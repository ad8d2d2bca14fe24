/* =================================================================================================
 * sccg.h -- C ABI of the B200-native SCCG hot path (libsccg_b200.so).
 *
 * The reference (Jan-Celin/SCCG-genome-compression) has no plugin / FFI interface: its hot path is a
 * set of free functions inside two executables.  Each entry point below replaces one of those
 * functions; the reference line it stands in for is cited.  Plain C, plain pointers and sizes.
 *
 * Conventions
 *   - every function returns SCCG_OK (0) or a negative SCCG_E_* code; sccg_last_error() gives text
 *     for the calling thread's most recent failure.  No exceptions cross this boundary.
 *   - host-pointer entry points: caller-owned input buffers, read-only, not retained after return;
 *     outputs are allocated by the library and released with sccg_free().
 *   - *_device entry points take DEVICE pointers (inputs already resident in HBM) and leave the
 *     result in device memory owned by the context (valid until the next call on that context).
 *     Every device input must be 16-byte aligned and have at least 16 READABLE bytes past its
 *     length (the kernels use 8/16-byte vector loads that may run past the last symbol; the
 *     content of that slack is irrelevant).  A cudaMalloc'ed buffer of len + 16 bytes qualifies.
 *   - one opaque context per GPU; calls on one context must be serialised by the caller, distinct
 *     contexts may be driven from distinct host threads.
 *   - there is NO CPU fallback: without a usable CUDA device sccg_create() fails.
 * ================================================================================================= */
#ifndef SCCG_H
#define SCCG_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCCG_OK 0
#define SCCG_E_CUDA (-1)        /* CUDA runtime / launch failure, or no device                            */
#define SCCG_E_ARG (-2)         /* invalid argument (NULL, negative size, size >= 2^31, unsupported k)    */
#define SCCG_E_FORMAT (-3)      /* malformed record stream: the reference would throw (stoi) -> exit 1    */
#define SCCG_E_BOUNDS (-4)      /* abs+len exceeds the reference: decompression.cpp:223-229 -> exit(1)    */
#define SCCG_E_NOMEM (-5)
#define SCCG_E_STOI (-6)        /* compress only: the target carries a literal '(' that makes the reference's text-level
                                 * delta_encode throw from stoi (compression.cpp:279) -> "Error: stoi", exit 1, and
                                 * compressed_genome.txt stays un-rewritten.  The output buffer IS filled with that
                                 * pre-delta image (release it as usual) so a caller can leave the same file behind. */

typedef struct sccg_ctx sccg_ctx;

/* vector<Position> of match_sequences (compression.cpp:20-24, :36) as struct-of-arrays.
 * Record i is a match iff lit_off[i+1] == lit_off[i]; then (p[i], l[i]) = (start_reference, length).
 * Otherwise it is a literal run lits[lit_off[i] .. lit_off[i+1]) and p[i] = -1, l[i] = 0. */
typedef struct {
    int64_t  n;
    int32_t* p;
    int32_t* l;
    int64_t* lit_off;   /* n + 1 entries */
    char*    lits;
} sccg_records;

/* phases whose device time the last call measured with CUDA events on the context's stream */
typedef struct {
    float h2d_ms;         /* host -> device copies (0 for *_device entry points)        */
    float kernels_ms;     /* every kernel of the call, first launch to last completion  */
    float d2h_ms;         /* device -> host copy of the result                          */
    float match_ms;       /* compress: segment-match (local) or index+parse (global)    */
    float serialize_ms;   /* compress: run lists + record text ; decompress: tokenizer  */
    float gather_ms;      /* decompress: reference-copy / literal gather + case/N/wrap  */
    int32_t launches;     /* kernels launched by the call                               */
    int32_t mode;         /* compress: 0 local, 1 global                                */
    int32_t front_steps;  /* global parse: exact steps the sequential front executed itself */
    int32_t spec_rounds;  /* global parse: speculation rounds (1 + number of "lost" re-speculations) */
    float index_ms;       /* global mode: reference k-mer index (hash + radix sort + bucket table)       */
    float parse_ms;       /* global mode: speculative chunk parse + exact front + concatenation        */
    float exchange_ms;    /* multi-GPU layer: the collective(s) of the last sccg_mgpu_* call           */
    int32_t index_stride; /* global mode: 1 = index of every reference k-mer, n = sampled index (every n-th position) */
} sccg_profile;

sccg_ctx*   sccg_create(int device);                 /* NULL on failure (see sccg_last_error)      */
void        sccg_destroy(sccg_ctx* ctx);
const char* sccg_last_error(void);
void        sccg_free(void* p);                      /* releases any buffer returned by the library */
void        sccg_records_free(sccg_records* r);
int         sccg_get_profile(sccg_ctx* ctx, sccg_profile* out);
const char* sccg_version(void);
/* copies n bytes of a device buffer returned by a *_device entry point to host memory (stream-ordered, blocking) */
int         sccg_download(sccg_ctx* ctx, const void* d_src, int64_t n, void* h_dst);

/* compress_genome minus file I/O and the external 7z stage (compression.cpp:320-579).
 * ref / tgt: raw symbols as read_genomes_from_files leaves them (:181-220): case preserved, no
 * newlines.  header: the target's first '>' line (must start with '>'), may be empty.  out: the final, delta-encoded
 * compressed_genome.txt image.  mode_out: 0 = local segment matching, 1 = global fallback. */
int sccg_compress(sccg_ctx* ctx, const char* ref, int64_t ref_len, const char* tgt, int64_t tgt_len,
                  const char* header, int64_t header_len, char** out, int64_t* out_len, int* mode_out);

/* same, inputs already in device memory; the encoded image stays on the device:
 * *d_out is owned by the context and valid until its next call. */
int sccg_compress_device(sccg_ctx* ctx, const void* d_ref, int64_t ref_len, const void* d_tgt, int64_t tgt_len,
                         const char* header, int64_t header_len, void** d_out, int64_t* out_len, int* mode_out);

/* match_sequences(Sr, St, k, m, global, offset)  (compression.cpp:36-179).
 * global == 0: one segment pair, nr and nt <= 1000 and 10 <= k <= 32 (the reference's own call sites, :401 k = 14 and :428
 *              k = 10; its match_sequences has no such limits, larger local inputs return SCCG_E_ARG here).
 * global != 0: whole sequences, any length < 2^31, 8 <= k <= 16 and 0 <= m <= 120 (:561 calls it with k = 14, m = 100). */
int sccg_match_sequences(sccg_ctx* ctx, const char* Sr, int64_t nr, const char* St, int64_t nt,
                         int k, int m, int global, int offset, sccg_records* out);

/* reconstruct_genome(reference, encoded, n_indices, lowercase_indices)  (decompression.cpp:117-279).
 * ref must already be prepared as decompress_genome does (:105-110).  out: the 50-column wrapped
 * sequence text ending in '\n' (what main writes after "<header>\n", :322). */
int sccg_reconstruct(sccg_ctx* ctx, const char* ref, int64_t ref_len, const char* encoded, int64_t enc_len,
                     const char* n_idx, int64_t n_len, const char* low_idx, int64_t low_len,
                     char** out, int64_t* out_len);

/* same, reference and the three text lines already in device memory; result stays on the device */
int sccg_reconstruct_device(sccg_ctx* ctx, const void* d_ref, int64_t ref_len, const void* d_encoded, int64_t enc_len,
                            const void* d_n_idx, int64_t n_len, const void* d_low_idx, int64_t low_len,
                            void** d_out, int64_t* out_len);

/* decompress_genome's in-memory part + reconstruct_genome + main's header line
 * (decompression.cpp:66-110, :117-279, :322): intermediate file image + raw reference symbols in,
 * reconstructed_genome.fa image out. */
int sccg_decompress(sccg_ctx* ctx, const char* ref_raw, int64_t ref_len, const char* intermediate, int64_t inter_len,
                    char** out, int64_t* out_len);

/* *_into variants: identical, but the result is written into a buffer of the caller instead of a fresh allocation
 * (page-locked host memory gives full PCIe speed).  If out_cap is too small they return SCCG_E_ARG and *out_len holds
 * the required size. */
int sccg_compress_into(sccg_ctx* ctx, const char* ref, int64_t ref_len, const char* tgt, int64_t tgt_len,
                       const char* header, int64_t header_len, char* out, int64_t out_cap, int64_t* out_len, int* mode_out);
int sccg_reconstruct_into(sccg_ctx* ctx, const char* ref, int64_t ref_len, const char* encoded, int64_t enc_len,
                          const char* n_idx, int64_t n_len, const char* low_idx, int64_t low_len,
                          char* out, int64_t out_cap, int64_t* out_len);
int sccg_decompress_into(sccg_ctx* ctx, const char* ref_raw, int64_t ref_len, const char* intermediate, int64_t inter_len,
                         char* out, int64_t out_cap, int64_t* out_len);

/* Output-range sharding of decompression over several GPUs: the part-th of n_parts contiguous pieces of the file image that
 * sccg_decompress would produce.  out receives the piece, *part_offset its offset inside the image, *part_len its length and
 * *total_len the length of the whole image.  Only the reference chunks the piece copies from are uploaded (local-mode files),
 * so N GPUs share the PCIe traffic of one pair; the pieces can be written straight to their offsets of the output file. */
int sccg_decompress_part(sccg_ctx* ctx, const char* ref_raw, int64_t ref_len, const char* intermediate, int64_t inter_len,
                         int part, int n_parts, char* out, int64_t out_cap, int64_t* part_offset, int64_t* part_len, int64_t* total_len);

/* Many targets against one reference (the reference repository's use case: every individual's chromosome against the same
 * reference chromosome, one `compress` / `decompress` process per pair -- compression.cpp:584-610, decompression.cpp:281-329 --
 * each of which re-reads the reference).  sccg_reference_set uploads the raw reference symbols once and keeps them in device
 * memory; the *_resident calls then move only the target (or the record file and the reconstructed text) over PCIe and give
 * exactly the bytes of sccg_compress_into / sccg_decompress_into with that reference.  The caller's reference buffer is free
 * again when sccg_reference_set returns. */
int sccg_reference_set(sccg_ctx* ctx, const char* ref, int64_t ref_len);
int sccg_reference_clear(sccg_ctx* ctx);
int sccg_compress_resident_into(sccg_ctx* ctx, const char* tgt, int64_t tgt_len, const char* header, int64_t header_len,
                                char* out, int64_t out_cap, int64_t* out_len, int* mode_out);
int sccg_decompress_resident_into(sccg_ctx* ctx, const char* intermediate, int64_t inter_len, char* out, int64_t out_cap, int64_t* out_len);

/* Region extraction: pieces of the decoded sequence without producing the whole image (what `samtools faidx` /
 * `bedtools getfasta` do with a plain FASTA).  D is the decoded sequence of the intermediate file: the reconstructed_genome.fa
 * image that sccg_decompress produces for the same inputs, without its first line ("<header>\n") and without any '\n' -- N runs
 * re-inserted, lowercase restored.  *seq_len receives len(D).  A region {start, end} is 0-based and half-open in D,
 * 0 <= start <= end <= len(D); empty regions are allowed, and regions may come in any order, overlap and repeat.  out receives
 * D[start_0:end_0] + D[start_1:end_1] + ... in the order given, with no separators: region i begins at the sum of the lengths
 * before it, and *out_len is the total.
 * Errors, in this order:
 *   SCCG_E_ARG before any device work: a NULL pointer with a non-zero count, start < 0 or start > end, a total of 2^31 bytes or
 *     more or n_regions >= 2^31, out_cap smaller than the total (*out_len then holds the required size);
 *   SCCG_E_FORMAT / SCCG_E_BOUNDS exactly when sccg_decompress fails on the same inputs, whatever the regions;
 *   SCCG_E_ARG when a region ends past len(D) (*seq_len holds len(D), so the caller can clamp).
 * Local-mode files upload and prepare only the reference chunks that the regions copy from; global-mode files need the whole
 * reference (every N of it is removed first).  Profile: h2d_ms (host -> device copies), serialize_ms (front end), gather_ms
 * (region gather), kernels_ms (all kernels), d2h_ms (device -> host copy of the result), launches. */
typedef struct { int64_t start, end; } sccg_region;
int sccg_extract(sccg_ctx* ctx, const char* ref_raw, int64_t ref_len, const char* intermediate, int64_t inter_len,
                 const sccg_region* regions, int64_t n_regions, char* out, int64_t out_cap, int64_t* out_len, int64_t* seq_len);
/* the same with the reference FASTA file image (as sccg_decompress_fasta takes it) */
int sccg_extract_fasta(sccg_ctx* ctx, const char* ref_file, int64_t ref_file_len, const char* intermediate, int64_t inter_len,
                       const sccg_region* regions, int64_t n_regions, char* out, int64_t out_cap, int64_t* out_len, int64_t* seq_len);
/* the same against the resident reference (sccg_reference_set; SCCG_E_ARG without one) */
int sccg_extract_resident(sccg_ctx* ctx, const char* intermediate, int64_t inter_len,
                          const sccg_region* regions, int64_t n_regions, char* out, int64_t out_cap, int64_t* out_len, int64_t* seq_len);

/* Archives: a record file opened once, then queried many times (what the index of `samtools faidx` does for a plain FASTA).
 * sccg_archive_open runs the decoder's front end of one intermediate file against the RESIDENT reference (sccg_reference_set)
 * and keeps the tables a gather reads (record bytes, segment tables, N runs, lowercase runs -- run lists out of order are
 * normalised here, once) in device memory owned by the handle; no later call on the context touches them.  It fails with
 * SCCG_E_FORMAT / SCCG_E_BOUNDS exactly when sccg_decompress_resident_into fails on the same file, and with SCCG_E_ARG without a
 * resident reference.  The first open of a local-mode (global-mode) file after sccg_reference_set prepares the upper-cased
 * (N-stripped and upper-cased) form of the resident reference, which then stays next to it.  Profile after an open:
 * serialize_ms (front end), kernels_ms, h2d_ms (record file upload).
 * sccg_archive_info: len(D) of the archive, its mode (0 local, 1 global) and the device memory it holds (any pointer may be NULL).
 * sccg_archive_close releases one archive; sccg_destroy releases every archive still open on the context.
 * An archive is bound to the resident reference it was opened against: after sccg_reference_set or sccg_reference_clear on
 * its context, a query that names it fails with SCCG_E_ARG (open it again); it can still be closed. */
typedef struct sccg_archive sccg_archive;
int sccg_archive_open(sccg_ctx* ctx, const char* intermediate, int64_t inter_len, sccg_archive** out);
int sccg_archive_info(const sccg_archive* a, int64_t* seq_len, int* mode, int64_t* device_bytes);
int sccg_archive_close(sccg_ctx* ctx, sccg_archive* a);

/* Pieces of any number of open archives in one call: query i is D_a[start:end] of archive archives[archive] (D as for
 * sccg_extract) when strand is 0, and its reverse complement when strand is 1 (`bedtools getfasta -s`, `samtools faidx -i`).
 * out receives the pieces in the order given, with no separators; *out_len is the total.  Complement, case kept: A<->T,
 * C<->G, R<->Y, K<->M, B<->V, D<->H; every other byte (S, W, N, anything else) maps to itself.
 * Errors, all SCCG_E_ARG and all before any device work, in this order: a NULL pointer with a non-zero count or a negative
 * count (2^31 or more archives or queries); then for each query in turn: an archive index out of range, a NULL archive, an
 * archive opened on another context, an archive whose resident reference has since been replaced or cleared, start < 0 or
 * start > end, end past len(D) of that archive, a strand other than 0 or 1; then a total of 2^31 bytes or more, and out_cap
 * smaller than the total (*out_len then holds the required size).
 * One host -> device copy (the query table), one launch, one device -> host copy.  Profile: h2d_ms, gather_ms, kernels_ms,
 * d2h_ms, launches. */
typedef struct { int64_t archive, start, end, strand; } sccg_query;
int sccg_archive_extract(sccg_ctx* ctx, sccg_archive* const* archives, int64_t n_archives, const sccg_query* queries, int64_t n_queries,
                         char* out, int64_t out_cap, int64_t* out_len);

/* Pattern search in windows of open archives: window w is D_a[start:end] of archives[archive] (D as for sccg_archive_extract:
 * N runs re-inserted, lowercase restored).  Pattern i is patterns[pattern_off[i] .. pattern_off[i+1]); 1 to 1024 patterns of
 * 1 to 64 bytes.  strands: 1 forward, 2 reverse complement, 3 both.
 * Match rule, per byte, after ASCII upper-casing both sides: pattern byte p matches D byte d when up(d) == up(p), or when p is
 * an IUPAC code (R Y S W K M B D H V N) and up(d) is one of A/C/G/T in its set.  So N in a pattern matches any base and N, an
 * N gap in D matches only pattern N, and any other byte matches only itself.
 * A hit (window w, pos, pattern i, strand s, mismatches k): D[pos, pos + len_i) lies inside window w and differs in exactly
 * k <= max_mismatches positions from pattern i (s = 0) or from its reverse complement (s = 1; the complement of
 * sccg_archive_extract, which maps the IUPAC codes).  pos is an absolute D coordinate, the leftmost base on either strand (BED).
 * Every hit is reported (overlapping occurrences, both strands of a palindrome, an occurrence once per window that holds it),
 * in (window, pos, pattern, strand) order.  Windows shorter than a pattern give no hits for it.
 * *n_hits always receives the total.  hits == NULL counts only.  When hits is given and the total exceeds hits_cap, the call
 * returns SCCG_E_ARG with the required count in *n_hits (hits then holds an unspecified prefix).
 * Errors, all SCCG_E_ARG and all before any device work, in this order: a NULL pointer with a non-zero count or a negative
 * count (2^31 or more archives, windows or patterns); a pattern count outside 1..1024, pattern_off not non-decreasing from 0
 * or a pattern length outside 1..64, max_mismatches < 0 or >= the shortest pattern's length, strands not in 1..3; then the
 * query checks of sccg_archive_extract over the windows (archive index out of range, NULL archive, another context, a
 * replaced or cleared resident reference, start < 0 or start > end, end past len(D)).
 * Windows may add up to any size: the call splits them into launches (SCCG_SEARCH_SPLIT: candidate positions per launch) and
 * copies the hits out after each.  Cost grows linearly with the number of patterns.  Profile: h2d_ms (window and pattern
 * tables), gather_ms (search kernels), kernels_ms, d2h_ms (hits), launches. */
typedef struct { int64_t archive, start, end; } sccg_window;
typedef struct { int64_t window, pos; int32_t pattern, strand, mismatches, reserved; } sccg_hit;
int sccg_archive_search(sccg_ctx* ctx, sccg_archive* const* archives, int64_t n_archives, const sccg_window* windows, int64_t n_windows,
                        const char* patterns, const int64_t* pattern_off, int64_t n_patterns, int max_mismatches, int strands,
                        sccg_hit* hits, int64_t hits_cap, int64_t* n_hits);

/* Pattern search with insertions and deletions: the inputs of sccg_archive_search (windows, archives, 1 to 1024 patterns of 1
 * to 64 bytes, strands 1/2/3, the per-byte match rule), with unit-cost Levenshtein distance ed(P, X) instead of mismatches: a
 * substitution is a pair of bytes that does not match under the rule, an insertion an extra D byte, a deletion a missing
 * pattern byte.  Strand 1 searches the reverse complement of the pattern (the same complement) on forward D.
 * A hit (window w, start, end, pattern i, strand s, edits): for window w = D_a[ws:we], pattern i (its reverse complement for
 * s = 1) and an end e with ws < e <= we, let d(e) = min over ws <= x <= e of ed(P, D[x:e]).  There is a hit iff
 * d(e) <= max_edits, with end = e, edits = d(e) and start = the largest x reaching d(e) (the shortest text).  start and end
 * are absolute D coordinates: [start, end) is a BED interval.  At most one hit per (w, e, i, s), in (window, end, pattern,
 * strand) order.  Hits are not clustered: every qualifying end is reported, so with max_edits >= 1 an exact occurrence
 * ending at e also gives 1-edit hits ending at e - 1 and e + 1.  Windows shorter than len_i - max_edits give no hits for i.
 * With max_edits = 0 the hits are exactly the sccg_archive_search hits with max_mismatches = 0 (start = pos,
 * end = pos + len_i).  For every sccg_archive_search hit (w, pos, i, s, m) there is a hit here at end = pos + len_i with
 * edits <= m.
 * *n_hits always receives the total.  hits == NULL counts only.  When hits is given and the total exceeds hits_cap, the call
 * returns SCCG_E_ARG with the required count in *n_hits (hits then holds an unspecified prefix).
 * Errors: those of sccg_archive_search, in the same order and all before any device work, with max_edits in place of
 * max_mismatches (>= 0 and below the shortest pattern's length).
 * Windows may add up to any size: the call splits them into launches (SCCG_SEARCH_SPLIT: candidate end positions per launch).
 * Cost grows linearly with the number of patterns.  Profile: h2d_ms (window and pattern tables), gather_ms (search kernels),
 * kernels_ms, d2h_ms (hits), launches. */
typedef struct { int64_t window, start, end; int32_t pattern, strand, edits, reserved; } sccg_edit_hit;
int sccg_archive_search_edits(sccg_ctx* ctx, sccg_archive* const* archives, int64_t n_archives, const sccg_window* windows, int64_t n_windows,
                              const char* patterns, const int64_t* pattern_off, int64_t n_patterns, int max_edits, int strands,
                              sccg_edit_hit* hits, int64_t hits_cap, int64_t* n_hits);

/* Differences of open archives from the resident reference, as normalised variant records.  R is the raw resident reference
 * (the bytes given to sccg_reference_set), D an archive's decoded sequence (as for sccg_archive_extract), up() ASCII
 * upper-casing of a-z; every comparison is on up() bytes, so lowercase is never a difference.  A record says that
 * up(R[pos:end]) is replaced by up(D[d_start:d_end]); its ALT bytes, exactly up(D[d_start:d_end]), are at alt + alt_off.
 * The records of an archive are a function of its record file and R alone:
 *  1. copy pieces: the decoder's token segments in D order, each (x, p, l) with up(D[x:x+l]) == up(R[p:p+l]) in raw
 *     coordinates (global mode: split wherever D skips a target N run or R skips a reference N run); literal runs and
 *     pieces with l = 0 are not pieces;
 *  2. anchors: with M = the maximum of p + l over all earlier pieces (0 at the start), piece (x, p, l) clipped at its start
 *     by s = max(0, M - p) is the anchor (x + s, p + s, l - s) when s < l.  Anchors increase strictly in D and in R;
 *  3. gaps: between consecutive anchors, before the first (from (0, 0)) and after the last (to (len(D), len(R))), the
 *     reference gap G_R and the D gap G_D.  Equal lengths: one substitution record per maximal run of differing positions.
 *     Different lengths: trim the longest common suffix, then the longest common prefix of what is left; both sides still
 *     non-empty make one complex record, otherwise one insertion (end == pos) or deletion (d_end == d_start);
 *  4. left-alignment: each insertion and deletion moves left one base at a time (pos, end, d_start and d_end decrease by
 *     1) while pos is greater than the end the previous record had at step 3 (0 for the first) and up(R[pos - 1]) equals
 *     the last byte of the allele (R[end - 1] for a deletion, the last ALT byte for an insertion): bcftools norm's
 *     left-alignment, bounded by the previous record, so records never overlap;
 *  5. windows: window w = {archive, start, end} is in REFERENCE coordinates (0 <= start <= end <= len(R)) and returns the
 *     records of its archive whose pos lies in [start, end) (a window that ends at len(R) also takes the insertions at
 *     pos = len(R)), each with window = w.  A window filters the records of the
 *     whole archive and never changes one; overlapping and repeated windows each report theirs.
 * Records come in (window, pos, d_start) order.  Per archive: pos_j >= end_{j-1} and d_start_j >= d_end_{j-1}, the stretches
 * between records are equally long and equal under up(), a substitution differs at every position, other records differ
 * in their first and in their last byte unless a side is empty, and splicing the ALTs into up(R) gives up(D).
 * Not done: realignment (the records are a faithful account of the encoding: permuted blocks appear as large complex
 * records), splitting complex records or MNPs (bcftools norm -a), genotypes or phasing.
 * *n_vars and *alt_len always receive the totals.  vars == NULL counts only.  When either cap is too small the call returns
 * SCCG_E_ARG with both totals set.  Errors, all SCCG_E_ARG and all before any device work, in this order: a NULL pointer with
 * a non-zero count or a negative count (2^31 or more archives or windows, a negative cap); then for each window the archive
 * checks of sccg_archive_extract (index out of range, NULL archive, another context, a replaced or cleared resident
 * reference), start < 0 or start > end, end > len(R); then the caps.  Profile: h2d_ms (archive and window tables), gather_ms
 * (variant kernels), kernels_ms, d2h_ms (records and ALT bytes), launches. */
typedef struct { int64_t window, pos, end, d_start, d_end, alt_off; } sccg_variant;
int sccg_archive_variants(sccg_ctx* ctx, sccg_archive* const* archives, int64_t n_archives, const sccg_window* windows, int64_t n_windows,
                          sccg_variant* vars, int64_t vars_cap, int64_t* n_vars, char* alt, int64_t alt_cap, int64_t* alt_len);

/* Coordinates lifted between the resident reference R and open archives D (R, D and up() as for sccg_archive_variants).
 * The records of archive a are its whole-archive records of sccg_archive_variants after step 4, in (pos, d_start) order
 * (windows play no part).  A record is a substitution when end - pos == d_end - d_start; otherwise it changes length.
 * Ownership: every reference base outside all [pos, end) spans lies in a stretch and is aligned one to one with a D base;
 * the D bases of a record, D[d_start:d_end], are owned by its pos (the rule by which a variants window reports a record).
 * from = 0, reference -> archive: query [s, e) with 0 <= s <= e <= len(R) lifts to [F(s), F+(e)), where F(b) is the number
 * of D bases whose owner or aligned reference base is < b, and F+(e) = F(e) except F+(len(R)) = len(D) (the end only: a
 * window that ends at len(R) also owns the records at pos = len(R), so [len(R), len(R)) owns a trailing insertion).  In
 * closed form, with j the last record with pos < b: F(b) = d_end_j + max(0, b - end_j), or b when there is none.
 * from = 1, archive -> reference: the mirror image.  [x, y) with 0 <= x <= y <= len(D) lifts to [G(x), G+(y)), the roles of
 * (pos, end) and (d_start, d_end) swapped: the reference bases of a record are owned by its d_start, and G+(len(D)) = len(R)
 * (so deletions at the end of D belong to a window that ends there).
 * Per query, in query order: start, end (the lifted interval; it may be empty, e.g. inside a deletion); same (source bases of
 * the query in stretches, copied identically); subst (source bases of the query inside substitution records); records (the
 * records the query owns: for from = 0 exactly what sccg_archive_variants reports for the window {archive, s, e}); flags:
 * SCCG_LIFT_START_INSIDE a record that begins before s reaches past it (the lifted start skips its ALT),
 * SCCG_LIFT_END_INSIDE an owned record reaches past e, SCCG_LIFT_LENGTH_CHANGE an owned record changes length; for from = 1
 * the same on the D side.  The sum same + subst + (the query's source bases inside length-changing records) is e - s.
 * Splice identity (from = 0): up(D[start:end]) equals up(R[s:e]) with each owned record's reference span replaced by its
 * ALT (a span that reaches past e taken whole) and the reference bases of [s, e) inside a record that begins before s
 * dropped.  For from = 1, the mirror: up(R[start:end]) equals up(D[x:y]) with each owned record's D span replaced by
 * up(R[pos:end]) (taken whole past y) and the D bases of [x, y) inside a record that begins before x dropped.
 * Lift tables: each archive's records are kept on the device as a compact sorted table (record bounds in both systems and
 * prefix sums of record lengths), one exactly-sized allocation held by the archive.  A call builds the tables of all its
 * archives that have none in one pipeline run; later calls only search.  sccg_archive_info's device_bytes includes the table
 * once built; sccg_archive_close and sccg_destroy release it.  A failed build (e.g. SCCG_E_NOMEM) leaves every archive
 * without a partial table and usable.  An archive whose resident reference was replaced fails the checks below, so a table
 * is never stale.
 * Errors, all SCCG_E_ARG and all before any device work, in this order: a NULL pointer with a non-zero count or a negative
 * count (2^31 or more archives or queries); then, the first failing check over all queries: the archive checks of
 * sccg_archive_extract (index out of range, NULL archive, another context, a replaced or cleared resident reference), from
 * not 0 or 1, start < 0 or start > end, end past len(R) (from = 0) or len(D) (from = 1).
 * Each query does two binary searches of its archive's table.  Profile: h2d_ms (query table), gather_ms (lift kernel),
 * kernels_ms (every kernel, table builds included: the build costs kernels_ms - gather_ms), d2h_ms (results), launches. */
typedef struct { int64_t archive, start, end; int32_t from, reserved; } sccg_lift_query;
typedef struct { int64_t start, end, same, subst, records; int32_t flags, reserved; } sccg_lift;
enum { SCCG_LIFT_START_INSIDE = 1, SCCG_LIFT_END_INSIDE = 2, SCCG_LIFT_LENGTH_CHANGE = 4 };
int sccg_archive_liftover(sccg_ctx* ctx, sccg_archive* const* archives, int64_t n_archives, const sccg_lift_query* queries, int64_t n_queries,
                          sccg_lift* out);

/* FASTA file images in: read_genomes_from_files (compression.cpp:181-220) and the reference reader of decompress_genome
 * (decompression.cpp:47-58) run on the device -- header lines skipped ('>' at a line start; in the target only the first one,
 * which becomes the header line of the output), isspace() bytes removed -- followed by sccg_compress / sccg_decompress.
 * ref_file / tgt_file: the raw bytes of the FASTA files.  The host never touches the symbols. */
int sccg_compress_fasta(sccg_ctx* ctx, const char* ref_file, int64_t ref_file_len, const char* tgt_file, int64_t tgt_file_len,
                        char** out, int64_t* out_len, int* mode_out);
int sccg_decompress_fasta(sccg_ctx* ctx, const char* ref_file, int64_t ref_file_len, const char* intermediate, int64_t inter_len,
                          char** out, int64_t* out_len);

/* *_into variants of the FASTA entry points, and page-locked host memory for their buffers (cudaMallocHost: copies run at full
 * PCIe speed and overlap with kernels; the batch drivers read the files straight into such buffers). */
void* sccg_pinned_alloc(int64_t bytes);              /* NULL on failure */
void  sccg_pinned_free(void* p);
int sccg_compress_fasta_into(sccg_ctx* ctx, const char* ref_file, int64_t ref_file_len, const char* tgt_file, int64_t tgt_file_len,
                             char* out, int64_t out_cap, int64_t* out_len, int* mode_out);
int sccg_decompress_fasta_into(sccg_ctx* ctx, const char* ref_file, int64_t ref_file_len, const char* intermediate, int64_t inter_len,
                               char* out, int64_t out_cap, int64_t* out_len);

/* Streaming decompression: the reconstructed_genome.fa image (decompression.cpp:316-323) is handed to `sink` piece by piece, in
 * order (offset = position of the piece in the image), from a page-locked double buffer owned by the context: while the sink
 * writes piece j to the output file, piece j + 1 crosses PCIe.  A non-zero return of the sink aborts the call.  Every error of
 * the record stream (SCCG_E_FORMAT / SCCG_E_BOUNDS) is reported BEFORE the first piece is delivered. */
typedef int (*sccg_sink_fn)(void* user, int64_t offset, const char* data, int64_t len);
int sccg_decompress_stream(sccg_ctx* ctx, const char* ref_raw, int64_t ref_len, const char* intermediate, int64_t inter_len,
                           sccg_sink_fn sink, void* user, int64_t* total_len);
int sccg_decompress_fasta_stream(sccg_ctx* ctx, const char* ref_file, int64_t ref_file_len, const char* intermediate, int64_t inter_len,
                                 sccg_sink_fn sink, void* user, int64_t* total_len);

/* One chromosome over several GPUs (the local segment-matching path, compression.cpp:381-481, sharded by segment range).
 * Shard r owns the segment pairs [seg_base, seg_base + n) and is given exactly the matching slices: ref[seg_base*1000 ..),
 * tgt[seg_base*1000 ..); the last shard's target slice runs to the end of the target.  sccg_shard_match does the matching and
 * reports the values that cross shard borders; the caller combines the reports of all shards into one sccg_shard_carry per
 * shard (sccg-genome-compression_b200/sharding.py: plan_carries) and sccg_shard_write then produces the shard's part of the
 * lowercase-run line and of the body.  Concatenating the parts in shard order (after "<header>\n", with "\n,\n" between the
 * two lines) gives exactly the file sccg_compress writes.  If any shard reports abort_inside / has_paren, or a border window
 * aborts, the pair must go through sccg_compress on one GPU (global mode / text-level delta). */
typedef struct {
    int64_t n_segments;
    int32_t abort_inside;       /* T2 abort condition met inside the shard (compression.cpp:462) */
    int32_t has_paren;          /* the target slice contains '(' */
    int32_t head_status[4];     /* first 4 segments: bit 0 = increments the T2 counter, bit 1 = can end an abort window */
    int32_t tail_status[4];     /* last 4 segments, in order */
    int32_t has_match;          /* at least one match token */
    int32_t last_p;             /* absolute reference position of the last match token */
    int64_t n_runs;             /* lowercase runs inside the target slice */
    int64_t first_run_start, first_run_len, last_run_start, last_run_len;   /* absolute target coordinates */
} sccg_shard_info;
typedef struct {
    int32_t prev_p;             /* p of the last match token of the shards before this one (0: none) */
    int32_t skip_first_run;     /* the first lowercase run continues a run of the previous shard */
    int64_t extra_last_len;     /* symbols the following shards add to the last lowercase run */
    int64_t prev_run_start;     /* start of the last run that begins before this shard (0: none) */
    int32_t last_run_reaches_end; /* the (lengthened) last run ends at the end of the target */
    int32_t reserved;
} sccg_shard_carry;
int sccg_shard_match(sccg_ctx* ctx, const char* ref_slice, int64_t ref_len, const char* tgt_slice, int64_t tgt_len,
                     int64_t seg_base, int is_last, sccg_shard_info* info);
int sccg_shard_write(sccg_ctx* ctx, const sccg_shard_carry* carry, char** low_part, int64_t* low_len, char** body_part, int64_t* body_len);

/* ---- Multi-GPU layer (host side in C++, NCCL C API underneath; csrc/sccg_mgpu.cuh) ------------------------------------------
 * The reference is one single-threaded process per FASTA pair (compression.cpp:584-610, decompression.cpp:281-329); a genome is
 * 24 invocations.  Here one rank (a process or a host thread) drives one GPU through its own sccg_ctx, and a communicator ties
 * the ranks of one job together.  NCCL carries only (a) the 128-byte border records of a segment-range sharded pair and (b) the
 * encoded record streams on their way to rank 0; no collective sits on a kernel's critical path.  libnccl.so.2 is bound at run
 * time: the single-GPU entry points above do not need it.
 *   sccg_mgpu_unique_id : rank 0 creates the rendezvous token (ncclGetUniqueId); the caller hands the 128 bytes to the other
 *                         ranks (torch.distributed / MPI broadcast, a file, or simply memory when the ranks are threads).
 *   sccg_mgpu_init      : joins the communicator; collective over all ranks.  ctx stays owned by the caller and must outlive it. */
#define SCCG_MGPU_ID_BYTES 128
typedef struct sccg_mgpu sccg_mgpu;
int  sccg_mgpu_unique_id(char* id128);
int  sccg_mgpu_init(sccg_ctx* ctx, const char* id128, int rank, int world, sccg_mgpu** out);
void sccg_mgpu_destroy(sccg_mgpu* g);
int  sccg_mgpu_rank(const sccg_mgpu* g);
int  sccg_mgpu_world(const sccg_mgpu* g);

/* (1) By chromosome.  sccg_mgpu_assign: longest-processing-time packing of n_items pairs (lengths[] = target symbols) onto
 * `world` ranks, deterministic; owner[i] = rank of pair i.  Every rank then runs compress_genome (compression.cpp:320-579) on
 * its own pairs with sccg_mgpu_compress_item (host buffers, pipelined upload) or ..._item_device (inputs resident in HBM): the
 * encoded image stays in device memory and is appended to the rank's outgoing streams (at most 64 per gather).
 * sccg_mgpu_gather (collective) moves every rank's streams to rank 0 -- sizes by ncclAllGather, payload by grouped
 * ncclSend / ncclRecv -- and copies them into `out` back to back; stream k is item_ids[k] at out + item_offs[k], item_lens[k]
 * bytes long.  On the other ranks out / item_* may be NULL.  Too small a buffer: SCCG_E_ARG with *total / *n_items set. */
int sccg_mgpu_assign(const int64_t* lengths, int n_items, int world, int32_t* owner);
int sccg_mgpu_compress_item(sccg_mgpu* g, int32_t item, const char* ref, int64_t ref_len, const char* tgt, int64_t tgt_len,
                            const char* header, int64_t header_len, int64_t* enc_len, int* mode_out);
int sccg_mgpu_compress_item_device(sccg_mgpu* g, int32_t item, const void* d_ref, int64_t ref_len, const void* d_tgt, int64_t tgt_len,
                                   const char* header, int64_t header_len, int64_t* enc_len, int* mode_out);
int sccg_mgpu_stash_device(sccg_mgpu* g, int32_t item, const void* d_data, int64_t len);
int sccg_mgpu_gather(sccg_mgpu* g, char* out, int64_t out_cap, int32_t* item_ids, int64_t* item_offs, int64_t* item_lens, int32_t cap_items,
                     int32_t* n_items, int64_t* total);
/* same, but the gathered streams stay in rank 0's device memory (*d_out: owned by the communicator, valid until its next gather;
 * sccg_download fetches pieces of it): the counterpart of sccg_compress_device for a job whose inputs are resident in HBM */
int sccg_mgpu_gather_device(sccg_mgpu* g, void** d_out, int32_t* item_ids, int64_t* item_offs, int64_t* item_lens, int32_t cap_items,
                            int32_t* n_items, int64_t* total);

/* (2) One pair over all ranks by segment range (the local path, compression.cpp:381-481).  Collective: every rank passes the
 * same host buffers but uploads and matches only its own slice; the border records travel in one ncclAllGather, every rank
 * derives the same carries, and the parts of the two text lines go to rank 0, which receives exactly the file sccg_compress
 * writes (*out_len = its length; 0 on the other ranks).  A pair that leaves the local path (T2 abort -> global mode, a '(' in
 * the target) or is too small to shard is compressed by rank 0 alone; *sharded_out tells which way it went. */
int sccg_mgpu_compress_sharded(sccg_mgpu* g, const char* ref, int64_t ref_len, const char* tgt, int64_t tgt_len, const char* header, int64_t header_len,
                               char* out, int64_t out_cap, int64_t* out_len, int* mode_out, int* sharded_out);

/* (3) Decompression of one pair by output range: this rank's piece of the reconstructed file image (sccg_decompress_part with
 * part = rank, n_parts = world).  Nothing is gathered: the pieces are written straight to their offsets of the output file. */
int sccg_mgpu_decompress_sharded(sccg_mgpu* g, const char* ref_raw, int64_t ref_len, const char* intermediate, int64_t inter_len,
                                 char* out, int64_t out_cap, int64_t* part_offset, int64_t* part_len, int64_t* total_len);

#ifdef __cplusplus
}
#endif
#endif /* SCCG_H */
