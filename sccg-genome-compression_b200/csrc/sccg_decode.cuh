// Record-decode (decompression): reconstruct_genome, decompression.cpp:117-279, on the device.
//
//   run-list parsers (:126-207)  -> parse_runs: number tokenizer + prefix sum of the deltas; runs stay
//                                   (start,len) pairs instead of one int per lowercase / N base
//   token decode (:210-236)      -> classify every byte of the body (literal / token start / inside
//                                   a token), three prefix sums (output offset, segment index, token
//                                   index), prefix sum of the token deltas -> absolute positions
//   N merge, tolower, 50-col wrap (:241-274) -> ONE output-centric gather kernel: every thread
//                                   produces 16 bytes of the final text straight from the reference /
//                                   the literal bytes (no intermediate "stripped" sequence in HBM)
//
// Input grammar.  Body tokens are read as the reference reads them: the token ends at the first ')', its two numbers go
// through std::stoi (leading isspace, '+' or '-', any number of leading zeros, whatever follows the digits is ignored).
// SCCG_E_FORMAT where that stoi throws, and for three pinned divergences (INTEGRATION.md section 5): a negative token
// length, a token whose ')' lies more than TOK_MAX bytes after its '(', and a token without ',' before its ')'.  Run
// lists: exactly what the compressor emits (N1 in SURVEY.md) plus the optional ',' after a tuple that the reference
// tolerates; other run-list text is SCCG_E_FORMAT (pinned too).  Run lists that are out of order or overlap are put in
// order first (reconstruct_normalize), as the reference's sort does.
#pragma once
#include "sccg_compress.cuh"
#include "sccg_strip.cuh"
#include "sccg_bulk.cuh"

#include <algorithm>
#include <utility>
#include <vector>

namespace sccg {

static const int TOK_MAX = 25;        // "(-2147483648,2147483647)" is 24 characters

enum DecScalar { D_ERR = 0, D_NSEG, D_NTOK, D_LS, D_LOW_ITEMS, D_N_ITEMS, D_NSUM, D_LSUM, D_STRIP, D_COUNT = 16 };
enum DecErr { DE_FORMAT = 1, DE_BOUNDS = 2, DE_LOW_UNSORTED = 4, DE_N_UNSORTED = 8 };   // the last two are no errors yet: reconstruct_normalize decides
static const u32 DE_HARD = DE_FORMAT | DE_BOUNDS, DE_SOFT = DE_LOW_UNSORTED | DE_N_UNSORTED;

__device__ __forceinline__ bool is_digit(u8 c) { return c >= '0' && c <= '9'; }

// std::stoi on s[i..] restricted to what the writers emit: optional '-', 1..10 digits, fits in int.
// returns the number of characters consumed, 0 on failure
__device__ __forceinline__ int parse_int(const u8* __restrict__ s, i64 i, i64 n, int* out) {
    int w = 0;
    bool neg = false;
    if (i < n && s[i] == '-') { neg = true; ++w; }
    i64 v = 0;
    int nd = 0;
    while (i + w < n && is_digit(s[i + w]) && nd < 11) { v = v * 10 + (s[i + w] - '0'); ++w; ++nd; }
    if (nd == 0 || nd > 10) return 0;
    if (neg) v = -v;
    if (v > 2147483647LL || v < -2147483648LL) return 0;
    *out = (int)v;
    return w;
}

// is byte i inside a "(...)" token that started before i?  (the last parenthesis in the TOK_MAX bytes before i is '(')
__device__ __forceinline__ bool inside_token(const u8* __restrict__ s, i64 i) {
    for (int d = 1; d <= TOK_MAX; ++d) {
        if (i - d < 0) return false;
        u8 c = s[i - d];
        if (c == '(') return true;
        if (c == ')') return false;
    }
    return false;
}

// byte i is copied to the output as a literal symbol (decompression.cpp:233)
__device__ __forceinline__ bool is_literal(const u8* __restrict__ s, i64 i) { return s[i] != '(' && !inside_token(s, i); }

// parses "(a,b)" at s[i]; returns its length in characters or 0
__device__ __forceinline__ int parse_tuple(const u8* __restrict__ s, i64 i, i64 n, int* a, int* b) {
    int w = 1;
    int k = parse_int(s, i + w, n, a);
    if (!k) return 0;
    w += k;
    if (i + w >= n || s[i + w] != ',') return 0;
    ++w;
    k = parse_int(s, i + w, n, b);
    if (!k) return 0;
    w += k;
    if (i + w >= n || s[i + w] != ')') return 0;
    return w + 1;
}

// a body token at s[i] == '(' (decompression.cpp:215-219): the token ends at the first ')' (where dec_chunk ends it), the
// delta is stoi from the byte after '(', the length is stoi from the byte after the first ',' inside the token.  Canonical
// tokens, all the writers emit, pass parse_tuple; anything else takes the stoi parse.  false -> SCCG_E_FORMAT: stoi throws,
// or one of two pinned classes.  A ')' more than TOK_MAX bytes after the '(' lies beyond the look-back that decides a
// chunk's entry state (dec_chunk would have classified the token's tail as literals), and a token without ',' before
// its ')' takes its length from the next ',' anywhere in the body in the reference (or from the body's first byte).
// The run lists keep parse_tuple / parse_int alone.
__device__ __forceinline__ bool parse_body_token(const u8* __restrict__ s, i64 i, i64 n, int* d, int* l) {
    if (parse_tuple(s, i, n, d, l)) return true;
    const u8* t = s + i;
    const int m = n - i - 1 < TOK_MAX ? (int)(n - i - 1) : TOK_MAX;      // bytes after the '(' the token may use
    int comma = 0, close = 0;
    for (int k = 1; k <= m; ++k) {
        if (t[k] == ')') { close = k; break; }
        if (t[k] == ',' && !comma) comma = k;
    }
    if (!close || !comma) return false;
    return dt_stoi(t, 1u, (u32)comma, d) && dt_stoi(t, (u32)comma + 1u, (u32)close, l);
}

// ------------------------------------------------------------------------------------------------
// body tokenizer (decompression.cpp:213-236): every thread owns 16 consecutive bytes of the record stream.  The state
// machine  outside --'('--> inside --')'--> outside  is evaluated on bit masks (byte-SWAR compares of the own 16 bytes
// and of the 32 bytes before them for the entry state), so a warp never serialises over per-byte branches:
//   token starts   "(d,l)"  -> one copy segment of l symbols taken from the reference
//   literal runs            -> one copy segment per maximal run of literal bytes
// Pass 1 (dec_count_k) leaves per-thread totals (decoded symbols, segments, tokens); after three scans, pass 2
// (dec_emit_k) rebuilds the masks and writes the compacted tables directly:
//   seg_dst[k] : offset of segment k in the decoded (N-free) sequence
//   seg_src[k] : literal run -> index into enc | SEG_LIT_FLAG ; token -> token index (absolute position filled later)
//   tok_delta[t], tok_len[t]
// No per-byte side arrays exist: the stream is read twice (2 B per encoded byte) + 24 B per 16-byte chunk.
// ------------------------------------------------------------------------------------------------
#define SEG_LIT_FLAG 0x4000000000000000LL
#define SEG_BAD_PTR (-1LL)               // seg_ptr of a token that failed the bounds check: no reader may dereference it
static const int DEC_T = 256;
static const int DEC_PER_THREAD = 16;

struct DecChunk { u32 tok, lit, segl; };       // bit b <=> byte i0 + b: token start / literal symbol / first byte of a literal run

__device__ __forceinline__ u32 paren_mask16(ulonglong2 v, u8 ch) { return movemask8(eq_flags8(v.x, ch)) | (movemask8(eq_flags8(v.y, ch)) << 8); }

// enc is 16-byte aligned with >= 16 readable bytes past ne; i0 is a multiple of 16 and < ne
__device__ __forceinline__ DecChunk dec_chunk(const u8* __restrict__ enc, i64 ne, i64 i0) {
    const ulonglong2 own = *reinterpret_cast<const ulonglong2*>(enc + i0);
    const i64 left = ne - i0;
    const u32 V = left >= 16 ? 0xffffu : ((1u << (int)left) - 1u);
    const u32 O = paren_mask16(own, '(') & V, C = paren_mask16(own, ')') & V;
    // entry state from the 32 bytes before the chunk (bit j <=> byte i0 - 32 + j)
    u32 Op = 0, Cp = 0;
    if (i0 >= 16) {
        const ulonglong2 p1 = *reinterpret_cast<const ulonglong2*>(enc + i0 - 16);
        Op = paren_mask16(p1, '(') << 16; Cp = paren_mask16(p1, ')') << 16;
        if (i0 >= 32) {
            const ulonglong2 p0 = *reinterpret_cast<const ulonglong2*>(enc + i0 - 32);
            Op |= paren_mask16(p0, '('); Cp |= paren_mask16(p0, ')');
        }
    }
    // inside_token(i0): the last parenthesis among bytes i0-25 .. i0-1 is '('      (bits 7..31)
    bool in = (Op & 0xffffff80u) > (Cp & 0xffffff80u);
    // is_literal(i0 - 1): not '(' and not inside a token that started in bytes i0-26 .. i0-2   (bits 6..30)
    const bool prev_lit = i0 > 0 && !(Op >> 31) && !((Op & 0x7fffffc0u) > (Cp & 0x7fffffc0u));
    u32 inside = 0;
    int last = 0;
    for (u32 pp = O | C; pp; pp &= pp - 1) {
        const int b = __ffs((int)pp) - 1;
        const bool is_open = (O >> b) & 1u;
        if (in) { inside |= (2u << b) - (1u << last); if (!is_open) in = false; }     // the token runs through its ')'
        else if (is_open) in = true;                                                   // a stray ')' is a literal (:233)
        last = b + 1;
    }
    if (in) inside |= 0x10000u - (1u << last);
    DecChunk c;
    c.tok = O & ~inside;
    c.lit = V & ~inside & ~c.tok;
    c.segl = c.lit & ~((c.lit << 1) | (prev_lit ? 1u : 0u));
    return c;
}

__global__ void __launch_bounds__(DEC_T) dec_count_k(const u8* __restrict__ enc, i64 ne, u32* __restrict__ th_sym, u32* __restrict__ th_seg, u32* __restrict__ th_tok,
                                                    u32* __restrict__ sc) {
    const i64 t = (i64)blockIdx.x * DEC_T + threadIdx.x;
    const i64 i0 = t * DEC_PER_THREAD;
    if (i0 >= ne) return;
    const DecChunk c = dec_chunk(enc, ne, i0);
    u32 sym = (u32)__popc(c.lit);
    for (u32 m = c.tok; m; m &= m - 1) {
        int d = 0, l = 0;
        if (!parse_body_token(enc, i0 + __ffs((int)m) - 1, ne, &d, &l) || l < 0) atomicOr(&sc[D_ERR], (u32)DE_FORMAT);
        else sym += (u32)l;
    }
    th_sym[t] = sym; th_seg[t] = (u32)__popc(c.tok | c.segl); th_tok[t] = (u32)__popc(c.tok);
}

// th_* hold exclusive prefixes by now
__global__ void __launch_bounds__(DEC_T) dec_emit_k(const u8* __restrict__ enc, i64 ne, const u32* __restrict__ th_sym, const u32* __restrict__ th_seg,
                                                   const u32* __restrict__ th_tok, u32* __restrict__ seg_dst, i64* __restrict__ seg_src,
                                                   int* __restrict__ tok_delta, int* __restrict__ tok_len) {
    const i64 t = (i64)blockIdx.x * DEC_T + threadIdx.x;
    const i64 i0 = t * DEC_PER_THREAD;
    if (i0 >= ne) return;
    const DecChunk c = dec_chunk(enc, ne, i0);
    u32 nseg = th_seg[t], ntok = th_tok[t];
    const u32 sym0 = th_sym[t];
    u32 tok_syms = 0;                                                  // symbols of the tokens seen so far in this chunk
    for (u32 m = c.tok | c.segl; m; m &= m - 1) {
        const int b = __ffs((int)m) - 1;
        const u32 at = sym0 + (u32)__popc(c.lit & ((1u << b) - 1u)) + tok_syms;
        seg_dst[nseg] = at;
        if ((c.tok >> b) & 1u) {
            int d = 0, l = 0;
            parse_body_token(enc, i0 + b, ne, &d, &l);                 // validated by dec_count_k
            seg_src[nseg] = (i64)ntok; tok_delta[ntok] = d; tok_len[ntok] = l;
            tok_syms += (u32)l; ++ntok;
        } else {
            seg_src[nseg] = (i64)(i0 + b) | SEG_LIT_FLAG;
        }
        ++nseg;
    }
}

// ------------------------------------------------------------------------------------------------
// run lists (decompression.cpp:126-207): "(d,len)" | "d," | "d"
// ------------------------------------------------------------------------------------------------
// 16 bytes of the list per thread, classified on bit masks like the body tokenizer above (a thread per byte and a flag word per
// byte cost 19 + 13 + 18 us on the 1.5 MB list of a chr1-sized file).  Same grammar checks as the reference's stoi / substr
// calls would make (decompression.cpp:126-207):
//   inside "(...)"  : digits, '-', ',' and the closing ')' only
//   outside         : '(' starts a tuple "(d,len)", len >= 0; a digit or '-' whose predecessor is neither starts a single "d"
//                     that must be followed by ',' or the end; ',' must follow a digit or ')'; nothing else
struct RunChunk { u32 items, tuples, err; };      // bit b <=> byte i0 + b: item start / tuple start / grammar error
__device__ __forceinline__ u64 digit_flags8(u64 w) {
    u64 x = w & SCCG_B7F;
    u64 ge = x + (u64)(0x80 - '0') * SCCG_B01, gt = x + (u64)(0x80 - '9' - 1) * SCCG_B01;
    return ge & ~gt & ~w & SCCG_B80;
}
__device__ __forceinline__ u32 eq_mask16(u64 lo, u64 hi, u8 ch) { return movemask8(eq_flags8(lo, ch)) | (movemask8(eq_flags8(hi, ch)) << 8); }
// s may have any alignment (it points into the file image); i0 is a multiple of 16 and < n; 16 readable bytes past n
__device__ __forceinline__ RunChunk run_chunk(const u8* __restrict__ s, i64 n, i64 i0) {
    const u64 a0 = ld_unaligned64(s + i0), a1 = ld_unaligned64(s + i0 + 8);
    const i64 left = n - i0;
    const u32 V = left >= 16 ? 0xffffu : ((1u << (int)left) - 1u);
    const u32 O = eq_mask16(a0, a1, '(') & V, C = eq_mask16(a0, a1, ')') & V, M = eq_mask16(a0, a1, ',') & V;
    const u32 Dg = (movemask8(digit_flags8(a0)) | (movemask8(digit_flags8(a1)) << 8)) & V;
    const u32 D = Dg | (eq_mask16(a0, a1, '-') & V);
    u32 Op = 0, Cp = 0;                                       // the 32 bytes before the chunk (bit j <=> byte i0 - 32 + j)
    if (i0 >= 16) {
        const u64 p2 = ld_unaligned64(s + i0 - 16), p3 = ld_unaligned64(s + i0 - 8);
        Op = eq_mask16(p2, p3, '(') << 16; Cp = eq_mask16(p2, p3, ')') << 16;
        if (i0 >= 32) {
            const u64 p0 = ld_unaligned64(s + i0 - 32), p1 = ld_unaligned64(s + i0 - 24);
            Op |= eq_mask16(p0, p1, '('); Cp |= eq_mask16(p0, p1, ')');
        }
    }
    bool in = (Op & 0xffffff80u) > (Cp & 0xffffff80u);        // inside_token(i0)
    u32 inside = 0;
    int last = 0;
    for (u32 pp = O | C; pp; pp &= pp - 1) {
        const int b = __ffs((int)pp) - 1;
        const bool is_open = (O >> b) & 1u;
        if (in) { inside |= (2u << b) - (1u << last); if (!is_open) in = false; }
        else if (is_open) in = true;
        last = b + 1;
    }
    if (in) inside |= 0x10000u - (1u << last);
    inside &= V;
    const u8 pb = i0 > 0 ? s[i0 - 1] : (u8)0;
    const u32 p_dg = is_digit(pb) ? 1u : 0u, p_dl = (is_digit(pb) || pb == '-') ? 1u : 0u, p_cl = pb == ')' ? 1u : 0u;
    RunChunk c;
    c.tuples = O & ~inside;
    const u32 lit = V & ~inside & ~c.tuples;
    c.items = c.tuples | (lit & D & ~((D << 1) | p_dl));
    c.err = (inside & ~(D | M | C)) | (lit & ~(D | M)) | (lit & M & ~((Dg << 1) | p_dg | (C << 1) | p_cl));
    return c;
}

static const int RUNS_T = 256;
__global__ void __launch_bounds__(RUNS_T) runs_count16_k(const u8* __restrict__ s, i64 n, u32* __restrict__ cnt, u32* __restrict__ masks, u32* __restrict__ sc) {
    const i64 t = (i64)blockIdx.x * RUNS_T + threadIdx.x;
    const i64 i0 = t * 16;
    if (i0 >= n) return;
    const RunChunk c = run_chunk(s, n, i0);
    bool bad = c.err != 0u;
    for (u32 m = c.items; m; m &= m - 1) {
        const int b = __ffs((int)m) - 1;
        int d = 0, l = 0;
        if ((c.tuples >> b) & 1u) { if (!parse_tuple(s, i0 + b, n, &d, &l) || l < 0) bad = true; }
        else { const int w = parse_int(s, i0 + b, n, &d); if (!w || (i0 + b + w < n && s[i0 + b + w] != ',')) bad = true; }
    }
    if (bad) atomicOr(&sc[D_ERR], (u32)DE_FORMAT);
    cnt[t] = (u32)__popc(c.items);
    masks[t] = c.items | (c.tuples << 16);
}
// cnt holds the exclusive prefix by now
__global__ void __launch_bounds__(RUNS_T) runs_emit16_k(const u8* __restrict__ s, i64 n, const u32* __restrict__ cnt, const u32* __restrict__ masks,
                                                        int* __restrict__ delta, int* __restrict__ len) {
    const i64 t = (i64)blockIdx.x * RUNS_T + threadIdx.x;
    const i64 i0 = t * 16;
    if (i0 >= n) return;
    const u32 mk = masks[t];
    u32 k = cnt[t];
    for (u32 m = mk & 0xffffu; m; m &= m - 1) {
        const int b = __ffs((int)m) - 1;
        int d = 0, l = 1;
        if ((mk >> (16 + b)) & 1u) { if (!parse_tuple(s, i0 + b, n, &d, &l)) { d = 0; l = 0; } }   // (validated by runs_count16_k; the caller does not get here after an error)
        else if (!parse_int(s, i0 + b, n, &d)) { d = 0; l = 0; }
        delta[k] = d; len[k] = l;
        ++k;
    }
}

// start[k] = prefix sum of deltas; validates ascending, non-overlapping runs
// start[k] = prefix sum of deltas.  The compressor only writes ascending, non-overlapping runs; the reference's parser expands
// whatever it reads into single positions and sorts them (decompression.cpp:138-164), so a list that is out of order or
// overlaps is legal input: it raises a soft flag and reconstruct_normalize puts it in order before it is used.
__global__ void runs_finish_k(const int* __restrict__ delta, const int* __restrict__ len, const u32* __restrict__ delta_excl, u32 K,
                              int* __restrict__ start, u32* __restrict__ sc, u32 soft_bit) {
    u32 k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    int st = (int)(delta_excl[k] + (u32)delta[k]);
    start[k] = st;
    if ((st < 0 && len[k] > 0) || len[k] < 0) atomicOr(&sc[D_ERR], (u32)DE_FORMAT);       // a negative position: undefined behaviour in the reference (:257)
    if (k > 0) {
        int pst = (int)delta_excl[k];                             // previous start
        if ((i64)st < (i64)pst + (i64)len[k - 1]) atomicOr(&sc[D_ERR], soft_bit);
    }
}

struct RunTable { int* start; int* len; u32* cum; u32 K; };        // cum[k] = sum of len[0..k)

static int parse_runs(sccg_ctx* c, const u8* d_text, i64 n, int slot_base, u32* sc, int sc_items, u32* sc_sum, u32 soft_bit, RunTable* out) {
    // slot_base: 4 consecutive buffer slots
    out->start = nullptr; out->len = nullptr; out->cum = nullptr; out->K = 0;
    if (n <= 0) {
        SCCG_TRY(buf(c, slot_base + 1, 4, &out->start));
        SCCG_TRY(buf(c, slot_base + 2, 4, &out->len));
        SCCG_TRY(buf(c, slot_base + 3, 4, &out->cum));
        return SCCG_OK;
    }
    const i64 nch = (n + 15) / 16;
    u32* cnt = nullptr;
    SCCG_TRY(buf(c, slot_base, (size_t)nch * 2 + 2, &cnt));
    u32* masks = cnt + nch + 1;
    unsigned g = div_up(nch, RUNS_T);
    LAUNCH(c, runs_count16_k, dim3(g), dim3(RUNS_T), 0, d_text, n, cnt, masks, sc);
    SCCG_TRY(scan_exclusive_u32(c, cnt, cnt, nch, sc + sc_items));
    u32 h[D_COUNT];
    SCCG_TRY(read_scalars(c, sc, h, D_COUNT));
    if (h[D_ERR] & DE_HARD) return set_error(SCCG_E_FORMAT, "malformed run list (the reference would throw from stoi or misbehave)");
    u32 K = h[sc_items];
    int *delta = nullptr;
    u32* excl = nullptr;
    SCCG_TRY(buf(c, slot_base + 1, (size_t)K + 1, &out->start));
    SCCG_TRY(buf(c, slot_base + 2, (size_t)K + 1, &out->len));
    SCCG_TRY(buf(c, slot_base + 3, (size_t)K + 1, &out->cum));
    SCCG_TRY(buf(c, B_TILE0, (size_t)K + 1, &delta));
    SCCG_TRY(buf(c, B_TILE1, (size_t)K + 1, &excl));
    out->K = K;
    if (K == 0) return SCCG_OK;
    LAUNCH(c, runs_emit16_k, dim3(g), dim3(RUNS_T), 0, d_text, n, (const u32*)cnt, (const u32*)masks, delta, out->len);
    SCCG_TRY(scan_exclusive_u32(c, (const u32*)delta, excl, (i64)K, nullptr));
    LAUNCH(c, runs_finish_k, dim3(div_up(K, 256)), dim3(256), 0, (const int*)delta, (const int*)out->len, (const u32*)excl, K, out->start, sc, soft_bit);
    SCCG_TRY(scan_exclusive_u32(c, (const u32*)out->len, out->cum, (i64)K, sc_sum));
    return SCCG_OK;
}

// ------------------------------------------------------------------------------------------------
// the gather: N merge (:244-252), tolower (:255-262), 50-column wrap (:266-274)
// ------------------------------------------------------------------------------------------------
// last k with arr[k] <= x, or -1
__device__ __forceinline__ int upper_idx_i32(const int* __restrict__ arr, int n, i64 x) {
    int lo = 0, hi = n;
    while (lo < hi) { int mid = (lo + hi) >> 1; if ((i64)arr[mid] <= x) lo = mid + 1; else hi = mid; }
    return lo - 1;
}
__device__ __forceinline__ int upper_idx_u32(const u32* __restrict__ arr, int n, i64 x) {
    int lo = 0, hi = n;
    while (lo < hi) { int mid = (lo + hi) >> 1; if ((i64)arr[mid] <= x) lo = mid + 1; else hi = mid; }
    return lo - 1;
}

struct GatherArgs {
    const u8* ref; const u8* enc;
    const u32* seg_dst; const i64* seg_src; const int* tok_abs; int nseg;
    const i64* seg_ptr;      // resolved source of segment k: literal run -> offset into enc | SEG_LIT_FLAG, token -> offset into ref
    const int4* tile_win;    // per 4 KiB tile of text: {first segment, first lowercase run, N symbols before the tile, staged path ok}
    const int* n_start; const int* n_len; const u32* n_cum; int n_k;
    const int* l_start; const int* l_len; int l_k;
    i64 Ls;          // symbols decoded from the record stream (N-free)
    i64 Lm;          // symbols in the N-merged sequence
    i64 total;       // bytes of wrapped text
    u8* out;
    u32 tile0;       // first tile of this launch (the text may be produced in several launches, see decompress_host)
    const u32* err;  // the decoder's error word: while a run list awaits normalisation (DE_SOFT) the tables must not be used
};

static const int GATHER_T = 256;
static const int GATHER_TILE = GATHER_T * 16;

// last k in [lo, hi] with arr[k] <= x, or lo - 1   (lo may be -1: then the search starts at 0)
__device__ __forceinline__ int bounded_upper_i32(const int* __restrict__ arr, int lo, int hi, i64 x) {
    int a = lo < 0 ? 0 : lo, b = hi + 1;
    while (a < b) { int mid = (a + b) >> 1; if ((i64)arr[mid] <= x) a = mid + 1; else b = mid; }
    return a - 1;
}
__device__ __forceinline__ int bounded_upper_u32(const u32* __restrict__ arr, int lo, int hi, i64 x) {
    int a = lo < 0 ? 0 : lo, b = hi + 1;
    while (a < b) { int mid = (a + b) >> 1; if ((i64)arr[mid] <= x) a = mid + 1; else b = mid; }
    return a - 1;
}

// symbol index (N-merged coordinates) shown at / just before output byte q
__device__ __forceinline__ i64 gather_sym_of(i64 q, i64 Lm) {
    i64 line = q / (WRAP + 1);
    int col = (int)(q - line * (WRAP + 1));
    i64 b = line * WRAP + (col < WRAP ? col : WRAP - 1);
    return b < Lm ? b : Lm - 1;
}
// N-free coordinate of merged symbol b (or of the first N-free symbol after it when b is an N)
__device__ __forceinline__ i64 gather_strip(const GatherArgs& a, i64 b) {
    int nk = upper_idx_i32(a.n_start, a.n_k, b);
    if (nk < 0) return b;
    i64 st = a.n_start[nk], ln = a.n_len[nk];
    if (b < st + ln) return st - (i64)a.n_cum[nk];
    return b - ((i64)a.n_cum[nk] + ln);
}

// warp-cooperative 32-ary search: last k with arr[k] <= x, or -1.  All 32 lanes, uniform arguments.
__device__ __forceinline__ int warp_upper_i32(const int* __restrict__ arr, int n, i64 x) {
    const int lane = lane_of();
    int lo = 0, hi = n;                                           // the count of elements <= x lies in [lo, hi]
    while (hi > lo) {
        int step = (hi - lo + 31) >> 5;
        int pi = lo + lane * step;
        bool le = pi < hi && (i64)arr[pi] <= x;
        int c = __popc(__ballot_sync(SCCG_FULL_MASK, le));
        if (c == 0) { hi = lo; break; }
        int nlo = lo + (c - 1) * step + 1;
        int nhi = lo + c * step; if (nhi > hi) nhi = hi;
        lo = nlo; hi = nhi;
    }
    return lo - 1;
}
__device__ __forceinline__ int warp_upper_u32(const u32* __restrict__ arr, int n, i64 x) {
    const int lane = lane_of();
    int lo = 0, hi = n;
    while (hi > lo) {
        int step = (hi - lo + 31) >> 5;
        int pi = lo + lane * step;
        bool le = pi < hi && (i64)arr[pi] <= x;
        int c = __popc(__ballot_sync(SCCG_FULL_MASK, le));
        if (c == 0) { hi = lo; break; }
        int nlo = lo + (c - 1) * step + 1;
        int nhi = lo + c * step; if (nhi > hi) nhi = hi;
        lo = nlo; hi = nhi;
    }
    return lo - 1;
}

// one symbol of the final text (slow path): N merge (:244-252), copy (:230-233), tolower (:255-262), wrap (:266-274)
__device__ __forceinline__ u8 gather_byte(const GatherArgs& a, const int* win, u32 q) {
    if ((i64)q == a.total - 1) return '\n';                       // the final newline (:274)
    u32 line = q / (u32)(WRAP + 1);
    int col = (int)(q - line * (u32)(WRAP + 1));
    if (col == WRAP) return '\n';
    i64 bb = (i64)line * WRAP + col;
    int nk = bounded_upper_i32(a.n_start, win[2], win[3], bb);
    i64 s = bb;
    bool is_n = false;
    if (nk >= 0) {
        i64 st = a.n_start[nk], ln = a.n_len[nk];
        if (bb < st + ln) is_n = true;
        else s = bb - ((i64)a.n_cum[nk] + ln);
    }
    u8 o = 'N';
    if (!is_n) {
        int sk = bounded_upper_u32(a.seg_dst, win[0], win[1], s);
        i64 src = a.seg_ptr[sk];
        i64 within = s - (i64)a.seg_dst[sk];
        if (src < 0) o = '?';                                     // SEG_BAD_PTR (the call returns an error)
        else o = (src & SEG_LIT_FLAG) ? a.enc[(src & ~SEG_LIT_FLAG) + within] : a.ref[src + within];
    }
    int lk = bounded_upper_i32(a.l_start, win[4], win[5], bb);
    if (lk >= 0 && bb < (i64)a.l_start[lk] + (i64)a.l_len[lk]) o = lower1(o);
    return o;
}

// Every thread owns one aligned 16-byte piece of the final text.  Fast path (the piece lies inside one copy segment,
// touches no N run and is entirely inside or outside a lowercase run): two unaligned 8-byte loads, SWAR tolower,
// newline spliced in with shifts, one 16-byte store.  Pieces that straddle a boundary are handed to the warp: 16 lanes
// per piece, one symbol per lane, so boundary pieces cost one pass instead of a 16-step serial loop in a single lane.
// (generic tile path: used for the rare tiles that contain re-inserted N runs; win = 6 ints of shared memory)
__device__ __forceinline__ void gather_tile_generic(const GatherArgs& a, int* win, i64 Q0, int byte_off) {
    const int lane = lane_of(), warp = (int)(threadIdx.x >> 5);
    const i64 Q1 = (Q0 + GATHER_TILE < a.total ? Q0 + GATHER_TILE : a.total) - 1;     // last byte of the tile
    if (a.Lm > 0) {
        // six 32-ary searches shared among the warps of the CTA
        for (int wi = warp; wi < 6; wi += (int)(blockDim.x >> 5)) {
            const i64 bq = gather_sym_of((wi & 1) ? Q1 : Q0, a.Lm);
            int r;
            if (wi < 2) {
                i64 sx = gather_strip(a, bq);
                if (sx > a.Ls - 1) sx = a.Ls - 1;
                r = a.nseg ? warp_upper_u32(a.seg_dst, a.nseg, sx) : -1;
            } else if (wi < 4) r = warp_upper_i32(a.n_start, a.n_k, bq);
            else r = warp_upper_i32(a.l_start, a.l_k, bq);
            if (lane == 0) win[wi] = r;
        }
    }
    __syncthreads();
    const i64 q0 = Q0 + byte_off + (i64)threadIdx.x * 16;
    const bool live = q0 < a.total;
    const u32 line0 = (u32)((u64)q0 / (u32)(WRAP + 1));
    const int col0 = (int)((u64)q0 - (u64)line0 * (WRAP + 1));
    const int c = WRAP - col0;                                   // offset of the '\n' inside this piece if < 16
    const i64 b = (i64)line0 * WRAP + col0;                      // first symbol of the piece
    const int ns = c < 16 ? 15 : 16;
    bool fast = live && (q0 + 16 <= a.total - 1) && a.Lm > 0;
    i64 noff = 0;
    int lower_all = 0, sk = -1;
    if (fast) {
        int nk = bounded_upper_i32(a.n_start, win[2], win[3], b + ns - 1);
        if (nk >= 0) {
            i64 en = (i64)a.n_start[nk] + a.n_len[nk];
            if (en > b) fast = false; else noff = (i64)a.n_cum[nk] + a.n_len[nk];
        }
    }
    if (fast) {
        i64 s = b - noff;
        sk = bounded_upper_u32(a.seg_dst, win[0], win[1], s);
        i64 seg_end = sk + 1 < a.nseg ? (i64)a.seg_dst[sk + 1] : a.Ls;
        if (sk < 0 || s + ns > seg_end || a.seg_ptr[sk] < 0) fast = false;
    }
    if (fast) {
        int lk = bounded_upper_i32(a.l_start, win[4], win[5], b + ns - 1);
        if (lk >= 0) {
            i64 ls = a.l_start[lk], le = ls + a.l_len[lk];
            if (le > b) { if (ls <= b && le >= b + ns) lower_all = 1; else fast = false; }
        }
    }
    if (fast) {
        i64 src = a.seg_ptr[sk];
        i64 within = (b - noff) - (i64)a.seg_dst[sk];
        const u8* sp = (src & SEG_LIT_FLAG) ? a.enc + (src & ~SEG_LIT_FLAG) + within : a.ref + src + within;
        u64 w0 = ld_unaligned64(sp), w1 = ld_unaligned64(sp + 8);
        if (lower_all) { w0 = lower8(w0); w1 = lower8(w1); }
        if (c < 8) {
            u64 lowmask = c ? (~0ull >> (64 - 8 * c)) : 0ull;
            u64 carry = w0 >> 56;
            w0 = (w0 & lowmask) | ((u64)'\n' << (8 * c)) | ((w0 & ~lowmask) << 8);
            w1 = (w1 << 8) | carry;
        } else if (c < 16) {
            int cc = c - 8;
            u64 lowmask = cc ? (~0ull >> (64 - 8 * cc)) : 0ull;
            w1 = (w1 & lowmask) | ((u64)'\n' << (8 * cc)) | ((w1 & ~lowmask) << 8);
        }
        ulonglong2 v; v.x = w0; v.y = w1;
        *reinterpret_cast<ulonglong2*>(a.out + q0) = v;
    }
    // ---- boundary pieces: two per round, 16 lanes each, one symbol per lane
    u32 slow = __ballot_sync(SCCG_FULL_MASK, live && !fast);
    const u32 my_q0 = (u32)q0;                                   // total < 2^32
    while (slow) {
        int s1 = __ffs((int)slow) - 1; slow &= slow - 1;
        int s2 = -1;
        if (slow) { s2 = __ffs((int)slow) - 1; slow &= slow - 1; }
        int src = lane < 16 ? s1 : s2;
        u32 pq0 = __shfl_sync(SCCG_FULL_MASK, my_q0, src < 0 ? 0 : src);
        if (src >= 0) {
            u32 q = pq0 + (u32)(lane & 15);
            if ((i64)q < a.total) a.out[q] = gather_byte(a, win, q);
        }
    }
}


// ---- staged tile path ------------------------------------------------------------------------------------------------
// dst (shared, any alignment) <- src (global, any alignment), n bytes; whole warp, uniform arguments.  8 bytes per lane and
// step; the source may be read up to 15 bytes past its end (buffers carry that slack).
__device__ __forceinline__ void warp_copy_g2s(u8* dst, const u8* __restrict__ src, u32 n) {
    const u32 lane = (u32)lane_of();
    if (n <= 32) {                                                 // literal runs are mostly one symbol: one byte per lane, done
        if (lane < n) dst[lane] = src[lane];
        return;
    }
    u32 head = (u32)((8u - ((u32)(uintptr_t)dst & 7u)) & 7u);
    if (head > n) head = n;
    if (lane < head) dst[lane] = src[lane];
    const u32 nw = (n - head) >> 3;
    u64* d64 = reinterpret_cast<u64*>(dst + head);
    // the source alignment is the same for every word of the segment: hoisted, and the 64-bit funnel is two 32-bit ones
    const uintptr_t sa = (uintptr_t)(src + head);
    const uint2* s2 = reinterpret_cast<const uint2*>(sa & ~(uintptr_t)7);
    const u32 sb = (u32)(sa & 7u);
    if (sb == 0) {
        for (u32 i = lane; i < nw; i += 32) { const uint2 a = s2[i]; d64[i] = (u64)a.x | ((u64)a.y << 32); }
    } else if (sb < 4) {
        const u32 sh = sb * 8u;
        for (u32 i = lane; i < nw; i += 32) {
            const uint2 a = s2[i], b = s2[i + 1];
            d64[i] = (u64)__funnelshift_r(a.x, a.y, sh) | ((u64)__funnelshift_r(a.y, b.x, sh) << 32);
        }
    } else {
        const u32 sh = (sb - 4u) * 8u;
        for (u32 i = lane; i < nw; i += 32) {
            const uint2 a = s2[i], b = s2[i + 1];
            d64[i] = (u64)__funnelshift_r(a.y, b.x, sh) | ((u64)__funnelshift_r(b.x, b.y, sh) << 32);
        }
    }
    const u32 done = head + (nw << 3);
    if (done + lane < n) dst[done + lane] = src[done + lane];
}
// tolower on n bytes of shared memory (decompression.cpp:255-262); whole warp, uniform arguments
__device__ __forceinline__ void warp_lower_smem(u8* p, u32 n) {
    const u32 lane = (u32)lane_of();
    u32 head = (u32)((8u - ((u32)(uintptr_t)p & 7u)) & 7u);
    if (head > n) head = n;
    if (lane < head) p[lane] = lower1(p[lane]);
    const u32 nw = (n - head) >> 3;
    u64* p64 = reinterpret_cast<u64*>(p + head);
    for (u32 i = lane; i < nw; i += 32) p64[i] = lower8(p64[i]);
    const u32 done = head + (nw << 3);
    if (done + lane < n) p[done + lane] = lower1(p[done + lane]);
}

static const int GATHER_PAD = 64;

// seg_ptr[k]: where segment k copies from (one dependent load less in the gather).  Token segments: abs = prefix sum of
// the deltas (decompression.cpp:220-222) and the bounds check (:223-229) happen here (token t belongs to exactly one segment).
__global__ void dec_resolve_k(const i64* __restrict__ seg_src, const int* __restrict__ tok_delta, const int* __restrict__ tok_len,
                              const u32* __restrict__ delta_excl, int nseg, i64 nr, int* __restrict__ tok_abs, i64* __restrict__ seg_ptr, u32* __restrict__ sc) {
    int k = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (k >= nseg) return;
    const i64 src = seg_src[k];
    if (src & SEG_LIT_FLAG) { seg_ptr[k] = src; return; }
    const int a = (int)(delta_excl[src] + (u32)tok_delta[src]);   // prev_abs_start + delta, int arithmetic
    tok_abs[src] = a;
    const int len = tok_len[src];                                 // >= 0 (dec_count_k)
    const i64 end = (i64)(int)((u32)a + (u32)len);                // `absolute_start + length` is evaluated in int (:223)
    i64 ptr = (i64)a;
    if (end > nr) { atomicOr(&sc[D_ERR], (u32)DE_BOUNDS); ptr = SEG_BAD_PTR; }
    else if (a < 0 || (i64)a + (i64)len > nr) {                   // substr(pos > size) throws out_of_range; a wrapped `end` would read past the reference
        atomicOr(&sc[D_ERR], (u32)DE_FORMAT); ptr = SEG_BAD_PTR;
    }
    seg_ptr[k] = ptr;                                             // SEG_BAD_PTR: the gather copies nothing for this segment (the call fails anyway)
}

// merged-coordinate symbol range [b0, b1) shown in the text bytes [Q0, Qe)
__device__ __forceinline__ void tile_symbols(i64 Q0, i64 Qe, i64 Lm, u32* b0, u32* b1) {
    const u32 l0 = (u32)Q0 / (u32)(WRAP + 1), c0 = (u32)Q0 - l0 * (u32)(WRAP + 1);
    const u32 l1 = (u32)Qe / (u32)(WRAP + 1), c1 = (u32)Qe - l1 * (u32)(WRAP + 1);
    *b0 = l0 * WRAP + (c0 < (u32)WRAP ? c0 : (u32)WRAP);
    u32 e = l1 * WRAP + (c1 < (u32)WRAP ? c1 : (u32)WRAP);
    if ((i64)e > Lm) e = (u32)Lm;
    *b1 = e;
}

// per tile: where its copy segments and lowercase runs start (the searches leave the gather's critical path)
__global__ void dec_tile_win_k(GatherArgs a, unsigned ntiles, int4* __restrict__ tile_win) {
    const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ntiles || (*a.err & DE_SOFT)) return;
    const i64 Q0 = (i64)t * GATHER_TILE;
    const i64 Qe = Q0 + GATHER_TILE < a.total ? Q0 + GATHER_TILE : a.total;
    int4 w = make_int4(0, 0, 0, 0);
    u32 b0 = 0, b1 = 0;
    bool staged = a.Lm > 0;
    if (staged) { tile_symbols(Q0, Qe, a.Lm, &b0, &b1); if (b1 <= b0) staged = false; }   // nothing but the final newline
    u32 noff = 0;
    if (staged && a.n_k) {
        const int nk = upper_idx_i32(a.n_start, a.n_k, (i64)b1 - 1);
        if (nk >= 0) {
            if ((i64)a.n_start[nk] + a.n_len[nk] > (i64)b0) staged = false;               // an N run inside the tile
            else noff = a.n_cum[nk] + (u32)a.n_len[nk];
        }
    }
    if (staged) {
        w.x = upper_idx_u32(a.seg_dst, a.nseg, (i64)(b0 - noff));                         // segment that holds the first symbol
        int lk = upper_idx_i32(a.l_start, a.l_k, (i64)b0);                                // first lowercase run that reaches into the tile
        if (lk < 0 || (i64)a.l_start[lk] + a.l_len[lk] <= (i64)b0) ++lk;
        w.y = lk; w.z = (int)noff; w.w = 1;
    }
    tile_win[t] = w;
}

// One small CTA produces one 4 KiB tile of the final text.  Tiles without re-inserted N (all but a handful):
//   1. the copy segments that overlap the tile are copied by whole warps, segment by segment, from the reference / the
//      literal bytes into a shared-memory image of the tile's symbols (coalesced 8-byte loads, no per-byte search);
//   2. the lowercase runs that overlap the tile are applied to that image, run by run (decompression.cpp:255-262);
//   3. every thread formats a few 16-byte pieces of text from the image: newline every 50 symbols (:266-274), 16-byte stores.
// Tiles that contain N runs take the generic per-piece path above (gather_tile_generic).
#ifndef SCCG_GATHER_CTA
#define SCCG_GATHER_CTA 64
#endif
static const int GATHER_CTA = SCCG_GATHER_CTA;             // threads per 4 KiB tile: fewer threads per tile = more tiles in flight per SM
static const int GATHER_ROUNDS = GATHER_TILE / 16 / GATHER_CTA;
// Copy-engine version of the segment copy: when source and destination have the same 16-byte phase (the image is placed so
// that this holds for every token on diagonal 0, i.e. nearly all of a local-mode file) the aligned middle of the segment is
// ONE cp.async.bulk issued by one lane; the lanes only move the <= 15 bytes before and after it.
__device__ __forceinline__ void warp_copy_g2s_bulk(u8* dst, const u8* __restrict__ src, u32 n, u64* bar) {
    const u32 lane = (u32)lane_of();
    if (n < 64u || (((u32)(uintptr_t)src ^ smem_phase16(dst)) & 15u) != 0u) { warp_copy_g2s(dst, src, n); return; }
    const u32 head = (16u - ((u32)(uintptr_t)src & 15u)) & 15u;
    const u32 mid = (n - head) & ~15u, tail = n - head - mid;
    if (lane == 0) { mbar_expect_tx(bar, mid); bulk_g2s(dst + head, src + head, mid, bar); }
    if (lane < head) dst[lane] = src[lane];
    if (lane >= 16u && lane - 16u < tail) dst[head + mid + (lane - 16u)] = src[head + mid + (lane - 16u)];
}

__global__ void __launch_bounds__(GATHER_CTA) dec_gather_k(GatherArgs a) {
    __shared__ int win[6];
    __align__(16) __shared__ u8 Araw[GATHER_TILE + GATHER_PAD + 16];     // symbols of the tile (no newlines yet)
    __align__(16) __shared__ u8 O[GATHER_TILE];                          // the tile as it goes to memory
    __align__(8) __shared__ u64 bar;
    const int warp = (int)(threadIdx.x >> 5);
    const unsigned tile = blockIdx.x + a.tile0;
    const i64 Q0 = (i64)tile * GATHER_TILE;
    const i64 Qe = Q0 + GATHER_TILE < a.total ? Q0 + GATHER_TILE : a.total;           // exclusive
    if (*a.err & DE_SOFT) return;                                 // a run list is out of order: the caller normalises it and launches again
    const int4 tw = a.tile_win[tile];
    if (!tw.w) {
        // generic path: one 16-byte piece per thread and round
        for (int r = 0; r < GATHER_ROUNDS; ++r) {
            gather_tile_generic(a, win, Q0, r * GATHER_CTA * 16);
            __syncthreads();
        }
        return;
    }
    if (threadIdx.x == 0) mbar_init(&bar, 1u);
    u32 b0, b1;
    tile_symbols(Q0, Qe, a.Lm, &b0, &b1);
    const u32 noff = (u32)tw.z;
    const u32 s0 = b0 - noff, s1 = b1 - noff;                                         // N-free coordinates of the tile's symbols
    // the image starts at the 16-byte phase of its first symbol's coordinate: a token that copies reference symbol x to decoded
    // symbol x (diagonal 0) then has equally aligned source and destination
    u8* const A = Araw + (s0 & 15u);
    __syncthreads();                                                                  // the mbarrier is initialised
    // ---- 1. copy segments -> image.  Warp w owns the segments first + w, first + w + NW, ...; their descriptors are fetched
    //      32 at a time, one per lane (one memory round trip), and handed out by shuffles
    const int lane = lane_of();
    const int NW = GATHER_CTA / 32;
    for (int kb = tw.x + warp; kb < a.nseg; kb += 32 * NW) {
        const int kk = kb + lane * NW;
        u32 md0 = 0xffffffffu, md1 = 0u;
        i64 mp = 0;
        if (kk < a.nseg) { md0 = a.seg_dst[kk]; md1 = kk + 1 < a.nseg ? a.seg_dst[kk + 1] : (u32)a.Ls; mp = a.seg_ptr[kk]; }
        bool done = false;
        for (int j = 0; j < 32; ++j) {
            const u32 d0 = __shfl_sync(SCCG_FULL_MASK, md0, j);
            if (d0 >= s1) { done = true; break; }                 // also the "no such segment" marker
            const u32 d1 = __shfl_sync(SCCG_FULL_MASK, md1, j);
            const i64 src = __shfl_sync(SCCG_FULL_MASK, mp, j);
            const u32 lo = d0 > s0 ? d0 : s0, hi = d1 < s1 ? d1 : s1;
            if (hi <= lo || src < 0) continue;                     // src < 0: SEG_BAD_PTR
            const u8* sp = (src & SEG_LIT_FLAG) ? a.enc + (src & ~SEG_LIT_FLAG) : a.ref + src;
            warp_copy_g2s_bulk(A + (lo - s0), sp + (lo - d0), hi - lo, &bar);
        }
        if (done) break;
    }
    // lowercase runs of this warp, fetched the same way while the copies are in flight
    int lkk = tw.y + warp + lane * NW;
    i64 ml0 = 0x7fffffffffffffffLL, ml1 = 0;
    if (lkk < a.l_k) { ml0 = a.l_start[lkk]; ml1 = ml0 + a.l_len[lkk]; }
    __syncthreads();                                              // every copy has been issued ...
    if (threadIdx.x == 0) mbar_arrive(&bar);
    mbar_wait(&bar, 0u);                                          // ... and has landed
    // ---- 2. lowercase runs (merged coordinates; image offset = b - b0)
    for (int lb = tw.y + warp; lb < a.l_k; lb += 32 * NW) {
        bool done = false;
        for (int j = 0; j < 32; ++j) {
            const i64 ls = __shfl_sync(SCCG_FULL_MASK, ml0, j);
            if (ls >= (i64)b1) { done = true; break; }
            const i64 le = __shfl_sync(SCCG_FULL_MASK, ml1, j);
            const u32 lo = ls > (i64)b0 ? (u32)ls : b0, hi = le < (i64)b1 ? (u32)le : b1;
            if (hi > lo) warp_lower_smem(A + (lo - b0), hi - lo);
        }
        if (done) break;
        lkk += 32 * NW;                                            // (rare) more than 32 runs per warp in one tile
        ml0 = 0x7fffffffffffffffLL; ml1 = 0;
        if (lkk < a.l_k) { ml0 = a.l_start[lkk]; ml1 = ml0 + a.l_len[lkk]; }
    }
    __syncthreads();
    // ---- 3. format: GATHER_ROUNDS x 16 bytes of text per thread, staged in O; a full tile leaves as ONE bulk store
    const bool full_tile = Qe - Q0 == GATHER_TILE && Qe < a.total;                    // (the last tile of the text carries the final newline: direct stores)
    const u32 aph = s0 & 15u;                                                         // phase of the image inside Araw
#pragma unroll
    for (int half = 0; half < GATHER_ROUNDS; ++half) {
        const u32 t16 = (u32)threadIdx.x + (u32)half * GATHER_CTA;
        const i64 q0 = Q0 + (i64)t16 * 16;
        if (q0 >= a.total) break;
        const u32 line0 = (u32)q0 / (u32)(WRAP + 1);
        const int col0 = (int)((u32)q0 - line0 * (u32)(WRAP + 1));
        const int c = WRAP - col0;                                   // offset of the '\n' inside this piece if < 16
        const u32 ao = line0 * WRAP + (u32)col0 - b0 + aph;          // offset of the first symbol of the piece inside Araw
        if (q0 + 16 <= a.total - 1) {
            const u32* A32 = reinterpret_cast<const u32*>(Araw);
            const u32 i = ao >> 2, sh = (ao & 3u) * 8u;
            const u32 x0 = A32[i], x1 = A32[i + 1], x2 = A32[i + 2], x3 = A32[i + 3], x4 = A32[i + 4];
            u64 w0 = (u64)__funnelshift_r(x0, x1, sh) | ((u64)__funnelshift_r(x1, x2, sh) << 32);
            u64 w1 = (u64)__funnelshift_r(x2, x3, sh) | ((u64)__funnelshift_r(x3, x4, sh) << 32);
            if (c < 8) {
                u64 lowmask = c ? (~0ull >> (64 - 8 * c)) : 0ull;
                u64 carry = w0 >> 56;
                w0 = (w0 & lowmask) | ((u64)'\n' << (8 * c)) | ((w0 & ~lowmask) << 8);
                w1 = (w1 << 8) | carry;
            } else if (c < 16) {
                int cc = c - 8;
                u64 lowmask = cc ? (~0ull >> (64 - 8 * cc)) : 0ull;
                w1 = (w1 & lowmask) | ((u64)'\n' << (8 * cc)) | ((w1 & ~lowmask) << 8);
            }
            ulonglong2 v; v.x = w0; v.y = w1;
            if (full_tile) *reinterpret_cast<ulonglong2*>(O + t16 * 16u) = v;
            else *reinterpret_cast<ulonglong2*>(a.out + q0) = v;
        } else {
            // the piece(s) at the very end of the text: the final newline (:274) does not sit on a line border
            u32 sym = ao;
            for (int d = 0; d < 16 && q0 + d < a.total; ++d) {
                const bool nl = (q0 + d == a.total - 1) || (col0 + d) % (WRAP + 1) == WRAP;
                a.out[q0 + d] = nl ? (u8)'\n' : Araw[sym];
                if (!nl) ++sym;
            }
        }
    }
    if (full_tile) {
        fence_smem_to_async();
        __syncthreads();
        if (threadIdx.x == 0) { bulk_s2g(a.out + Q0, O, (u32)GATHER_TILE); bulk_wait_read(); }
    }
}

// reconstruct_genome.  header_reserve bytes are left free in front of the text (multiple of 16) so that the caller
// can place "<header>\n" right before it.  *d_out points at the text itself.
struct ReconPlan {
    GatherArgs a; u32* sc; int* tok_len; u32 ntok; unsigned ntiles; RunTable lows, ns; u32 soft;
    i64 nr; const int* tok_delta; const u32* delta_excl;        // inputs of dec_resolve_k
};

// The front end of reconstruct_genome, shared by the whole-image decoder and region extraction: run lists, tokenizer, sizes,
// the segment tables (plan->a without an output: a.out / a.tile_win stay NULL).  Reads no reference symbols.  On return the
// main lane may still be producing delta_excl (tokens) and the side lane the lowercase-run table (event ev_side[3]).
static int reconstruct_front(sccg_ctx* c, i64 nr, const u8* d_enc, i64 ne, const u8* d_n, i64 nn, const u8* d_low, i64 nl, ReconPlan* plan) {
    u32* sc = nullptr;
    SCCG_TRY(buf(c, B_SCALARS, (size_t)S_COUNT, &sc));
    SCCG_CK(cudaMemsetAsync(sc, 0, sizeof(u32) * S_COUNT, c->stream));
    SCCG_CK(cudaEventRecord(c->ev[0], c->stream));

    RunTable lows, ns;
    SCCG_CK(cudaEventRecord(c->ev_side[2], c->stream));
    SCCG_CK(cudaStreamWaitEvent(c->side_stream, c->ev_side[2], 0));

    // ---- body tokenizer: count per 16-byte chunk, scan, emit the compacted tables
    const i64 nth = (ne + DEC_PER_THREAD - 1) / DEC_PER_THREAD;
    const unsigned dblocks = div_up(nth > 0 ? nth : 1, DEC_T);
    u32 *th_sym = nullptr, *th_seg = nullptr, *th_tok = nullptr;
    const size_t th_stride = ((size_t)nth + 4) & ~(size_t)3;                    // keeps the three arrays 16-byte aligned
    SCCG_TRY(buf(c, B_TOK_FLAG, th_stride * 3 + 4, &th_sym));
    th_seg = th_sym + th_stride; th_tok = th_seg + th_stride;
    if (ne > 0) LAUNCH(c, dec_count_k, dim3(dblocks), dim3(DEC_T), 0, d_enc, ne, th_sym, th_seg, th_tok, sc);
    SCCG_TRY(scan_exclusive_u32x3(c, th_sym, th_stride, nth, sc + D_LS, sc + D_NSEG, sc + D_NTOK));     // three counters, one launch
    // ---- the two run lists are parsed on the side lane while the tokenizer kernels run
    {
        SideLane side(c);
        SCCG_TRY(parse_runs(c, d_low, nl, B_NUM0, sc, D_LOW_ITEMS, sc + D_LSUM, DE_LOW_UNSORTED, &lows));     // slots B_NUM0..B_NUM3
        SCCG_TRY(parse_runs(c, d_n, nn, B_NUM4, sc, D_N_ITEMS, sc + D_NSUM, DE_N_UNSORTED, &ns));          // slots B_NUM4, B_NUM5, B_LRUN_S, B_LRUN_E
        SCCG_CK(cudaEventRecord(c->ev_side[3], c->stream));
    }
    // the run tables are needed by the gather only (and the N total by the sizes, global-mode files): the main lane does not
    // wait for the side lane before it reads the tokenizer totals
    if (ns.K) SCCG_CK(cudaStreamWaitEvent(c->stream, c->ev_side[3], 0));
    u32 h[D_COUNT];
    SCCG_TRY(read_scalars(c, sc, h, D_COUNT));
    if (h[D_ERR] & DE_FORMAT) return set_error(SCCG_E_FORMAT, "malformed record stream (the reference would throw from stoi)");
    const u32 nseg = h[D_NSEG], ntok = h[D_NTOK];
    const i64 Ls = h[D_LS];
    const i64 nsum = ns.K ? (i64)h[D_NSUM] : 0;

    u32* seg_dst = nullptr; i64* seg_src = nullptr; int *tok_delta = nullptr, *tok_len = nullptr, *tok_abs = nullptr; u32* delta_excl = nullptr;
    SCCG_TRY(buf(c, B_TOK_POS, (size_t)nseg + 1, &seg_dst));
    SCCG_TRY(buf(c, B_ITEM_SRC, (size_t)nseg + 1, &seg_src));
    SCCG_TRY(buf(c, B_ITEM_OFF, (size_t)ntok * 3 + 3, &tok_delta));
    tok_len = tok_delta + ntok + 1; tok_abs = tok_len + ntok + 1;
    SCCG_TRY(buf(c, B_TILE2, (size_t)ntok + 1, &delta_excl));
    if (ne > 0) {
        LAUNCH(c, dec_emit_k, dim3(dblocks), dim3(DEC_T), 0, d_enc, ne, (const u32*)th_sym, (const u32*)th_seg, (const u32*)th_tok, seg_dst, seg_src, tok_delta, tok_len);
    }
    SCCG_CK(cudaEventRecord(c->ev_side[4], c->stream));                         // seg_dst complete: the per-tile windows can be searched (side lane)
    if (ntok > 0) {
        SCCG_TRY(scan_exclusive_u32(c, (const u32*)tok_delta, delta_excl, (i64)ntok, nullptr));
    }
    SCCG_CK(cudaEventRecord(c->ev[1], c->stream));

    // ---- sizes: N-merged length, wrapped text length
    const i64 Lm = Ls + nsum;
    if (ns.K) {
        // the last N run must end inside the merged sequence: otherwise the reference's merge loop (:244-252) runs
        // past the end of the decoded string (undefined behaviour there, SCCG_E_FORMAT here)
        int last[2] = {0, 0};
        SCCG_CK(cudaMemcpyAsync(&last[0], ns.start + (ns.K - 1), sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaMemcpyAsync(&last[1], ns.len + (ns.K - 1), sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaStreamSynchronize(c->stream));
        if ((i64)last[0] + (i64)last[1] > Lm) return set_error(SCCG_E_FORMAT, "N run list reaches past the end of the decoded sequence");
    }
    const i64 nchunks = (Lm + WRAP - 1) / WRAP;
    const i64 total = Lm > 0 ? Lm + nchunks : 1;
    if (total >= 0xffffffffLL) return set_error(SCCG_E_ARG, "decoded output would exceed 4 GiB");
    plan->lows = lows; plan->ns = ns; plan->soft = 0;
    GatherArgs& a = plan->a;
    a.ref = nullptr; a.enc = d_enc; a.seg_dst = seg_dst; a.seg_src = seg_src; a.tok_abs = tok_abs; a.nseg = (int)nseg;
    a.n_start = ns.start; a.n_len = ns.len; a.n_cum = ns.cum; a.n_k = (int)ns.K;
    a.l_start = lows.start; a.l_len = lows.len; a.l_k = (int)lows.K;
    a.Ls = Ls; a.Lm = Lm; a.total = total; a.out = nullptr; a.tile0 = 0; a.err = sc + D_ERR; a.tile_win = nullptr;
    plan->sc = sc; plan->tok_len = tok_len; plan->ntok = ntok; plan->ntiles = 0;
    plan->nr = nr; plan->tok_delta = tok_delta; plan->delta_excl = delta_excl;
    // resolved segment sources: the gathers start from two table loads
    i64* seg_ptr = nullptr;
    SCCG_TRY(buf(c, B_SEG_PTR, (size_t)nseg + 1, &seg_ptr));
    a.seg_ptr = seg_ptr;
    return SCCG_OK;
}

// seg_ptr of every segment and the bounds check of every token (main lane)
static int reconstruct_resolve(sccg_ctx* c, const ReconPlan* plan) {
    const GatherArgs& a = plan->a;
    if (a.nseg) LAUNCH(c, dec_resolve_k, dim3(div_up(a.nseg, 256)), dim3(256), 0, a.seg_src, plan->tok_delta, (const int*)plan->tok_len,
                       plan->delta_excl, a.nseg, plan->nr, const_cast<int*>(a.tok_abs), const_cast<i64*>(a.seg_ptr), plan->sc);
    return SCCG_OK;
}

// everything of reconstruct_genome that does not read the reference symbols: front end, output buffer, per-tile windows
static int reconstruct_prepare(sccg_ctx* c, i64 nr, const u8* d_enc, i64 ne, const u8* d_n, i64 nn, const u8* d_low, i64 nl,
                               i64 header_reserve, ReconPlan* plan) {
    SCCG_TRY(reconstruct_front(c, nr, d_enc, ne, d_n, nn, d_low, nl, plan));
    GatherArgs& a = plan->a;
    u8* out = nullptr;
    SCCG_TRY(buf(c, B_OUT, (size_t)(header_reserve + a.total + 32), &out));
    a.out = out + header_reserve;
    plan->ntiles = div_up(a.total, GATHER_TILE);
    // per-tile entry points: the gather itself starts from two table loads
    int4* tile_win = nullptr;
    SCCG_TRY(buf(c, B_TILE_WIN, (size_t)plan->ntiles + 1, &tile_win));
    a.tile_win = tile_win;
    {   // the window searches need the run tables (made on the side lane) and seg_dst: they run there, next to the token scan
        // and dec_resolve_k of the main lane
        SideLane side(c);
        SCCG_CK(cudaStreamWaitEvent(c->stream, c->ev_side[4], 0));
        LAUNCH(c, dec_tile_win_k, dim3(div_up(plan->ntiles, 128)), dim3(128), 0, a, plan->ntiles, tile_win);
        SCCG_CK(cudaEventRecord(c->ev_side[5], c->stream));
    }
    SCCG_TRY(reconstruct_resolve(c, plan));
    SCCG_CK(cudaStreamWaitEvent(c->stream, c->ev_side[5], 0));                  // run tables + windows complete (device-side wait)
    SCCG_CK(cudaEventRecord(c->ev[1], c->stream));                              // everything up to here is "tokenizer" time
    return SCCG_OK;
}

// Run lists the compressor cannot have written but the reference's parser accepts (positions are expanded and SORTED there,
// decompression.cpp:138-164 / :176-207): runs out of order, lowercase runs that overlap.  Rare and off the hot path: the
// (start, length) tables come to the host, are sorted -- lowercase: overlapping runs united (tolower is idempotent); N: an
// overlap or a run past the end makes the reference's merge loop read out of range (:244-252) and stays an error -- and go
// back.  Clears the soft flags.
static int normalize_runs(sccg_ctx* c, ReconPlan* plan) {
    GatherArgs& a = plan->a;
    for (int which = 0; which < 2; ++which) {
        const u32 bit = which == 0 ? DE_LOW_UNSORTED : DE_N_UNSORTED;
        if (!(plan->soft & bit)) continue;
        RunTable& t = which == 0 ? plan->lows : plan->ns;
        const u32 K = t.K;
        std::vector<int> st(K), ln(K);
        SCCG_CK(cudaMemcpyAsync(st.data(), t.start, sizeof(int) * K, cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaMemcpyAsync(ln.data(), t.len, sizeof(int) * K, cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaStreamSynchronize(c->stream));
        std::vector<std::pair<i64, i64>> runs;                      // [start, end)
        for (u32 k = 0; k < K; ++k) if (ln[k] > 0) runs.push_back(std::make_pair((i64)st[k], (i64)st[k] + ln[k]));
        std::sort(runs.begin(), runs.end());
        std::vector<std::pair<i64, i64>> outr;
        for (const auto& r : runs) {
            if (!outr.empty() && r.first < outr.back().second) {
                if (which == 1) return set_error(SCCG_E_FORMAT, "N run list with overlapping runs (the reference reads out of range)");
                if (r.second > outr.back().second) outr.back().second = r.second;
            } else outr.push_back(r);
        }
        if (which == 1 && !outr.empty() && outr.back().second > a.Lm) return set_error(SCCG_E_FORMAT, "N run list reaches past the end of the decoded sequence");
        const u32 K2 = (u32)outr.size();                          // <= K: the tables are large enough
        std::vector<u32> cum(K2 + 1, 0u);
        for (u32 k = 0; k < K2; ++k) { st[k] = (int)outr[k].first; ln[k] = (int)(outr[k].second - outr[k].first); cum[k + 1] = cum[k] + (u32)ln[k]; }
        if (K2) {
            SCCG_CK(cudaMemcpyAsync(t.start, st.data(), sizeof(int) * K2, cudaMemcpyHostToDevice, c->stream));
            SCCG_CK(cudaMemcpyAsync(t.len, ln.data(), sizeof(int) * K2, cudaMemcpyHostToDevice, c->stream));
            SCCG_CK(cudaMemcpyAsync(t.cum, cum.data(), sizeof(u32) * K2, cudaMemcpyHostToDevice, c->stream));
        }
        SCCG_CK(cudaStreamSynchronize(c->stream));                  // (pageable sources)
        t.K = K2;
        if (which == 0) a.l_k = (int)K2; else a.n_k = (int)K2;
    }
    plan->soft = 0;
    SCCG_CK(cudaMemsetAsync(plan->sc + D_ERR, 0, sizeof(u32), c->stream));
    return SCCG_OK;
}
// the same for the whole-image decoder: the per-tile windows are searched again
static int reconstruct_normalize(sccg_ctx* c, ReconPlan* plan) {
    SCCG_TRY(normalize_runs(c, plan));
    const GatherArgs& a = plan->a;
    LAUNCH(c, dec_tile_win_k, dim3(div_up(plan->ntiles, 128)), dim3(128), 0, a, plan->ntiles, const_cast<int4*>(a.tile_win));
    return SCCG_OK;
}

// tiles [tile0, tile0 + ntiles) of the final text
static int reconstruct_gather(sccg_ctx* c, const ReconPlan* plan, const u8* d_ref, unsigned tile0, unsigned ntiles) {
    GatherArgs a = plan->a;
    a.ref = d_ref; a.tile0 = tile0;
    if (ntiles) LAUNCH(c, dec_gather_k, dim3(ntiles), dim3(GATHER_CTA), 0, a);
    return SCCG_OK;
}

static int reconstruct_finish(sccg_ctx* c, const ReconPlan* plan) {
    SCCG_CK(cudaEventRecord(c->ev[2], c->stream));
    u32 h[D_COUNT];
    SCCG_TRY(read_scalars(c, plan->sc, h, D_COUNT));
    if (h[D_ERR] & DE_BOUNDS) return set_error(SCCG_E_BOUNDS, "ERROR: absolute_start + length exceeds reference genome size");
    if (h[D_ERR] & DE_HARD) return set_error(SCCG_E_FORMAT, "malformed record stream or run list");
    const_cast<ReconPlan*>(plan)->soft = h[D_ERR] & DE_SOFT;       // a run list out of order: the caller normalises it and gathers again
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->ev[0], c->ev[2]); c->prof.kernels_ms = ms;
    cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]); c->prof.serialize_ms = ms;
    cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]); c->prof.gather_ms = ms;
    return SCCG_OK;
}

// reconstruct_genome in one go (reference already resident and prepared)
static int reconstruct_device(sccg_ctx* c, const u8* d_ref, i64 nr, const u8* d_enc, i64 ne, const u8* d_n, i64 nn, const u8* d_low, i64 nl,
                              i64 header_reserve, u8** d_out, i64* out_len) {
    ReconPlan plan;
    SCCG_TRY(reconstruct_prepare(c, nr, d_enc, ne, d_n, nn, d_low, nl, header_reserve, &plan));
    SCCG_TRY(reconstruct_gather(c, &plan, d_ref, 0, plan.ntiles));
    SCCG_TRY(reconstruct_finish(c, &plan));
    if (plan.soft) {                                               // a run list out of order (legal for the reference's parser): once more, in order
        SCCG_TRY(reconstruct_normalize(c, &plan));
        SCCG_TRY(reconstruct_gather(c, &plan, d_ref, 0, plan.ntiles));
        SCCG_TRY(reconstruct_finish(c, &plan));
    }
    *d_out = plan.a.out;
    *out_len = plan.a.total;
    return SCCG_OK;
}

// ------------------------------------------------------------------------------------------------
// pipelined decompression: the reference streams in over PCIe in chunks while the text streams out
// ------------------------------------------------------------------------------------------------
// output byte (wrapped text) at which symbol s of the decoded, N-free sequence appears
__device__ __forceinline__ i64 out_byte_of_sym(const GatherArgs& a, i64 s) {
    i64 b = s;
    if (a.n_k) {
        int lo = 0, hi = a.n_k;                                   // last N run that lies before symbol s
        while (lo < hi) { int mid = (lo + hi) >> 1; if ((i64)a.n_start[mid] - (i64)a.n_cum[mid] <= s) lo = mid + 1; else hi = mid; }
        if (lo > 0) b = s + (i64)a.n_cum[lo - 1] + (i64)a.n_len[lo - 1];
    }
    return b + b / WRAP;
}
// need_hi[j] = one past the last reference symbol that the tokens feeding output chunk j copy from
// need_lo[j]: the first one (0xffffffff: chunk j copies nothing from the reference)
__global__ void dec_need_k(GatherArgs a, const int* __restrict__ tok_len, i64 chunk_bytes, u32* __restrict__ need_hi, u32* __restrict__ need_lo) {
    const int k = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    u32 hi = 0, lo = 0xffffffffu;
    i64 c0 = -1, c1 = -2;
    if (*a.err & DE_SOFT) return;                                 // (uniform) tables not usable yet
    if (k < a.nseg) {
        const i64 src = a.seg_src[k];
        const i64 s0 = a.seg_dst[k], s1 = k + 1 < a.nseg ? (i64)a.seg_dst[k + 1] : a.Ls;
        if (!(src & SEG_LIT_FLAG) && s1 > s0 && a.seg_ptr[k] >= 0) {
            lo = (u32)a.tok_abs[src];
            hi = (u32)((i64)a.tok_abs[src] + (i64)tok_len[src]);
            c0 = out_byte_of_sym(a, s0) / chunk_bytes; c1 = out_byte_of_sym(a, s1 - 1) / chunk_bytes;
        }
    }
    // neighbouring segments feed the same output chunk: one atomic per warp instead of one per segment
    const i64 cw = (i64)__reduce_max_sync(SCCG_FULL_MASK, (int)c0);           // chunk of the token segments of this warp (-1: none)
    if (__all_sync(SCCG_FULL_MASK, (c0 == cw && c1 == cw) || c1 < c0)) {
        const u32 m = __reduce_max_sync(SCCG_FULL_MASK, hi);
        const u32 mlo = __reduce_min_sync(SCCG_FULL_MASK, lo);
        if (lane_of() == 0 && cw >= 0 && m) { atomicMax(&need_hi[cw], m); atomicMin(&need_lo[cw], mlo); }
        return;
    }
    for (i64 cj = c0; cj <= c1; ++cj) { atomicMax(&need_hi[cj], hi); atomicMin(&need_lo[cj], lo); }
}

static const int PIPE_MAX_CHUNKS = 64;


// the lines of an intermediate file (decompression.cpp:66-101): optional "<header>", lowercase runs, N runs, body
struct InterLines { const char* header; i64 nh; const char* low; i64 nl; const char* nline; i64 nn; const char* body; i64 nb; bool local_mode; };
static int split_intermediate(const char* inter, i64 inter_len, InterLines* L) {
    i64 cur = 0;
    auto next_line = [&](const char** b, i64* n) -> bool {
        if (cur >= inter_len) return false;
        const char* q = (const char*)memchr(inter + cur, '\n', (size_t)(inter_len - cur));
        *b = inter + cur;
        if (q) { *n = (q - inter) - cur; cur = (q - inter) + 1; } else { *n = inter_len - cur; cur = inter_len; }
        return true;
    };
    const char* first = inter; i64 n0 = 0;
    if (!next_line(&first, &n0)) return set_error(SCCG_E_FORMAT, "Greska pri citanju datoteke (empty intermediate file)");
    L->nh = 0; L->header = inter;
    if (n0 > 0 && first[0] == '>') {
        L->header = first; L->nh = n0;
        if (!next_line(&L->low, &L->nl)) return set_error(SCCG_E_FORMAT, "Greska pri citanju indeksa malih slova");
    } else { L->low = first; L->nl = n0; }
    if (!next_line(&L->nline, &L->nn)) return set_error(SCCG_E_FORMAT, "Greska pri citanju indeksa nepoznatih nukleotida");
    if (!next_line(&L->body, &L->nb)) return set_error(SCCG_E_FORMAT, "Greska pri citanju kodiranog genoma");
    L->local_mode = (L->nn == 1 && L->nline[0] == ',');                          // :105
    return SCCG_OK;
}
// the three text lines -> device (a local-mode file's N line "," stays on the host: nothing is re-inserted)
static int upload_lines(sccg_ctx* c, const InterLines& L, u8** d_enc, u8** d_n, u8** d_low) {
    SCCG_TRY(upload(c, B_ENC, L.body, L.nb, d_enc));
    SCCG_TRY(upload(c, B_NIDX, L.nline, L.local_mode ? 0 : L.nn, d_n));
    SCCG_TRY(upload(c, B_LOW, L.low, L.nl, d_low));
    return SCCG_OK;
}
// the decoder's error word after the front end -> error code (the soft flags are handled by the caller)
static int decoder_flags_error(u32 flags) {
    if (flags & DE_BOUNDS) return set_error(SCCG_E_BOUNDS, "ERROR: absolute_start + length exceeds reference genome size");
    if (flags & DE_HARD) return set_error(SCCG_E_FORMAT, "malformed record stream or run list");
    return SCCG_OK;
}

// decompress_genome's in-memory part (decompression.cpp:66-110) + reconstruct_genome + main's "<header>\n" (:322)
// d_raw_in != NULL: the raw reference symbols are already in device memory (FASTA ingest on the device); ref_raw is unused then
// part / n_parts (n_parts > 1): only the part-th of n_parts contiguous pieces of the file image is produced -- output-range
// sharding over several GPUs (SURVEY 8e (4)): dst receives the piece, *part_off its offset in the image, *out_len its length,
// *total_len the length of the whole image; only the reference chunks that piece copies from are uploaded.
struct PartSpec { int part, n_parts; int64_t* part_off; int64_t* total_len; };
// streaming delivery (sccg_decompress*_stream): the image is handed to fn piece by piece, in order, from a page-locked double
// buffer: while fn works on piece j (writes it to the output file), piece j + 1 is on its way over PCIe
struct SinkSpec { sccg_sink_fn fn; void* user; };
static int decompress_host_impl(sccg_ctx* c, const char* ref_raw, i64 ref_len, const char* inter, i64 inter_len, char* dst, i64 dst_cap, char** out, int64_t* out_len,
                                const u8* d_raw_in, const PartSpec* ps, const SinkSpec* sink);
static int decompress_host(sccg_ctx* c, const char* ref_raw, i64 ref_len, const char* inter, i64 inter_len, char* dst, i64 dst_cap, char** out, int64_t* out_len,
                           const u8* d_raw_in = nullptr, const PartSpec* ps = nullptr, const SinkSpec* sink = nullptr) {
    const int rc = decompress_host_impl(c, ref_raw, ref_len, inter, inter_len, dst, dst_cap, out, out_len, d_raw_in, ps, sink);
    if (rc != SCCG_OK && c->pipe_ready) {
        // an error return must not leave copies from / into the caller's buffers in flight
        cudaStreamSynchronize(c->s_h2d); cudaStreamSynchronize(c->s_d2h); cudaStreamSynchronize(c->main_stream);
    }
    return rc;
}
static int decompress_host_impl(sccg_ctx* c, const char* ref_raw, i64 ref_len, const char* inter, i64 inter_len, char* dst, i64 dst_cap, char** out, int64_t* out_len,
                                const u8* d_raw_in, const PartSpec* ps, const SinkSpec* sink) {
    const bool parts = ps && ps->n_parts > 1;
    if (sink && parts) return set_error(SCCG_E_ARG, "streaming and output-range sharding cannot be combined");
    // ---- the 3 / 4 getline calls (:66-101)
    InterLines L;
    SCCG_TRY(split_intermediate(inter, inter_len, &L));
    const char* header = L.header; const i64 nh = L.nh, nl = L.nl, nn = L.nn, nb = L.nb;
    const bool local_mode = L.local_mode;
    // ---- uploads: the three text lines first (small), then the reference in chunks on its own copy stream
    SCCG_TRY(pipe_streams(c));
    u8 *d_raw = nullptr, *d_ref = nullptr, *d_enc = nullptr, *d_n = nullptr, *d_low = nullptr;
    SCCG_CK(cudaEventRecord(c->ev[4], c->stream));
    SCCG_TRY(upload_lines(c, L, &d_enc, &d_n, &d_low));
    if (d_raw_in) d_raw = const_cast<u8*>(d_raw_in);
    else SCCG_TRY(buf(c, B_TGT, (size_t)ref_len + 128, &d_raw));
    SCCG_TRY(buf(c, B_REF, (size_t)ref_len + 128, &d_ref));
    const i64 rchunk = pipe_chunk_bytes(ref_len);
    const int n_rch = ref_len > 0 ? (int)((ref_len + rchunk - 1) / rchunk) : 0;
    if (getenv("SCCG_PIPE_POISON")) {                                        // tests: a chunk used before it was uploaded / prepared shows up
        SCCG_CK(cudaMemsetAsync(d_ref, 0xEE, (size_t)ref_len, c->stream));
        if (!d_raw_in) SCCG_CK(cudaMemsetAsync(d_raw, 0xEE, (size_t)ref_len, c->stream));
    }
    SCCG_CK(cudaEventRecord(c->ev_pipe[0], c->stream));                      // buffers may have been (re)allocated: order the copy stream after it
    SCCG_CK(cudaStreamWaitEvent(c->s_h2d, c->ev_pipe[0], 0));
    auto enqueue_ref = [&](int i0, int i1) -> int {                          // reference chunks [i0, i1) -> device, one event each
        for (int i = i0; i < i1; ++i) {
            const i64 off = (i64)i * rchunk, len = (ref_len - off) < rchunk ? (ref_len - off) : rchunk;
            if (!d_raw_in) SCCG_CK(cudaMemcpyAsync(d_raw + off, ref_raw + off, (size_t)len, cudaMemcpyHostToDevice, c->s_h2d));
            SCCG_CK(cudaEventRecord(c->ev_h2d[i], c->s_h2d));
        }
        return SCCG_OK;
    };
    const bool defer_upload = parts && local_mode;                            // a piece of a local-mode file needs a piece of the reference only
    if (!defer_upload) {
        SCCG_TRY(enqueue_ref(0, n_rch));
        SCCG_CK(cudaEventRecord(c->ev[5], c->s_h2d));
    }
    u32* sc = nullptr;
    SCCG_TRY(buf(c, B_SCALARS, (size_t)S_COUNT, &sc));
    // ---- reference preparation (:105-110): global mode erases every N (needs the whole reference), local mode only upper-cases
    i64 nr = ref_len;
    int prepared = 0;                                                        // reference chunks already upper-cased (local mode)
    if (!local_mode) {
        SCCG_CK(cudaStreamWaitEvent(c->stream, c->ev[5], 0));
        SCCG_TRY(strip_n<0>(c, d_raw, ref_len, d_ref, B_TILE3, sc + D_STRIP, &nr));
        prepared = n_rch;
    }
    const i64 reserve = ((nh + 1) + 15) & ~(i64)15;
    ReconPlan plan;
    SCCG_TRY(reconstruct_prepare(c, nr, d_enc, nb, d_n, local_mode ? 0 : nn, d_low, nl, reserve, &plan));
    u8* d_text = plan.a.out;
    const i64 n = plan.a.total;
    // "<header>\n" right in front of the text (:322; an absent header still yields the "\n")
    // (a header line of any length: it is copied straight from the caller's file image, where its '\n' follows it -- the image
    // stays valid until the final synchronisation of this call; no header: the lone "\n" comes from the staging area)
    if (nh > 0) {
        SCCG_CK(cudaMemcpyAsync(d_text - (nh + 1), header, (size_t)nh + 1, cudaMemcpyHostToDevice, c->stream));
    } else {
        char* hdr_stage = (char*)c->h_pinned + 4096;                          // scalars live in the first bytes of the staging area
        hdr_stage[0] = '\n';
        SCCG_CK(cudaMemcpyAsync(d_text - 1, hdr_stage, 1, cudaMemcpyHostToDevice, c->stream));
    }
    // ---- result buffer
    const i64 full = n + nh + 1;
    *out_len = full;
    if (parts) *ps->total_len = full;
    char* h_dst = dst;
    if (sink) {
        // pieces are sized by the library: nothing to check
    } else if (parts) {
        if (!dst) return set_error(SCCG_E_ARG, "null argument");
    } else if (dst && dst_cap < full) {
        return set_error(SCCG_E_ARG, "output buffer too small (required size returned in *out_len)");
    }
    // ---- which part of the reference does every output chunk need?
    const unsigned tiles_per_chunk = pipe_tiles_per_chunk(plan.ntiles);
    const int n_och = (int)((plan.ntiles + tiles_per_chunk - 1) / tiles_per_chunk);
    u32 need[PIPE_MAX_CHUNKS], need_lo[PIPE_MAX_CHUNKS];
    for (int j = 0; j < n_och; ++j) { need[j] = 0xffffffffu; need_lo[j] = 0u; }
    {
        // one host round trip: the decoder's error word (every flag is set by now: tokenizer, run lists, bounds check of every
        // token -- nothing is gathered, let alone delivered, from a malformed file) and, for files of several chunks, the
        // reference range every output chunk needs
        const bool need_block = local_mode && plan.a.nseg > 0 && (n_och > 1 || parts);
        u32* d_need = nullptr;                                               // [0, 64): need_hi, [64, 128): need_lo
        SCCG_TRY(buf(c, B_NEED, 2 * PIPE_MAX_CHUNKS, &d_need));
        u32* h_need = (u32*)((char*)c->h_pinned + 8192);
        for (int attempt = 0; attempt < 2; ++attempt) {
            if (need_block) {
                SCCG_CK(cudaMemsetAsync(d_need, 0, sizeof(u32) * PIPE_MAX_CHUNKS, c->stream));
                SCCG_CK(cudaMemsetAsync(d_need + PIPE_MAX_CHUNKS, 0xff, sizeof(u32) * PIPE_MAX_CHUNKS, c->stream));
                LAUNCH(c, dec_need_k, dim3(div_up(plan.a.nseg, 256)), dim3(256), 0, plan.a, (const int*)plan.tok_len, (i64)tiles_per_chunk * GATHER_TILE, d_need,
                       d_need + PIPE_MAX_CHUNKS);
                SCCG_CK(cudaMemcpyAsync(h_need, d_need, sizeof(u32) * 2 * PIPE_MAX_CHUNKS, cudaMemcpyDeviceToHost, c->stream));
            }
            SCCG_CK(cudaMemcpyAsync(h_need + 2 * PIPE_MAX_CHUNKS, sc + D_ERR, sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
            SCCG_CK(cudaStreamSynchronize(c->stream));
            const u32 flags = h_need[2 * PIPE_MAX_CHUNKS];
            SCCG_TRY(decoder_flags_error(flags));
            if (!(flags & DE_SOFT)) break;
            plan.soft = flags & DE_SOFT;                                     // a run list out of order (legal for the reference's parser): sort it, ask again
            SCCG_TRY(reconstruct_normalize(c, &plan));
        }
        if (need_block) {
            memcpy(need, h_need, sizeof(u32) * (size_t)n_och);
            memcpy(need_lo, h_need + PIPE_MAX_CHUNKS, sizeof(u32) * (size_t)n_och);
        }
    }
    // ---- the output chunks of this call: all of them, or the part-th of n_parts contiguous groups
    int j_begin = 0, j_end = n_och;
    i64 img_base = 0;                                                        // offset of h_dst[0] inside the file image
    if (parts) {
        j_begin = (int)((i64)n_och * ps->part / ps->n_parts); j_end = (int)((i64)n_och * (ps->part + 1) / ps->n_parts);
        const i64 pb0 = j_begin == 0 ? 0 : (nh + 1) + (i64)j_begin * tiles_per_chunk * GATHER_TILE;       // offsets in the file image
        i64 pb1 = (nh + 1) + (i64)j_end * tiles_per_chunk * GATHER_TILE; if (pb1 > full || j_end == n_och) pb1 = full;
        if (j_end <= j_begin) pb1 = pb0;
        *ps->part_off = pb0; *out_len = pb1 - pb0;
        if (dst_cap < pb1 - pb0) return set_error(SCCG_E_ARG, "output buffer too small (required size returned in *out_len)");
        img_base = pb0;                                                      // image offset x lands at dst[x - pb0]
        if (defer_upload) {
            u32 lo = 0xffffffffu, hi = 0u;
            for (int j = j_begin; j < j_end; ++j) { if (need_lo[j] < lo) lo = need_lo[j]; if (need[j] != 0xffffffffu && need[j] > hi) hi = need[j]; if (need[j] == 0xffffffffu) { lo = 0; hi = (u32)ref_len; } }
            int i0 = 0, i1 = 0;
            if (hi > lo) { i0 = (int)(lo / rchunk); i1 = (int)(((i64)hi + 32 + rchunk - 1) / rchunk); if (i1 > n_rch) i1 = n_rch; }
            SCCG_TRY(enqueue_ref(i0, i1));
            SCCG_CK(cudaEventRecord(c->ev[5], c->s_h2d));
            prepared = i0;
        }
    }
    if (sink) {
        const size_t need_bytes = (size_t)tiles_per_chunk * GATHER_TILE + (size_t)nh + 64;
        if (c->h_stream_cap < need_bytes) {
            for (int i = 0; i < 2; ++i) { if (c->h_stream[i]) cudaFreeHost(c->h_stream[i]); c->h_stream[i] = nullptr; }
            c->h_stream_cap = 0;
            for (int i = 0; i < 2; ++i) if (cudaMallocHost(&c->h_stream[i], need_bytes) != cudaSuccess) { cudaGetLastError(); return set_error(SCCG_E_NOMEM, "page-locked stream buffers"); }
            c->h_stream_cap = need_bytes;
        }
    } else if (!dst) {                                                       // allocated last: no early return can leak it
        h_dst = (char*)malloc((size_t)full + 1);
        if (!h_dst) return set_error(SCCG_E_NOMEM, "malloc of the result failed");
        h_dst[full] = 0;
    }
    // ---- gather chunk by chunk; every finished chunk goes home on the D2H stream while the next ones are produced
    int rc = SCCG_OK;
    cudaError_t ce = cudaSuccess;
    for (int j = j_begin; j < j_end && rc == SCCG_OK && ce == cudaSuccess; ++j) {
        i64 want = need[j] == 0xffffffffu ? ref_len : (i64)need[j] + 32;     // reference symbols [.., want) must be resident
        if (want > ref_len) want = ref_len;
        while (prepared < n_rch && (i64)prepared * rchunk < want && rc == SCCG_OK) {
            const i64 off = (i64)prepared * rchunk, len = (ref_len - off) < rchunk ? (ref_len - off) : rchunk;
            ce = cudaStreamWaitEvent(c->stream, c->ev_h2d[prepared], 0);
            if (ce != cudaSuccess) break;
            c->prof.launches++;
            SCCG_LAUNCH(upper_k, dim3(div_up(len, 256 * 16)), dim3(256), 0, c->stream, (const u8*)(d_raw + off), len, d_ref + off);
            ++prepared;
        }
        if (ce != cudaSuccess) break;
        const unsigned t0 = (unsigned)j * tiles_per_chunk;
        const unsigned tn = plan.ntiles - t0 < tiles_per_chunk ? plan.ntiles - t0 : tiles_per_chunk;
        rc = reconstruct_gather(c, &plan, d_ref, t0, tn);
        if (rc != SCCG_OK) break;
        if (j == j_begin) cudaEventRecord(c->ev[6], c->stream);
        ce = cudaEventRecord(c->ev_g[j], c->stream);
        if (ce == cudaSuccess) ce = cudaStreamWaitEvent(c->s_d2h, c->ev_g[j], 0);
        // bytes of the device image [-(nh+1), n): chunk 0 also carries the header line
        const i64 b0 = j == 0 ? -(nh + 1) : (i64)t0 * GATHER_TILE;
        i64 b1 = ((i64)t0 + tn) * GATHER_TILE; if (b1 > n) b1 = n;
        if (sink) continue;                                                  // the pieces go home below, two in flight at most
        if (ce == cudaSuccess && b1 > b0) ce = cudaMemcpyAsync(h_dst + ((nh + 1) + b0 - img_base), d_text + b0, (size_t)(b1 - b0), cudaMemcpyDeviceToHost, c->s_d2h);
    }
    if (sink && rc == SCCG_OK && ce == cudaSuccess) {
        auto piece = [&](int j, i64* b0, i64* b1) {                          // bytes [b0, b1) of the device image [-(nh+1), n)
            const unsigned t0 = (unsigned)j * tiles_per_chunk;
            const unsigned tn = plan.ntiles - t0 < tiles_per_chunk ? plan.ntiles - t0 : tiles_per_chunk;
            *b0 = j == 0 ? -(nh + 1) : (i64)t0 * GATHER_TILE;
            *b1 = ((i64)t0 + tn) * GATHER_TILE; if (*b1 > n) *b1 = n;
        };
        auto send_home = [&](int j) -> cudaError_t {
            i64 b0, b1; piece(j, &b0, &b1);
            cudaError_t e2 = cudaStreamWaitEvent(c->s_d2h, c->ev_g[j], 0);
            if (e2 == cudaSuccess && b1 > b0) e2 = cudaMemcpyAsync(c->h_stream[j & 1], d_text + b0, (size_t)(b1 - b0), cudaMemcpyDeviceToHost, c->s_d2h);
            if (e2 == cudaSuccess) e2 = cudaEventRecord(c->ev_d2h[j], c->s_d2h);
            return e2;
        };
        for (int j = 0; j < n_och && j < 2 && ce == cudaSuccess; ++j) ce = send_home(j);
        for (int j = 0; j < n_och && ce == cudaSuccess && rc == SCCG_OK; ++j) {
            ce = cudaEventSynchronize(c->ev_d2h[j]);
            if (ce != cudaSuccess) break;
            i64 b0, b1; piece(j, &b0, &b1);
            if (b1 > b0 && sink->fn(sink->user, (nh + 1) + b0, (const char*)c->h_stream[j & 1], b1 - b0) != 0) rc = set_error(SCCG_E_ARG, "the output sink reported a failure");
            if (j + 2 < n_och && rc == SCCG_OK) ce = send_home(j + 2);        // this buffer is free again
        }
    }
    if (ce == cudaSuccess) ce = cudaEventRecord(c->ev[7], c->s_d2h);
    if (rc == SCCG_OK && ce == cudaSuccess) rc = reconstruct_finish(c, &plan);       // synchronises the compute stream, reads the error flags
    cudaError_t ce2 = cudaStreamSynchronize(c->s_d2h);
    cudaError_t ce3 = cudaStreamSynchronize(c->s_h2d);
    if (rc == SCCG_OK && (ce != cudaSuccess || ce2 != cudaSuccess || ce3 != cudaSuccess))
        rc = set_error(SCCG_E_CUDA, "pipelined decompression failed: %s", cudaGetErrorString(ce != cudaSuccess ? ce : (ce2 != cudaSuccess ? ce2 : ce3)));
    if (rc != SCCG_OK) { if (!dst && !sink) free(h_dst); return rc; }
    if (!dst && !sink) *out = h_dst;
    cudaEventElapsedTime(&c->prof.h2d_ms, c->ev[4], c->ev[5]);
    cudaEventElapsedTime(&c->prof.d2h_ms, c->ev[6], c->ev[7]);
    return SCCG_OK;
}

}  // namespace sccg
