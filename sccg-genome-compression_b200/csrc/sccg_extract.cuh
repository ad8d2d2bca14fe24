// Region extraction: D[start_0:end_0] + D[start_1:end_1] + ... of the decoded sequence D of an intermediate file (the
// reconstructed_genome.fa image without its header line and newlines), without producing the whole image.
//
//   front end          -> reconstruct_front + dec_resolve_k: the same tokenizer, run lists, segment tables and bounds checks as
//                         the whole-image decoder (so the same errors, whatever regions are asked for)
//   region table       -> host: r_start[i], r_off[i] (output offset of region i, int prefix of the lengths); one upload
//   reference          -> local-mode files: only the chunks that the tokens feeding the regions copy from (ext_need_k, one bit
//                         per chunk) are uploaded / upper-cased; global mode strips N from the whole reference as decompress does
//   ext_gather_k       -> one CTA per 4 KiB of output: region pieces built in a shared-memory image of the tile from the
//                         reference / literal bytes, N runs and lowercase runs applied, the tile leaves with one bulk store
#pragma once
#include "sccg_decode.cuh"

#include <new>

namespace sccg {

static const int EXT_T = 128;                 // threads per output tile
static const int EXT_TILE = GATHER_TILE;      // 4 KiB of output per CTA
static const int EXT_NW = EXT_T / 32;
// Tiles with at least this many region pieces take the lane-per-region path (a thread per piece, per-symbol bounded searches)
// instead of the warp-per-piece path (32-ary searches + warp copies): a warp per 1-bp piece spends its searches on one byte.
// SCCG_EXT_LANE_MIN overrides it (tests force either path).
static const u32 EXT_LANE_MIN = 64;
// granularity of the host's union of the regions (the chunk selection of local-mode files): coarser than a region only adds
// reference symbols to a chunk that is uploaded anyway in all but border cases
static const int EXT_IV_SHIFT = 12;

struct ExtArgs {
    const GatherArgs* g;     // tables of the decoded sequence of each archive (device memory; reconstruct_front); out, tile_win,
                             // seg_src, tok_abs and err of an entry are not used
    const u32* r_start;      // region i is D[r_start[i], r_start[i] + len_i) of archive r_tag[i] >> 1 ...
    const u32* r_off;        // ... and lands at out[r_off[i], r_off[i + 1]); r_off[n_reg] = total
    const u32* r_tag;        // archive << 1 | strand (1: the reverse complement of the region); NULL: archive 0, strand 0 throughout
    int n_reg;
    u32 total;               // output bytes
    u8* out;                 // 16-byte aligned, 16 writable bytes of slack past total
    u32 lane_min;
    const u32* err;          // the decoder's error word of a call that has just run the front end (DE_SOFT: return at once), or NULL
};

// complement of one byte, case kept: A-T, C-G, R-Y, K-M, B-V, D-H; every other byte (S, W, N, non-letters) maps to itself.
// (c | 0x20) is a lowercase letter only for letters, and the xor of two upper-case letters leaves the case bit alone.
__host__ __device__ __forceinline__ u8 comp_byte(u32 c) {
    switch (c | 0x20u) {
        case 'a': case 't': return (u8)(c ^ ('A' ^ 'T'));
        case 'c': case 'g': return (u8)(c ^ ('C' ^ 'G'));
        case 'r': case 'y': return (u8)(c ^ ('R' ^ 'Y'));
        case 'k': case 'm': return (u8)(c ^ ('K' ^ 'M'));
        case 'b': case 'v': return (u8)(c ^ ('B' ^ 'V'));
        case 'd': case 'h': return (u8)(c ^ ('D' ^ 'H'));
        default: return (u8)c;
    }
}

// search ranges of the per-symbol lookups: segments, N runs, lowercase runs
struct ExtWin { int s0, s1, n0, n1, l0, l1; };

// symbol b of D (merged coordinates): gather_byte without the wrap
__device__ __forceinline__ u8 ext_sym(const GatherArgs& a, const ExtWin& w, i64 b) {
    int nk = a.n_k ? bounded_upper_i32(a.n_start, w.n0, w.n1, b) : -1;
    i64 s = b;
    bool is_n = false;
    if (nk >= 0) {
        const i64 st = a.n_start[nk], ln = a.n_len[nk];
        if (b < st + ln) is_n = true;
        else s = b - ((i64)a.n_cum[nk] + ln);
    }
    u8 o = 'N';
    if (!is_n) {
        const int sk = bounded_upper_u32(a.seg_dst, w.s0, w.s1, s);
        const i64 src = a.seg_ptr[sk];
        const i64 within = s - (i64)a.seg_dst[sk];
        if (src < 0) o = '?';                                         // SEG_BAD_PTR (the call has returned an error before)
        else o = (src & SEG_LIT_FLAG) ? a.enc[(src & ~SEG_LIT_FLAG) + within] : a.ref[src + within];
    }
    const int lk = a.l_k ? bounded_upper_i32(a.l_start, w.l0, w.l1, b) : -1;
    if (lk >= 0 && b < (i64)a.l_start[lk] + (i64)a.l_len[lk]) o = lower1(o);
    return o;
}

// piece D[b0, b0 + n) -> dst (shared), a symbol at a time; minus strand: its reverse complement (ct: complement table)
__device__ __forceinline__ void ext_piece_lane(const GatherArgs& a, const ExtWin& w, i64 b0, u32 n, bool minus, const u8* ct, u8* dst) {
    if (minus) for (u32 i = 0; i < n; ++i) dst[i] = ct[ext_sym(a, w, b0 + (n - 1 - i))];
    else for (u32 i = 0; i < n; ++i) dst[i] = ext_sym(a, w, b0 + i);
}

// N-free symbols [s, se) -> dst (shared); whole warp, uniform arguments.  The copy segments are fetched 32 at a time, one per
// lane, and handed out by shuffles (as in dec_gather_k)
__device__ __forceinline__ void ext_copy_warp(const GatherArgs& a, i64 s, i64 se, u8* dst, u64* bar) {
    const int lane = lane_of();
    const int sk = warp_upper_u32(a.seg_dst, a.nseg, s);
    for (int kb = sk; kb < a.nseg; kb += 32) {
        const int kk = kb + lane;
        i64 md0 = 0x7fffffffffffffffLL, md1 = 0, mp = 0;
        if (kk < a.nseg) { md0 = a.seg_dst[kk]; md1 = kk + 1 < a.nseg ? (i64)a.seg_dst[kk + 1] : a.Ls; mp = a.seg_ptr[kk]; }
        bool done = false;
        for (int j = 0; j < 32; ++j) {
            const i64 d0 = __shfl_sync(SCCG_FULL_MASK, md0, j);
            if (d0 >= se) { done = true; break; }
            const i64 d1 = __shfl_sync(SCCG_FULL_MASK, md1, j);
            const i64 src = __shfl_sync(SCCG_FULL_MASK, mp, j);
            const i64 lo = d0 > s ? d0 : s, hi = d1 < se ? d1 : se;
            if (hi <= lo || src < 0) continue;                        // src < 0: SEG_BAD_PTR
            const u8* sp = (src & SEG_LIT_FLAG) ? a.enc + (src & ~SEG_LIT_FLAG) : a.ref + src;
            warp_copy_g2s_bulk(dst + (lo - s), sp + (lo - d0), (u32)(hi - lo), bar);
        }
        if (done) break;
    }
}

// one region piece D[b0, b1) -> dst (shared), without the lowercase runs; whole warp, uniform arguments.  Stretches inside N
// runs become 'N', the others are copied from their N-free coordinates.
__device__ __forceinline__ void ext_piece_warp(const GatherArgs& a, i64 b0, i64 b1, u8* dst, u64* bar) {
    const int lane = lane_of();
    int nk = a.n_k ? warp_upper_i32(a.n_start, a.n_k, b0) : -1;     // last N run that starts at or before b
    i64 b = b0;
    while (b < b1) {
        i64 noff = 0;
        if (nk >= 0) {
            const i64 en = (i64)a.n_start[nk] + a.n_len[nk];
            if (b < en) {                                             // inside N run nk
                const i64 e = en < b1 ? en : b1;
                for (i64 i = b + lane; i < e; i += 32) dst[i - b0] = 'N';
                b = e;
                continue;
            }
            noff = (i64)a.n_cum[nk] + a.n_len[nk];
        }
        const i64 nxt = nk + 1 < a.n_k ? (i64)a.n_start[nk + 1] : b1;
        if (b >= nxt) { ++nk; continue; }
        const i64 e = nxt < b1 ? nxt : b1;
        ext_copy_warp(a, b - noff, e - noff, dst + (b - b0), bar);
        b = e;
    }
}

// the lowercase runs that overlap D[b0, b1) -> dst (shared); whole warp, uniform arguments
__device__ __forceinline__ void ext_lower_warp(const GatherArgs& a, i64 b0, i64 b1, u8* dst) {
    const int lane = lane_of();
    int lk = warp_upper_i32(a.l_start, a.l_k, b0);
    if (lk < 0 || (i64)a.l_start[lk] + a.l_len[lk] <= b0) ++lk;       // first run that reaches into the piece
    for (int kb = lk; kb < a.l_k; kb += 32) {
        const int kk = kb + lane;
        i64 ml0 = 0x7fffffffffffffffLL, ml1 = 0;
        if (kk < a.l_k) { ml0 = a.l_start[kk]; ml1 = ml0 + a.l_len[kk]; }
        bool done = false;
        for (int j = 0; j < 32; ++j) {
            const i64 ls = __shfl_sync(SCCG_FULL_MASK, ml0, j);
            if (ls >= b1) { done = true; break; }
            const i64 le = __shfl_sync(SCCG_FULL_MASK, ml1, j);
            const i64 lo = ls > b0 ? ls : b0, hi = le < b1 ? le : b1;
            if (hi > lo) warp_lower_smem(dst + (lo - b0), (u32)(hi - lo));
        }
        if (done) break;
    }
}

// n bytes of shared memory -> their reverse complement, in place; whole warp, uniform arguments
__device__ __forceinline__ void ext_revcomp_warp(u8* p, u32 n, const u8* ct) {
    for (u32 j = (u32)lane_of(); j < (n + 1) / 2; j += 32) {
        const u8 x = p[j], y = p[n - 1 - j];
        p[j] = ct[y];
        p[n - 1 - j] = ct[x];                                         // (the middle byte of an odd n: the same value twice)
    }
}

// piece of region r inside the output bytes [Q0, Qe): D[*b0, *b0 + len) lands at out[*q, *q + len), reversed and complemented
// when strand (*tag & 1) is 1 -- then the tile's part of the piece comes from the mirrored part of the region
__device__ __forceinline__ u32 ext_piece(const ExtArgs& e, int r, u32 Q0, u32 Qe, i64* b0, u32* q, u32* tag) {
    const u32 o0 = e.r_off[r], o1 = e.r_off[r + 1];
    const u32 q0 = o0 > Q0 ? o0 : Q0, q1 = o1 < Qe ? o1 : Qe;
    *tag = e.r_tag ? e.r_tag[r] : 0u;
    *b0 = (i64)e.r_start[r] + ((*tag & 1u) ? (i64)o1 - (i64)q1 : (i64)q0 - (i64)o0);
    *q = q0;
    return q1 > q0 ? q1 - q0 : 0u;
}

// (8 CTAs per SM: without a floor ptxas settles on 48 registers and spills; 56 registers keep 9 CTAs of 4.6 KiB resident)
__global__ void __launch_bounds__(EXT_T, 8) ext_gather_k(ExtArgs e) {
    __shared__ int sh[2];                                            // first and last region that reach into the tile
    __shared__ int win[6];
    __shared__ i64 span[2 * EXT_NW];
    __align__(16) __shared__ u8 O[EXT_TILE];                          // the tile as it goes to memory
    __align__(8) __shared__ u64 bar;
    __align__(8) __shared__ GatherArgs A;                             // the tables of the tile's archive, when all its pieces share one
    __shared__ u8 CT[256];                                            // complement table, when a piece is on the minus strand
    if (e.err && (*e.err & DE_SOFT)) return;                          // a run list is out of order: the caller normalises it and launches again
    const int warp = (int)(threadIdx.x >> 5), lane = lane_of();
    const u32 Q0 = blockIdx.x * (u32)EXT_TILE;
    const u32 Qe = e.total - Q0 < (u32)EXT_TILE ? e.total : Q0 + (u32)EXT_TILE;
    if (threadIdx.x == 0) mbar_init(&bar, 1u);
    static_assert(sizeof(GatherArgs) % 8 == 0, "GatherArgs is copied in 8-byte words");
    const int nw8 = (int)(sizeof(GatherArgs) / 8);
    if (warp < 2) {
        const int r = warp_upper_u32(e.r_off, e.n_reg, warp ? (i64)Qe - 1 : (i64)Q0);
        if (lane == 0) sh[warp] = r;
    } else if (!e.r_tag) {                                            // one archive: its tables load while warps 0, 1 search
        for (int i = (int)threadIdx.x - 64; i < nw8; i += EXT_T - 64) reinterpret_cast<u64*>(&A)[i] = reinterpret_cast<const u64*>(e.g)[i];
    }
    __syncthreads();                                                  // (also: the mbarrier is initialised)
    const int r0 = sh[0], r1 = sh[1];
    int mixed = 0;
    if (e.r_tag) {                                                    // (block-uniform)
        const u32 arch0 = e.r_tag[r0] >> 1;
        int minus = 0;
        for (int r = r0 + (int)threadIdx.x; r <= r1; r += EXT_T) { const u32 t = e.r_tag[r]; mixed |= (t >> 1) != arch0; minus |= (int)(t & 1u); }
        mixed = __syncthreads_or(mixed);
        minus = __syncthreads_or(minus);
        if (minus) for (int i = (int)threadIdx.x; i < 256; i += EXT_T) CT[i] = comp_byte((u32)i);
        if (!mixed) for (int i = (int)threadIdx.x; i < nw8; i += EXT_T) reinterpret_cast<u64*>(&A)[i] = reinterpret_cast<const u64*>(e.g + arch0)[i];
        __syncthreads();
    }
    const bool lanes = (u32)(r1 - r0 + 1) >= e.lane_min;
    if (lanes) {
        // ---- many short pieces: a thread per piece, one bounded search per symbol and table.  When the pieces of the tile
        //      share one archive, the search ranges cover the pieces of the whole tile (six 32-ary searches shared among the
        //      warps, as in gather_tile_generic); a tile that mixes archives searches each archive's whole tables.
        if (!mixed) {
            const GatherArgs& a = A;
            i64 lo = 0x7fffffffffffffffLL, hi = -1;
            for (int r = r0 + (int)threadIdx.x; r <= r1; r += EXT_T) {
                i64 b0; u32 q, tag;
                const u32 n = ext_piece(e, r, Q0, Qe, &b0, &q, &tag);
                if (n) { lo = b0 < lo ? b0 : lo; hi = b0 + n - 1 > hi ? b0 + n - 1 : hi; }
            }
            for (int d = 16; d; d >>= 1) {
                const i64 l2 = __shfl_xor_sync(SCCG_FULL_MASK, lo, d), h2 = __shfl_xor_sync(SCCG_FULL_MASK, hi, d);
                lo = l2 < lo ? l2 : lo; hi = h2 > hi ? h2 : hi;
            }
            if (lane == 0) { span[warp] = lo; span[EXT_NW + warp] = hi; }
            __syncthreads();
            lo = span[0]; hi = span[EXT_NW];
            for (int w = 1; w < EXT_NW; ++w) { lo = span[w] < lo ? span[w] : lo; hi = span[EXT_NW + w] > hi ? span[EXT_NW + w] : hi; }
            if (hi >= lo) {
                for (int wi = warp; wi < 6; wi += EXT_NW) {
                    const i64 bq = (wi & 1) ? hi : lo;
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
        }
        for (int r = r0 + (int)threadIdx.x; r <= r1; r += EXT_T) {
            i64 b0; u32 q, tag;
            const u32 n = ext_piece(e, r, Q0, Qe, &b0, &q, &tag);
            if (!n) continue;
            if (!mixed) {
                ext_piece_lane(A, ExtWin{win[0], win[1], win[2], win[3], win[4], win[5]}, b0, n, tag & 1u, CT, O + (q - Q0));
            } else {
                const GatherArgs& g = e.g[tag >> 1];
                ext_piece_lane(g, ExtWin{0, g.nseg - 1, 0, g.n_k - 1, 0, g.l_k - 1}, b0, n, tag & 1u, CT, O + (q - Q0));
            }
        }
    } else {
        // ---- few pieces: warp w builds pieces r0 + w, r0 + w + EXT_NW, ... with warp copies (bulk copies where the 16-byte
        //      phases of source and tile agree, e.g. one region of a local-mode file that starts on a 16-byte boundary)
        for (int r = r0 + warp; r <= r1; r += EXT_NW) {
            i64 b0; u32 q, tag;
            const u32 n = ext_piece(e, r, Q0, Qe, &b0, &q, &tag);
            if (!n) continue;
            if (!mixed) ext_piece_warp(A, b0, b0 + n, O + (q - Q0), &bar);
            else ext_piece_warp(e.g[tag >> 1], b0, b0 + n, O + (q - Q0), &bar);
        }
    }
    __syncthreads();                                                  // every copy has been issued ...
    if (threadIdx.x == 0) mbar_arrive(&bar);
    mbar_wait(&bar, 0u);                                              // ... and has landed
    if (!lanes) {
        // lowercase runs over the forward piece; a minus-strand piece is then reversed and complemented within its own span
        for (int r = r0 + warp; r <= r1; r += EXT_NW) {
            i64 b0; u32 q, tag;
            const u32 n = ext_piece(e, r, Q0, Qe, &b0, &q, &tag);
            if (!n) continue;
            const GatherArgs& a = mixed ? e.g[tag >> 1] : A;
            if (a.l_k) ext_lower_warp(a, b0, b0 + n, O + (q - Q0));
            if (tag & 1u) { __syncwarp(); ext_revcomp_warp(O + (q - Q0), n, CT); }
        }
        __syncthreads();
    }
    // ---- the tile leaves: one bulk store when it is whole, 16-byte stores otherwise (the output buffer has slack past total)
    if (Qe - Q0 == (u32)EXT_TILE) {
        fence_smem_to_async();
        __syncthreads();
        if (threadIdx.x == 0) { bulk_s2g(e.out + Q0, O, (u32)EXT_TILE); bulk_wait_read(); }
    } else {
        for (u32 i = threadIdx.x * 16u; i < Qe - Q0; i += EXT_T * 16u)
            *reinterpret_cast<ulonglong2*>(e.out + Q0 + i) = *reinterpret_cast<const ulonglong2*>(O + i);
    }
}

// Local-mode files: bit j of *need <=> reference chunk j holds symbols that a token copies into the regions.  iv_lo / iv_hi:
// the regions united into sorted, disjoint intervals of D (= N-free coordinates: a local-mode file re-inserts no N).  A thread
// per copy segment; one atomic per warp.
__global__ void ext_need_k(GatherArgs a, const u32* __restrict__ iv_lo, const u32* __restrict__ iv_hi, int n_iv, i64 chunk, u32* __restrict__ need) {
    const int k = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    u32 bits = 0;
    if (k < a.nseg) {
        const i64 src = a.seg_src[k], p = a.seg_ptr[k];
        const i64 s0 = a.seg_dst[k], s1 = k + 1 < a.nseg ? (i64)a.seg_dst[k + 1] : a.Ls;
        if (!(src & SEG_LIT_FLAG) && p >= 0 && s1 > s0 && n_iv > 0) {
            const int i1 = upper_idx_u32(iv_lo, n_iv, s1 - 1);           // last interval that starts before s1
            const int i0 = upper_idx_u32(iv_hi, n_iv, s0) + 1;           // first interval that ends after s0
            if (i1 >= 0 && i0 <= i1) {
                const i64 lo = iv_lo[i0] > s0 ? (i64)iv_lo[i0] : s0, hi = iv_hi[i1] < s1 ? (i64)iv_hi[i1] : s1;
                const i64 c0 = (p + (lo - s0)) / chunk;
                i64 c1 = (p + (hi - s0) + 32 - 1) / chunk;                // the warp copies may read up to 32 bytes past a segment
                if (c1 > 31) c1 = 31;
                if (c0 <= c1) bits = (c1 - c0 >= 31 ? 0xffffffffu : ((2u << (c1 - c0)) - 1u)) << c0;
            }
        }
    }
    bits = __reduce_or_sync(SCCG_FULL_MASK, bits);
    if (lane_of() == 0 && bits) atomicOr(need, bits);
}

static u32 ext_lane_min() {
    if (const char* s = getenv("SCCG_EXT_LANE_MIN")) return (u32)strtoul(s, nullptr, 10);
    return EXT_LANE_MIN;
}

// the page-locked staging area of the region / query tables (grow-only)
static int ext_staging(sccg_ctx* c, size_t bytes) {
    if (c->h_ext_cap >= bytes) return SCCG_OK;
    if (c->h_ext) { SCCG_CK(cudaStreamSynchronize(c->stream)); cudaFreeHost(c->h_ext); }
    c->h_ext = nullptr; c->h_ext_cap = 0;
    if (cudaMallocHost(&c->h_ext, bytes + bytes / 8) != cudaSuccess) { cudaGetLastError(); c->h_ext = nullptr; return set_error(SCCG_E_NOMEM, "page-locked region table"); }
    c->h_ext_cap = bytes + bytes / 8;
    return SCCG_OK;
}

// the decoder's error word after the front end (one host round trip; d_extra / h_extra: one more word fetched with it): a run
// list out of order is normalised and the word read again
static int front_settle(sccg_ctx* c, ReconPlan* plan, const u32* d_extra, u32* h_extra) {
    u32* h_flags = (u32*)((char*)c->h_pinned + 8192);
    for (int attempt = 0; attempt < 2; ++attempt) {
        if (d_extra && attempt == 0) SCCG_CK(cudaMemcpyAsync(h_flags + 1, d_extra, sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaMemcpyAsync(h_flags, plan->sc + D_ERR, sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaStreamSynchronize(c->stream));
        if (d_extra && attempt == 0) *h_extra = h_flags[1];
        const u32 flags = h_flags[0];
        SCCG_TRY(decoder_flags_error(flags));
        if (!(flags & DE_SOFT)) break;
        plan->soft = flags & DE_SOFT;                                        // a run list out of order (legal for the reference's parser)
        SCCG_TRY(normalize_runs(c, plan));
    }
    return SCCG_OK;
}

static size_t align_up(size_t n, size_t a) { return (n + a - 1) / a * a; }

// the argument checks of sccg_extract* that need no decoding (include/sccg.h); *out_len = the total on success and when out_cap
// is too small
static int extract_check_regions(const sccg_region* regions, i64 n_regions, const char* out, i64 out_cap, int64_t* out_len, int64_t* seq_len,
                                 i64* total_out = nullptr, i64* max_end_out = nullptr) {
    if (!out_len || !seq_len || n_regions < 0 || (n_regions > 0 && !regions)) return set_error(SCCG_E_ARG, "null argument");
    if (n_regions >= 0x80000000LL) return set_error(SCCG_E_ARG, "at most 2^31 - 1 regions per call");
    i64 total = 0, max_end = 0;
    for (i64 i = 0; i < n_regions; ++i) {
        const i64 s = regions[i].start, t = regions[i].end;
        if (s < 0 || s > t) return set_error(SCCG_E_ARG, "a region must have 0 <= start <= end");
        if (t - s >= 0x80000000LL - total) return set_error(SCCG_E_ARG, "the regions add up to 2^31 bytes or more");
        total += t - s;
        if (t > max_end) max_end = t;
    }
    *out_len = total;
    if (total > 0 && !out) return set_error(SCCG_E_ARG, "null argument");
    if (out_cap < total) return set_error(SCCG_E_ARG, "output buffer too small (required size returned in *out_len)");
    if (total_out) *total_out = total;
    if (max_end_out) *max_end_out = max_end;
    return SCCG_OK;
}

// sccg_extract*: ref_raw (host, ref_len symbols) or d_raw_in (raw symbols already in device memory: FASTA ingest, resident
// reference).  Argument errors first, before any device work (include/sccg.h).
static int extract_host_impl(sccg_ctx* c, const char* ref_raw, i64 ref_len, const u8* d_raw_in, const char* inter, i64 inter_len,
                             const sccg_region* regions, i64 n_regions, char* out, i64 out_cap, int64_t* out_len, int64_t* seq_len) {
    i64 total = 0, max_end = 0;
    SCCG_TRY(extract_check_regions(regions, n_regions, out, out_cap, out_len, seq_len, &total, &max_end));
    // ---- the lines of the file, uploads
    InterLines L;
    SCCG_TRY(split_intermediate(inter, inter_len, &L));
    const bool local_mode = L.local_mode;
    u8 *d_raw = nullptr, *d_ref = nullptr, *d_enc = nullptr, *d_n = nullptr, *d_low = nullptr;
    // region table (and, local mode, the union of the regions at 4 KiB granularity) through the page-locked staging area
    std::vector<u32> iv;                                                     // lo0, hi0, lo1, hi1, ...
    if (local_mode && total > 0) {
        const i64 lim = max_end < 0x7fffffffLL ? max_end : 0x7fffffffLL;     // (a larger end fails below, before any gather)
        const i64 nblk = (lim >> EXT_IV_SHIFT) + 2;
        std::vector<int> diff((size_t)nblk, 0);
        for (i64 i = 0; i < n_regions; ++i) {
            const i64 s = regions[i].start, t = regions[i].end < lim ? regions[i].end : lim;
            if (t > s) { ++diff[(size_t)(s >> EXT_IV_SHIFT)]; --diff[(size_t)(((t - 1) >> EXT_IV_SHIFT) + 1)]; }
        }
        int run = 0;
        for (i64 b = 0; b < nblk; ++b) {
            const bool was = run > 0;
            run += diff[(size_t)b];
            if (run > 0 && !was) iv.push_back((u32)(b << EXT_IV_SHIFT));
            if (run == 0 && was) { const i64 h = b << EXT_IV_SHIFT; iv.push_back((u32)(h < lim ? h : lim)); }
        }
    }
    const int n_iv = (int)(iv.size() / 2);
    // [region table | interval table | GatherArgs of the one archive, copied once the front end has made it]
    const size_t reg_bytes = sizeof(u32) * ((size_t)n_regions * 2 + 1);
    const size_t g_off = align_up(sizeof(u32) * ((size_t)n_regions * 2 + 1 + iv.size()), 16);
    SCCG_TRY(ext_staging(c, g_off + sizeof(GatherArgs)));
    u32* h_start = (u32*)c->h_ext;
    u32* h_off = h_start + n_regions;
    {
        u32 off = 0;
        for (i64 i = 0; i < n_regions; ++i) {
            const i64 s = regions[i].start;
            h_start[i] = (u32)(s < 0x7fffffffLL ? s : 0x7fffffffLL);        // (start <= end <= Lm < 2^31 once the call gets to the gather)
            h_off[i] = off;
            off += (u32)(regions[i].end - s);
        }
        h_off[n_regions] = off;
    }
    u32* h_iv = h_off + n_regions + 1;
    for (size_t i = 0; i < iv.size(); i += 2) { h_iv[i / 2] = iv[i]; h_iv[n_iv + i / 2] = iv[i + 1]; }
    SCCG_CK(cudaEventRecord(c->ev[4], c->stream));                         // (h2d_ms: copies only, not the host work above)
    SCCG_TRY(upload_lines(c, L, &d_enc, &d_n, &d_low));
    u8* d_tab = nullptr; u32* d_iv = nullptr;
    SCCG_TRY(buf(c, B_EXT_REG, align_up(reg_bytes, 16) + sizeof(GatherArgs), &d_tab));
    u32* d_reg = (u32*)d_tab;
    GatherArgs* d_g = (GatherArgs*)(d_tab + align_up(reg_bytes, 16));
    SCCG_TRY(buf(c, B_EXT_IV, (size_t)n_iv * 2 + 1, &d_iv));
    SCCG_CK(cudaMemcpyAsync(d_reg, h_start, reg_bytes, cudaMemcpyHostToDevice, c->stream));
    if (n_iv) SCCG_CK(cudaMemcpyAsync(d_iv, h_iv, sizeof(u32) * 2 * (size_t)n_iv, cudaMemcpyHostToDevice, c->stream));
    // ---- reference buffers; global mode: the whole reference, N stripped (decompression.cpp:105-110)
    if (d_raw_in) d_raw = const_cast<u8*>(d_raw_in);
    else SCCG_TRY(buf(c, B_TGT, (size_t)ref_len + 128, &d_raw));
    SCCG_TRY(buf(c, B_REF, (size_t)ref_len + 128, &d_ref));
    if (getenv("SCCG_PIPE_POISON")) {                                        // tests: a chunk used before it was uploaded / prepared shows up
        SCCG_CK(cudaMemsetAsync(d_ref, 0xEE, (size_t)ref_len, c->stream));
        if (!d_raw_in) SCCG_CK(cudaMemsetAsync(d_raw, 0xEE, (size_t)ref_len, c->stream));
    }
    u32* sc = nullptr;
    SCCG_TRY(buf(c, B_SCALARS, (size_t)S_COUNT, &sc));
    i64 nr = ref_len;
    if (!local_mode) {
        if (!d_raw_in && ref_len > 0) SCCG_CK(cudaMemcpyAsync(d_raw, ref_raw, (size_t)ref_len, cudaMemcpyHostToDevice, c->stream));
        SCCG_CK(cudaEventRecord(c->ev[5], c->stream));
        SCCG_TRY(strip_n<0>(c, d_raw, ref_len, d_ref, B_TILE3, sc + D_STRIP, &nr));
    } else {
        SCCG_CK(cudaEventRecord(c->ev[5], c->stream));
    }
    // ---- front end: the decoder's tables and every error check of sccg_decompress
    ReconPlan plan;
    SCCG_TRY(reconstruct_front(c, nr, d_enc, L.nb, d_n, local_mode ? 0 : L.nn, d_low, L.nl, &plan));
    SCCG_TRY(reconstruct_resolve(c, &plan));
    SCCG_CK(cudaStreamWaitEvent(c->stream, c->ev_side[3], 0));              // run tables complete (side lane)
    SCCG_CK(cudaEventRecord(c->ev[1], c->stream));
    // ---- one host round trip: the error word and the reference chunks the regions need
    const i64 rchunk = pipe_chunk_bytes(ref_len);
    const int n_rch = ref_len > 0 ? (int)((ref_len + rchunk - 1) / rchunk) : 0;
    u32* d_need = nullptr;
    SCCG_TRY(buf(c, B_NEED, 2, &d_need));
    const bool need_pass = local_mode && plan.a.nseg > 0 && n_iv > 0 && n_rch > 0;
    if (need_pass) {
        SCCG_CK(cudaMemsetAsync(d_need, 0, sizeof(u32), c->stream));
        LAUNCH(c, ext_need_k, dim3(div_up(plan.a.nseg, 256)), dim3(256), 0, plan.a, (const u32*)d_iv, (const u32*)(d_iv + n_iv), n_iv, rchunk, d_need);
    }
    u32 need = 0;                                                            // the reference chunks the regions need
    SCCG_TRY(front_settle(c, &plan, need_pass ? d_need : nullptr, &need));
    const i64 Lm = plan.a.Lm;
    *seq_len = Lm;
    if (max_end > Lm) return set_error(SCCG_E_ARG, "a region ends past the end of the decoded sequence (its length returned in *seq_len)");
    // ---- local mode: upload (host reference) and upper-case only the chunks the regions copy from
    const bool ref_chunks = local_mode && need;
    if (ref_chunks) {
        SCCG_CK(cudaEventRecord(c->ev_x[0], c->stream));
        for (int j = 0; j < n_rch && j < 32; ++j) {
            if (!((need >> j) & 1u) || d_raw_in) continue;
            const i64 off = (i64)j * rchunk, len = (ref_len - off) < rchunk ? (ref_len - off) : rchunk;
            SCCG_CK(cudaMemcpyAsync(d_raw + off, ref_raw + off, (size_t)len, cudaMemcpyHostToDevice, c->stream));
        }
        SCCG_CK(cudaEventRecord(c->ev_x[1], c->stream));
        for (int j = 0; j < n_rch && j < 32; ++j) {
            if (!((need >> j) & 1u)) continue;
            const i64 off = (i64)j * rchunk, len = (ref_len - off) < rchunk ? (ref_len - off) : rchunk;
            LAUNCH(c, upper_k, dim3(div_up(len, 256 * 16)), dim3(256), 0, (const u8*)(d_raw + off), len, d_ref + off);
        }
    }
    // ---- the gather (again after a normalisation: the first launch returned at once) and the result
    u8* d_out = nullptr;
    SCCG_TRY(buf(c, B_OUT, (size_t)total + 32, &d_out));
    GatherArgs* h_g = (GatherArgs*)((char*)c->h_ext + g_off);
    *h_g = plan.a; h_g->ref = d_ref;
    SCCG_CK(cudaMemcpyAsync(d_g, h_g, sizeof(GatherArgs), cudaMemcpyHostToDevice, c->stream));
    ExtArgs e;
    e.g = d_g; e.r_start = d_reg; e.r_off = d_reg + n_regions; e.r_tag = nullptr; e.n_reg = (int)n_regions; e.total = (u32)total; e.out = d_out;
    e.lane_min = ext_lane_min(); e.err = plan.sc + D_ERR;
    SCCG_CK(cudaEventRecord(c->ev[3], c->stream));
    const unsigned ntiles = div_up(total, EXT_TILE);
    if (ntiles) LAUNCH(c, ext_gather_k, dim3(ntiles), dim3(EXT_T), 0, e);
    SCCG_CK(cudaEventRecord(c->ev[2], c->stream));
    SCCG_CK(cudaEventRecord(c->ev[6], c->stream));
    if (total > 0) SCCG_CK(cudaMemcpyAsync(out, d_out, (size_t)total, cudaMemcpyDeviceToHost, c->stream));
    SCCG_CK(cudaEventRecord(c->ev[7], c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    float ms = 0.f, ref_ms = 0.f;
    if (ref_chunks) cudaEventElapsedTime(&ref_ms, c->ev_x[0], c->ev_x[1]);
    cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]); c->prof.h2d_ms = ms + ref_ms;
    cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]); c->prof.serialize_ms = ms;
    cudaEventElapsedTime(&ms, c->ev[3], c->ev[2]); c->prof.gather_ms = ms;
    cudaEventElapsedTime(&ms, c->ev[0], c->ev[2]); c->prof.kernels_ms = ms;
    cudaEventElapsedTime(&ms, c->ev[6], c->ev[7]); c->prof.d2h_ms = ms;
    return SCCG_OK;
}

static int extract_host(sccg_ctx* c, const char* ref_raw, i64 ref_len, const u8* d_raw_in, const char* inter, i64 inter_len,
                        const sccg_region* regions, i64 n_regions, char* out, i64 out_cap, int64_t* out_len, int64_t* seq_len) {
    const int rc = extract_host_impl(c, ref_raw, ref_len, d_raw_in, inter, inter_len, regions, n_regions, out, out_cap, out_len, seq_len);
    if (rc != SCCG_OK) cudaStreamSynchronize(c->main_stream);             // no copy from the caller's buffers stays in flight
    return rc;
}

// ------------------------------------------------------------------------------------------------
// archives: the front end of one record file run once, its tables kept in device memory of their own
// ------------------------------------------------------------------------------------------------
}  // namespace sccg

struct sccg_archive {
    sccg_ctx* ctx;
    sccg_archive *prev, *next;     // the context's list of open archives
    unsigned gen;                  // resident reference generation the archive was opened against
    int mode;                      // 0: local-mode file, 1: global mode
    sccg::GatherArgs g;            // the tables (in mem) and the reference form they read; seg_src, tok_abs, err, out unused
    void* mem;                     // one exactly-sized allocation: record bytes, seg_dst, seg_ptr, N runs, lowercase runs
    long long device_bytes;        // mem, plus lift once built
    void* lift;                    // the lift table (sccg_liftover.cuh), one exactly-sized allocation built by the first liftover call
    long long lift_n;              // its records
};

namespace sccg {

// the resident reference in the form files of this mode read it (decompress_host_impl: local mode upper-cases, global mode erases
// every N first), built once per resident reference
static int reference_form(sccg_ctx* c, int form) {
    if (c->res_form[form]) return SCCG_OK;
    const i64 n = c->res_ref_len;
    u8* p = nullptr;
    if (cudaMalloc(&p, (size_t)n + 128) != cudaSuccess) { cudaGetLastError(); return set_error(SCCG_E_NOMEM, "cudaMalloc of the prepared reference failed"); }
    i64 len = n;
    int rc = cudaMemsetAsync(p, 0, (size_t)n + 128, c->stream) == cudaSuccess ? SCCG_OK : set_error(SCCG_E_CUDA, "cudaMemsetAsync failed");
    if (rc == SCCG_OK && form == 0 && n > 0) LAUNCH(c, upper_k, dim3(div_up(n, 256 * 16)), dim3(256), 0, (const u8*)c->res_ref, n, p);
    if (rc == SCCG_OK && form == 1) {
        u32* sc = nullptr;
        rc = buf(c, B_SCALARS, (size_t)S_COUNT, &sc);
        if (rc == SCCG_OK) rc = strip_n<0>(c, c->res_ref, n, p, B_TILE3, sc + D_STRIP, &len);
    }
    if (rc != SCCG_OK) { cudaStreamSynchronize(c->stream); cudaFree(p); return rc; }
    c->res_form[form] = p; c->res_form_len[form] = len;
    return SCCG_OK;
}

// the resident reference changes: the prepared forms go, and archives opened against it are stale from now on
static void reference_changed(sccg_ctx* c) {
    ++c->res_gen;
    for (int f = 0; f < 2; ++f) {
        if (c->res_form[f]) { cudaStreamSynchronize(c->main_stream); cudaFree(c->res_form[f]); }
        c->res_form[f] = nullptr; c->res_form_len[f] = 0;
    }
    if (c->res_nrun) { cudaStreamSynchronize(c->main_stream); cudaFree(c->res_nrun); }
    c->res_nrun = nullptr; c->res_nrun_k = 0;
}

static void archive_free(sccg_archive* a) {
    if (a->mem) cudaFree(a->mem);
    if (a->lift) cudaFree(a->lift);
    delete a;
}

static int archive_build(sccg_ctx* c, const char* inter, i64 inter_len, sccg_archive* a) {
    InterLines L;
    SCCG_TRY(split_intermediate(inter, inter_len, &L));
    const int form = L.local_mode ? 0 : 1;
    SCCG_TRY(reference_form(c, form));
    u8 *d_enc = nullptr, *d_n = nullptr, *d_low = nullptr;
    SCCG_CK(cudaEventRecord(c->ev[4], c->stream));
    SCCG_TRY(upload_lines(c, L, &d_enc, &d_n, &d_low));
    // ---- front end: the decoder's tables and every error check of sccg_decompress_resident_into; run lists normalised here
    ReconPlan plan;
    SCCG_TRY(reconstruct_front(c, c->res_form_len[form], d_enc, L.nb, d_n, L.local_mode ? 0 : L.nn, d_low, L.nl, &plan));
    SCCG_TRY(reconstruct_resolve(c, &plan));
    SCCG_CK(cudaStreamWaitEvent(c->stream, c->ev_side[3], 0));              // run tables complete (side lane)
    SCCG_CK(cudaEventRecord(c->ev[1], c->stream));
    SCCG_TRY(front_settle(c, &plan, nullptr, nullptr));
    // ---- the tables a gather reads move into the archive's own memory (the slots they were built in belong to the next call)
    const GatherArgs& p = plan.a;
    const size_t nseg = (size_t)p.nseg, nk = (size_t)p.n_k, lk = (size_t)p.l_k;
    const size_t sz[8] = {(size_t)L.nb + 128, 4 * (nseg + 1), 8 * (nseg + 1), 4 * (nk + 1), 4 * (nk + 1), 4 * (nk + 1), 4 * (lk + 1), 4 * (lk + 1)};
    size_t off[8], total = 0;
    for (int i = 0; i < 8; ++i) { off[i] = total; total += align_up(sz[i], 16); }
    if (cudaMalloc(&a->mem, total) != cudaSuccess) { cudaGetLastError(); a->mem = nullptr; return set_error(SCCG_E_NOMEM, "cudaMalloc of the archive tables failed"); }
    a->device_bytes = (long long)total;
    u8* m = (u8*)a->mem;
    const void* src[8] = {p.enc, p.seg_dst, p.seg_ptr, p.n_start, p.n_len, p.n_cum, p.l_start, p.l_len};
    const size_t cnt[8] = {(size_t)L.nb, 4 * nseg, 8 * nseg, 4 * nk, 4 * nk, 4 * nk, 4 * lk, 4 * lk};
    SCCG_CK(cudaMemsetAsync(m, 0, total, c->stream));                      // (the slack past the record bytes included)
    for (int i = 0; i < 8; ++i) if (cnt[i]) SCCG_CK(cudaMemcpyAsync(m + off[i], src[i], cnt[i], cudaMemcpyDeviceToDevice, c->stream));
    SCCG_CK(cudaEventRecord(c->ev[2], c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    GatherArgs& g = a->g;
    g = p;
    g.ref = c->res_form[form]; g.enc = m + off[0];
    g.seg_dst = (const u32*)(m + off[1]); g.seg_ptr = (const i64*)(m + off[2]);
    g.n_start = (const int*)(m + off[3]); g.n_len = (const int*)(m + off[4]); g.n_cum = (const u32*)(m + off[5]);
    g.l_start = (const int*)(m + off[6]); g.l_len = (const int*)(m + off[7]);
    g.seg_src = nullptr; g.tok_abs = nullptr; g.tile_win = nullptr; g.out = nullptr; g.err = nullptr;
    a->mode = form;
    a->gen = c->res_gen;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]); c->prof.serialize_ms = ms;
    cudaEventElapsedTime(&ms, c->ev[0], c->ev[2]); c->prof.kernels_ms = ms;
    cudaEventElapsedTime(&ms, c->ev[4], c->ev[0]); c->prof.h2d_ms = ms;
    return SCCG_OK;
}

static int archive_open(sccg_ctx* c, const char* inter, i64 inter_len, sccg_archive** out) {
    sccg_archive* a = new (std::nothrow) sccg_archive();
    if (!a) return set_error(SCCG_E_NOMEM, "out of host memory");
    memset(a, 0, sizeof *a);
    a->ctx = c;
    const int rc = archive_build(c, inter, inter_len, a);
    if (rc != SCCG_OK) { cudaStreamSynchronize(c->main_stream); archive_free(a); return rc; }
    a->next = c->archives;
    if (c->archives) c->archives->prev = a;
    c->archives = a;
    *out = a;
    return SCCG_OK;
}

static void archive_unlink(sccg_ctx* c, sccg_archive* a) {
    if (a->prev) a->prev->next = a->next; else c->archives = a->next;
    if (a->next) a->next->prev = a->prev;
}

// the checks of one query (sccg_archive_extract) or window (sccg_archive_search) in the order of include/sccg.h: the index of
// the first that fails, ARCHIVE_QUERY_OK when none does
static const char* const archive_query_why[] = {"a query names an archive index out of range", "null argument",
                                                "a query names an archive opened on another context",
                                                "a query names an archive opened against a resident reference that has since been replaced or cleared",
                                                "a query must have 0 <= start <= end", "a query ends past the end of its archive's decoded sequence",
                                                "a query's strand must be 0 or 1"};
static const int ARCHIVE_QUERY_OK = 6;
static int archive_query_fault(const sccg_ctx* c, sccg_archive* const* archives, i64 n_archives, i64 archive, i64 start, i64 end) {
    const sccg_archive* a = archive >= 0 && archive < n_archives ? archives[archive] : nullptr;
    return (archive < 0 || archive >= n_archives) ? 0 : !a ? 1 : a->ctx != c ? 2 : a->gen != c->res_gen ? 3
         : (start < 0 || start > end) ? 4 : end > a->g.Lm ? 5 : ARCHIVE_QUERY_OK;
}

// sccg_archive_extract: argument checks (include/sccg.h, in that order), then one copy of the query table, one gather, one copy back
static int archive_extract_impl(sccg_ctx* c, sccg_archive* const* archives, i64 n_archives, const sccg_query* queries, i64 n_queries,
                                char* out, i64 out_cap, int64_t* out_len) {
    if (!out_len || n_archives < 0 || n_queries < 0 || (n_archives > 0 && !archives) || (n_queries > 0 && !queries))
        return set_error(SCCG_E_ARG, "null argument");
    if (n_archives >= 0x80000000LL || n_queries >= 0x80000000LL) return set_error(SCCG_E_ARG, "at most 2^31 - 1 archives and queries per call");
    // one pass; the error reported is the first of the list in include/sccg.h that any query commits
    int first = 7;
    i64 total = 0;
    for (i64 i = 0; i < n_queries && first > 0; ++i) {
        const sccg_query& q = queries[i];
        const int f = archive_query_fault(c, archives, n_archives, q.archive, q.start, q.end);
        const int bad = f < ARCHIVE_QUERY_OK ? f : (q.strand != 0 && q.strand != 1) ? 6 : 7;
        if (bad < first) first = bad;
        if (bad == 7) total += q.end - q.start;                              // (< 2^31 each, < 2^31 queries: no overflow)
    }
    if (first < 7) return set_error(SCCG_E_ARG, archive_query_why[first]);
    if (total >= 0x80000000LL) return set_error(SCCG_E_ARG, "the queries add up to 2^31 bytes or more");
    *out_len = total;
    if (total > 0 && !out) return set_error(SCCG_E_ARG, "null argument");
    if (out_cap < total) return set_error(SCCG_E_ARG, "output buffer too small (required size returned in *out_len)");
    if (total == 0) return SCCG_OK;
    // ---- [GatherArgs of every archive | r_start | r_off | r_tag] through the page-locked staging area, one copy
    const size_t ga_bytes = sizeof(GatherArgs) * (size_t)n_archives;
    const size_t bytes = ga_bytes + sizeof(u32) * (3 * (size_t)n_queries + 1);
    SCCG_TRY(ext_staging(c, bytes));
    GatherArgs* h_g = (GatherArgs*)c->h_ext;
    for (i64 k = 0; k < n_archives; ++k) {
        const sccg_archive* a = archives[k];
        if (a && a->ctx == c && a->gen == c->res_gen) h_g[k] = a->g;
        else memset(&h_g[k], 0, sizeof(GatherArgs));                      // (named by no query)
    }
    u32* h_start = (u32*)((char*)c->h_ext + ga_bytes);
    u32* h_off = h_start + n_queries;
    u32* h_tag = h_off + n_queries + 1;
    u32 off = 0;
    for (i64 i = 0; i < n_queries; ++i) {
        const sccg_query& q = queries[i];
        h_start[i] = (u32)q.start; h_off[i] = off; h_tag[i] = ((u32)q.archive << 1) | (u32)q.strand;
        off += (u32)(q.end - q.start);
    }
    h_off[n_queries] = off;
    u8* d_tab = nullptr; u8* d_out = nullptr;
    SCCG_TRY(buf(c, B_EXT_REG, bytes, &d_tab));
    SCCG_TRY(buf(c, B_OUT, (size_t)total + 32, &d_out));
    SCCG_CK(cudaEventRecord(c->ev[4], c->stream));
    SCCG_CK(cudaMemcpyAsync(d_tab, c->h_ext, bytes, cudaMemcpyHostToDevice, c->stream));
    SCCG_CK(cudaEventRecord(c->ev[5], c->stream));
    ExtArgs e;
    e.g = (const GatherArgs*)d_tab;
    e.r_start = (const u32*)(d_tab + ga_bytes); e.r_off = e.r_start + n_queries; e.r_tag = e.r_off + n_queries + 1;
    e.n_reg = (int)n_queries; e.total = (u32)total; e.out = d_out; e.lane_min = ext_lane_min(); e.err = nullptr;
    SCCG_CK(cudaEventRecord(c->ev[3], c->stream));
    LAUNCH(c, ext_gather_k, dim3(div_up(total, EXT_TILE)), dim3(EXT_T), 0, e);
    SCCG_CK(cudaEventRecord(c->ev[2], c->stream));
    SCCG_CK(cudaMemcpyAsync(out, d_out, (size_t)total, cudaMemcpyDeviceToHost, c->stream));
    SCCG_CK(cudaEventRecord(c->ev[7], c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]); c->prof.h2d_ms = ms;
    cudaEventElapsedTime(&ms, c->ev[3], c->ev[2]); c->prof.gather_ms = ms; c->prof.kernels_ms = ms;
    cudaEventElapsedTime(&ms, c->ev[2], c->ev[7]); c->prof.d2h_ms = ms;
    return SCCG_OK;
}

}  // namespace sccg
