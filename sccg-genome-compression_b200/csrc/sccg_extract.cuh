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
    GatherArgs g;            // tables of the decoded sequence (reconstruct_front); g.out and g.tile_win are not used
    const u32* r_start;      // region i is D[r_start[i], r_start[i] + len_i) ...
    const u32* r_off;        // ... and lands at out[r_off[i], r_off[i + 1]); r_off[n_reg] = total
    int n_reg;
    u32 total;               // output bytes
    u8* out;                 // 16-byte aligned, 16 writable bytes of slack past total
    u32 lane_min;
};

// symbol b of D (merged coordinates): gather_byte without the wrap.  win: search ranges {seg lo, hi, N lo, hi, lower lo, hi}
__device__ __forceinline__ u8 ext_sym(const GatherArgs& a, const int* win, i64 b) {
    int nk = a.n_k ? bounded_upper_i32(a.n_start, win[2], win[3], b) : -1;
    i64 s = b;
    bool is_n = false;
    if (nk >= 0) {
        const i64 st = a.n_start[nk], ln = a.n_len[nk];
        if (b < st + ln) is_n = true;
        else s = b - ((i64)a.n_cum[nk] + ln);
    }
    u8 o = 'N';
    if (!is_n) {
        const int sk = bounded_upper_u32(a.seg_dst, win[0], win[1], s);
        const i64 src = a.seg_ptr[sk];
        const i64 within = s - (i64)a.seg_dst[sk];
        if (src < 0) o = '?';                                         // SEG_BAD_PTR (the call has returned an error before)
        else o = (src & SEG_LIT_FLAG) ? a.enc[(src & ~SEG_LIT_FLAG) + within] : a.ref[src + within];
    }
    const int lk = a.l_k ? bounded_upper_i32(a.l_start, win[4], win[5], b) : -1;
    if (lk >= 0 && b < (i64)a.l_start[lk] + (i64)a.l_len[lk]) o = lower1(o);
    return o;
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

// piece of region r inside the output bytes [Q0, Qe): D[*b0, *b0 + len) lands at out[*q, *q + len)
__device__ __forceinline__ u32 ext_piece(const ExtArgs& e, int r, u32 Q0, u32 Qe, i64* b0, u32* q) {
    const u32 o0 = e.r_off[r], o1 = e.r_off[r + 1];
    const u32 q0 = o0 > Q0 ? o0 : Q0, q1 = o1 < Qe ? o1 : Qe;
    *b0 = (i64)e.r_start[r] + (q0 - o0);
    *q = q0;
    return q1 > q0 ? q1 - q0 : 0u;
}

__global__ void __launch_bounds__(EXT_T) ext_gather_k(ExtArgs e) {
    __shared__ int sh[2];                                            // first and last region that reach into the tile
    __shared__ int win[6];
    __shared__ i64 span[2 * EXT_NW];
    __align__(16) __shared__ u8 O[EXT_TILE];                          // the tile as it goes to memory
    __align__(8) __shared__ u64 bar;
    const GatherArgs& a = e.g;
    if (*a.err & DE_SOFT) return;                                     // a run list is out of order: the caller normalises it and launches again
    const int warp = (int)(threadIdx.x >> 5), lane = lane_of();
    const u32 Q0 = blockIdx.x * (u32)EXT_TILE;
    const u32 Qe = e.total - Q0 < (u32)EXT_TILE ? e.total : Q0 + (u32)EXT_TILE;
    if (threadIdx.x == 0) mbar_init(&bar, 1u);
    if (warp < 2) {
        const int r = warp_upper_u32(e.r_off, e.n_reg, warp ? (i64)Qe - 1 : (i64)Q0);
        if (lane == 0) sh[warp] = r;
    }
    __syncthreads();                                                  // (also: the mbarrier is initialised)
    const int r0 = sh[0], r1 = sh[1];
    const bool lanes = (u32)(r1 - r0 + 1) >= e.lane_min;
    if (lanes) {
        // ---- many short pieces: a thread per piece, one bounded search per symbol and table.  The search ranges cover the
        //      pieces of the whole tile (six 32-ary searches shared among the warps, as in gather_tile_generic)
        i64 lo = 0x7fffffffffffffffLL, hi = -1;
        for (int r = r0 + (int)threadIdx.x; r <= r1; r += EXT_T) {
            i64 b0; u32 q;
            const u32 n = ext_piece(e, r, Q0, Qe, &b0, &q);
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
        for (int r = r0 + (int)threadIdx.x; r <= r1; r += EXT_T) {
            i64 b0; u32 q;
            const u32 n = ext_piece(e, r, Q0, Qe, &b0, &q);
            for (u32 i = 0; i < n; ++i) O[q - Q0 + i] = ext_sym(a, win, b0 + i);
        }
    } else {
        // ---- few pieces: warp w builds pieces r0 + w, r0 + w + EXT_NW, ... with warp copies (bulk copies where the 16-byte
        //      phases of source and tile agree, e.g. one region of a local-mode file that starts on a 16-byte boundary)
        for (int r = r0 + warp; r <= r1; r += EXT_NW) {
            i64 b0; u32 q;
            const u32 n = ext_piece(e, r, Q0, Qe, &b0, &q);
            if (n) ext_piece_warp(a, b0, b0 + n, O + (q - Q0), &bar);
        }
    }
    __syncthreads();                                                  // every copy has been issued ...
    if (threadIdx.x == 0) mbar_arrive(&bar);
    mbar_wait(&bar, 0u);                                              // ... and has landed
    if (!lanes && a.l_k) {
        for (int r = r0 + warp; r <= r1; r += EXT_NW) {
            i64 b0; u32 q;
            const u32 n = ext_piece(e, r, Q0, Qe, &b0, &q);
            if (n) ext_lower_warp(a, b0, b0 + n, O + (q - Q0));
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
    const size_t table_bytes = sizeof(u32) * ((size_t)n_regions * 2 + 1 + iv.size());
    if (c->h_ext_cap < table_bytes) {
        if (c->h_ext) { SCCG_CK(cudaStreamSynchronize(c->stream)); cudaFreeHost(c->h_ext); }
        c->h_ext = nullptr; c->h_ext_cap = 0;
        if (cudaMallocHost(&c->h_ext, table_bytes + table_bytes / 8) != cudaSuccess) { cudaGetLastError(); c->h_ext = nullptr; return set_error(SCCG_E_NOMEM, "page-locked region table"); }
        c->h_ext_cap = table_bytes + table_bytes / 8;
    }
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
    u32* d_reg = nullptr; u32* d_iv = nullptr;
    SCCG_TRY(buf(c, B_EXT_REG, (size_t)n_regions * 2 + 1, &d_reg));
    SCCG_TRY(buf(c, B_EXT_IV, (size_t)n_iv * 2 + 1, &d_iv));
    SCCG_CK(cudaMemcpyAsync(d_reg, h_start, sizeof(u32) * ((size_t)n_regions * 2 + 1), cudaMemcpyHostToDevice, c->stream));
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
    u32* h_flags = (u32*)((char*)c->h_pinned + 8192);                       // [0]: error word, [1]: chunk bits
    const bool need_pass = local_mode && plan.a.nseg > 0 && n_iv > 0 && n_rch > 0;
    if (need_pass) {
        SCCG_CK(cudaMemsetAsync(d_need, 0, sizeof(u32), c->stream));
        LAUNCH(c, ext_need_k, dim3(div_up(plan.a.nseg, 256)), dim3(256), 0, plan.a, (const u32*)d_iv, (const u32*)(d_iv + n_iv), n_iv, rchunk, d_need);
    }
    for (int attempt = 0; attempt < 2; ++attempt) {
        if (need_pass && attempt == 0) SCCG_CK(cudaMemcpyAsync(h_flags + 1, d_need, sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaMemcpyAsync(h_flags, plan.sc + D_ERR, sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaStreamSynchronize(c->stream));
        const u32 flags = h_flags[0];
        SCCG_TRY(decoder_flags_error(flags));
        if (!(flags & DE_SOFT)) break;
        plan.soft = flags & DE_SOFT;                                         // a run list out of order (legal for the reference's parser)
        SCCG_TRY(normalize_runs(c, &plan));
    }
    const u32 need = need_pass ? h_flags[1] : 0u;
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
    ExtArgs e;
    e.g = plan.a; e.g.ref = d_ref;
    e.r_start = d_reg; e.r_off = d_reg + n_regions; e.n_reg = (int)n_regions; e.total = (u32)total; e.out = d_out; e.lane_min = ext_lane_min();
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

}  // namespace sccg
