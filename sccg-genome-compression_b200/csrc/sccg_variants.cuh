// Variant records of open archives (sccg_archive_variants, include/sccg.h): the stretches between the copies of a record file,
// compared with the reference bytes they replace.  All archives named by the windows go through one pipeline; their elements
// (copy segments, plus one end sentinel per archive) are concatenated in archive order, so every per-archive scan is one scan:
//   vr_key_k / max scan     -> M = the largest reference end of the earlier copies (a key (archive + 1) << 32 | end keeps the
//                              archives apart in one unsegmented prefix maximum)
//   vr_anchor_k (count)     -> the anchor of each copy (clipped by M), split at N runs in global mode: the number of pieces
//   sum scan, vr_anchor_k   -> the anchors in raw coordinates, the sentinel (len(D), len(R)) closing each archive
//   vr_gap_k / sum scan     -> gap j runs from anchor j - 1 (or (0, 0)) to anchor j; its width max(|G_R|, |G_D|) places it in
//                              the gap-byte space, which is tiled at 4 KiB per CTA: a long gap spreads over many CTAs
//   vr_trim_k               -> gaps of unequal length: first difference from each end (per-gap atomicMin)
//   vr_count_k / sum scan   -> records per tile; one host read of the total sizes the record table
//   vr_emit_k, vr_align_k   -> the records of step 3, then each insertion / deletion left-aligned (thread per record)
//   vr_win_k, two sum scans -> per window: its records (two binary searches) and their ALT bytes; one host read of the totals
//   vr_out_k, vr_alt_k      -> the records of every window, then their ALT bytes (one thread per byte, read through ext_sym)
// D bytes are read with ext_sym (sccg_extract.cuh): literal bytes from the record bytes, copies from the reference form, N runs
// applied.  DESIGN.md §4 note 15 explains why this equals the sequential definition of include/sccg.h.
#pragma once
#include "sccg_extract.cuh"

namespace sccg {

static const int VR_T = 256;
static const int VR_I = 4;                      // scan elements per thread
static const int VR_STILE = VR_T * VR_I;
static const int VR_BPT = 16;                   // gap bytes per thread
static const int VR_TILE = VR_T * VR_BPT;       // 4 KiB of gap bytes per CTA
enum { SC_A = 0, SC_W, SC_NT, SC_NR, SC_NV, SC_AL, SC_RN, SC_COUNT };

// ---- exclusive u64 scans (sum or maximum; both have identity 0) in three launches: tile totals, one CTA over the tile
//      totals, tiles again.  The element count may live in device memory (n_dev) with a host bound sizing the grids.
struct VrSum { static __device__ __forceinline__ u64 op(u64 a, u64 b) { return a + b; } };
struct VrMax { static __device__ __forceinline__ u64 op(u64 a, u64 b) { return a > b ? a : b; } };

template <class Op> __device__ __forceinline__ u64 vr_block_excl(u64 v, u64* sm, u64* total) {
    const int lane = lane_of(), w = (int)(threadIdx.x >> 5), nw = (int)(blockDim.x >> 5);
    u64 incl = v;
    for (int d = 1; d < 32; d <<= 1) { const u64 y = __shfl_up_sync(SCCG_FULL_MASK, incl, d); if (lane >= d) incl = Op::op(incl, y); }
    u64 ex = __shfl_up_sync(SCCG_FULL_MASK, incl, 1);
    if (lane == 0) ex = 0;
    if (lane == 31) sm[w] = incl;
    __syncthreads();
    if (w == 0) {
        const u64 s = lane < nw ? sm[lane] : 0;
        u64 si = s;
        for (int d = 1; d < 32; d <<= 1) { const u64 y = __shfl_up_sync(SCCG_FULL_MASK, si, d); if (lane >= d) si = Op::op(si, y); }
        u64 se = __shfl_up_sync(SCCG_FULL_MASK, si, 1);
        if (lane == 0) se = 0;
        sm[lane] = se;
        if (lane == 31) sm[32] = si;
    }
    __syncthreads();
    const u64 r = Op::op(sm[w], ex);
    *total = sm[32];
    __syncthreads();
    return r;
}

template <class Op> __global__ void __launch_bounds__(VR_T) vr_scan_up_k(const u64* in, const u64* n_dev, u64 n_host, u64* agg) {
    __shared__ u64 sm[33];
    const u64 n = n_dev ? *n_dev : n_host;
    const u64 base = (u64)blockIdx.x * VR_STILE + threadIdx.x * VR_I;
    if ((u64)blockIdx.x * VR_STILE >= n) return;
    u64 v = 0;
    for (int j = 0; j < VR_I; ++j) if (base + j < n) v = Op::op(v, in[base + j]);
    u64 tot;
    vr_block_excl<Op>(v, sm, &tot);
    if (threadIdx.x == 0) agg[blockIdx.x] = tot;
}

template <class Op> __global__ void __launch_bounds__(VR_T) vr_scan_top_k(u64* agg, const u64* n_dev, u64 n_host, u64* total) {
    __shared__ u64 sm[33];
    const u64 n = n_dev ? *n_dev : n_host;
    const u64 nt = (n + VR_STILE - 1) / VR_STILE;
    u64 carry = 0;
    for (u64 b = 0; b < nt; b += VR_T) {
        const u64 i = b + threadIdx.x;
        const u64 v = i < nt ? agg[i] : 0;
        u64 tot;
        const u64 ex = vr_block_excl<Op>(v, sm, &tot);
        if (i < nt) agg[i] = Op::op(carry, ex);
        carry = Op::op(carry, tot);
    }
    if (threadIdx.x == 0 && total) *total = carry;
}

template <class Op> __global__ void __launch_bounds__(VR_T) vr_scan_down_k(const u64* in, u64* out, const u64* n_dev, u64 n_host, const u64* agg) {
    __shared__ u64 sm[33];
    const u64 n = n_dev ? *n_dev : n_host;
    if ((u64)blockIdx.x * VR_STILE >= n) return;
    const u64 base = (u64)blockIdx.x * VR_STILE + threadIdx.x * VR_I;
    u64 v[VR_I], s = 0;
    for (int j = 0; j < VR_I; ++j) { v[j] = base + j < n ? in[base + j] : 0; s = Op::op(s, v[j]); }
    u64 tot;
    u64 acc = Op::op(agg[blockIdx.x], vr_block_excl<Op>(s, sm, &tot));
    for (int j = 0; j < VR_I; ++j) { if (base + j < n) out[base + j] = acc; acc = Op::op(acc, v[j]); }
}

// out[i] = op of in[0 .. i) (in may alias out); n elements, in device memory at n_dev when given, at most n_bound; *total
// (device, optional) = op of all n.  agg: slot B_VR_AGG.
template <class Op> static int vr_scan(sccg_ctx* c, const u64* in, u64* out, const u64* n_dev, u64 n_bound, u64* total) {
    const unsigned nt = div_up((long long)(n_bound > 0 ? n_bound : 1), VR_STILE);
    u64* agg = nullptr;
    SCCG_TRY(buf(c, B_VR_AGG, (size_t)nt, &agg));
    LAUNCH(c, vr_scan_up_k<Op>, dim3(nt), dim3(VR_T), 0, in, n_dev, n_bound, agg);
    LAUNCH(c, vr_scan_top_k<Op>, dim3(1), dim3(VR_T), 0, agg, n_dev, n_bound, total);
    LAUNCH(c, vr_scan_down_k<Op>, dim3(nt), dim3(VR_T), 0, in, out, n_dev, n_bound, (const u64*)agg);
    return SCCG_OK;
}

// ---- the N runs of the resident reference (raw coordinates), for global-mode archives: run k begins before stripped
//      symbol rn_sp[k] of the N-stripped form, and stripped symbol q is raw symbol q + rn_add[k] (k: the last run with
//      rn_sp[k] <= q).  Built once per resident reference, next to its forms.
__global__ void __launch_bounds__(VR_T) vr_nrun_k(const u8* R, i64 n, u64* cnt_s, u64* cnt_e, const u64* off_s, const u64* off_e, u32* st, u32* en) {
    __shared__ u64 sm[33];
    const i64 b0 = (i64)blockIdx.x * VR_TILE + (i64)threadIdx.x * VR_BPT;
    u32 ms = 0, me = 0;                                              // run starts / run ends among the thread's bytes
    for (int i = 0; i < VR_BPT; ++i) {
        const i64 b = b0 + i;
        if (b >= n || R[b] != 'N') continue;
        if (b == 0 || R[b - 1] != 'N') ms |= 1u << i;
        if (b + 1 == n || R[b + 1] != 'N') me |= 1u << i;
    }
    u64 ts, te;
    const u64 xs = vr_block_excl<VrSum>((u64)__popc(ms), sm, &ts);
    const u64 xe = vr_block_excl<VrSum>((u64)__popc(me), sm, &te);
    if (!st) { if (threadIdx.x == 0) { cnt_s[blockIdx.x] = ts; cnt_e[blockIdx.x] = te; } return; }
    u64 os = off_s[blockIdx.x] + xs, oe = off_e[blockIdx.x] + xe;
    for (; ms; ms &= ms - 1) st[os++] = (u32)(b0 + __ffs((int)ms) - 1);
    for (; me; me &= me - 1) en[oe++] = (u32)(b0 + __ffs((int)me));  // (exclusive end)
}

// run lengths (scanned into cum[k], the N symbols before run k), then rn_sp = start - cum and rn_add = cum + len in place
__global__ void vr_nrun_len_k(const u32* st, const u32* en, u64 k_n, u64* len) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < k_n) len[k] = en[k] - st[k];
}
__global__ void vr_nrun_fin_k(u32* st, u32* en, u64 k_n, const u64* cum) {
    const u64 k = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= k_n) return;
    const u32 s = st[k], e = en[k];
    st[k] = s - (u32)cum[k];                                          // rn_sp (in place)
    en[k] = (u32)cum[k] + (e - s);                                     // rn_add (in place)
}

static int reference_nruns(sccg_ctx* c) {
    if (c->res_nrun) return SCCG_OK;
    const i64 n = c->res_ref_len;
    const unsigned nt = div_up(n > 0 ? n : 1, VR_TILE);
    u64 *cs = nullptr, *ce = nullptr, *sc = nullptr;
    SCCG_TRY(buf(c, B_VR_KEY, 2 * (size_t)nt, &cs));
    ce = cs + nt;
    SCCG_TRY(buf(c, B_VR_SC, SC_COUNT, &sc));
    LAUNCH(c, vr_nrun_k, dim3(nt), dim3(VR_T), 0, (const u8*)c->res_ref, n, cs, ce, (const u64*)nullptr, (const u64*)nullptr, (u32*)nullptr, (u32*)nullptr);
    SCCG_TRY(vr_scan<VrSum>(c, cs, cs, nullptr, nt, sc + SC_RN));
    SCCG_TRY(vr_scan<VrSum>(c, ce, ce, nullptr, nt, nullptr));
    u64* h = (u64*)c->h_pinned;
    SCCG_CK(cudaMemcpyAsync(h, sc + SC_RN, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    const u64 k_n = *h;
    void* p = nullptr;
    if (cudaMalloc(&p, sizeof(u32) * 2 * (k_n + 1)) != cudaSuccess) { cudaGetLastError(); return set_error(SCCG_E_NOMEM, "cudaMalloc of the reference N runs failed"); }
    u32* st = (u32*)p; u32* en = st + k_n + 1;
    u64* len = nullptr;
    int rc = buf(c, B_VR_CNT, (size_t)k_n + 1, &len);
    if (rc == SCCG_OK && k_n > 0) {
        LAUNCH(c, vr_nrun_k, dim3(nt), dim3(VR_T), 0, (const u8*)c->res_ref, n, cs, ce, (const u64*)cs, (const u64*)ce, st, en);
        LAUNCH(c, vr_nrun_len_k, dim3(div_up((long long)k_n, VR_T)), dim3(VR_T), 0, (const u32*)st, (const u32*)en, k_n, len);
        rc = vr_scan<VrSum>(c, len, len, nullptr, k_n, nullptr);
        if (rc == SCCG_OK) LAUNCH(c, vr_nrun_fin_k, dim3(div_up((long long)k_n, VR_T)), dim3(VR_T), 0, st, en, k_n, (const u64*)len);
    }
    if (rc != SCCG_OK) { cudaStreamSynchronize(c->stream); cudaFree(p); return rc; }
    c->res_nrun = p; c->res_nrun_k = (long long)k_n;
    return SCCG_OK;
}

// ---- the pipeline
struct VrArch {
    GatherArgs g;            // the archive's tables (sccg_archive::g)
    i64 e0;                  // its first element (segments, then the sentinel)
    i64 dlen;                // len(D)
    int mode;                // 0 local, 1 global
    int pad;
};
struct VrAnchor { i64 x, p, l, k; };          // raw D / R coordinates, archive ordinal
struct VrWin { i64 start, end, k; };
struct VrGap { i64 lx, lp, nd, nr; int k; };

struct VrArgs {
    const VrArch* arch; int n_arch;
    const u8* R; i64 rlen;                    // raw resident reference
    const u32* rn_sp; const u32* rn_add; int rn_k;
    u64 n_elem;
    u64* key;                                 // per element: copy key, then M (max scan)
    u64* cnt;                                 // per element: pieces of its anchor, then their offset (sum scan)
    VrAnchor* anc;
    u64* goff;                                // per gap: width, then offset in the gap-byte space
    u32* suf; u32* pre;                       // per gap of unequal length: first difference from the end / from the start
    u64* tcnt;                                // per tile: records, then their offset
    sccg_variant* rec3;                       // records of step 3 (window = archive ordinal)
    sccg_variant* recf;                       // left-aligned
    u64* sc;
};

__device__ __forceinline__ u8 vr_r(const VrArgs& a, i64 q) { return upper1(a.R[q]); }
__device__ __forceinline__ u8 vr_d(const GatherArgs& g, i64 b) { return upper1(ext_sym(g, ExtWin{0, g.nseg - 1, 0, g.n_k - 1, 0, -1}, b)); }

__device__ __forceinline__ int vr_arch_of(const VrArgs& a, u64 e) {
    int lo = 0, hi = a.n_arch;
    while (hi - lo > 1) { const int m = (lo + hi) >> 1; if ((u64)a.arch[m].e0 <= e) lo = m; else hi = m; }
    return lo;
}

// copy segment j: N-free start x, reference-form start p, length l (0 for a literal run)
__device__ __forceinline__ void vr_seg(const GatherArgs& g, int j, i64* x, i64* p, i64* l) {
    const i64 src = g.seg_ptr[j];
    *x = g.seg_dst[j];
    const i64 x1 = j + 1 < g.nseg ? (i64)g.seg_dst[j + 1] : g.Ls;
    *p = src;
    *l = (src < 0 || (src & SEG_LIT_FLAG)) ? 0 : x1 - *x;
}

__global__ void __launch_bounds__(VR_T) vr_key_k(VrArgs a) {
    const u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.n_elem) return;
    const int k = vr_arch_of(a, e);
    const GatherArgs& g = a.arch[k].g;
    const i64 j = (i64)e - a.arch[k].e0;
    u64 key = 0;
    if (j < g.nseg) {
        i64 x, p, l;
        vr_seg(g, (int)j, &x, &p, &l);
        if (l > 0) key = ((u64)(k + 1) << 32) | (u64)(p + l);
    }
    a.key[e] = key;
}

// last target N run k with n_start[k] - n_cum[k] <= x (its N-free position), or -1
__device__ __forceinline__ int vr_last_tp(const GatherArgs& g, i64 x) {
    int lo = 0, hi = g.n_k;
    while (lo < hi) { const int m = (lo + hi) >> 1; if ((i64)g.n_start[m] - (i64)g.n_cum[m] <= x) lo = m + 1; else hi = m; }
    return lo - 1;
}
__device__ __forceinline__ int vr_last_sp(const VrArgs& a, i64 q) {
    int lo = 0, hi = a.rn_k;
    while (lo < hi) { const int m = (lo + hi) >> 1; if ((i64)a.rn_sp[m] <= q) lo = m + 1; else hi = m; }
    return lo - 1;
}

// the pieces of element e's anchor in raw coordinates (out == NULL: counted only).  M: the maximum scan at e.
__device__ u64 vr_anchor_walk(const VrArgs& a, u64 e, u64 M, VrAnchor* out) {
    const int k = vr_arch_of(a, e);
    const VrArch& A = a.arch[k];
    const GatherArgs& g = A.g;
    const i64 j = (i64)e - A.e0;
    if (j == g.nseg) { if (out) *out = VrAnchor{A.dlen, a.rlen, 0, k}; return 1; }       // the sentinel closes the archive
    i64 x, p, l;
    vr_seg(g, (int)j, &x, &p, &l);
    if (l <= 0) return 0;
    const i64 m = (M >> 32) == (u64)(k + 1) ? (i64)(M & 0xffffffffu) : 0;
    const i64 s = m > p ? m - p : 0;
    if (s >= l) return 0;
    x += s; p += s; l -= s;
    if (A.mode == 0) { if (out) *out = VrAnchor{x, p, l, k}; return 1; }
    // global mode: x is N-free, p N-stripped; split where D skips a target N run or R skips a reference N run
    int kt = vr_last_tp(g, x), kr = vr_last_sp(a, p);
    i64 dx = kt >= 0 ? (i64)g.n_cum[kt] + g.n_len[kt] : 0, rx = kr >= 0 ? (i64)a.rn_add[kr] : 0;
    u64 n = 0;
    for (i64 o = 0; o < l;) {
        const i64 nt = kt + 1 < g.n_k ? (i64)g.n_start[kt + 1] - (i64)g.n_cum[kt + 1] - x : l;
        const i64 nr = kr + 1 < a.rn_k ? (i64)a.rn_sp[kr + 1] - p : l;
        i64 cut = nt < nr ? nt : nr;
        cut = cut < l ? cut : l;
        if (cut > o) { if (out) out[n] = VrAnchor{x + o + dx, p + o + rx, cut - o, k}; ++n; }
        if (cut == nt && nt < l) { ++kt; dx = (i64)g.n_cum[kt] + g.n_len[kt]; }
        if (cut == nr && nr < l) { ++kr; rx = a.rn_add[kr]; }
        o = cut;
    }
    return n;
}

__global__ void __launch_bounds__(VR_T) vr_anchor_k(VrArgs a, int emit) {
    const u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.n_elem) return;
    if (emit) vr_anchor_walk(a, e, a.key[e], a.anc + a.cnt[e]);
    else a.cnt[e] = vr_anchor_walk(a, e, a.key[e], nullptr);
}

__device__ __forceinline__ VrGap vr_gap(const VrArgs& a, u64 j) {
    const VrAnchor r = a.anc[j];
    i64 x0 = 0, p0 = 0;
    if (j > 0) { const VrAnchor q = a.anc[j - 1]; if (q.k == r.k) { x0 = q.x + q.l; p0 = q.p + q.l; } }
    return VrGap{x0, p0, r.x - x0, r.p - p0, (int)r.k};
}

__global__ void __launch_bounds__(VR_T) vr_gap_k(VrArgs a) {
    const u64 A = a.sc[SC_A];
    for (u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x; j < A; j += (u64)gridDim.x * blockDim.x) {
        const VrGap G = vr_gap(a, j);
        const i64 m = G.nd < G.nr ? G.nd : G.nr;
        a.goff[j] = (u64)(G.nd > G.nr ? G.nd : G.nr);
        a.suf[j] = (u32)m; a.pre[j] = (u32)m;
    }
}

// the thread's bytes of gap-byte tile t in byte order: gap j, its geometry G, byte i of the gap
struct VrCursor {
    u64 b, be, j, A, g0;
    VrGap G;
    __device__ __forceinline__ VrCursor(const VrArgs& a, u64 t) {
        const u64 W = a.sc[SC_W];
        A = a.sc[SC_A];
        b = t * VR_TILE + (u64)threadIdx.x * VR_BPT;
        be = b + VR_BPT < W ? b + VR_BPT : W;
        u64 lo = 0, hi = A;                                           // last gap with goff <= b
        if (b < be) while (hi - lo > 1) { const u64 m = (lo + hi) >> 1; if (a.goff[m] <= b) lo = m; else hi = m; }
        j = lo;
        if (b < be) { G = vr_gap(a, j); g0 = a.goff[j]; }
    }
    __device__ __forceinline__ bool more() const { return b < be; }
    __device__ __forceinline__ i64 i() const { return (i64)(b - g0); }
    __device__ __forceinline__ void next(const VrArgs& a) {
        if (++b >= be) return;
        bool moved = false;
        while (j + 1 < A && a.goff[j + 1] <= b) { ++j; moved = true; }
        if (moved) { G = vr_gap(a, j); g0 = a.goff[j]; }
    }
};

__device__ __forceinline__ bool vr_diff(const VrArgs& a, const VrGap& G, i64 i) {
    return vr_r(a, G.lp + i) != vr_d(a.arch[G.k].g, G.lx + i);
}

__global__ void __launch_bounds__(VR_T) vr_trim_k(VrArgs a) {
    const u64 NT = (a.sc[SC_W] + VR_TILE - 1) / VR_TILE;
    if (blockIdx.x == 0 && threadIdx.x == 0) a.sc[SC_NT] = NT;
    for (u64 t = blockIdx.x; t < NT; t += gridDim.x) {
        u64 cj = ~0ull;
        u32 cs = ~0u, cp = ~0u;                                        // first difference from the end / the start in gap cj
        for (VrCursor c(a, t); c.more(); c.next(a)) {
            const VrGap& G = c.G;
            const i64 m = G.nd < G.nr ? G.nd : G.nr, i = c.i();
            if (G.nd == G.nr || i >= m) continue;
            if (c.j != cj) {
                if (cj != ~0ull && cs != ~0u) atomicMin(&a.suf[cj], cs);
                if (cj != ~0ull && cp != ~0u) atomicMin(&a.pre[cj], cp);
                cj = c.j; cs = cp = ~0u;
            }
            const GatherArgs& g = a.arch[G.k].g;
            if (cs == ~0u && vr_r(a, G.lp + G.nr - 1 - i) != vr_d(g, G.lx + G.nd - 1 - i)) cs = (u32)i;
            if (cp == ~0u && vr_r(a, G.lp + i) != vr_d(g, G.lx + i)) cp = (u32)i;
        }
        if (cj != ~0ull && cs != ~0u) atomicMin(&a.suf[cj], cs);
        if (cj != ~0ull && cp != ~0u) atomicMin(&a.pre[cj], cp);
    }
}

// the record starts among the thread's bytes of tile t: a gap of unequal length has one record, at its byte 0; a gap of equal
// length one per maximal run of differing positions.  Returns their number; EMIT: writes the records from rec3[r] on.
template <bool EMIT> __device__ __forceinline__ u32 vr_starts(const VrArgs& a, u64 t, u64 r) {
    u64 pj = ~0ull;
    i64 pi = -2;
    bool pd = false;
    u32 n = 0;
    for (VrCursor c(a, t); c.more(); c.next(a)) {
        const VrGap& G = c.G;
        const i64 i = c.i();
        bool start;
        if (G.nd != G.nr) {
            start = i == 0;
        } else {
            const bool d = vr_diff(a, G, i);
            const bool prev = i == 0 ? false : (c.j == pj && i == pi + 1) ? pd : vr_diff(a, G, i - 1);
            pj = c.j; pi = i; pd = d;
            start = d && !prev;
        }
        if (!start) continue;
        ++n;
        if (!EMIT) continue;
        sccg_variant v;
        v.window = G.k; v.alt_off = 0;
        if (G.nd != G.nr) {
            const i64 m = G.nd < G.nr ? G.nd : G.nr, suf = a.suf[c.j];
            const i64 pre = (i64)a.pre[c.j] < m - suf ? (i64)a.pre[c.j] : m - suf;
            v.pos = G.lp + pre; v.end = G.lp + G.nr - suf; v.d_start = G.lx + pre; v.d_end = G.lx + G.nd - suf;
        } else {
            i64 e = i + 1;
            while (e < G.nd && vr_diff(a, G, e)) ++e;
            v.pos = G.lp + i; v.end = G.lp + e; v.d_start = G.lx + i; v.d_end = G.lx + e;
        }
        a.rec3[r++] = v;
    }
    return n;
}

__global__ void __launch_bounds__(VR_T) vr_count_k(VrArgs a) {
    __shared__ u32 sm[40];
    const u64 NT = a.sc[SC_NT];
    for (u64 t = blockIdx.x; t < NT; t += gridDim.x) {
        const u32 n = vr_starts<false>(a, t, 0);
        u32 tot;
        block_scan_excl(n, sm, &tot);
        if (threadIdx.x == 0) a.tcnt[t] = tot;
    }
}

__global__ void __launch_bounds__(VR_T) vr_emit_k(VrArgs a) {
    __shared__ u32 sm[40];
    const u64 NT = a.sc[SC_NT];
    for (u64 t = blockIdx.x; t < NT; t += gridDim.x) {
        const u32 n = vr_starts<false>(a, t, 0);
        u32 tot;
        const u64 r = a.tcnt[t] + block_scan_excl(n, sm, &tot);
        vr_starts<true>(a, t, r);
    }
}

// left-alignment of insertions and deletions, bounded by the step-3 end of the previous record of the archive
__global__ void __launch_bounds__(VR_T) vr_align_k(VrArgs a, u64 nr) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < nr; r += (u64)gridDim.x * blockDim.x) {
        sccg_variant v = a.rec3[r];
        const bool del = v.d_end == v.d_start, ins = v.end == v.pos;
        if (del != ins) {
            const i64 bound = (r > 0 && a.rec3[r - 1].window == v.window) ? a.rec3[r - 1].end : 0;
            const GatherArgs& g = a.arch[v.window].g;
            while (v.pos > bound) {
                const u8 last = del ? vr_r(a, v.end - 1) : vr_d(g, v.d_end - 1);
                if (vr_r(a, v.pos - 1) != last) break;
                --v.pos; --v.end; --v.d_start; --v.d_end;
            }
        }
        a.recf[r] = v;
    }
}

__global__ void __launch_bounds__(VR_T) vr_altlen_k(const sccg_variant* rec, u64 nr, u64* len) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < nr; r += (u64)gridDim.x * blockDim.x) len[r] = (u64)(rec[r].d_end - rec[r].d_start);
}

// first record at or after (archive k, pos)
__device__ __forceinline__ u64 vr_lower(const sccg_variant* rec, u64 n, i64 k, i64 pos) {
    u64 lo = 0, hi = n;
    while (lo < hi) {
        const u64 m = (lo + hi) >> 1;
        const sccg_variant& v = rec[m];
        if (v.window < k || (v.window == k && v.pos < pos)) lo = m + 1; else hi = m;
    }
    return lo;
}

// per window: its records [wlo, wlo + wcnt) and their ALT bytes (P: exclusive ALT-length prefix over the records, P[nr] the total)
// (a window that ends at len(R) also takes the insertions at len(R))
__global__ void __launch_bounds__(VR_T) vr_win_k(const sccg_variant* rec, u64 nr, const u64* P, const VrWin* win, u64 nw, i64 rlen, u64* wcnt, u64* walt,
                                                 u64* wlo) {
    const u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nw) return;
    const VrWin W = win[w];
    const u64 lo = vr_lower(rec, nr, W.k, W.start), hi = vr_lower(rec, nr, W.k, W.end == rlen ? rlen + 1 : W.end);
    wcnt[w] = hi - lo; walt[w] = P[hi] - P[lo]; wlo[w] = lo;
}

// last i < n with off[i] <= x
__device__ __forceinline__ u64 vr_upper(const u64* off, u64 n, u64 x) {
    u64 lo = 0, hi = n;
    while (hi - lo > 1) { const u64 m = (lo + hi) >> 1; if (off[m] <= x) lo = m; else hi = m; }
    return lo;
}

__global__ void __launch_bounds__(VR_T) vr_out_k(const sccg_variant* rec, const u64* P, u64 nw, const u64* woff, const u64* waoff, const u64* wlo,
                                                 u64 nv, sccg_variant* out) {
    for (u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x; j < nv; j += (u64)gridDim.x * blockDim.x) {
        const u64 w = vr_upper(woff, nw, j);
        const u64 r = wlo[w] + (j - woff[w]);
        sccg_variant v = rec[r];
        v.window = (i64)w;
        v.alt_off = (i64)(waoff[w] + P[r] - P[wlo[w]]);
        out[j] = v;
    }
}

__global__ void __launch_bounds__(VR_T) vr_alt_k(VrArgs a, const sccg_variant* out, u64 nv, const VrWin* win, u64 al, u8* alt) {
    for (u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x; q < al; q += (u64)gridDim.x * blockDim.x) {
        u64 lo = 0, hi = nv;                                          // the last record whose ALT starts at or before q
        while (hi - lo > 1) { const u64 m = (lo + hi) >> 1; if ((u64)out[m].alt_off <= q) lo = m; else hi = m; }
        const sccg_variant v = out[lo];
        alt[q] = vr_d(a.arch[win[v.window].k].g, v.d_start + (i64)(q - (u64)v.alt_off));
    }
}

// steps 1-4 of include/sccg.h for the archives arcs[0 .. n_arch) (a record's window is the archive's ordinal there): the
// staging table [VrArch of each archive | tail_bytes that fill(tail) writes] goes over in one copy (ev[4] -> ev[5]), and *d_tail
// is the device copy of the tail.  Runs the anchors, gaps and per-tile record counts (ev[3] -> ev[2], added to *ms) and reads
// the record total once into *nr; rec3 / recf are then sized for it.  vr_records_emit writes the records into a->recf.
template <class Fill>
static int vr_records_count(sccg_ctx* c, sccg_archive* const* arcs, int n_arch, size_t tail_bytes, Fill fill, VrArgs* out, u8** d_tail, u64* nr, float* ms) {
    int n_global = 0;
    u64 n_elem = 0, anc_bound = 0, byte_bound = 0;
    for (int k = 0; k < n_arch; ++k) {
        const sccg_archive* a = arcs[k];
        n_elem += (u64)a->g.nseg + 1;
        anc_bound += (u64)a->g.nseg + 1 + (a->mode ? (u64)a->g.n_k : 0);
        byte_bound += (u64)a->g.Lm + (u64)c->res_ref_len;
        n_global += a->mode == 1;
    }
    if (n_global) {                                                          // a reference N run splits at most one anchor per archive
        SCCG_TRY(reference_nruns(c));
        anc_bound += (u64)n_global * (u64)c->res_nrun_k;
    }
    const u64 tile_bound = byte_bound / VR_TILE + 1;
    // ---- staging: [VrArch of each archive | the caller's tail], one copy
    const size_t arch_bytes = align_up(sizeof(VrArch) * (size_t)n_arch, 16);
    SCCG_TRY(ext_staging(c, arch_bytes + tail_bytes));
    VrArch* h_arch = (VrArch*)c->h_ext;
    {
        i64 e0 = 0;
        for (int k = 0; k < n_arch; ++k) {
            const sccg_archive* a = arcs[k];
            VrArch& A = h_arch[k];
            memset(&A, 0, sizeof A);
            A.g = a->g; A.e0 = e0; A.dlen = a->g.Lm; A.mode = a->mode;
            e0 += a->g.nseg + 1;
        }
        fill((char*)c->h_ext + arch_bytes);
    }
    u8* d_tab = nullptr; u64* sc = nullptr;
    SCCG_TRY(buf(c, B_VR_TAB, arch_bytes + tail_bytes, &d_tab));
    SCCG_TRY(buf(c, B_VR_SC, SC_COUNT, &sc));
    VrArgs a;
    memset(&a, 0, sizeof a);
    a.arch = (const VrArch*)d_tab; a.n_arch = n_arch;
    a.R = c->res_ref; a.rlen = c->res_ref_len;
    if (n_global) { a.rn_sp = (const u32*)c->res_nrun; a.rn_add = a.rn_sp + c->res_nrun_k + 1; a.rn_k = (int)c->res_nrun_k; }
    a.n_elem = n_elem; a.sc = sc;
    SCCG_TRY(buf(c, B_VR_KEY, (size_t)n_elem, &a.key));
    SCCG_TRY(buf(c, B_VR_CNT, (size_t)n_elem, &a.cnt));
    SCCG_TRY(buf(c, B_VR_ANC, (size_t)anc_bound, &a.anc));
    u8* gp = nullptr;
    SCCG_TRY(buf(c, B_VR_GAP, (size_t)anc_bound * 16, &gp));
    a.goff = (u64*)gp; a.suf = (u32*)(gp + 8 * anc_bound); a.pre = a.suf + anc_bound;
    SCCG_TRY(buf(c, B_VR_TILE, (size_t)tile_bound, &a.tcnt));
    *d_tail = d_tab + arch_bytes;
    SCCG_CK(cudaEventRecord(c->ev[4], c->stream));
    SCCG_CK(cudaMemcpyAsync(d_tab, c->h_ext, arch_bytes + tail_bytes, cudaMemcpyHostToDevice, c->stream));
    SCCG_CK(cudaEventRecord(c->ev[5], c->stream));
    // ---- anchors, gaps, records per tile
    const unsigned grid = (unsigned)(c->sm_count > 0 ? c->sm_count : 1) * 8u;
    const unsigned eg = div_up((long long)n_elem, VR_T);
    SCCG_CK(cudaEventRecord(c->ev[3], c->stream));
    LAUNCH(c, vr_key_k, dim3(eg), dim3(VR_T), 0, a);
    SCCG_TRY(vr_scan<VrMax>(c, a.key, a.key, nullptr, n_elem, nullptr));
    LAUNCH(c, vr_anchor_k, dim3(eg), dim3(VR_T), 0, a, 0);
    SCCG_TRY(vr_scan<VrSum>(c, a.cnt, a.cnt, nullptr, n_elem, sc + SC_A));
    LAUNCH(c, vr_anchor_k, dim3(eg), dim3(VR_T), 0, a, 1);
    LAUNCH(c, vr_gap_k, dim3(grid), dim3(VR_T), 0, a);
    SCCG_TRY(vr_scan<VrSum>(c, a.goff, a.goff, sc + SC_A, anc_bound, sc + SC_W));
    LAUNCH(c, vr_trim_k, dim3(grid), dim3(VR_T), 0, a);
    LAUNCH(c, vr_count_k, dim3(grid), dim3(VR_T), 0, a);
    SCCG_TRY(vr_scan<VrSum>(c, a.tcnt, a.tcnt, sc + SC_NT, tile_bound, sc + SC_NR));
    SCCG_CK(cudaEventRecord(c->ev[2], c->stream));
    u64* h = (u64*)c->h_pinned;
    SCCG_CK(cudaMemcpyAsync(h, sc + SC_NR, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    float t = 0.f;
    cudaEventElapsedTime(&t, c->ev[3], c->ev[2]); *ms += t;
    *nr = h[0];
    SCCG_TRY(buf(c, B_VR_REC3, (size_t)*nr * 2 + 2, &a.rec3));
    a.recf = a.rec3 + *nr + 1;
    *out = a;
    return SCCG_OK;
}

// the nr records of step 3, then each insertion / deletion left-aligned (step 4), into a.recf
static int vr_records_emit(sccg_ctx* c, const VrArgs& a, u64 nr) {
    const unsigned grid = (unsigned)(c->sm_count > 0 ? c->sm_count : 1) * 8u;
    const unsigned rg = nr ? (div_up((long long)nr, VR_T) < grid ? div_up((long long)nr, VR_T) : grid) : 1;
    LAUNCH(c, vr_emit_k, dim3(grid), dim3(VR_T), 0, a);
    LAUNCH(c, vr_align_k, dim3(rg), dim3(VR_T), 0, a, nr);
    return SCCG_OK;
}

// sccg_archive_variants: argument checks (include/sccg.h, in that order), then the pipeline above
static int archive_variants_impl(sccg_ctx* c, sccg_archive* const* archives, i64 n_archives, const sccg_window* windows, i64 n_windows,
                                 sccg_variant* vars, i64 vars_cap, int64_t* n_vars, char* alt, i64 alt_cap, int64_t* alt_len) {
    if (!n_vars || !alt_len || n_archives < 0 || n_windows < 0 || vars_cap < 0 || alt_cap < 0 || (n_archives > 0 && !archives) ||
        (n_windows > 0 && !windows))
        return set_error(SCCG_E_ARG, "null argument");
    *n_vars = 0; *alt_len = 0;
    if (n_archives >= 0x80000000LL || n_windows >= 0x80000000LL) return set_error(SCCG_E_ARG, "at most 2^31 - 1 archives and windows per call");
    int first = ARCHIVE_QUERY_OK;
    for (i64 i = 0; i < n_windows && first > 0; ++i) {
        const sccg_window& W = windows[i];
        const int f = archive_query_fault(c, archives, n_archives, W.archive, W.start, W.end);
        const int bad = f < 4 ? f : (W.start < 0 || W.start > W.end) ? 4 : W.end > c->res_ref_len ? 5 : ARCHIVE_QUERY_OK;
        if (bad < first) first = bad;
    }
    if (first == 5) return set_error(SCCG_E_ARG, "a window ends past the end of the resident reference");
    if (first < ARCHIVE_QUERY_OK) return set_error(SCCG_E_ARG, archive_query_why[first]);
    if (n_windows == 0) return SCCG_OK;
    // ---- the archives the windows name, in index order, then the records of steps 1-4 with the window table in the same copy
    std::vector<int> ord((size_t)n_archives, -1);
    for (i64 i = 0; i < n_windows; ++i) ord[(size_t)windows[i].archive] = 0;
    std::vector<sccg_archive*> named;
    for (i64 k = 0; k < n_archives; ++k)
        if (ord[(size_t)k] >= 0) { ord[(size_t)k] = (int)named.size(); named.push_back(archives[k]); }
    const size_t win_bytes = sizeof(VrWin) * (size_t)n_windows;
    auto fill = [&](void* tail) {
        VrWin* h_win = (VrWin*)tail;
        for (i64 i = 0; i < n_windows; ++i) h_win[i] = VrWin{windows[i].start, windows[i].end, ord[(size_t)windows[i].archive]};
    };
    VrArgs a;
    u8* d_tail = nullptr;
    u64 nr = 0;
    float ms = 0.f, gat = 0.f;
    SCCG_TRY(vr_records_count(c, named.data(), (int)named.size(), win_bytes, fill, &a, &d_tail, &nr, &gat));
    const VrWin* d_win = (const VrWin*)d_tail;
    u64* sc = a.sc;
    u64* h = (u64*)c->h_pinned;
    // ---- records, left-alignment, the windows
    u64 *P = nullptr, *wt = nullptr;
    SCCG_TRY(buf(c, B_VR_P, (size_t)nr + 1, &P));
    SCCG_TRY(buf(c, B_VR_WIN, 5 * (size_t)n_windows, &wt));
    u64 *woff = wt, *waoff = wt + n_windows, *wlo = wt + 2 * n_windows;
    const unsigned grid = (unsigned)(c->sm_count > 0 ? c->sm_count : 1) * 8u;
    const unsigned rg = nr ? (div_up((long long)nr, VR_T) < grid ? div_up((long long)nr, VR_T) : grid) : 1;
    SCCG_CK(cudaEventRecord(c->ev[3], c->stream));
    SCCG_TRY(vr_records_emit(c, a, nr));
    LAUNCH(c, vr_altlen_k, dim3(rg), dim3(VR_T), 0, (const sccg_variant*)a.recf, nr, P);
    SCCG_TRY(vr_scan<VrSum>(c, P, P, nullptr, nr, P + nr));
    LAUNCH(c, vr_win_k, dim3(div_up(n_windows, VR_T)), dim3(VR_T), 0, (const sccg_variant*)a.recf, nr, (const u64*)P, d_win, (u64)n_windows, a.rlen, woff, waoff, wlo);
    SCCG_TRY(vr_scan<VrSum>(c, woff, woff, nullptr, (u64)n_windows, sc + SC_NV));
    SCCG_TRY(vr_scan<VrSum>(c, waoff, waoff, nullptr, (u64)n_windows, sc + SC_AL));
    SCCG_CK(cudaEventRecord(c->ev[2], c->stream));
    SCCG_CK(cudaMemcpyAsync(h, sc + SC_NV, 2 * sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    cudaEventElapsedTime(&ms, c->ev[3], c->ev[2]); gat += ms;
    const u64 nv = h[0], al = h[1];
    *n_vars = (int64_t)nv; *alt_len = (int64_t)al;
    c->prof.gather_ms = gat; c->prof.kernels_ms = gat;
    cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]); c->prof.h2d_ms = ms;
    if (!vars) return SCCG_OK;
    if (al > 0 && !alt) return set_error(SCCG_E_ARG, "null argument");
    if ((u64)vars_cap < nv || (u64)alt_cap < al) return set_error(SCCG_E_ARG, "record or ALT buffer too small (required sizes returned in *n_vars and *alt_len)");
    if (nv == 0) return SCCG_OK;
    // ---- the records of every window, their ALT bytes, one copy of each
    sccg_variant* d_out = nullptr; u8* d_alt = nullptr;
    SCCG_TRY(buf(c, B_VR_OUT, (size_t)nv, &d_out));
    SCCG_TRY(buf(c, B_OUT, (size_t)al + 16, &d_alt));
    const unsigned og = div_up((long long)nv, VR_T) < grid ? div_up((long long)nv, VR_T) : grid;
    const unsigned ag = al ? (div_up((long long)al, VR_T) < grid ? div_up((long long)al, VR_T) : grid) : 1;
    SCCG_CK(cudaEventRecord(c->ev[3], c->stream));
    LAUNCH(c, vr_out_k, dim3(og), dim3(VR_T), 0, (const sccg_variant*)a.recf, (const u64*)P, (u64)n_windows, (const u64*)woff, (const u64*)waoff,
           (const u64*)wlo, nv, d_out);
    if (al) LAUNCH(c, vr_alt_k, dim3(ag), dim3(VR_T), 0, a, (const sccg_variant*)d_out, nv, d_win, al, d_alt);
    SCCG_CK(cudaEventRecord(c->ev[2], c->stream));
    SCCG_CK(cudaMemcpyAsync(vars, d_out, sizeof(sccg_variant) * (size_t)nv, cudaMemcpyDeviceToHost, c->stream));
    if (al) SCCG_CK(cudaMemcpyAsync(alt, d_alt, (size_t)al, cudaMemcpyDeviceToHost, c->stream));
    SCCG_CK(cudaEventRecord(c->ev[7], c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    cudaEventElapsedTime(&ms, c->ev[3], c->ev[2]); gat += ms;
    c->prof.gather_ms = gat; c->prof.kernels_ms = gat;
    cudaEventElapsedTime(&ms, c->ev[2], c->ev[7]); c->prof.d2h_ms = ms;
    return SCCG_OK;
}

}  // namespace sccg
