// Edit-distance pattern search over open archives (sccg_archive_search_edits, include/sccg.h): every end of an alignment of up
// to 1024 patterns of 1 to 64 bytes within max_edits unit-cost edits (substitutions, insertions, deletions), on either strand,
// inside windows of D of any open archive.  The image, the tile build and the region tables are those of sccg_search.cuh; the
// candidates are end positions, so a window cut over launches carries look-behind instead of look-ahead.
//
//   image            -> the concatenation of the windows; a window that does not fit a launch is cut into pieces, each with the
//                       L = maxlen + max_edits - 1 bytes of its window before its first candidate end (an alignment with at most
//                       k edits spans at most m + k bytes of D)
//   srch_edit_count_k-> one CTA per 4096 candidate ends: the tile and up to 128 bytes before it built in shared memory by
//                       srch_build; each thread runs Myers' bit-parallel column DP (search mode: free start in D) for every
//                       pattern over its 32 ends, from m + k bytes before its first end (never before the start of the region),
//                       restarting at every region start; hits of each tile
//   scan             -> scan_exclusive_u32 of the tile counts: each tile's first hit, and the launch total (one round trip)
//   srch_edit_emit_k -> the tiles that hold hits built again and counted again; each end that holds a hit runs an anchored DP
//                       backward from the end (the reversed pattern against D read backward) for every pattern and strand: the
//                       least score over at most m + k bytes is d(e), the fewest bytes reaching it give the start; written as
//                       sccg_edit_hit in (window, end, pattern, strand) order
#pragma once
#include "sccg_search.cuh"

namespace sccg {

static const int SE_BEHIND = 128;                               // room for the look-behind: L <= 64 + 63 - 1 bytes
// the Peq slot of a lowercased byte l is (l >> 1) & 7: 0 for a, 1 c, 2 t, 3 g, 7 n; SE_LET holds those letters at their slots
static const u64 SE_LET = 0x6e00000067746361ull;
static const u32 SE_OTHER = 4;                                  // the slot of every other byte (Peq 0 in the table)

struct EditArgs {
    ExtArgs x;               // the launch's image, as for SrchArgs
    const u32* r_win;        // window index of region i
    const u32* r_cend;       // (= r_off[i + 1]: no look-ahead)
    const u32* r_cbeg;       // candidate ends of region i: the ends of image bytes [r_cbeg[i], r_off[i + 1]); bytes before are look-behind
    const u64* peq;          // peq[((i * 2 + strand) * 2 + dir) * 8 + slot]: bit j where byte j of the pattern (dir 0) or of the
                             // reversed pattern (dir 1) matches the slot's letter
    const u16* desc;         // pattern byte descriptors, as for SrchArgs (the Peq of a byte outside the five slots)
    const u8* plen;
    int n_pat, strands, kmax;
    u32* tile_cnt;           // count pass: hits of each tile
    const u32* tile_off;     // emit pass: their exclusive scan
    sccg_edit_hit* hits;     // emit pass: the launch's hits
};

struct EditSmem {
    __align__(16) u8 O[SE_BEHIND + SRCH_TILE];   // image bytes [Qb, Q0 + SRCH_TILE), Qb = Q0 - min(Q0, 128); zero past the last
    u8 S[SE_BEHIND + SRCH_TILE];                 // the Peq slot of each byte of O
    u32 red[33];
    int sh[2];
    __align__(8) u64 bar;
};

// one column of Myers' DP (Hyyro's formulation) for text byte with match mask eq; sc tracks the bottom row (score of the whole
// pattern).  Search mode: the top row is 0 (an alignment may start anywhere); anchored: the top row grows by one per column.
template <bool ANCHORED>
__device__ __forceinline__ void edit_step(u64 eq, u64 top, u64& Pv, u64& Mv, int& sc) {
    const u64 Xv = eq | Mv;
    const u64 Xh = (((eq & Pv) + Pv) ^ Pv) | eq;
    u64 Ph = Mv | ~(Xh | Pv);
    u64 Mh = Pv & Xh;
    sc += (int)((Ph & top) != 0) - (int)((Mh & top) != 0);
    Ph = (Ph << 1) | (ANCHORED ? 1ull : 0ull);
    Mh <<= 1;
    Pv = Mh | ~(Xv | Ph);
    Mv = Ph & Xv;
}

// Peq of a byte outside the five slots, from the descriptors of the pattern (rev: of the reversed pattern)
__device__ __forceinline__ u64 edit_peq_other(const u16* ds, u32 m, u32 b, bool rev) {
    u64 eq = 0;
    for (u32 j = 0; j < m; ++j)
        if (srch_match(ds[j], b)) eq |= 1ull << (rev ? m - 1u - j : j);
    return eq;
}

__device__ __forceinline__ u64 edit_eq(const EditArgs& a, const EditSmem& s, const u64* pq, int ps, u32 m, u32 i, bool rev) {
    const u32 sl = s.S[i];
    u64 eq = __ldg(pq + sl);
    if (sl == SE_OTHER) eq = edit_peq_other(a.desc + (size_t)ps * SRCH_MAXLEN, m, s.O[i], rev);
    return eq;
}

// the ends of image bytes [q0, qe) (in cand) within kmax edits of pattern pi on strands st0 .. st0 + NS - 1: the search-mode DP
// from image byte p0 of region r, restarted at each region start; bit i of hit[t] for the end of byte q0 + i
template <int NS>
__device__ __forceinline__ void edit_fwd(const EditArgs& a, const EditSmem& s, u32 Qb, int pi, int st0, u32 m, u32 p0, int r,
                                         u32 q0, u32 qe, u32 cand, u32* hit) {
    const u64 top = 1ull << (m - 1u);
    const u64* pq[NS];
    u64 Pv[NS], Mv[NS];
    int sc[NS];
#pragma unroll
    for (int t = 0; t < NS; ++t) { pq[t] = a.peq + (size_t)((pi * 2 + st0 + t) * 2) * 8; Pv[t] = ~0ull; Mv[t] = 0; sc[t] = (int)m; hit[t] = 0; }
    u32 nxt = a.x.r_off[r + 1];
    for (u32 p = p0; p < qe; ++p) {
        if (p == nxt) {                                               // a new region: its alignments start in it
#pragma unroll
            for (int t = 0; t < NS; ++t) { Pv[t] = ~0ull; Mv[t] = 0; sc[t] = (int)m; }
            nxt = a.x.r_off[++r + 1];
        }
        const u32 bit = p - q0;
#pragma unroll
        for (int t = 0; t < NS; ++t) {
            edit_step<false>(edit_eq(a, s, pq[t], pi * 2 + st0 + t, m, p - Qb, false), top, Pv[t], Mv[t], sc[t]);
            if (bit < 32u) hit[t] |= (u32)(sc[t] <= a.kmax) << bit;
        }
    }
#pragma unroll
    for (int t = 0; t < NS; ++t) hit[t] &= cand;
}

// count (EMIT = false) or emit pass of one tile: candidate ends of image bytes [Q0, Q0 + 4096)
template <bool EMIT>
__device__ __forceinline__ void edit_tile(const EditArgs& a, EditSmem& s) {
    const ExtArgs& e = a.x;
    if (EMIT && a.tile_cnt[blockIdx.x] == 0) return;                  // the count pass found nothing here: no second build
    const u32 Q0 = blockIdx.x * (u32)SRCH_TILE;
    const u32 Qb = Q0 - (Q0 < (u32)SE_BEHIND ? Q0 : (u32)SE_BEHIND);
    const u32 Qe = e.total - Q0 < (u32)SRCH_TILE ? e.total : Q0 + (u32)SRCH_TILE;
    srch_build(e, Qb, Qe, s);
    for (u32 i = threadIdx.x; i < (u32)sizeof(s.O); i += SRCH_T) {
        const u32 l = s.O[i] | 0x20u, sl = (l >> 1) & 7u;
        s.S[i] = (u8)(((u32)(SE_LET >> (8u * sl)) & 0xffu) == l ? sl : SE_OTHER);
    }
    // ---- this thread's candidate ends: one region holding all 32 as candidates is the common case
    const u32 q0 = Q0 + threadIdx.x * 32u;
    const u32 qe = e.total - q0 < 32u ? e.total : q0 + 32u;
    u32 cand = 0;
    int rq = -1;
    if (q0 < e.total) {
        rq = bounded_upper_u32(e.r_off, s.sh[0], s.sh[1], (i64)q0);
        if (a.r_cbeg[rq] <= q0 && e.r_off[rq + 1] >= qe) cand = qe - q0 == 32u ? 0xffffffffu : (1u << (qe - q0)) - 1u;
        else {
            int r = rq;
            for (u32 q = q0; q < qe; ++q) {
                while (e.r_off[r + 1] <= q) ++r;
                cand |= (u32)(q >= a.r_cbeg[r]) << (q - q0);
            }
        }
    }
    __syncthreads();
    // ---- every pattern: both strands in one pass where both are searched (two independent chains)
    u32 cnt = 0, anyhit = 0;
    if (cand) {
        for (int pi = 0; pi < a.n_pat; ++pi) {
            const u32 m = a.plen[pi], span = m + (u32)a.kmax;
            const u32 p0 = q0 + 1u >= e.r_off[rq] + span ? q0 + 1u - span : e.r_off[rq];
            u32 h[2];
            if (a.strands == 3) edit_fwd<2>(a, s, Qb, pi, 0, m, p0, rq, q0, qe, cand, h);
            else { edit_fwd<1>(a, s, Qb, pi, a.strands >> 1, m, p0, rq, q0, qe, cand, h); h[1] = 0; }
            cnt += (u32)(__popc(h[0]) + __popc(h[1]));
            anyhit |= h[0] | h[1];
        }
    }
    if (!EMIT) {
        cnt = __reduce_add_sync(SCCG_FULL_MASK, cnt);
        if (lane_of() == 0) s.red[threadIdx.x >> 5] = cnt;
        __syncthreads();
        if (threadIdx.x == 0) {
            u32 t = 0;
            for (int w = 0; w < SRCH_T / 32; ++w) t += s.red[w];
            a.tile_cnt[blockIdx.x] = t;
        }
        return;
    }
    // ---- emit: this thread's hits start at the tile's offset plus the block scan of the counts; ends in order, then patterns,
    //      then strands.  For each: the anchored DP backward from the end over at most m + k bytes of its region; after j bytes
    //      its score is ed(P, D[end - j, end)).  The least score is d(end) when it is <= k (note 14 of DESIGN.md section 4); the
    //      first j that reaches it gives the largest start.
    u32 tot = 0;
    u32 at = a.tile_off[blockIdx.x] + block_scan_excl(cnt, s.red, &tot);
    int r = rq;
    while (anyhit) {
        const u32 i = (u32)(__ffs((int)anyhit) - 1);
        anyhit &= anyhit - 1u;
        const u32 q = q0 + i;
        while (e.r_off[r + 1] <= q) ++r;
        const u32 back = q + 1u - e.r_off[r];                         // bytes of the region up to the end
        const i64 end = (i64)e.r_start[r] + (i64)back;
        for (int pi = 0; pi < a.n_pat; ++pi) {
            const u32 m = a.plen[pi], span = m + (u32)a.kmax, J = back < span ? back : span;
            const u64 top = 1ull << (m - 1u);
            for (int st = 0; st < 2; ++st) {
                if (!((a.strands >> st) & 1)) continue;
                const u64* pq = a.peq + (size_t)((pi * 2 + st) * 2 + 1) * 8;
                u64 Pv = ~0ull, Mv = 0;
                int sc = (int)m, best = (int)m;
                u32 bj = 0;
                for (u32 j = 1; j <= J; ++j) {
                    edit_step<true>(edit_eq(a, s, pq, pi * 2 + st, m, q + 1u - j - Qb, true), top, Pv, Mv, sc);
                    if (sc < best) { best = sc; bj = j; }
                }
                if (best > a.kmax) continue;
                sccg_edit_hit hh;
                hh.window = (int64_t)a.r_win[r]; hh.start = end - (i64)bj; hh.end = end; hh.pattern = pi; hh.strand = st;
                hh.edits = best; hh.reserved = 0;
                a.hits[at++] = hh;
            }
        }
    }
}

__global__ void __launch_bounds__(SRCH_T, 8) srch_edit_count_k(EditArgs a) {
    __shared__ EditSmem s;
    edit_tile<false>(a, s);
}

__global__ void __launch_bounds__(SRCH_T, 8) srch_edit_emit_k(EditArgs a) {
    __shared__ EditSmem s;
    edit_tile<true>(a, s);
}

static void search_launch(sccg_ctx* c, unsigned ntiles, const EditArgs& sa, bool emit) {
    if (emit) LAUNCH(c, srch_edit_emit_k, dim3(ntiles), dim3(SRCH_T), 0, sa);
    else LAUNCH(c, srch_edit_count_k, dim3(ntiles), dim3(SRCH_T), 0, sa);
}

// sccg_archive_search_edits: the checks of sccg_archive_search, the pattern tables (descriptors and Peq masks) once, then the
// launches (windows of at least minlen - max_edits bytes, cut with maxlen + max_edits - 1 bytes of look-behind)
static int archive_search_edits_impl(sccg_ctx* c, sccg_archive* const* archives, i64 n_archives, const sccg_window* windows, i64 n_windows,
                                     const char* patterns, const int64_t* pattern_off, i64 n_patterns, int max_edits, int strands,
                                     sccg_edit_hit* hits, i64 hits_cap, int64_t* n_hits) {
    i64 minlen = 0, maxlen = 0;
    SCCG_TRY(search_check(c, archives, n_archives, windows, n_windows, patterns, pattern_off, n_patterns, max_edits,
                          "max_edits must be >= 0 and below the shortest pattern's length", strands, hits_cap, n_hits, &minlen, &maxlen));
    if (n_windows == 0) return SCCG_OK;
    const int ns = (strands & 1) + (strands >> 1);
    i64 lim = search_split();
    const i64 hit_lim = 0xffffffffLL / (n_patterns * ns);             // a launch's hits fit 32 bits
    lim = lim < hit_lim ? lim : hit_lim;
    SearchCut cut;
    search_cut(windows, n_windows, minlen - max_edits, 0, maxlen + max_edits - 1, lim, cut);
    // ---- staging: [GatherArgs of every archive | Peq masks | descriptors | lengths] once, then the region table per launch
    const size_t ga_bytes = sizeof(GatherArgs) * (size_t)n_archives;
    const size_t peq_off = align_up(ga_bytes, 16), peq_bytes = sizeof(u64) * (size_t)n_patterns * 32;
    const size_t desc_off = peq_off + peq_bytes, desc_bytes = sizeof(u16) * (size_t)n_patterns * 2 * SRCH_MAXLEN;
    const size_t tab_bytes = align_up(desc_off + desc_bytes + (size_t)n_patterns, 16);
    const size_t reg_bytes = sizeof(u32) * (6 * cut.max_reg + 1);
    SCCG_TRY(ext_staging(c, tab_bytes + reg_bytes));
    u8* h = (u8*)c->h_ext;
    search_stage_archives(c, archives, n_archives, (GatherArgs*)h);
    u64* h_peq = (u64*)(h + peq_off);
    u16* h_desc = (u16*)(h + desc_off);
    u8* h_len = h + desc_off + desc_bytes;
    static const u32 slot_letter[8] = {'a', 'c', 't', 'g', 0, 0, 0, 'n'};
    for (i64 i = 0; i < n_patterns; ++i) {
        const u32 m = (u32)(pattern_off[i + 1] - pattern_off[i]);
        h_len[i] = (u8)m;
        search_stage_desc((const u8*)patterns + pattern_off[i], m, h_desc + i * 2 * SRCH_MAXLEN);
        for (int st = 0; st < 2; ++st) {
            const u16* ds = h_desc + (i * 2 + st) * SRCH_MAXLEN;
            u64* fw = h_peq + (i * 2 + st) * 16;
            for (int sl = 0; sl < 8; ++sl) {
                u64 f = 0, rv = 0;
                for (u32 j = 0; slot_letter[sl] && j < m; ++j)
                    if (srch_match(ds[j], slot_letter[sl])) { f |= 1ull << j; rv |= 1ull << (m - 1u - j); }
                fw[sl] = f; fw[8 + sl] = rv;
            }
        }
    }
    u8* d_tab = nullptr; u32* d_reg = nullptr;
    SCCG_TRY(buf(c, B_SRCH_TAB, tab_bytes, &d_tab));
    SCCG_TRY(buf(c, B_SRCH_REG, 6 * cut.max_reg + 1, &d_reg));
    SCCG_CK(cudaEventRecord(c->ev[4], c->stream));
    SCCG_CK(cudaMemcpyAsync(d_tab, h, tab_bytes, cudaMemcpyHostToDevice, c->stream));
    EditArgs sa;
    sa.x.g = (const GatherArgs*)d_tab; sa.x.out = nullptr; sa.x.lane_min = ext_lane_min(); sa.x.err = nullptr;
    sa.peq = (const u64*)(d_tab + peq_off); sa.desc = (const u16*)(d_tab + desc_off); sa.plen = d_tab + desc_off + desc_bytes;
    sa.n_pat = (int)n_patterns; sa.strands = strands; sa.kmax = max_edits;
    return search_launches(c, cut, (u32*)(h + tab_bytes), d_reg, sa, hits, hits_cap, n_hits);
}

}  // namespace sccg
