// Pattern search over open archives (sccg_archive_search, include/sccg.h): every occurrence of up to 1024 patterns of 1 to 64
// bytes, with up to max_mismatches Hamming mismatches, on either strand, inside windows of D of any open archive.
//
//   image            -> the concatenation of the windows: the image sccg_archive_extract would produce for the queries
//                       (archive, start, end, 0).  The host cuts it into launches whose image fits 32-bit offsets (and whose
//                       hit count fits 32 bits); a window that does not fit is cut into pieces that overlap by the look-ahead
//   srch_count_k     -> one CTA per 4096 candidate start positions: the tile and maxlen - 1 bytes of look-ahead are built in
//                       shared memory with the piece helpers of ext_gather_k, then matched with A/C/G/T/N bit-planes; hits of
//                       each tile
//   scan             -> scan_exclusive_u32 of the tile counts: each tile's first hit, and the launch total (one round trip)
//   srch_emit_k      -> the tiles that hold hits built again; the positions that hold a hit are re-evaluated one by one in
//                       (pattern, strand) order and written as sccg_hit, in (window, pos, pattern, strand) order
#pragma once
#include "sccg_extract.cuh"
#include "sccg_scan.cuh"

namespace sccg {

static const int SRCH_T = EXT_T;                                // 128 threads, 32 candidate positions each
static const int SRCH_TILE = SRCH_T * 32;                       // candidate positions per CTA
static const int SRCH_MAXLEN = 64;
static const int SRCH_BYTES = SRCH_TILE + 64;                   // the tile, the look-ahead and the last thread's 96-byte window
static const int SRCH_WORDS = SRCH_BYTES / 32;                  // 32-position words of each bit-plane
static const int SRCH_MAXPAT = 1024;
// candidate positions per launch; SCCG_SEARCH_SPLIT overrides it (tests force many launches)
static const i64 SRCH_SPLIT = 1ll << 30;

// pattern byte descriptors (host-made; desc[(i * 2 + strand) * 64 + j]): bits 0-3 the bases of A, C, G, T it matches, bit 4
// 'N' / 'n', bit 5 the byte in bits 8-15 itself (bit 6: either case of that letter)
static const u32 SD_N = 16u, SD_OTHER = 32u, SD_FOLD = 64u;

struct SrchArgs {
    ExtArgs x;               // the launch's image: r_start, r_off, r_tag (archive << 1), n_reg, total (image bytes), g, lane_min
    const u32* r_win;        // window index of region i (a window cut over launches makes several regions)
    const u32* r_cend;       // candidate positions of region i: image [r_off[i], r_cend[i]); bytes past it are look-ahead
    const u32* r_cbeg;       // (= r_off: no look-behind; the edit-distance engine's table has it)
    const u16* desc;         // pattern byte descriptors, both strands (the minus strand: the reverse complement)
    const u8* plen;
    int n_pat, strands, kmax;
    u32 maxlen;
    u32* tile_cnt;           // count pass: hits of each tile
    const u32* tile_off;     // emit pass: their exclusive scan
    sccg_hit* hits;          // emit pass: the launch's hits
};

struct SrchSmem {
    __align__(16) u8 O[SRCH_BYTES];       // image bytes [Q0, Q0 + SRCH_BYTES), zero past the tile's last byte
    u8 room[SRCH_TILE];                   // bytes of its window from each candidate on (capped at 64; 0: not a candidate)
    u32 pl[5][SRCH_WORDS];                // A, C, G, T, N bit-planes (case-blind)
    u32 red[33];
    int sh[2];
    __align__(8) u64 bar;
};

// one bit per byte of x (already | 0x20) equal to the byte repeated in rep: byte i -> bit i
__device__ __forceinline__ u32 srch_eq4(u32 x, u32 rep) {
    const u32 y = x ^ rep;
    const u32 z = ~(((y & 0x7f7f7f7fu) + 0x7f7f7f7fu) | y | 0x7f7f7f7fu);     // 0x80 exactly in the zero bytes of y
    return (z * 0x00204081u) >> 28;                                              // bits 7, 15, 23, 31 -> 28 .. 31
}

// the match rule of one pattern byte descriptor against one byte of D
__host__ __device__ __forceinline__ bool srch_match(u32 d, u32 b) {
    const u32 l = b | 0x20u;
    if (((d & 1u) && l == 'a') || ((d & 2u) && l == 'c') || ((d & 4u) && l == 'g') || ((d & 8u) && l == 't') || ((d & SD_N) && l == 'n')) return true;
    if (!(d & SD_OTHER)) return false;
    const u32 x = d >> 8;
    return (d & SD_FOLD) ? l == (x | 0x20u) : b == x;
}

// image bytes [Q0, Qe) -> s.O: every piece that reaches into them, without the lowercase pass (the match is case-blind; the
// lane path's ext_sym still lowers, which changes nothing here).  Tiles of lane_min pieces or more: a thread per piece, as in
// ext_gather_k, searching each archive's whole tables.  Others: warp w builds the pieces that meet the w-th quarter of the
// bytes, clipped to it, so a tile made of one long piece keeps every warp busy.  Q0 is a multiple of 16; s.O is zero past
// the last byte.  (S: SrchSmem, or the shared memory of the edit-distance engine, sccg_search_edit.cuh)
template <class S>
__device__ __forceinline__ void srch_build(const ExtArgs& e, u32 Q0, u32 Qe, S& s) {
    const int warp = (int)(threadIdx.x >> 5), lane = lane_of();
    if (threadIdx.x == 0) mbar_init(&s.bar, 1u);
    if (warp < 2) {
        const int r = warp_upper_u32(e.r_off, e.n_reg, warp ? (i64)Qe - 1 : (i64)Q0);
        if (lane == 0) s.sh[warp] = r;
    }
    __syncthreads();
    const int r0 = s.sh[0], r1 = s.sh[1];
    if ((u32)(r1 - r0 + 1) >= e.lane_min) {
        for (int r = r0 + (int)threadIdx.x; r <= r1; r += SRCH_T) {
            i64 b0; u32 q, tag;
            const u32 n = ext_piece(e, r, Q0, Qe, &b0, &q, &tag);
            if (!n) continue;
            const GatherArgs& g = e.g[tag >> 1];
            ext_piece_lane(g, ExtWin{0, g.nseg - 1, 0, g.n_k - 1, 0, g.l_k - 1}, b0, n, false, nullptr, s.O + (q - Q0));
        }
    } else {
        const u32 nb = Qe - Q0;
        const u32 W0 = Q0 + (warp ? ((nb * (u32)warp / 4u) & ~15u) : 0u);
        const u32 We = warp == SRCH_T / 32 - 1 ? Qe : Q0 + ((nb * (u32)(warp + 1) / 4u) & ~15u);
        for (int r = r0; r <= r1 && W0 < We; ++r) {
            i64 b0; u32 q, tag;
            const u32 n = ext_piece(e, r, W0, We, &b0, &q, &tag);
            if (n) ext_piece_warp(e.g[tag >> 1], b0, b0 + n, s.O + (q - Q0), &s.bar);
        }
    }
    __syncthreads();                                                  // every copy has been issued ...
    if (threadIdx.x == 0) mbar_arrive(&s.bar);
    mbar_wait(&s.bar, 0u);                                            // ... and has landed
    for (u32 i = Qe - Q0 + threadIdx.x; i < (u32)sizeof(s.O); i += SRCH_T) s.O[i] = 0;
    __syncthreads();
}

// count (EMIT = false) or emit pass of one tile: candidate positions [Q0, Q0 + 4096) of the launch's image
template <bool EMIT>
__device__ __forceinline__ void srch_tile(const SrchArgs& a, SrchSmem& s) {
    const ExtArgs& e = a.x;
    if (EMIT && a.tile_cnt[blockIdx.x] == 0) return;                  // the count pass found nothing here: no second build
    const u32 Q0 = blockIdx.x * (u32)SRCH_TILE;
    const u32 Qe = e.total - Q0 < (u32)SRCH_TILE + a.maxlen - 1u ? e.total : Q0 + (u32)SRCH_TILE + a.maxlen - 1u;
    srch_build(e, Q0, Qe, s);
    const u32 P0 = threadIdx.x * 32u;
    const u32 q0 = Q0 + P0;
    // ---- bit-planes of this thread's 32 bytes; threads 0, 1 also make the two words past the tile
    for (u32 wd = threadIdx.x; wd < (u32)SRCH_WORDS; wd += SRCH_T) {
        u32 pa = 0, pc = 0, pg = 0, pt = 0, pn = 0;
        const u32* w4 = reinterpret_cast<const u32*>(s.O + wd * 32u);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const u32 x = w4[k] | 0x20202020u;
            pa |= srch_eq4(x, 0x61616161u) << (4 * k);
            pc |= srch_eq4(x, 0x63636363u) << (4 * k);
            pg |= srch_eq4(x, 0x67676767u) << (4 * k);
            pt |= srch_eq4(x, 0x74747474u) << (4 * k);
            pn |= srch_eq4(x, 0x6e6e6e6eu) << (4 * k);
        }
        s.pl[0][wd] = pa; s.pl[1][wd] = pc; s.pl[2][wd] = pg; s.pl[3][wd] = pt; s.pl[4][wd] = pn;
    }
    // ---- the room of each candidate: one window holding all 32 positions and 64 bytes past the last is the common case
    bool full = false, any_cand = q0 < e.total;
    int rq = -1;
    if (any_cand) {
        rq = bounded_upper_u32(e.r_off, s.sh[0], s.sh[1], (i64)q0);
        full = a.r_cend[rq] >= q0 + 32u && e.r_off[rq + 1] >= q0 + 31u + (u32)SRCH_MAXLEN;
        if (!full) {
            int r = rq;
            for (u32 i = 0; i < 32u; ++i) {
                const u32 q = q0 + i;
                u32 rm = 0;
                if (q < e.total) {
                    while (e.r_off[r + 1] <= q) ++r;
                    if (q < a.r_cend[r]) { rm = e.r_off[r + 1] - q; rm = rm < (u32)SRCH_MAXLEN ? rm : (u32)SRCH_MAXLEN; }
                }
                s.room[P0 + i] = (u8)rm;
            }
        }
    }
    __syncthreads();
    u32 A[3], Cp[3], G[3], T[3], N[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const u32 wd = threadIdx.x + (u32)k;
        A[k] = s.pl[0][wd]; Cp[k] = s.pl[1][wd]; G[k] = s.pl[2][wd]; T[k] = s.pl[3][wd]; N[k] = s.pl[4][wd];
    }
    // ---- every pattern and strand: positions with at most kmax mismatches (bit-sliced counters; a position is dead once its
    //      count reaches kmax + 1)
    const u32 kp1 = (u32)a.kmax + 1u;
    const int nb = 32 - __clz((int)kp1);                              // bits of kmax + 1 (<= 7)
    u32 cnt = 0, anyhit = 0, vlen = 0xffffffffu, valid = any_cand && full ? 0xffffffffu : 0u;
    if (any_cand) {
        for (int pi = 0; pi < a.n_pat; ++pi) {
            const u32 len = a.plen[pi];
            if (!full && len != vlen) {
                valid = 0;
                for (u32 i = 0; i < 32u; ++i) valid |= (u32)(s.room[P0 + i] >= len) << i;
                vlen = len;
            }
            if (!valid) continue;
            for (int st = 0; st < 2; ++st) {
                if (!((a.strands >> st) & 1)) continue;
                const u16* ds = a.desc + ((size_t)pi * 2 + st) * SRCH_MAXLEN;
                u32 dead = ~valid, c[7] = {0, 0, 0, 0, 0, 0, 0};
                for (u32 j = 0; j < len; ++j) {
                    const u32 d = ds[j];
                    const bool hw = j >= 32u;
                    const u32 sa = 0u - (d & 1u), sc = 0u - ((d >> 1) & 1u), sg = 0u - ((d >> 2) & 1u), stt = 0u - ((d >> 3) & 1u), sn = 0u - ((d >> 4) & 1u);
                    const u32 lo = ((hw ? A[1] : A[0]) & sa) | ((hw ? Cp[1] : Cp[0]) & sc) | ((hw ? G[1] : G[0]) & sg) | ((hw ? T[1] : T[0]) & stt) | ((hw ? N[1] : N[0]) & sn);
                    const u32 hi = ((hw ? A[2] : A[1]) & sa) | ((hw ? Cp[2] : Cp[1]) & sc) | ((hw ? G[2] : G[1]) & sg) | ((hw ? T[2] : T[1]) & stt) | ((hw ? N[2] : N[1]) & sn);
                    u32 m = __funnelshift_r(lo, hi, j & 31u);
                    if (d & SD_OTHER) {                               // a byte other than A, C, G, T, N of the pattern: compared as is
                        const u32 x = d >> 8;
                        for (u32 i = 0; i < 32u; ++i) {
                            const u32 b = s.O[P0 + j + i];
                            m |= (u32)((d & SD_FOLD) ? (b | 0x20u) == (x | 0x20u) : b == x) << i;
                        }
                    }
                    u32 carry = ~m & ~dead;
#pragma unroll
                    for (int b = 0; b < 7; ++b) if (b < nb) { const u32 t = c[b] & carry; c[b] ^= carry; carry = t; }
                    u32 eq = 0xffffffffu;
#pragma unroll
                    for (int b = 0; b < 7; ++b) if (b < nb) eq &= ((kp1 >> b) & 1u) ? c[b] : ~c[b];
                    dead |= eq;
                    if (dead == 0xffffffffu) break;
                }
                cnt += (u32)__popc(~dead);
                anyhit |= ~dead;
            }
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
    // ---- emit: this thread's hits start at the tile's offset plus the block scan of the counts; positions in order, then
    //      patterns, then strands
    u32 tot = 0;
    u32 at = a.tile_off[blockIdx.x] + block_scan_excl(cnt, s.red, &tot);
    int r = rq;
    while (anyhit) {
        const u32 i = (u32)(__ffs((int)anyhit) - 1);
        anyhit &= anyhit - 1u;
        const u32 q = q0 + i;
        while (e.r_off[r + 1] <= q) ++r;
        const u32 rm = full ? (u32)SRCH_MAXLEN : s.room[P0 + i];
        const i64 pos = (i64)e.r_start[r] + (i64)(q - e.r_off[r]);
        for (int pi = 0; pi < a.n_pat; ++pi) {
            const u32 len = a.plen[pi];
            if (rm < len) continue;
            for (int st = 0; st < 2; ++st) {
                if (!((a.strands >> st) & 1)) continue;
                const u16* ds = a.desc + ((size_t)pi * 2 + st) * SRCH_MAXLEN;
                int mm = 0;
                for (u32 j = 0; j < len && mm <= a.kmax; ++j) mm += !srch_match(ds[j], s.O[P0 + i + j]);
                if (mm > a.kmax) continue;
                sccg_hit h;
                h.window = (int64_t)a.r_win[r]; h.pos = pos; h.pattern = pi; h.strand = st; h.mismatches = mm; h.reserved = 0;
                a.hits[at++] = h;
            }
        }
    }
}

__global__ void __launch_bounds__(SRCH_T, 8) srch_count_k(SrchArgs a) {
    __shared__ SrchSmem s;
    srch_tile<false>(a, s);
}

__global__ void __launch_bounds__(SRCH_T, 8) srch_emit_k(SrchArgs a) {
    __shared__ SrchSmem s;
    srch_tile<true>(a, s);
}

static i64 search_split() {
    i64 v = SRCH_SPLIT;
    if (const char* s = getenv("SCCG_SEARCH_SPLIT")) { const long long x = atoll(s); if (x >= 1) v = x; }
    return v < (1ll << 31) - 4 * SRCH_TILE ? v : (1ll << 31) - 4 * SRCH_TILE;
}

// the byte descriptor of pattern byte p (SD_*): after upper-casing, A/C/G/T match themselves; an IUPAC code matches the bases of
// its set and itself; every other byte matches only itself (either case of a letter)
static u16 search_desc(u8 p) {
    const u32 P = (p >= 'a' && p <= 'z') ? p - 32u : p;
    static const char codes[] = "ACGTRYSWKMBDHVN";
    static const u8 sets[] = {1, 2, 4, 8, 1 | 4, 2 | 8, 2 | 4, 1 | 8, 4 | 8, 1 | 2, 2 | 4 | 8, 1 | 4 | 8, 1 | 2 | 8, 1 | 2 | 4, 15};
    for (int i = 0; i < 15; ++i) {
        if ((u32)codes[i] != P) continue;
        if (i < 4) return sets[i];
        if (P == 'N') return (u16)(15u | SD_N);
        return (u16)(sets[i] | SD_OTHER | SD_FOLD | (P << 8));
    }
    return (u16)(SD_OTHER | ((P >= 'A' && P <= 'Z') ? SD_FOLD : 0u) | (P << 8));
}

// the argument checks of sccg_archive_search and sccg_archive_search_edits (include/sccg.h, in that order; k_why: the message
// for k out of range) -> the shortest and the longest pattern
static int search_check(sccg_ctx* c, sccg_archive* const* archives, i64 n_archives, const sccg_window* windows, i64 n_windows,
                        const char* patterns, const int64_t* pattern_off, i64 n_patterns, int k, const char* k_why, int strands,
                        i64 hits_cap, int64_t* n_hits, i64* minlen_out, i64* maxlen_out) {
    if (!n_hits || n_archives < 0 || n_windows < 0 || n_patterns < 0 || hits_cap < 0 || (n_archives > 0 && !archives) ||
        (n_windows > 0 && !windows) || (n_patterns > 0 && (!pattern_off || !patterns)))
        return set_error(SCCG_E_ARG, "null argument");
    *n_hits = 0;
    if (n_archives >= 0x80000000LL || n_windows >= 0x80000000LL || n_patterns >= 0x80000000LL)
        return set_error(SCCG_E_ARG, "at most 2^31 - 1 archives, windows and patterns per call");
    // ---- patterns
    if (n_patterns < 1 || n_patterns > SRCH_MAXPAT) return set_error(SCCG_E_ARG, "a search takes 1 to 1024 patterns");
    if (pattern_off[0] != 0) return set_error(SCCG_E_ARG, "pattern_off must start at 0");
    i64 minlen = SRCH_MAXLEN, maxlen = 1;
    for (i64 i = 0; i < n_patterns; ++i) {
        const i64 len = pattern_off[i + 1] - pattern_off[i];
        if (len < 1 || len > SRCH_MAXLEN) return set_error(SCCG_E_ARG, "every pattern must be 1 to 64 bytes long (pattern_off non-decreasing from 0)");
        minlen = len < minlen ? len : minlen;
        maxlen = len > maxlen ? len : maxlen;
    }
    if (k < 0 || k >= minlen) return set_error(SCCG_E_ARG, k_why);
    if (strands < 1 || strands > 3) return set_error(SCCG_E_ARG, "strands must be 1 (forward), 2 (reverse complement) or 3 (both)");
    // ---- windows: the query checks of sccg_archive_extract
    int first = ARCHIVE_QUERY_OK;
    for (i64 i = 0; i < n_windows && first > 0; ++i) {
        const int bad = archive_query_fault(c, archives, n_archives, windows[i].archive, windows[i].start, windows[i].end);
        if (bad < first) first = bad;
    }
    if (first < ARCHIVE_QUERY_OK) return set_error(SCCG_E_ARG, archive_query_why[first]);
    *minlen_out = minlen; *maxlen_out = maxlen;
    return SCCG_OK;
}

// the regions of a search's launches: the windows of at least min_win bytes, cut into pieces of at most `lim` candidate positions
// per launch.  Region i is D[rs[i], rs[i] + rlen[i]) of archive rarch[i]; its candidates are bytes [rlo[i], rhi[i]) of it; the
// bytes before them (at most `behind`) and past them (at most `ahead`) are those of its window that a cut left out of the piece.
struct SearchCut {
    std::vector<u32> rs, rlen, rlo, rhi, rwin, rarch;
    std::vector<size_t> launch_end;                                   // regions [launch_end[k - 1], launch_end[k]) make launch k
    size_t max_reg = 0;
};

static void search_cut(const sccg_window* windows, i64 n_windows, i64 min_win, i64 ahead, i64 behind, i64 lim, SearchCut& o) {
    i64 left = lim;
    for (i64 w = 0; w < n_windows; ++w) {
        const sccg_window& W = windows[w];
        if (W.end - W.start < min_win) continue;                        // no pattern fits
        for (i64 s = W.start; s < W.end;) {
            const i64 take = W.end - s < left ? W.end - s : left;
            const i64 ce = s + take, be = ce + ahead < W.end ? ce + ahead : W.end, bs = s - behind > W.start ? s - behind : W.start;
            o.rs.push_back((u32)bs); o.rlen.push_back((u32)(be - bs)); o.rlo.push_back((u32)(s - bs)); o.rhi.push_back((u32)(ce - bs));
            o.rwin.push_back((u32)w); o.rarch.push_back((u32)W.archive);
            left -= take;
            s = ce;
            if (left == 0) { o.launch_end.push_back(o.rs.size()); left = lim; }
        }
    }
    if (o.launch_end.empty() || o.launch_end.back() != o.rs.size()) o.launch_end.push_back(o.rs.size());
    for (size_t k = 0, b = 0; k < o.launch_end.size(); b = o.launch_end[k++]) o.max_reg = o.launch_end[k] - b > o.max_reg ? o.launch_end[k] - b : o.max_reg;
}

static void search_launch(sccg_ctx* c, unsigned ntiles, const SrchArgs& sa, bool emit) {
    if (emit) LAUNCH(c, srch_emit_k, dim3(ntiles), dim3(SRCH_T), 0, sa);
    else LAUNCH(c, srch_count_k, dim3(ntiles), dim3(SRCH_T), 0, sa);
}

// the launches of either engine (Args: SrchArgs or EditArgs, with their search_launch): per launch one copy of the region table
// [r_start | r_off | r_tag | r_win | r_cend | r_cbeg] from h_reg to d_reg, the count pass, the scan and one round trip for the
// total, and (while the hits fit hits_cap) the emit pass and one copy of its hits.  The table copy of the call is timed from
// c->ev[4] on.
template <class Args, class Hit>
static int search_launches(sccg_ctx* c, const SearchCut& cut, u32* h_reg, u32* d_reg, Args& sa, Hit* hits, i64 hits_cap, int64_t* n_hits) {
    float h2d = 0.f, gat = 0.f, ker = 0.f, d2h = 0.f, ms = 0.f;
    u32* h_total = (u32*)((char*)c->h_pinned + 8192);
    u32* d_tile = nullptr;
    i64 found = 0;
    bool over = false;
    for (size_t k = 0, b = 0; k < cut.launch_end.size(); b = cut.launch_end[k++]) {
        const size_t n = cut.launch_end[k] - b;
        if (n == 0) continue;
        if (k > 0) { SCCG_CK(cudaEventRecord(c->ev[4], c->stream)); }
        u32* r_start = h_reg; u32* r_off = r_start + n; u32* r_tag = r_off + n + 1; u32* r_win = r_tag + n; u32* r_cend = r_win + n;
        u32* r_cbeg = r_cend + n;
        u32 off = 0;
        for (size_t i = 0; i < n; ++i) {
            r_start[i] = cut.rs[b + i]; r_off[i] = off; r_tag[i] = cut.rarch[b + i] << 1; r_win[i] = cut.rwin[b + i];
            r_cend[i] = off + cut.rhi[b + i]; r_cbeg[i] = off + cut.rlo[b + i];
            off += cut.rlen[b + i];
        }
        r_off[n] = off;
        const unsigned ntiles = div_up(off, SRCH_TILE);
        SCCG_TRY(buf(c, B_SRCH_TILE, 2 * (size_t)ntiles + 1, &d_tile));
        SCCG_CK(cudaMemcpyAsync(d_reg, h_reg, sizeof(u32) * (6 * n + 1), cudaMemcpyHostToDevice, c->stream));
        SCCG_CK(cudaEventRecord(c->ev[5], c->stream));
        sa.x.r_start = d_reg; sa.x.r_off = d_reg + n; sa.x.r_tag = d_reg + 2 * n + 1; sa.r_win = d_reg + 3 * n + 1; sa.r_cend = d_reg + 4 * n + 1;
        sa.r_cbeg = d_reg + 5 * n + 1;
        sa.x.n_reg = (int)n; sa.x.total = off;
        sa.tile_cnt = d_tile; sa.tile_off = d_tile + ntiles; sa.hits = nullptr;
        SCCG_CK(cudaEventRecord(c->ev[3], c->stream));
        search_launch(c, ntiles, sa, false);
        SCCG_CK(cudaEventRecord(c->ev[2], c->stream));
        SCCG_TRY(scan_exclusive_u32(c, d_tile, d_tile + ntiles, (i64)ntiles, d_tile + 2 * ntiles));
        SCCG_CK(cudaEventRecord(c->ev[1], c->stream));
        SCCG_CK(cudaMemcpyAsync(h_total, d_tile + 2 * ntiles, sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaStreamSynchronize(c->stream));
        cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]); h2d += ms;
        cudaEventElapsedTime(&ms, c->ev[3], c->ev[2]); gat += ms;
        cudaEventElapsedTime(&ms, c->ev[3], c->ev[1]); ker += ms;
        const i64 t = (i64)*h_total;
        found += t;
        if (!hits || over || t == 0) continue;
        if (found > hits_cap) { over = true; continue; }                  // the remaining launches are only counted
        Hit* d_hits = nullptr;
        SCCG_TRY(buf(c, B_SRCH_HITS, (size_t)t, &d_hits));
        sa.hits = d_hits;
        SCCG_CK(cudaEventRecord(c->ev[3], c->stream));
        search_launch(c, ntiles, sa, true);
        SCCG_CK(cudaEventRecord(c->ev[2], c->stream));
        SCCG_CK(cudaMemcpyAsync(hits + (found - t), d_hits, sizeof(Hit) * (size_t)t, cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaEventRecord(c->ev[7], c->stream));
        SCCG_CK(cudaStreamSynchronize(c->stream));
        cudaEventElapsedTime(&ms, c->ev[3], c->ev[2]); gat += ms; ker += ms;
        cudaEventElapsedTime(&ms, c->ev[2], c->ev[7]); d2h += ms;
    }
    c->prof.h2d_ms = h2d; c->prof.gather_ms = gat; c->prof.kernels_ms = ker; c->prof.d2h_ms = d2h;
    *n_hits = found;
    if (over) return set_error(SCCG_E_ARG, "hit buffer too small (required count returned in *n_hits)");
    return SCCG_OK;
}

// the GatherArgs of every archive a window may name (a stale or foreign one is named by no window: zeros)
static void search_stage_archives(const sccg_ctx* c, sccg_archive* const* archives, i64 n_archives, GatherArgs* h_g) {
    for (i64 k = 0; k < n_archives; ++k) {
        const sccg_archive* a = archives[k];
        if (a && a->ctx == c && a->gen == c->res_gen) h_g[k] = a->g;
        else memset(&h_g[k], 0, sizeof(GatherArgs));
    }
}

// the byte descriptors of pattern i (len bytes at p), both strands (the minus strand: the reverse complement), zero past len
static void search_stage_desc(const u8* p, i64 len, u16* d) {
    for (i64 j = 0; j < SRCH_MAXLEN; ++j) {
        d[j] = j < len ? search_desc(p[j]) : 0;
        d[SRCH_MAXLEN + j] = j < len ? search_desc(comp_byte(p[len - 1 - j])) : 0;
    }
}

// sccg_archive_search: argument checks, the pattern tables once, then the launches (windows cut with maxlen - 1 bytes of
// look-ahead)
static int archive_search_impl(sccg_ctx* c, sccg_archive* const* archives, i64 n_archives, const sccg_window* windows, i64 n_windows,
                               const char* patterns, const int64_t* pattern_off, i64 n_patterns, int max_mismatches, int strands,
                               sccg_hit* hits, i64 hits_cap, int64_t* n_hits) {
    i64 minlen = 0, maxlen = 0;
    SCCG_TRY(search_check(c, archives, n_archives, windows, n_windows, patterns, pattern_off, n_patterns, max_mismatches,
                          "max_mismatches must be >= 0 and below the shortest pattern's length", strands, hits_cap, n_hits, &minlen, &maxlen));
    if (n_windows == 0) return SCCG_OK;
    const int ns = (strands & 1) + (strands >> 1);
    i64 lim = search_split();
    const i64 hit_lim = 0xffffffffLL / (n_patterns * ns);             // a launch's hits fit 32 bits
    lim = lim < hit_lim ? lim : hit_lim;
    SearchCut cut;
    search_cut(windows, n_windows, minlen, maxlen - 1, 0, lim, cut);
    // ---- staging: [GatherArgs of every archive | descriptors | lengths] once, then the region table per launch
    const size_t ga_bytes = sizeof(GatherArgs) * (size_t)n_archives;
    const size_t desc_off = align_up(ga_bytes, 16), desc_bytes = sizeof(u16) * (size_t)n_patterns * 2 * SRCH_MAXLEN;
    const size_t tab_bytes = align_up(desc_off + desc_bytes + (size_t)n_patterns, 16);
    const size_t reg_bytes = sizeof(u32) * (6 * cut.max_reg + 1);
    SCCG_TRY(ext_staging(c, tab_bytes + reg_bytes));
    u8* h = (u8*)c->h_ext;
    search_stage_archives(c, archives, n_archives, (GatherArgs*)h);
    u16* h_desc = (u16*)(h + desc_off);
    u8* h_len = h + desc_off + desc_bytes;
    for (i64 i = 0; i < n_patterns; ++i) {
        h_len[i] = (u8)(pattern_off[i + 1] - pattern_off[i]);
        search_stage_desc((const u8*)patterns + pattern_off[i], h_len[i], h_desc + i * 2 * SRCH_MAXLEN);
    }
    u8* d_tab = nullptr; u32* d_reg = nullptr;
    SCCG_TRY(buf(c, B_SRCH_TAB, tab_bytes, &d_tab));
    SCCG_TRY(buf(c, B_SRCH_REG, 6 * cut.max_reg + 1, &d_reg));
    SCCG_CK(cudaEventRecord(c->ev[4], c->stream));
    SCCG_CK(cudaMemcpyAsync(d_tab, h, tab_bytes, cudaMemcpyHostToDevice, c->stream));
    SrchArgs sa;
    sa.x.g = (const GatherArgs*)d_tab; sa.x.out = nullptr; sa.x.lane_min = ext_lane_min(); sa.x.err = nullptr;
    sa.desc = (const u16*)(d_tab + desc_off); sa.plen = d_tab + desc_off + desc_bytes;
    sa.n_pat = (int)n_patterns; sa.strands = strands; sa.kmax = max_mismatches; sa.maxlen = (u32)maxlen;
    return search_launches(c, cut, (u32*)(h + tab_bytes), d_reg, sa, hits, hits_cap, n_hits);
}

}  // namespace sccg
