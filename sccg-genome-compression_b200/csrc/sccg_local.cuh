// Local (segment-aligned) match-and-encode: one warp per 1000-symbol segment pair.
//   reference: match_sequences compression.cpp:36-179 called per segment from the driver :395-474.
//
// Per segment the warp
//   1. stages r_i and t_i (upper-cased on the fly, :369-370) in shared memory with coalesced 8-byte
//      loads and builds the diagonal-0 mismatch bitmap in the same pass;
//   2. takes the exact fast path when t_i == r_i (the single candidate p = 0 of length 1000 cannot
//      be tied, see DESIGN.md), otherwise
//   3. builds the k-mer index of r_i as a chained hash table in shared memory (:41-47; bucket order
//      is irrelevant because candidate selection is evaluated as an order-independent reduction that
//      equals the reference's ascending-p fold incl. its `pn == 0` quirk, :114-130) and
//   4. runs the greedy parse (:64-161) warp-uniformly: cooperative k-mer hash (REDUX), chain walk,
//      32-lane extension with ballot (extend_alignment :27-34); k = 14 first, k' = 10 if no match
//      (:401, :428).
// Output: one packed u32 per match (tpos | p << 10 | l << 20) in a fixed 100-entry slot per segment
// and one u32 of per-segment status; literals are implied by the gaps between matches.
#pragma once
#include "sccg_scan.cuh"

namespace sccg {

#ifndef SCCG_LM_WARPS
#define SCCG_LM_WARPS 4
#endif
static const int LM_WARPS = SCCG_LM_WARPS;    // 4 warps x 6.6 KB per CTA, 8 CTAs = 32 warps per SM (shared memory and registers both full)
static const int LM_CTAS_PER_SM = 32 / LM_WARPS;
static const int LM_HT_BITS = 9;              // 512 chain heads for <= 987 k-mers (false positives die on a 4-byte tag)
static const int LM_HT = 1 << LM_HT_BITS;
static const int LM_SEQ_PAD = 1040;
static const int LM_SLOT = 100;               // max matches per segment: 1000 / k' (k' = 10)
// k-mer hash: h = sum over the k-mer of c_i * 2^(s * (k-1-i)) mod 2^32 with s = ceil(32 / k): symbols older than the
// last ceil(32/s) <= k have left the 32-bit register, so sliding by one symbol is a single multiply-add with the
// incoming symbol (no outgoing term).  Collisions are harmless: every chain entry is verified symbol by symbol.
__host__ __device__ __forceinline__ int lm_hash_shift(int k) { return (32 + k - 1) / k; }

struct LmWarpSmem {
    u8 r[LM_SEQ_PAD];
    u8 t[LM_SEQ_PAD];
    u32 head[LM_HT];       // 0 = empty, else chain entry: (p + 1) | 6 tag bits of the k-mer hash << 10
    u16 next[1024];        // chain: 0 = end, else entry of the next position
    u32 mlist[LM_SLOT + 4];
    u16 mis[32];           // diagonal-hypothesis path: mismatching symbols, ascending, + sentinel
    u16 qv[32];            //   looked-up windows: position | clean << 15
};

// seginfo layout
#define SEGINFO_NMATCH(x) ((x) & 0xffu)
#define SEGINFO_LIT(x) (((x) >> 8) & 0x7ffu)
#define SEGINFO_ALLN(x) (((x) >> 20) & 1u)
#define SEGINFO_BAD(x) (((x) >> 21) & 1u)

__device__ __forceinline__ u32 lm_mix(u32 h) { return h * 0x9E3779B1u; }
__device__ __forceinline__ u32 lm_bucket(u32 hm) { return hm >> (32 - LM_HT_BITS); }
__device__ __forceinline__ u32 lm_tag(u32 hm) { return (hm >> (32 - LM_HT_BITS - 16)) & 0xfc00u; }   // 6 tag bits at bit 10

__device__ __forceinline__ u32 ld_unaligned32(const u8* base, int off) {
    const u32* w = reinterpret_cast<const u32*>(base);
    int q = off >> 2;
    return __funnelshift_r(w[q], w[q + 1], (u32)(off & 3) * 8u);
}

// min(maxl, length of the common prefix of r[p..] and t[j..]); all 32 lanes, uniform arguments
__device__ __forceinline__ int warp_lcp(const u8* r, int p, const u8* t, int j, int maxl) {
    const int lane = lane_of();
    for (int base = 0; base < maxl; base += 128) {
        int o = base + 4 * lane;
        u32 diff = 0xffffffffu;                               // beyond maxl counts as a mismatch at o
        if (o < maxl) diff = ld_unaligned32(r, p + o) ^ ld_unaligned32(t, j + o);
        u32 bal = __ballot_sync(SCCG_FULL_MASK, diff != 0u);
        if (bal) {
            int src = __ffs((int)bal) - 1;
            u32 d = __shfl_sync(SCCG_FULL_MASK, diff, src);
            int l = base + 4 * src + ((__ffs((int)d) - 1) >> 3);
            return l < maxl ? l : maxl;
        }
    }
    return maxl;
}

// Diagonal 0 (p == j, by far the most common candidate): wm[it] bit `lane` is set iff the 8-byte word 32*it+lane of r
// and t differ inside [0, Lmin).  Returns min(Lmin - j, lcp(r[j..], t[j..])); uniform, no shuffles.
__device__ __forceinline__ int diag_lcp(const LmWarpSmem& S, const u32 (&wm)[4], int j, int Lmin) {
    const u64* r64 = reinterpret_cast<const u64*>(S.r);
    const u64* t64 = reinterpret_cast<const u64*>(S.t);
    const int w = j >> 3;
    const int lim = Lmin - j;
    u64 x = (r64[w] ^ t64[w]) >> (8 * (j & 7));                   // symbols j.. of the first word
    if (x) { int l = (__ffsll((long long)x) - 1) >> 3; return l < lim ? l : lim; }
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        u32 m = wm[it];
        int lo = 32 * it;
        if (lo + 31 <= w) m = 0u;
        else if (lo <= w) m &= 0xfffffffeu << (w - lo);           // words > w only
        if (m) {
            int q = lo + __ffs((int)m) - 1;
            u64 y = r64[q] ^ t64[q];
            int l = 8 * q + ((__ffsll((long long)y) - 1) >> 3) - j;
            return l < lim ? l : lim;
        }
    }
    return lim;
}

// Runs of one symbol (the border of an N block, poly-A): every position of such a run of r holds the same k-mer, a bucket with
// hundreds of entries -- a chain the parse would walk entry by entry, with one extension each.  The k-mers of LONG runs are
// kept out of the chains: lm_runs lists the maximal runs of r of at least max(k, 15) symbols (S.mis = first symbol, S.qv = one
// past the last; the diagonal-hypothesis path is done with both arrays when the generic path starts), and a looked-up k-mer
// that is itself a run of one symbol gets those candidates from the list in closed form (lm_fold_runs) and the rest -- runs
// shorter than 15 -- from its chain as usual.  Returns the number of runs, or -1 if there are more than LM_MAX_RUNS (then
// every k-mer goes into the chains and nothing changes).
// 15 symbols because such a run contains an 8-byte aligned word of 8 equal symbols: the test "does this segment have a long
// run at all" is four 8-byte loads and compares per lane, and almost always says no.
// In the listing pass the lanes look at their eight 4-byte words of r; the lane that owns the FIRST word of 4 equal symbols of
// a run measures the run.
static const int LM_MAX_RUNS = 32;
static const int LM_RUN_MIN = 15;
__device__ __forceinline__ int lm_runs(LmWarpSmem& S, int Lr, int k) {
    const int lane = lane_of();
    const u32* r32 = reinterpret_cast<const u32*>(S.r);
    {
        bool cand = false;
#pragma unroll
        for (int it = 0; it < 4; ++it) {
            const u64 x = reinterpret_cast<const u64*>(S.r)[lane + 32 * it];
            cand = cand || (x == ((x << 8) | (x >> 56)) && 8 * (lane + 32 * it) + 8 <= Lr);
        }
        if (!__any_sync(SCCG_FULL_MASK, cand)) return 0;
    }
    const int min_len = k > LM_RUN_MIN ? k : LM_RUN_MIN;
    int n_runs = 0;
    for (int it = 0; it < 8; ++it) {                                             // word q = 32 * it + lane: uniform trip count
        const int q = 32 * it + lane;
        int a = 0, b = 0;
        bool first = false;
        if (4 * q + 4 <= Lr) {
            const u32 x = r32[q];
            if (x == __funnelshift_r(x, x, 8)) {                                 // 4 equal symbols
                const u8 sym = (u8)x;
                first = q == 0 || r32[q - 1] != x;                               // the word before belongs to the same run: not mine
                if (first) {
                    a = 4 * q; while (a > 0 && S.r[a - 1] == sym) --a;           // <= 3 steps (the word before is not all sym)
                    int qq = q + 1;
                    while (4 * qq + 4 <= Lr && r32[qq] == x) ++qq;               // whole words of the run, then <= 3 symbols
                    b = 4 * qq; while (b < Lr && S.r[b] == sym) ++b;
                    first = b - a >= min_len;
                }
            }
        }
        const u32 bal = __ballot_sync(SCCG_FULL_MASK, first);
        if (bal) {
            const int slot = n_runs + __popc(bal & ((1u << lane) - 1u));
            if (first && slot < LM_MAX_RUNS) { S.mis[slot] = (u16)a; S.qv[slot] = (u16)b; }
            n_runs += __popc(bal);
        }
    }
    __syncwarp();
    return n_runs <= LM_MAX_RUNS ? n_runs : -1;
}

// k-mer index of r[0..Lr) (compression.cpp:41-47) as a chained hash table; k-mers inside the n_runs listed runs of one
// symbol are left out (see lm_runs)
__device__ __forceinline__ void lm_build_index(LmWarpSmem& S, int Lr, int k, int n_runs) {
    const int lane = lane_of();
    for (int x = lane; x < LM_HT; x += 32) S.head[x] = 0u;
    __syncwarp();
    int nk = Lr - k + 1;
    if (nk > 0) {
        const u32 mul = 1u << lm_hash_shift(k);
        int chunk = (nk + 31) >> 5;                                              // <= 31 positions per lane
        int p = lane * chunk;
        int p1 = p + chunk < nk ? p + chunk : nk;
        if (p < p1) {
            u32 skip = 0u;                                                       // bit i: the k-mer at p + i lies inside a listed run
            for (int i = 0; i < n_runs; ++i) {
                const int lo = (int)S.mis[i] - p, hi = (int)S.qv[i] - k - p;     // positions lo .. hi of this lane's chunk
                if (hi >= 0 && lo < 32) skip |= (hi >= 31 ? 0xffffffffu : (2u << hi) - 1u) & (lo <= 0 ? 0xffffffffu : ~((1u << lo) - 1u));
            }
            const int p0 = p;
            u32 h = 0u;
            for (int i = 0; i < k - 1; ++i) h = h * mul + S.r[p + i];
            const u8* in = S.r + (k - 1);
            for (; p < p1; ++p) {
                h = h * mul + in[p];                                             // slide: symbol p + k - 1 enters
                if ((skip >> (p - p0)) & 1u) continue;
                u32 hm = lm_mix(h);
                u32 old = atomicExch(&S.head[lm_bucket(hm)], (u32)(p + 1) | lm_tag(hm));
                S.next[p] = (u16)old;
            }
        }
    }
    __syncwarp();
}

// one lane, one candidate: min(maxl, lcp(r[p..], t[j..])) with 8-byte compares (used when a bucket is crowded, H7)
__device__ __forceinline__ int lane_lcp(const u8* r, int p, const u8* t, int j, int maxl) {
    int l = 0;
    while (l < maxl) {
        u32 a0 = ld_unaligned32(r, p + l), b0 = ld_unaligned32(t, j + l);
        if (a0 != b0) { l += (__ffs((int)(a0 ^ b0)) - 1) >> 3; break; }
        u32 a1 = ld_unaligned32(r, p + l + 4), b1 = ld_unaligned32(t, j + l + 4);
        if (a1 != b1) { l += 4 + ((__ffs((int)(a1 ^ b1)) - 1) >> 3); break; }
        l += 8;
    }
    return l < maxl ? l : maxl;
}

__device__ __forceinline__ u32 mad_u32(u32 a, u32 b, u32 c) {
#if defined(__CUDA_ARCH__)
    u32 d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));   // one IMAD (the compiler would emit shift + add for b = 2^s)
    return d;
#else
    return a * b + c;
#endif
}
// r[p..p+k) == t[j..j+k)  (k <= 32, both in shared memory with >= 8 bytes of slack)
__device__ __forceinline__ bool kmer_equal_smem(const u8* r, int p, const u8* t, int j, int k) {
    for (int o = 0; o < k; o += 4) {
        u32 d = ld_unaligned32(r, p + o) ^ ld_unaligned32(t, j + o);
        if (k - o < 4) d &= (1u << (8 * (k - o))) - 1u;
        if (d) return false;
    }
    return true;
}

// running state of the candidate fold (compression.cpp:114-130 as an order-independent reduction):
// longest length; among the longest: how many, is p == 0 among them, and min (|p - e| << 16 | p) over p != 0
struct LmFold { int best_l; int cnt; bool zero_in; u32 best_key; };
__device__ __forceinline__ void lm_fold_one(LmFold& f, int p, int l, int e) {
    if (l > f.best_l) { f.best_l = l; f.cnt = 0; f.zero_in = false; f.best_key = 0xffffffffu; }     // :127-128
    if (l == f.best_l) {                                                                             // :124-126
        ++f.cnt;
        if (p == 0) f.zero_in = true;
        else {
            int d = p - e; if (d < 0) d = -d;
            u32 key = ((u32)d << 16) | (u32)p;
            if (key < f.best_key) f.best_key = key;
        }
    }
}

// Candidates of a looked-up k-mer t[j..j+k) that is a run of one symbol sym (see lm_runs), folded in closed form.  tr = length
// of the run of sym in t from j on (>= k).  In a run [a, b) of sym in r the candidates are p = a .. b - k, with rr = b - p
// symbols of the run ahead of them:
//   rr < tr: the reference leaves the run first, l = rr          rr > tr: the target leaves it first, l = tr
//   rr == tr (p* = b - tr): both leave it together, l = tr + lcp(r[b..], t[j+tr..])
// so if tr > b - a the longest is p = a alone (l = b - a); else p* is the longest if it gets past the run, and if it does not
// every p in [a, p*] ties at l = tr (the tie-break of :124-126 picks the one nearest to e: a clamp).  All lanes, uniform.
__device__ __forceinline__ void lm_fold_runs(LmWarpSmem& S, LmFold& f, int n_runs, u8 sym, int j, int tr, int e, int Lr, int Lt) {
    for (int i = 0; i < n_runs; ++i) {
        const int a = (int)S.mis[i], b = (int)S.qv[i];
        if (S.r[a] != sym) continue;
        if (tr > b - a) { lm_fold_one(f, a, b - a, e); continue; }
        const int ps = b - tr;
        int ext = 0;
        if (b < Lr && j + tr < Lt) ext = warp_lcp(S.r, b, S.t, j + tr, (Lr - b) < (Lt - j - tr) ? (Lr - b) : (Lt - j - tr));
        if (ext > 0) { lm_fold_one(f, ps, tr + ext, e); continue; }
        // a .. ps all reach exactly tr
        if (tr > f.best_l) { f.best_l = tr; f.cnt = 0; f.zero_in = false; f.best_key = 0xffffffffu; }
        if (tr == f.best_l) {
            f.cnt += ps - a + 1;
            if (a == 0) f.zero_in = true;
            const int lo = a > 1 ? a : 1;
            if (lo <= ps) {
                const int pn = e < lo ? lo : (e > ps ? ps : e);
                int d = pn - e; if (d < 0) d = -d;
                const u32 key = ((u32)d << 16) | (u32)pn;
                if (key < f.best_key) f.best_key = key;
            }
        }
    }
}
// length of the run of sym in t from j on (t[j] == sym), capped at Lt - j; all lanes, uniform
__device__ __forceinline__ int lm_run_len_t(const LmWarpSmem& S, u8 sym, int j, int Lt) {
    const int lane = lane_of();
    const u32 pat = (u32)sym * 0x01010101u;
    const int maxl = Lt - j;
    for (int base = 0; base < maxl; base += 128) {
        const int o = base + 4 * lane;
        u32 diff = 0xffffffffu;
        if (o < maxl) diff = ld_unaligned32(S.t, j + o) ^ pat;
        const u32 bal = __ballot_sync(SCCG_FULL_MASK, diff != 0u);
        if (bal) {
            const int src = __ffs((int)bal) - 1;
            const u32 d = __shfl_sync(SCCG_FULL_MASK, diff, src);
            const int l = base + 4 * src + ((__ffs((int)d) - 1) >> 3);
            return l < maxl ? l : maxl;
        }
    }
    return maxl;
}

// the greedy parse of one segment (compression.cpp:64-167); returns the number of matches, stored in S.mlist
__device__ __forceinline__ int lm_parse(LmWarpSmem& S, const u32 (&wm)[4], int Lr, int Lt, int k, u32 powk, int n_runs) {
    const int Lmin = Lr < Lt ? Lr : Lt;
    const int lane = lane_of();
    int j = 0, e = -1, nmatch = 0, misses = 0;
    const u32 mul = 1u << lm_hash_shift(k);
    while (j < Lt - k + 1) {                                                     // :64
#ifndef SCCG_NO_LOOKAHEAD
        if (misses >= 2) {
            // look-ahead after two literal steps in a row: lane x probes position j + x on its own (hash, bucket, chain,
            // full k-mer compare).  Positions before the first one that has a candidate are literal steps (:77-81), so
            // they are skipped 32 at a time; segments without any match (and the literal stretches of divergent ones)
            // cost 1/32 of the lock-step walk.  (Near-identical segments never get here: one miss per substitution.)
            const int jj = j + lane;
            bool hit = false;
            if (jj < Lt - k + 1) {
                u32 h = 0u;
                bool one_sym = n_runs > 0;                                       // (only worth knowing when r has runs at all)
                for (int x = 0; x < k; ++x) { const u8 cx = S.t[jj + x]; h = mad_u32(h, mul, cx); one_sym = one_sym && cx == S.t[jj]; }
                if (one_sym) {                                                   // a run of one symbol occurs in every listed run of that symbol (and maybe in shorter ones: chain)
                    for (int i = 0; i < n_runs; ++i) hit = hit || S.r[S.mis[i]] == S.t[jj];
                }
                const u32 hm = lm_mix(h);
                const u32 qt = lm_tag(hm), t4 = ld_unaligned32(S.t, jj);
                for (u32 c = S.head[lm_bucket(hm)]; c && !hit;) {
                    const int p = (int)(c & 0x3ffu) - 1;
                    if ((c & 0xfc00u) == qt && ld_unaligned32(S.r, p) == t4 && kmer_equal_smem(S.r, p, S.t, jj, k)) hit = true;
                    c = S.next[p];
                }
            }
            const u32 bal = __ballot_sync(SCCG_FULL_MASK, hit);
            if (!bal) { j += 32; continue; }
            j += __ffs((int)bal) - 1;
        }
#endif
        u32 term = lane < k ? (u32)S.t[j + lane] * powk : 0u;
        u32 hm = lm_mix(__reduce_add_sync(SCCG_FULL_MASK, term));
        u32 c = S.head[lm_bucket(hm)];
        const u32 qtag = lm_tag(hm);                                             // already positioned at bit 10
        const u32 tag = ld_unaligned32(S.t, j);
        LmFold f; f.best_l = 0; f.cnt = 0; f.zero_in = false; f.best_key = 0xffffffffu;
        bool diag_folded = false;                                                // the diagonal candidate (p == j) has been folded: crowded buckets take it ahead of its turn
        if (n_runs > 0 && __all_sync(SCCG_FULL_MASK, lane >= k || S.t[j + lane] == S.t[j])) {
            // the looked-up k-mer is a run of one symbol: its candidates inside the listed (long) runs of r come from the list, the
            // chain below only holds those of shorter runs
            const u8 sym = S.t[j];
            lm_fold_runs(S, f, n_runs, sym, j, lm_run_len_t(S, sym, j, Lt), e, Lr, Lt);
            for (int i = 0; i < n_runs; ++i) diag_folded = diag_folded || (j >= (int)S.mis[i] && j + k <= (int)S.qv[i]);   // p == j is one of the listed candidates
        }
        while (c) {                                                              // :114 every candidate of the bucket
            // gather up to 32 chain entries whose first 4 symbols match (hash-chain false positives die here)
            int myp = -1, nb = 0;
            while (c && nb < 32) {
                int p = (int)(c & 0x3ffu) - 1;
                u32 ctag = c & 0xfc00u;
                c = S.next[p];
                if (ctag == qtag && ld_unaligned32(S.r, p) == tag) { if (lane == nb) myp = p; ++nb; }
            }
            if (nb <= 2) {
                // the common case: extend cooperatively, 128 symbols per step (extend_alignment :27-34)
                for (int i = 0; i < nb; ++i) {
                    int p = __shfl_sync(SCCG_FULL_MASK, myp, i);
                    if (p == j) { if (diag_folded) continue; diag_folded = true; }
                    int maxl = (Lr - p) < (Lt - j) ? (Lr - p) : (Lt - j);
                    int l = (p == j) ? diag_lcp(S, wm, j, Lmin) : warp_lcp(S.r, p, S.t, j, maxl);
                    if (l >= k) lm_fold_one(f, p, l, e);
                }
            } else {
                // crowded bucket (low-complexity sequence, the border of an N run): one candidate per lane.  A candidate can
                // only enter the fold if it reaches the best length so far (best_l never shrinks), so the diagonal candidate --
                // usually the longest by far, and free to extend -- is folded first and every other candidate is dropped by one
                // 4-byte compare at the far end of that length unless it really gets there.  (Without this the border segment of
                // the chr1-sized pair's N block, 297 occurrences of N^14, took 117 us and was the last warp of the launch.)
                if (!diag_folded) {
                    diag_folded = true;                                          // (or it is no candidate at all: same thing for the lanes below)
                    if (j < Lmin - k + 1 && kmer_equal_smem(S.r, j, S.t, j, k)) {
                        const int ld = diag_lcp(S, wm, j, Lmin);
                        if (ld >= k) lm_fold_one(f, j, ld, e);
                    }
                }
                int l = 0;
                if (myp >= 0 && myp != j) {
                    int maxl = (Lr - myp) < (Lt - j) ? (Lr - myp) : (Lt - j);
                    const int need = f.best_l;                                   // >= 4 whenever it is set (k >= 10)
                    if (maxl >= need && (need < 4 || ld_unaligned32(S.r, myp + need - 4) == ld_unaligned32(S.t, j + need - 4))) {
                        l = lane_lcp(S.r, myp, S.t, j, maxl);
                        if (l < k) l = 0;
                    }
                }
                int bmax = (int)__reduce_max_sync(SCCG_FULL_MASK, (u32)l);
                if (bmax > 0) {
                    if (bmax > f.best_l) { f.best_l = bmax; f.cnt = 0; f.zero_in = false; f.best_key = 0xffffffffu; }
                    if (bmax == f.best_l) {
                        bool is = l == bmax;
                        f.cnt += __popc(__ballot_sync(SCCG_FULL_MASK, is));
                        if (__any_sync(SCCG_FULL_MASK, is && myp == 0)) f.zero_in = true;
                        u32 key = 0xffffffffu;
                        if (is && myp != 0) { int d = myp - e; if (d < 0) d = -d; key = ((u32)d << 16) | (u32)myp; }
                        key = __reduce_min_sync(SCCG_FULL_MASK, key);
                        if (key < f.best_key) f.best_key = key;
                    }
                }
            }
        }
        if (f.best_l == 0) { ++j; ++misses; continue; }                          // :77-81 literal
        misses = 0;
        // p = 0 survives only when it is the single longest candidate (`pn1 == 0` is "unset", :125)
        int p_sel = (f.cnt == 1 && f.zero_in) ? 0 : (int)(f.best_key & 0xffffu);
        if (lane == 0) S.mlist[nmatch] = (u32)j | ((u32)p_sel << 10) | ((u32)f.best_l << 20);
        ++nmatch;
        e = p_sel + f.best_l - 1;                                                // :149
        j += f.best_l;                                                           // :159
    }
    return nmatch;
}

// ------------------------------------------------------------------------------------------------
// Diagonal-hypothesis parse (the common near-identical segment: a few substitutions, Lr == Lt).
//
// If every k-mer the greedy parse looks up has no occurrence in r other than the one on diagonal 0 (p == j), the parse is
// fully determined by the positions where r and t differ: a window t[j..j+k) without a mismatch matches at p = j and
// extends to the next mismatch (single candidate: no tie, `pn == 0` cannot be displaced, :114-130); a window that
// contains a mismatch has no candidate and yields a literal (:77-81).  With the mismatch positions m_0 < m_1 < ... and the
// mismatch-free intervals [a_i, b_i) = [m_(i-1) + 1, m_i) between them that parse is, in closed form:
//     interval of length >= k : one looked-up window at a_i (clean) -> match (a_i, a_i, b_i - a_i), the index jumps to b_i
//     shorter interval        : every position of it is a looked-up window that contains m_i -> literals
//     every m_i               : a looked-up window that starts with a mismatch -> literal
// (windows must start at j <= L - k, :64).  So the warp works lane-parallel, no serial walk:
//   1. mismatching symbols from the word ballots of the diagonal compare: the warp visits the (usually one or two) differing
//      8-byte words in position order, lanes 0-7 test one symbol of the word each, a ballot gives each mismatch its slot,
//   2. lane i owns interval i: its looked-up windows (<= 32 in total, else the generic path runs) and its match,
//   3. PROOF of the hypothesis.  An occurrence of a looked-up k-mer t[j..j+k) at r[p..p+k) implies that the 8-byte chunk
//      of r at the next multiple of 4, a = ceil4(p), equals the 8 bytes of t at u = j + (a - p), u in {j .. j+3}
//      (u + 8 <= j + k needs k >= 11).  So the <= 4 * 32 chunks t[u..u+8) go into a hash table keyed by content (entry e on
//      lane e % 32: a segment with <= 8 looked-up windows stores one entry per lane) and every lane probes the 250 four-aligned chunks of r (8 per lane, straight from two 16-byte shared-memory loads): 8
//      instructions per chunk and no per-position work at all.  A table entry carries u: a hit with a == u is the
//      diagonal itself (the expected occurrence of a clean window, no occurrence at all for a window with a mismatch) and is
//      ignored by construction (the XOR below is 0); any other hit is checked symbol by symbol, and a real occurrence --
//      a repeat in r, an off-diagonal occurrence of a mutated k-mer -- rejects the hypothesis.
// Rejection falls back to the exact generic path (index + parse), so the result is always the reference's.
// ------------------------------------------------------------------------------------------------
static const int DV_MAX_MISWORDS = 16;        // mismatching 8-byte words (one warp-uniform round each in step 1)
static const int DV_MAX_MIS = 30;             // mismatching symbols (+ sentinel <= 32 intervals, one per lane)
static const int DV_TAB = 1024;               // table slots: S.head and S.next together (4 KiB)

__device__ __forceinline__ u32 dv_hash(u32 lo, u32 hi) { return (lo * 0x9E3779B1u + hi) * 0x85EBCA6Bu; }
// table entry / probe value: hash bits 11..31, bit 10 set (an empty slot is 0), symbol position in bits 0..9
__device__ __forceinline__ u32 dv_slot(u32 e, u32 alt_shift) { return (e >> alt_shift) & (u32)(DV_TAB - 1); }   // alt_shift: 22, or 12 on the retry

// table entry e of the proof: the chunk t[u .. u+8), u = (position of looked-up window e / 4) + e % 4
__device__ __forceinline__ u32 dv_entry(const LmWarpSmem& S, int e) {
    const int u = (int)(S.qv[e >> 2] & 0x3ffu) + (e & 3);
    const u32* t32 = reinterpret_cast<const u32*>(S.t);
    const int w = u >> 2;
    const u32 sh = (u32)(u & 3) * 8u;
    const u32 b0 = t32[w], b1 = t32[w + 1], b2 = t32[w + 2];
    return (dv_hash(__funnelshift_r(b0, b1, sh), __funnelshift_r(b1, b2, sh)) & ~1023u) | 1024u | (u32)u;
}
enum { DV_STORE = 0, DV_CHECK = 1, DV_CLEAR = 2 };
__device__ __forceinline__ void dv_tab_one(u32* tab, u32 x, u32 alt, int op, bool& coll) {
    u32& s = tab[dv_slot(x, alt)];
    if (op == DV_STORE) s = x;
    else if (op == DV_CHECK) coll |= s != x;
    else s = 0u;
}
// one pass over the ne = 4 * nq entries, entry e on lane e % 32.  en0: this lane's entry `lane` (0: none); the later rounds
// (more than 8 looked-up windows) are recomputed.  DV_CHECK returns true if another entry holds one of this lane's slots.
__device__ __forceinline__ bool dv_tab_pass(const LmWarpSmem& S, u32* tab, u32 en0, int ne, u32 alt, int op) {
    bool coll = false;
    if (en0) dv_tab_one(tab, en0, alt, op, coll);
#pragma unroll 1
    for (int e = 32 + lane_of(); e < ne; e += 32) dv_tab_one(tab, dv_entry(S, e), alt, op, coll);
    return coll;
}

// returns the number of matches (written to gmatches, their summed length in covered), or 0 when the hypothesis was
// rejected / not applicable.  tab_clean (in/out): the 4 KiB table region is all zero.
__device__ __forceinline__ int lm_diag_parse(LmWarpSmem& S, const u32 (&wm)[4], int L, int k, bool& tab_clean,
                                             u32* __restrict__ gmatches, int& covered) {
    const int lane = lane_of();
    if (__popc(wm[0]) + __popc(wm[1]) + __popc(wm[2]) + __popc(wm[3]) > DV_MAX_MISWORDS) return 0;
    // ---- 1. mismatching symbols, ascending: bit `lane` of wm[it] is word 32 * it + lane (S.r / S.t hold the upper-cased pair)
    int c = 0;
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        for (u32 m = wm[it]; m; m &= m - 1) {                      // uniform
            const int pos = 8 * (32 * it + __ffs((int)m) - 1) + lane;
            const bool mis = lane < 8 && pos < L && S.r[pos] != S.t[pos];
            const u32 bal = __ballot_sync(SCCG_FULL_MASK, mis);
            const int slot = c + __popc(bal & ((1u << lane) - 1u));
            if (mis && slot < DV_MAX_MIS) S.mis[slot] = (u16)pos;
            c += __popc(bal);
        }
    }
    if (c > DV_MAX_MIS) return 0;
    if (lane == 0) S.mis[c] = (u16)L;                               // sentinel
    __syncwarp();
    // ---- 2. lane i owns the mismatch-free interval [a, b) before mismatch i (i == c: the tail up to L)
    const bool act = lane <= c;
    int a = 0, b = L;
    if (act) { a = lane ? (int)S.mis[lane - 1] + 1 : 0; b = (int)S.mis[lane]; }
    const int len = b - a;
    const bool lng = act && len >= k;
    int nshort = 0;
    if (act && !lng) { const int hi = b < L - k + 1 ? b : L - k + 1; nshort = hi > a ? hi - a : 0; }
    const int qmis = (act && lane < c && b <= L - k) ? 1 : 0;       // the window that starts at the mismatch itself
    const u32 pk = (u32)((lng ? 1 : nshort) + qmis) | (lng ? 0x10000u : 0u);
    const u32 incl2 = warp_scan_incl(pk);
    const u32 tot2 = __shfl_sync(SCCG_FULL_MASK, incl2, 31);
    const int nq = (int)(tot2 & 0xffffu), nmatch = (int)(tot2 >> 16);
    if (nq > 32 || nmatch == 0) return 0;
    {
        u32 qo = (incl2 - pk) & 0xffffu;
        if (lng) {
            S.qv[qo++] = (u16)(a | 0x8000);
            gmatches[(incl2 - pk) >> 16] = (u32)a | ((u32)a << 10) | ((u32)len << 20);
        } else {
            for (int x = 0; x < nshort; ++x) S.qv[qo++] = (u16)(a + x);
        }
        if (qmis) S.qv[qo] = (u16)b;
    }
    covered = (int)__reduce_add_sync(SCCG_FULL_MASK, lng ? (u32)len : 0u);
    u32* tab = S.head;                                              // head[512] and next[1024] are adjacent: 1024 u32 slots
    if (!tab_clean) {
        uint4* t4 = reinterpret_cast<uint4*>(tab);
#pragma unroll
        for (int x = 0; x < DV_TAB / 4 / 32; ++x) t4[lane + 32 * x] = make_uint4(0u, 0u, 0u, 0u);
        tab_clean = true;
    }
    __syncwarp();
    // ---- 3a. the chunks t[u .. u+8), u = j .. j+3, of the looked-up windows j
    const int ne = 4 * nq;
    const u32 en0 = lane < ne ? dv_entry(S, lane) : 0u;
    u32 alt = 22u;
    for (;;) {
        dv_tab_pass(S, tab, en0, ne, alt, DV_STORE);
        __syncwarp();
        const bool coll = dv_tab_pass(S, tab, en0, ne, alt, DV_CHECK);   // two different chunks in one slot (equal chunks of neighbouring windows coincide)
        if (!__any_sync(SCCG_FULL_MASK, coll)) break;
        __syncwarp();
        dv_tab_pass(S, tab, en0, ne, alt, DV_CLEAR);
        __syncwarp();
        if (alt == 12u) return 0;                                   // collides under both slot functions (or equal chunks at different positions): generic path
        alt = 12u;
    }
    // ---- 3b. probe: lane owns the chunks at a = 16 * lane + 4 * x and 512 + 16 * lane + 4 * x, x = 0 .. 3
    bool bad = false;
    {
        const uint4 x0 = reinterpret_cast<const uint4*>(S.r)[lane], x1 = reinterpret_cast<const uint4*>(S.r)[32 + lane];
        const u32 y0 = reinterpret_cast<const u32*>(S.r)[4 * lane + 4], y1 = reinterpret_cast<const u32*>(S.r)[128 + 4 * lane + 4];
        const u32 rr[10] = {x0.x, x0.y, x0.z, x0.w, y0, x1.x, x1.y, x1.z, x1.w, y1};
        const u32 A = (u32)(16 * lane) | 1024u;
        bool hit = false;
#pragma unroll
        for (int x = 0; x < 8; ++x) {
            const int wi = x < 4 ? x : x + 1;
            const u32 h = dv_hash(rr[wi], rr[wi + 1]);
            const u32 ent = tab[(h >> alt) & (u32)(DV_TAB - 1)];
            const u32 pos = (x < 4 ? 0u : 512u) | (u32)(4 * (x & 3));           // A | pos = 1024 | a (disjoint bits)
            const u32 xo = ((h & ~1023u) | A) ^ ent ^ pos;                      // 0: the diagonal chunk itself; 1..1023: same content, other position
            hit |= (xo - 1u) < 1023u;
        }
        if (__any_sync(SCCG_FULL_MASK, hit)) {
            // rare: some chunk of r has the content of a looked-up chunk at another position -- is it a whole k-mer?  One real
            // occurrence rejects the hypothesis, so the warp leaves at the first one any lane finds (a segment with a shifted
            // stretch -- an insertion and a deletion a few dozen symbols apart -- has dozens of them: checking them all cost
            // such a segment 50 k cycles, half of its total).
#pragma unroll 1
            for (int x = 0; x < 8; ++x) {
                if (hit) {
                    const int ra = (x < 4 ? 0 : 512) + 16 * lane + 4 * (x & 3);
                    const u32* r32 = reinterpret_cast<const u32*>(S.r) + (ra >> 2);   // (re-read: indexing the register copy would put it on the stack)
                    const u32 h = dv_hash(r32[0], r32[1]);
                    const u32 ent = tab[(h >> alt) & (u32)(DV_TAB - 1)];
                    const u32 xo = ((h & ~1023u) | 1024u | (u32)ra) ^ ent;
                    if ((xo - 1u) < 1023u) {
                        const int u = (int)(ent & 1023u);
#pragma unroll 1
                        for (int v = 0; v < nq && !bad; ++v) {
                            const int j = (int)(S.qv[v] & 0x3ffu);
                            const int d = u - j;
                            if (d < 0 || d > 3) continue;
                            const int pp = ra - d;
                            if (pp >= 0 && pp <= L - k && kmer_equal_smem(S.r, pp, S.t, j, k)) bad = true;
                        }
                    }
                }
                if (__any_sync(SCCG_FULL_MASK, bad)) break;
            }
        }
    }
    __syncwarp();
    dv_tab_pass(S, tab, en0, ne, alt, DV_CLEAR);                    // leave the table clean for the next segment
    __syncwarp();
    return __any_sync(SCCG_FULL_MASK, bad) ? 0 : nmatch;
}

#ifdef SCCG_SEG_TIMING
// development aid (tools/seg_timing.py, separate build): clock64() ticks spent per segment
__device__ unsigned long long* g_seg_cycles = nullptr;
#endif
#ifdef SCCG_SEG_STATS
// development aid (tools/seg_stats.py, separate build): how many segments took which path
__device__ unsigned long long g_seg_stats[8];      // 0 identical, 1 diagonal accepted, 2 generic (diagonal not tried / rejected), 3 second pass
#define SEG_STAT(i) do { if (lane == 0) atomicAdd(&g_seg_stats[i], 1ull); } while (0)
#else
#define SEG_STAT(i) do { } while (0)
#endif

// raw (not yet upper-cased) 8-byte words of the segment pair at symbol offset off: lane holds words lane, lane+32, lane+64, lane+96
__device__ __forceinline__ void lm_fetch(const u8* __restrict__ ref, const u8* __restrict__ tgt, i64 off, int Lr, int Lt, int lane, u64 (&rw)[4], u64 (&tw)[4]) {
    const u64* pr = reinterpret_cast<const u64*>(ref + off) + lane;
    const u64* pt = reinterpret_cast<const u64*>(tgt + off) + lane;
    if (Lr == SEG && Lt == SEG) {                              // uniform; 1000 symbols = 125 words: no per-word guards
#pragma unroll
        for (int it = 0; it < 3; ++it) { rw[it] = __ldg(pr + 32 * it); tw[it] = __ldg(pt + 32 * it); }
        rw[3] = 0ull; tw[3] = 0ull;
        if (lane < SEG / 8 - 96) { rw[3] = __ldg(pr + 96); tw[3] = __ldg(pt + 96); }
    } else {
#pragma unroll
        for (int it = 0; it < 4; ++it) {
            const int b0 = 8 * (lane + 32 * it);
            rw[it] = b0 < Lr ? __ldg(pr + 32 * it) : 0ull;
            tw[it] = b0 < Lt ? __ldg(pt + 32 * it) : 0ull;
        }
    }
}

// k1 > 0 always; k2 == 0 disables the second pass (function-level match_sequences).
// One launch handles the segments [seg_begin, n_iter) (the host entry points launch one range per uploaded chunk of the
// reference); n_total is the number of segment pairs of the whole job (T2 windows look across launch borders).
// work_counter: device u32, zero before the launch; hands out the segments after the pre-assigned ones.
// abort_flag (optional): seginfo must be preset to 0xffffffff ("not done"); as soon as some warp sees the T2 abort
// condition of the driver (:454-473: a failed, non-all-N segment ending a run of 5 counter increments) among finished
// segments it raises the flag and every warp stops claiming work -- the local attempt is discarded anyway (:466-472).
#ifndef SCCG_LM_CLAIM
#define SCCG_LM_CLAIM 2             // segments claimed per atomic
#endif
#ifndef SCCG_LM_MIN_CTAS
#define SCCG_LM_MIN_CTAS (32 / SCCG_LM_WARPS)   // 32 warps x 32 lanes x 64 registers = the whole register file of an SM
#endif
// CLAIM: consecutive segments per claim (SCCG_LM_CLAIM for the bulk launches; 1 for the abort probe, which wants the
// segments of a T2 window on different warps)
// MODE (two-phase launches, device-resident pairs of 64 K segments and more).  6 % of the segments of a near-identical pair take
// the generic path at 20-90 k cycles each, everything else 2-6 k.  The bulk launch (LM_DEFER) only QUEUES those segments and a
// second launch (LM_QUEUE) works the queue off.  Measured on the chr1-sized pair: the two launches alone take as long as the
// single one did (175 + 48 us against 208 -- the work is issue-bound, and neither fewer warps per SM nor heaviest-first order
// in the second launch changed that), but the queue launch leaves room for the run-list kernels of the side lane, which
// otherwise only start when the persistent CTAs of the matcher retire: compress step 0.359 -> 0.337 ms.
//   LM_INLINE: everything in one launch (abort probe, pipelined uploads, small pairs, function-level calls)
//   LM_DEFER : queue[atomicAdd(q_ctl, 1)] = seg for every segment that is neither identical nor decided by the diagonal path
//   LM_QUEUE : segment ids come from queue[0 .. *q_ctl); CLAIM 1, work_counter a fresh counter
enum { LM_INLINE = 0, LM_DEFER = 1, LM_QUEUE = 2 };
template <int CLAIM, int MODE>
__device__ __forceinline__ void seg_match_body(const u8* __restrict__ ref, i64 nr, const u8* __restrict__ tgt, i64 nt,
                                               int seg_begin, int n_iter, int n_total, int k1, int k2, u32* seginfo, u32* __restrict__ matches,
                                               u32* __restrict__ work_counter, u32* abort_flag, int use_diag, u32* queue, u32* q_ctl) {
    SCCG_DYN_SMEM(smem_raw);
    LmWarpSmem& S = reinterpret_cast<LmWarpSmem*>(smem_raw)[threadIdx.x >> 5];
    const int lane = lane_of();
    const int warps_total = (int)(gridDim.x * (blockDim.x >> 5));
    const int warp_global = (int)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5));
#ifndef SCCG_NO_EARLY_ABORT
    // the abort probe (or an earlier launch of the same attempt) has already raised the flag: nothing of this launch is used
    if (abort_flag && __any_sync(SCCG_FULL_MASK, __ldcg(abort_flag) != 0u)) return;
#endif

    // 2^(s*(k-1-lane)) for the cooperative k-mer hash of a target position (0 once the symbol has left the register)
    u32 pow1 = 0u, pow2 = 0u;
    {
        int sh = lm_hash_shift(k1) * (k1 - 1 - lane);
        if (lane < k1 && sh < 32) pow1 = 1u << sh;
        sh = k2 > 0 ? lm_hash_shift(k2) * (k2 - 1 - lane) : 32;
        if (lane < k2 && sh < 32) pow2 = 1u << sh;
    }

    // segments are claimed dynamically (their cost varies by an order of magnitude); the next segment is pulled into L2
    // while the current one is parsed and loaded when its turn comes (31 other warps of the SM cover that L2 latency)
    u64 nrw[4], ntw[4];
    const int claim = CLAIM;                                           // compile-time: a run-time claim size cost 15 % (registers in the hot loop)
    const int claim_base = seg_begin + warps_total * claim;            // the first warps_total * claim segments are pre-assigned
    int claimed_used = 0;
    bool tab_clean = false;                                   // S.head + S.next all zero (kept by the diagonal-hypothesis path)
    const u8* const pf_base = (lane < 8 ? ref : tgt) + 128 * (lane & 7);      // L2 prefetch of the next pair: lanes 0-7 the reference, 8-15 the target
    int seg = seg_begin + warp_global * claim < n_iter ? seg_begin + warp_global * claim : n_iter;
    const int nq = MODE == LM_QUEUE ? (int)*q_ctl : 0;                   // (written by the launch before this one)
    if (MODE == LM_QUEUE) seg = warp_global < nq ? (int)queue[warp_global] : n_iter;
    if (MODE == LM_QUEUE) use_diag = 0;                                  // queued segments have been through the cheap paths
    while (seg < n_iter) {
        const i64 off = (i64)seg * SEG;
        const int Lr = (int)((nr - off) < SEG ? (nr - off) : SEG);
        const int Lt = (int)((nt - off) < SEG ? (nt - off) : SEG);
        const int Lmin = Lr < Lt ? Lr : Lt;
        lm_fetch(ref, tgt, off, Lr, Lt, lane, nrw, ntw);
        __syncwarp();                                        // previous segment fully consumed
#ifdef SCCG_SEG_TIMING
        const long long t_begin = clock64();
        long long t_ph[6] = {0, 0, 0, 0, 0, 0};
#define SEG_PHASE(i) t_ph[i] = clock64()
#else
#define SEG_PHASE(i)
#endif
        u32 wm[4];                                           // diagonal-0 mismatch flags per 8-byte word (uniform)
        // upper-case in place (:369-370) and compare on the diagonal, all in registers: an identical pair never touches shared memory
#pragma unroll
        for (int it = 0; it < 4; ++it) {
            u64 rw = nrw[it], tw = ntw[it];
            if (rw & 0x2020202020202020ULL) rw = upper8(rw);                 // only bytes with bit 5 can be a-z
            if (tw & 0x2020202020202020ULL) tw = upper8(tw);
            nrw[it] = rw; ntw[it] = tw;
            wm[it] = __ballot_sync(SCCG_FULL_MASK, rw != tw);
        }
        if (Lr != SEG || Lt != SEG) {
            // a shorter (last) pair: only the first Lmin symbols are on the diagonal (full pairs: the words past the end were
            // fetched as 0 on both sides, nothing to mask)
            const int wv = Lmin >> 3, rem = Lmin & 7;
#pragma unroll
            for (int it = 0; it < 4; ++it) {
                const int q = lane + 32 * it;
                const u64 diff = nrw[it] ^ ntw[it];
                const bool d = q < wv ? diff != 0ull : (q == wv && rem ? (diff & (~0ull >> (64 - 8 * rem))) != 0ull : false);
                wm[it] = __ballot_sync(SCCG_FULL_MASK, d);
            }
        }
        // claim the next segment: SCCG_LM_CLAIM consecutive segments per atomic (one hot L2 address for the whole grid)
        int next_seg = seg + 1;
        if (++claimed_used >= claim) {
            if (lane == 0) {
                next_seg = (int)atomicAdd(work_counter, 1u) * claim + claim_base;
            }
            claimed_used = 0;
            next_seg = __shfl_sync(SCCG_FULL_MASK, next_seg, 0);
        }
        if (MODE == LM_QUEUE) next_seg = next_seg < nq ? (int)queue[next_seg] : n_iter;      // (claim_base = warps in the grid: queue index -> segment)
#ifndef SCCG_NO_EARLY_ABORT
        // checked before every segment (the flag lives in its own cache line, away from the claim atomics): a failing
        // segment is expensive, and after the abort nothing of this launch is used (:466-472)
        // (the vote makes the decision warp-uniform by construction: lanes that disagreed about the flag would leave the loop
        // at different segments and hang the collectives below)
        if (abort_flag && __any_sync(SCCG_FULL_MASK, __ldcg(abort_flag) != 0u)) next_seg = n_iter;
#endif
        if (next_seg + 1 < n_iter && lane < 16) {             // pull the next segment (a full pair: not the last one) into L2 only: no registers held across the parse
#ifndef SCCG_EMU
            asm volatile("prefetch.global.L2 [%0];" :: "l"(pf_base + (i64)next_seg * SEG));
#else
            (void)pf_base;
#endif
        }
        int nmatch = 0, covered = 0;
        bool direct = false;                                 // the matches are already in global memory
        if (Lr == Lt && Lt >= k1 && (wm[0] | wm[1] | wm[2] | wm[3]) == 0u) {
            // t_i == r_i: candidate p = 0 extends to Lt; any other p gives l <= Lr - p < Lt -> untied
            if (lane == 0) matches[(i64)seg * LM_SLOT] = 0u | (0u << 10) | ((u32)Lt << 20);
            nmatch = 1; covered = Lt; direct = true;
            SEG_STAT(0);
        } else {
#pragma unroll
            for (int it = 0; it < 4; ++it) {
                reinterpret_cast<u64*>(S.r)[lane + 32 * it] = nrw[it];
                reinterpret_cast<u64*>(S.t)[lane + 32 * it] = ntw[it];
            }
            if (lane < 2) reinterpret_cast<u64*>(S.r)[128 + lane] = 0ull, reinterpret_cast<u64*>(S.t)[128 + lane] = 0ull;
            __syncwarp();
            SEG_PHASE(0);
            if (use_diag && Lr == Lt && Lt >= k1 && k1 >= 11 &&
                (nmatch = lm_diag_parse(S, wm, Lt, k1, tab_clean, matches + (i64)seg * LM_SLOT, covered)) > 0) {
                // near-identical segment: parse determined by the mismatch positions, hypothesis proven against all of r
                direct = true;
                SEG_STAT(1);
            } else if (MODE == LM_DEFER) {
                if (lane == 0) queue[atomicAdd(q_ctl, 1u)] = (u32)seg;
                tab_clean = false;
                seg = next_seg;
                continue;                                     // seginfo[seg] stays "not done" until the queue launch
            } else {
                SEG_STAT(2);
                tab_clean = false;
                // pass 1 with k (compression.cpp:401), pass 2 with k' only if pass 1 found no match (:428); one copy of the code
#pragma unroll 1
                for (int pass = 0; pass < 2; ++pass) {
                    const int k = pass ? k2 : k1;
                    if (k <= 0) break;
#ifndef SCCG_NO_EARLY_ABORT
                    if (abort_flag) {                                                     // the launch is being discarded: do not start an expensive pass
                        u32 stop = lane == 0 ? __ldcg(abort_flag) : 0u;
                        if (__shfl_sync(SCCG_FULL_MASK, stop, 0)) break;
                    }
#endif
                    if (pass) SEG_STAT(3);
                    if (!pass) SEG_PHASE(1);
                    int n_runs = lm_runs(S, Lr, k);
                    if (n_runs < 0) n_runs = 0;                                   // too many runs to list: every k-mer goes into the chains
                    if (!pass) SEG_PHASE(2);
                    lm_build_index(S, Lr, k, n_runs);
                    if (!pass) SEG_PHASE(3);
                    nmatch = lm_parse(S, wm, Lr, Lt, k, pass ? pow2 : pow1, n_runs);
                    if (!pass) SEG_PHASE(4);
                    if (nmatch) break;
                }
            }
        }
        __syncwarp();
        if (!direct) {
            covered = 0;                                     // (a rejected diagonal hypothesis may have left its own sum behind)
            for (int m = lane; m < nmatch; m += 32) {
                u32 pk = S.mlist[m];
                matches[(i64)seg * LM_SLOT + m] = pk;
                covered += (int)(pk >> 20);
            }
            covered = __reduce_add_sync(SCCG_FULL_MASK, covered);
        }
        // "segment consists only of N" (:419, :455) matters only where the driver would count the segment: compute it there
        int all_n = 0;
        if (nmatch == 0 || 2 * (Lt - covered) > Lt) {
            int mine = 1;
            for (int b0 = 8 * lane; b0 < Lt; b0 += 256) {
                const u64 nx = reinterpret_cast<const u64*>(S.t)[b0 >> 3] ^ 0x4E4E4E4E4E4E4E4EULL;     // 'N' * 8
                const int vt = Lt - b0;
                if (vt >= 8 ? nx != 0ull : (nx & (~0ull >> (64 - 8 * vt))) != 0ull) mine = 0;
            }
            all_n = __all_sync(SCCG_FULL_MASK, mine);
        }
        if (lane == 0) {
            int lit = Lt - covered;                                              // count_mismatches :413
            u32 bad = (2 * lit > Lt) ? 1u : 0u;                                  // (float)lit / Lt > 0.5f  :417-419
            u32 info = (u32)nmatch | ((u32)lit << 8) | ((u32)(all_n ? 1 : 0) << 20) | (bad << 21);
#ifndef SCCG_NO_EARLY_ABORT
            if (abort_flag) {
                *reinterpret_cast<volatile u32*>(seginfo + seg) = info;
                if (!all_n && (nmatch == 0 || bad)) {
                    // this segment increments the counter: test the five windows of 5 consecutive segments that contain it
                    __threadfence();
                    for (int end = seg; end <= seg + T2_LIMIT && end < n_total; ++end) {
                        if (end < T2_LIMIT) continue;
                        bool all_inc = true;
                        for (int d = 0; d <= T2_LIMIT && all_inc; ++d) {
                            u32 x = *reinterpret_cast<volatile u32*>(seginfo + end - d);
                            bool inc = x != 0xffffffffu && !SEGINFO_ALLN(x) && (SEGINFO_NMATCH(x) == 0 || SEGINFO_BAD(x));
                            if (d == 0 && inc && SEGINFO_NMATCH(x) != 0) inc = false;     // the window must END with a failed segment
                            all_inc = inc;
                        }
                        if (all_inc) { atomicOr(abort_flag, 1u); break; }
                    }
                }
            } else
#endif
            {
                seginfo[seg] = info;
            }
        }
#ifdef SCCG_SEG_TIMING
        if (lane == 0 && g_seg_cycles) {
            const long long t_end = clock64();
            g_seg_cycles[seg] = (unsigned long long)(t_end - t_begin);
            // phases (generic segments): the tool allocates 6 arrays of n_total entries behind the totals
            if (t_ph[1]) {
                g_seg_cycles[(size_t)n_total * 1 + seg] = (unsigned long long)(t_ph[0] - t_begin);
                g_seg_cycles[(size_t)n_total * 2 + seg] = (unsigned long long)(t_ph[1] - t_ph[0]);
                g_seg_cycles[(size_t)n_total * 3 + seg] = (unsigned long long)(t_ph[2] - t_ph[1]);
                g_seg_cycles[(size_t)n_total * 4 + seg] = (unsigned long long)(t_ph[3] - t_ph[2]);
                g_seg_cycles[(size_t)n_total * 5 + seg] = (unsigned long long)(t_ph[4] - t_ph[3]);
                g_seg_cycles[(size_t)n_total * 6 + seg] = (unsigned long long)(t_end - t_ph[4]);
            }
        }
#endif
        seg = next_seg;
    }
}

template <int CLAIM>
__global__ void __launch_bounds__(LM_WARPS * 32, SCCG_LM_MIN_CTAS) seg_match_k(const u8* __restrict__ ref, i64 nr, const u8* __restrict__ tgt, i64 nt,
                                                            int seg_begin, int n_iter, int n_total, int k1, int k2, u32* seginfo, u32* __restrict__ matches,
                                                            u32* __restrict__ work_counter, u32* abort_flag, int use_diag) {
    seg_match_body<CLAIM, LM_INLINE>(ref, nr, tgt, nt, seg_begin, n_iter, n_total, k1, k2, seginfo, matches, work_counter, abort_flag, use_diag, nullptr, nullptr);
}
// the two launches of a device-resident pair
__global__ void __launch_bounds__(LM_WARPS * 32, SCCG_LM_MIN_CTAS) seg_match_defer_k(const u8* __restrict__ ref, i64 nr, const u8* __restrict__ tgt, i64 nt,
                                                            int seg_begin, int n_iter, int n_total, int k1, int k2, u32* seginfo, u32* __restrict__ matches,
                                                            u32* __restrict__ work_counter, u32* abort_flag, int use_diag, u32* queue, u32* q_ctl) {
    seg_match_body<SCCG_LM_CLAIM, LM_DEFER>(ref, nr, tgt, nt, seg_begin, n_iter, n_total, k1, k2, seginfo, matches, work_counter, abort_flag, use_diag, queue, q_ctl);
}
__global__ void __launch_bounds__(LM_WARPS * 32, SCCG_LM_MIN_CTAS) seg_match_queue_k(const u8* __restrict__ ref, i64 nr, const u8* __restrict__ tgt, i64 nt,
                                                            int n_total, int k1, int k2, u32* seginfo, u32* __restrict__ matches,
                                                            u32* __restrict__ work_counter, u32* abort_flag, u32* queue, u32* q_ctl) {
    seg_match_body<1, LM_QUEUE>(ref, nr, tgt, nt, 0, n_total, n_total, k1, k2, seginfo, matches, work_counter, abort_flag, 0, queue, q_ctl);
}

// Segment driver bookkeeping (compression.cpp:395-474): T2 abort test, delta chain carry, text size.
// One thread per segment.
// absolute != 0: tokens carry the absolute p as the reference writes them BEFORE delta_encode (:406-415); used when the
// text-level delta pass (sccg_delta.cuh) has to reproduce delta_encode on a body that contains literal '('.
__global__ void seg_bytes_k(const u32* __restrict__ seginfo, const u32* __restrict__ matches, int n_iter,
                            u32* __restrict__ seg_bytes, int* __restrict__ seg_prev_p, u32* __restrict__ d_abort, int absolute,
                            int seg_base, int carry_prev) {
    int i = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (i >= n_iter) return;
    if (*d_abort) return;                                    // raised early by seg_match_k: seginfo is incomplete and will be discarded
    u32 info = seginfo[i];
    int nmatch = (int)SEGINFO_NMATCH(info);
    if (nmatch == 0) {
        // both passes failed (:454-473).  counter > T2 <=> this and the 4 preceding segments all incremented it
        if (!SEGINFO_ALLN(info) && i >= T2_LIMIT) {
            bool all_inc = true;
            for (int d = 1; d <= T2_LIMIT; ++d) {
                u32 x = seginfo[i - d];
                bool inc = !SEGINFO_ALLN(x) && (SEGINFO_NMATCH(x) == 0 || SEGINFO_BAD(x));
                all_inc = all_inc && inc;
            }
            if (all_inc) atomicOr(d_abort, 1u);
        }
        seg_bytes[i] = 0u;                                   // silently dropped segment
        seg_prev_p[i] = 0;
        return;
    }
    // p of the previous match in file order (delta_encode :258).  seg_base / carry_prev: this launch covers the segments
    // seg_base .. of a chromosome that is sharded over several GPUs; carry_prev is the last match of the shards before it
    int prev = carry_prev;
    for (int s = i - 1; s >= 0; --s) {
        u32 x = seginfo[s];
        int nm = (int)SEGINFO_NMATCH(x);
        if (nm) { prev = (s + seg_base) * SEG + (int)((matches[(i64)s * LM_SLOT + nm - 1] >> 10) & 0x3ffu); break; }
    }
    seg_prev_p[i] = prev;
    u32 bytes = SEGINFO_LIT(info);
    int pp = prev;
    for (int m = 0; m < nmatch; ++m) {
        u32 pk = matches[(i64)i * LM_SLOT + m];
        int p_abs = (i + seg_base) * SEG + (int)((pk >> 10) & 0x3ffu);
        bytes += 3u + (u32)dec_len_i32(absolute ? p_abs : p_abs - pp) + (u32)dec_len_u32(pk >> 20);
        pp = p_abs;
    }
    seg_bytes[i] = bytes;
}

// writes "(dp,l)" at o, returns its length
__device__ __forceinline__ int write_token(u8* o, int dp, int l) {
    int w = 0;
    o[w++] = '(';
    w += write_dec_i32(o + w, dp);
    o[w++] = ',';
    w += write_dec_i32(o + w, l);
    o[w++] = ')';
    return w;
}

// one segment written by the whole warp (many matches or long literal runs)
__device__ __forceinline__ void seg_write_coop(const u8* __restrict__ tgt, i64 nt, const u32* __restrict__ matches, int seg, int nmatch,
                                               u8* __restrict__ base, int prevp, int absolute, int seg_base) {
    const int lane = lane_of();
    const i64 toff = (i64)seg * SEG;
    const int Lt = (int)((nt - toff) < SEG ? (nt - toff) : SEG);
    int prev_end = 0;
    u32 cursor = 0;
    for (int c0 = 0; c0 < nmatch; c0 += 32) {
        int m = c0 + lane;
        bool valid = m < nmatch;
        u32 pk = valid ? matches[(i64)seg * LM_SLOT + m] : 0u;
        int tpos = (int)(pk & 0x3ffu), l = (int)(pk >> 20);
        int p_abs = (seg + seg_base) * SEG + (int)((pk >> 10) & 0x3ffu);
        int te = tpos + l;
        int pp = __shfl_up_sync(SCCG_FULL_MASK, p_abs, 1);
        int pe = __shfl_up_sync(SCCG_FULL_MASK, te, 1);
        if (lane == 0) { pp = prevp; pe = prev_end; }
        if (absolute) pp = 0;
        int gap = valid ? tpos - pe : 0;
        int tok = valid ? 3 + dec_len_i32(p_abs - pp) + dec_len_u32((u32)l) : 0;
        u32 mine = (u32)(gap + tok);
        u32 incl = warp_scan_incl(mine);
        u32 o = cursor + incl - mine;
        if (valid) {
            if (gap <= 8) for (int x = 0; x < gap; ++x) base[o + x] = upper1(tgt[toff + pe + x]);
            write_token(base + o + gap, p_abs - pp, l);
        }
        u32 big = __ballot_sync(SCCG_FULL_MASK, valid && gap > 8);   // long literal runs: whole warp copies
        while (big) {
            int src = __ffs((int)big) - 1; big &= big - 1;
            int g = __shfl_sync(SCCG_FULL_MASK, gap, src);
            int s0 = __shfl_sync(SCCG_FULL_MASK, pe, src);
            u32 o0 = __shfl_sync(SCCG_FULL_MASK, o, src);
            for (int x = lane; x < g; x += 32) base[o0 + x] = upper1(tgt[toff + s0 + x]);
        }
        int lastl = (nmatch - 1 - c0) < 31 ? (nmatch - 1 - c0) : 31;
        prevp = __shfl_sync(SCCG_FULL_MASK, p_abs, lastl);
        prev_end = __shfl_sync(SCCG_FULL_MASK, te, lastl);
        cursor += __shfl_sync(SCCG_FULL_MASK, incl, 31);
    }
    for (int x = prev_end + lane; x < Lt; x += 32) base[cursor + (u32)(x - prev_end)] = upper1(tgt[toff + x]);   // trailing literals :164-167
}

// Record writer (compression.cpp:406-415) fused with delta_encode (:222-304).  A warp takes 32 consecutive segments:
// the usual segment (a few tokens, a few literals) is written by its own lane, segments with many matches or long
// literal runs are handed to the whole warp one after the other.
// The records of 32 light segments are one contiguous piece of the body (~ 0.7 KB): the lanes assemble it in shared memory,
// at the 16-byte phase of its place in the image, and the warp stores it with 16-byte vectors -- instead of ~ 25 byte stores
// per lane, each touching 32 different sectors.  d_total (optional): body bytes of all segments; NULL: direct stores only.
static const int SW_STAGE = 2304;                 // per warp; a piece that does not fit (or a warp with a heavy segment) goes out directly
__global__ void __launch_bounds__(256) seg_write_k(const u8* __restrict__ tgt, i64 nt, const u32* __restrict__ seginfo, const u32* __restrict__ matches,
                                                   const u32* __restrict__ seg_off, const int* __restrict__ seg_prev_p, int n_iter,
                                                   u8* __restrict__ out, const u32* __restrict__ d_body_base, int absolute, int seg_base,
                                                   const u32* __restrict__ d_total) {
    __align__(16) __shared__ u8 stage_all[8][SW_STAGE];
    const int lane = lane_of();
    const int warps_total = (int)(gridDim.x * (blockDim.x >> 5));
    if (*d_body_base == 0xffffffffu) return;                       // BODY_BASE_NONE: no local-mode image (abort) or not in this buffer
    u8* body = out + *d_body_base;
    u8* const stage = stage_all[threadIdx.x >> 5];
    for (int seg0 = (int)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32; seg0 < n_iter; seg0 += warps_total * 32) {
        const int seg = seg0 + lane;
        // everything a light segment needs is fetched up front, in parallel (one round trip instead of a chain of five):
        // status, text offset, delta carry and the first four matches (the slot is 400 bytes: 16-byte aligned)
        u32 info = 0u, off0 = 0u; int prev0 = 0;
        uint4 m4 = make_uint4(0u, 0u, 0u, 0u);
        if (seg < n_iter) {
            info = seginfo[seg]; off0 = seg_off[seg]; prev0 = seg_prev_p[seg];
            m4 = *reinterpret_cast<const uint4*>(matches + (i64)seg * LM_SLOT);
        }
        const int nmatch = (int)SEGINFO_NMATCH(info);
        const bool light = nmatch > 0 && nmatch <= 6 && SEGINFO_LIT(info) <= 24;
        const u32 heavy_lanes = __ballot_sync(SCCG_FULL_MASK, nmatch > 0 && !light);
        // the piece of the body these 32 segments fill
        const u32 first = __shfl_sync(SCCG_FULL_MASK, off0, 0);
        u32 piece = 0;
        bool staged = false;
        if (d_total && heavy_lanes == 0u) {
            const u32 end = seg0 + 32 < n_iter ? seg_off[seg0 + 32] : *d_total;
            piece = end - first;
            staged = piece + 16u <= (u32)SW_STAGE;
        }
        const u32 phase = (u32)((uintptr_t)(body + first) & 15u);
        if (light) {
            const i64 toff = (i64)seg * SEG;
            const int Lt = (int)((nt - toff) < SEG ? (nt - toff) : SEG);
            u8* o = staged ? stage + phase + (off0 - first) : body + off0;
            int pp = prev0, pe = 0;
            for (int m = 0; m < nmatch; ++m) {
                u32 pk = m == 0 ? m4.x : m == 1 ? m4.y : m == 2 ? m4.z : m == 3 ? m4.w : matches[(i64)seg * LM_SLOT + m];
                int tpos = (int)(pk & 0x3ffu), l = (int)(pk >> 20);
                int p_abs = (seg + seg_base) * SEG + (int)((pk >> 10) & 0x3ffu);
                for (int x = pe; x < tpos; ++x) *o++ = upper1(tgt[toff + x]);
                o += write_token(o, absolute ? p_abs : p_abs - pp, l);
                pp = p_abs; pe = tpos + l;
            }
            for (int x = pe; x < Lt; ++x) *o++ = upper1(tgt[toff + x]);
        }
        if (staged) {
            __syncwarp();
            u8* dst = body + first;
            const u8* src = stage + phase;
            u32 head = (16u - phase) & 15u;
            if (head > piece) head = piece;
            const u32 mid = (piece - head) & ~15u, tail = piece - head - mid;
            if ((u32)lane < head) dst[lane] = src[lane];
            for (u32 x = (u32)lane * 16u; x < mid; x += 512u) *reinterpret_cast<uint4*>(dst + head + x) = *reinterpret_cast<const uint4*>(src + head + x);
            if ((u32)lane < tail) dst[head + mid + lane] = src[head + mid + lane];
            __syncwarp();                                              // the stage is free again
        }
        u32 heavy = heavy_lanes;
        while (heavy) {
            int src = __ffs((int)heavy) - 1; heavy &= heavy - 1;
            int hseg = seg0 + src;
            int hn = __shfl_sync(SCCG_FULL_MASK, nmatch, src);
            seg_write_coop(tgt, nt, matches, hseg, hn, body + seg_off[hseg], seg_prev_p[hseg], absolute, seg_base);
        }
    }
}

// out[i] = toupper(src[i])  (leftover target segments, compression.cpp:476-481; global literals)
__global__ void upper_copy_k(const u8* __restrict__ src, i64 n, u8* __restrict__ out, const u32* __restrict__ d_base, u32 extra, const u32* __restrict__ d_extra) {
    if (d_base && *d_base == 0xffffffffu) return;                  // BODY_BASE_NONE (see put_separators_k)
    u8* dst = out + (d_base ? *d_base : 0u) + extra + (d_extra ? *d_extra : 0u);
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) dst[i] = upper1(src[i]);
}

}  // namespace sccg
