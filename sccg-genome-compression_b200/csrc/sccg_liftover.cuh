// Coordinates lifted between the resident reference and open archives (sccg_archive_liftover, include/sccg.h).
// Lift table of an archive: its whole-archive variant records (steps 1-4 of sccg_archive_variants, run by the same
// vr_records_count / vr_records_emit) as u32 columns, n records (len(R), len(D) < 2^31, records do not overlap):
//   pos[n] end[n] d_start[n] d_end[n], then four exclusive prefixes of n + 1 entries each over the records:
//   LT_PR reference lengths, LT_PD D lengths, LT_PS substitution lengths (equal on both sides), LT_PN length-changing records.
// Build, for every archive of a call without a table, in one pipeline run:
//   vr_records_count, vr_records_emit -> the records of all archives (record window = build ordinal), one host read of the total
//   lt_bounds_k                       -> the first record of each archive; one host read of these sizes the tables
//   lt_len_k / one sum scan           -> the four prefixes over all records, laid end to end ([PR | PD | PS | PN])
//   lt_fill_k                         -> each archive's columns and prefixes (relative to its first record) into its table
// Lift: lt_lift_k, one thread per query, two binary searches of the table (by pos for from = 0, by d_start for from = 1) and
// constant arithmetic.  DESIGN.md §4 note 16 explains why the closed form equals the ownership definition of include/sccg.h.
#pragma once
#include "sccg_variants.cuh"

#include <unordered_set>

namespace sccg {

enum { LT_PR = 0, LT_PD, LT_PS, LT_PN };
static inline size_t lt_words(u64 n) { return 8 * (size_t)n + 4; }

struct LtArch { const u32* t; i64 n, dlen, pad; };            // per archive index of a lift call (zero when no query names it)

__global__ void __launch_bounds__(VR_T) lt_bounds_k(const sccg_variant* rec, u64 nr, int n_build, u64* lo) {
    const int k = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (k <= n_build) lo[k] = vr_lower(rec, nr, k, 0);
}

// x[q * nr + r], q = LT_PR .. LT_PN: the lengths (and the length-change indicator) the prefixes sum
__global__ void __launch_bounds__(VR_T) lt_len_k(const sccg_variant* rec, u64 nr, u64* x) {
    for (u64 r = (u64)blockIdx.x * blockDim.x + threadIdx.x; r < nr; r += (u64)gridDim.x * blockDim.x) {
        const sccg_variant v = rec[r];
        const u64 lr = (u64)(v.end - v.pos), ld = (u64)(v.d_end - v.d_start);
        x[r] = lr; x[nr + r] = ld; x[2 * nr + r] = lr == ld ? lr : 0; x[3 * nr + r] = lr != ld;
    }
}

// items r < nr: record r into its archive's table; items nr + k: the closing prefix entries of archive k
__global__ void __launch_bounds__(VR_T) lt_fill_k(const sccg_variant* rec, u64 nr, const u64* x, const u64* lo, u32* const* tab, int n_build) {
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < nr + (u64)n_build; t += (u64)gridDim.x * blockDim.x) {
        const int k = t < nr ? (int)rec[t].window : (int)(t - nr);
        const u64 l = lo[k], n = lo[k + 1] - l;
        u32* T = tab[k];
        const u64 i = t < nr ? t - l : n, g = t < nr ? t : l + n;
        if (t < nr) {
            const sccg_variant v = rec[t];
            T[i] = (u32)v.pos; T[n + i] = (u32)v.end; T[2 * n + i] = (u32)v.d_start; T[3 * n + i] = (u32)v.d_end;
        }
        for (int q = 0; q < 4; ++q) T[4 * n + (u64)q * (n + 1) + i] = (u32)(x[(u64)q * nr + g] - x[(u64)q * nr + l]);
    }
}

// last record whose key is < b, or -1
__device__ __forceinline__ i64 lt_last(const u32* key, i64 n, i64 b) {
    i64 lo = 0, hi = n;
    while (lo < hi) { const i64 m = (lo + hi) >> 1; if ((i64)key[m] < b) lo = m + 1; else hi = m; }
    return lo - 1;
}

// one side of a table: the source columns (k, ke), the target columns (o, oe), the source-length prefix, the substitution
// prefix, the length-change prefix
struct LtSide {
    const u32 *k, *ke, *o, *oe, *pk, *ps, *pn;
    __device__ __forceinline__ LtSide(const LtArch& A, int from) {
        const u32* t = A.t;
        const i64 n = A.n;
        const u32* P = t + 4 * n;
        k = t + (from ? 2 * n : 0); ke = k + n;
        o = t + (from ? 0 : 2 * n); oe = o + n;
        pk = P + (from ? LT_PD : LT_PR) * (n + 1); ps = P + LT_PS * (n + 1); pn = P + LT_PN * (n + 1);
    }
    // F(b) with j = lt_last(k, n, b)
    __device__ __forceinline__ i64 lift(i64 j, i64 b) const { return j < 0 ? b : (i64)oe[j] + (b > (i64)ke[j] ? b - (i64)ke[j] : 0); }
    // source bases < b inside records (sub: inside substitution records)
    __device__ __forceinline__ i64 inside(i64 j, i64 b, bool sub) const {
        if (j < 0) return 0;
        const i64 part = (b < (i64)ke[j] ? b : (i64)ke[j]) - (i64)k[j];
        const bool is_sub = ke[j] - k[j] == oe[j] - o[j];
        return sub ? (i64)ps[j] + (is_sub ? part : 0) : (i64)pk[j] + part;
    }
};

__global__ void __launch_bounds__(VR_T) lt_lift_k(const LtArch* arch, const sccg_lift_query* qs, i64 nq, i64 rlen, sccg_lift* out) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    const sccg_lift_query q = qs[i];
    const LtArch A = arch[q.archive];
    const LtSide S(A, q.from);
    const i64 ls = q.from ? A.dlen : rlen, lt = q.from ? rlen : A.dlen, s = q.start, e = q.end;
    const i64 js = lt_last(S.k, A.n, s), je = lt_last(S.k, A.n, e == ls ? e + 1 : e);   // (the len rule: records at ls too)
    sccg_lift r;
    r.start = S.lift(js, s);
    r.end = e == ls ? lt : S.lift(je, e);
    r.same = (e - s) - (S.inside(je, e, false) - S.inside(js, s, false));
    r.subst = S.inside(je, e, true) - S.inside(js, s, true);
    r.records = je - js;
    int f = 0;
    if (js >= 0 && (i64)S.ke[js] > s) f |= SCCG_LIFT_START_INSIDE;
    if (je > js && (i64)S.ke[je] > e) f |= SCCG_LIFT_END_INSIDE;
    if (S.pn[je + 1] != S.pn[js + 1]) f |= SCCG_LIFT_LENGTH_CHANGE;
    r.flags = f; r.reserved = 0;
    out[i] = r;
}

// the lift tables of arcs[0 .. n) (none has one): all built, or none (*ms: kernel time)
static int lift_tables(sccg_ctx* c, const std::vector<sccg_archive*>& arcs, float* ms) {
    const int n = (int)arcs.size();
    VrArgs a;
    u8* d_tail = nullptr;
    u64 nr = 0;
    SCCG_TRY(vr_records_count(c, arcs.data(), n, 0, [](void*) {}, &a, &d_tail, &nr, ms));
    u64 *lo = nullptr, *x = nullptr;
    SCCG_TRY(buf(c, B_LT_LO, 2 * (size_t)n + 1, &lo));                      // [lo of each archive, nr | table pointers]
    SCCG_TRY(buf(c, B_LT_X, 4 * (size_t)nr + 1, &x));
    SCCG_TRY(ext_staging(c, sizeof(u64) * (2 * (size_t)n + 1)));
    const unsigned grid = (unsigned)(c->sm_count > 0 ? c->sm_count : 1) * 8u;
    const unsigned rg = nr ? (div_up((long long)nr, VR_T) < grid ? div_up((long long)nr, VR_T) : grid) : 1;
    SCCG_CK(cudaEventRecord(c->ev[3], c->stream));
    SCCG_TRY(vr_records_emit(c, a, nr));
    LAUNCH(c, lt_bounds_k, dim3(div_up((long long)n + 1, VR_T)), dim3(VR_T), 0, (const sccg_variant*)a.recf, nr, n, lo);
    if (nr) LAUNCH(c, lt_len_k, dim3(rg), dim3(VR_T), 0, (const sccg_variant*)a.recf, nr, x);
    SCCG_TRY(vr_scan<VrSum>(c, x, x, nullptr, 4 * nr, x + 4 * nr));
    SCCG_CK(cudaEventRecord(c->ev[2], c->stream));
    u64* h_lo = (u64*)c->h_ext;
    SCCG_CK(cudaMemcpyAsync(h_lo, lo, sizeof(u64) * ((size_t)n + 1), cudaMemcpyDeviceToHost, c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    float t = 0.f;
    cudaEventElapsedTime(&t, c->ev[3], c->ev[2]); *ms += t;
    // ---- one exactly-sized allocation per archive; any failure releases those of this call
    std::vector<void*> mem((size_t)n, nullptr);
    auto release = [&](int rc) { cudaStreamSynchronize(c->stream); for (void* p : mem) if (p) cudaFree(p); return rc; };
    u32** h_tab = (u32**)(h_lo + n + 1);
    for (int k = 0; k < n; ++k) {
        if (cudaMalloc(&mem[(size_t)k], sizeof(u32) * lt_words(h_lo[k + 1] - h_lo[k])) != cudaSuccess) {
            cudaGetLastError(); mem[(size_t)k] = nullptr;
            return release(set_error(SCCG_E_NOMEM, "cudaMalloc of a lift table failed"));
        }
        h_tab[k] = (u32*)mem[(size_t)k];
    }
    u32** d_tab = (u32**)(lo + n + 1);
    const unsigned fg = div_up((long long)(nr + (u64)n), VR_T) < grid ? div_up((long long)(nr + (u64)n), VR_T) : grid;
    if (cudaMemcpyAsync(d_tab, h_tab, sizeof(u32*) * (size_t)n, cudaMemcpyHostToDevice, c->stream) != cudaSuccess ||
        cudaEventRecord(c->ev[3], c->stream) != cudaSuccess)
        return release(set_error(SCCG_E_CUDA, "lift table upload failed"));
    LAUNCH(c, lt_fill_k, dim3(fg), dim3(VR_T), 0, (const sccg_variant*)a.recf, nr, (const u64*)x, (const u64*)lo, (u32* const*)d_tab, n);
    if (cudaEventRecord(c->ev[2], c->stream) != cudaSuccess || cudaStreamSynchronize(c->stream) != cudaSuccess)
        return release(set_error(SCCG_E_CUDA, "lift table build failed: %s", cudaGetErrorString(cudaGetLastError())));
    cudaEventElapsedTime(&t, c->ev[3], c->ev[2]); *ms += t;
    for (int k = 0; k < n; ++k) {
        sccg_archive* A = arcs[(size_t)k];
        A->lift = mem[(size_t)k]; A->lift_n = (long long)(h_lo[k + 1] - h_lo[k]);
        A->device_bytes += (long long)(sizeof(u32) * lt_words((u64)A->lift_n));
    }
    return SCCG_OK;
}

// sccg_archive_liftover: argument checks (include/sccg.h, in that order), the missing tables, then one copy of the query
// table, one launch, one copy back
static int archive_liftover_impl(sccg_ctx* c, sccg_archive* const* archives, i64 n_archives, const sccg_lift_query* queries, i64 n_queries,
                                 sccg_lift* out) {
    if (n_archives < 0 || n_queries < 0 || (n_archives > 0 && !archives) || (n_queries > 0 && (!queries || !out)))
        return set_error(SCCG_E_ARG, "null argument");
    if (n_archives >= 0x80000000LL || n_queries >= 0x80000000LL) return set_error(SCCG_E_ARG, "at most 2^31 - 1 archives and queries per call");
    int first = 7;                                                           // 0-3 archive checks, 4 from, 5 start, 6 end
    for (i64 i = 0; i < n_queries && first > 0; ++i) {
        const sccg_lift_query& q = queries[i];
        const int f = archive_query_fault(c, archives, n_archives, q.archive, 0, 0);
        const int bad = f < 4 ? f : (q.from != 0 && q.from != 1) ? 4 : (q.start < 0 || q.start > q.end) ? 5
                      : q.end > (q.from ? archives[q.archive]->g.Lm : c->res_ref_len) ? 6 : 7;
        if (bad < first) first = bad;
    }
    if (first < 4) return set_error(SCCG_E_ARG, archive_query_why[first]);
    if (first == 4) return set_error(SCCG_E_ARG, "a query's from must be 0 (reference) or 1 (archive)");
    if (first == 5) return set_error(SCCG_E_ARG, archive_query_why[4]);
    if (first == 6) return set_error(SCCG_E_ARG, "a query ends past the end of its source sequence (len(R) for from = 0, len(D) for from = 1)");
    if (n_queries == 0) return SCCG_OK;
    // ---- the tables the queries still need, each archive once however often it is listed
    std::vector<sccg_archive*> need;
    {
        std::unordered_set<const sccg_archive*> seen;
        for (i64 i = 0; i < n_queries; ++i) {
            sccg_archive* a = archives[queries[i].archive];
            if (!a->lift && seen.insert(a).second) need.push_back(a);
        }
    }
    float build = 0.f, ms = 0.f;
    if (!need.empty()) SCCG_TRY(lift_tables(c, need, &build));
    // ---- [LtArch of every archive | the queries] through the page-locked staging area, one copy
    const size_t arch_bytes = sizeof(LtArch) * (size_t)n_archives, q_bytes = sizeof(sccg_lift_query) * (size_t)n_queries;
    SCCG_TRY(ext_staging(c, arch_bytes + q_bytes));
    LtArch* h_arch = (LtArch*)c->h_ext;
    memset(h_arch, 0, arch_bytes);
    for (i64 i = 0; i < n_queries; ++i) {
        const sccg_archive* a = archives[queries[i].archive];
        h_arch[queries[i].archive] = LtArch{(const u32*)a->lift, (i64)a->lift_n, (i64)a->g.Lm, 0};
    }
    memcpy((char*)c->h_ext + arch_bytes, queries, q_bytes);
    u8* d_tab = nullptr; sccg_lift* d_out = nullptr;
    SCCG_TRY(buf(c, B_LT_Q, arch_bytes + q_bytes, &d_tab));
    SCCG_TRY(buf(c, B_LT_OUT, (size_t)n_queries, &d_out));
    SCCG_CK(cudaEventRecord(c->ev[4], c->stream));
    SCCG_CK(cudaMemcpyAsync(d_tab, c->h_ext, arch_bytes + q_bytes, cudaMemcpyHostToDevice, c->stream));
    SCCG_CK(cudaEventRecord(c->ev[5], c->stream));
    SCCG_CK(cudaEventRecord(c->ev[3], c->stream));
    LAUNCH(c, lt_lift_k, dim3(div_up(n_queries, VR_T)), dim3(VR_T), 0, (const LtArch*)d_tab, (const sccg_lift_query*)(d_tab + arch_bytes), n_queries,
           (i64)c->res_ref_len, d_out);
    SCCG_CK(cudaEventRecord(c->ev[2], c->stream));
    SCCG_CK(cudaMemcpyAsync(out, d_out, sizeof(sccg_lift) * (size_t)n_queries, cudaMemcpyDeviceToHost, c->stream));
    SCCG_CK(cudaEventRecord(c->ev[7], c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]); c->prof.h2d_ms = ms;
    cudaEventElapsedTime(&ms, c->ev[3], c->ev[2]); c->prof.gather_ms = ms; c->prof.kernels_ms = build + ms;
    cudaEventElapsedTime(&ms, c->ev[2], c->ev[7]); c->prof.d2h_ms = ms;
    return SCCG_OK;
}

}  // namespace sccg
