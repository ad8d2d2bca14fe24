// libsccg_b200.so -- C ABI (include/sccg.h) over the sm_100a kernels.  No CPU fallback: without a
// CUDA device sccg_create() fails and every other entry point needs a context.
#include "sccg_compress.cuh"
#include "sccg_global.cuh"
#include "sccg_decode.cuh"
#include "sccg_extract.cuh"
#include "sccg_search.cuh"
#include "sccg_search_edit.cuh"
#include "sccg_variants.cuh"
#include "sccg_liftover.cuh"
#include "sccg_fasta.cuh"
#include "sccg_shard.cuh"
#include "sccg_mgpu.cuh"

#include <new>
#include <time.h>

using namespace sccg;

namespace sccg {

static int check_sizes(i64 a, i64 b) {
    if (a < 0 || b < 0 || a >= 0x7fffffffLL || b >= 0x7fffffffLL) return set_error(SCCG_E_ARG, "sequence length must be in [0, 2^31-1)");
    return SCCG_OK;
}

// called at the start of every entry point except sccg_shard_write: besides the profile it invalidates the state that
// sccg_shard_match leaves behind (the buffers it points into are about to be reused)
static void prof_reset(sccg_ctx* c) { memset(&c->prof, 0, sizeof c->prof); c->shard.valid = 0; }

// read_genomes_from_files only ever yields a header that starts with '>' (compression.cpp:208-213); delta_encode keys its
// line skipping on that byte (:237), so anything else would shift the text it rewrites
static int check_header(const char* header, int64_t header_len) {
    if (header_len > 0 && header[0] != '>') return set_error(SCCG_E_ARG, "header must be empty or start with '>'");
    if (header_len > 0 && memchr(header, '\n', (size_t)header_len)) return set_error(SCCG_E_ARG, "header must be a single line");
    return SCCG_OK;
}
static int stoi_failure() {
    return set_error(SCCG_E_STOI, "stoi (a literal '(' in the target breaks the reference's delta_encode; the output holds the un-rewritten image)");
}

}  // namespace sccg

extern "C" {

const char* sccg_version(void) {
#ifdef SCCG_EMU
    return "sccg-b200 0.1 (SIMT emulator build: kernel logic tests only)";
#else
    return "sccg-b200 0.1 (sm_100a)";
#endif
}

const char* sccg_last_error(void) { return g_last_error.c_str(); }

static double wall_s() { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec; }

sccg_ctx* sccg_create(int device) {
    const bool timing = getenv("SCCG_TIMING") != nullptr;
    const double t_begin = wall_s();
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    const double t_count = wall_s();
    if (e != cudaSuccess || ndev <= 0) {
        set_error(SCCG_E_CUDA, "no CUDA device available (%s): this library has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        return nullptr;
    }
    if (device < 0 || device >= ndev) { set_error(SCCG_E_ARG, "device index out of range"); return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) { set_error(SCCG_E_CUDA, "cudaSetDevice failed"); return nullptr; }
    cudaFree(0);                                                               // forces the primary context into existence here (timed below)
    const double t_ctx = wall_s();
    sccg_ctx* c = new (std::nothrow) sccg_ctx();
    if (!c) { set_error(SCCG_E_NOMEM, "out of host memory"); return nullptr; }
    memset(c, 0, sizeof *c);
    c->device = device;
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (c->sm_count <= 0) c->sm_count = 148;
    c->h_pinned_cap = 1 << 20;
    { const char* e = getenv("SCCG_NO_DIAG"); c->use_diag = (e && atoi(e) != 0) ? 0 : 1; }    // tests: force the generic segment parse
    // (stream priorities for either lane were measured: main first 0.343 -> 0.389 ms per chr1-sized pair, side first no change)
    bool ok = cudaStreamCreate(&c->main_stream) == cudaSuccess && cudaStreamCreate(&c->side_stream) == cudaSuccess &&
              cudaMallocHost(&c->h_pinned, c->h_pinned_cap) == cudaSuccess;
    c->stream = c->main_stream;
    for (int i = 0; ok && i < 6; ++i) ok = cudaEventCreate(&c->ev_side[i]) == cudaSuccess;
    for (int i = 0; ok && i < 8; ++i) ok = cudaEventCreate(&c->ev[i]) == cudaSuccess;
    for (int i = 0; ok && i < 4; ++i) ok = cudaEventCreate(&c->ev_x[i]) == cudaSuccess;
    if (!ok) { set_error(SCCG_E_CUDA, "context setup failed: %s", cudaGetErrorString(cudaGetLastError())); sccg_destroy(c); return nullptr; }
    if (timing) fprintf(stderr, "timing: sccg_create: driver init %.3f s, device context %.3f s, streams / events / staging %.3f s\n", t_count - t_begin, t_ctx - t_count, wall_s() - t_ctx);
    return c;
}

void sccg_destroy(sccg_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    for (int i = 0; i < B_NSLOTS; ++i) if (c->bufs[i].p) cudaFree(c->bufs[i].p);
    if (c->h_pinned) cudaFreeHost(c->h_pinned);
    if (c->res_ref) cudaFree(c->res_ref);
    while (c->archives) { sccg_archive* a = c->archives; archive_unlink(c, a); archive_free(a); }
    for (int f = 0; f < 2; ++f) if (c->res_form[f]) cudaFree(c->res_form[f]);
    if (c->res_nrun) cudaFree(c->res_nrun);
    for (int i = 0; i < 8; ++i) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    for (int i = 0; i < 4; ++i) if (c->ev_x[i]) cudaEventDestroy(c->ev_x[i]);
    if (c->main_stream) cudaStreamDestroy(c->main_stream);
    if (c->side_stream) cudaStreamDestroy(c->side_stream);
    for (int i = 0; i < 6; ++i) if (c->ev_side[i]) cudaEventDestroy(c->ev_side[i]);
    if (c->pipe_ready) {
        cudaStreamDestroy(c->s_h2d); cudaStreamDestroy(c->s_d2h);
        for (int i = 0; i < 2; ++i) cudaEventDestroy(c->ev_pipe[i]);
        for (int i = 0; i < 64; ++i) { cudaEventDestroy(c->ev_h2d[i]); cudaEventDestroy(c->ev_g[i]); cudaEventDestroy(c->ev_d2h[i]); }
    }
    for (int i = 0; i < 2; ++i) if (c->h_stream[i]) cudaFreeHost(c->h_stream[i]);
    if (c->h_ext) cudaFreeHost(c->h_ext);
    delete c;
}

void sccg_free(void* p) { free(p); }

void sccg_records_free(sccg_records* r) {
    if (!r) return;
    free(r->p); free(r->l); free(r->lit_off); free(r->lits);
    memset(r, 0, sizeof *r);
}

int sccg_download(sccg_ctx* c, const void* d_src, int64_t n, void* h_dst) {
    if (!c || n < 0 || (n > 0 && (!d_src || !h_dst))) return set_error(SCCG_E_ARG, "null argument");
    SCCG_CK(cudaSetDevice(c->device));
    if (n > 0) {
        SCCG_CK(cudaMemcpyAsync(h_dst, d_src, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaStreamSynchronize(c->stream));
    }
    return SCCG_OK;
}

int sccg_get_profile(sccg_ctx* c, sccg_profile* out) {
    if (!c || !out) return set_error(SCCG_E_ARG, "null argument");
    *out = c->prof;
    return SCCG_OK;
}

int sccg_compress_device(sccg_ctx* c, const void* d_ref, int64_t ref_len, const void* d_tgt, int64_t tgt_len,
                         const char* header, int64_t header_len, void** d_out, int64_t* out_len, int* mode_out) {
    if (!c || !d_out || !out_len || (header_len > 0 && !header)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_len, tgt_len));
    SCCG_TRY(check_header(header, header_len));
    if (((uintptr_t)d_ref | (uintptr_t)d_tgt) & 15) return set_error(SCCG_E_ARG, "device inputs must be 16-byte aligned");
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    CompressResult res;
    SCCG_TRY(compress_device(c, (const u8*)d_ref, ref_len, (const u8*)d_tgt, tgt_len, header, header_len < 0 ? 0 : header_len, &res, nullptr));
    *d_out = res.d_out; *out_len = res.out_len;
    if (mode_out) *mode_out = res.mode;
    return res.stoi_failed ? stoi_failure() : SCCG_OK;
}

static int compress_host(sccg_ctx* c, const char* ref, int64_t ref_len, const char* tgt, int64_t tgt_len, const char* header, int64_t header_len,
                         char* dst, int64_t dst_cap, char** out, int64_t* out_len, int* mode_out) {
    if (!c || !out_len || (ref_len > 0 && !ref) || (tgt_len > 0 && !tgt) || (header_len > 0 && !header)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_len, tgt_len));
    SCCG_TRY(check_header(header, header_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    u8 *d_ref = nullptr, *d_tgt = nullptr;
    ChunkArrival arr;
    SCCG_TRY(enqueue_pair_upload(c, ref, ref_len, tgt, tgt_len, &d_ref, &d_tgt, &arr));
    CompressResult res;
    int rc_c = compress_device(c, d_ref, ref_len, d_tgt, tgt_len, header, header_len < 0 ? 0 : header_len, &res, &arr);
    SCCG_CK(cudaStreamSynchronize(c->s_h2d));                                 // the caller's buffers are no longer in use
    if (rc_c != SCCG_OK) return rc_c;
    SCCG_CK(cudaEventRecord(c->ev[6], c->stream));
    SCCG_TRY(deliver(c, res.d_out, res.out_len, dst, dst_cap, out, out_len));
    SCCG_CK(cudaEventRecord(c->ev[7], c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    cudaEventElapsedTime(&c->prof.h2d_ms, c->ev[4], c->ev[5]);
    cudaEventElapsedTime(&c->prof.d2h_ms, c->ev[6], c->ev[7]);
    if (mode_out) *mode_out = res.mode;
    return res.stoi_failed ? stoi_failure() : SCCG_OK;
}

int sccg_compress(sccg_ctx* c, const char* ref, int64_t ref_len, const char* tgt, int64_t tgt_len,
                  const char* header, int64_t header_len, char** out, int64_t* out_len, int* mode_out) {
    if (!out) return set_error(SCCG_E_ARG, "null argument");
    return compress_host(c, ref, ref_len, tgt, tgt_len, header, header_len, nullptr, 0, out, out_len, mode_out);
}

int sccg_compress_into(sccg_ctx* c, const char* ref, int64_t ref_len, const char* tgt, int64_t tgt_len,
                       const char* header, int64_t header_len, char* out, int64_t out_cap, int64_t* out_len, int* mode_out) {
    if (!out) return set_error(SCCG_E_ARG, "null argument");
    return compress_host(c, ref, ref_len, tgt, tgt_len, header, header_len, out, out_cap, nullptr, out_len, mode_out);
}

// ---- resident reference: many targets against one reference (the reference goes over PCIe once) ------------------------
int sccg_reference_set(sccg_ctx* c, const char* ref, int64_t ref_len) {
    if (!c || ref_len < 0 || (ref_len > 0 && !ref)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_len, 0));
    SCCG_CK(cudaSetDevice(c->device));
    reference_changed(c);
    const size_t need = (size_t)ref_len + 128;
    if (need > c->res_ref_cap) {
        if (c->res_ref) { SCCG_CK(cudaStreamSynchronize(c->main_stream)); cudaFree(c->res_ref); c->res_ref = nullptr; c->res_ref_cap = 0; }
        c->res_ref_set = 0; c->res_ref_len = 0;                                // no resident reference until the new one is complete
        void* p = nullptr;
        if (cudaMalloc(&p, need) != cudaSuccess) { cudaGetLastError(); return set_error(SCCG_E_NOMEM, "cudaMalloc of the resident reference failed"); }
        c->res_ref = (u8*)p; c->res_ref_cap = need;
    }
    c->res_ref_set = 0;
    if (ref_len > 0) SCCG_CK(cudaMemcpyAsync(c->res_ref, ref, (size_t)ref_len, cudaMemcpyHostToDevice, c->main_stream));
    SCCG_CK(cudaMemsetAsync(c->res_ref + ref_len, 0, 128, c->main_stream));
    SCCG_CK(cudaStreamSynchronize(c->main_stream));                            // the caller's buffer is free again
    c->res_ref_len = ref_len;
    c->res_ref_set = 1;
    return SCCG_OK;
}

int sccg_reference_clear(sccg_ctx* c) {
    if (!c) return set_error(SCCG_E_ARG, "null argument");
    SCCG_CK(cudaSetDevice(c->device));
    reference_changed(c);
    if (c->res_ref) { SCCG_CK(cudaStreamSynchronize(c->main_stream)); cudaFree(c->res_ref); }
    c->res_ref = nullptr; c->res_ref_cap = 0; c->res_ref_len = 0; c->res_ref_set = 0;
    return SCCG_OK;
}

// compress_genome against the resident reference: only the target travels, in chunks, and the matcher starts on every
// chunk as it lands
int sccg_compress_resident_into(sccg_ctx* c, const char* tgt, int64_t tgt_len, const char* header, int64_t header_len,
                                char* dst, int64_t dst_cap, int64_t* out_len, int* mode_out) {
    if (!c || !dst || !out_len || (tgt_len > 0 && !tgt) || (header_len > 0 && !header)) return set_error(SCCG_E_ARG, "null argument");
    if (!c->res_ref_set) return set_error(SCCG_E_ARG, "no resident reference (call sccg_reference_set first)");
    SCCG_TRY(check_sizes(c->res_ref_len, tgt_len));
    SCCG_TRY(check_header(header, header_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    u8* d_tgt = nullptr;
    SCCG_TRY(pipe_streams(c));
    SCCG_TRY(buf(c, B_TGT, (size_t)tgt_len + 128, &d_tgt));
    if (getenv("SCCG_PIPE_POISON")) SCCG_CK(cudaMemsetAsync(d_tgt, 0xEE, (size_t)tgt_len, c->stream));     // tests: a chunk read before it arrived shows up
    SCCG_CK(cudaEventRecord(c->ev[4], c->stream));
    SCCG_CK(cudaStreamWaitEvent(c->s_h2d, c->ev[4], 0));
    ChunkArrival arr;
    arr.chunk = pipe_chunk_bytes(tgt_len);
    arr.n = tgt_len > 0 ? (int)((tgt_len + arr.chunk - 1) / arr.chunk) : 0;
    arr.ev_ref = c->ev_h2d; arr.ev_tgt = c->ev_pipe[1]; arr.tgt_chunked = 1;
    for (int i = 0; i < arr.n; ++i) {
        const i64 off = (i64)i * arr.chunk, len = (tgt_len - off) < arr.chunk ? (tgt_len - off) : arr.chunk;
        SCCG_CK(cudaMemcpyAsync(d_tgt + off, tgt + off, (size_t)len, cudaMemcpyHostToDevice, c->s_h2d));
        SCCG_CK(cudaEventRecord(arr.ev_ref[i], c->s_h2d));
    }
    SCCG_CK(cudaMemsetAsync(d_tgt + tgt_len, 0, 64, c->s_h2d));
    SCCG_CK(cudaEventRecord(arr.ev_tgt, c->s_h2d));
    SCCG_CK(cudaEventRecord(c->ev[5], c->s_h2d));
    CompressResult res;
    int rc_c = compress_device(c, c->res_ref, c->res_ref_len, d_tgt, tgt_len, header, header_len < 0 ? 0 : header_len, &res, &arr);
    SCCG_CK(cudaStreamSynchronize(c->s_h2d));                                 // the caller's buffer is no longer in use
    if (rc_c != SCCG_OK) return rc_c;
    SCCG_CK(cudaEventRecord(c->ev[6], c->stream));
    SCCG_TRY(deliver(c, res.d_out, res.out_len, dst, dst_cap, nullptr, out_len));
    SCCG_CK(cudaEventRecord(c->ev[7], c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    cudaEventElapsedTime(&c->prof.h2d_ms, c->ev[4], c->ev[5]);
    cudaEventElapsedTime(&c->prof.d2h_ms, c->ev[6], c->ev[7]);
    if (mode_out) *mode_out = res.mode;
    return res.stoi_failed ? stoi_failure() : SCCG_OK;
}

// decompress_genome against the resident reference: the record file goes up, the text comes back in chunks
int sccg_decompress_resident_into(sccg_ctx* c, const char* inter, int64_t inter_len, char* out, int64_t out_cap, int64_t* out_len) {
    if (!c || !out || !out_len || (inter_len > 0 && !inter)) return set_error(SCCG_E_ARG, "null argument");
    if (!c->res_ref_set) return set_error(SCCG_E_ARG, "no resident reference (call sccg_reference_set first)");
    SCCG_TRY(check_sizes(c->res_ref_len, inter_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    return decompress_host(c, nullptr, c->res_ref_len, inter, inter_len, out, out_cap, nullptr, out_len, c->res_ref);
}

int sccg_match_sequences(sccg_ctx* c, const char* Sr, int64_t nr, const char* St, int64_t nt,
                         int k, int m, int global, int offset, sccg_records* out) {
    if (!c || !out || (nr > 0 && !Sr) || (nt > 0 && !St)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(nr, nt));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    memset(out, 0, sizeof *out);
    u8 *d_ref = nullptr, *d_tgt = nullptr;
    SCCG_TRY(upload(c, B_REF, Sr, nr, &d_ref));
    SCCG_TRY(upload(c, B_TGT, St, nt, &d_tgt));
    if (global) return match_sequences_global(c, d_ref, nr, d_tgt, nt, St, k, m, offset, out);

    // local: one segment pair through the segment kernel, single pass with the caller's k
    if (nr > SEG || nt > SEG) return set_error(SCCG_E_ARG, "local match_sequences takes one segment pair (<= 1000 symbols each)");
    if (k < K2 || k > 32) return set_error(SCCG_E_ARG, "local match_sequences supports 10 <= k <= 32");
    u32 *seginfo = nullptr, *matches = nullptr, *sc = nullptr;
    SCCG_TRY(buf(c, B_SCALARS, (size_t)S_COUNT, &sc));
    SCCG_CK(cudaMemsetAsync(sc, 0, sizeof(u32) * S_COUNT, c->stream));
    SCCG_TRY(buf(c, B_SEGINFO, 2, &seginfo));
    SCCG_TRY(buf(c, B_MATCH, LM_SLOT + 1, &matches));
    int nmatch = 0;
    u32 h_matches[LM_SLOT];
    if (nt > 0) {
        // the kernel upper-cases on load (the reference driver does so before calling, :369-370); callers pass
        // upper-cased symbols, for which this is the identity
        const size_t smem = sizeof(LmWarpSmem) * LM_WARPS;
        SCCG_SET_MAX_SMEM(seg_match_k<SCCG_LM_CLAIM>, smem);
        LAUNCH(c, seg_match_k<SCCG_LM_CLAIM>, dim3(1), dim3(LM_WARPS * 32), smem, (const u8*)d_ref, (i64)(nr > 0 ? nr : 0), (const u8*)d_tgt, nt, 0, 1, 1, k, 0, seginfo, matches, sc + S_WORK, (u32*)nullptr, c->use_diag);
        u32 info = 0;
        SCCG_CK(cudaMemcpyAsync(&info, seginfo, sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaMemcpyAsync(h_matches, matches, sizeof(u32) * LM_SLOT, cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaStreamSynchronize(c->stream));
        nmatch = (int)SEGINFO_NMATCH(info);
    }
    // vector<Position>: alternating literal / match records (compression.cpp:97-108, :152-156, :164-167)
    int64_t cap = 2 * (int64_t)nmatch + 2;
    out->p = (int32_t*)malloc(sizeof(int32_t) * (size_t)cap);
    out->l = (int32_t*)malloc(sizeof(int32_t) * (size_t)cap);
    out->lit_off = (int64_t*)malloc(sizeof(int64_t) * (size_t)(cap + 1));
    out->lits = (char*)malloc((size_t)nt + 1);
    if (!out->p || !out->l || !out->lit_off || !out->lits) { sccg_records_free(out); return set_error(SCCG_E_NOMEM, "out of host memory"); }
    int64_t n = 0, lit = 0;
    int pos = 0;
    for (int i = 0; i <= nmatch; ++i) {
        int tpos = i < nmatch ? (int)(h_matches[i] & 0x3ffu) : (int)nt;
        if (tpos > pos) {
            out->p[n] = -1; out->l[n] = 0; out->lit_off[n] = lit;
            memcpy(out->lits + lit, St + pos, (size_t)(tpos - pos));
            lit += tpos - pos; ++n;
        }
        if (i < nmatch) {
            out->p[n] = (int)((h_matches[i] >> 10) & 0x3ffu) + offset;
            out->l[n] = (int)(h_matches[i] >> 20);
            out->lit_off[n] = lit; ++n;
            pos = tpos + out->l[n - 1];
        }
    }
    out->lit_off[n] = lit;
    out->n = n;
    (void)m;
    return SCCG_OK;
}

int sccg_reconstruct_device(sccg_ctx* c, const void* d_ref, int64_t ref_len, const void* d_encoded, int64_t enc_len,
                            const void* d_n_idx, int64_t n_len, const void* d_low_idx, int64_t low_len,
                            void** d_out, int64_t* out_len) {
    if (!c || !d_out || !out_len) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_len, enc_len));
    SCCG_TRY(check_sizes(n_len, low_len));
    if (((uintptr_t)d_ref | (uintptr_t)d_encoded | (uintptr_t)d_n_idx | (uintptr_t)d_low_idx) & 15) return set_error(SCCG_E_ARG, "device inputs must be 16-byte aligned");
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    u8* out = nullptr; i64 n = 0;
    SCCG_TRY(reconstruct_device(c, (const u8*)d_ref, ref_len, (const u8*)d_encoded, enc_len, (const u8*)d_n_idx, n_len,
                                (const u8*)d_low_idx, low_len, 0, &out, &n));
    *d_out = out; *out_len = n;
    return SCCG_OK;
}

static int reconstruct_host(sccg_ctx* c, const char* ref, int64_t ref_len, const char* encoded, int64_t enc_len, const char* n_idx, int64_t n_len,
                            const char* low_idx, int64_t low_len, char* dst, int64_t dst_cap, char** out, int64_t* out_len) {
    if (!c || !out_len || (ref_len > 0 && !ref) || (enc_len > 0 && !encoded) || (n_len > 0 && !n_idx) || (low_len > 0 && !low_idx))
        return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_len, enc_len));
    SCCG_TRY(check_sizes(n_len, low_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    u8 *d_ref = nullptr, *d_enc = nullptr, *d_n = nullptr, *d_low = nullptr;
    SCCG_CK(cudaEventRecord(c->ev[4], c->stream));
    SCCG_TRY(upload(c, B_REF, ref, ref_len, &d_ref));
    SCCG_TRY(upload(c, B_ENC, encoded, enc_len, &d_enc));
    SCCG_TRY(upload(c, B_NIDX, n_idx, n_len, &d_n));
    SCCG_TRY(upload(c, B_LOW, low_idx, low_len, &d_low));
    SCCG_CK(cudaEventRecord(c->ev[5], c->stream));
    u8* d_res = nullptr; i64 n = 0;
    SCCG_TRY(reconstruct_device(c, d_ref, ref_len, d_enc, enc_len, d_n, n_len, d_low, low_len, 0, &d_res, &n));
    SCCG_CK(cudaEventRecord(c->ev[6], c->stream));
    SCCG_TRY(deliver(c, d_res, n, dst, dst_cap, out, out_len));
    SCCG_CK(cudaEventRecord(c->ev[7], c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    cudaEventElapsedTime(&c->prof.h2d_ms, c->ev[4], c->ev[5]);
    cudaEventElapsedTime(&c->prof.d2h_ms, c->ev[6], c->ev[7]);
    return SCCG_OK;
}

int sccg_reconstruct(sccg_ctx* c, const char* ref, int64_t ref_len, const char* encoded, int64_t enc_len,
                     const char* n_idx, int64_t n_len, const char* low_idx, int64_t low_len, char** out, int64_t* out_len) {
    if (!out) return set_error(SCCG_E_ARG, "null argument");
    return reconstruct_host(c, ref, ref_len, encoded, enc_len, n_idx, n_len, low_idx, low_len, nullptr, 0, out, out_len);
}

int sccg_reconstruct_into(sccg_ctx* c, const char* ref, int64_t ref_len, const char* encoded, int64_t enc_len,
                          const char* n_idx, int64_t n_len, const char* low_idx, int64_t low_len, char* out, int64_t out_cap, int64_t* out_len) {
    if (!out) return set_error(SCCG_E_ARG, "null argument");
    return reconstruct_host(c, ref, ref_len, encoded, enc_len, n_idx, n_len, low_idx, low_len, out, out_cap, nullptr, out_len);
}

int sccg_decompress(sccg_ctx* c, const char* ref_raw, int64_t ref_len, const char* inter, int64_t inter_len, char** out, int64_t* out_len) {
    if (!c || !out || !out_len || (ref_len > 0 && !ref_raw) || (inter_len > 0 && !inter)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_len, inter_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    return decompress_host(c, ref_raw, ref_len, inter, inter_len, nullptr, 0, out, out_len);
}

int sccg_decompress_into(sccg_ctx* c, const char* ref_raw, int64_t ref_len, const char* inter, int64_t inter_len, char* out, int64_t out_cap, int64_t* out_len) {
    if (!c || !out || !out_len || (ref_len > 0 && !ref_raw) || (inter_len > 0 && !inter)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_len, inter_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    return decompress_host(c, ref_raw, ref_len, inter, inter_len, out, out_cap, nullptr, out_len);
}

// ---- FASTA images in, FASTA handling on the device (SURVEY 8f.1) -------------------------------------------------------
static int upload_file(sccg_ctx* c, int slot, const char* h, int64_t n, u8** d) {
    SCCG_TRY(buf(c, slot, (size_t)(n > 0 ? n : 1) + 128, d));
    if (n > 0) SCCG_CK(cudaMemcpyAsync(*d, h, (size_t)n, cudaMemcpyHostToDevice, c->stream));
    SCCG_CK(cudaMemsetAsync(*d + (n > 0 ? n : 0), 0, 64, c->stream));
    return SCCG_OK;
}

// the two file images travel on the copy stream -- target first -- while the compute stream already strips the target; with
// page-locked sources (sccg_pinned_alloc) the copies run at full PCIe speed and asynchronously
static int compress_fasta_impl(sccg_ctx* c, const char* ref_file, int64_t ref_file_len, const char* tgt_file, int64_t tgt_file_len,
                               char* dst, int64_t dst_cap, char** out, int64_t* out_len, int* mode_out) {
    if (!c || !out_len || (ref_file_len > 0 && !ref_file) || (tgt_file_len > 0 && !tgt_file)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_file_len, tgt_file_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    SCCG_TRY(pipe_streams(c));
    u8 *d_rf = nullptr, *d_tf = nullptr;
    u32* sc = nullptr;
    SCCG_TRY(buf(c, B_SCALARS, (size_t)S_COUNT, &sc));
    SCCG_TRY(buf(c, B_FILE_R, (size_t)(ref_file_len > 0 ? ref_file_len : 1) + 128, &d_rf));
    SCCG_TRY(buf(c, B_FILE_T, (size_t)(tgt_file_len > 0 ? tgt_file_len : 1) + 128, &d_tf));
    SCCG_CK(cudaEventRecord(c->ev[4], c->stream));
    SCCG_CK(cudaStreamWaitEvent(c->s_h2d, c->ev[4], 0));                      // (the buffers may just have been reallocated)
    if (tgt_file_len > 0) SCCG_CK(cudaMemcpyAsync(d_tf, tgt_file, (size_t)tgt_file_len, cudaMemcpyHostToDevice, c->s_h2d));
    SCCG_CK(cudaMemsetAsync(d_tf + (tgt_file_len > 0 ? tgt_file_len : 0), 0, 64, c->s_h2d));
    SCCG_CK(cudaEventRecord(c->ev_pipe[1], c->s_h2d));
    if (ref_file_len > 0) SCCG_CK(cudaMemcpyAsync(d_rf, ref_file, (size_t)ref_file_len, cudaMemcpyHostToDevice, c->s_h2d));
    SCCG_CK(cudaMemsetAsync(d_rf + (ref_file_len > 0 ? ref_file_len : 0), 0, 64, c->s_h2d));
    SCCG_CK(cudaEventRecord(c->ev[5], c->s_h2d));
    FastaSeq R, T;
    SCCG_CK(cudaStreamWaitEvent(c->stream, c->ev_pipe[1], 0));
    int rc = fasta_ingest(c, d_tf, tgt_file_len, true, B_TGT, B_FA_TMP, B_FA_RNG, sc + S_G7, &T);       // :207-219
    if (rc == SCCG_OK) { SCCG_CK(cudaStreamWaitEvent(c->stream, c->ev[5], 0)); rc = fasta_ingest(c, d_rf, ref_file_len, false, B_REF, B_FA_TMP, B_FA_RNG, sc + S_G7, &R); }   // compression.cpp:193-200
    CompressResult res;
    if (rc == SCCG_OK) {
        const char* header = T.hdr_start >= 0 ? tgt_file + T.hdr_start : "";
        const int64_t nh = T.hdr_start >= 0 ? T.hdr_end - T.hdr_start : 0;
        rc = compress_device(c, R.d_seq, R.len, T.d_seq, T.len, header, nh, &res, nullptr);
    }
    SCCG_CK(cudaStreamSynchronize(c->s_h2d));                                 // the caller's buffers are no longer in use
    if (rc != SCCG_OK) return rc;
    SCCG_CK(cudaEventRecord(c->ev[6], c->stream));
    SCCG_TRY(deliver(c, res.d_out, res.out_len, dst, dst_cap, out, out_len));
    SCCG_CK(cudaEventRecord(c->ev[7], c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    cudaEventElapsedTime(&c->prof.h2d_ms, c->ev[4], c->ev[5]);
    cudaEventElapsedTime(&c->prof.d2h_ms, c->ev[6], c->ev[7]);
    if (mode_out) *mode_out = res.mode;
    return res.stoi_failed ? stoi_failure() : SCCG_OK;
}

int sccg_compress_fasta(sccg_ctx* c, const char* ref_file, int64_t ref_file_len, const char* tgt_file, int64_t tgt_file_len,
                        char** out, int64_t* out_len, int* mode_out) {
    if (!out) return set_error(SCCG_E_ARG, "null argument");
    return compress_fasta_impl(c, ref_file, ref_file_len, tgt_file, tgt_file_len, nullptr, 0, out, out_len, mode_out);
}

int sccg_compress_fasta_into(sccg_ctx* c, const char* ref_file, int64_t ref_file_len, const char* tgt_file, int64_t tgt_file_len,
                             char* out, int64_t out_cap, int64_t* out_len, int* mode_out) {
    if (!out) return set_error(SCCG_E_ARG, "null argument");
    return compress_fasta_impl(c, ref_file, ref_file_len, tgt_file, tgt_file_len, out, out_cap, nullptr, out_len, mode_out);
}

static int decompress_fasta_impl(sccg_ctx* c, const char* ref_file, int64_t ref_file_len, const char* inter, int64_t inter_len, char* dst, int64_t dst_cap,
                                 char** out, int64_t* out_len, const SinkSpec* sink) {
    if (!c || !out_len || (ref_file_len > 0 && !ref_file) || (inter_len > 0 && !inter)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_file_len, inter_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    u8* d_rf = nullptr;
    u32* sc = nullptr;
    SCCG_TRY(buf(c, B_SCALARS, (size_t)S_COUNT, &sc));
    SCCG_TRY(upload_file(c, B_FILE_R, ref_file, ref_file_len, &d_rf));
    FastaSeq R;
    SCCG_TRY(fasta_ingest(c, d_rf, ref_file_len, false, B_TGT, B_FA_TMP, B_FA_RNG, sc + S_G7, &R));      // decompression.cpp:47-58
    return decompress_host(c, nullptr, R.len, inter, inter_len, dst, dst_cap, out, out_len, R.d_seq, nullptr, sink);
}

int sccg_decompress_fasta(sccg_ctx* c, const char* ref_file, int64_t ref_file_len, const char* inter, int64_t inter_len, char** out, int64_t* out_len) {
    if (!out) return set_error(SCCG_E_ARG, "null argument");
    return decompress_fasta_impl(c, ref_file, ref_file_len, inter, inter_len, nullptr, 0, out, out_len, nullptr);
}

int sccg_decompress_fasta_into(sccg_ctx* c, const char* ref_file, int64_t ref_file_len, const char* inter, int64_t inter_len, char* out, int64_t out_cap,
                               int64_t* out_len) {
    if (!out) return set_error(SCCG_E_ARG, "null argument");
    return decompress_fasta_impl(c, ref_file, ref_file_len, inter, inter_len, out, out_cap, nullptr, out_len, nullptr);
}

int sccg_decompress_fasta_stream(sccg_ctx* c, const char* ref_file, int64_t ref_file_len, const char* inter, int64_t inter_len, sccg_sink_fn sink, void* user,
                                 int64_t* total_len) {
    if (!sink) return set_error(SCCG_E_ARG, "null argument");
    SinkSpec sp{sink, user};
    return decompress_fasta_impl(c, ref_file, ref_file_len, inter, inter_len, nullptr, 0, nullptr, total_len, &sp);
}

int sccg_decompress_stream(sccg_ctx* c, const char* ref_raw, int64_t ref_len, const char* inter, int64_t inter_len, sccg_sink_fn sink, void* user, int64_t* total_len) {
    if (!c || !sink || !total_len || (ref_len > 0 && !ref_raw) || (inter_len > 0 && !inter)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_len, inter_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    SinkSpec sp{sink, user};
    return decompress_host(c, ref_raw, ref_len, inter, inter_len, nullptr, 0, nullptr, total_len, nullptr, nullptr, &sp);
}

// ---- region extraction (csrc/sccg_extract.cuh) ----------------------------------------------------------------------------
int sccg_extract(sccg_ctx* c, const char* ref_raw, int64_t ref_len, const char* inter, int64_t inter_len, const sccg_region* regions, int64_t n_regions,
                 char* out, int64_t out_cap, int64_t* out_len, int64_t* seq_len) {
    if (!c || (ref_len > 0 && !ref_raw) || (inter_len > 0 && !inter)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_len, inter_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    return extract_host(c, ref_raw, ref_len, nullptr, inter, inter_len, regions, n_regions, out, out_cap, out_len, seq_len);
}

int sccg_extract_fasta(sccg_ctx* c, const char* ref_file, int64_t ref_file_len, const char* inter, int64_t inter_len, const sccg_region* regions,
                       int64_t n_regions, char* out, int64_t out_cap, int64_t* out_len, int64_t* seq_len) {
    if (!c || (ref_file_len > 0 && !ref_file) || (inter_len > 0 && !inter)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_file_len, inter_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    // the region list is checked before the reference FASTA goes to the device (argument errors come before any device work)
    SCCG_TRY(extract_check_regions(regions, n_regions, out, out_cap, out_len, seq_len));
    u8* d_rf = nullptr;
    u32* sc = nullptr;
    SCCG_TRY(buf(c, B_SCALARS, (size_t)S_COUNT, &sc));
    SCCG_TRY(upload_file(c, B_FILE_R, ref_file, ref_file_len, &d_rf));
    FastaSeq R;
    SCCG_TRY(fasta_ingest(c, d_rf, ref_file_len, false, B_TGT, B_FA_TMP, B_FA_RNG, sc + S_G7, &R));      // decompression.cpp:47-58
    return extract_host(c, nullptr, R.len, R.d_seq, inter, inter_len, regions, n_regions, out, out_cap, out_len, seq_len);
}

int sccg_extract_resident(sccg_ctx* c, const char* inter, int64_t inter_len, const sccg_region* regions, int64_t n_regions,
                          char* out, int64_t out_cap, int64_t* out_len, int64_t* seq_len) {
    if (!c || (inter_len > 0 && !inter)) return set_error(SCCG_E_ARG, "null argument");
    if (!c->res_ref_set) return set_error(SCCG_E_ARG, "no resident reference (call sccg_reference_set first)");
    SCCG_TRY(check_sizes(c->res_ref_len, inter_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    return extract_host(c, nullptr, c->res_ref_len, c->res_ref, inter, inter_len, regions, n_regions, out, out_cap, out_len, seq_len);
}

// ---- archives: record files decoded once and kept open on the device (csrc/sccg_extract.cuh) --------------------------------
int sccg_archive_open(sccg_ctx* c, const char* inter, int64_t inter_len, sccg_archive** out) {
    if (!c || !out || (inter_len > 0 && !inter)) return set_error(SCCG_E_ARG, "null argument");
    if (!c->res_ref_set) return set_error(SCCG_E_ARG, "no resident reference (call sccg_reference_set first)");
    SCCG_TRY(check_sizes(c->res_ref_len, inter_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    return archive_open(c, inter, inter_len, out);
}

int sccg_archive_info(const sccg_archive* a, int64_t* seq_len, int* mode, int64_t* device_bytes) {
    if (!a) return set_error(SCCG_E_ARG, "null argument");
    if (seq_len) *seq_len = a->g.Lm;
    if (mode) *mode = a->mode;
    if (device_bytes) *device_bytes = a->device_bytes;
    return SCCG_OK;
}

int sccg_archive_close(sccg_ctx* c, sccg_archive* a) {
    if (!c || !a) return set_error(SCCG_E_ARG, "null argument");
    if (a->ctx != c) return set_error(SCCG_E_ARG, "the archive was opened on another context");
    SCCG_CK(cudaSetDevice(c->device));
    SCCG_CK(cudaStreamSynchronize(c->main_stream));
    archive_unlink(c, a);
    archive_free(a);
    return SCCG_OK;
}

int sccg_archive_extract(sccg_ctx* c, sccg_archive* const* archives, int64_t n_archives, const sccg_query* queries, int64_t n_queries,
                         char* out, int64_t out_cap, int64_t* out_len) {
    if (!c) return set_error(SCCG_E_ARG, "null argument");
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    const int rc = archive_extract_impl(c, archives, n_archives, queries, n_queries, out, out_cap, out_len);
    if (rc != SCCG_OK) cudaStreamSynchronize(c->main_stream);              // no copy into the caller's buffer stays in flight
    return rc;
}

int sccg_archive_search(sccg_ctx* c, sccg_archive* const* archives, int64_t n_archives, const sccg_window* windows, int64_t n_windows,
                        const char* patterns, const int64_t* pattern_off, int64_t n_patterns, int max_mismatches, int strands,
                        sccg_hit* hits, int64_t hits_cap, int64_t* n_hits) {
    if (!c) return set_error(SCCG_E_ARG, "null argument");
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    const int rc = archive_search_impl(c, archives, n_archives, windows, n_windows, patterns, pattern_off, n_patterns, max_mismatches,
                                       strands, hits, hits_cap, n_hits);
    if (rc != SCCG_OK) cudaStreamSynchronize(c->main_stream);              // no copy into the caller's buffer stays in flight
    return rc;
}

int sccg_archive_search_edits(sccg_ctx* c, sccg_archive* const* archives, int64_t n_archives, const sccg_window* windows, int64_t n_windows,
                              const char* patterns, const int64_t* pattern_off, int64_t n_patterns, int max_edits, int strands,
                              sccg_edit_hit* hits, int64_t hits_cap, int64_t* n_hits) {
    if (!c) return set_error(SCCG_E_ARG, "null argument");
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    const int rc = archive_search_edits_impl(c, archives, n_archives, windows, n_windows, patterns, pattern_off, n_patterns, max_edits,
                                             strands, hits, hits_cap, n_hits);
    if (rc != SCCG_OK) cudaStreamSynchronize(c->main_stream);              // no copy into the caller's buffer stays in flight
    return rc;
}

int sccg_archive_variants(sccg_ctx* c, sccg_archive* const* archives, int64_t n_archives, const sccg_window* windows, int64_t n_windows,
                          sccg_variant* vars, int64_t vars_cap, int64_t* n_vars, char* alt, int64_t alt_cap, int64_t* alt_len) {
    if (!c) return set_error(SCCG_E_ARG, "null argument");
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    const int rc = archive_variants_impl(c, archives, n_archives, windows, n_windows, vars, vars_cap, n_vars, alt, alt_cap, alt_len);
    if (rc != SCCG_OK) cudaStreamSynchronize(c->main_stream);              // no copy into the caller's buffers stays in flight
    return rc;
}

int sccg_archive_liftover(sccg_ctx* c, sccg_archive* const* archives, int64_t n_archives, const sccg_lift_query* queries, int64_t n_queries,
                          sccg_lift* out) {
    if (!c) return set_error(SCCG_E_ARG, "null argument");
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    const int rc = archive_liftover_impl(c, archives, n_archives, queries, n_queries, out);
    if (rc != SCCG_OK) cudaStreamSynchronize(c->main_stream);              // no copy into the caller's buffer stays in flight
    return rc;
}

void* sccg_pinned_alloc(int64_t bytes) {
    void* p = nullptr;
    if (bytes <= 0 || cudaMallocHost(&p, (size_t)bytes) != cudaSuccess) { cudaGetLastError(); set_error(SCCG_E_NOMEM, "page-locked allocation failed"); return nullptr; }
    return p;
}
void sccg_pinned_free(void* p) { if (p) cudaFreeHost(p); }

int sccg_shard_match(sccg_ctx* c, const char* ref_slice, int64_t ref_len, const char* tgt_slice, int64_t tgt_len, int64_t seg_base, int is_last,
                     sccg_shard_info* info) {
    if (!c || !info || (ref_len > 0 && !ref_slice) || (tgt_len > 0 && !tgt_slice) || seg_base < 0) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_len, tgt_len));
    if ((seg_base + (tgt_len + SEG - 1) / SEG) * SEG >= 0x7fffffffLL) return set_error(SCCG_E_ARG, "sequence length must be in [0, 2^31-1)");
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    u8 *d_ref = nullptr, *d_tgt = nullptr;
    ChunkArrival arr;
    SCCG_TRY(enqueue_pair_upload(c, ref_slice, ref_len, tgt_slice, tgt_len, &d_ref, &d_tgt, &arr));
    ShardBorder* d_border = nullptr;
    int rc = shard_match(c, d_ref, ref_len, d_tgt, tgt_len, seg_base, is_last, &arr, &d_border);
    SCCG_CK(cudaStreamSynchronize(c->s_h2d));                                 // the caller's buffers are no longer in use
    if (rc != SCCG_OK) { c->shard.valid = 0; return rc; }
    ShardBorder hb;
    SCCG_CK(cudaMemcpyAsync(&hb, d_border, sizeof hb, cudaMemcpyDeviceToHost, c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    shard_info_from_border(hb, info);
    return SCCG_OK;
}

int sccg_shard_write(sccg_ctx* c, const sccg_shard_carry* carry, char** low_part, int64_t* low_len, char** body_part, int64_t* body_len) {
    if (!c || !carry || !low_part || !low_len || !body_part || !body_len) return set_error(SCCG_E_ARG, "null argument");
    SCCG_CK(cudaSetDevice(c->device));
    u8 *d_low = nullptr, *d_body = nullptr; i64 nl = 0, nb = 0;
    SCCG_TRY(shard_write(c, carry, &d_low, &nl, &d_body, &nb));
    SCCG_TRY(download(c, d_low, nl, low_part));
    int rc = download(c, d_body, nb, body_part);
    if (rc != SCCG_OK) { free(*low_part); *low_part = nullptr; return rc; }
    *low_len = nl; *body_len = nb;
    return SCCG_OK;
}

// ---- multi-GPU layer (csrc/sccg_mgpu.cuh) ---------------------------------------------------------------------------------
int sccg_mgpu_unique_id(char* id128) {
    if (!id128) return set_error(SCCG_E_ARG, "null argument");
    return mg_unique_id(id128);
}

int sccg_mgpu_init(sccg_ctx* c, const char* id128, int rank, int world, sccg_mgpu** out) {
    if (!c || !id128 || !out) return set_error(SCCG_E_ARG, "null argument");
    *out = nullptr;
    return mg_init(c, id128, rank, world, out);
}

void sccg_mgpu_destroy(sccg_mgpu* g) { mg_destroy(g); }
int sccg_mgpu_rank(const sccg_mgpu* g) { return g ? g->rank : -1; }
int sccg_mgpu_world(const sccg_mgpu* g) { return g ? g->world : 0; }

int sccg_mgpu_assign(const int64_t* lengths, int n_items, int world, int32_t* owner) {
    if (n_items < 0 || world < 1 || (n_items > 0 && (!lengths || !owner))) return set_error(SCCG_E_ARG, "invalid argument");
    mg_assign(lengths, n_items, world, owner);
    return SCCG_OK;
}

int sccg_mgpu_stash_device(sccg_mgpu* g, int32_t item, const void* d_data, int64_t len) {
    if (!g || len < 0 || (len > 0 && !d_data)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_CK(cudaSetDevice(g->ctx->device));
    return mg_stash(g, item, d_data, len);
}

// compress_genome of one pair of this rank; the encoded image stays on the device and joins the rank's outgoing streams
static int mg_compress_item(sccg_mgpu* g, int32_t item, const char* ref, int64_t ref_len, const char* tgt, int64_t tgt_len, const char* header, int64_t header_len,
                            int device_inputs, int64_t* enc_len, int* mode_out) {
    sccg_ctx* c = g->ctx;
    SCCG_TRY(check_sizes(ref_len, tgt_len));
    SCCG_TRY(check_header(header, header_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    CompressResult res;
    if (device_inputs) {
        if (((uintptr_t)ref | (uintptr_t)tgt) & 15) return set_error(SCCG_E_ARG, "device inputs must be 16-byte aligned");
        SCCG_TRY(compress_device(c, (const u8*)ref, ref_len, (const u8*)tgt, tgt_len, header, header_len < 0 ? 0 : header_len, &res, nullptr));
    } else {
        u8 *d_ref = nullptr, *d_tgt = nullptr;
        ChunkArrival arr;
        SCCG_TRY(enqueue_pair_upload(c, ref, ref_len, tgt, tgt_len, &d_ref, &d_tgt, &arr));
        int rc_c = compress_device(c, d_ref, ref_len, d_tgt, tgt_len, header, header_len < 0 ? 0 : header_len, &res, &arr);
        SCCG_CK(cudaStreamSynchronize(c->s_h2d));                             // the caller's buffers are no longer in use
        if (rc_c != SCCG_OK) return rc_c;
        cudaEventElapsedTime(&c->prof.h2d_ms, c->ev[4], c->ev[5]);
    }
    SCCG_TRY(mg_stash(g, item, res.d_out, res.out_len));
    if (enc_len) *enc_len = res.out_len;
    if (mode_out) *mode_out = res.mode;
    return res.stoi_failed ? stoi_failure() : SCCG_OK;
}

int sccg_mgpu_compress_item(sccg_mgpu* g, int32_t item, const char* ref, int64_t ref_len, const char* tgt, int64_t tgt_len, const char* header, int64_t header_len,
                            int64_t* enc_len, int* mode_out) {
    if (!g || (ref_len > 0 && !ref) || (tgt_len > 0 && !tgt) || (header_len > 0 && !header)) return set_error(SCCG_E_ARG, "null argument");
    return mg_compress_item(g, item, ref, ref_len, tgt, tgt_len, header, header_len, 0, enc_len, mode_out);
}

int sccg_mgpu_compress_item_device(sccg_mgpu* g, int32_t item, const void* d_ref, int64_t ref_len, const void* d_tgt, int64_t tgt_len, const char* header,
                                   int64_t header_len, int64_t* enc_len, int* mode_out) {
    if (!g || (ref_len > 0 && !d_ref) || (tgt_len > 0 && !d_tgt) || (header_len > 0 && !header)) return set_error(SCCG_E_ARG, "null argument");
    return mg_compress_item(g, item, (const char*)d_ref, ref_len, (const char*)d_tgt, tgt_len, header, header_len, 1, enc_len, mode_out);
}

int sccg_mgpu_gather(sccg_mgpu* g, char* out, int64_t out_cap, int32_t* item_ids, int64_t* item_offs, int64_t* item_lens, int32_t cap_items,
                     int32_t* n_items, int64_t* total) {
    if (!g) return set_error(SCCG_E_ARG, "null argument");
    if (g->rank == 0 && (!out || !item_ids || !item_offs || !item_lens)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_CK(cudaSetDevice(g->ctx->device));
    return mg_gather(g, out, out_cap, nullptr, item_ids, item_offs, item_lens, cap_items, n_items, total);
}

int sccg_mgpu_gather_device(sccg_mgpu* g, void** d_out, int32_t* item_ids, int64_t* item_offs, int64_t* item_lens, int32_t cap_items,
                            int32_t* n_items, int64_t* total) {
    if (!g) return set_error(SCCG_E_ARG, "null argument");
    if (g->rank == 0 && (!d_out || !item_ids || !item_offs || !item_lens)) return set_error(SCCG_E_ARG, "null argument");
    SCCG_CK(cudaSetDevice(g->ctx->device));
    return mg_gather(g, nullptr, 0, d_out, item_ids, item_offs, item_lens, cap_items, n_items, total);
}

// One pair, segment pairs spread over all ranks (compression.cpp:381-481 sharded by segment range).  Collective: every rank
// passes the same pair but only touches -- and only uploads -- its own slices.  Rank 0 receives the file image.
int sccg_mgpu_compress_sharded(sccg_mgpu* g, const char* ref, int64_t ref_len, const char* tgt, int64_t tgt_len, const char* header, int64_t header_len,
                               char* out, int64_t out_cap, int64_t* out_len, int* mode_out, int* sharded_out) {
    if (!g || !out_len || (ref_len > 0 && !ref) || (tgt_len > 0 && !tgt) || (header_len > 0 && !header)) return set_error(SCCG_E_ARG, "null argument");
    sccg_ctx* c = g->ctx;
    const int W = g->world, rank = g->rank;
    if (rank == 0 && !out) return set_error(SCCG_E_ARG, "null argument");
    SCCG_TRY(check_sizes(ref_len, tgt_len));
    SCCG_TRY(check_header(header, header_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    if (header_len < 0) header_len = 0;
    cudaStream_t s = c->main_stream;
    std::vector<i64> ra, rb;
    std::vector<sccg_shard_carry> carries;
    bool sharded = mg_segment_ranges(ref_len, tgt_len, W, &ra, &rb);
    if (sharded) {
        const i64 a = ra[rank], b = rb[rank];
        const int is_last = rank == W - 1;
        const i64 r_end = b * SEG < ref_len ? b * SEG : ref_len;
        const i64 rl = r_end - a * SEG, tl = is_last ? tgt_len - a * SEG : (b - a) * SEG;
        u8 *d_ref = nullptr, *d_tgt = nullptr;
        ChunkArrival arr;
        ShardBorder* d_border = nullptr;
        int rc = enqueue_pair_upload(c, ref + a * SEG, rl, tgt + a * SEG, tl, &d_ref, &d_tgt, &arr);
        if (rc == SCCG_OK) rc = shard_match(c, d_ref, rl, d_tgt, tl, a, is_last, &arr, &d_border);
        if (c->pipe_ready) cudaStreamSynchronize(c->s_h2d);                   // the caller's buffers are no longer in use
        const void* send = d_border;
        if (rc != SCCG_OK) {                                                  // a failed rank still takes part in the exchange and tells the others
            ShardBorder* eb = (ShardBorder*)g->h_meta;
            memset(eb, 0, sizeof *eb); eb->pad[0] = -1;
            SCCG_CK(cudaMemcpyAsync(g->d_meta, eb, sizeof *eb, cudaMemcpyHostToDevice, s));
            send = g->d_meta;
        }
        SCCG_TRY(g->tr->all_gather(send, g->d_border_all, sizeof(ShardBorder), s));
        SCCG_CK(cudaMemcpyAsync(g->h_border, g->d_border_all, sizeof(ShardBorder) * (size_t)W, cudaMemcpyDeviceToHost, s));
        SCCG_CK(cudaStreamSynchronize(s));
        if (rc != SCCG_OK) { c->shard.valid = 0; return rc; }
        for (int r = 0; r < W; ++r) if (g->h_border[r].pad[0] == -1) { c->shard.valid = 0; return set_error(SCCG_E_CUDA, "sharded compress: another rank failed in its match phase"); }
        sharded = mg_plan_carries(g->h_border, ra, rb, tgt_len, &carries);
    }
    g->last_sharded = sharded ? 1 : 0;
    if (sharded_out) *sharded_out = g->last_sharded;
    if (!sharded) {                                                           // T2 abort (-> global mode), '(' in the target, tiny pair: rank 0 alone
        c->shard.valid = 0;
        *out_len = 0;
        if (rank != 0) { if (mode_out) *mode_out = -1; return SCCG_OK; }
        return compress_host(c, ref, ref_len, tgt, tgt_len, header, header_len, out, out_cap, nullptr, out_len, mode_out);
    }
    // ---- write phase: sizes first (device), one all-gather tells every rank every size
    u8 *d_low = nullptr, *d_body = nullptr;
    i64 my_body = 0;
    u32* sc = (u32*)c->bufs[B_SCALARS].p;
    SCCG_TRY(shard_write_sizes(c, &carries[rank], &d_low));
    SCCG_TRY(g->tr->all_gather(sc, g->d_meta_all, 64, s));
    const u32* hs = (const u32*)(g->h_meta + MG_META_I64);
    SCCG_CK(cudaMemcpyAsync((void*)hs, g->d_meta_all, 64 * (size_t)W, cudaMemcpyDeviceToHost, s));
    SCCG_CK(cudaStreamSynchronize(s));
    SCCG_TRY(shard_write_body(c, hs[rank * 16 + S_BODY_MAIN], &d_body, &my_body));
    const i64 n_rseg = (ref_len + SEG - 1) / SEG, n_tseg = (tgt_len + SEG - 1) / SEG, n_iter = n_rseg < n_tseg ? n_rseg : n_tseg;
    const i64 leftover = n_tseg > n_iter ? tgt_len - n_iter * SEG : 0;
    std::vector<i64> low_len(W), body_len(W);
    i64 low_sum = 0, body_sum = 0;
    for (int r = 0; r < W; ++r) {
        low_len[r] = hs[r * 16 + S_LOW_TEXT]; body_len[r] = (i64)hs[r * 16 + S_BODY_MAIN] + (r == W - 1 ? leftover : 0);
        low_sum += low_len[r]; body_sum += body_len[r];
    }
    const i64 hdr_bytes = header_len > 0 ? header_len + 1 : 0;
    const i64 total = hdr_bytes + low_sum + 3 + body_sum;
    *out_len = rank == 0 ? total : 0;
    if (mode_out) *mode_out = 0;
    int rc = SCCG_OK;
    if (rank == 0) {
        if (total > out_cap) rc = set_error(SCCG_E_ARG, "output buffer too small (required size returned in *out_len)");
        SCCG_TRY(mg_grow(&g->d_recv, &g->recv_cap, (size_t)total + 64, 0, s));
        u8* img = g->d_recv;
        SCCG_TRY(write_header(c, img, header, header_len));
        char* sep = (char*)c->h_pinned + 12288;
        sep[0] = '\n'; sep[1] = ','; sep[2] = '\n';
        SCCG_CK(cudaMemcpyAsync(img + hdr_bytes + low_sum, sep, 3, cudaMemcpyHostToDevice, s));
        std::vector<MgP2P> recvs;
        i64 lo = hdr_bytes, bo = hdr_bytes + low_sum + 3;
        for (int r = 0; r < W; ++r) {
            if (r == 0) {
                if (low_len[0]) SCCG_CK(cudaMemcpyAsync(img + lo, d_low, (size_t)low_len[0], cudaMemcpyDeviceToDevice, s));
                if (body_len[0]) SCCG_CK(cudaMemcpyAsync(img + bo, d_body, (size_t)body_len[0], cudaMemcpyDeviceToDevice, s));
            } else {
                if (low_len[r]) recvs.push_back(MgP2P{img + lo, (size_t)low_len[r], r});
                if (body_len[r]) recvs.push_back(MgP2P{img + bo, (size_t)body_len[r], r});
            }
            lo += low_len[r]; bo += body_len[r];
        }
        SCCG_TRY(g->tr->p2p(nullptr, 0, recvs.data(), (int)recvs.size(), s));
        if (rc == SCCG_OK && total > 0) SCCG_CK(cudaMemcpyAsync(out, img, (size_t)total, cudaMemcpyDeviceToHost, s));
    } else {
        MgP2P sends[2]; int ns = 0;
        if (low_len[rank]) sends[ns++] = MgP2P{d_low, (size_t)low_len[rank], 0};
        if (body_len[rank]) sends[ns++] = MgP2P{d_body, (size_t)body_len[rank], 0};
        SCCG_TRY(g->tr->p2p(sends, ns, nullptr, 0, s));
    }
    SCCG_CK(cudaStreamSynchronize(s));
    if (c->pipe_ready) cudaEventElapsedTime(&c->prof.h2d_ms, c->ev[4], c->ev[5]);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]) == cudaSuccess) c->prof.match_ms = ms;
    return rc;
}

// the rank-th of world contiguous pieces of the reconstructed file image (sccg_decompress_part); nothing is gathered: every
// rank writes its piece at *part_offset of the output file
int sccg_mgpu_decompress_sharded(sccg_mgpu* g, const char* ref_raw, int64_t ref_len, const char* intermediate, int64_t inter_len,
                                 char* out, int64_t out_cap, int64_t* part_offset, int64_t* part_len, int64_t* total_len) {
    if (!g) return set_error(SCCG_E_ARG, "null argument");
    return sccg_decompress_part(g->ctx, ref_raw, ref_len, intermediate, inter_len, g->rank, g->world, out, out_cap, part_offset, part_len, total_len);
}

#ifdef SCCG_SEG_STATS
int sccg_debug_seg_stats(unsigned long long* out8, int reset) {
    if (cudaMemcpyFromSymbol(out8, sccg::g_seg_stats, sizeof(unsigned long long) * 8) != cudaSuccess) return -1;
    if (reset) { unsigned long long z[8] = {0}; if (cudaMemcpyToSymbol(sccg::g_seg_stats, z, sizeof z) != cudaSuccess) return -1; }
    return 0;
}
#endif
int sccg_decompress_part(sccg_ctx* c, const char* ref_raw, int64_t ref_len, const char* inter, int64_t inter_len, int part, int n_parts,
                         char* out, int64_t out_cap, int64_t* part_offset, int64_t* part_len, int64_t* total_len) {
    if (!c || !out || !part_offset || !part_len || !total_len || (ref_len > 0 && !ref_raw) || (inter_len > 0 && !inter)) return set_error(SCCG_E_ARG, "null argument");
    if (n_parts < 1 || part < 0 || part >= n_parts) return set_error(SCCG_E_ARG, "part index out of range");
    SCCG_TRY(check_sizes(ref_len, inter_len));
    SCCG_CK(cudaSetDevice(c->device));
    prof_reset(c);
    if (n_parts == 1) {
        *part_offset = 0;
        int rc = decompress_host(c, ref_raw, ref_len, inter, inter_len, out, out_cap, nullptr, part_len);
        *total_len = *part_len;
        return rc;
    }
    PartSpec ps; ps.part = part; ps.n_parts = n_parts; ps.part_off = part_offset; ps.total_len = total_len;
    return decompress_host(c, ref_raw, ref_len, inter, inter_len, out, out_cap, nullptr, part_len, nullptr, &ps);
}

#ifdef SCCG_SEG_TIMING
int sccg_debug_seg_timing(void* d_cycles) {
    unsigned long long* p = (unsigned long long*)d_cycles;
    return cudaMemcpyToSymbol(sccg::g_seg_cycles, &p, sizeof p) == cudaSuccess ? 0 : -1;
}
#endif

}  // extern "C"
