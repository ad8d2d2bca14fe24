// Context, grow-only device buffers, error plumbing, launch accounting.
#pragma once
#include "sccg_common.cuh"
#include "../../include/sccg.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>

namespace sccg {

static thread_local std::string g_last_error;

static int set_error(int code, const char* fmt, const char* a = "", const char* b = "") {
    char buf[512];
    snprintf(buf, sizeof buf, fmt, a, b);
    g_last_error = buf;
    return code;
}

#define SCCG_CK(call)                                                                               \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess) return sccg::set_error(SCCG_E_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

// grow-only device buffer slots (one cudaMalloc per slot after warm-up)
enum Slot {
    B_REF = 0, B_TGT, B_OUT, B_OUT2, B_SEGINFO, B_MATCH, B_SEGBYTES, B_SEGPREV, B_SCAN0, B_SCAN1, B_SCAN2, B_SCAN3, B_SCALARS,
    B_RUN_CNT, B_RUN_MASK, B_NRUN_MASK, B_RUN_START, B_RUN_END, B_RUN_BYTES, B_RUN_TEXT, B_NRUN_CNT, B_NRUN_START, B_NRUN_END, B_NRUN_BYTES, B_NRUN_TEXT,
    B_ENC, B_NIDX, B_LOW, B_TOK_FLAG, B_TOK_POS, B_ITEM_OFF, B_ITEM_SRC, B_NUM0, B_NUM1, B_NUM2, B_NUM3, B_NUM4, B_NUM5,
    B_LRUN_S, B_LRUN_E, B_NRUNS_S, B_NRUNS_E, B_NRUNS_CUM, B_TILE0, B_TILE1, B_TILE2, B_TILE3, B_SEG_PTR, B_TILE_WIN, B_FILE_R, B_FILE_T, B_FA_TMP, B_FA_RNG, B_NEED,
    B_GREF, B_GTGT, B_GKEYS, B_GVALS, B_GKEYS2, B_GVALS2, B_GHIST, B_GOFFS, B_GBUCKET, B_GREC, B_GLIT, B_GTMP0, B_GTMP1, B_GTMP2, B_GTMP3, B_GFIRST, B_SHARD,
    B_EXT_REG, B_EXT_IV, B_SRCH_TAB, B_SRCH_REG, B_SRCH_TILE, B_SRCH_HITS,
    B_VR_AGG, B_VR_SC, B_VR_TAB, B_VR_KEY, B_VR_CNT, B_VR_ANC, B_VR_GAP, B_VR_TILE, B_VR_REC3, B_VR_P, B_VR_WIN, B_VR_OUT,
    B_LT_LO, B_LT_X, B_LT_Q, B_LT_OUT,
    B_NSLOTS
};

struct DevBuf { void* p; size_t cap; };

}  // namespace sccg

namespace sccg {
// what sccg_shard_match leaves behind for sccg_shard_write (the device buffers stay in their slots)
struct ShardState { int valid; const unsigned char* d_tgt; long long nt; int n_iter; long long seg_base; int is_last; unsigned low_k; long long leftover; };
}

struct sccg_ctx {
    int device;
    int sm_count;
    cudaStream_t stream;
    sccg::DevBuf bufs[sccg::B_NSLOTS];
    void* h_pinned;            // small pinned staging area for scalars
    size_t h_pinned_cap;
    cudaEvent_t ev[8];
    cudaEvent_t ev_x[4];           // phase marks inside a call (global mode: index / parse; multi-GPU: exchange)
    sccg_profile prof;
    unsigned scan_epoch[2];        // single-pass scan, per lane (0 = main stream, 1 = side stream): epoch of the last launch,
    unsigned scan_counter_base[2]; //   tiles handed out so far
    int scan_counter_ready[2];
    cudaStream_t main_stream, side_stream;   // `stream` is the lane the helpers currently enqueue on (main_stream except inside SideLane)
    cudaEvent_t ev_side[6];
    unsigned char* res_ref; long long res_ref_len; size_t res_ref_cap; int res_ref_set;      // resident reference (sccg_reference_set): raw symbols, kept across calls
    int use_diag;                  // seg_match_k: try the diagonal-hypothesis parse first (SCCG_NO_DIAG=1 disables it)
    cudaStream_t s_h2d, s_d2h;     // copy streams of the pipelined host entry points (created on first use)
    cudaEvent_t ev_pipe[2], ev_h2d[64], ev_g[64], ev_d2h[64];
    void* h_stream[2]; size_t h_stream_cap;      // page-locked double buffer of the streaming decompressor (sccg_decompress*_stream)
    int pipe_ready;
    sccg::ShardState shard;
    void* h_ext; size_t h_ext_cap;   // page-locked staging of the region tables (sccg_extract*, sccg_archive_extract, sccg_archive_search), grow-only
    unsigned res_gen;                // resident reference generation: sccg_reference_set / _clear advance it (archives opened before go stale)
    unsigned char* res_form[2]; long long res_form_len[2];   // the resident reference as archives read it: [0] upper-cased (local-mode
                                                              // files), [1] N-stripped and upper-cased (global mode); built at first need
    sccg_archive* archives;          // open archives (sccg_destroy releases them)
    void* res_nrun; long long res_nrun_k;   // the resident reference's N runs for sccg_archive_variants (sccg_variants.cuh), built at first need
};

namespace sccg {

static int buf_reserve(sccg_ctx* c, int slot, size_t bytes, void** out) {
    DevBuf& b = c->bufs[slot];
    bytes = (bytes + 255) & ~(size_t)255;
    if (bytes < 256) bytes = 256;
    if (b.cap < bytes) {
        if (b.p) { cudaFree(b.p); b.p = nullptr; b.cap = 0; }
        size_t want = bytes + bytes / 8;                       // a little headroom against regrowth
        cudaError_t e = cudaMalloc(&b.p, want);
        if (e != cudaSuccess) { cudaGetLastError(); e = cudaMalloc(&b.p, want = bytes); }
        if (e != cudaSuccess) { b.p = nullptr; return set_error(SCCG_E_NOMEM, "cudaMalloc failed: %s", cudaGetErrorString(e)); }
        b.cap = want;
    }
    *out = b.p;
    return SCCG_OK;
}
template <typename T> static int buf(sccg_ctx* c, int slot, size_t count, T** out) {
    void* p = nullptr;
    int rc = buf_reserve(c, slot, count * sizeof(T) + 64, &p);   // +64: vector loads may run past the end
    *out = (T*)p;
    return rc;
}

#define SCCG_TRY(expr) do { int rc_ = (expr); if (rc_ != SCCG_OK) return rc_; } while (0)

// every kernel launch goes through here so that gpu_launches can be reported
#define LAUNCH(ctx, kernel, grid, block, smem, ...)                      \
    do {                                                                 \
        SCCG_LAUNCH(kernel, grid, block, smem, (ctx)->stream, __VA_ARGS__); \
        (ctx)->prof.launches++;                                          \
    } while (0)

static inline unsigned div_up(long long a, long long b) { return (unsigned)((a + b - 1) / b); }

// copies a host buffer into a grow-only device slot (pageable source: cudaMemcpyAsync stages it)
static int upload(sccg_ctx* c, int slot, const void* h, i64 n, u8** d) {
    SCCG_TRY(buf(c, slot, (size_t)n + 64, d));
    if (n > 0) SCCG_CK(cudaMemcpyAsync(*d, h, (size_t)n, cudaMemcpyHostToDevice, c->stream));
    return SCCG_OK;
}

static int download(sccg_ctx* c, const u8* d, i64 n, char** out) {
    char* h = (char*)malloc((size_t)n + 1);
    if (!h) return set_error(SCCG_E_NOMEM, "malloc of the result failed");
    if (n > 0) {
        cudaError_t e = cudaMemcpyAsync(h, d, (size_t)n, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) { free(h); return set_error(SCCG_E_CUDA, "result download failed: %s", cudaGetErrorString(e)); }
    }
    h[n] = 0;
    *out = h;
    return SCCG_OK;
}

// Independent work (the lowercase-run pipeline of compress) is enqueued on a second stream so that it runs underneath the
// ALU-bound segment matcher: inside a SideLane scope every helper that uses c->stream targets the side stream.
struct SideLane {
    sccg_ctx* c;
    explicit SideLane(sccg_ctx* ctx) : c(ctx) { c->stream = c->side_stream; }
    ~SideLane() { c->stream = c->main_stream; }
};
static inline int lane_of_stream(const sccg_ctx* c) { return c->stream == c->side_stream ? 1 : 0; }

// copy streams and events of the pipelined host entry points
static int pipe_streams(sccg_ctx* c) {
    if (c->pipe_ready) return SCCG_OK;
    SCCG_CK(cudaStreamCreate(&c->s_h2d));
    SCCG_CK(cudaStreamCreate(&c->s_d2h));
    for (int i = 0; i < 2; ++i) SCCG_CK(cudaEventCreate(&c->ev_pipe[i]));
    for (int i = 0; i < 64; ++i) { SCCG_CK(cudaEventCreate(&c->ev_h2d[i])); SCCG_CK(cudaEventCreate(&c->ev_g[i])); SCCG_CK(cudaEventCreate(&c->ev_d2h[i])); }
    c->pipe_ready = 1;
    return SCCG_OK;
}
// reference chunk of the pipelined upload: <= 32 chunks, multiples of 1 MiB (SCCG_PIPE_CHUNK overrides it, tests use tiny chunks)
static i64 pipe_chunk_bytes(i64 n) {
    i64 ch = 16ll << 20;
    if (const char* e = getenv("SCCG_PIPE_CHUNK")) { long long v = atoll(e); if (v >= 4096) ch = (v + 4095) & ~4095ll; }
    while ((n + ch - 1) / ch > 32) ch *= 2;
    return ch;
}
// output chunk of the pipelined download in gather tiles (4 KiB each): <= 32 chunks
static unsigned pipe_tiles_per_chunk(unsigned ntiles) {
    unsigned t = 4096;                                             // 16 MiB
    if (const char* e = getenv("SCCG_PIPE_CHUNK")) { long long v = atoll(e); if (v >= 4096) t = (unsigned)((v + 4095) / 4096); }
    while ((ntiles + t - 1) / t > 32) t *= 2;
    return t;
}

// result delivery: either into a buffer of the caller (dst != NULL; pin it for full PCIe speed) or into a fresh malloc
static int deliver(sccg_ctx* c, const u8* d, i64 n, char* dst, i64 dst_cap, char** out_alloc, int64_t* out_len) {
    *out_len = n;
    if (!dst) return download(c, d, n, out_alloc);
    if (dst_cap < n) return set_error(SCCG_E_ARG, "output buffer too small (required size returned in *out_len)");
    if (n > 0) {
        SCCG_CK(cudaMemcpyAsync(dst, d, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
        SCCG_CK(cudaStreamSynchronize(c->stream));
    }
    return SCCG_OK;
}



}  // namespace sccg
