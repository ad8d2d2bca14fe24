// Text-level delta_encode (compression.cpp:222-304) on the device.
//
// The record writers fuse the delta chain at RECORD level (DESIGN.md 4.8), which equals the reference's text-level
// pass whenever every '(' of the body belongs to a match token.  A target that carries a literal '(' (an inlined
// `>header (alt)` of a later FASTA record, SURVEY N2 / experiment J) makes the reference's `find('(')` / `find(')')`
// loop (:262-292) pair that literal with the next ')' and feed stoi with target symbols: the delta chain is poisoned
// or the program dies in stoi.  Parity means reproducing exactly that, so when the target contains '(' anywhere the
// writers emit the PRE-delta body (absolute p, what :406-415 / :564-573 write) and this pass replays :258-292 on it.
//
// The loop of the reference is sequential, but its only state is (cursor, previous_start_ref): one warp streams the
// body once -- wide ballot searches for the next '(' / ')' / ',', a serial stoi on <= 12 bytes, wide copies.  It is a
// rare-input path (one warp, ~1 GB/s on literal-heavy bodies) and is never taken for ACGTN targets.
#pragma once
#include "sccg_scan.cuh"

namespace sccg {

enum { DT_LEN = 0, DT_ERR = 1, DT_TOKENS = 2, DT_PARENS = 3 };     // u32 slots of the result block

// first index in [from, end) with s[idx] == ch, else `end`.  s is 8-byte aligned; the buffer has >= 8 readable bytes past
// `end`.  All 32 lanes, uniform arguments; 1 KB per round.
__device__ __forceinline__ u32 warp_find_byte(const u8* __restrict__ s, u32 from, u32 end, u8 ch) {
    const int lane = lane_of();
    const u64* w64 = reinterpret_cast<const u64*>(s);
    for (u32 w0 = from >> 3; (w0 << 3) < end; w0 += 128) {
        u32 m[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const u32 wi = w0 + (u32)lane + 32u * (u32)u;
            const u32 b = wi << 3;
            u32 mm = 0;
            if (b < end) {
                mm = movemask8(eq_flags8(w64[wi], ch));
                if (b < from) mm &= 0xffu << (from - b);               // bytes before `from`
                if (end - b < 8) mm &= (1u << (end - b)) - 1u;         // bytes at or past `end`
            }
            m[u] = mm;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            u32 bal = __ballot_sync(SCCG_FULL_MASK, m[u] != 0u);
            if (bal) {
                int src = __ffs((int)bal) - 1;
                u32 mm = __shfl_sync(SCCG_FULL_MASK, m[u], src);
                return ((w0 + (u32)src + 32u * (u32)u) << 3) + (u32)(__ffs((int)mm) - 1);
            }
        }
    }
    return end;
}

// dst[0..len) = src[0..len); all 32 lanes, uniform arguments; the source buffer has >= 16 readable bytes past its end
__device__ __forceinline__ void warp_copy_bytes(u8* __restrict__ dst, const u8* __restrict__ src, u32 len) {
    const int lane = lane_of();
    if (len < 64) {
        for (u32 x = (u32)lane; x < len; x += 32) dst[x] = src[x];
        return;
    }
    u32 head = (u32)((8 - ((uintptr_t)dst & 7)) & 7);                  // bytes until dst is 8-byte aligned
    if ((u32)lane < head) dst[lane] = src[lane];
    const u32 words = (len - head) >> 3;
    u64* d64 = reinterpret_cast<u64*>(dst + head);
    const u8* s = src + head;
    for (u32 w = (u32)lane; w < words; w += 32) d64[w] = ld_unaligned64(s + 8 * (size_t)w);
    const u32 done = head + (words << 3);
    if (done + (u32)lane < len) dst[done + lane] = src[done + lane];   // < 8 tail bytes
}

// in[start..end) -> out (written from out[0]); res[DT_LEN] = bytes written, res[DT_ERR] != 0 iff stoi would have thrown
// (then the reference leaves the file un-rewritten and exits 1).  `in` is the 8-byte aligned file image, offsets are
// absolute.  One warp.
__global__ void __launch_bounds__(32) delta_text_k(const u8* __restrict__ in, u32 start, u32 end, u8* __restrict__ out, u32* __restrict__ res) {
    const int lane = lane_of();
    u32 cur = start;                          // everything before `cur` has been emitted
    u32 o = 0;
    u32 prev = 0;                             // previous_start_ref (:258), int arithmetic modulo 2^32
    u32 ntok = 0;
    bool err = false;
    while (cur < end) {
        const u32 open = warp_find_byte(in, cur, end, '(');                   // :263
        if (open >= end) break;
        const u32 sp = open + 1;                                              // start_pos :267
        const u32 close = warp_find_byte(in, sp, end, ')');                   // :268
        if (close >= end) break;                                              // :269-270
        const u32 comma = warp_find_byte(in, sp, close, ',');                 // :273 token.find(',')
        if (comma >= close) {                                                 // :274-277 no comma: resume after the ')'
            warp_copy_bytes(out + o, in + cur, close + 1 - cur);
            o += close + 1 - cur; cur = close + 1;
            continue;
        }
        int p = 0;
        if (!dt_stoi(in, sp, comma, &p)) { err = true; break; }               // :279 throws
        const u32 delta = (u32)p - prev;                                      // :280
        prev = (u32)p;                                                        // :282
        warp_copy_bytes(out + o, in + cur, sp - cur);                         // text up to and including '('
        o += sp - cur;
        const int w = dec_len_i32((int)delta);
        if (lane == 0) write_dec_i32(out + o, (int)delta);                    // :284 to_string(delta)
        __syncwarp();
        o += (u32)w;
        warp_copy_bytes(out + o, in + comma, close - comma);                  //      + token.substr(comma_pos)
        o += close - comma;
        cur = close;                                                          // :292 the search resumes at the ')'
        ++ntok;
    }
    if (!err && cur < end) { warp_copy_bytes(out + o, in + cur, end - cur); o += end - cur; }
    if (lane == 0) { res[DT_LEN] = o; res[DT_ERR] = err ? 1u : 0u; res[DT_TOKENS] = ntok; }
}

// res[DT_PARENS] += number of '(' in s[start..end): bound for the size of the rewritten body
__global__ void __launch_bounds__(256) count_parens_k(const u8* __restrict__ s, u32 start, u32 end, u32* __restrict__ res) {
    u32 cnt = 0;
    for (u32 i = start + blockIdx.x * blockDim.x + threadIdx.x; i < end; i += gridDim.x * blockDim.x) cnt += s[i] == '(';
    cnt = __reduce_add_sync(SCCG_FULL_MASK, cnt);
    if (lane_of() == 0 && cnt) atomicAdd(&res[DT_PARENS], cnt);
}

// Replays delta_encode on the pre-delta file image d_file[0..file_len) whose body starts at body_base.  On success
// *d_final / *final_len describe the rewritten image (a different buffer); *stoi_failed reports the reference's exception.
static int delta_text_pass(sccg_ctx* c, const u8* d_file, i64 file_len, u32 body_base, u32* sc_res, u8** d_final, i64* final_len, bool* stoi_failed) {
    SCCG_CK(cudaMemsetAsync(sc_res, 0, sizeof(u32) * 4, c->stream));
    const u32 end = (u32)file_len;
    if (end > body_base) {
        unsigned g = div_up((i64)end - body_base, 256 * 64);
        unsigned capg = (unsigned)c->sm_count * 8u;
        LAUNCH(c, count_parens_k, dim3(g < capg ? g : capg), dim3(256), 0, d_file, body_base, end, sc_res);
    }
    SCCG_CK(cudaMemcpyAsync(c->h_pinned, sc_res, sizeof(u32) * 4, cudaMemcpyDeviceToHost, c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    const u64 parens = ((u32*)c->h_pinned)[DT_PARENS];
    const u64 cap = (u64)file_len + 11ull * parens + 64;                      // to_string(delta) is at most 11 characters
    if (cap >= 0xffffffffull) return set_error(SCCG_E_ARG, "encoded output would exceed 4 GiB");
    u8* fin = nullptr;
    SCCG_TRY(buf(c, B_OUT2, (size_t)cap, &fin));
    if (body_base) SCCG_CK(cudaMemcpyAsync(fin, d_file, body_base, cudaMemcpyDeviceToDevice, c->stream));
    LAUNCH(c, delta_text_k, dim3(1), dim3(32), 0, d_file, body_base, end, fin + body_base, sc_res);
    SCCG_CK(cudaMemcpyAsync(c->h_pinned, sc_res, sizeof(u32) * 4, cudaMemcpyDeviceToHost, c->stream));
    SCCG_CK(cudaStreamSynchronize(c->stream));
    const u32* h = (const u32*)c->h_pinned;
    *stoi_failed = h[DT_ERR] != 0;
    *d_final = fin;
    *final_len = (i64)body_base + h[DT_LEN];
    return SCCG_OK;
}

}  // namespace sccg
