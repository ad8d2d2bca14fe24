// Shared device helpers: byte-SWAR on 64-bit words, decimal formatting, warp/block scans.
#pragma once
#include "sccg_compat.h"

namespace sccg {

typedef unsigned long long u64;
typedef unsigned int u32;
typedef unsigned short u16;
typedef unsigned char u8;
typedef long long i64;

static const int SEG = 1000;        // segment length L (compression.cpp:375)
static const int K1 = 14;           // primary k-mer length (compression.cpp:373)
static const int K2 = 10;           // secondary k-mer length (compression.cpp:374)
static const int GLOBAL_M = 100;    // global search distance m (compression.cpp:376)
static const int T2_LIMIT = 4;      // consecutive bad segments tolerated (compression.cpp:378)
static const int WRAP = 50;         // output line width (decompression.cpp:267)

#define SCCG_B01 0x0101010101010101ULL
#define SCCG_B7F 0x7f7f7f7f7f7f7f7fULL
#define SCCG_B80 0x8080808080808080ULL

// bit 7 of every byte that is an ASCII lowercase letter (C-locale islower, compression.cpp:345)
__device__ __forceinline__ u64 lower_flags8(u64 w) {
    u64 x = w & SCCG_B7F;
    u64 ge_a = x + (u64)(0x80 - 'a') * SCCG_B01;         // bit7 <=> (b & 0x7f) >= 'a'
    u64 gt_z = x + (u64)(0x80 - 'z' - 1) * SCCG_B01;     // bit7 <=> (b & 0x7f) >  'z'
    return ge_a & ~gt_z & ~w & SCCG_B80;
}
// ::toupper on 8 bytes (compression.cpp:369-370)
__device__ __forceinline__ u64 upper8(u64 w) { return w ^ (lower_flags8(w) >> 2); }
// ::tolower on 8 bytes: only 'A'..'Z' change (decompression.cpp:257)
__device__ __forceinline__ u64 lower8(u64 w) {
    u64 x = w & SCCG_B7F;
    u64 ge_a = x + (u64)(0x80 - 'A') * SCCG_B01;
    u64 gt_z = x + (u64)(0x80 - 'Z' - 1) * SCCG_B01;
    return w | ((ge_a & ~gt_z & ~w & SCCG_B80) >> 2);
}
// bit 7 of every non-zero byte
__device__ __forceinline__ u64 nonzero_flags8(u64 d) { return (((d & SCCG_B7F) + SCCG_B7F) | d) & SCCG_B80; }
// bit 7 of every byte equal to c
__device__ __forceinline__ u64 eq_flags8(u64 w, u8 c) { return ~nonzero_flags8(w ^ ((u64)c * SCCG_B01)) & SCCG_B80; }
// gathers the bit-7 flags of 8 bytes into 8 bits (byte j -> bit j)
__device__ __forceinline__ u32 movemask8(u64 flags) { return (u32)(((flags >> 7) * 0x0102040810204080ULL) >> 56); }

__device__ __forceinline__ u8 upper1(u8 c) { return (c >= 'a' && c <= 'z') ? (u8)(c - 32) : c; }
__device__ __forceinline__ u8 lower1(u8 c) { return (c >= 'A' && c <= 'Z') ? (u8)(c + 32) : c; }

// std::stoi(s[a..b)) as the reference calls it (compression.cpp:279, decompression.cpp:218-219): leading isspace skipped,
// optional sign, >= 1 digit, stops at the first non-digit, value must fit in int.  Returns false where stoi throws.
__device__ __forceinline__ bool dt_stoi(const u8* __restrict__ s, u32 a, u32 b, int* out) {
    while (a < b && (s[a] == ' ' || (s[a] >= 9 && s[a] <= 13))) ++a;
    bool neg = false;
    if (a < b && (s[a] == '-' || s[a] == '+')) { neg = s[a] == '-'; ++a; }
    if (a >= b || s[a] < '0' || s[a] > '9') return false;                     // invalid_argument
    i64 v = 0;
    while (a < b && s[a] >= '0' && s[a] <= '9') {
        v = v * 10 + (s[a] - '0');
        if (v > 2147483648LL) return false;                                    // out_of_range
        ++a;
    }
    if (neg) v = -v;
    if (v > 2147483647LL || v < -2147483648LL) return false;
    *out = (int)v;
    return true;
}

// number of characters operator<<(int) / std::to_string(int) prints
__device__ __forceinline__ int dec_len_u32(u32 v) {
    int n = 1;
    if (v >= 100000000u) { v /= 100000000u; n += 8; }
    if (v >= 10000u) { v /= 10000u; n += 4; }
    if (v >= 100u) { v /= 100u; n += 2; }
    if (v >= 10u) n += 1;
    return n;
}
__device__ __forceinline__ int dec_len_i32(int v) {
    return v < 0 ? 1 + dec_len_u32((u32)(-(i64)v)) : dec_len_u32((u32)v);
}
// writes v in decimal at dst, returns the number of characters written
__device__ __forceinline__ int write_dec_i32(u8* dst, int v) {
    u32 a = v < 0 ? (u32)(-(i64)v) : (u32)v;
    int n = dec_len_u32(a), off = 0;
    if (v < 0) { dst[0] = '-'; off = 1; }
    for (int i = n - 1; i >= 0; --i) { dst[off + i] = (u8)('0' + a % 10u); a /= 10u; }
    return off + n;
}

// 8 bytes at an arbitrary address (global or shared): two aligned loads + funnel shift.  Reads up to 15 bytes past p:
// every buffer this library allocates carries >= 64 bytes of slack.
__device__ __forceinline__ u64 ld_unaligned64(const u8* p) {
    uintptr_t a = (uintptr_t)p;
    const u64* q = reinterpret_cast<const u64*>(a & ~(uintptr_t)7);
    u32 sh = (u32)(a & 7) * 8u;
    u64 lo = q[0];
    if (sh == 0) return lo;
    return (lo >> sh) | (q[1] << (64u - sh));
}

__device__ __forceinline__ int lane_of() { return (int)(threadIdx.x & 31); }

// inclusive warp scan (all 32 lanes must call)
__device__ __forceinline__ u32 warp_scan_incl(u32 v) {
    const int lane = lane_of();
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        u32 y = __shfl_up_sync(SCCG_FULL_MASK, v, d);
        if (lane >= d) v += y;
    }
    return v;
}

// Exclusive block scan of one value per thread; blockDim.x <= 1024, multiple of 32; `total` = block sum.
// smem32: at least 33 u32 of shared scratch.  Contains three __syncthreads().
__device__ __forceinline__ u32 block_scan_excl(u32 v, u32* smem32, u32* total) {
    const int lane = lane_of(), w = (int)(threadIdx.x >> 5), nw = (int)(blockDim.x >> 5);
    u32 incl = warp_scan_incl(v);
    if (lane == 31) smem32[w] = incl;
    __syncthreads();
    if (w == 0) {
        u32 s = lane < nw ? smem32[lane] : 0u;
        u32 si = warp_scan_incl(s);
        smem32[lane] = si - s;               // exclusive warp offsets
        if (lane == 31) smem32[32] = si;
    }
    __syncthreads();
    u32 base = smem32[w];
    *total = smem32[32];
    __syncthreads();                         // smem32 may be reused by the caller right away
    return base + incl - v;
}

// Stream compaction, store side: every thread of the block keeps the bytes of its 16-byte piece (x, y) selected by the
// mask m; the block's kept bytes (tot of them, this thread's start at excl) go to dst[0 .. tot).  They are packed in shared
// memory at the same 16-byte phase as dst and leave as aligned 16-byte stores (byte stores only in the first and last
// partial block), instead of one global byte store per kept byte.  stage: 16-byte aligned, blockDim.x * 16 + 32 bytes.
__device__ __forceinline__ void block_compact_store(u8* stage, u8* __restrict__ dst, u32 excl, u32 m, u64 x, u64 y, u32 tot) {
    const u32 a = (u32)((uintptr_t)dst & 15);
    u32 pos = a + excl;
    if (m == 0xffffu && (pos & 3u) == 0u) {
        u32* s32 = reinterpret_cast<u32*>(stage + pos);
        s32[0] = (u32)x; s32[1] = (u32)(x >> 32); s32[2] = (u32)y; s32[3] = (u32)(y >> 32);
    } else {
        while (m) {
            const int b = __ffs((int)m) - 1; m &= m - 1;
            const u64 w = b < 8 ? x : y;
            stage[pos++] = (u8)(w >> (8 * (b & 7)));
        }
    }
    __syncthreads();
    u8* base = dst - a;                                    // 16-byte aligned; bytes [a, end) of the staged image belong to this block
    const u32 end = a + tot;
    for (u32 q = threadIdx.x * 16u; q < end; q += blockDim.x * 16u) {
        if (q >= a && q + 16u <= end) *reinterpret_cast<uint4*>(base + q) = *reinterpret_cast<const uint4*>(stage + q);
        else for (u32 b = q > a ? q : a; b < q + 16u && b < end; ++b) base[b] = stage[b];
    }
}

}  // namespace sccg
