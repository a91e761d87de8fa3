// pfp_fp.cuh -- the phrase fingerprint (stands in for kr_hash(), newscan.cpp:229-239) shared by
// the streaming kernel, the border/long-phrase kernel and the dictionary stages.
//
// A phrase is cut into 16-byte chunks c = 0,1,.. from its first byte (zero padded behind its
// end); chunk c lies in segment c >> 9 (8 KB) and uses NH key words 4*(c & 511)...  Two NH sums
// (UMAC's universal family over 32-bit words, the second with the key shifted by one chunk,
// "Toeplitz") are taken per segment and the segments are combined as
//     fp = sum_seg FOLD^seg * NH(seg)      (mod 2^64, FOLD odd),
// which is additive over ANY partition of the chunks -- what lets a streaming pass hand the
// pieces of one phrase to different threads, warps and tiles and just add them up.
#pragma once
#include "pfp_common.cuh"
#include "pfp_stages.cuh"

__device__ __forceinline__ u64 rotl64(u64 x, int r) { return (x << r) | (x >> (64 - r)); }
__device__ __forceinline__ u64 fmix64(u64 k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdULL;
    k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL;
    k ^= k >> 33;
    return k;
}

// never 0: 0 marks an empty slot of the dictionary table
__device__ __forceinline__ u64 sort_key_of(u64 fa, u64 fb) {
    u64 k = fmix64(fa ^ rotl64(fb, 29) ^ 0x9E3779B97F4A7C15ULL);
    return k ? k : 0x9E3779B97F4A7C15ULL;
}

// 32-bit digest of the 128-bit fingerprint, independent of the table key: words that share a key
// must agree on it (never 0: 0 marks a slot whose digest is not written yet)
__device__ __forceinline__ u32 check_of(const PhraseFp &r) {
    u64 x = (r.fpa + 0x632BE59BD9B4E019ULL) * 0xD1342543DE82EF95ULL;
    x ^= (rotl64(r.fpb, 23) + 0x2545F4914F6CDD1DULL) * 0xAF251AF3B0F025B5ULL;
    x ^= x >> 29;
    u32 c = (u32)(x ^ (x >> 32));
    return c ? c : 1u;
}

__device__ __forceinline__ void store_rec(PhraseFp *rec, u64 j, u64 fa, u64 fb) {
    *reinterpret_cast<uint4 *>(rec + j) = make_uint4((u32)fa, (u32)(fa >> 32), (u32)fb, (u32)(fb >> 32));
}

// base^e mod 2^64 (long phrases only)
static __device__ __noinline__ u64 fold_pow(u64 base, u32 e) {
    u64 r = 1;
    while (e) {
        if (e & 1u) r *= base;
        base *= base;
        e >>= 1;
    }
    return r;
}
