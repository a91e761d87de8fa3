// pfp_table.cuh -- the dictionary table of K3, shared by the stand-alone insert kernel
// (pfp_phrase.cu) and the insert fused into the streaming K2 pass (pfp_stream.cu).
#pragma once
#include "pfp_common.cuh"
#include "pfp_stages.cuh"
#include "pfp_fp.cuh"

// Open addressing, linear probing, 16-byte slots {key, val, check}; key 0 = empty.
// A warp first groups its lanes by key (match.any) so that runs of identical phrases cost one
// atomic per warp instead of 32.  `chk` is a 32-bit digest of the full 128-bit fingerprint and
// the length, independent of the key: every phrase that lands in a slot must agree with it, or
// the parse stops with PFPB200_E_COLLISION (the reference compares strings, newscan.cpp:282-286).
// `val` is the word's occurrence count in table_insert_k, and word id + 1 in the fused K2 pass
// (0 until its creator stored it).
struct __align__(16) DictSlot { u64 key; u32 val; u32 chk; };
constexpr u32 TABLE_MAX_PROBES = 2048;
constexpr u32 UID_PENDING = 0x80000000u;       // fused K2 pass: uid[j] = UID_PENDING | slot, resolved by table_pending_k

__device__ __forceinline__ u32 check_of(const PhraseFp &r) {
    u64 x = (r.fpa + 0x632BE59BD9B4E019ULL) * 0xD1342543DE82EF95ULL;
    x ^= (rotl64(r.fpb, 23) + 0x2545F4914F6CDD1DULL) * 0xAF251AF3B0F025B5ULL;
    x ^= x >> 29;
    u32 c = (u32)(x ^ (x >> 32));
    return c ? c : 1u;
}

int pfp_table_init(pfpb200_ctx *ctx, DictSlot *tab, u64 cap);     // all slots empty (pfp_phrase.cu)

// One probe sequence: a plain 16-byte load of the slot first -- on repetitive inputs nine phrases
// in ten find their word already there and finish with one fire-and-forget add to its count --
// and a CAS only on an empty slot.  The thread that wins the CAS is the word's creator.  Word ids
// are not handed out here: table_insert_k leaves the slot in uid[] with a creator bit, and
// table_compact_k numbers the words afterwards, in the order of their creators' records (one scan
// over the records, no counter that every creator has to wait for).
struct Probe { u64 slot; bool placed; bool creator; u32 seen_chk; u32 seen_val; };

__device__ __forceinline__ Probe table_probe(DictSlot *__restrict__ tab, u64 cap, u64 slot, uint4 sv, u64 k) {
    Probe r{slot, false, false, 0u, 0u};
    u32 probes = 0;
    for (;;) {
        const u64 key = ((u64)sv.y << 32) | sv.x;
        if (key == k) { r.placed = true; r.seen_val = sv.z; r.seen_chk = sv.w; break; }
        if (key == 0ull) {
            const u64 prev = atomicCAS((unsigned long long *)&tab[r.slot].key, 0ull, (unsigned long long)k);
            if (prev == 0ull) { r.placed = true; r.creator = true; break; }
            if (prev == k) { r.placed = true; break; }
        }
        if (++probes > TABLE_MAX_PROBES) break;               // table too small for this input
        r.slot = (r.slot + 1 == cap) ? 0 : r.slot + 1;
        sv = __ldcg(reinterpret_cast<const uint4 *>(tab + r.slot));
    }
    return r;
}

