// pfp_phrase.cu -- K2 in its per-phrase form, K3 dictionary table, phrase pool, dictionary merge.
//
// K2 replaces save_update_word() (newscan.cpp:245-304): from consecutive trigger positions it
// derives every phrase (start, length), its `.last` byte (:296) and `.sai` value (:299-301), and
// a fingerprint standing in for kr_hash() (:229-239).  The reference's 64-bit hash only ever
// reaches the private .parse_old file, so its VALUE is not part of the contract; what matters is
// that equal phrases get equal ids and different phrases different ones.  The fingerprint is
// two NH sums (UMAC's universal family: sum of (x_2i + k_2i)(x_2i+1 + k_2i+1) mod 2^64 over
// 32-bit words, Toeplitz-shifted keys), segments of 8 KB weighted by powers of an odd constant,
// plus the length (pfp_fp.cuh).  The streaming form of K2 (pfp_stream.cu) is what normally runs;
// the kernels here take over for w > 32, for tiles denser than it handles, and for the listed
// phrases (borders, very long ones).
//
// K3 replaces the std::map<uint64_t,word_stats> updates (:256-288) with an open-addressing table
// in HBM (table_insert_k) and numbers the words in the text order of their creators with one scan
// over the records (table_compact_k); a collision of the 64-bit key is detected through an
// independent check digest, as the reference detects its own (:282-286).
#include "pfp_common.cuh"
#include "pfp_stages.cuh"
#include "pfp_fp.cuh"
#include <stdlib.h>

// 16 bytes of a phrase at phrase offset o (multiple of 16), zero beyond the phrase end.
// fast path: aligned 32-bit loads + funnel shift by the byte misalignment of the phrase start
__device__ __forceinline__ void load_chunk(const TextView &tv, i64 s0, u64 len, u64 o, bool special,
                                           u32 x[4]) {
    const u32 nbv = (u32)((len - o) < 16 ? (len - o) : 16);
    if (!special) {
        const i64 loc = s0 + (i64)o - tv.pos0;            // offset of the chunk in the buffer
        const u8 *p = tv.T + loc;
        const u32 bs = (u32)((uintptr_t)p & 3);
        const u32 *p4 = reinterpret_cast<const u32 *>(p - bs);
        u32 W[5];
        if ((u64)loc + 20 <= tv.n_buf) {                  // interior: five unconditional loads
#pragma unroll
            for (int j = 0; j < 5; j++) W[j] = __ldg(p4 + j);
        } else {
            const u32 need = bs + nbv;                    // bytes needed counted from p4
#pragma unroll
            for (int j = 0; j < 5; j++) W[j] = (4u * j < need) ? __ldg(p4 + j) : 0u;
        }
#pragma unroll
        for (int j = 0; j < 4; j++) x[j] = __funnelshift_r(W[j], W[j + 1], 8 * bs);
    } else {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            u32 v = 0;
            for (int b = 0; b < 4; b++) {
                u32 k = 4 * j + b;
                if (k < nbv) v |= (u32)tv_byte(tv, s0 + (i64)o + k) << (8 * b);
            }
            x[j] = v;
        }
    }
    if (nbv < 16) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            u32 lo = 4u * j;
            u32 nb = nbv > lo ? nbv - lo : 0;
            if (nb < 4) x[j] &= (nb == 0) ? 0u : ((1u << (8 * nb)) - 1u);
        }
    }
}

// 16 bytes of a phrase at p (20 readable bytes guaranteed by the caller), in two halves so that
// the loads of the next chunk can be in flight while the current one is hashed:
// fetch = five aligned 32-bit loads; finish = funnel shift by the misalignment and zero the
// bytes past the phrase end (rem = bytes left from p), without branches
struct ChunkRaw { u32 W[5]; u32 bs; };

__device__ __forceinline__ void chunk_fetch(const u8 *p, ChunkRaw &r) {
    r.bs = (u32)((uintptr_t)p & 3);
    const u32 *p4 = reinterpret_cast<const u32 *>(p - r.bs);
#pragma unroll
    for (int j = 0; j < 5; j++) r.W[j] = __ldg(p4 + j);
}

__device__ __forceinline__ void chunk_finish(const ChunkRaw &r, u32 rem, u32 x[4]) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
        u32 v = __funnelshift_r(r.W[j], r.W[j + 1], 8 * r.bs);
        int nb = (int)rem - 4 * j;                    // valid bytes of word j, clamped to 0..4
        nb = nb < 0 ? 0 : (nb > 4 ? 4 : nb);
        x[j] = v & __funnelshift_rc(0xFFFFFFFFu, 0u, 8u * (4u - (u32)nb));
    }
}

__device__ __forceinline__ void nh_chunk(const u32 *__restrict__ sk, u32 c, const u32 x[4], u64 &pa,
                                         u64 &pb) {
    const uint4 k0 = *reinterpret_cast<const uint4 *>(sk + 4 * c);
    const uint4 k1 = *reinterpret_cast<const uint4 *>(sk + 4 * c + 4);
    pa += (u64)(x[0] + k0.x) * (u64)(x[1] + k0.y) + (u64)(x[2] + k0.z) * (u64)(x[3] + k0.w);
    pb += (u64)(x[0] + k1.x) * (u64)(x[1] + k1.y) + (u64)(x[2] + k1.z) * (u64)(x[3] + k1.w);
}

// .last and .sai of every phrase: one thread per phrase, coalesced stores
__global__ void phrase_records_k(TextView tv, const u64 *__restrict__ ends, u64 j0, u64 P, u32 w,
                                 u8 *__restrict__ last, u8 *__restrict__ sai) {
    u64 j = j0 + (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= P) return;
    i64 e = (i64)ends[j];
    last[j] = tv_byte(tv, e - (i64)w);                          // newscan.cpp:296
    if (sai) {                                                  // newscan.cpp:299-301
        u64 pos = (u64)(e + 1);
        u8 *d = sai + j * PFP_IBYTES;
#pragma unroll
        for (int b = 0; b < PFP_IBYTES; b++) d[b] = (u8)(pos >> (8 * b));
    }
}

constexpr int PH_T = 256;
constexpr int PH_WARPS = PH_T / 32;
constexpr int PH_PER_BLOCK = PH_T;                   // one phrase per thread of a warp block

// A warp takes 32 consecutive phrases, flattens them into their 16-byte chunks and gives every
// lane the same number of consecutive chunks (phrase lengths are geometric: giving lanes whole
// phrases would leave most of the warp idle).  NH sums are additive, so a lane adds what it
// accumulated to the phrase's shared-memory accumulator whenever it crosses a phrase boundary
// (dealing chunks round-robin instead costs two shared atomics per chunk: measured 1.6x slower).
// Phrases longer than one NH segment (8 KB) go to phrase_hash_long_k.
__global__ void __launch_bounds__(PH_T) phrase_hash_k(TextView tv, PhraseArrays ph, u64 P,
                                                      i64 first_start, u32 w,
                                                      const u32 *__restrict__ keytab,
                                                      u32 *__restrict__ long_list,
                                                      u32 *__restrict__ long_count, u32 long_cap,
                                                      u64 *__restrict__ flags) {
    __shared__ __align__(16) u32 sk[NH_KEY_WORDS];
    __shared__ const u8 *s_ptr[PH_WARPS][32];
    __shared__ u32 s_len[PH_WARPS][32];
    __shared__ u32 s_pre[PH_WARPS][33];
    __shared__ unsigned long long s_acc[PH_WARPS][32][2];
    for (int i = threadIdx.x; i < NH_KEY_WORDS; i += PH_T) sk[i] = keytab[i];
    __syncthreads();
    const u32 lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    for (u64 j0 = ((u64)blockIdx.x * PH_WARPS + wp) * 32; j0 < P; j0 += (u64)gridDim.x * PH_PER_BLOCK) {
        const u64 j = j0 + lane;
        const bool valid = j < P;
        i64 e = valid ? (i64)ph.ends[j] : 0;
        i64 prev = __shfl_up_sync(0xffffffffu, e, 1);
        if (lane == 0) prev = (j0 > 0) ? (i64)ph.ends[j0 - 1] : 0;
        const i64 s0 = (j == 0) ? first_start : prev - (i64)w + 1;
        const u64 len = valid ? (u64)(e - s0 + 1) : 0;
        // the long kernel takes phrases beyond one NH segment, phrases touching the virtual
        // borders of the text, and phrases within 20 bytes of the end of the buffer
        const bool slow = valid && (len > NH_SEG_BYTES || s0 < tv.pos0 || e >= tv.n_global ||
                                    (u64)(e - tv.pos0) + 24 > tv.n_buf);
        if (slow) {
            if (len > 0xFFFFFFFFull) atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_LIMIT);
            else {
                const u32 li = atomicAdd(long_count, 1u);
                if (li < long_cap) long_list[li] = (u32)j;
                else atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_INTERNAL);   // cannot happen: cap = P
            }
        }
        const u32 mylen = slow ? 0u : (u32)len;
        const u32 nch = (mylen + 15) >> 4;
        const u32 incl = warp_incl_scan(nch);
        const u32 T = __shfl_sync(0xffffffffu, incl, 31);
        const u8 *myptr = tv.T + (s0 - tv.pos0);
        s_ptr[wp][lane] = myptr;
        s_len[wp][lane] = mylen;
        s_pre[wp][lane] = incl - nch;
        if (lane == 31) s_pre[wp][32] = T;
        s_acc[wp][lane][0] = 0ull;
        s_acc[wp][lane][1] = 0ull;
        __syncwarp();
        const u32 K = (T + 31) >> 5;
        u32 g = lane * K;
        const u32 g1 = (g + K < T) ? g + K : T;
        // A phrase finished inside the lane that started it is stored at once.  A phrase that
        // spans lanes is the sum of: the tail partial of the lane where it starts, the whole sum
        // of every lane lying inside it (pass-through), the head partial of the lane where it
        // ends -- combined by one segmented warp scan, no atomics.
        u64 head_a = 0, head_b = 0, tail_a = 0, tail_b = 0;
        u32 head_q = 0xFFFFFFFFu;
        bool pass = false;
        if (g < g1) {
            u32 lo = 0, hi = 32;              // phrase holding chunk g: pre[lo] <= g < pre[lo+1]
#pragma unroll
            for (int it = 0; it < 5; it++) {
                u32 mid = (lo + hi) >> 1;
                if (s_pre[wp][mid] <= g) lo = mid; else hi = mid;
            }
            u32 q = lo;
            u32 c = g - s_pre[wp][q];
            bool cont = c != 0;               // the first partial continues an earlier lane's phrase
            const u8 *qp = s_ptr[wp][q];
            u32 qlen = s_len[wp][q];
            u32 qnch = (qlen + 15) >> 4;
            u64 pa = 0, pb = 0;
            ChunkRaw cur;
            chunk_fetch(qp + 16u * c, cur);
            for (; g < g1; g++) {
                // where the next chunk lives: same phrase, or the start of the next one
                u32 nq = q, nc = c + 1, nlen = qlen, nnch = qnch;
                const u8 *np = qp;
                const bool ends = nc == qnch;
                if (ends) {
                    nc = 0;
                    do { nq++; } while (nq < 31 && s_len[wp][nq] == 0);
                    np = s_ptr[wp][nq & 31];
                    nlen = s_len[wp][nq & 31];
                    nnch = (nlen + 15) >> 4;
                }
                ChunkRaw nxt;
                if (g + 1 < g1) chunk_fetch(np + 16u * nc, nxt);      // in flight during the hashing below
                u32 x[4];
                chunk_finish(cur, qlen - 16u * c, x);
                nh_chunk(sk, c, x, pa, pb);
                if (ends) {
                    if (cont) { head_a = pa; head_b = pb; head_q = q; cont = false; }
                    else { s_acc[wp][q][0] = pa; s_acc[wp][q][1] = pb; }
                    pa = pb = 0;
                }
                q = nq; c = nc; qp = np; qlen = nlen; qnch = nnch;
                cur = nxt;
            }
            if (c != 0) { tail_a = pa; tail_b = pb; pass = cont; }
        }
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            u64 ta = __shfl_up_sync(0xffffffffu, tail_a, o);
            u64 tb = __shfl_up_sync(0xffffffffu, tail_b, o);
            int tp = __shfl_up_sync(0xffffffffu, (int)pass, o);
            if (lane >= (u32)o && pass) { tail_a += ta; tail_b += tb; pass = tp != 0; }
        }
        u64 ca = __shfl_up_sync(0xffffffffu, tail_a, 1);
        u64 cb = __shfl_up_sync(0xffffffffu, tail_b, 1);
        if (head_q != 0xFFFFFFFFu) {
            s_acc[wp][head_q][0] = head_a + (lane ? ca : 0ull);
            s_acc[wp][head_q][1] = head_b + (lane ? cb : 0ull);
        }
        __syncwarp();
        if (valid && !slow) store_rec(ph.rec, j, s_acc[wp][lane][0], s_acc[wp][lane][1]);
        __syncwarp();
    }
}

// Listed phrases (longer than one NH segment, touching the text borders, or left over by the
// streaming pass): one warp per phrase, lanes stride over its 16-byte chunks; the chunks of
// segment s enter the sum with weight FOLD^s (pfp_fp.cuh).  Six CTAs per SM hold it at 40 registers
// (48 resident warps); left to itself ptxas takes 46.
__global__ void __launch_bounds__(PH_T, 6) phrase_hash_long_k(TextView tv, PhraseArrays ph,
                                                              i64 first_start, u32 w,
                                                              const u32 *__restrict__ keytab,
                                                              const u32 *__restrict__ long_list,
                                                              const u32 *__restrict__ long_count, u32 long_cap,
                                                              u64 *__restrict__ flags) {
    __shared__ __align__(16) u32 sk[NH_KEY_WORDS];
    for (int i = threadIdx.x; i < NH_KEY_WORDS; i += PH_T) sk[i] = keytab[i];
    __syncthreads();
    const u32 lane = threadIdx.x & 31;
    const u32 nlong = min(*long_count, long_cap);
    for (u32 q = blockIdx.x * PH_WARPS + (threadIdx.x >> 5); q < nlong; q += gridDim.x * PH_WARPS) {
        const u64 j = long_list[q];
        const i64 e = (i64)ph.ends[j];
        const i64 s0 = (j == 0) ? first_start : (i64)ph.ends[j - 1] - (i64)w + 1;
        const u64 len = (u64)(e - s0 + 1);
        const bool special = (s0 < 0) || (e >= tv.n_global);
        const u64 nch = (len + 15) >> 4;
        u64 fa = 0, fb = 0, pa = 0, pb = 0, wa = 1, wb = 1;
        u64 seg = 0;
        for (u64 c = lane; c < nch; c += 32) {
            const u64 sg = c >> 9;
            if (sg != seg) {                       // leave segment `seg`: weigh what was gathered in it
                fa += wa * pa; fb += wb * pb;
                pa = pb = 0;
                for (; seg < sg; seg++) { wa *= NH_FOLD_A; wb *= NH_FOLD_B; }
            }
            u32 x[4];
            load_chunk(tv, s0, len, 16ull * c, special, x);
            nh_chunk(sk, (u32)(c & 511u), x, pa, pb);
        }
        fa += wa * pa; fb += wb * pb;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            fa += __shfl_xor_sync(0xffffffffu, fa, o);
            fb += __shfl_xor_sync(0xffffffffu, fb, o);
        }
        if (lane == 0) {
            if (len > 0xFFFFFFFFull) atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_LIMIT);
            store_rec(ph.rec, j, fa, fb);
        }
    }
}

// ---- K3: dictionary table ---------------------------------------------------------------------------------
// Open addressing, linear probing, 16-byte slots {key, val, check}; key 0 = empty.
// A warp first groups its lanes by key (match.any) so that runs of identical phrases cost one
// atomic per warp instead of 32.  `chk` is a 32-bit digest of the full 128-bit fingerprint and
// the length, independent of the key: every phrase that lands in a slot must agree with it, or
// the parse stops with PFPB200_E_COLLISION (the reference compares strings, newscan.cpp:282-286).
// `val` is the word's occurrence count.
struct __align__(16) DictSlot { u64 key; u32 val; u32 chk; };
constexpr u32 TABLE_MAX_PROBES = 2048;

// One probe sequence: a plain 16-byte load of the slot first -- on repetitive inputs nine phrases
// in ten find their word already there and finish with one fire-and-forget add to its count --
// and a CAS only on an empty slot.  The thread that wins the CAS is the word's creator.  Word ids
// are not handed out here: table_insert_k leaves the slot in uid[] with a creator bit, and
// table_compact_k numbers the words afterwards, in the order of their creators' records (one scan
// over the records, no counter that every creator has to wait for).
struct Probe { u64 slot; bool placed; bool creator; u32 seen_chk; };

__device__ __forceinline__ Probe table_probe(DictSlot *__restrict__ tab, u64 cap, u64 slot, uint4 sv, u64 k) {
    Probe r{slot, false, false, 0u};
    u32 probes = 0;
    for (;;) {
        const u64 key = ((u64)sv.y << 32) | sv.x;
        if (key == k) { r.placed = true; r.seen_chk = sv.w; break; }
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

__global__ void table_init_k(DictSlot *__restrict__ tab, u64 cap) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cap) *reinterpret_cast<uint4 *>(tab + i) = make_uint4(0u, 0u, 0u, 0u);
}

constexpr int TI_T = 256;

// uid[j] = slot of record j's word, with UID_CREATOR set on the record whose thread won the CAS of
// the empty slot.  Occurrences add up in the slot's val: popc(peers) per leader of a match.any
// group, or weight[j] per record (words of several shards being merged, newscan.cpp:277-281).
// No thread waits for another: no barrier, no counter; table_compact_k numbers the words.  The
// kernel is latency-bound on the table: one record per thread and round at 32 registers (all 64
// warps of an SM resident) measured faster than 2 or 4 records in flight per thread at 38 / 64
// registers (DESIGN.md §3b).
__global__ void __launch_bounds__(TI_T, 8) table_insert_k(const PhraseFp *__restrict__ rec, u64 P,
                                                         DictSlot *__restrict__ tab, u64 cap,
                                                         const u32 *__restrict__ weight,
                                                         u32 weak /* test hook: keep 2 fingerprint bits */,
                                                         u32 *__restrict__ uid, u64 *__restrict__ flags) {
    const u32 lane = threadIdx.x & 31;
    for (u64 b0 = (u64)blockIdx.x * TI_T; b0 < P; b0 += (u64)gridDim.x * TI_T) {
        const u64 j = b0 + threadIdx.x;
        PhraseFp r;
        r.fpa = 0; r.fpb = 0;
        u64 k = 0;
        if (j < P) {                                  // streamed once: keep it out of the table's way in L2
            const uint4 a = __ldcs(reinterpret_cast<const uint4 *>(rec + j));
            r.fpa = ((u64)a.y << 32) | a.x; r.fpb = ((u64)a.w << 32) | a.z;
            if (weak) { r.fpa &= 3ull; r.fpb = 0; }
            k = sort_key_of(r.fpa, r.fpb);
        }
        const u32 chk = j < P ? check_of(r) : 0u;
        const u32 peers = __match_any_sync(0xffffffffu, k);
        const int leader = __ffs(peers) - 1;
        const bool lead = j < P && (int)lane == leader;
        u32 res = 0;                                  // table full: any valid slot, the stage is rerun
        if (lead) {
            const u64 s0 = __umul64hi(k, cap);
            const Probe pr = table_probe(tab, cap, s0, __ldcg(reinterpret_cast<const uint4 *>(tab + s0)), k);
            if (pr.placed) {
                res = (u32)pr.slot | (pr.creator ? UID_CREATOR : 0u);
                u32 seen = pr.seen_chk;
                if (seen == 0u) seen = atomicCAS(&tab[pr.slot].chk, 0u, chk);   // creator, or racing with it
                if (seen != 0u && seen != chk) atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_COLLISION);
                if (!weight) atomicAdd(&tab[pr.slot].val, (u32)__popc(peers));
            } else {
                atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_TABLE_FULL);
            }
        }
        const u32 slot = __shfl_sync(0xffffffffu, res, leader) & ~UID_CREATOR;
        const u32 lchk = __shfl_sync(0xffffffffu, chk, leader);
        if (j < P) {
            if (chk != lchk) atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_COLLISION);
            __stcs(uid + j, lead ? res : slot);
            if (weight) {
                const u32 c = weight[j];
                const u32 old = atomicAdd(&tab[slot].val, c);
                if (old + c < old) atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_LIMIT);
            }
        }
    }
}

constexpr int TC_T = 256;
constexpr int TC_I = 4;                              // consecutive records per thread
constexpr int TC_TILE = TC_T * TC_I;

__device__ __forceinline__ void load_uids(const u32 *__restrict__ uid, u64 n, u64 j, u32 v[TC_I]) {
    if (j + TC_I <= n) {                             // j is a multiple of 4: one aligned 16-byte load
        const uint4 a = __ldcs(reinterpret_cast<const uint4 *>(uid + j));
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
    } else {
#pragma unroll
        for (int i = 0; i < TC_I; i++) v[i] = j + i < n ? uid[j + i] : 0u;
    }
}

// creators per tile of TC_TILE records
__global__ void __launch_bounds__(TC_T) table_creators_k(const u32 *__restrict__ uid, u64 n,
                                                         u32 *__restrict__ tile_count) {
    __shared__ u32 sm[9];
    u32 v[TC_I];
    load_uids(uid, n, (u64)blockIdx.x * TC_TILE + (u64)threadIdx.x * TC_I, v);
    u32 c = 0;
#pragma unroll
    for (int i = 0; i < TC_I; i++) c += v[i] >> 31;
    u32 total;
    block_excl_scan_256(c, &total, sm);
    if (threadIdx.x == 0) tile_count[blockIdx.x] = total;
}

// Numbers the words in the order of their creators' records (tile_base: exclusive scan of
// table_creators_k's counts) and writes, at each word id u: its representative record, count,
// slot, length and start, and the creator's uid[] becomes the word id (creator bit kept).  The
// length comes from len_in[rep] when given (merge), else from ends[]
// (phrase j = text from ends[j-1]-w+1, or first_start for j = 0, to ends[j]).  Every load of a
// thread's creators is issued before its first store.  flags[2] / flags[3] get the largest and
// the total word length.
__global__ void __launch_bounds__(TC_T, 6) table_compact_k(u32 *__restrict__ uid, u64 n,
                                                        const u32 *__restrict__ tile_base,
                                                        const DictSlot *__restrict__ tab,
                                                        const u32 *__restrict__ len_in,
                                                        const u64 *__restrict__ ends, i64 first_start, u32 w,
                                                        u32 *__restrict__ slot_of_word,
                                                        u32 *__restrict__ rep, u32 *__restrict__ count,
                                                        u32 *__restrict__ ulen, u32 *__restrict__ uwords,
                                                        i64 *__restrict__ ustart /* may be null */,
                                                        u64 *__restrict__ flags) {
    __shared__ u32 sm[9];
    __shared__ u32 s_max;
    __shared__ unsigned long long s_sum;
    if (threadIdx.x == 0) { s_max = 0; s_sum = 0; }
    const u64 j0 = (u64)blockIdx.x * TC_TILE + (u64)threadIdx.x * TC_I;
    u32 v[TC_I];
    load_uids(uid, n, j0, v);
    u32 c = 0;
#pragma unroll
    for (int i = 0; i < TC_I; i++) c += v[i] >> 31;
    u32 cnt[TC_I], len[TC_I];
    i64 st[TC_I];
#pragma unroll
    for (int i = 0; i < TC_I; i++) {
        const u64 j = j0 + i;
        const bool cr = (v[i] & UID_CREATOR) != 0;
        cnt[i] = cr ? tab[v[i] & ~UID_CREATOR].val : 0u;
        if (len_in) {
            len[i] = cr ? len_in[j] : 0u;
            st[i] = 0;
        } else {
            st[i] = cr ? (j ? (i64)ends[j - 1] - (i64)w + 1 : first_start) : 0;
            len[i] = cr ? (u32)((i64)ends[j] - st[i] + 1) : 0u;        // > 2^32-1 was flagged by K2
        }
    }
    u32 total;
    u32 u = block_excl_scan_256(c, &total, sm) + tile_base[blockIdx.x];
    u32 mx = 0;
    u64 sum = 0;
#pragma unroll
    for (int i = 0; i < TC_I; i++) {
        if (!(v[i] & UID_CREATOR)) continue;
        slot_of_word[u] = v[i] & ~UID_CREATOR;
        uid[j0 + i] = u | UID_CREATOR;
        rep[u] = (u32)(j0 + i); count[u] = cnt[i]; ulen[u] = len[i]; uwords[u] = (len[i] + 7) >> 3;
        if (ustart) ustart[u] = st[i];
        mx = max(mx, len[i]);
        sum += len[i];
        u++;
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if ((threadIdx.x & 31) == 0 && sum) { atomicMax(&s_max, mx); atomicAdd(&s_sum, (unsigned long long)sum); }
    __syncthreads();
    if (threadIdx.x == 0 && s_sum) {
        atomicMax((unsigned long long *)&flags[2], (unsigned long long)s_max);
        atomicAdd((unsigned long long *)&flags[3], s_sum);
    }
}

// d_ptr non-null: the number of words is read there (a merge that has not read it back yet)
__global__ void word_of_slot_k(const u32 *__restrict__ slot_of_word, u64 d, const u64 *__restrict__ d_ptr,
                               u32 *__restrict__ word_of_slot) {
    const u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < (d_ptr ? *d_ptr : d)) word_of_slot[slot_of_word[u]] = (u32)u;
}

__device__ __forceinline__ u32 word_of(u32 v, const u32 *__restrict__ word_of_slot) {
    return (v & UID_CREATOR) ? v & ~UID_CREATOR : word_of_slot[v];
}

// uid[j]: word id with the creator bit, or table slot -> word id
__global__ void uid_words_k(u32 *__restrict__ uid, u64 n, const u32 *__restrict__ word_of_slot) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 j = 4 * q;
    if (j + 4 <= n) {
        uint4 v = __ldcs(reinterpret_cast<const uint4 *>(uid) + q);
        v.x = word_of(v.x, word_of_slot); v.y = word_of(v.y, word_of_slot);
        v.z = word_of(v.z, word_of_slot); v.w = word_of(v.w, word_of_slot);
        __stcs(reinterpret_cast<uint4 *>(uid) + q, v);
    } else {
        for (u64 i = j; i < n; i++) uid[i] = word_of(uid[i], word_of_slot);
    }
}

// uid[0..n) -> word ids; at most d_max words, their number in d_ptr on the device when not null
static int uid_words(pfpb200_ctx *ctx, DictArrays *D, u64 n, u64 d_max, const u64 *d_ptr) {
    if (n && d_max) {
        u32 *word_of_slot = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &word_of_slot, D->slots));
        word_of_slot_k<<<pfp_blocks(d_max, 256), 256, 0, ctx->stream>>>(D->slot_of_word, d_max, d_ptr, word_of_slot);
        PFP_LAUNCHED(ctx);
        uid_words_k<<<pfp_blocks((n + 3) / 4, 256), 256, 0, ctx->stream>>>(D->uid, n, word_of_slot);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_free_now(ctx, word_of_slot));
    }
    PFP_TRY(pfp_free_now(ctx, D->slot_of_word));
    D->slot_of_word = nullptr;
    return PFPB200_OK;
}

int pfp_uid_words(pfpb200_ctx *ctx, DictArrays *D, u64 n) {
    return D->slot_of_word ? uid_words(ctx, D, n, D->d, nullptr) : PFPB200_OK;
}

// The table part of a dedup: n records into a fresh table of cap slots, then word ids in the order
// of the creators' records.  rep/count/ulen/uwords/ustart/slot_of_word are written for the d words,
// flags[1] = d, flags[2] = largest, flags[3] = total word length; uid[] as DictArrays::slot_of_word
// describes it.
static int table_words(pfpb200_ctx *ctx, const PhraseFp *rec, u64 n, DictSlot *tab, u64 cap,
                       const u32 *weight, const u32 *len_in, const u64 *ends, i64 first_start, u32 w,
                       u32 *uid, const DictArrays &D) {
    table_init_k<<<pfp_blocks(cap, 256), 256, 0, ctx->stream>>>(tab, cap);
    PFP_LAUNCHED(ctx);
    PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[1], 0, 3 * sizeof(u64), ctx->stream));
    if (n == 0) return PFPB200_OK;
    int per_sm = 0;                                  // a grid of resident CTAs strides over the records
    PFP_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, table_insert_k, TI_T, 0));
    const u64 want = (n + TI_T - 1) / TI_T;
    const u64 resident = (u64)ctx->sm_count * (per_sm > 0 ? per_sm : 1);
    table_insert_k<<<(u32)(want < resident ? want : resident), TI_T, 0, ctx->stream>>>(
        rec, n, tab, cap, weight, ctx->weak_fp, uid, ctx->d_flags);
    PFP_LAUNCHED(ctx);
    const u32 nt = pfp_blocks(n, TC_TILE);
    u32 *tile = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &tile, nt));
    table_creators_k<<<nt, TC_T, 0, ctx->stream>>>(uid, n, tile);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pfp_exclusive_scan_u32(ctx, tile, tile, nt, reinterpret_cast<u32 *>(&ctx->d_flags[1])));
    table_compact_k<<<nt, TC_T, 0, ctx->stream>>>(uid, n, tile, tab, len_in, ends, first_start, w, D.slot_of_word,
                                                  D.rep, D.count, D.ulen, D.uwords, D.ustart, ctx->d_flags);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pfp_free_now(ctx, tile));
    return PFPB200_OK;
}

// phrase pool: every distinct word once, zero padded to 8 bytes, 8-byte aligned
// 8-byte word k of the phrase that starts at global position s0 and is len bytes long (zero
// behind its end); special: the phrase touches a virtual border of the text
__device__ __forceinline__ u64 phrase_word8(const TextView &tv, i64 s0, u64 len, u64 k, bool special) {
    const u64 o = 8 * k;
    const u32 nbv = (u32)((len - o) < 8 ? (len - o) : 8);
    u64 v = 0;
    if (!special) {
        const u8 *p = tv.T + (s0 + (i64)o - tv.pos0);
        const u32 bs = (u32)((uintptr_t)p & 7);
        const u64 *p8 = reinterpret_cast<const u64 *>(p - bs);
        const u64 lo = __ldg(p8);
        if (bs) {
            const u64 hi = (bs + nbv > 8) ? __ldg(p8 + 1) : 0ull;
            v = (lo >> (8 * bs)) | (hi << (64 - 8 * bs));
        } else v = lo;
    } else {
        for (u32 b = 0; b < nbv; b++) v |= (u64)tv_byte(tv, s0 + (i64)o + b) << (8 * b);
    }
    if (nbv < 8) v &= (1ull << (8 * nbv)) - 1ull;
    return v;
}

// The copy is organised by OUTPUT: the pool offsets ascend with the word id, so the 32 words of a
// warp fill one contiguous span of the pool; every lane takes consecutive 8-byte slots of that span
// (coalesced stores, all lanes busy whatever the word lengths), finds the word a slot belongs to by
// a binary search over the warp's 32 offsets (shuffles) and fetches its bytes from the text.
// Eight lanes per word instead measured slower (DESIGN.md §3b).
__global__ void __launch_bounds__(PH_T) pool_copy_span_k(TextView tv, const i64 *__restrict__ ustart,
                                                         const u32 *__restrict__ ulen,
                                                         const u64 *__restrict__ uoff, u64 d,
                                                         u64 *__restrict__ pool) {
    const u32 lane = threadIdx.x & 31;
    for (u64 u0 = ((u64)blockIdx.x * PH_WARPS + (threadIdx.x >> 5)) * 32; u0 < d; u0 += (u64)gridDim.x * PH_WARPS * 32) {
        const u64 u = u0 + lane;
        const bool have = u < d;
        const i64 s0 = have ? ustart[u] : 0;
        const u32 len = have ? ulen[u] : 0u;
        const u64 off = have ? uoff[u] : 0ull;
        const u64 base = __shfl_sync(0xffffffffu, off, 0);
        const u32 nw = (len + 7) >> 3;
        u32 rel = have ? (u32)(off - base) : 0xFFFFFFFFu;              // lanes past the end never match
        const u32 endrel = have ? rel + nw : 0u;
        u32 total = endrel;                                            // span length: max over the lanes
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) total = max(total, __shfl_xor_sync(0xffffffffu, total, o));
        const bool special = have && (s0 < 0 || s0 + (i64)len > tv.n_global);
        for (u32 k0 = 0; k0 < total; k0 += 32) {
            const u32 k = k0 + lane;
            u32 j = 0;                                                 // largest lane with rel <= k
#pragma unroll
            for (int step = 16; step > 0; step >>= 1) {
                const u32 t = __shfl_sync(0xffffffffu, rel, (j + step) & 31);
                if (j + step < 32 && t <= k) j += step;
            }
            const u32 rj = __shfl_sync(0xffffffffu, rel, j);
            const u32 lj = __shfl_sync(0xffffffffu, len, j);
            const i64 sj = __shfl_sync(0xffffffffu, s0, j);
            const int spj = __shfl_sync(0xffffffffu, (int)special, j);
            if (k < total) pool[base + k] = phrase_word8(tv, sj, lj, k - rj, spj != 0);
        }
    }
}

// PFPB200_F_VERIFY: every phrase is compared byte for byte with the pool copy of the word it was
// given -- what the reference does on every map hit (newscan.cpp:282-286).  With it a wrong merge
// of two different phrases is impossible, whatever the fingerprints say: the parse either is
// exact or stops with PFPB200_E_COLLISION.  One warp per phrase.
__global__ void __launch_bounds__(PH_T) verify_phrases_k(TextView tv, const u64 *__restrict__ ends,
                                                         i64 first_start, u32 w, u64 P,
                                                         const u32 *__restrict__ uid,
                                                         const u32 *__restrict__ ulen,
                                                         const u64 *__restrict__ uoff,
                                                         const u64 *__restrict__ pool,
                                                         u64 *__restrict__ flags) {
    const u32 lane = threadIdx.x & 31;
    for (u64 j = (u64)blockIdx.x * PH_WARPS + (threadIdx.x >> 5); j < P; j += (u64)gridDim.x * PH_WARPS) {
        const i64 e = (i64)ends[j];
        const i64 s0 = (j == 0) ? first_start : (i64)ends[j - 1] - (i64)w + 1;
        const u64 len = (u64)(e - s0 + 1);
        const u32 u = uid[j];
        bool bad = len != (u64)ulen[u];
        if (!bad) {
            const bool special = (s0 < 0) || (e >= tv.n_global);
            const u64 *src = pool + uoff[u];
            const u64 nw = (len + 7) >> 3;
            for (u64 k = lane; k < nw; k += 32) bad |= phrase_word8(tv, s0, len, k, special) != src[k];
        }
        if (__any_sync(0xffffffffu, bad) && lane == 0)
            atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_COLLISION);
    }
}

// the same for the entries of a dictionary merge: entry i against the representative entry of
// the word it was merged into (both in the received pool)
__global__ void __launch_bounds__(PH_T) verify_entries_k(u64 n, const u32 *__restrict__ uid_of_entry,
                                                         const u32 *__restrict__ rep,
                                                         const u32 *__restrict__ len_in,
                                                         const u64 *__restrict__ in_off,
                                                         const u64 *__restrict__ pool,
                                                         u64 *__restrict__ flags) {
    const u32 lane = threadIdx.x & 31;
    for (u64 i = (u64)blockIdx.x * PH_WARPS + (threadIdx.x >> 5); i < n; i += (u64)gridDim.x * PH_WARPS) {
        const u32 r = rep[uid_of_entry[i]];
        if (r == (u32)i) continue;
        bool bad = len_in[i] != len_in[r];
        if (!bad) {
            const u64 *a = pool + in_off[i], *b = pool + in_off[r];
            const u64 nw = ((u64)len_in[i] + 7) >> 3;
            for (u64 k = lane; k < nw; k += 32) bad |= a[k] != b[k];
        }
        if (__any_sync(0xffffffffu, bad) && lane == 0)
            atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_COLLISION);
    }
}

// ------------------------------------------------------------------------------------------
// host orchestration
// ------------------------------------------------------------------------------------------
// fingerprints of the phrases listed in long_list[0..*long_count): any length, any position
int pfp_hash_list(pfpb200_ctx *ctx, const TextView &tv, const PhraseArrays &ph, i64 first_start, u32 w,
                  const u32 *long_list, const u32 *long_count, u64 max_count) {
    u64 want = (max_count + PH_WARPS - 1) / PH_WARPS;
    u64 maxb = (u64)ctx->sm_count * 8;
    u32 nlb = (u32)(want < maxb ? want : maxb);
    if (nlb == 0) nlb = 1;
    phrase_hash_long_k<<<nlb, PH_T, 0, ctx->stream>>>(tv, ph, first_start, w, ctx->d_keys, long_list,
                                                      long_count, (u32)(max_count < 0xFFFFFFFFull ? max_count : 0xFFFFFFFFull),
                                                      ctx->d_flags);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

// .last/.sai of the phrases [j0, P)
int pfp_records_range(pfpb200_ctx *ctx, const TextView &tv, const PhraseArrays &ph, u64 j0, u64 P, u32 w) {
    if (j0 >= P) return PFPB200_OK;
    phrase_records_k<<<pfp_blocks(P - j0, 256), 256, 0, ctx->stream>>>(tv, ph.ends, j0, P, w, ph.last, ph.sai);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

int pfp_hash_stage(pfpb200_ctx *ctx, const TextView &tv, const PhraseArrays &ph, u64 P,
                   i64 first_start, u32 w) {
    u32 *long_list = nullptr, *long_count = nullptr;
    // every phrase may be listed: all of them are longer than one NH segment when w >= 8192, and up
    // to 24 short ones can end within the last 24 bytes of the buffer (4 bytes per phrase)
    const u64 cap = P + 8;
    PFP_TRY(pfp_alloc_t(ctx, &long_list, (size_t)cap));
    PFP_TRY(pfp_alloc_t(ctx, &long_count, 1));
    PFP_CUDA(ctx, cudaMemsetAsync(long_count, 0, sizeof(u32), ctx->stream));
    phrase_records_k<<<pfp_blocks(P, 256), 256, 0, ctx->stream>>>(tv, ph.ends, 0, P, w, ph.last, ph.sai);
    PFP_LAUNCHED(ctx);
    u64 want = (P + PH_PER_BLOCK - 1) / PH_PER_BLOCK;
    u64 maxb = (u64)ctx->sm_count * 32;
    u32 nb = (u32)(want < maxb ? want : maxb);
    if (nb == 0) nb = 1;
    phrase_hash_k<<<nb, PH_T, 0, ctx->stream>>>(tv, ph, P, first_start, w, ctx->d_keys, long_list, long_count,
                                                (u32)cap, ctx->d_flags);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pfp_hash_list(ctx, tv, ph, first_start, w, long_list, long_count, cap));
    PFP_TRY(pfp_free_now(ctx, long_list));
    PFP_TRY(pfp_free_now(ctx, long_count));
    return PFPB200_OK;
}

// Inserts every phrase into the dictionary table and numbers the distinct words in the text order
// of their creators; when the stage is done rep[], ulen[], uwords[], ustart[] and count[] are
// complete, and uid[] holds table slots that D->slot_of_word relates to the words (pfp_uid_words
// turns them into word ids; the remap of the .dict stage reads them as they are).
// Reads d (and length stats) back to the host: one synchronisation.
int pfp_dedup_stage(pfpb200_ctx *ctx, const PhraseArrays &ph, u64 P, i64 first_start, u32 w, DictArrays *D) {
    // Capacity: without a hint 1.5 P (load factor <= 2/3 even if every phrase is distinct).  The
    // distinct/phrase ratio of the previous parse on this context sizes the table 2x the expected
    // dictionary instead, which keeps it several times smaller on repetitive inputs -- small
    // enough to live in L2; if that guess turns out too small the insert kernel says so and the
    // stage reruns with the safe size.  Slots are addressed by fastrange (mulhi(key, cap)), so the
    // capacity need not be a power of two.  The per-word arrays are sized by the capacity.
    if (P >= 0x7FFFFFFEull) return pfp_fail(ctx, PFPB200_E_LIMIT, "more than 2^31-2 phrases in one shard");
    DictSlot *tab = nullptr;
    u64 cap = 0, d = 0;
    PFP_TRY(pfp_alloc_t(ctx, &D->uid, P));
    for (int attempt = 0;; attempt++) {
        double want = (double)P * 1.5;
        if (attempt == 0 && ctx->dedup_ratio > 0.0) {
            double guess = ctx->dedup_ratio * (double)P * 2.0;
            if (guess < want) want = guess;
        }
        cap = (u64)want + 1024;
        if (cap >= 0x7FFFFFFFull) cap = 0x7FFFFFFEull;
        const u64 wcap = cap < P ? cap : P;            // there are at most min(cap, P) words
        PFP_TRY(pfp_alloc_t(ctx, &tab, cap));
        PFP_TRY(pfp_alloc_t(ctx, &D->slot_of_word, wcap));
        PFP_TRY(pfp_alloc_t(ctx, &D->rep, wcap));
        PFP_TRY(pfp_alloc_t(ctx, &D->count, wcap));
        PFP_TRY(pfp_alloc_t(ctx, &D->ulen, wcap));
        PFP_TRY(pfp_alloc_t(ctx, &D->uwords, wcap));
        PFP_TRY(pfp_alloc_t(ctx, &D->ustart, wcap));
        PFP_TRY(table_words(ctx, ph.rec, P, tab, cap, nullptr, nullptr, ph.ends, first_start, w, D->uid, *D));
        PFP_CUDA(ctx, cudaMemcpyAsync(ctx->h_flags, ctx->d_flags, 4 * sizeof(u64), cudaMemcpyDeviceToHost,
                                      ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (ctx->h_flags[0] & PFP_ERRBIT_LIMIT)
            return pfp_fail(ctx, PFPB200_E_LIMIT, "a phrase is longer than 2^32-1 bytes");
        d = ctx->h_flags[1];
        const bool full = (ctx->h_flags[0] & PFP_ERRBIT_TABLE_FULL) != 0 || (double)d > 0.85 * (double)cap;
        if (!full) break;
        if (attempt > 0) return pfp_fail(ctx, PFPB200_E_INTERNAL, "dictionary table overflow");
        // undo and retry with the safe capacity
        void *fr[] = {tab, D->slot_of_word, D->rep, D->count, D->ulen, D->uwords, D->ustart};
        for (void *q : fr) PFP_TRY(pfp_free_now(ctx, q));
        ctx->dedup_ratio = 0.0;
        const u64 keep = ctx->h_flags[0] & ~(PFP_ERRBIT_TABLE_FULL | PFP_ERRBIT_COLLISION);
        PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->d_flags[0], &keep, sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    D->slots = cap;
    ctx->dedup_ratio = (double)d / (double)P;
    if (d > 0x7FFFFFFEull)
        return pfp_fail(ctx, PFPB200_E_LIMIT, "%llu distinct words exceed the limit 2^31-2",
                        (unsigned long long)d);
    D->d = d;
    D->max_len = (u32)ctx->h_flags[2];
    D->sum_len = ctx->h_flags[3];
    PFP_TRY(pfp_free_now(ctx, tab));
    return PFPB200_OK;
}

// Builds the pool of distinct words.  One synchronisation (pool size, max / total word length).
int pfp_pool_stage(pfpb200_ctx *ctx, const TextView &tv, DictArrays *D) {
    u64 d = D->d;
    PFP_TRY(pfp_alloc_t(ctx, &D->uoff, d));
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, D->uwords, D->uoff, d, &ctx->d_flags[1]));
    PFP_CUDA(ctx, cudaMemcpyAsync(ctx->h_flags, ctx->d_flags, 4 * sizeof(u64), cudaMemcpyDeviceToHost,
                                  ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->h_flags[0] & PFP_ERRBIT_COLLISION)
        return pfp_fail(ctx, PFPB200_E_COLLISION, "fingerprint collision between different phrases");
    D->pool_words = ctx->h_flags[1];
    D->max_len = (u32)ctx->h_flags[2];
    D->sum_len = ctx->h_flags[3];
    PFP_TRY(pfp_alloc_t(ctx, &D->pool, (size_t)D->pool_words));
    u64 want = (d + 32ull * PH_WARPS - 1) / (32ull * PH_WARPS);
    u64 maxb = (u64)ctx->sm_count * 32;
    pool_copy_span_k<<<(u32)(want < maxb ? (want ? want : 1) : maxb), PH_T, 0, ctx->stream>>>(
        tv, D->ustart, D->ulen, D->uoff, d, D->pool);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

// PFPB200_F_VERIFY for a merge whose pool arrived after the dedup (pfpb200_dict_merge_finish)
int pfp_merge_verify(pfpb200_ctx *ctx, u64 n, const u32 *uid_of_entry, const u32 *rep, const u32 *len_in,
                     const u32 *uwords_in, const u64 *pool) {
    if (n == 0) return PFPB200_OK;
    u64 *in_off = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &in_off, n));
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, uwords_in, in_off, n, nullptr));
    u64 want = (n + PH_WARPS - 1) / PH_WARPS;
    u64 maxb = (u64)ctx->sm_count * 32;
    verify_entries_k<<<(u32)(want < maxb ? want : maxb), PH_T, 0, ctx->stream>>>(n, uid_of_entry, rep, len_in, in_off, pool,
                                                                                ctx->d_flags);
    PFP_LAUNCHED(ctx);
    PFP_CUDA(ctx, cudaMemcpyAsync(ctx->h_flags, ctx->d_flags, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    PFP_TRY(pfp_free_now(ctx, in_off));
    if (ctx->h_flags[0] & PFP_ERRBIT_COLLISION)
        return pfp_fail(ctx, PFPB200_E_COLLISION, "two different words share a fingerprint (found by the verify pass)");
    return PFPB200_OK;
}

// PFPB200_F_VERIFY for a parse: after the pool exists.  The caller reads flags[0] back.
int pfp_verify_stage(pfpb200_ctx *ctx, const TextView &tv, const u64 *ends, i64 first_start, u32 w, u64 P,
                     const DictArrays &D) {
    if (P == 0) return PFPB200_OK;
    u64 want = (P + PH_WARPS - 1) / PH_WARPS;
    u64 maxb = (u64)ctx->sm_count * 32;
    verify_phrases_k<<<(u32)(want < maxb ? want : maxb), PH_T, 0, ctx->stream>>>(
        tv, ends, first_start, w, P, D.uid, D.ulen, D.uoff, D.pool, ctx->d_flags);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

// ------------------------------------------------------------------------------------------
// dictionary merge: words (fingerprint, length, count, pool bytes) coming from several shards
// ------------------------------------------------------------------------------------------
// the incoming words as fingerprint records, so that the dictionary-table kernels above dedup them
__global__ void merge_recs_k(const u64 *__restrict__ fpa, const u64 *__restrict__ fpb, u64 n,
                             PhraseFp *__restrict__ rec) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) store_rec(rec, i, fpa[i], fpb[i]);
}

// a merged word lives where its representative entry lives in the received pool
__global__ void merge_words_k(const u32 *__restrict__ rep, const u32 *__restrict__ uwords_in,
                              const u64 *__restrict__ in_off, const u64 *__restrict__ d_ptr,
                              u32 *__restrict__ uwords, u64 *__restrict__ uoff) {
    u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= *d_ptr) return;
    const u32 r = rep[u];
    uwords[u] = uwords_in[r];
    uoff[u] = in_off[r];
}

// per-word fingerprints of a shard's local dictionary (what a shard exports)
__global__ void gather_word_fp_k(const u32 *__restrict__ rep, const PhraseFp *__restrict__ rec,
                                 u64 d, u64 *__restrict__ wfpa, u64 *__restrict__ wfpb) {
    u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= d) return;
    u32 j = rep[u];
    wfpa[u] = rec[j].fpa;
    wfpb[u] = rec[j].fpb;
}

int pfp_gather_word_fp(pfpb200_ctx *ctx, const DictArrays &D, const PhraseArrays &ph, u64 *wfpa,
                       u64 *wfpb) {
    gather_word_fp_k<<<pfp_blocks(D.d, 256), 256, 0, ctx->stream>>>(D.rep, ph.rec, D.d, wfpa, wfpb);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

// Merges n input words into the distinct set D with the dictionary table (word ids in the order of
// their creators' entries); uid_of_entry[i] = merged word of input entry i, occurrences summed per word.
// One synchronisation.
int pfp_merge_stage(pfpb200_ctx *ctx, u64 n, const u64 *fpa, const u64 *fpb, const u32 *len,
                    const u32 *count_in, const u32 *uwords_in, const u64 *pool, u64 pool_words,
                    bool verify, DictArrays *D, u32 **uid_of_entry) {
    const int TB = 256;
    if (n >= 0x7FFFFFFEull / 2) return pfp_fail(ctx, PFPB200_E_LIMIT, "too many words to merge");
    PhraseFp *rec = nullptr;
    DictSlot *tab = nullptr;
    u64 *in_off = nullptr;
    const u64 cap = n + n / 2 + 1024;                  // load factor <= 2/3 even if nothing merges
    PFP_TRY(pfp_alloc_t(ctx, &rec, n));
    PFP_TRY(pfp_alloc_t(ctx, &tab, cap));
    PFP_TRY(pfp_alloc_t(ctx, &D->slot_of_word, n));
    PFP_TRY(pfp_alloc_t(ctx, &in_off, n));
    PFP_TRY(pfp_alloc_t(ctx, uid_of_entry, n));
    PFP_TRY(pfp_alloc_t(ctx, &D->rep, n));
    PFP_TRY(pfp_alloc_t(ctx, &D->count, n));
    PFP_TRY(pfp_alloc_t(ctx, &D->ulen, n));
    PFP_TRY(pfp_alloc_t(ctx, &D->uwords, n));
    PFP_TRY(pfp_alloc_t(ctx, &D->uoff, n));
    D->uid = *uid_of_entry;
    merge_recs_k<<<pfp_blocks(n, TB), TB, 0, ctx->stream>>>(fpa, fpb, n, rec);
    PFP_LAUNCHED(ctx);
    PFP_TRY(table_words(ctx, rec, n, tab, cap, count_in, len, nullptr, 0, 0, *uid_of_entry, *D));
    D->slots = cap;
    PFP_TRY(uid_words(ctx, D, n, n, reinterpret_cast<const u64 *>(&ctx->d_flags[1])));
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, uwords_in, in_off, n, nullptr));
    merge_words_k<<<pfp_blocks(n, TB), TB, 0, ctx->stream>>>(D->rep, uwords_in, in_off,
                                                             reinterpret_cast<const u64 *>(&ctx->d_flags[1]),
                                                             D->uwords, D->uoff);
    PFP_LAUNCHED(ctx);
    if (verify) {
        u64 want = (n + PH_WARPS - 1) / PH_WARPS;
        u64 maxb = (u64)ctx->sm_count * 32;
        verify_entries_k<<<(u32)(want < maxb ? want : maxb), PH_T, 0, ctx->stream>>>(
            n, *uid_of_entry, D->rep, len, in_off, pool, ctx->d_flags);
        PFP_LAUNCHED(ctx);
    }
    PFP_CUDA(ctx, cudaMemcpyAsync(ctx->h_flags, ctx->d_flags, 4 * sizeof(u64), cudaMemcpyDeviceToHost,
                                  ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->h_flags[0] & PFP_ERRBIT_COLLISION)
        return pfp_fail(ctx, PFPB200_E_COLLISION, "fingerprint collision between different phrases");
    if (ctx->h_flags[0] & PFP_ERRBIT_TABLE_FULL)
        return pfp_fail(ctx, PFPB200_E_INTERNAL, "dictionary table overflow in the merge");
    if (ctx->h_flags[0] & PFP_ERRBIT_LIMIT)
        return pfp_fail(ctx, PFPB200_E_LIMIT, "a word occurs more than 2^32-1 times");
    const u64 d = ctx->h_flags[1];
    if (d > 0x7FFFFFFEull)
        return pfp_fail(ctx, PFPB200_E_LIMIT, "%llu distinct words exceed the limit 2^31-2",
                        (unsigned long long)d);
    D->d = d;
    D->pool = const_cast<u64 *>(pool);
    D->pool_words = pool_words;
    D->max_len = (u32)ctx->h_flags[2];
    D->sum_len = ctx->h_flags[3];
    void *fr[] = {rec, tab, in_off};
    for (void *q : fr) PFP_TRY(pfp_free_now(ctx, q));
    return PFPB200_OK;
}
