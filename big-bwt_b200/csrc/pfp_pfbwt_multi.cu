// pfp_pfbwt_multi.cu -- the kernels of the sharded pfbwt (pfpb200_multi_pfbwt_file): the last stage
// of the pipeline spread over the GPUs of a pfpb200_multi handle, for dictionaries of 4 GB and more.
// pfp_multi.cu owns the threads and the barriers and calls the steps below on every rank.
//
// The algorithm is the one of pfp_pfbwt.cu (its comment says what each step computes), with
// 64-bit positions and ranks, and the dictionary suffixes partitioned over the ranks:
//   * every rank holds the whole dictionary and the parse-side streams and derives the same word
//     structure and dense alphabet codes;
//   * a suffix belongs to the rank whose range holds its FIRST KEY (h0 dense-coded symbols, cut
//     behind the terminator); equal first keys never straddle two ranks, so rank g's sorted
//     suffixes are the global slots [base_g, base_g + M_g) and no group of the doubling is ever split;
//   * the rank array is stored by position, block g on rank g, and read / written with direct
//     peer loads and stores (PmRanks); a round is "gather rank(i+h)" | barrier | "sort, scatter
//     the changed ranks" | barrier, so no rank ever reads a partly updated array;
//   * the emission (count / easy / hard) runs on each rank's slice: a group of equal suffixes is
//     whole on one rank, so the merge of the .ilist cursors stays local.
#include "pfp_common.cuh"
#include "pfp_stages.cuh"

constexpr int PM_T = 256;
constexpr u64 PM_BATCH = (u64)1 << 30;          // occurrences sorted at once in the hard groups
constexpr u32 PM_BIG = 512;                     // easy members with more occurrences get a CTA instead of a thread
constexpr u64 PM_CHUNK = (u64)1 << 30;          // dictionary positions per pass of the partition

__device__ __forceinline__ bool pm_term(u8 c) { return c <= PFP_END_OF_WORD; }

__device__ __forceinline__ u64 pm_rank_get(const PmRanks &R, u64 j) {
    const u64 o = j / R.per;
    return R.blk[o][j - o * R.per];
}
__device__ __forceinline__ void pm_rank_put(const PmRanks &R, u64 j, u64 v) {
    const u64 o = j / R.per;
    R.blk[o][j - o * R.per] = v;
}

// ---- 1. word structure -------------------------------------------------------------------------------
__global__ void __launch_bounds__(PM_T) pm_flags_k(const u8 *__restrict__ d, u64 N, u8 *__restrict__ flag) {
    const u64 t = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (t < N) flag[t] = pm_term(d[t]) ? 1 : 0;
}

__global__ void __launch_bounds__(PM_T) pm_wend_k(const u8 *__restrict__ flag, const u32 *__restrict__ wid, u64 N,
                                                  u64 *__restrict__ wend) {
    const u64 t = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (t < N && flag[t]) wend[wid[t]] = t;
}

// ---- 2. first keys and the partition ------------------------------------------------------------------
struct PmCodes { u8 code[256]; };

__device__ __forceinline__ u64 pm_first_key(const u8 *__restrict__ d, u64 N, const u8 *code, int h0, int bs, u64 t) {
    u64 k = 0;
    bool live = !pm_term(d[t]);
    for (int i = 0; i < h0; i++) {
        u32 c = 0;
        if (live) {
            const u8 b = t + i < N ? d[t + i] : (u8)0;
            c = code[b];
            if (pm_term(b)) live = false;                            // the terminator itself is part of the key
        }
        k = (k << bs) | c;
    }
    return k;
}

struct PmRange { u64 lo, hi; int has_lo, has_hi; };
__device__ __forceinline__ bool pm_in(const PmRange &r, u64 k) { return (!r.has_lo || k >= r.lo) && (!r.has_hi || k < r.hi); }

__global__ void __launch_bounds__(PM_T) pm_sample_k(const u8 *__restrict__ d, u64 N, PmCodes cd, int h0, int bs, u64 lo,
                                                    u64 step, u32 ns, u64 *__restrict__ out) {
    __shared__ u8 code[256];
    code[threadIdx.x] = cd.code[threadIdx.x];
    __syncthreads();
    const u32 i = blockIdx.x * PM_T + threadIdx.x;
    if (i < ns) out[i] = pm_first_key(d, N, code, h0, bs, lo + (u64)i * step);
}

__global__ void __launch_bounds__(PM_T) pm_count_k(const u8 *__restrict__ d, u64 N, PmCodes cd, int h0, int bs, PmRange rg,
                                                   unsigned long long *__restrict__ total) {
    __shared__ u8 code[256];
    __shared__ u32 cnt;
    code[threadIdx.x] = cd.code[threadIdx.x];
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    u32 n = 0;
    for (u64 t = (u64)blockIdx.x * PM_T + threadIdx.x; t < N; t += (u64)gridDim.x * PM_T)
        n += pm_in(rg, pm_first_key(d, N, code, h0, bs, t)) ? 1u : 0u;
    n = __reduce_add_sync(0xffffffffu, n);
    if ((threadIdx.x & 31) == 0 && n) atomicAdd(&cnt, n);
    __syncthreads();
    if (threadIdx.x == 0 && cnt) atomicAdd(total, (unsigned long long)cnt);
}

__global__ void __launch_bounds__(PM_T) pm_in_k(const u8 *__restrict__ d, u64 N, PmCodes cd, int h0, int bs, PmRange rg,
                                                u64 c0, u64 n, u8 *__restrict__ flag) {
    __shared__ u8 code[256];
    code[threadIdx.x] = cd.code[threadIdx.x];
    __syncthreads();
    const u64 t = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (t < n) flag[t] = pm_in(rg, pm_first_key(d, N, code, h0, bs, c0 + t)) ? 1 : 0;
}

// the owned positions of chunk [c0, c0 + n), in position order from element e0 on: position, length
// to the terminator, first key; val = element id, slot = local slot of the first sort
__global__ void __launch_bounds__(PM_T) pm_collect_k(const u8 *__restrict__ d, u64 N, PmCodes cd, int h0, int bs,
                                                     const u8 *__restrict__ flag, const u32 *__restrict__ scan, u64 c0,
                                                     u64 n, u64 e0, const u32 *__restrict__ wid,
                                                     const u64 *__restrict__ wend, u64 *__restrict__ pos,
                                                     u32 *__restrict__ sl, u64 *__restrict__ key, u32 *__restrict__ val,
                                                     u32 *__restrict__ slot) {
    __shared__ u8 code[256];
    code[threadIdx.x] = cd.code[threadIdx.x];
    __syncthreads();
    const u64 t = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (t >= n || !flag[t]) return;
    const u64 s = c0 + t, e = e0 + scan[t];
    pos[e] = s;
    sl[e] = (u32)(wend[wid[s]] - s);
    key[e] = pm_first_key(d, N, code, h0, bs, s);
    val[e] = (u32)e;
    slot[e] = (u32)e;
}

// ---- 3. prefix doubling ---------------------------------------------------------------------------------
__global__ void __launch_bounds__(PM_T) pm_gflags_k(const u64 *__restrict__ key, u64 M, u8 *__restrict__ flag) {
    const u64 k = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (k < M) flag[k] = (k == 0 || key[k] != key[k - 1]) ? 1 : 0;
}

// split key form: the sorted key holds the old group only, the second half sits per element in lo[]
__global__ void __launch_bounds__(PM_T) pm_gflags2_k(const u64 *__restrict__ key, const u32 *__restrict__ val,
                                                     const u64 *__restrict__ lo, u64 M, u8 *__restrict__ flag) {
    const u64 k = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (k < M) flag[k] = (k == 0 || key[k] != key[k - 1] || lo[val[k]] != lo[val[k - 1]]) ? 1 : 0;
}

__global__ void __launch_bounds__(PM_T) pm_heads_k(const u8 *__restrict__ flag, const u32 *__restrict__ escan,
                                                   const u32 *__restrict__ slot, u64 M, u32 *__restrict__ head) {
    const u64 k = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (k < M && flag[k]) head[escan[k]] = slot[k];
}

// rank = global slot where the group starts (base + local slot); a suffix leaves when it is alone in
// its group or compared to its end (length + terminator <= h); its rank is stored (into the owner's
// block) only when it changed.  hi_shift: where the old local rank sits in the sorted key (-1: first round)
__global__ void __launch_bounds__(PM_T) pm_update_k(const u8 *__restrict__ flag, const u32 *__restrict__ escan,
                                                    const u32 *__restrict__ slot, const u32 *__restrict__ val,
                                                    const u64 *__restrict__ key, int hi_shift,
                                                    const u32 *__restrict__ head, const u64 *__restrict__ pos,
                                                    const u32 *__restrict__ sl, u64 M, u64 h, u64 base, PmRanks R,
                                                    u64 *__restrict__ sa_pos, u32 *__restrict__ sa_grp,
                                                    u32 *__restrict__ rs, u8 *__restrict__ keep) {
    const u64 k = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (k >= M) return;
    const u32 f = flag[k], e = val[k];
    const u32 r = head[escan[k] + f - 1u];
    const bool single = f && (k + 1 == M || flag[k + 1]);
    const bool done = (u64)sl[e] + 1 <= h;                          // bytes of the suffix + its terminator
    const bool same = hi_shift >= 0 && (u32)(key[k] >> hi_shift) == r;
    const u64 s = pos[e];
    if (!same) pm_rank_put(R, s, base + r);
    rs[k] = r;
    const bool stay = !(single || done);
    keep[k] = stay ? 1 : 0;
    if (!stay) {
        sa_pos[slot[k]] = s;
        sa_grp[slot[k]] = r;
    }
}

// the survivors, compacted, with the key of the next round: (old local rank, rank(i+h), done bit) --
// packed into one u64, or (split) the low part here and the old rank per element in hi[]
__global__ void __launch_bounds__(PM_T) pm_gather_k(const u8 *__restrict__ keep, const u32 *__restrict__ kscan,
                                                    const u32 *__restrict__ slot, const u32 *__restrict__ val,
                                                    const u32 *__restrict__ rs, const u64 *__restrict__ pos,
                                                    const u32 *__restrict__ sl, PmRanks R, u64 M, u64 h, int bn,
                                                    int split, u32 *__restrict__ slot2, u32 *__restrict__ val2,
                                                    u64 *__restrict__ key2, u32 *__restrict__ hi, u64 *__restrict__ lo_e) {
    const u64 k = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (k >= M || !keep[k]) return;
    const u32 p = kscan[k], e = val[k], l = sl[e];
    const u64 r2 = h <= l ? pm_rank_get(R, pos[e] + h) : 0u;       // the terminator's rank is 0
    const u64 lo = (r2 << 1) | (((u64)l + 1 <= 2 * h) ? 1u : 0u);
    slot2[p] = slot[k];
    val2[p] = e;
    if (split) {
        key2[p] = lo;
        hi[e] = rs[k];
        lo_e[e] = lo;
    } else {
        key2[p] = ((u64)rs[k] << (bn + 1)) | lo;
    }
}

__global__ void __launch_bounds__(PM_T) pm_hikey_k(const u32 *__restrict__ val, const u32 *__restrict__ hi, u64 M,
                                                   u64 *__restrict__ key) {
    const u64 k = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (k < M) key[k] = hi[val[k]];
}

// ---- 4. emission on the rank's slice ------------------------------------------------------------------------
struct PmView {
    const u8 *d;
    const u64 *sa_pos;          // per local slot: suffix position
    const u32 *sa_grp;          // per local slot: local rank (start of its group)
    const u32 *wid, *occ, *istart;
    const u64 *wend;
    uint2 *mrec;                // per slot: {word, suffix length}
    u16 *mc;                    // per slot: char in front | whole word << 8 | counts << 9
    u64 N;                      // slots of this rank
    u32 w;
};
__device__ __forceinline__ bool pm_member(const PmView &v, u64 k, u32 &word, u32 &len, bool &full, u8 &c) {
    const u32 m = v.mc[k];
    const uint2 r = v.mrec[k];
    word = r.x; len = r.y;
    full = (m & 0x100u) != 0;
    c = (u8)m;
    return (m & 0x200u) != 0;
}

__global__ void __launch_bounds__(PM_T) pm_member_k(PmView v, u32 *__restrict__ cnt, u8 *__restrict__ newgrp) {
    const u64 k = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (k >= v.N) return;
    const u64 s = v.sa_pos[k];
    newgrp[k] = (k == 0 || v.sa_grp[k] != v.sa_grp[k - 1]) ? 1 : 0;
    u32 word = 0, len = 0, n = 0, m = 0;
    if (!pm_term(v.d[s])) {
        word = v.wid[s];
        len = (u32)(v.wend[word] - s);
        if (len > v.w) {
            const bool full = s == 0 || v.d[s - 1] == PFP_END_OF_WORD;
            const u32 c = (s <= 1) ? 0u : v.d[s - 1];                // d[0] = 0 is the EOF char of the final BWT
            m = c | (full ? 0x100u : 0u) | 0x200u;
            n = v.occ[word];
        }
    }
    v.mrec[k] = make_uint2(word, len);
    v.mc[k] = (u16)m;
    cnt[k] = n;
}

__global__ void __launch_bounds__(PM_T) pm_first_k(const u8 *__restrict__ newgrp, const u32 *__restrict__ gscan, u64 N,
                                                   u32 *__restrict__ first) {
    const u64 k = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (k < N && newgrp[k]) first[gscan[k]] = (u32)k;
}

__global__ void __launch_bounds__(PM_T) pm_mixed_k(PmView v, const u8 *__restrict__ newgrp, const u32 *__restrict__ gscan,
                                                   const u32 *__restrict__ first, u8 *__restrict__ mixed) {
    const u64 k = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (k >= v.N || newgrp[k]) return;
    u32 word, len; bool full; u8 c, c0;
    if (!pm_member(v, k, word, len, full, c)) return;
    const u32 g = gscan[k] + newgrp[k] - 1u;
    pm_member(v, first[g], word, len, full, c0);
    if (c != c0) mixed[g] = 1;
}

__global__ void __launch_bounds__(PM_T) pm_hard_k(const u32 *__restrict__ cnt, const u8 *__restrict__ newgrp,
                                                  const u32 *__restrict__ gscan, const u8 *__restrict__ mixed, u64 N,
                                                  int want_sa, u32 *__restrict__ hcnt) {
    const u64 k = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (k >= N) return;
    const bool alone = newgrp[k] && (k + 1 == N || newgrp[k + 1]);
    const u32 g = gscan[k] + newgrp[k] - 1u;
    hcnt[k] = (!alone && (want_sa || mixed[g])) ? cnt[k] : 0u;
}

__device__ __forceinline__ u64 pm_get5(const u8 *__restrict__ a, u64 i) {
    u64 x = 0;
#pragma unroll
    for (int j = PFP_IBYTES - 1; j >= 0; j--) x = (x << 8) | a[i * PFP_IBYTES + j];
    return x;
}
__device__ __forceinline__ void pm_put5(u8 *__restrict__ a, u64 i, u64 x) {
#pragma unroll
    for (int j = 0; j < PFP_IBYTES; j++) a[i * PFP_IBYTES + j] = (u8)(x >> (8 * j));
}

__global__ void __launch_bounds__(PM_T) pm_easy_k(PmView v, const u32 *__restrict__ cnt, const u32 *__restrict__ hcnt,
                                                  const u64 *__restrict__ off, const u32 *__restrict__ ilist,
                                                  const u8 *__restrict__ bwlast, const u8 *__restrict__ bwsai,
                                                  u8 *__restrict__ bwt, u8 *__restrict__ sa5, u32 *__restrict__ big,
                                                  u32 *__restrict__ big_n, u32 big_cap) {
    const u64 k = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (k >= v.N || cnt[k] == 0 || hcnt[k] != 0) return;
    u32 word, len; bool full; u8 c;
    pm_member(v, k, word, len, full, c);
    const u32 n = cnt[k];
    if (n > PM_BIG) {
        const u32 i = atomicAdd(big_n, 1u);
        if (i < big_cap) big[i] = (u32)k;
        return;
    }
    const u64 o = off[k];
    const u32 is = v.istart[word] + 1u;                              // ilist[0] is the end symbol's entry
    for (u32 j = 0; j < n; j++) {
        const u32 ip = (full || sa5) ? ilist[is + j] : 0u;
        bwt[o + j] = full ? bwlast[ip] : c;
        if (sa5) pm_put5(sa5, o + j, (full && word == 0) ? pm_get5(bwsai, 0) - v.w : pm_get5(bwsai, ip) - len);
    }
}

__global__ void __launch_bounds__(PM_T) pm_easy_big_k(PmView v, const u32 *__restrict__ big, const u32 *__restrict__ big_n,
                                                      u32 big_cap, const u32 *__restrict__ cnt, const u64 *__restrict__ off,
                                                      const u32 *__restrict__ ilist, const u8 *__restrict__ bwlast,
                                                      const u8 *__restrict__ bwsai, u8 *__restrict__ bwt,
                                                      u8 *__restrict__ sa5) {
    const u32 nbig = min(*big_n, big_cap);
    for (u32 b = blockIdx.x; b < nbig; b += gridDim.x) {
        const u64 k = big[b];
        u32 word, len; bool full; u8 c;
        pm_member(v, k, word, len, full, c);
        const u32 n = cnt[k];
        const u64 o = off[k];
        const u32 is = v.istart[word] + 1u;
        for (u32 j = threadIdx.x; j < n; j += PM_T) {
            const u32 ip = (full || sa5) ? ilist[is + j] : 0u;
            bwt[o + j] = full ? bwlast[ip] : c;
            if (sa5) pm_put5(sa5, o + j, (full && word == 0) ? pm_get5(bwsai, 0) - v.w : pm_get5(bwsai, ip) - len);
        }
    }
}

__global__ void __launch_bounds__(PM_T) pm_gen_k(PmView v, const u32 *__restrict__ hcnt, const u64 *__restrict__ hoff,
                                                 const u32 *__restrict__ gscan, const u8 *__restrict__ newgrp,
                                                 const u32 *__restrict__ ilist, u64 k0, u64 k1, u64 e0, u32 g0,
                                                 u64 *__restrict__ key, u32 *__restrict__ val) {
    const u64 k = k0 + (u64)blockIdx.x * PM_T + threadIdx.x;
    if (k >= k1 || hcnt[k] == 0) return;
    const u32 word = v.mrec[k].x;
    const u32 is = v.istart[word] + 1u, n = hcnt[k];
    const u64 g = (u64)(gscan[k] + newgrp[k] - 1u - g0) << 32;
    const u64 e = hoff[k] - e0;
    for (u32 j = 0; j < n; j++) {
        key[e + j] = g | ilist[is + j];
        val[e + j] = (u32)k;
    }
}

__global__ void __launch_bounds__(PM_T) pm_scatter_k(PmView v, const u64 *__restrict__ key, const u32 *__restrict__ val,
                                                     u64 ne, u64 e0, u32 g0, const u32 *__restrict__ first,
                                                     const u64 *__restrict__ off, const u64 *__restrict__ hoff,
                                                     const u8 *__restrict__ bwsai, u8 *__restrict__ bwt,
                                                     u8 *__restrict__ sa5) {
    const u64 e = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (e >= ne) return;
    const u64 kk = key[e];
    const u32 k = val[e], f = first[(u32)(kk >> 32) + g0];
    const u64 pos = off[f] + (e0 + e - hoff[f]);
    u32 word, len; bool full; u8 c;
    pm_member(v, k, word, len, full, c);
    bwt[pos] = c;
    if (sa5) pm_put5(sa5, pos, pm_get5(bwsai, (u32)kk) - len);
}

__global__ void pm_batch_k(const u64 *__restrict__ hoff, const u32 *__restrict__ gscan, const u8 *__restrict__ newgrp,
                           const u32 *__restrict__ first, u64 ngroups, u64 ka, u64 N, u64 cap, u64 *__restrict__ out) {
    const u64 target = hoff[ka] + cap;
    u64 kb = N;
    if (hoff[N] > target) {
        u64 a = ka, b = N;
        while (a < b) {
            const u64 m = (a + b) >> 1;
            if (hoff[m] <= target) a = m + 1; else b = m;
        }
        const u64 kl = a - 1;
        const u64 g = gscan[kl] + newgrp[kl] - 1u;
        kb = first[g];
        if (kb <= ka) kb = g + 1 < ngroups ? first[g + 1] : N;
    }
    const u64 ga = gscan[ka] + newgrp[ka] - 1u;
    out[0] = kb;
    out[1] = hoff[kb];
    out[2] = ga;
    out[3] = kb < N ? gscan[kb] + newgrp[kb] - 1u - ga : ngroups - ga;
}

// runs of the BWT at the piece's edges: prev / next = the chars of the neighbouring non-empty pieces (-1: none)
__global__ void __launch_bounds__(PM_T) pm_runs_k(const u8 *__restrict__ bwt, u64 n, int at_end, int prev, int next,
                                                  u32 *__restrict__ flag) {
    const u64 i = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (i >= n) return;
    bool f;
    if (at_end) f = i + 1 == n ? (next < 0 || bwt[i] != (u8)next) : bwt[i + 1] != bwt[i];
    else f = i == 0 ? (prev < 0 || bwt[0] != (u8)prev) : bwt[i] != bwt[i - 1];
    flag[i] = f ? 1u : 0u;
}
__global__ void __launch_bounds__(PM_T) pm_sample_sa_k(const u32 *__restrict__ flag, const u64 *__restrict__ fscan,
                                                       const u8 *__restrict__ sa5, u64 n, u64 off, u8 *__restrict__ out) {
    const u64 i = (u64)blockIdx.x * PM_T + threadIdx.x;
    if (i >= n || !flag[i]) return;
    const u64 o = fscan[i];
    pm_put5(out, 2 * o, off + i);                                    // (global BWT position, suffix-array value)
    pm_put5(out, 2 * o + 1, pm_get5(sa5, i));
}

// ---- host side -----------------------------------------------------------------------------------------------
static int pm_bits(u64 v) {
    int b = 1;
    while (b < 64 && (v >> b) != 0) b++;
    return b;
}

#define PM_LAUNCH(ctx, n, kernel, ...)                                                          \
    do {                                                                                        \
        if ((n) > 0) {                                                                          \
            kernel<<<pfp_blocks((n), PM_T), PM_T, 0, (ctx)->stream>>>(__VA_ARGS__);              \
            PFP_LAUNCHED(ctx);                                                                  \
        }                                                                                       \
    } while (0)

static int pm_sync_read(pfpb200_ctx *ctx, int slot, int n) {
    PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[slot], &ctx->d_flags[slot], n * sizeof(u64), cudaMemcpyDeviceToHost,
                                  ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return PFPB200_OK;
}

int pm_words(pfpb200_ctx *ctx, PmState &S) {
    const u64 N = S.N;
    PFP_CUDA(ctx, cudaMemsetAsync(ctx->d_flags, 0, 12 * sizeof(u64), ctx->stream));
    PFP_TRY(pfp_alloc_t(ctx, &S.tflag, N));
    PFP_TRY(pfp_alloc_t(ctx, &S.wid, N));
    PFP_TRY(pfp_alloc_t(ctx, &S.wend, S.dwords + 2));
    PFP_TRY(pfp_alloc_t(ctx, &S.istart, S.dwords + 1));
    PM_LAUNCH(ctx, N, pm_flags_k, S.d, N, S.tflag);
    PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, S.tflag, S.wid, N, reinterpret_cast<u32 *>(&ctx->d_flags[1])));
    PFP_TRY(pfp_exclusive_scan_u32(ctx, S.occ, S.istart, S.dwords, reinterpret_cast<u32 *>(&ctx->d_flags[2])));
    PFP_TRY(pm_sync_read(ctx, 1, 2));
    if ((u32)ctx->h_flags[1] != S.dwords + 1)
        return pfp_fail(ctx, PFPB200_E_ARG, "the dictionary holds %u words, .occ %llu", (u32)ctx->h_flags[1] - 1,
                        (unsigned long long)S.dwords);
    if ((u64)(u32)ctx->h_flags[2] + 1 != S.psize) return pfp_fail(ctx, PFPB200_E_ARG, "sum of .occ + 1 != size of .ilist");
    PM_LAUNCH(ctx, N, pm_wend_k, S.tflag, S.wid, N, S.wend);
    PFP_TRY(pfp_free_now(ctx, S.tflag));                             // the word ids and ends are all that is kept
    S.tflag = nullptr;
    // the dense alphabet codes of the first key, as the single-GPU path derives them
    u32 *present = reinterpret_cast<u32 *>(&ctx->d_flags[8]);
    PFP_TRY(pfp_dict_alphabet(ctx, S.d, N, present));
    PFP_TRY(pm_sync_read(ctx, 8, 4));
    memset(S.code, 0, sizeof(S.code));
    u32 sigma = 1;
    S.code[0] = S.code[1] = 1;
    const u32 *pm = reinterpret_cast<const u32 *>(&ctx->h_flags[8]);
    for (u32 c = 2; c < 256; c++)
        if (pm[c >> 5] & (1u << (c & 31))) S.code[c] = (u8)++sigma;
    S.bs = pm_bits(sigma);
    S.h0 = 64 / S.bs > 32 ? 32 : 64 / S.bs;
    return PFPB200_OK;
}

static PmCodes pm_codes(const PmState &S) {
    PmCodes cd;
    memcpy(cd.code, S.code, 256);
    return cd;
}

int pm_sample(pfpb200_ctx *ctx, PmState &S, u64 lo, u64 hi, u32 want, u64 *h_out, u32 *got) {
    *got = 0;
    if (hi <= lo) return PFPB200_OK;
    const u64 n = hi - lo;
    const u32 ns = (u32)(n < want ? n : want);
    u64 *d_out = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &d_out, ns));
    pm_sample_k<<<pfp_blocks(ns, PM_T), PM_T, 0, ctx->stream>>>(S.d, S.N, pm_codes(S), S.h0, S.bs, lo, n / ns, ns, d_out);
    PFP_LAUNCHED(ctx);
    PFP_CUDA(ctx, cudaMemcpyAsync(h_out, d_out, ns * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    PFP_TRY(pfp_free_now(ctx, d_out));
    *got = ns;
    return PFPB200_OK;
}

int pm_count(pfpb200_ctx *ctx, PmState &S, u64 klo, u64 khi, int has_lo, int has_hi, u64 *count) {
    S.rg_lo = klo; S.rg_hi = khi; S.rg_has_lo = has_lo; S.rg_has_hi = has_hi;
    const PmRange rg{klo, khi, has_lo, has_hi};
    PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[1], 0, sizeof(u64), ctx->stream));
    pm_count_k<<<ctx->sm_count * 8, PM_T, 0, ctx->stream>>>(S.d, S.N, pm_codes(S), S.h0, S.bs, rg,
                                                            reinterpret_cast<unsigned long long *>(&ctx->d_flags[1]));
    PFP_LAUNCHED(ctx);
    PFP_TRY(pm_sync_read(ctx, 1, 1));
    *count = ctx->h_flags[1];
    return PFPB200_OK;
}

int pm_collect(pfpb200_ctx *ctx, PmState &S, int split) {
    const u64 M = S.M0, N = S.N;
    S.split = split;
    S.bn = pm_bits(N);
    S.bm = pm_bits(M);
    PFP_TRY(pfp_alloc_t(ctx, &S.pos, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.sl, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.k0, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.k1, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.v0, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.v1, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.slot, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.slot2, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.head, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.escan, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.rs, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.flag, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.keep, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.sa_pos, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.sa_grp, M));
    if (split) {
        PFP_TRY(pfp_alloc_t(ctx, &S.hi, M));
        PFP_TRY(pfp_alloc_t(ctx, &S.lo, M));
    }
    const PmRange rg{S.rg_lo, S.rg_hi, S.rg_has_lo, S.rg_has_hi};
    if (M) {
        const u64 chunk = N < PM_CHUNK ? N : PM_CHUNK;
        u8 *cf = nullptr;
        u32 *cs = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &cf, chunk));
        PFP_TRY(pfp_alloc_t(ctx, &cs, chunk));
        u64 e0 = 0;
        for (u64 c0 = 0; c0 < N && e0 < M; c0 += chunk) {
            const u64 n = N - c0 < chunk ? N - c0 : chunk;
            pm_in_k<<<pfp_blocks(n, PM_T), PM_T, 0, ctx->stream>>>(S.d, N, pm_codes(S), S.h0, S.bs, rg, c0, n, cf);
            PFP_LAUNCHED(ctx);
            PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, cf, cs, n, reinterpret_cast<u32 *>(&ctx->d_flags[1])));
            pm_collect_k<<<pfp_blocks(n, PM_T), PM_T, 0, ctx->stream>>>(S.d, N, pm_codes(S), S.h0, S.bs, cf, cs, c0, n, e0,
                                                                        S.wid, S.wend, S.pos, S.sl, S.k0, S.v0, S.slot);
            PFP_LAUNCHED(ctx);
            PFP_TRY(pm_sync_read(ctx, 1, 1));
            e0 += (u32)ctx->h_flags[1];
        }
        PFP_TRY(pfp_free_now(ctx, cf));
        PFP_TRY(pfp_free_now(ctx, cs));
        if (e0 != M) return pfp_fail(ctx, PFPB200_E_INTERNAL, "pfbwt: partition counted %llu suffixes, collected %llu",
                                     (unsigned long long)M, (unsigned long long)e0);
    }
    PFP_TRY(pfp_radix_sort_pairs(ctx, S.k0, S.v0, S.k1, S.v1, M, 0, S.h0 * S.bs, &S.ks, &S.vs));
    S.M = M;
    return PFPB200_OK;
}

int pm_update(pfpb200_ctx *ctx, PmState &S, const PmRanks &R, u64 h, int first, u64 *active) {
    const u64 M = S.M;
    int hi_shift = -1;
    if (!first) hi_shift = S.split ? 0 : S.bn + 1;
    if (S.split && !first) PM_LAUNCH(ctx, M, pm_gflags2_k, S.ks, S.vs, S.lo, M, S.flag);
    else PM_LAUNCH(ctx, M, pm_gflags_k, S.ks, M, S.flag);
    PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, S.flag, S.escan, M, nullptr));
    PM_LAUNCH(ctx, M, pm_heads_k, S.flag, S.escan, S.slot, M, S.head);
    PM_LAUNCH(ctx, M, pm_update_k, S.flag, S.escan, S.slot, S.vs, S.ks, hi_shift, S.head, S.pos, S.sl, M, h, S.base, R,
              S.sa_pos, S.sa_grp, S.rs, S.keep);
    PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, S.keep, S.escan, M, reinterpret_cast<u32 *>(&ctx->d_flags[1])));
    PFP_TRY(pm_sync_read(ctx, 1, 1));
    S.M2 = M ? (u32)ctx->h_flags[1] : 0;
    *active = S.M2;
    return PFPB200_OK;
}

int pm_gather(pfpb200_ctx *ctx, PmState &S, const PmRanks &R, u64 h) {
    const u64 M = S.M;
    S.ko = S.ks == S.k0 ? S.k1 : S.k0;
    S.vo = S.vs == S.v0 ? S.v1 : S.v0;
    PM_LAUNCH(ctx, M, pm_gather_k, S.keep, S.escan, S.slot, S.vs, S.rs, S.pos, S.sl, R, M, h, S.bn, S.split, S.slot2, S.vo,
              S.ko, S.hi, S.lo);
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return PFPB200_OK;
}

int pm_sort(pfpb200_ctx *ctx, PmState &S) {
    { u32 *t = S.slot; S.slot = S.slot2; S.slot2 = t; }
    const u64 M = S.M = S.M2;
    if (!S.split) return pfp_radix_sort_pairs(ctx, S.ko, S.vo, S.ks, S.vs, M, 0, S.bm + S.bn + 1, &S.ks, &S.vs);
    // two stable LSD sorts: (rank(i+h), done) first, then the old local rank
    u64 *ka; u32 *va;
    PFP_TRY(pfp_radix_sort_pairs(ctx, S.ko, S.vo, S.ks, S.vs, M, 0, S.bn + 1, &ka, &va));
    u64 *kb = ka == S.k0 ? S.k1 : S.k0;
    u32 *vb = va == S.v0 ? S.v1 : S.v0;
    PM_LAUNCH(ctx, M, pm_hikey_k, va, S.hi, M, kb);
    return pfp_radix_sort_pairs(ctx, kb, va, ka, vb, M, 0, S.bm, &S.ks, &S.vs);
}

int pm_sort_done(pfpb200_ctx *ctx, PmState &S) {
    PFP_TRY(pfp_free_now(ctx, S.k0)); PFP_TRY(pfp_free_now(ctx, S.k1)); PFP_TRY(pfp_free_now(ctx, S.v0));
    PFP_TRY(pfp_free_now(ctx, S.v1)); PFP_TRY(pfp_free_now(ctx, S.slot)); PFP_TRY(pfp_free_now(ctx, S.slot2));
    PFP_TRY(pfp_free_now(ctx, S.head)); PFP_TRY(pfp_free_now(ctx, S.keep)); PFP_TRY(pfp_free_now(ctx, S.rs));
    PFP_TRY(pfp_free_now(ctx, S.pos)); PFP_TRY(pfp_free_now(ctx, S.sl)); PFP_TRY(pfp_free_now(ctx, S.hi));
    PFP_TRY(pfp_free_now(ctx, S.lo));
    S.lo = nullptr;
    S.k0 = S.k1 = S.ks = nullptr; S.v0 = S.v1 = S.vs = nullptr;
    S.slot = S.slot2 = S.head = S.rs = S.hi = nullptr; S.keep = nullptr; S.pos = nullptr; S.sl = nullptr;
    return PFPB200_OK;
}

// per slot: occurrences, member record, group starts -> this rank's chars
int pm_count_chars(pfpb200_ctx *ctx, PmState &S) {
    const u64 N = S.M0;
    PFP_TRY(pfp_alloc_t(ctx, &S.mrec, N));
    PFP_TRY(pfp_alloc_t(ctx, &S.mc, N));
    PFP_TRY(pfp_alloc_t(ctx, &S.cnt, N));
    PFP_TRY(pfp_alloc_t(ctx, &S.off, N + 1));
    S.newgrp = S.flag;
    S.gscan = S.escan;
    const PmView V{S.d, S.sa_pos, S.sa_grp, S.wid, S.occ, S.istart, S.wend, S.mrec, S.mc, N, S.w};
    PM_LAUNCH(ctx, N, pm_member_k, V, S.cnt, S.newgrp);
    PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, S.newgrp, S.gscan, N, reinterpret_cast<u32 *>(&ctx->d_flags[1])));
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, S.cnt, S.off, N, &ctx->d_flags[2]));
    PFP_TRY(pm_sync_read(ctx, 1, 2));
    S.ngroups = N ? (u32)ctx->h_flags[1] : 0;
    S.chars = N ? ctx->h_flags[2] : 0;
    return PFPB200_OK;
}

// easy and hard members into this rank's piece of the BWT (and SA)
int pm_fill(pfpb200_ctx *ctx, PmState &S) {
    const u64 N = S.M0, n_bwt = S.chars;
    const bool want_sa = (S.flags & (PFPB200_PFBWT_SA | PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA)) != 0;
    const PmView V{S.d, S.sa_pos, S.sa_grp, S.wid, S.occ, S.istart, S.wend, S.mrec, S.mc, N, S.w};
    u32 *hcnt = nullptr, *first = nullptr;
    u8 *mixed = nullptr;
    u64 *hoff = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &hcnt, N));
    PFP_TRY(pfp_alloc_t(ctx, &hoff, N + 1));
    PFP_TRY(pfp_alloc_t(ctx, &first, S.ngroups + 1));
    PFP_TRY(pfp_alloc_t(ctx, &mixed, S.ngroups + 1));
    PFP_CUDA(ctx, cudaMemsetAsync(mixed, 0, S.ngroups + 1, ctx->stream));
    PM_LAUNCH(ctx, N, pm_first_k, S.newgrp, S.gscan, N, first);
    PM_LAUNCH(ctx, N, pm_mixed_k, V, S.newgrp, S.gscan, first, mixed);
    PM_LAUNCH(ctx, N, pm_hard_k, S.cnt, S.newgrp, S.gscan, mixed, N, want_sa ? 1 : 0, hcnt);
    PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[3], 0, sizeof(u64), ctx->stream));
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, hcnt, hoff, N, &ctx->d_flags[3]));
    PFP_CUDA(ctx, cudaMemcpyAsync(&hoff[N], &ctx->d_flags[3], sizeof(u64), cudaMemcpyDeviceToDevice, ctx->stream));
    PFP_TRY(pm_sync_read(ctx, 3, 1));
    const u64 n_hard = S.n_hard = ctx->h_flags[3];
    PFP_TRY(pfp_alloc_t(ctx, &S.bwt, n_bwt));
    if (want_sa) PFP_TRY(pfp_alloc_t(ctx, &S.sa5, n_bwt * PFP_IBYTES));
    const u32 big_cap = (u32)(n_bwt / PM_BIG + 1);
    u32 *big = nullptr, *big_n = reinterpret_cast<u32 *>(&ctx->d_flags[6]);
    PFP_TRY(pfp_alloc_t(ctx, &big, big_cap));
    PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[6], 0, sizeof(u64), ctx->stream));
    PM_LAUNCH(ctx, N, pm_easy_k, V, S.cnt, hcnt, S.off, S.ilist, S.bwlast, S.bwsai, S.bwt, S.sa5, big, big_n, big_cap);
    if (N) {
        pm_easy_big_k<<<ctx->sm_count * 8, PM_T, 0, ctx->stream>>>(V, big, big_n, big_cap, S.cnt, S.off, S.ilist, S.bwlast,
                                                                  S.bwsai, S.bwt, S.sa5);
        PFP_LAUNCHED(ctx);
    }
    if (n_hard) {
        const u64 cap = n_hard < PM_BATCH ? n_hard : PM_BATCH;
        u64 *hk0 = nullptr, *hk1 = nullptr;
        u32 *hv0 = nullptr, *hv1 = nullptr;
        u64 ka = 0, ea = 0, buf = 0;
        while (ka < N && ea < n_hard) {
            pm_batch_k<<<1, 1, 0, ctx->stream>>>(hoff, S.gscan, S.newgrp, first, S.ngroups, ka, N, cap, &ctx->d_flags[4]);
            PFP_LAUNCHED(ctx);
            PFP_TRY(pm_sync_read(ctx, 4, 4));
            const u64 kb = ctx->h_flags[4], eb = ctx->h_flags[5], ng = ctx->h_flags[7];
            const u32 g0 = (u32)ctx->h_flags[6];
            const u64 ne = eb - ea;
            if (ne >= 0xFFFFFFFEull)
                return pfp_fail(ctx, PFPB200_E_LIMIT, "pfbwt: one group of equal suffixes with 2^32 occurrences");
            if (ne) {
                if (ne > buf) {
                    if (hk0) { PFP_TRY(pfp_free_now(ctx, hk0)); PFP_TRY(pfp_free_now(ctx, hk1)); PFP_TRY(pfp_free_now(ctx, hv0)); PFP_TRY(pfp_free_now(ctx, hv1)); }
                    buf = ne > cap ? ne : cap;
                    PFP_TRY(pfp_alloc_t(ctx, &hk0, buf));
                    PFP_TRY(pfp_alloc_t(ctx, &hk1, buf));
                    PFP_TRY(pfp_alloc_t(ctx, &hv0, buf));
                    PFP_TRY(pfp_alloc_t(ctx, &hv1, buf));
                }
                pm_gen_k<<<pfp_blocks(kb - ka, PM_T), PM_T, 0, ctx->stream>>>(V, hcnt, hoff, S.gscan, S.newgrp, S.ilist, ka, kb,
                                                                             ea, g0, hk0, hv0);
                PFP_LAUNCHED(ctx);
                u64 *sk = nullptr;
                u32 *sv = nullptr;
                PFP_TRY(pfp_radix_sort_pairs(ctx, hk0, hv0, hk1, hv1, ne, 0, 32 + pm_bits(ng), &sk, &sv));
                pm_scatter_k<<<pfp_blocks(ne, PM_T), PM_T, 0, ctx->stream>>>(V, sk, sv, ne, ea, g0, first, S.off, hoff,
                                                                            S.bwsai, S.bwt, S.sa5);
                PFP_LAUNCHED(ctx);
            }
            ka = kb;
            ea = eb;
        }
    }
    if (n_bwt) {                                                     // the edge chars, for the runs across pieces
        PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[9], S.bwt, 1, cudaMemcpyDeviceToHost, ctx->stream));
        PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[10], S.bwt + n_bwt - 1, 1, cudaMemcpyDeviceToHost, ctx->stream));
    }
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    S.c_first = n_bwt ? (int)*(const u8 *)&ctx->h_flags[9] : -1;
    S.c_last = n_bwt ? (int)*(const u8 *)&ctx->h_flags[10] : -1;
    return PFPB200_OK;
}

// the (global position, SA value) pairs at the starts (at_end = 0) / ends of the runs inside this piece
int pm_samples(pfpb200_ctx *ctx, PmState &S, int at_end, int prev, int next, u64 off) {
    const u64 n = S.chars;
    u8 **outp = at_end ? &S.esa : &S.ssa;
    u64 *nr = at_end ? &S.n_esa : &S.n_ssa;
    *nr = 0;
    if (n == 0) return PFPB200_OK;
    u32 *rf = nullptr;
    u64 *rscan = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &rf, n));
    PFP_TRY(pfp_alloc_t(ctx, &rscan, n));
    PM_LAUNCH(ctx, n, pm_runs_k, S.bwt, n, at_end, prev, next, rf);
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, rf, rscan, n, &ctx->d_flags[5]));
    PFP_TRY(pm_sync_read(ctx, 5, 1));
    *nr = ctx->h_flags[5];
    PFP_TRY(pfp_alloc_t(ctx, outp, *nr * 2 * PFP_IBYTES));
    PM_LAUNCH(ctx, n, pm_sample_sa_k, rf, rscan, S.sa5, n, off, *outp);
    PFP_TRY(pfp_free_now(ctx, rf));
    PFP_TRY(pfp_free_now(ctx, rscan));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return PFPB200_OK;
}
