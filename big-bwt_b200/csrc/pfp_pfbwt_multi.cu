// pfp_pfbwt_multi.cu -- the sharded suffix sort of pfbwt (pfpb200_multi_pfbwt_file): the last stage
// of the pipeline spread over the GPUs of a pfpb200_multi handle, for dictionaries of 4 GB and more.
// pfp_multi.cu owns the threads and the barriers and calls the steps below on every rank.
//
// The word structure, the emission and the sampled suffix array are the ones of pfp_pfbwt.cu (pb_words,
// pb_plan, pb_write_windows, pb_samples; its comment says what each step computes).  What is here is the suffix sort
// that one GPU cannot do, with 64-bit positions and ranks and the dictionary suffixes partitioned over
// the ranks:
//   * every rank holds the whole dictionary and the parse-side streams and derives the same word
//     structure (word ends, no word per position) and dense alphabet codes;
//   * a suffix belongs to the rank whose range holds its FIRST KEY (h0 dense-coded symbols, cut
//     behind the terminator); equal first keys never straddle two ranks, so rank g's sorted
//     suffixes are the global slots [base_g, base_g + M_g) and no group of the doubling is ever split;
//   * the rank array is stored by position, block g on rank g, and read / written with direct
//     peer loads and stores (PmRanks); a round is "gather rank(i+h)" | barrier | "sort, scatter
//     the changed ranks" | barrier, so no rank ever reads a partly updated array;
//   * the emission runs on each rank's slice (sa_pos / sa_grp / sa_word, read through PbSplitSlots): a
//     group of equal suffixes is whole on one rank, so the merge of the .ilist cursors stays local.
#include "pfp_common.cuh"
#include "pfp_stages.cuh"

__device__ __forceinline__ u64 pm_rank_get(const PmRanks &R, u64 j) {
    const u64 o = j / R.per;
    return R.blk[o][j - o * R.per];
}
__device__ __forceinline__ void pm_rank_put(const PmRanks &R, u64 j, u64 v) {
    const u64 o = j / R.per;
    R.blk[o][j - o * R.per] = v;
}

// ---- 1. the partition by first key -------------------------------------------------------------------------
struct PmRange { u64 lo, hi; int has_lo, has_hi; };
__device__ __forceinline__ bool pm_in(const PmRange &r, u64 k) { return (!r.has_lo || k >= r.lo) && (!r.has_hi || k < r.hi); }

__global__ void __launch_bounds__(PB_T) pm_sample_k(const u8 *__restrict__ d, u64 N, PbCodes cd, int h0, int bs, u64 lo,
                                                    u64 step, u32 ns, u64 *__restrict__ out) {
    __shared__ u8 code[256];
    code[threadIdx.x] = cd.code[threadIdx.x];
    __syncthreads();
    const u32 i = blockIdx.x * PB_T + threadIdx.x;
    if (i < ns) out[i] = pb_first_key(d, N, code, h0, bs, lo + (u64)i * step);
}

__global__ void __launch_bounds__(PB_T) pm_count_k(const u8 *__restrict__ d, u64 N, PbCodes cd, int h0, int bs, PmRange rg,
                                                   unsigned long long *__restrict__ total) {
    __shared__ u8 code[256];
    __shared__ u32 cnt;
    code[threadIdx.x] = cd.code[threadIdx.x];
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    u32 n = 0;
    for (u64 t = (u64)blockIdx.x * PB_T + threadIdx.x; t < N; t += (u64)gridDim.x * PB_T)
        n += pm_in(rg, pb_first_key(d, N, code, h0, bs, t)) ? 1u : 0u;
    n = __reduce_add_sync(0xffffffffu, n);
    if ((threadIdx.x & 31) == 0 && n) atomicAdd(&cnt, n);
    __syncthreads();
    if (threadIdx.x == 0 && cnt) atomicAdd(total, (unsigned long long)cnt);
}

__global__ void __launch_bounds__(PB_T) pm_in_k(const u8 *__restrict__ d, u64 N, PbCodes cd, int h0, int bs, PmRange rg,
                                                u64 c0, u64 n, u8 *__restrict__ flag) {
    __shared__ u8 code[256];
    code[threadIdx.x] = cd.code[threadIdx.x];
    __syncthreads();
    const u64 t = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (t < n) flag[t] = pm_in(rg, pb_first_key(d, N, code, h0, bs, c0 + t)) ? 1 : 0;
}

// the owned positions of chunk [c0, c0 + n), in position order from element e0 on: position, word,
// length to the terminator, first key; val = element id, slot = local slot of the first sort.  The word
// of s is the first k with wend[k] >= s (nw word ends): a binary search, on the same path for the
// neighbouring positions of a warp.
__global__ void __launch_bounds__(PB_T) pm_collect_k(const u8 *__restrict__ d, u64 N, PbCodes cd, int h0, int bs,
                                                     const u8 *__restrict__ flag, const u32 *__restrict__ scan, u64 c0,
                                                     u64 n, u64 e0, const u64 *__restrict__ wend, u64 nw,
                                                     u64 *__restrict__ pos, u32 *__restrict__ we, u32 *__restrict__ sl,
                                                     u64 *__restrict__ key, u32 *__restrict__ val,
                                                     u32 *__restrict__ slot) {
    __shared__ u8 code[256];
    code[threadIdx.x] = cd.code[threadIdx.x];
    __syncthreads();
    const u64 t = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (t >= n || !flag[t]) return;
    const u64 s = c0 + t, e = e0 + scan[t];
    u64 a = 0, b = nw - 1;                                       // wend[nw - 1] = N - 1 >= s
    while (a < b) {
        const u64 m = (a + b) >> 1;
        if (wend[m] < s) a = m + 1; else b = m;
    }
    pos[e] = s;
    we[e] = (u32)a;
    sl[e] = (u32)(wend[a] - s);
    key[e] = pb_first_key(d, N, code, h0, bs, s);
    val[e] = (u32)e;
    slot[e] = (u32)e;
}

// ---- 2. prefix doubling ---------------------------------------------------------------------------------
// split key form: the sorted key holds the old group only, the second half sits per element in lo[]
__global__ void __launch_bounds__(PB_T) pm_gflags2_k(const u64 *__restrict__ key, const u32 *__restrict__ val,
                                                     const u64 *__restrict__ lo, u64 M, u8 *__restrict__ flag) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k < M) flag[k] = (k == 0 || key[k] != key[k - 1] || lo[val[k]] != lo[val[k - 1]]) ? 1 : 0;
}

// rank = global slot where the group starts (base + local slot); a suffix leaves when it is alone in
// its group or compared to its end (length + terminator <= h); its rank is stored (into the owner's
// block) only when it changed.  hi_shift: where the old local rank sits in the sorted key (-1: first round)
__global__ void __launch_bounds__(PB_T) pm_update_k(const u8 *__restrict__ flag, const u32 *__restrict__ escan,
                                                    const u32 *__restrict__ slot, const u32 *__restrict__ val,
                                                    const u64 *__restrict__ key, int hi_shift,
                                                    const u32 *__restrict__ head, const u64 *__restrict__ pos,
                                                    const u32 *__restrict__ sl, const u32 *__restrict__ we, u64 M,
                                                    u64 h, u64 base, PmRanks R, u64 *__restrict__ sa_pos,
                                                    u32 *__restrict__ sa_grp, u32 *__restrict__ sa_word,
                                                    u32 *__restrict__ rs, u8 *__restrict__ keep) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
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
        sa_word[slot[k]] = we[e];
    }
}

// the survivors, compacted, with the key of the next round: (old local rank, rank(i+h), done bit) --
// packed into one u64, or (split) the low part here and the old rank per element in hi[]
__global__ void __launch_bounds__(PB_T) pm_gather_k(const u8 *__restrict__ keep, const u32 *__restrict__ kscan,
                                                    const u32 *__restrict__ slot, const u32 *__restrict__ val,
                                                    const u32 *__restrict__ rs, const u64 *__restrict__ pos,
                                                    const u32 *__restrict__ sl, PmRanks R, u64 M, u64 h, int bn,
                                                    int split, u32 *__restrict__ slot2, u32 *__restrict__ val2,
                                                    u64 *__restrict__ key2, u32 *__restrict__ hi, u64 *__restrict__ lo_e) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
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

__global__ void __launch_bounds__(PB_T) pm_hikey_k(const u32 *__restrict__ val, const u32 *__restrict__ hi, u64 M,
                                                   u64 *__restrict__ key) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k < M) key[k] = hi[val[k]];
}

// ---- host side -----------------------------------------------------------------------------------------------
int pm_sample(pfpb200_ctx *ctx, PmState &S, u64 lo, u64 hi, u32 want, u64 *h_out, u32 *got) {
    *got = 0;
    if (hi <= lo) return PFPB200_OK;
    const u64 n = hi - lo;
    const u32 ns = (u32)(n < want ? n : want);
    u64 *d_out = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &d_out, ns));
    pm_sample_k<<<pfp_blocks(ns, PB_T), PB_T, 0, ctx->stream>>>(S.in.d, S.in.N, S.wd.cd, S.wd.h0, S.wd.bs, lo, n / ns, ns, d_out);
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
    pm_count_k<<<ctx->sm_count * 8, PB_T, 0, ctx->stream>>>(S.in.d, S.in.N, S.wd.cd, S.wd.h0, S.wd.bs, rg,
                                                            reinterpret_cast<unsigned long long *>(&ctx->d_flags[1]));
    PFP_LAUNCHED(ctx);
    PFP_TRY(pb_sync_read(ctx, 1, 1));
    *count = ctx->h_flags[1];
    return PFPB200_OK;
}

int pm_collect(pfpb200_ctx *ctx, PmState &S, int split) {
    const u64 M = S.M0, N = S.in.N;
    S.split = split;
    S.bn = pb_bits(N);
    S.bm = pb_bits(M);
    PFP_TRY(pfp_alloc_t(ctx, &S.pos, M));
    PFP_TRY(pfp_alloc_t(ctx, &S.we, M));
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
    PFP_TRY(pfp_alloc_t(ctx, &S.sa_word, M));
    if (split) {
        PFP_TRY(pfp_alloc_t(ctx, &S.hi, M));
        PFP_TRY(pfp_alloc_t(ctx, &S.lo, M));
    }
    const PmRange rg{S.rg_lo, S.rg_hi, S.rg_has_lo, S.rg_has_hi};
    if (M) {
        const u64 chunk = N < PB_CHUNK ? N : PB_CHUNK;
        u8 *cf = nullptr;
        u32 *cs = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &cf, chunk));
        PFP_TRY(pfp_alloc_t(ctx, &cs, chunk));
        u64 e0 = 0;
        for (u64 c0 = 0; c0 < N && e0 < M; c0 += chunk) {
            const u64 n = N - c0 < chunk ? N - c0 : chunk;
            pm_in_k<<<pfp_blocks(n, PB_T), PB_T, 0, ctx->stream>>>(S.in.d, N, S.wd.cd, S.wd.h0, S.wd.bs, rg, c0, n, cf);
            PFP_LAUNCHED(ctx);
            PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, cf, cs, n, reinterpret_cast<u32 *>(&ctx->d_flags[1])));
            pm_collect_k<<<pfp_blocks(n, PB_T), PB_T, 0, ctx->stream>>>(S.in.d, N, S.wd.cd, S.wd.h0, S.wd.bs, cf, cs, c0, n, e0,
                                                                        S.wd.wend, S.in.dwords + 1, S.pos, S.we, S.sl, S.k0,
                                                                        S.v0, S.slot);
            PFP_LAUNCHED(ctx);
            PFP_TRY(pb_sync_read(ctx, 1, 1));
            e0 += (u32)ctx->h_flags[1];
        }
        PFP_TRY(pfp_free_now(ctx, cf));
        PFP_TRY(pfp_free_now(ctx, cs));
        if (e0 != M) return pfp_fail(ctx, PFPB200_E_INTERNAL, "pfbwt: partition counted %llu suffixes, collected %llu",
                                     (unsigned long long)M, (unsigned long long)e0);
    }
    PFP_TRY(pfp_radix_sort_pairs(ctx, S.k0, S.v0, S.k1, S.v1, M, 0, S.wd.h0 * S.wd.bs, &S.ks, &S.vs));
    S.M = M;
    return PFPB200_OK;
}

int pm_update(pfpb200_ctx *ctx, PmState &S, const PmRanks &R, u64 h, int first, u64 *active) {
    const u64 M = S.M;
    int hi_shift = -1;
    if (!first) hi_shift = S.split ? 0 : S.bn + 1;
    if (S.split && !first) PB_LAUNCH(ctx, M, pm_gflags2_k, S.ks, S.vs, S.lo, M, S.flag);
    else PB_LAUNCH(ctx, M, pb_gflags_k, S.ks, M, S.flag);
    PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, S.flag, S.escan, M, nullptr));
    PB_LAUNCH(ctx, M, pb_heads_k, S.flag, S.escan, S.slot, M, S.head);
    PB_LAUNCH(ctx, M, pm_update_k, S.flag, S.escan, S.slot, S.vs, S.ks, hi_shift, S.head, S.pos, S.sl, S.we, M, h, S.base,
              R, S.sa_pos, S.sa_grp, S.sa_word, S.rs, S.keep);
    PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, S.keep, S.escan, M, reinterpret_cast<u32 *>(&ctx->d_flags[1])));
    PFP_TRY(pb_sync_read(ctx, 1, 1));
    S.M2 = M ? (u32)ctx->h_flags[1] : 0;
    *active = S.M2;
    return PFPB200_OK;
}

int pm_gather(pfpb200_ctx *ctx, PmState &S, const PmRanks &R, u64 h) {
    const u64 M = S.M;
    S.ko = S.ks == S.k0 ? S.k1 : S.k0;
    S.vo = S.vs == S.v0 ? S.v1 : S.v0;
    PB_LAUNCH(ctx, M, pm_gather_k, S.keep, S.escan, S.slot, S.vs, S.rs, S.pos, S.sl, R, M, h, S.bn, S.split, S.slot2, S.vo,
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
    PB_LAUNCH(ctx, M, pm_hikey_k, va, S.hi, M, kb);
    return pfp_radix_sort_pairs(ctx, kb, va, ka, vb, M, 0, S.bm, &S.ks, &S.vs);
}

int pm_sort_done(pfpb200_ctx *ctx, PmState &S) {
    PFP_TRY(pfp_free_now(ctx, S.k0)); PFP_TRY(pfp_free_now(ctx, S.k1)); PFP_TRY(pfp_free_now(ctx, S.v0));
    PFP_TRY(pfp_free_now(ctx, S.v1)); PFP_TRY(pfp_free_now(ctx, S.slot)); PFP_TRY(pfp_free_now(ctx, S.slot2));
    PFP_TRY(pfp_free_now(ctx, S.head)); PFP_TRY(pfp_free_now(ctx, S.keep)); PFP_TRY(pfp_free_now(ctx, S.rs));
    PFP_TRY(pfp_free_now(ctx, S.pos)); PFP_TRY(pfp_free_now(ctx, S.sl)); PFP_TRY(pfp_free_now(ctx, S.hi));
    PFP_TRY(pfp_free_now(ctx, S.lo)); PFP_TRY(pfp_free_now(ctx, S.we));
    S.lo = nullptr;
    S.k0 = S.k1 = S.ks = nullptr; S.v0 = S.v1 = S.vs = nullptr;
    S.slot = S.slot2 = S.head = S.rs = S.hi = S.we = nullptr; S.keep = nullptr; S.pos = nullptr; S.sl = nullptr;
    return PFPB200_OK;
}


// the plan of the emission on this rank's slice; the sorted slots are not read after it
int pm_plan(pfpb200_ctx *ctx, PmState &S) {
    PFP_TRY(pb_plan(ctx, S.in, S.wd, PbSplitSlots{S.sa_pos, S.sa_grp, S.sa_word}, S.M0, S.flag, S.escan, &S.plan));
    PFP_TRY(pfp_free_now(ctx, S.sa_pos)); PFP_TRY(pfp_free_now(ctx, S.sa_grp)); PFP_TRY(pfp_free_now(ctx, S.sa_word));
    S.sa_pos = nullptr; S.sa_grp = S.sa_word = nullptr;
    return PFPB200_OK;
}
