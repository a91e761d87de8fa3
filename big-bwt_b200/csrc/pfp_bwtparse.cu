// pfp_bwtparse.cu -- the stage after the parse: suffix array of the parse, its BWT, the inverted
// list and the permuted .last / .sai streams.  SURVEY.md section 8(f) row 3.
//
// Replaces bwtparse.c of the reference (main(), bwtparse.c:218-322): there sacak_int() (gSACA-K,
// gsa/gsacak.c) sorts the suffixes of T[0..n] (the n parse symbols + the end symbol T[n] = 0) on
// one core, then three loops build BWT / .bwlast / .bwsai (:243-272) and the inverted list by a
// counting sort (:294-298).  Here, for a parse resident in HBM:
//   * suffix array by PREFIX DOUBLING on ranks: round r sorts the pairs (rank of the first h
//     symbols, rank of the next h symbols) with the library's own LSD radix sort, h = 2, 4, 8, ...
//     -- the end symbol is unique and the smallest, so no suffix is a prefix of another and a
//     position past the end never has to be compared (its rank is read as 0).  A round is: keys
//     from ranks (one gather), radix passes over exactly 2 ceil(log2 N) key bits, group flags,
//     a scan, the new ranks.  A suffix's rank is the POSITION where its group starts, so ranks stay
//     valid while only some groups are refined: a suffix alone in its group is final and leaves
//     the active list (Larsson-Sadakane discarding) -- the last rounds sort a few per cent of the
//     suffixes.  It stops when the active list is empty.  A repetitive pan-genome parse needs
//     log2(longest repeat in phrases) + 1 rounds (8 for 100 haplotypes at 0.1 % divergence).
//   * BWT[i] = T[SA[i] - 1], bwlast[i] = last[SA[i] - 2], bwsai[i] = sai[SA[i] - 1] with the special
//     cases of bwtparse.c:246-270: gathers;
//   * ilist = positions i sorted stably by BWT[i] (bwtparse.c:294-298 is a counting sort with the
//     F[] array built from .occ): the same radix sort on (BWT[i], i) -- .occ is not needed.
// Outputs are byte-identical to the reference's .ilist / .bwlast / .bwsai (tests/test_bwtparse_gpu.py
// runs the unmodified bwtparse beside it; tests/golden/golden_bwtparse.npz holds its outputs).
#include "pfp_common.cuh"
#include "pfp_stages.cuh"
#include <errno.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

constexpr int BP_T = 256;

// first round: the pair of the first two symbols; T[n] = 0 is the end symbol (bwtparse.c:114)
__global__ void __launch_bounds__(BP_T) bp_init_k(const u32 *__restrict__ parse, u64 n, u64 *__restrict__ key,
                                                  u32 *__restrict__ val) {
    const u64 i = (u64)blockIdx.x * BP_T + threadIdx.x;
    if (i > n) return;
    const u64 t0 = i < n ? parse[i] : 0u, t1 = i + 1 < n ? parse[i + 1] : 0u;
    key[i] = (t0 << 32) | t1;
    val[i] = (u32)i;
}

// flag[k] = 1 where a new group of equal keys starts (sorted order of the active suffixes)
__global__ void __launch_bounds__(BP_T) bp_flags_k(const u64 *__restrict__ key, u64 M, u8 *__restrict__ flag) {
    const u64 k = (u64)blockIdx.x * BP_T + threadIdx.x;
    if (k >= M) return;
    flag[k] = (k == 0 || key[k] != key[k - 1]) ? 1 : 0;
}

__global__ void __launch_bounds__(BP_T) bp_iota_k(u32 *__restrict__ a, u64 n) {
    const u64 i = (u64)blockIdx.x * BP_T + threadIdx.x;
    if (i < n) a[i] = (u32)i;
}

// head[g] = slot (position in the suffix array) where group g of the active list starts
__global__ void __launch_bounds__(BP_T) bp_heads_k(const u8 *__restrict__ flag, const u32 *__restrict__ escan,
                                                   const u32 *__restrict__ slot, u64 M, u32 *__restrict__ head) {
    const u64 k = (u64)blockIdx.x * BP_T + threadIdx.x;
    if (k < M && flag[k]) head[escan[k]] = slot[k];
}

// the sorted active suffixes go back to their slots; a suffix's rank is the slot where its group
// starts (stable under refinement: only the groups that are split change); keep[k] = 0 for a group
// of one -- that suffix is in its final place and leaves the active list
__global__ void __launch_bounds__(BP_T) bp_update_k(const u8 *__restrict__ flag, const u32 *__restrict__ escan,
                                                    const u32 *__restrict__ slot, const u32 *__restrict__ val,
                                                    const u32 *__restrict__ head, u64 M, u32 *__restrict__ sa,
                                                    u32 *__restrict__ rank, u32 *__restrict__ rs,
                                                    u8 *__restrict__ keep) {
    const u64 k = (u64)blockIdx.x * BP_T + threadIdx.x;
    if (k >= M) return;
    const u32 f = flag[k], s = val[k];
    const u32 r = head[escan[k] + f - 1u];
    sa[slot[k]] = s;
    rank[s] = r;
    rs[k] = r;
    keep[k] = (f && (k + 1 == M || flag[k + 1])) ? 0 : 1;
}

// the suffixes that stay active, in order, with the next round's key: (rank, rank h symbols on)
__global__ void __launch_bounds__(BP_T) bp_compact_k(const u8 *__restrict__ keep, const u32 *__restrict__ kscan,
                                                     const u32 *__restrict__ slot, const u32 *__restrict__ val,
                                                     const u32 *__restrict__ rs, const u32 *__restrict__ rank, u64 M,
                                                     u64 N, u64 h, int b, u32 *__restrict__ slot2,
                                                     u32 *__restrict__ val2, u64 *__restrict__ key2) {
    const u64 k = (u64)blockIdx.x * BP_T + threadIdx.x;
    if (k >= M || !keep[k]) return;
    const u32 p = kscan[k], s = val[k];
    const u64 j = (u64)s + h;
    slot2[p] = slot[k];
    val2[p] = s;
    key2[p] = ((u64)rs[k] << b) | (j < N ? (u64)rank[j] + 1u : 0u);
}

// BWT of the parse and the permuted .last / .sai (bwtparse.c:243-272); SA[0] = n by construction
__global__ void __launch_bounds__(BP_T) bp_emit_k(const u32 *__restrict__ sa, const u32 *__restrict__ parse,
                                                  const u8 *__restrict__ last, const u8 *__restrict__ sai, u64 n,
                                                  u64 *__restrict__ bwt_key, u32 *__restrict__ pos,
                                                  u8 *__restrict__ bwlast, u8 *__restrict__ bwsai,
                                                  unsigned long long *__restrict__ flags) {
    const u64 i = (u64)blockIdx.x * BP_T + threadIdx.x;
    if (i > n) return;
    const u64 s = sa[i];
    if ((i == 0) != (s == n) || (s == 0 && i != 1)) atomicOr(flags, PFP_ERRBIT_INTERNAL);   // the asserts of :244,:250
    u32 sym = 0;
    u8 lc = 0;
    if (s != 0) {
        sym = parse[s - 1];
        lc = s == 1 ? last[n - 1] : last[s - 2];
    }
    bwt_key[i] = sym;
    pos[i] = (u32)i;
    bwlast[i] = lc;
    if (bwsai) {
#pragma unroll
        for (int k = 0; k < PFP_IBYTES; k++) bwsai[i * PFP_IBYTES + k] = s ? sai[(s - 1) * PFP_IBYTES + k] : (u8)0;
    }
}

__global__ void __launch_bounds__(BP_T) bp_max_k(const u32 *__restrict__ parse, u64 n, u32 *__restrict__ out) {
    u32 m = 0;
    for (u64 i = (u64)blockIdx.x * BP_T + threadIdx.x; i < n; i += (u64)gridDim.x * BP_T) m = max(m, parse[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

// The outputs of a parse on this context stay valid (they are the natural inputs here); only the
// outputs of the previous bwtparse call are given back.
static int bp_begin(pfpb200_ctx *ctx) {
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    pfp_release_scratch(ctx);
    for (int k = 0; k < 3; k++) {
        void *p = ctx->bp_out[k];
        ctx->bp_out[k] = nullptr;
        if (!p) continue;
        for (size_t i = 0; i < ctx->held.size(); i++)
            if (ctx->held[i] == p) {
                ctx->held[i] = ctx->held.back();
                ctx->held.pop_back();
                ctx->scratch.push_back(p);            // released with the scratch just below
                break;
            }
    }
    pfp_release_scratch(ctx);
    ctx->err[0] = 0;
    PFP_CUDA(ctx, cudaMemsetAsync(ctx->d_flags, 0, 3 * sizeof(u64), ctx->stream));
    return PFPB200_OK;
}

static int bits_for(u64 v) {   // bits needed to write values 0 .. v
    int b = 1;
    while (b < 64 && (v >> b) != 0) b++;
    return b;
}

// d_parse[n], d_last[n], d_sai[5n] (or null) on the device -> held device outputs
static int bwtparse_device_impl(pfpb200_ctx *ctx, const u32 *d_parse, u64 n, const u8 *d_last, const u8 *d_sai,
                                pfpb200_bwtparse_result *res) {
    memset(res, 0, sizeof(*res));
    if (n < 2) return pfp_fail(ctx, PFPB200_E_ARG, "bwtparse: the parse must hold at least two phrases");   // assert(n>1), :241
    if (n >= 0xFFFFFFFEull) return pfp_fail(ctx, PFPB200_E_LIMIT, "Input containing more than 2^32-2 phrases!");   // :101
    const u64 N = n + 1;
    const u32 nb = pfp_blocks(N, BP_T);
    PfpEvents evs(3);
    if (!evs.ok) return pfp_fail(ctx, PFPB200_E_CUDA, "cudaEventCreate failed");
    const u32 launches0 = ctx->launches;
    PFP_CUDA(ctx, cudaEventRecord(evs[0], ctx->stream));
    u64 *k0 = nullptr, *k1 = nullptr;
    u32 *v0 = nullptr, *v1 = nullptr, *rank = nullptr, *rs = nullptr, *escan = nullptr, *sa = nullptr;
    u32 *slot = nullptr, *slot2 = nullptr, *head = nullptr;
    u8 *flag = nullptr, *keep = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &k0, N));
    PFP_TRY(pfp_alloc_t(ctx, &k1, N));
    PFP_TRY(pfp_alloc_t(ctx, &v0, N));
    PFP_TRY(pfp_alloc_t(ctx, &v1, N));
    PFP_TRY(pfp_alloc_t(ctx, &sa, N));
    PFP_TRY(pfp_alloc_t(ctx, &rank, N));
    PFP_TRY(pfp_alloc_t(ctx, &rs, N));
    PFP_TRY(pfp_alloc_t(ctx, &escan, N));
    PFP_TRY(pfp_alloc_t(ctx, &slot, N));
    PFP_TRY(pfp_alloc_t(ctx, &slot2, N));
    PFP_TRY(pfp_alloc_t(ctx, &head, N));
    PFP_TRY(pfp_alloc_t(ctx, &flag, N));
    PFP_TRY(pfp_alloc_t(ctx, &keep, N));
    // largest symbol: key bits of the first round and of the inverted list
    u32 *d_max = reinterpret_cast<u32 *>(&ctx->d_flags[2]);
    PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[1], 0, 2 * sizeof(u64), ctx->stream));
    bp_max_k<<<ctx->sm_count * 4, BP_T, 0, ctx->stream>>>(d_parse, n, d_max);
    PFP_LAUNCHED(ctx);
    PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[2], &ctx->d_flags[2], sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    bp_init_k<<<nb, BP_T, 0, ctx->stream>>>(d_parse, n, k0, v0);
    PFP_LAUNCHED(ctx);
    bp_iota_k<<<nb, BP_T, 0, ctx->stream>>>(slot, N);
    PFP_LAUNCHED(ctx);
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const u32 kmax = (u32)ctx->h_flags[2];
    const int sym_bits = bits_for(kmax);
    const int b = bits_for(N);                            // bits of a rank + 1
    u64 *ks = nullptr;
    u32 *vs = nullptr;
    // round 1: all suffixes by their first two symbols.  The low half sorts over sym_bits, the high half starts at bit 32
    PFP_TRY(pfp_radix_sort_pairs(ctx, k0, v0, k1, v1, N, 0, sym_bits, &ks, &vs));
    {
        u64 *ko = ks == k0 ? k1 : k0;
        u32 *vo = vs == v0 ? v1 : v0;
        PFP_TRY(pfp_radix_sort_pairs(ctx, ks, vs, ko, vo, N, 32, 32 + sym_bits, &ks, &vs));
    }
    u32 rounds = 1;
    u64 M = N;                                            // suffixes still in a group of two or more
    u32 *d_cnt = reinterpret_cast<u32 *>(&ctx->d_flags[1]);
    for (u64 h = 2;; h *= 2, rounds++) {
        // (ks, vs)[0..M): the active suffixes sorted by (rank, rank of the next h / 2 symbols); slot[k] = where the k-th goes
        const u32 mb = pfp_blocks(M, BP_T);
        bp_flags_k<<<mb, BP_T, 0, ctx->stream>>>(ks, M, flag);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, flag, escan, M, nullptr));
        bp_heads_k<<<mb, BP_T, 0, ctx->stream>>>(flag, escan, slot, M, head);
        PFP_LAUNCHED(ctx);
        bp_update_k<<<mb, BP_T, 0, ctx->stream>>>(flag, escan, slot, vs, head, M, sa, rank, rs, keep);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, keep, escan, M, d_cnt));
        PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[1], &ctx->d_flags[1], sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        const u64 M2 = (u32)ctx->h_flags[1];
        if (M2 == 0) break;                               // every suffix has its own rank: sa[] is the suffix array
        if (h >= 2 * N) return pfp_fail(ctx, PFPB200_E_INTERNAL, "bwtparse: prefix doubling did not converge");
        u64 *ko = ks == k0 ? k1 : k0;
        u32 *vo = vs == v0 ? v1 : v0;
        bp_compact_k<<<mb, BP_T, 0, ctx->stream>>>(keep, escan, slot, vs, rs, rank, M, N, h, b, slot2, vo, ko);
        PFP_LAUNCHED(ctx);
        { u32 *t = slot; slot = slot2; slot2 = t; }
        M = M2;
        PFP_TRY(pfp_radix_sort_pairs(ctx, ko, vo, ks, vs, M, 0, 2 * b, &ks, &vs));
    }
    PFP_CUDA(ctx, cudaEventRecord(evs[1], ctx->stream));
    // BWT, .bwlast, .bwsai, then the inverted list = positions sorted stably by BWT symbol
    u32 *ilist = nullptr;
    u8 *bwlast = nullptr, *bwsai = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &bwlast, N, true));
    if (d_sai) PFP_TRY(pfp_alloc_t(ctx, &bwsai, N * PFP_IBYTES, true));
    PFP_TRY(pfp_alloc_t(ctx, &ilist, N, true));
    u64 *bk = k0;                                          // the sort buffers are free: the suffix array has its own
    u32 *bv = v0;
    bp_emit_k<<<nb, BP_T, 0, ctx->stream>>>(sa, d_parse, d_last, d_sai, n, bk, bv, bwlast, bwsai,
                                            reinterpret_cast<unsigned long long *>(&ctx->d_flags[0]));
    PFP_LAUNCHED(ctx);
    u64 *ik = nullptr;
    u32 *iv = nullptr;
    PFP_TRY(pfp_radix_sort_pairs(ctx, bk, bv, k1, v1, N, 0, sym_bits, &ik, &iv));
    PFP_CUDA(ctx, cudaMemcpyAsync(ilist, iv, N * sizeof(u32), cudaMemcpyDeviceToDevice, ctx->stream));
    PFP_CUDA(ctx, cudaEventRecord(evs[2], ctx->stream));
    PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[0], &ctx->d_flags[0], sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->h_flags[0] & PFP_ERRBIT_INTERNAL)
        return pfp_fail(ctx, PFPB200_E_INTERNAL, "bwtparse: the parse does not start with its smallest, unique phrase");
    ctx->bp_out[0] = ilist; ctx->bp_out[1] = bwlast; ctx->bp_out[2] = bwsai;
    res->ilist = ilist;
    res->bwlast = bwlast;
    res->bwsai = bwsai;
    res->n_out = N;
    res->alphabet = (u64)kmax + 1;
    res->rounds = rounds;
    res->launches = ctx->launches - launches0;
    cudaEventElapsedTime(&res->ms_sa, evs[0], evs[1]);
    cudaEventElapsedTime(&res->ms_lists, evs[1], evs[2]);
    res->ms_total = res->ms_sa + res->ms_lists;
    return PFPB200_OK;
}

extern "C" int pfpb200_bwtparse_device(pfpb200_ctx *ctx, const uint32_t *d_parse, uint64_t n_phrases,
                                       const uint8_t *d_last, const uint8_t *d_sai,
                                       pfpb200_bwtparse_result *res) {
    if (!ctx || !d_parse || !d_last || !res) return PFPB200_E_ARG;
    PFP_TRY(bp_begin(ctx));
    const int rc = bwtparse_device_impl(ctx, d_parse, n_phrases, d_last, d_sai, res);
    pfp_release_scratch(ctx);
    return rc;
}

extern "C" int pfpb200_bwtparse_host(pfpb200_ctx *ctx, const uint32_t *parse, uint64_t n, const uint8_t *last,
                                     const uint8_t *sai, uint32_t *ilist, uint8_t *bwlast, uint8_t *bwsai,
                                     pfpb200_bwtparse_result *res) {
    if (!ctx || !parse || !last || !ilist || !bwlast || !res || (sai && !bwsai)) return PFPB200_E_ARG;
    PFP_TRY(bp_begin(ctx));
    u32 *d_parse = nullptr;
    u8 *d_last = nullptr, *d_sai = nullptr;
    int rc = pfp_alloc_t(ctx, &d_parse, n);
    if (rc == PFPB200_OK) rc = pfp_alloc_t(ctx, &d_last, n);
    if (rc == PFPB200_OK && sai) rc = pfp_alloc_t(ctx, &d_sai, n * PFP_IBYTES);
    if (rc != PFPB200_OK) { pfp_release_scratch(ctx); return rc; }
    auto copy = [&](void *d, const void *s, size_t bytes, cudaMemcpyKind k) {
        return bytes == 0 || cudaMemcpyAsync(d, s, bytes, k, ctx->stream) == cudaSuccess;
    };
    bool ok = copy(d_parse, parse, n * sizeof(u32), cudaMemcpyHostToDevice) &&
              copy(d_last, last, n, cudaMemcpyHostToDevice) &&
              (!sai || copy(d_sai, sai, n * PFP_IBYTES, cudaMemcpyHostToDevice));
    if (!ok) { pfp_release_scratch(ctx); return pfp_fail(ctx, PFPB200_E_CUDA, "bwtparse: host to device copy failed"); }
    rc = bwtparse_device_impl(ctx, d_parse, n, d_last, d_sai, res);
    if (rc == PFPB200_OK) {
        ok = copy(ilist, res->ilist, res->n_out * sizeof(u32), cudaMemcpyDeviceToHost) &&
             copy(bwlast, res->bwlast, res->n_out, cudaMemcpyDeviceToHost) &&
             (!sai || copy(bwsai, res->bwsai, res->n_out * PFP_IBYTES, cudaMemcpyDeviceToHost)) &&
             cudaStreamSynchronize(ctx->stream) == cudaSuccess;
        if (!ok) rc = pfp_fail(ctx, PFPB200_E_CUDA, "bwtparse: device to host copy failed");
    }
    pfp_release_scratch(ctx);
    return rc;
}

// ---- files: <base>.parse, <base>[.<i>].last, <base>[.<i>].sai -> <base>.ilist .bwlast .bwsai ----------------
static int open_size(const char *name, u64 *size) {
    const int fd = open(name, O_RDONLY);
    if (fd < 0) return -1;
    struct stat st;
    if (fstat(fd, &st) != 0) { close(fd); return -1; }
    *size = (u64)st.st_size;
    return fd;
}

// the .last / .sai stream of `want` bytes, in one file or in nseg segment files <base>.<i>.<ext>
// (mopen_aux_file / mfread, utils.c:57-110), streamed to d_dst
static int segments_to_device(pfpb200_ctx *ctx, const char *base, const char *ext, int nseg, u64 want, u8 *d_dst) {
    char name[4096];
    u64 got = 0;
    for (int i = 0; i < (nseg > 0 ? nseg : 1); i++) {
        if (nseg > 0) snprintf(name, sizeof(name), "%s.%d.%s", base, i, ext);
        else snprintf(name, sizeof(name), "%s.%s", base, ext);
        u64 sz = 0;
        const int fd = open_size(name, &sz);
        if (fd < 0) return pfp_fail(ctx, PFPB200_E_IO, "cannot open %s: %s", name, strerror(errno));
        if (got + sz > want) sz = want - got;
        const int rc = sz ? pfp_file_to_device(ctx, fd, 0, sz, d_dst + got) : PFPB200_OK;
        close(fd);
        if (rc != PFPB200_OK) return rc;
        got += sz;
    }
    if (got != want) return pfp_fail(ctx, PFPB200_E_IO, "%s: %llu bytes, %llu expected", ext, (unsigned long long)got,
                                     (unsigned long long)want);
    return PFPB200_OK;
}

// ---- the bounded path: a parse whose in-HBM sort does not fit (DESIGN.md §6e) -----------------------------
// Resident: the parse, .last, .sai, sa[N], rank[N] (the slot where a suffix's group starts) and a byte
// per slot marking group starts.  Round 1 sorts the suffixes by their first two symbols in windows of
// first-symbol ranges; every later round sorts the members of the groups of two or more in windows of
// whole groups, in slot order.  A window reads ranks that earlier windows of the same round have already
// refined (Larsson-Sadakane): every group is refined as a whole and every rank stays consistent with the
// suffix order, so the keys still sort each group by a prefix of at least 2h symbols.  The outputs are
// written to the files in windows: .bwlast / .bwsai over slot ranges, .ilist over symbol ranges.
constexpr int BW_I = 16;
constexpr u64 BW_BLK = (u64)BP_T * BW_I;   // positions per block of the counting and collecting kernels

// positions i < len whose value lies in [c0, c1)
struct BwSym {
    const u32 *v;
    u64 len, c0, c1;
    __device__ __forceinline__ bool operator()(u64 i) const { return i < len && v[i] >= c0 && v[i] < c1; }
};
// slots s < hi whose group has two or more members (gstart[N] = 1 ends the last group)
struct BwActive {
    const u8 *gstart;
    u64 hi;
    __device__ __forceinline__ bool operator()(u64 s) const { return s < hi && !(gstart[s] && gstart[s + 1]); }
};

// cnt[b] = matches among positions [lo + b BW_BLK, lo + (b + 1) BW_BLK)
template <class Pred>
__global__ void __launch_bounds__(BP_T) bw_count_k(Pred p, u64 lo, u32 *__restrict__ cnt) {
    const u64 base = lo + (u64)blockIdx.x * BW_BLK + threadIdx.x;
    u32 c = 0;
    for (int r = 0; r < BW_I; r++) c += (u32)__syncthreads_count(p(base + (u64)r * BP_T));
    if (threadIdx.x == 0) cnt[blockIdx.x] = c;
}

// the matches of a block in position order, from out index boff[block] on: calls f(position, index)
template <class Pred, class F>
__device__ __forceinline__ void bw_collect(Pred p, u64 lo, const u32 *__restrict__ boff, F f) {
    __shared__ u32 sm[9];
    const u64 base = lo + (u64)blockIdx.x * BW_BLK + threadIdx.x;
    u32 o = boff[blockIdx.x];
    for (int r = 0; r < BW_I; r++) {
        const u64 i = base + (u64)r * BP_T;
        const bool m = p(i);
        u32 tot;
        const u32 ex = block_excl_scan_256(m ? 1u : 0u, &tot, sm);
        if (m) f(i, o + ex);
        o += tot;
    }
}

// round 1 and the inverted list: key = (v[i] - c0) << 32 | v[i + 1] (0 past the end), val = i.  Round 1
// sorts both halves (its first two symbols), the inverted list only the high one.
__global__ void __launch_bounds__(BP_T) bw_select_k(BwSym p, const u32 *__restrict__ boff, u64 *__restrict__ key,
                                                    u32 *__restrict__ val) {
    bw_collect(p, 0, boff, [&](u64 i, u32 k) {
        key[k] = ((u64)(p.v[i] - p.c0) << 32) | (i + 1 < p.len ? p.v[i + 1] : 0u);
        val[k] = (u32)i;
    });
}

// a later round: the active slots of the window [lo, p.hi) in slot order, with the key (rank - lo, rank
// h symbols on + 1) of the suffix in them
__global__ void __launch_bounds__(BP_T) bw_active_k(BwActive p, u64 lo, const u32 *__restrict__ boff,
                                                    const u32 *__restrict__ sa, const u32 *__restrict__ rank, u64 N,
                                                    u64 h, int b, u32 *__restrict__ slot, u64 *__restrict__ key,
                                                    u32 *__restrict__ val) {
    bw_collect(p, lo, boff, [&](u64 s, u32 k) {
        const u32 v = sa[s];
        const u64 j = (u64)v + h;
        slot[k] = (u32)s;
        val[k] = v;
        key[k] = ((u64)(rank[v] - lo) << b) | (j < N ? (u64)rank[j] + 1u : 0u);
    });
}

__global__ void __launch_bounds__(BP_T) bw_iota_k(u32 *__restrict__ a, u64 m, u64 base) {
    const u64 k = (u64)blockIdx.x * BP_T + threadIdx.x;
    if (k < m) a[k] = (u32)(base + k);
}

// slot 0 holds the end suffix n, alone in its group; gstart[N] closes the last group
__global__ void bw_init_k(u32 *__restrict__ sa, u32 *__restrict__ rank, u8 *__restrict__ gstart, u64 n) {
    sa[0] = (u32)n;
    rank[n] = 0;
    gstart[0] = 1;
    gstart[n + 1] = 1;
}

// the sorted window back into place: suffix, its group's first slot, and the group starts
__global__ void __launch_bounds__(BP_T) bw_update_k(const u8 *__restrict__ flag, const u32 *__restrict__ escan,
                                                    const u32 *__restrict__ slot, const u32 *__restrict__ val,
                                                    const u32 *__restrict__ head, u64 m, u32 *__restrict__ sa,
                                                    u32 *__restrict__ rank, u8 *__restrict__ gstart) {
    const u64 k = (u64)blockIdx.x * BP_T + threadIdx.x;
    if (k >= m) return;
    const u32 f = flag[k], s = val[k], sl = slot[k];
    sa[sl] = s;
    rank[s] = head[escan[k] + f - 1u];
    gstart[sl] = (u8)f;
}

// occurrences of the symbols c0 <= c < c1 of the parse, into cnt[c - c0]
__global__ void __launch_bounds__(BP_T) bw_hist_k(const u32 *__restrict__ parse, u64 n, u64 c0, u64 c1,
                                                  u32 *__restrict__ cnt) {
    for (u64 i0 = (u64)blockIdx.x * BP_T; i0 < n; i0 += (u64)gridDim.x * BP_T) {
        const u64 i = i0 + threadIdx.x;
        const u64 v = i < n ? parse[i] : c1;
        const bool ok = v >= c0 && v < c1;
        const u32 peers = __match_any_sync(0xffffffffu, ok ? v : c1);
        if (ok && (peers & lanemask_lt()) == 0) atomicAdd(&cnt[v - c0], (u32)__popc(peers));
    }
}

// The end of a window that starts at group start a: the last group start s in [lo, hi] (s > a) with
// base + (active slots in [lo, s)) <= cap, 0 if there is none.  One CTA over hi - lo <= BW_BLK slots.
__global__ void __launch_bounds__(BP_T) bw_cut_k(const u8 *__restrict__ gstart, u64 a, u64 lo, u64 hi, u64 base,
                                                 u64 cap, unsigned long long *__restrict__ out) {
    __shared__ u32 sm[9];
    __shared__ unsigned long long best;
    if (threadIdx.x == 0) best = 0;
    u64 run = base;
    for (u64 s0 = lo; s0 <= hi; s0 += BP_T) {
        const u64 s = s0 + threadIdx.x;
        const bool in = s <= hi;
        const bool act = s < hi && !(gstart[s] && gstart[s + 1]);
        u32 tot;
        const u32 ex = block_excl_scan_256(act ? 1u : 0u, &tot, sm);
        if (in && s > a && gstart[s] && run + ex <= cap) atomicMax(&best, (unsigned long long)s);
        run += tot;
    }
    __syncthreads();
    if (threadIdx.x == 0) *out = best;
}

// the last (first = 0) or first (first = 1) group start in [lo, hi); out preset by the caller
__global__ void __launch_bounds__(BP_T) bw_find_k(const u8 *__restrict__ gstart, u64 lo, u64 hi, int first,
                                                  unsigned long long *__restrict__ out) {
    for (u64 s = lo + (u64)blockIdx.x * BP_T + threadIdx.x; s < hi; s += (u64)gridDim.x * BP_T)
        if (gstart[s]) {
            if (first) atomicMin(out, (unsigned long long)s);
            else atomicMax(out, (unsigned long long)s);
        }
}

// slots [a, a + m): BWT of the parse (as u32, into bwt[a + k]), .bwlast and .bwsai of the window
// (bwtparse.c:243-272, the checks of bp_emit_k)
__global__ void __launch_bounds__(BP_T) bw_emit_k(const u32 *__restrict__ sa, const u32 *__restrict__ parse,
                                                  const u8 *__restrict__ last, const u8 *__restrict__ sai, u64 n,
                                                  u64 a, u64 m, u32 *__restrict__ bwt, u8 *__restrict__ bwlast,
                                                  u8 *__restrict__ bwsai, unsigned long long *__restrict__ flags) {
    const u64 k = (u64)blockIdx.x * BP_T + threadIdx.x;
    if (k >= m) return;
    const u64 i = a + k, s = sa[i];
    if ((i == 0) != (s == n) || (s == 0 && i != 1)) atomicOr(flags, PFP_ERRBIT_INTERNAL);
    u32 sym = 0;
    u8 lc = 0;
    if (s != 0) {
        sym = parse[s - 1];
        lc = s == 1 ? last[n - 1] : last[s - 2];
    }
    bwt[i] = sym;
    bwlast[k] = lc;
    if (bwsai) {
#pragma unroll
        for (int j = 0; j < PFP_IBYTES; j++) bwsai[k * PFP_IBYTES + j] = s ? sai[(s - 1) * PFP_IBYTES + j] : (u8)0;
    }
}

static u64 ceil_div(u64 a, u64 b) { return (a + b - 1) / b; }
constexpr u64 BP_ALLOC_SLACK = 512;        // pfp_alloc rounds every request up to 512 bytes

// device bytes of bwtparse_device_impl with its inputs in HBM, from its allocations: .parse .last [.sai],
// k0 k1 v0 v1 sa rank rs escan slot slot2 head flag keep, the radix sort's histograms and the scans'
// partial sums, and the outputs, allocated while the sort's buffers are still live
static u64 bp_inhbm_bytes(u64 n, bool sai) {
    const u64 N = n + 1;
    return n * (4 + 1 + (sai ? PFP_IBYTES : 0)) + N * 54 + 1024 * ceil_div(N, 4096) + 8 * ceil_div(N, 2048) +
           N * (1 + (sai ? PFP_IBYTES : 0) + 4) + 24 * BP_ALLOC_SLACK;
}
// the bounded path outside its windows: the inputs, sa rank gstart, two arrays of block counts
static u64 bw_resident_bytes(u64 n, bool sai) {
    const u64 N = n + 1;
    return n * (4 + 1 + (sai ? PFP_IBYTES : 0)) + N * 9 + 1 + 8 * ceil_div(N, BW_BLK) + 8 * BP_ALLOC_SLACK;
}
// one sort window of m suffixes: k0 k1 v0 v1 slot escan head flag, histograms and partial sums
static u64 bw_window_bytes(u64 m) {
    return m * 37 + 1024 * ceil_div(m, 4096) + 8 * ceil_div(m, 2048) + 11 * BP_ALLOC_SLACK;
}

// PFPB200_BWTPARSE_BUDGET=<bytes>, else the free device memory plus what the arena holds unused
static int bw_budget(pfpb200_ctx *ctx, u64 *budget) {
    const char *ev = getenv("PFPB200_BWTPARSE_BUDGET");
    if (ev && atoll(ev) > 0) {
        *budget = (u64)atoll(ev);
        return PFPB200_OK;
    }
    size_t fr = 0, tot = 0;
    PFP_CUDA(ctx, cudaMemGetInfo(&fr, &tot));
    *budget = (u64)fr + (u64)(ctx->arena.total - ctx->arena.in_use);
    return PFPB200_OK;
}

// flags, heads and the update of a sorted window (ks, vs)[0, m) whose k-th suffix goes to slot[k]
static int bw_refine(pfpb200_ctx *ctx, const u64 *ks, const u32 *vs, const u32 *slot, u64 m, u8 *flag, u32 *escan,
                     u32 *head, u32 *sa, u32 *rank, u8 *gstart) {
    const u32 mb = pfp_blocks(m, BP_T);
    bp_flags_k<<<mb, BP_T, 0, ctx->stream>>>(ks, m, flag);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, flag, escan, m, nullptr));
    bp_heads_k<<<mb, BP_T, 0, ctx->stream>>>(flag, escan, slot, m, head);
    PFP_LAUNCHED(ctx);
    bw_update_k<<<mb, BP_T, 0, ctx->stream>>>(flag, escan, slot, vs, head, m, sa, rank, gstart);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

// the buffers of one sort window of m suffixes
struct BwWin {
    u64 *k0 = nullptr, *k1 = nullptr;
    u32 *v0 = nullptr, *v1 = nullptr, *slot = nullptr, *escan = nullptr, *head = nullptr;
    u8 *flag = nullptr;
};
static int bw_win_alloc(pfpb200_ctx *ctx, u64 m, BwWin *w) {
    PFP_TRY(pfp_alloc_t(ctx, &w->k0, m)); PFP_TRY(pfp_alloc_t(ctx, &w->k1, m));
    PFP_TRY(pfp_alloc_t(ctx, &w->v0, m)); PFP_TRY(pfp_alloc_t(ctx, &w->v1, m));
    PFP_TRY(pfp_alloc_t(ctx, &w->slot, m)); PFP_TRY(pfp_alloc_t(ctx, &w->escan, m));
    PFP_TRY(pfp_alloc_t(ctx, &w->head, m)); PFP_TRY(pfp_alloc_t(ctx, &w->flag, m));
    return PFPB200_OK;
}
static int bw_win_free(pfpb200_ctx *ctx, BwWin *w) {
    void *p[8] = {w->k0, w->k1, w->v0, w->v1, w->slot, w->escan, w->head, w->flag};
    for (void *q : p) PFP_TRY(pfp_free_now(ctx, q));
    *w = BwWin();
    return PFPB200_OK;
}

// windows [c0, c1) of whole symbols whose counts cnt[c] (+ 1 for symbol 0 when extra0) sum to at most cap;
// a symbol with more gets a window of its own.  Empty windows are left out.
static std::vector<std::pair<u64, u64>> bw_sym_windows(const std::vector<u32> &cnt, bool extra0, u64 cap) {
    std::vector<std::pair<u64, u64>> w;
    const u64 A = cnt.size();
    for (u64 c0 = 0; c0 < A;) {
        u64 m = cnt[c0] + (extra0 && c0 == 0), c1 = c0 + 1;
        while (c1 < A && m + cnt[c1] <= cap) m += cnt[c1++];
        if (m) w.push_back({c0, c1});
        c0 = c1;
    }
    return w;
}

// stable compaction of the positions i < len with v[i] in [c0, c1) into (key, val) (bw_select_k)
static int bw_select(pfpb200_ctx *ctx, const u32 *v, u64 len, u64 c0, u64 c1, u32 *bcnt, u64 *key, u32 *val) {
    const BwSym p{v, len, c0, c1};
    const u32 nb = pfp_blocks(len, (u32)BW_BLK);
    bw_count_k<<<nb, BP_T, 0, ctx->stream>>>(p, 0, bcnt);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pfp_exclusive_scan_u32(ctx, bcnt, bcnt, nb, nullptr));
    bw_select_k<<<nb, BP_T, 0, ctx->stream>>>(p, bcnt, key, val);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

static int bw_open(pfpb200_ctx *ctx, const char *base, const char *ext, int *fd, char *name, size_t cap) {
    snprintf(name, cap, "%s.%s", base, ext);
    *fd = open(name, O_WRONLY | O_CREAT | O_TRUNC, 0666);
    if (*fd < 0) return pfp_fail(ctx, PFPB200_E_IO, "%s: %s", name, strerror(errno));
    return PFPB200_OK;
}

struct BwFiles {
    int fd[3] = {-1, -1, -1};
    char name[3][4096];
    ~BwFiles() {
        for (int i = 0; i < 3; i++)
            if (fd[i] >= 0) close(fd[i]);
    }
};

// <base>.parse (fd, n phrases), .last [.sai] -> <base>.ilist .bwlast [.bwsai] within `budget` device bytes;
// *windows = the windows of round 1
static int bwtparse_bounded(pfpb200_ctx *ctx, int fd_parse, const char *base, u64 n, int sa_info, int nseg, u64 budget,
                            pfpb200_bwtparse_result *res, u64 *windows) {
    memset(res, 0, sizeof(*res));
    if (n < 2) return pfp_fail(ctx, PFPB200_E_ARG, "bwtparse: the parse must hold at least two phrases");
    if (n >= 0xFFFFFFFEull) return pfp_fail(ctx, PFPB200_E_LIMIT, "Input containing more than 2^32-2 phrases!");
    const u64 N = n + 1;
    const u64 resident = bw_resident_bytes(n, sa_info != 0);
    if (resident + bw_window_bytes(1) > budget)
        return pfp_fail(ctx, PFPB200_E_NOMEM,
                        "bwtparse: %llu phrases need at least %llu bytes of device memory (%llu resident + %llu for the "
                        "smallest window), %llu available",
                        (unsigned long long)n, (unsigned long long)(resident + bw_window_bytes(1)),
                        (unsigned long long)resident, (unsigned long long)bw_window_bytes(1), (unsigned long long)budget);
    const u64 room = budget - resident;
    u64 cap = 1, hi = N;                                   // the most suffixes of a sort window that fits
    while (cap < hi) {
        const u64 mid = cap + (hi - cap + 1) / 2;
        if (bw_window_bytes(mid) <= room) cap = mid; else hi = mid - 1;
    }
    const u64 emit_unit = 1 + (sa_info ? PFP_IBYTES : 0);
    u64 cap_e = (room > 2 * BP_ALLOC_SLACK ? room - 2 * BP_ALLOC_SLACK : 0) / emit_unit;
    if (cap_e < cap) cap_e = cap;
    PfpEvents evs(3);
    if (!evs.ok) return pfp_fail(ctx, PFPB200_E_CUDA, "cudaEventCreate failed");
    const u32 launches0 = ctx->launches;
    // ---- the resident arrays
    u32 *parse = nullptr, *sa = nullptr, *rank = nullptr, *bcnt = nullptr, *wcnt = nullptr;
    u8 *last = nullptr, *sai = nullptr, *gstart = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &parse, n));
    PFP_TRY(pfp_file_to_device(ctx, fd_parse, 0, n * 4, reinterpret_cast<u8 *>(parse)));
    PFP_TRY(pfp_alloc_t(ctx, &last, n));
    PFP_TRY(segments_to_device(ctx, base, "last", nseg, n, last));
    if (sa_info) {
        PFP_TRY(pfp_alloc_t(ctx, &sai, n * PFP_IBYTES));
        PFP_TRY(segments_to_device(ctx, base, "sai", nseg, n * PFP_IBYTES, sai));
    }
    const u64 nblk = ceil_div(N, BW_BLK);
    PFP_TRY(pfp_alloc_t(ctx, &sa, N));
    PFP_TRY(pfp_alloc_t(ctx, &rank, N));
    PFP_TRY(pfp_alloc_t(ctx, &gstart, N + 1));
    PFP_TRY(pfp_alloc_t(ctx, &bcnt, nblk));
    PFP_TRY(pfp_alloc_t(ctx, &wcnt, nblk));
    PFP_CUDA(ctx, cudaEventRecord(evs[0], ctx->stream));
    // ---- symbol counts: the slot bases of round 1 and the offsets of the inverted list
    u32 *d_max = reinterpret_cast<u32 *>(&ctx->d_flags[2]);
    PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[1], 0, 4 * sizeof(u64), ctx->stream));
    bp_max_k<<<ctx->sm_count * 4, BP_T, 0, ctx->stream>>>(parse, n, d_max);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pb_sync_read(ctx, 2, 1));
    const u64 kmax = (u32)ctx->h_flags[2];
    std::vector<u32> cnt(kmax + 1);
    {                                                      // in alphabet ranges whose counts fit the window room
        const u64 A = kmax + 1, per = (room - BP_ALLOC_SLACK) / 4 < A ? (room - BP_ALLOC_SLACK) / 4 : A;
        u32 *d_cnt = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &d_cnt, per));
        for (u64 c0 = 0; c0 < A; c0 += per) {
            const u64 c1 = c0 + per < A ? c0 + per : A;
            PFP_CUDA(ctx, cudaMemsetAsync(d_cnt, 0, (c1 - c0) * sizeof(u32), ctx->stream));
            bw_hist_k<<<ctx->sm_count * 4, BP_T, 0, ctx->stream>>>(parse, n, c0, c1, d_cnt);
            PFP_LAUNCHED(ctx);
            PFP_CUDA(ctx, cudaMemcpyAsync(&cnt[c0], d_cnt, (c1 - c0) * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
            PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        }
        PFP_TRY(pfp_free_now(ctx, d_cnt));
    }
    std::vector<u64> C(kmax + 2);                          // C[c] = 1 + occurrences of the symbols below c
    C[0] = 1;
    for (u64 c = 0; c <= kmax; c++) C[c + 1] = C[c] + cnt[c];
    const int sym_bits = bits_for(kmax);
    const int b = bits_for(N);
    // ---- round 1: the suffixes by their first two symbols, in windows of first-symbol ranges
    PFP_CUDA(ctx, cudaMemsetAsync(gstart, 0, N + 1, ctx->stream));
    bw_init_k<<<1, 1, 0, ctx->stream>>>(sa, rank, gstart, n);
    PFP_LAUNCHED(ctx);
    const auto w1 = bw_sym_windows(cnt, false, cap);
    *windows = w1.size();
    for (const auto &cw : w1) {
        const u64 c0 = cw.first, c1 = cw.second, m = C[c1] - C[c0];
        BwWin W;
        PFP_TRY(bw_win_alloc(ctx, m, &W));
        PFP_TRY(bw_select(ctx, parse, n, c0, c1, bcnt, W.k0, W.v0));
        u64 *ks = nullptr;
        u32 *vs = nullptr;
        PFP_TRY(pfp_radix_sort_pairs(ctx, W.k0, W.v0, W.k1, W.v1, m, 0, sym_bits, &ks, &vs));
        {
            u64 *ko = ks == W.k0 ? W.k1 : W.k0;
            u32 *vo = vs == W.v0 ? W.v1 : W.v0;
            PFP_TRY(pfp_radix_sort_pairs(ctx, ks, vs, ko, vo, m, 32, 32 + bits_for(c1 - 1 - c0), &ks, &vs));
        }
        bw_iota_k<<<pfp_blocks(m, BP_T), BP_T, 0, ctx->stream>>>(W.slot, m, C[c0]);
        PFP_LAUNCHED(ctx);
        PFP_TRY(bw_refine(ctx, ks, vs, W.slot, m, W.flag, W.escan, W.head, sa, rank, gstart));
        PFP_TRY(bw_win_free(ctx, &W));
    }
    // ---- rounds h = 2, 4, ...: the active slots in windows of whole groups
    u32 rounds = 1;
    std::vector<u32> hc(nblk);
    unsigned long long *d_pos = reinterpret_cast<unsigned long long *>(&ctx->d_flags[3]);
    auto find = [&](u64 lo, u64 hi, int first, u64 *s) -> int {   // bw_find_k; *s = 0 / N + 1: none
        ctx->h_flags[3] = first ? N + 1 : 0;
        PFP_CUDA(ctx, cudaMemcpyAsync(d_pos, &ctx->h_flags[3], sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
        u32 g = pfp_blocks(hi - lo, BP_T);
        if (g > (u32)ctx->sm_count * 8) g = (u32)ctx->sm_count * 8;
        bw_find_k<<<g, BP_T, 0, ctx->stream>>>(gstart, lo, hi, first, d_pos);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pb_sync_read(ctx, 3, 1));
        *s = ctx->h_flags[3];
        return PFPB200_OK;
    };
    for (u64 h = 2;; h *= 2) {
        bw_count_k<<<(u32)nblk, BP_T, 0, ctx->stream>>>(BwActive{gstart, N}, 0, bcnt);
        PFP_LAUNCHED(ctx);
        PFP_CUDA(ctx, cudaMemcpyAsync(hc.data(), bcnt, nblk * sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        u64 active = 0;
        for (u32 c : hc) active += c;
        if (active == 0) break;                            // every suffix has its own group: sa[] is the suffix array
        if (h >= 2 * N) return pfp_fail(ctx, PFPB200_E_INTERNAL, "bwtparse: prefix doubling did not converge");
        rounds++;
        for (u64 a = 0; a < N;) {
            // whole blocks while their counts fit (the first one counted in full), then the cut: the last
            // group start that keeps the window within cap, else the end of the group at a
            u64 j = a / BW_BLK, acc = 0;
            while (j < nblk && acc + hc[j] <= cap) acc += hc[j++];
            u64 e = N;
            if (j < nblk) {
                const u64 lo = j * BW_BLK > a ? j * BW_BLK : a, hi = (j + 1) * BW_BLK < N ? (j + 1) * BW_BLK : N;
                bw_cut_k<<<1, BP_T, 0, ctx->stream>>>(gstart, a, lo, hi, acc, cap, d_pos);
                PFP_LAUNCHED(ctx);
                PFP_TRY(pb_sync_read(ctx, 3, 1));
                e = ctx->h_flags[3];
                if (e == 0 && lo > a) PFP_TRY(find(a + 1, lo + 1, 0, &e));
                // none: the group at a alone holds more than cap; it ends at the first group start behind lo
                // (gstart[N] = 1), searched in ranges that double
                for (u64 from = lo + 1, len = BW_BLK; e == 0; from += len, len *= 2) {
                    const u64 to = from + len < N + 1 ? from + len : N + 1;
                    PFP_TRY(find(from, to, 1, &e));
                    if (e > N) e = 0;
                    if (e == 0 && to == N + 1)
                        return pfp_fail(ctx, PFPB200_E_INTERNAL, "bwtparse: no group start behind slot %llu", (unsigned long long)a);
                }
            }
            // the window [a, e): its active slots, their keys, the sort and the update
            const u32 nb = pfp_blocks(e - a, (u32)BW_BLK);
            const BwActive p{gstart, e};
            u32 *d_m = reinterpret_cast<u32 *>(&ctx->d_flags[1]);
            bw_count_k<<<nb, BP_T, 0, ctx->stream>>>(p, a, wcnt);
            PFP_LAUNCHED(ctx);
            PFP_TRY(pfp_exclusive_scan_u32(ctx, wcnt, wcnt, nb, d_m));
            PFP_TRY(pb_sync_read(ctx, 1, 1));
            const u64 m = (u32)ctx->h_flags[1];
            if (m) {
                BwWin W;
                PFP_TRY(bw_win_alloc(ctx, m, &W));
                bw_active_k<<<nb, BP_T, 0, ctx->stream>>>(p, a, wcnt, sa, rank, N, h, b, W.slot, W.k0, W.v0);
                PFP_LAUNCHED(ctx);
                u64 *ks = nullptr;
                u32 *vs = nullptr;
                PFP_TRY(pfp_radix_sort_pairs(ctx, W.k0, W.v0, W.k1, W.v1, m, 0, b + bits_for(e - 1 - a), &ks, &vs));
                PFP_TRY(bw_refine(ctx, ks, vs, W.slot, m, W.flag, W.escan, W.head, sa, rank, gstart));
                PFP_TRY(bw_win_free(ctx, &W));
            }
            a = e;
        }
    }
    PFP_CUDA(ctx, cudaEventRecord(evs[1], ctx->stream));
    // ---- .bwlast / .bwsai in slot windows; the parse's BWT (u32) goes into rank's memory
    BwFiles F;
    PFP_TRY(bw_open(ctx, base, "bwlast", &F.fd[0], F.name[0], sizeof(F.name[0])));
    if (sa_info) PFP_TRY(bw_open(ctx, base, "bwsai", &F.fd[1], F.name[1], sizeof(F.name[1])));
    PFP_TRY(bw_open(ctx, base, "ilist", &F.fd[2], F.name[2], sizeof(F.name[2])));
    u32 *bwt = rank;
    {
        const u64 m0 = cap_e < N ? cap_e : N;
        u8 *bl = nullptr, *bs = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &bl, m0));
        if (sa_info) PFP_TRY(pfp_alloc_t(ctx, &bs, m0 * PFP_IBYTES));
        for (u64 a = 0; a < N; a += m0) {
            const u64 m = N - a < m0 ? N - a : m0;
            bw_emit_k<<<pfp_blocks(m, BP_T), BP_T, 0, ctx->stream>>>(sa, parse, last, sai, n, a, m, bwt, bl, bs,
                                                                     reinterpret_cast<unsigned long long *>(&ctx->d_flags[0]));
            PFP_LAUNCHED(ctx);
            PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            PFP_TRY(pfp_device_to_fd(ctx, F.fd[0], a, bl, m, F.name[0]));
            if (sa_info) PFP_TRY(pfp_device_to_fd(ctx, F.fd[1], a * PFP_IBYTES, bs, m * PFP_IBYTES, F.name[1]));
        }
        PFP_TRY(pfp_free_now(ctx, bl));
        PFP_TRY(pfp_free_now(ctx, bs));
    }
    PFP_TRY(pb_sync_read(ctx, 0, 1));
    if (ctx->h_flags[0] & PFP_ERRBIT_INTERNAL)
        return pfp_fail(ctx, PFPB200_E_INTERNAL, "bwtparse: the parse does not start with its smallest, unique phrase");
    // ---- .ilist: the positions of every symbol range, in order, at offset F[c0] (F[0] = 0, F[c] = C[c] above)
    for (const auto &cw : bw_sym_windows(cnt, true, cap)) {
        const u64 c0 = cw.first, c1 = cw.second;
        const u64 f0 = c0 ? C[c0] : 0, m = C[c1] - f0;
        BwWin W;
        PFP_TRY(bw_win_alloc(ctx, m, &W));
        PFP_TRY(bw_select(ctx, bwt, N, c0, c1, bcnt, W.k0, W.v0));
        u64 *ks = W.k0;
        u32 *vs = W.v0;
        if (c1 - c0 > 1) PFP_TRY(pfp_radix_sort_pairs(ctx, W.k0, W.v0, W.k1, W.v1, m, 32, 32 + bits_for(c1 - 1 - c0), &ks, &vs));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        PFP_TRY(pfp_device_to_fd(ctx, F.fd[2], f0 * 4, vs, m * 4, F.name[2]));
        PFP_TRY(bw_win_free(ctx, &W));
    }
    PFP_CUDA(ctx, cudaEventRecord(evs[2], ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 3; i++) {
        if (F.fd[i] < 0) continue;
        const int r = close(F.fd[i]);
        F.fd[i] = -1;
        if (r != 0) return pfp_fail(ctx, PFPB200_E_IO, "%s: write error: %s", F.name[i], strerror(errno));
    }
    res->n_out = N;
    res->alphabet = kmax + 1;
    res->rounds = rounds;
    res->launches = ctx->launches - launches0;
    cudaEventElapsedTime(&res->ms_sa, evs[0], evs[1]);
    cudaEventElapsedTime(&res->ms_lists, evs[1], evs[2]);
    res->ms_total = res->ms_sa + res->ms_lists;
    return PFPB200_OK;
}

extern "C" int pfpb200_bwtparse_file(pfpb200_ctx *ctx, const char *basename, int sa_info, int nseg,
                                     pfpb200_bwtparse_result *res) {
    if (!ctx || !basename || !res) return PFPB200_E_ARG;
    PFP_TRY(bp_begin(ctx));
    ctx->bp_windows = ctx->bp_peak = 0;
    ctx->arena.peak = ctx->arena.in_use;                  // pfpb200_bwtparse_plan reports this call's peak
    char name[4096];
    snprintf(name, sizeof(name), "%s.parse", basename);
    u64 bytes = 0;
    const int fd = open_size(name, &bytes);
    if (fd < 0) return pfp_fail(ctx, PFPB200_E_IO, "cannot open %s: %s", name, strerror(errno));
    if (bytes % 4 != 0) {
        close(fd);
        return pfp_fail(ctx, PFPB200_E_ARG, "Invalid input file: size not multiple of 4");      // bwtparse.c:81
    }
    const u64 n = bytes / 4;
    // the in-HBM path when its allocations fit the device memory available to the call, else the bounded one
    u64 budget = 0;
    int rc = bw_budget(ctx, &budget);
    if (rc == PFPB200_OK && bp_inhbm_bytes(n, sa_info != 0) > budget) {
        u64 windows = 0;
        rc = bwtparse_bounded(ctx, fd, basename, n, sa_info, nseg, budget, res, &windows);
        close(fd);
        if (rc == PFPB200_OK) ctx->bp_windows = windows;
        ctx->bp_peak = ctx->arena.peak;
        pfp_release_scratch(ctx);
        return rc;
    }
    if (rc != PFPB200_OK) { close(fd); return rc; }
    u32 *d_parse = nullptr;
    u8 *d_last = nullptr, *d_sai = nullptr;
    rc = pfp_alloc_t(ctx, &d_parse, n);
    if (rc == PFPB200_OK && n) rc = pfp_file_to_device(ctx, fd, 0, bytes, reinterpret_cast<u8 *>(d_parse));
    close(fd);
    if (rc == PFPB200_OK) rc = pfp_alloc_t(ctx, &d_last, n);
    if (rc == PFPB200_OK) rc = segments_to_device(ctx, basename, "last", nseg, n, d_last);
    if (rc == PFPB200_OK && sa_info) rc = pfp_alloc_t(ctx, &d_sai, n * PFP_IBYTES);
    if (rc == PFPB200_OK && sa_info) rc = segments_to_device(ctx, basename, "sai", nseg, n * PFP_IBYTES, d_sai);
    if (rc == PFPB200_OK) rc = bwtparse_device_impl(ctx, d_parse, n, d_last, d_sai, res);
    if (rc == PFPB200_OK) {
        snprintf(name, sizeof(name), "%s.bwlast", basename);
        rc = pfp_device_to_file(ctx, name, res->bwlast, res->n_out);
    }
    if (rc == PFPB200_OK && sa_info) {
        snprintf(name, sizeof(name), "%s.bwsai", basename);
        rc = pfp_device_to_file(ctx, name, res->bwsai, res->n_out * PFP_IBYTES);
    }
    if (rc == PFPB200_OK) {
        snprintf(name, sizeof(name), "%s.ilist", basename);
        rc = pfp_device_to_file(ctx, name, res->ilist, res->n_out * sizeof(u32));
    }
    if (rc == PFPB200_OK) ctx->bp_windows = 1;
    ctx->bp_peak = ctx->arena.peak;
    pfp_release_scratch(ctx);
    return rc;
}

extern "C" int pfpb200_bwtparse_plan(const pfpb200_ctx *ctx, uint64_t *windows, uint64_t *peak_device_bytes) {
    if (!ctx) return PFPB200_E_ARG;
    if (windows) *windows = ctx->bp_windows;
    if (peak_device_bytes) *peak_device_bytes = ctx->bp_peak;
    return PFPB200_OK;
}
