// pfp_prims.cu -- device-wide primitives written for this pipeline: exclusive scan and a
// stable LSD radix sort of (u64 key, u32 value) pairs.  HBM-bound integer work: coalesced
// striped loads, warp-level multisplit (match.any) for ranking, shared-memory staging so the
// scatter leaves the SM as contiguous per-bucket runs.
#include "pfp_common.cuh"
#include <stdarg.h>

// ------------------------------------------------------------------------------------------
// context helpers
// ------------------------------------------------------------------------------------------
int pfp_fail(pfpb200_ctx *ctx, int code, const char *fmt, ...) {
    if (ctx) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(ctx->err, sizeof(ctx->err), fmt, ap);
        va_end(ap);
    }
    return code;
}

// ---- arena ---------------------------------------------------------------------------------------
static void arena_insert_free(PfpArena &A, PfpBlock b) {
    size_t i = 0;
    while (i < A.free_list.size() && A.free_list[i].p < b.p) i++;
    A.free_list.insert(A.free_list.begin() + i, b);
    // coalesce with the right then the left neighbour (never across slabs: slabs are not adjacent
    // in general, and if they are, merging is still a valid contiguous device range only within
    // one allocation -- so check slab membership)
    auto same_slab = [&](char *x, char *y) {
        for (auto &s : A.slabs)
            if (x >= s.p && x < s.p + s.n) return y >= s.p && y < s.p + s.n;
        return false;
    };
    if (i + 1 < A.free_list.size() && A.free_list[i].p + A.free_list[i].n == A.free_list[i + 1].p &&
        same_slab(A.free_list[i].p, A.free_list[i + 1].p)) {
        A.free_list[i].n += A.free_list[i + 1].n;
        A.free_list.erase(A.free_list.begin() + i + 1);
    }
    if (i > 0 && A.free_list[i - 1].p + A.free_list[i - 1].n == A.free_list[i].p &&
        same_slab(A.free_list[i - 1].p, A.free_list[i].p)) {
        A.free_list[i - 1].n += A.free_list[i].n;
        A.free_list.erase(A.free_list.begin() + i);
    }
}

static void *arena_take(PfpArena &A, size_t bytes) {
    for (size_t i = 0; i < A.free_list.size(); i++) {
        if (A.free_list[i].n >= bytes) {
            char *p = A.free_list[i].p;
            if (A.free_list[i].n == bytes) A.free_list.erase(A.free_list.begin() + i);
            else { A.free_list[i].p += bytes; A.free_list[i].n -= bytes; }
            A.used.push_back({p, bytes});
            A.in_use += bytes;
            if (A.in_use > A.peak) A.peak = A.in_use;
            return p;
        }
    }
    return nullptr;
}

static void arena_give(PfpArena &A, void *p) {
    for (size_t i = 0; i < A.used.size(); i++)
        if (A.used[i].p == (char *)p) {
            PfpBlock b = A.used[i];
            A.used[i] = A.used.back();
            A.used.pop_back();
            A.in_use -= b.n;
            arena_insert_free(A, b);
            return;
        }
}

void pfp_arena_destroy(pfpb200_ctx *ctx) {
    for (auto &s : ctx->arena.slabs) cudaFree(s.p);
    ctx->arena = PfpArena();
}

// Called between calls, when nothing is in use: fold several slabs into one so that the next
// call sees a single contiguous range at least as large as the last peak.
int pfp_arena_consolidate(pfpb200_ctx *ctx) {
    PfpArena &A = ctx->arena;
    if (A.slabs.size() <= 1 || A.in_use != 0) return PFPB200_OK;
    size_t want = A.total;
    cudaStreamSynchronize(ctx->stream);
    for (auto &s : A.slabs) cudaFree(s.p);
    A.slabs.clear();
    A.free_list.clear();
    A.total = 0;
    void *p = nullptr;
    if (cudaMalloc(&p, want) != cudaSuccess) { cudaGetLastError(); return PFPB200_OK; }  // grow lazily again
    A.slabs.push_back({(char *)p, want});
    A.free_list.push_back({(char *)p, want});
    A.total = want;
    return PFPB200_OK;
}

void pfp_arena_trim(pfpb200_ctx *ctx) {
    PfpArena &A = ctx->arena;
    cudaStreamSynchronize(ctx->stream);
    for (size_t i = 0; i < A.slabs.size();) {
        const PfpBlock s = A.slabs[i];
        size_t f = 0;
        while (f < A.free_list.size() && !(A.free_list[f].p == s.p && A.free_list[f].n == s.n)) f++;
        if (f == A.free_list.size()) { i++; continue; }          // something in it is in use
        cudaFree(s.p);
        A.free_list.erase(A.free_list.begin() + f);
        A.slabs.erase(A.slabs.begin() + i);
        A.total -= s.n;
    }
}

int pfp_alloc(pfpb200_ctx *ctx, void **p, size_t bytes, bool held) {
    *p = nullptr;
    if (bytes == 0) bytes = 16;
    bytes = (bytes + 511) & ~(size_t)511;
    PfpArena &A = ctx->arena;
    void *q = arena_take(A, bytes);
    if (!q) {
        // grow: a new slab of at least the request, at least 256 MB, at least half of what we have
        size_t slab = bytes;
        if (slab < ((size_t)256 << 20)) slab = (size_t)256 << 20;
        if (slab < A.total / 2) slab = A.total / 2;
        void *base = nullptr;
        cudaError_t e = cudaMalloc(&base, slab);
        if (e != cudaSuccess && slab > bytes) { cudaGetLastError(); slab = bytes; e = cudaMalloc(&base, slab); }
        if (e != cudaSuccess) {
            cudaGetLastError();
            return pfp_fail(ctx, PFPB200_E_NOMEM, "device allocation of %zu bytes failed: %s", bytes,
                            cudaGetErrorString(e));
        }
        A.slabs.push_back({(char *)base, slab});
        A.total += slab;
        arena_insert_free(A, {(char *)base, slab});
        q = arena_take(A, bytes);
        if (!q) return pfp_fail(ctx, PFPB200_E_INTERNAL, "arena inconsistency");
    }
    *p = q;
    (held ? ctx->held : ctx->scratch).push_back(q);
    return PFPB200_OK;
}

// One slab of `bytes` up front (when the arena holds less): a parse whose size is known then reaches
// the driver once instead of at every stage -- with peer access enabled every cudaMalloc is mapped
// into all the peer GPUs, tens of milliseconds each.  Best effort: a failure leaves the arena as it is.
void pfp_arena_reserve(pfpb200_ctx *ctx, size_t bytes) {
    PfpArena &A = ctx->arena;
    if (A.total >= bytes) return;
    size_t want = ((bytes - A.total) + ((size_t)1 << 20) - 1) & ~(((size_t)1 << 20) - 1);
    void *base = nullptr;
    if (cudaMalloc(&base, want) != cudaSuccess) { cudaGetLastError(); return; }
    A.slabs.push_back({(char *)base, want});
    A.total += want;
    arena_insert_free(A, {(char *)base, want});
}

int pfp_free_now(pfpb200_ctx *ctx, void *p) {
    if (!p) return PFPB200_OK;
    for (size_t i = 0; i < ctx->scratch.size(); i++)
        if (ctx->scratch[i] == p) {
            ctx->scratch[i] = ctx->scratch.back();
            ctx->scratch.pop_back();
            arena_give(ctx->arena, p);
            return PFPB200_OK;
        }
    return PFPB200_OK;
}

void pfp_release_scratch(pfpb200_ctx *ctx) {
    for (void *p : ctx->scratch) arena_give(ctx->arena, p);
    ctx->scratch.clear();
}

void pfp_release_held(pfpb200_ctx *ctx) {
    for (void *p : ctx->held) arena_give(ctx->arena, p);
    ctx->held.clear();
    ctx->bp_out[0] = ctx->bp_out[1] = ctx->bp_out[2] = nullptr;
    ctx->up_out = nullptr;
    ctx->pb_out[0] = ctx->pb_out[1] = ctx->pb_out[2] = ctx->pb_out[3] = nullptr;
}

// ------------------------------------------------------------------------------------------
// exclusive scan: reduce tiles -> scan the tile sums (recursively) -> scan tiles with offsets
// ------------------------------------------------------------------------------------------
constexpr int SC_T = 256;
constexpr int SC_I = 8;
constexpr int SC_TILE = SC_T * SC_I;

template <typename T>
__device__ __forceinline__ T warp_incl_scan_t(T v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane_id() >= (u32)o) v += t;
    }
    return v;
}

template <typename T>
__device__ __forceinline__ T block_excl_scan_t(T v, T *total, T *sm /* 9 */) {
    T inc = warp_incl_scan_t<T>(v);
    u32 w = threadIdx.x >> 5;
    __syncthreads();
    if (lane_id() == 31) sm[w] = inc;
    __syncthreads();
    if (threadIdx.x < 32) {
        T x = threadIdx.x < 8 ? sm[threadIdx.x] : (T)0;
        T xi = warp_incl_scan_t<T>(x);
        if (threadIdx.x < 8) sm[threadIdx.x] = xi - x;
        if (threadIdx.x == 7) sm[8] = xi;
    }
    __syncthreads();
    *total = sm[8];
    return inc - v + sm[w];
}

template <typename TIn, typename TOut>
__global__ void __launch_bounds__(SC_T) scan_reduce_k(const TIn *__restrict__ in, u64 n,
                                                      TOut *__restrict__ partial) {
    __shared__ TOut sm[9];
    u64 base = (u64)blockIdx.x * SC_TILE;
    TOut s = 0;
#pragma unroll
    for (int k = 0; k < SC_I; k++) {
        u64 i = base + (u64)k * SC_T + threadIdx.x;
        if (i < n) s += (TOut)in[i];
    }
    TOut total;
    block_excl_scan_t<TOut>(s, &total, sm);
    if (threadIdx.x == 0) partial[blockIdx.x] = total;
}

template <typename TIn, typename TOut>
__global__ void __launch_bounds__(SC_T) scan_apply_k(const TIn *in,   // may alias out
                                                     TOut *out, u64 n,
                                                     const TOut *__restrict__ tile_prefix,
                                                     TOut *__restrict__ d_total) {
    __shared__ TOut sm[9];
    u64 base = (u64)blockIdx.x * SC_TILE + (u64)threadIdx.x * SC_I;
    TOut v[SC_I];
    TOut s = 0;
#pragma unroll
    for (int k = 0; k < SC_I; k++) {
        u64 i = base + k;
        v[k] = (i < n) ? (TOut)in[i] : (TOut)0;
        s += v[k];
    }
    TOut total;
    TOut ex = block_excl_scan_t<TOut>(s, &total, sm);
    if (tile_prefix) ex += tile_prefix[blockIdx.x];
#pragma unroll
    for (int k = 0; k < SC_I; k++) {
        u64 i = base + k;
        if (i < n) {
            out[i] = ex;
            if (d_total && i == n - 1) *d_total = ex + v[k];
        }
        ex += v[k];
    }
}

template <typename TIn, typename TOut>
static int exclusive_scan_impl(pfpb200_ctx *ctx, const TIn *in, TOut *out, u64 n, TOut *d_total) {
    if (n == 0) {
        if (d_total) PFP_CUDA(ctx, cudaMemsetAsync(d_total, 0, sizeof(TOut), ctx->stream));
        return PFPB200_OK;
    }
    u32 nb = pfp_blocks(n, SC_TILE);
    if (nb == 1) {
        scan_apply_k<TIn, TOut><<<1, SC_T, 0, ctx->stream>>>(in, out, n, nullptr, d_total);
        PFP_LAUNCHED(ctx);
        return PFPB200_OK;
    }
    TOut *partial = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &partial, nb));
    scan_reduce_k<TIn, TOut><<<nb, SC_T, 0, ctx->stream>>>(in, n, partial);
    PFP_LAUNCHED(ctx);
    PFP_TRY((exclusive_scan_impl<TOut, TOut>(ctx, partial, partial, nb, nullptr)));
    scan_apply_k<TIn, TOut><<<nb, SC_T, 0, ctx->stream>>>(in, out, n, partial, d_total);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pfp_free_now(ctx, partial));
    return PFPB200_OK;
}

int pfp_exclusive_scan_u32(pfpb200_ctx *ctx, const u32 *in, u32 *out, u64 n, u32 *d_total) {
    return exclusive_scan_impl<u32, u32>(ctx, in, out, n, d_total);
}
int pfp_exclusive_scan_u32_u64(pfpb200_ctx *ctx, const u32 *in, u64 *out, u64 n, u64 *d_total) {
    return exclusive_scan_impl<u32, u64>(ctx, in, out, n, d_total);
}
int pfp_exclusive_scan_u8_u32(pfpb200_ctx *ctx, const u8 *in, u32 *out, u64 n, u32 *d_total) {
    return exclusive_scan_impl<u8, u32>(ctx, in, out, n, d_total);
}

// ------------------------------------------------------------------------------------------
// radix sort: per pass  histogram -> scan -> ranked scatter   (8-bit digits)
// ------------------------------------------------------------------------------------------
constexpr int RS_T = 256;
constexpr int RS_I = 8;
constexpr int RS_TILE = RS_T * RS_I;   // 4096 pairs per CTA
constexpr int RS_WARPS = RS_T / 32;
constexpr int RS_SUB = RS_TILE / RS_WARPS;   // 512 consecutive items per warp

__global__ void __launch_bounds__(RS_T) rs_hist_k(const u64 *__restrict__ keys, u64 n, int shift,
                                                  u32 *__restrict__ hist, u32 nblocks) {
    __shared__ u32 h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    u64 base = (u64)blockIdx.x * RS_TILE;
#pragma unroll 4
    for (int k = 0; k < RS_I; k++) {
        u64 i = base + (u64)k * RS_T + threadIdx.x;
        bool valid = i < n;
        u32 d = valid ? (u32)((keys[i] >> shift) & 255) : 256u;
        u32 peers = __match_any_sync(0xffffffffu, d);
        if (valid && (peers & lanemask_lt()) == 0) atomicAdd(&h[d], __popc(peers));
    }
    __syncthreads();
    hist[(u64)threadIdx.x * nblocks + blockIdx.x] = h[threadIdx.x];
}

struct RsSmem {
    u64 key[RS_TILE];
    u32 val[RS_TILE];
    u32 wcnt[RS_WARPS][256];
    u32 tile_start[256];
    u32 gbase[256];
    u32 scan_sm[9];
};

__global__ void __launch_bounds__(RS_T) rs_scatter_k(const u64 *__restrict__ kin,
                                                     const u32 *__restrict__ vin,
                                                     u64 *__restrict__ kout, u32 *__restrict__ vout,
                                                     u64 n, int shift,
                                                     const u32 *__restrict__ offs, u32 nblocks) {
    extern __shared__ __align__(16) unsigned char rs_raw[];
    RsSmem &S = *reinterpret_cast<RsSmem *>(rs_raw);
    const u32 t = threadIdx.x, wi = t >> 5, ln = t & 31;
    const u64 base = (u64)blockIdx.x * RS_TILE;
    const u32 count = (u32)((n - base) < (u64)RS_TILE ? (n - base) : (u64)RS_TILE);

    for (int i = t; i < RS_WARPS * 256; i += RS_T) (&S.wcnt[0][0])[i] = 0;
    __syncthreads();

    u64 k[RS_I];
    u32 v[RS_I];
    u32 pos[RS_I];
#pragma unroll
    for (int r = 0; r < RS_I; r++) {
        u32 idx = wi * RS_SUB + r * 32 + ln;
        bool valid = idx < count;
        k[r] = valid ? kin[base + idx] : 0;
        v[r] = valid ? vin[base + idx] : 0;
    }
    // warp-level multisplit: rank of each item among equal digits, in (round, lane) order
#pragma unroll
    for (int r = 0; r < RS_I; r++) {
        u32 idx = wi * RS_SUB + r * 32 + ln;
        bool valid = idx < count;
        u32 d = valid ? (u32)((k[r] >> shift) & 255) : 256u;
        u32 peers = __match_any_sync(0xffffffffu, d);
        u32 rank = __popc(peers & lanemask_lt());
        u32 prev = valid ? S.wcnt[wi][d] : 0;
        pos[r] = prev + rank;
        __syncwarp();
        if (valid && rank == 0) S.wcnt[wi][d] = prev + __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    // thread t owns digit t: exclusive scan over the warps, then over the digits
    u32 run = 0;
#pragma unroll
    for (int w2 = 0; w2 < RS_WARPS; w2++) {
        u32 c = S.wcnt[w2][t];
        S.wcnt[w2][t] = run;
        run += c;
    }
    u32 tot;
    u32 ts = block_excl_scan_256(run, &tot, S.scan_sm);
    S.tile_start[t] = ts;
    S.gbase[t] = offs[(u64)t * nblocks + blockIdx.x] - ts;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < RS_I; r++) {
        u32 idx = wi * RS_SUB + r * 32 + ln;
        if (idx < count) {
            u32 d = (u32)((k[r] >> shift) & 255);
            u32 lp = S.tile_start[d] + S.wcnt[wi][d] + pos[r];
            S.key[lp] = k[r];
            S.val[lp] = v[r];
        }
    }
    __syncthreads();
    for (u32 i = t; i < count; i += RS_T) {
        u64 key = S.key[i];
        u32 d = (u32)((key >> shift) & 255);
        u32 g = S.gbase[d] + i;
        kout[g] = key;
        vout[g] = S.val[i];
    }
}

int pfp_prims_init(pfpb200_ctx *ctx) {
    PFP_CUDA(ctx, cudaFuncSetAttribute(rs_scatter_k, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)sizeof(RsSmem)));
    return PFPB200_OK;
}

int pfp_radix_sort_pairs(pfpb200_ctx *ctx, u64 *k0, u32 *v0, u64 *k1, u32 *v1, u64 n,
                         int begin_bit, int end_bit, u64 **res_k, u32 **res_v) {
    *res_k = k0;
    *res_v = v0;
    if (n <= 1 || end_bit <= begin_bit) return PFPB200_OK;
    if (n >= 0xFFFFFFFFull) return pfp_fail(ctx, PFPB200_E_LIMIT, "radix sort: too many items");
    u32 nb = pfp_blocks(n, RS_TILE);
    u32 *hist = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &hist, (size_t)256 * nb));
    u64 *ka = k0, *kb = k1;
    u32 *va = v0, *vb = v1;
    for (int shift = begin_bit; shift < end_bit; shift += 8) {
        rs_hist_k<<<nb, RS_T, 0, ctx->stream>>>(ka, n, shift, hist, nb);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_exclusive_scan_u32(ctx, hist, hist, (u64)256 * nb, nullptr));
        rs_scatter_k<<<nb, RS_T, sizeof(RsSmem), ctx->stream>>>(ka, va, kb, vb, n, shift, hist, nb);
        PFP_LAUNCHED(ctx);
        u64 *tk = ka; ka = kb; kb = tk;
        u32 *tv = va; va = vb; vb = tv;
    }
    PFP_TRY(pfp_free_now(ctx, hist));
    *res_k = ka;
    *res_v = va;
    return PFPB200_OK;
}
