// pfp_common.cuh -- context, error handling and device primitives shared by all stages.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <vector>
#include "pfp_arith.h"
#include "../../include/pfpb200.h"

typedef uint64_t u64;
typedef uint32_t u32;
typedef uint16_t u16;
typedef uint8_t u8;
typedef int64_t i64;

// Device scratch arena: a few big cudaMalloc'd slabs carved by a first-fit free list on the
// host.  All work of a context is ordered on one stream, so a block freed on the host may be
// handed out again at once.  After the first call on a workload no allocation reaches the driver.
struct PfpBlock { char *p; size_t n; };
struct PfpArena {
    std::vector<PfpBlock> slabs;
    std::vector<PfpBlock> free_list;   // sorted by address, coalesced
    std::vector<PfpBlock> used;
    size_t in_use = 0, peak = 0, total = 0;
};

// ---- trigger bits of a buffer (K1a output) ------------------------------------------------------
// Positions are counted in "q" coordinates: byte offsets from the 16-byte aligned address A at
// or below the buffer start; global text position = q + pos_bias.  Bit q of `mask` (little
// endian 32-bit words) is set iff an owned trigger ends at q.  Tiles of PFP_TILE positions.
constexpr int PFP_TILE_T = 256;                        // threads per tile CTA
constexpr int PFP_TILE_RUN = 128;                      // positions per thread
constexpr int PFP_TILE = PFP_TILE_T * PFP_TILE_RUN;    // 32768 positions per tile
struct ScanBits {
    const uint4 *A;
    u64 q_end;          // q of the first byte behind the buffer
    u64 pos_bias;       // global position of q = 0 (may wrap below zero; arithmetic is modular)
    u32 ntiles;         // 0: nothing was scanned (empty range)
    uint4 *mask;        // [ntiles * 256] = 128 bits per thread run
    u32 *tile_cnt;      // [ntiles] triggers per tile
    u64 *tile_off;      // [ntiles] triggers before the tile
    u64 total;          // all triggers
    u32 max_tile_cnt;   // largest tile_cnt
};

// pinned ring of the overlapped file I/O (pfp_ingest.cu): IO_THREADS workers, two slots each
constexpr int PFP_IO_THREADS = 4;
constexpr size_t PFP_IO_CHUNK = (size_t)8 << 20;
struct PfpIo {
    bool ready = false;
    void *slot[PFP_IO_THREADS][2] = {{nullptr}};
    cudaEvent_t ev[PFP_IO_THREADS][2] = {{nullptr}};
    cudaStream_t stream[PFP_IO_THREADS] = {nullptr};
};

struct pfpb200_ctx {
    int device = 0;
    PfpIo io;
    PfpArena arena;
    int sm_count = 148;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    u32 launches = 0;
    bool k1_rolling = false;       // PFPB200_K1=rolling: always the rolling-arithmetic scan kernel
    // byte values present in the text, as a by-product of the DNA form of K1 (8 x 32 bits): rows that
    // the interval form takes hold only A C G T, the others record their bytes.  Valid for the words of
    // a single-GPU parse; lets the ranking skip its own pass over the words' first bytes.
    u32 *d_alpha = nullptr;
    bool alpha_valid = false;
    void *iv_etab = nullptr;       // interval form of the DNA scan, tables of (iv_w, iv_p): 1024 x {a16 + 2, b16} (w <= 10)
    void *iv_xtab = nullptr;       //   or 256 x {f1 f0, f3 f2} (w <= 16); and the exact partial hashes {Ah, Bl} / {F0..F3}
    u32 iv_w = 0, iv_p = 0, iv_cthr = 0;
    int iv_skip = 0;               // > 0: the last scan found text that is not DNA, use the rolling kernel for this many calls
    bool rank_chunk_passes = false;  // PFPB200_RANK_CHUNK_PASSES=1: mid-size tie groups by chunk passes instead of LCP walks (A/B)
    bool rank_warp_passes = false;   // PFPB200_RANK_WARP_PASSES=1: tie groups of 2..32 words by warp chunk passes instead of LCP walks (A/B)
    bool legacy_k2 = false;        // PFPB200_LEGACY_K2=1: per-phrase K2 kernels (A/B measurements)
    u32 weak_fp = 0;               // PFPB200_TEST_WEAK_FP=1 (tests): 2-bit fingerprints, so that PFPB200_F_VERIFY has collisions to catch
    double dedup_ratio = 0.0;      // distinct words / phrases of the previous parse (table sizing hint)
    u64 plan_chunks = 0, plan_peak = 0;   // pfpb200_parse_plan: chunks (0: one-shot) and arena peak of the last parse_file
    u64 pb_windows = 0, pb_peak = 0;      // pfpb200_pfbwt_plan: output windows and arena peak of the last pfbwt file call
    u64 bp_windows = 0, bp_peak = 0;      // pfpb200_bwtparse_plan: round-1 windows (1: in HBM) and arena peak of the last bwtparse file call
    char err[512] = {0};
    std::vector<void *> scratch;   // freed at the end of every call
    std::vector<void *> held;      // outputs: freed at the start of the next call / destroy
    void *bp_out[3] = {nullptr, nullptr, nullptr};   // held outputs of the last pfpb200_bwtparse_* call
    void *up_out = nullptr;        // held output of the last pfpb200_unparse_device call
    void *pb_out[4] = {nullptr, nullptr, nullptr, nullptr};   // held outputs of the last pfpb200_pfbwt_* call
    void *pin_buf[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // host outputs of parse_host,
    size_t pin_cap[5] = {0, 0, 0, 0, 0};                                 // kept and grown across calls
    // parse_host: .last/.sai are final after K2 and travel to the host on a second stream while
    // the dictionary stages run
    // K5 (remap) needs only the ranks: it runs here while the .dict bytes are gathered on the main stream
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t ev_aux0 = nullptr, ev_aux1 = nullptr;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_k2 = nullptr, ev_copy = nullptr;
    bool early_copy = false;       // set by parse_host for the duration of the call
    bool early_done = false;       // the copies were issued (ev_copy marks their end)
    // persistent small device state
    u32 *d_keys = nullptr;         // NH key table (phrase fingerprints)
    u64 *d_flags = nullptr;        // [0] error bits, [1..] counters read back by the host
    u64 *h_flags = nullptr;        // pinned mirror
    // state carried from pfpb200_dict_merge_begin to pfpb200_dict_merge_finish
    struct {
        u64 n_in = 0, d = 0, sum_len = 0;
        u32 max_len = 0;
        u32 *uid_of_entry = nullptr, *rep = nullptr, *count = nullptr, *ulen = nullptr, *uwords = nullptr;
        u64 *uoff = nullptr;
        const u32 *len_in = nullptr, *uwords_in = nullptr;
    } mg;
    // state carried between the pfpb200_shard_* calls of one sharded parse
    struct {
        pfpb200_shard desc;
        pfpb200_opts opts;
        u64 *ends = nullptr;
        bool ends_emitted = true;      // false: shard_words' streaming pass still has to write ends[]
        ScanBits bits;                 // trigger bits of the shard, kept from shard_scan to shard_words
        u64 n_trig = 0, P = 0, d = 0;
        u32 *uid = nullptr;
        // local dictionary of the shard (held until the next parse)
        u64 *wfpa = nullptr, *wfpb = nullptr, *pool = nullptr, *uoff = nullptr, pool_words = 0;
        u32 *ulen = nullptr, *count = nullptr, *uwords = nullptr;
        // routing plan kept between pfpb200_shard_route_plan and pfpb200_shard_route_push
        u32 *route_perm = nullptr;
        u64 *route_ooff = nullptr;
        u64 route_words_to[PFPB200_MAX_RANKS] = {0}, route_pool_to[PFPB200_MAX_RANKS] = {0};
    } sh;
};

#define PFP_FLAG_SLOTS 16
#define PFP_ERRBIT_COLLISION 1ull
#define PFP_ERRBIT_LIMIT 2ull
#define PFP_ERRBIT_INTERNAL 4ull
#define PFP_ERRBIT_TABLE_FULL 8ull

int pfp_fail(pfpb200_ctx *ctx, int code, const char *fmt, ...);

#define PFP_CUDA(ctx, call)                                                                 \
    do {                                                                                    \
        cudaError_t e_ = (call);                                                            \
        if (e_ != cudaSuccess)                                                              \
            return pfp_fail((ctx), e_ == cudaErrorMemoryAllocation ? PFPB200_E_NOMEM        \
                                                                   : PFPB200_E_CUDA,        \
                            "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
    } while (0)

#define PFP_TRY(expr)                 \
    do {                              \
        int rc_ = (expr);             \
        if (rc_ != PFPB200_OK) return rc_; \
    } while (0)

// counts a launch and checks it
#define PFP_LAUNCHED(ctx)                                                                   \
    do {                                                                                    \
        (ctx)->launches++;                                                                  \
        cudaError_t e_ = cudaGetLastError();                                                \
        if (e_ != cudaSuccess)                                                              \
            return pfp_fail((ctx), PFPB200_E_CUDA, "%s:%d launch: %s", __FILE__, __LINE__,  \
                            cudaGetErrorString(e_));                                        \
    } while (0)

// ---- scratch memory (stream-ordered pool) ----------------------------------------------
int pfp_alloc(pfpb200_ctx *ctx, void **p, size_t bytes, bool held = false);
int pfp_free_now(pfpb200_ctx *ctx, void *p);   // early release of one scratch buffer
void pfp_release_scratch(pfpb200_ctx *ctx);
void pfp_release_held(pfpb200_ctx *ctx);
void pfp_arena_destroy(pfpb200_ctx *ctx);
int pfp_arena_consolidate(pfpb200_ctx *ctx);
void pfp_arena_trim(pfpb200_ctx *ctx);   // slabs with nothing in use go back to the driver
void pfp_arena_reserve(pfpb200_ctx *ctx, size_t bytes);

template <typename T>
static inline int pfp_alloc_t(pfpb200_ctx *ctx, T **p, size_t count, bool held = false) {
    return pfp_alloc(ctx, (void **)p, (count ? count : 1) * sizeof(T), held);
}

// Function attributes (dynamic shared memory limits) and constant memory are per DEVICE.  Every
// translation unit sets its own in pfpb200_create() -- unconditionally, once per context, on the
// context's device -- so there is no process-wide "already done" state for host threads to race on.
int pfp_scan_init(pfpb200_ctx *ctx);
int pfp_stream_init(pfpb200_ctx *ctx);
int pfp_prims_init(pfpb200_ctx *ctx);
int pfp_rank_init(pfpb200_ctx *ctx);

// a handful of CUDA events that are destroyed on every exit path of the scope that made them
struct PfpEvents {
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    bool ok = true;
    explicit PfpEvents(int n) {
        for (int i = 0; i < n && i < 4; i++)
            if (cudaEventCreate(&ev[i]) != cudaSuccess) { ev[i] = nullptr; ok = false; }
    }
    ~PfpEvents() {
        for (int i = 0; i < 4; i++)
            if (ev[i]) cudaEventDestroy(ev[i]);
    }
    PfpEvents(const PfpEvents &) = delete;
    PfpEvents &operator=(const PfpEvents &) = delete;
    cudaEvent_t operator[](int i) const { return ev[i]; }
};

static inline u32 pfp_blocks(u64 n, u32 per_block) { return (u32)((n + per_block - 1) / per_block); }

// ---- primitives (pfp_prims.cu) -----------------------------------------------------------
// out[i] = sum_{j<i} in[j]; if d_total != null, *d_total = sum of all (device pointer).
int pfp_exclusive_scan_u32(pfpb200_ctx *ctx, const u32 *in, u32 *out, u64 n, u32 *d_total);
int pfp_exclusive_scan_u32_u64(pfpb200_ctx *ctx, const u32 *in, u64 *out, u64 n, u64 *d_total);
int pfp_exclusive_scan_u8_u32(pfpb200_ctx *ctx, const u8 *in, u32 *out, u64 n, u32 *d_total);

// Stable LSD radix sort of (u64 key, u32 value) pairs on key bits [begin_bit, end_bit).
// Ping-pongs between (k0,v0) and (k1,v1); *res_k/*res_v point at the sorted pair on return.
int pfp_radix_sort_pairs(pfpb200_ctx *ctx, u64 *k0, u32 *v0, u64 *k1, u32 *v1, u64 n,
                         int begin_bit, int end_bit, u64 **res_k, u32 **res_v);

// ---- small device helpers ---------------------------------------------------------------------
__device__ __forceinline__ u32 lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ u32 lanemask_lt() {
    u32 m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}
__device__ __forceinline__ u32 warp_incl_scan(u32 v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane_id() >= (u32)o) v += t;
    }
    return v;
}
// exclusive scan over a 256-thread block; returns exclusive prefix, *total = block sum
__device__ __forceinline__ u32 block_excl_scan_256(u32 v, u32 *total, u32 *sm /*>=9 u32*/) {
    u32 inc = warp_incl_scan(v);
    u32 w = threadIdx.x >> 5;
    __syncthreads();   // protect sm from a previous use
    if (lane_id() == 31) sm[w] = inc;
    __syncthreads();
    if (threadIdx.x < 32) {
        u32 x = threadIdx.x < 8 ? sm[threadIdx.x] : 0;
        u32 xi = warp_incl_scan(x);
        if (threadIdx.x < 8) sm[threadIdx.x] = xi - x;
        if (threadIdx.x == 7) sm[8] = xi;
    }
    __syncthreads();
    *total = sm[8];
    return inc - v + sm[w];
}
