// pfp_api.cu -- the C ABI of libpfpb200.so (include/pfpb200.h): context management and the
// orchestration of the stages K1..K5 for one GPU.
#include "pfp_common.cuh"
#include "pfp_stages.cuh"
#include <errno.h>
#include <fcntl.h>
#include <stdlib.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>

extern "C" {
int pfp_io_read_file(const char *path, int gz_ok, uint8_t **buf, uint64_t *n, char *err, size_t errlen);
int pfp_io_write_outputs(const char *path, const pfpb200_opts *opts, const pfpb200_outputs *o,
                         char *err, size_t errlen);
}

static double wall_sec() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

__global__ void set_u64_k(u64 *p, u64 v) { *p = v; }

// first position holding a byte <= 0x02 (newscan.cpp:364), or n: 16-byte loads, the classic
// "has a byte below k" word test, exact position only in the rare word that trips it
__global__ void __launch_bounds__(256) first_invalid_k(const u8 *__restrict__ t, u64 n,
                                                       unsigned long long *__restrict__ first) {
    const u64 stride = (u64)gridDim.x * blockDim.x * 16;
    for (u64 i = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * 16; i < n; i += stride) {
        bool hit = false;
        if (i + 16 <= n && (((uintptr_t)(t + i)) & 15) == 0) {
            uint4 v = __ldg(reinterpret_cast<const uint4 *>(t + i));
            u32 w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; k++) hit |= ((w[k] - 0x03030303u) & ~w[k] & 0x80808080u) != 0;
        } else hit = true;
        if (hit) {
            u64 e = i + 16 < n ? i + 16 : n;
            for (u64 j = i; j < e; j++)
                if (t[j] <= PFP_DOLLAR) { atomicMin(first, (unsigned long long)j); break; }
        }
    }
}

// *d_first (device u64, caller-initialised to n) = first position of text[0..n) holding a byte
// <= 0x02, where the reference stops reading (newscan.cpp:364)
int pfp_first_invalid(pfpb200_ctx *ctx, const u8 *d_text, u64 n, u64 *d_first) {
    if (n == 0) return PFPB200_OK;
    first_invalid_k<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(d_text, n,
                                                               reinterpret_cast<unsigned long long *>(d_first));
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

extern "C" int pfpb200_abi_version(void) { return PFPB200_ABI_VERSION; }

extern "C" const char *pfpb200_strerror(int code) {
    switch (code) {
        case PFPB200_OK: return "ok";
        case PFPB200_E_ARG: return "invalid argument";
        case PFPB200_E_IO: return "file I/O error";
        case PFPB200_E_CUDA: return "CUDA error (no usable GPU or kernel failure)";
        case PFPB200_E_NOMEM: return "out of memory";
        case PFPB200_E_LIMIT: return "algorithm limit exceeded";
        case PFPB200_E_COLLISION: return "fingerprint collision";
        case PFPB200_E_INTERNAL: return "internal error";
        default: return "unknown error";
    }
}

extern "C" uint32_t pfpb200_launch_count(const pfpb200_ctx *ctx) { return ctx ? ctx->launches : 0; }

extern "C" const char *pfpb200_last_error(const pfpb200_ctx *ctx) { return ctx ? ctx->err : ""; }

static u64 splitmix64(u64 &s) {
    u64 z = (s += 0x9E3779B97F4A7C15ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

extern "C" int pfpb200_create(int device, pfpb200_ctx **out) {
    if (!out) return PFPB200_E_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
        cudaGetLastError();
        return PFPB200_E_CUDA;   // no CPU fallback: without a GPU there is no product
    }
    pfpb200_ctx *ctx = new (std::nothrow) pfpb200_ctx();
    if (!ctx) return PFPB200_E_NOMEM;
    ctx->device = device;
    { const char *ev = getenv("PFPB200_LEGACY_K2"); ctx->legacy_k2 = ev && atoi(ev) != 0; }
    { const char *ev = getenv("PFPB200_K1"); ctx->k1_rolling = ev && strcmp(ev, "rolling") == 0; }
    { const char *ev = getenv("PFPB200_TEST_WEAK_FP"); ctx->weak_fp = (ev && atoi(ev) != 0) ? 1u : 0u; }
    { const char *ev = getenv("PFPB200_RANK_CHUNK_PASSES"); ctx->rank_chunk_passes = ev && atoi(ev) != 0; }
    { const char *ev = getenv("PFPB200_RANK_WARP_PASSES"); ctx->rank_warp_passes = ev && atoi(ev) != 0; }
    auto bail = [&](int code) { pfpb200_destroy(ctx); return code; };
    if (cudaSetDevice(device) != cudaSuccess) return bail(PFPB200_E_CUDA);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return bail(PFPB200_E_CUDA);
    ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(PFPB200_E_CUDA);
    ctx->stream = ctx->own_stream;
    if (cudaMalloc(&ctx->d_flags, PFP_FLAG_SLOTS * sizeof(u64)) != cudaSuccess ||
        cudaMallocHost(&ctx->h_flags, PFP_FLAG_SLOTS * sizeof(u64)) != cudaSuccess ||
        cudaMalloc(&ctx->d_keys, NH_KEY_WORDS * sizeof(u32)) != cudaSuccess ||
        cudaMalloc(&ctx->d_alpha, 8 * sizeof(u32)) != cudaSuccess)
        return bail(PFPB200_E_NOMEM);
    u32 hk[NH_KEY_WORDS];
    u64 seed = 0x5bd1e9955bd1e995ULL;
    for (u32 i = 0; i < NH_KEY_WORDS; i++) hk[i] = (u32)(splitmix64(seed) >> 32);
    if (cudaMemcpy(ctx->d_keys, hk, sizeof(hk), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemset(ctx->d_flags, 0, PFP_FLAG_SLOTS * sizeof(u64)) != cudaSuccess)
        return bail(PFPB200_E_CUDA);
    // fail here, loudly, if the library carries no kernel image for this GPU
    set_u64_k<<<1, 1, 0, ctx->stream>>>(&ctx->d_flags[15], 1);
    if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(ctx->stream) != cudaSuccess)
        return bail(PFPB200_E_CUDA);
    if (cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_aux0, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_aux1, cudaEventDisableTiming) != cudaSuccess)
        return bail(PFPB200_E_CUDA);
    // per-device kernel attributes and constants of every stage (see pfp_common.cuh)
    if (pfp_scan_init(ctx) || pfp_stream_init(ctx) || pfp_prims_init(ctx) || pfp_rank_init(ctx))
        return bail(PFPB200_E_CUDA);
    *out = ctx;
    return PFPB200_OK;
}

extern "C" void pfpb200_destroy(pfpb200_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    pfp_release_scratch(ctx);
    pfp_release_held(ctx);
    pfp_arena_destroy(ctx);
    if (ctx->own_stream) { cudaStreamSynchronize(ctx->own_stream); cudaStreamDestroy(ctx->own_stream); }
    if (ctx->d_flags) cudaFree(ctx->d_flags);
    if (ctx->h_flags) cudaFreeHost(ctx->h_flags);
    if (ctx->d_keys) cudaFree(ctx->d_keys);
    if (ctx->iv_etab) cudaFree(ctx->iv_etab);
    if (ctx->iv_xtab) cudaFree(ctx->iv_xtab);
    if (ctx->d_alpha) cudaFree(ctx->d_alpha);
    pfp_io_destroy(ctx);
    for (int i = 0; i < 5; i++)
        if (ctx->pin_buf[i]) cudaFreeHost(ctx->pin_buf[i]);
    if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
    if (ctx->aux_stream) { cudaStreamSynchronize(ctx->aux_stream); cudaStreamDestroy(ctx->aux_stream); }
    if (ctx->ev_aux0) cudaEventDestroy(ctx->ev_aux0);
    if (ctx->ev_aux1) cudaEventDestroy(ctx->ev_aux1);
    if (ctx->ev_k2) cudaEventDestroy(ctx->ev_k2);
    if (ctx->ev_copy) cudaEventDestroy(ctx->ev_copy);
    delete ctx;
}

extern "C" int pfpb200_set_stream(pfpb200_ctx *ctx, void *cuda_stream) {
    if (!ctx) return PFPB200_E_ARG;
    cudaStreamSynchronize(ctx->stream);
    pfp_release_scratch(ctx);
    pfp_release_held(ctx);
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return PFPB200_OK;
}

static int check_opts(pfpb200_ctx *ctx, const pfpb200_opts *o) {
    if (!ctx) return PFPB200_E_ARG;
    if (!o) return pfp_fail(ctx, PFPB200_E_ARG, "null options");
    if (o->w < 4) return pfp_fail(ctx, PFPB200_E_ARG, "Windows size must be at least 4");   // newscan.cpp:537
    if (o->p < 10) return pfp_fail(ctx, PFPB200_E_ARG, "Modulus must be at least 10");      // newscan.cpp:541
    if (o->w > 65536) return pfp_fail(ctx, PFPB200_E_ARG, "window size too large");
    if (o->nseg < 0) return pfp_fail(ctx, PFPB200_E_ARG, "Number of threads cannot be negative");
    return PFPB200_OK;
}

static int begin_call(pfpb200_ctx *ctx) {
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    pfp_release_scratch(ctx);
    pfp_release_held(ctx);
    PFP_TRY(pfp_arena_consolidate(ctx));
    ctx->launches = 0;
    ctx->err[0] = 0;
    PFP_CUDA(ctx, cudaMemsetAsync(ctx->d_flags, 0, PFP_FLAG_SLOTS * sizeof(u64), ctx->stream));
    return PFPB200_OK;
}

struct StageTimer {
    cudaEvent_t ev[10] = {nullptr};
    int n = 0;
    int init() {
        for (int i = 0; i < 10; i++)
            if (cudaEventCreate(&ev[i]) != cudaSuccess) { ev[i] = nullptr; return -1; }
        return 0;
    }
    void mark(cudaStream_t s) { cudaEventRecord(ev[n++], s); }
    float ms(int a, int b) { float t = 0; cudaEventElapsedTime(&t, ev[a], ev[b]); return t; }
    ~StageTimer() {
        for (int i = 0; i < 10; i++)
            if (ev[i]) cudaEventDestroy(ev[i]);
    }
};

// pinned host buffer `slot` of the context, grown on demand
static int pfp_pin(pfpb200_ctx *ctx, int slot, void **h, size_t bytes) {
    if (bytes > ctx->pin_cap[slot]) {
        if (ctx->pin_buf[slot]) cudaFreeHost(ctx->pin_buf[slot]);
        ctx->pin_buf[slot] = nullptr;
        ctx->pin_cap[slot] = 0;
        size_t cap = bytes + bytes / 8 + 4096;
        if (cudaMallocHost(&ctx->pin_buf[slot], cap) != cudaSuccess) {
            cudaGetLastError();
            return pfp_fail(ctx, PFPB200_E_NOMEM, "pinned host allocation of %zu bytes failed", cap);
        }
        ctx->pin_cap[slot] = cap;
    }
    *h = ctx->pin_buf[slot];
    return PFPB200_OK;
}

// text resident on the device -> all outputs on the device
static int parse_device_impl(pfpb200_ctx *ctx, const u8 *d_text, u64 n, const pfpb200_opts *o,
                             pfpb200_outputs *out, pfpb200_stats *st) {
    const u32 w = o->w, p = o->p;
    StageTimer tm;
    if (tm.init()) return pfp_fail(ctx, PFPB200_E_CUDA, "cudaEventCreate failed");
    int rc = PFPB200_OK;
    auto run = [&]() -> int {
        tm.mark(ctx->stream);                                           // 0
        // K1: trigger bits
        ScanBits sb;
        float ms_scan = 0, ms_emit = 0;
        PFP_TRY(pfp_scan_bits(ctx, d_text, n, 0, 0, n, w, p, false, &sb, &ms_scan));
        const u64 k = sb.total;
        const u64 P = k + 1;
        if (P >= 0xFFFFFFFFull)
            return pfp_fail(ctx, PFPB200_E_LIMIT, "the parse contains %llu words, more than 2^32-2",
                            (unsigned long long)P);                     // bigbwt:110-114
        u64 *ends = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &ends, P));
        set_u64_k<<<1, 1, 0, ctx->stream>>>(ends + k, n + w - 1);       // final word (:376-377)
        PFP_LAUNCHED(ctx);
        tm.mark(ctx->stream);                                           // 1
        // K2: positions, .last, .sai and fingerprints in one pass over text + bits
        PhraseArrays ph{};
        ph.ends = ends;
        PFP_TRY(pfp_alloc_t(ctx, &ph.last, P, true));
        if (o->flags & PFPB200_F_SAI) PFP_TRY(pfp_alloc_t(ctx, &ph.sai, P * PFP_IBYTES, true));
        TextView tv{d_text, n, 0, (i64)n};
        DictArrays D;
        PFP_TRY(pfp_alloc_t(ctx, &ph.rec, P));
        if (pfp_stream_ok(sb, w) && !ctx->legacy_k2) PFP_TRY(pfp_stream_stage(ctx, sb, tv, ph, P, -1, w, true));
        else {                                                          // any window size
            PFP_TRY(pfp_scan_emit(ctx, sb, ends));
            PFP_TRY(pfp_hash_stage(ctx, tv, ph, P, -1, w));
        }
        PFP_TRY(pfp_scan_bits_free(ctx, &sb));
        tm.mark(ctx->stream);                                           // 2
        if (ctx->early_copy) {          // .last/.sai are final: to the host while K3/K4 run
            void *h_last = nullptr, *h_sai = nullptr;
            PFP_TRY(pfp_pin(ctx, 3, &h_last, P));
            if (ph.sai) PFP_TRY(pfp_pin(ctx, 4, &h_sai, P * PFP_IBYTES));
            if (!ctx->copy_stream) {
                PFP_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
                PFP_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_k2, cudaEventDisableTiming));
                PFP_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_copy, cudaEventDisableTiming));
            }
            PFP_CUDA(ctx, cudaEventRecord(ctx->ev_k2, ctx->stream));
            PFP_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_k2, 0));
            PFP_CUDA(ctx, cudaMemcpyAsync(h_last, ph.last, P, cudaMemcpyDeviceToHost, ctx->copy_stream));
            if (ph.sai)
                PFP_CUDA(ctx, cudaMemcpyAsync(h_sai, ph.sai, P * PFP_IBYTES, cudaMemcpyDeviceToHost, ctx->copy_stream));
            PFP_CUDA(ctx, cudaEventRecord(ctx->ev_copy, ctx->copy_stream));
            ctx->early_done = true;
        }
        // K3
        PFP_TRY(pfp_dedup_stage(ctx, ph, P, -1, w, &D));
        PFP_TRY(pfp_free_now(ctx, ph.rec));
        PFP_TRY(pfp_pool_stage(ctx, tv, &D));
        if (o->flags & PFPB200_F_VERIFY) {
            PFP_TRY(pfp_uid_words(ctx, &D, P));
            PFP_TRY(pfp_verify_stage(ctx, tv, ends, -1, w, P, D));
        }
        tm.mark(ctx->stream);                                           // 3
        // K4
        u32 *order = nullptr, rounds = 0;
        PFP_TRY(pfp_rank_stage(ctx, D, &order, &rounds, ctx->alpha_valid));
        tm.mark(ctx->stream);                                           // 4
        u8 *dict = nullptr;
        u32 *occ = nullptr, *rank_of_uid = nullptr;
        u64 dict_bytes = 0;
        // K5 (remap) runs on the aux stream beside the .dict gather: it only needs the ranks
        u32 *parse = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &parse, P, true));
        PFP_TRY(pfp_dict_stage(ctx, D, order, (o->flags & PFPB200_F_COMPRESS) ? w : 0, &dict,
                               &dict_bytes, &occ, &rank_of_uid, D.uid, P, parse));
        tm.mark(ctx->stream);                                           // 5
        tm.mark(ctx->stream);                                           // 6
        PFP_CUDA(ctx, cudaMemcpyAsync(ctx->h_flags, ctx->d_flags, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        PFP_CUDA(ctx, cudaGetLastError());
        if (ctx->h_flags[0] & PFP_ERRBIT_COLLISION)
            return pfp_fail(ctx, PFPB200_E_COLLISION, "two different phrases share a fingerprint (found by the verify pass)");
        out->dict = dict; out->dict_bytes = dict_bytes;
        out->occ = occ; out->n_distinct = D.d;
        out->parse = parse; out->n_phrases = P;
        out->last = ph.last;
        out->sai = ph.sai;
        if (st) {
            st->n_text = n; st->n_phrases = P; st->n_distinct = D.d;
            st->sum_word_len = D.sum_len; st->dict_bytes = dict_bytes;
            st->alg_bytes = n + 4 * P + P + ((o->flags & PFPB200_F_SAI) ? 5 * P : 0) + dict_bytes + 4 * D.d;
            st->rank_rounds = rounds;
            st->launches = ctx->launches;
            st->ms_total = tm.ms(0, 6);
            st->ms_scan = ms_scan; st->ms_emit = ms_emit;
            st->ms_hash = tm.ms(1, 2); st->ms_dedup = tm.ms(2, 3); st->ms_rank = tm.ms(3, 4);
            st->ms_dict = tm.ms(4, 5); st->ms_remap = tm.ms(5, 6);
        }
        return PFPB200_OK;
    };
    rc = run();
    if (rc != PFPB200_OK) cudaStreamSynchronize(ctx->stream);
    pfp_release_scratch(ctx);
    return rc;
}

extern "C" int pfpb200_parse_device(pfpb200_ctx *ctx, const uint8_t *d_text, uint64_t n_text,
                                    const pfpb200_opts *opts, pfpb200_outputs *dev_out,
                                    pfpb200_stats *stats) {
    PFP_TRY(check_opts(ctx, opts));
    if (!dev_out || (n_text && !d_text)) return pfp_fail(ctx, PFPB200_E_ARG, "null buffer");
    if (stats) memset(stats, 0, sizeof(*stats));
    memset(dev_out, 0, sizeof(*dev_out));
    PFP_TRY(begin_call(ctx));
    return parse_device_impl(ctx, d_text, n_text, opts, dev_out, stats);
}

extern "C" int pfpb200_memcpy_d2h(pfpb200_ctx *ctx, void *dst_host, const void *src_device,
                                  uint64_t bytes) {
    if (!ctx || (bytes && (!dst_host || !src_device))) return PFPB200_E_ARG;
    if (bytes == 0) return PFPB200_OK;
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    PFP_CUDA(ctx, cudaMemcpyAsync(dst_host, src_device, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return PFPB200_OK;
}

extern "C" int pfpb200_parse_host(pfpb200_ctx *ctx, const uint8_t *text, uint64_t n_text,
                                  const pfpb200_opts *opts, pfpb200_outputs *host_out,
                                  pfpb200_stats *stats) {
    PFP_TRY(check_opts(ctx, opts));
    if (!host_out || (n_text && !text)) return pfp_fail(ctx, PFPB200_E_ARG, "null buffer");
    if (stats) memset(stats, 0, sizeof(*stats));
    memset(host_out, 0, sizeof(*host_out));
    PFP_TRY(begin_call(ctx));
    PfpEvents evs(4);
    if (!evs.ok) return pfp_fail(ctx, PFPB200_E_CUDA, "cudaEventCreate failed");
    const cudaEvent_t e0 = evs[0], e1 = evs[1], e2 = evs[2], e3 = evs[3];
    u8 *d_text = nullptr;
    PFP_TRY(pfp_alloc(ctx, (void **)&d_text, n_text, true));
    cudaEventRecord(e0, ctx->stream);
    if (n_text) PFP_CUDA(ctx, cudaMemcpyAsync(d_text, text, n_text, cudaMemcpyHostToDevice, ctx->stream));
    // the cut at the first invalid byte is found on the device, at HBM speed
    u64 n = n_text;
    if (n_text) {
        set_u64_k<<<1, 1, 0, ctx->stream>>>(&ctx->d_flags[14], n_text);
        PFP_LAUNCHED(ctx);
        first_invalid_k<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(
            d_text, n_text, reinterpret_cast<unsigned long long *>(&ctx->d_flags[14]));
        PFP_LAUNCHED(ctx);
        PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[14], &ctx->d_flags[14], sizeof(u64),
                                      cudaMemcpyDeviceToHost, ctx->stream));
    }
    cudaEventRecord(e1, ctx->stream);
    if (n_text) {
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        n = ctx->h_flags[14];
    }
    if (n < n_text && (opts->flags & PFPB200_F_VERBOSE))
        fprintf(stderr, "Invalid char found in input file: no additional chars will be read\n");
    pfpb200_outputs dv;
    memset(&dv, 0, sizeof(dv));
    ctx->early_copy = true;
    ctx->early_done = false;
    int rc = parse_device_impl(ctx, d_text, n, opts, &dv, stats);
    ctx->early_copy = false;
    if (rc != PFPB200_OK) {
        if (ctx->early_done) cudaEventSynchronize(ctx->ev_copy);
        return rc;
    }
    // device -> pinned host
    const u64 P = dv.n_phrases, d = dv.n_distinct;
    void *h_dict = nullptr, *h_occ = nullptr, *h_parse = nullptr, *h_last = nullptr, *h_sai = nullptr;
    PFP_TRY(pfp_pin(ctx, 0, &h_dict, dv.dict_bytes));
    PFP_TRY(pfp_pin(ctx, 1, &h_occ, d * 4));
    PFP_TRY(pfp_pin(ctx, 2, &h_parse, P * 4));
    PFP_TRY(pfp_pin(ctx, 3, &h_last, P));
    if (dv.sai) PFP_TRY(pfp_pin(ctx, 4, &h_sai, P * PFP_IBYTES));
    cudaEventRecord(e2, ctx->stream);
    PFP_CUDA(ctx, cudaMemcpyAsync(h_dict, dv.dict, dv.dict_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaMemcpyAsync(h_occ, dv.occ, d * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaMemcpyAsync(h_parse, dv.parse, P * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (ctx->early_done) {              // .last/.sai left on the copy stream right after K2
        PFP_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_copy, 0));
    } else {
        PFP_CUDA(ctx, cudaMemcpyAsync(h_last, dv.last, P, cudaMemcpyDeviceToHost, ctx->stream));
        if (dv.sai)
            PFP_CUDA(ctx, cudaMemcpyAsync(h_sai, dv.sai, P * PFP_IBYTES, cudaMemcpyDeviceToHost, ctx->stream));
    }
    cudaEventRecord(e3, ctx->stream);
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (stats) {
        cudaEventElapsedTime(&stats->ms_h2d, e0, e1);
        cudaEventElapsedTime(&stats->ms_d2h, e2, e3);
    }
    host_out->dict = (const u8 *)h_dict; host_out->dict_bytes = dv.dict_bytes;
    host_out->occ = (const u32 *)h_occ; host_out->n_distinct = d;
    host_out->parse = (const u32 *)h_parse; host_out->n_phrases = P;
    host_out->last = (const u8 *)h_last;
    host_out->sai = (const u8 *)h_sai;
    // the device copies are no longer needed
    pfp_release_held(ctx);
    return PFPB200_OK;
}

// the five files straight from the device outputs, D2H chunks overlapped with the writes
static int write_outputs_from_device(pfpb200_ctx *ctx, const char *path, const pfpb200_opts *o,
                                     const pfpb200_outputs &dv) {
    char name[4096];
    auto put = [&](const char *ext, int seg, const void *p, u64 bytes) -> int {
        if (seg < 0) snprintf(name, sizeof(name), "%s.%s", path, ext);              // utils.c:33-41
        else snprintf(name, sizeof(name), "%s.%d.%s", path, seg, ext);              // utils.c:44-54
        return pfp_device_to_file(ctx, name, p, bytes);
    };
    const u64 P = dv.n_phrases;
    PFP_TRY(put((o->flags & PFPB200_F_COMPRESS) ? "dicz" : "dict", -1, dv.dict, dv.dict_bytes));
    PFP_TRY(put("occ", -1, dv.occ, 4 * dv.n_distinct));
    PFP_TRY(put("parse", -1, dv.parse, 4 * P));
    const int T = o->nseg;
    if (T <= 0) {
        PFP_TRY(put("last", -1, dv.last, P));
        if (dv.sai) PFP_TRY(put("sai", -1, dv.sai, PFP_IBYTES * P));
    } else {
        // newscan.hpp:274-276: one .last/.sai segment per helper thread; bwtparse -t T reads them
        // back to back (bwtparse.c:179,195; utils.c:57-105), so any split is equivalent
        const u64 per = (P + (u64)T - 1) / (u64)T;
        for (int s = 0; s < T; s++) {
            u64 a = (u64)s * per, b = a + per;
            if (a > P) a = P;
            if (b > P) b = P;
            PFP_TRY(put("last", s, dv.last + a, b - a));
            if (dv.sai) PFP_TRY(put("sai", s, dv.sai + PFP_IBYTES * a, PFP_IBYTES * (b - a)));
        }
    }
    return PFPB200_OK;
}

// parse_host semantics for text that is already on the device: cut at the first byte <= 0x02
static int cut_and_parse_device(pfpb200_ctx *ctx, const u8 *d_text, u64 n_text, const pfpb200_opts *opts,
                                pfpb200_outputs *dv, pfpb200_stats *stats) {
    u64 n = n_text;
    if (n_text) {
        set_u64_k<<<1, 1, 0, ctx->stream>>>(&ctx->d_flags[14], n_text);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_first_invalid(ctx, d_text, n_text, &ctx->d_flags[14]));
        PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[14], &ctx->d_flags[14], sizeof(u64), cudaMemcpyDeviceToHost,
                                      ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        n = ctx->h_flags[14];
    }
    if (n < n_text) fprintf(stderr, "Invalid char found in input file: no additional chars will be read\n");
    return parse_device_impl(ctx, d_text, n, opts, dv, stats);
}

// file -> text in HBM -> the five streams in HBM; write_files: also into <path>.dict ... (parse_file)
static int parse_file_impl(pfpb200_ctx *ctx, const char *path, const pfpb200_opts *opts, pfpb200_stats *stats,
                           bool write_files, pfpb200_outputs *dv_out);

extern "C" int pfpb200_parse_file(pfpb200_ctx *ctx, const char *path, const pfpb200_opts *opts,
                                  pfpb200_stats *stats) {
    const int rc = parse_file_impl(ctx, path, opts, stats, true, nullptr);
    if (ctx && rc == PFPB200_OK) pfp_release_held(ctx);
    return rc;
}

// `bigbwt <file> -w W -p P [-f] [-S | -s -e]` in one call (bigbwt:66-150 runs newscan, bwtparse and
// pfbwt as three processes that hand each other files): the input streams into HBM, the three stages
// run there, and only <path>.bwt (and .sa / .ssa / .esa) are written -- with keep_files != 0 also the
// intermediate files the reference leaves behind with `bigbwt -k`.
extern "C" int pfpb200_bigbwt_file(pfpb200_ctx *ctx, const char *path, const pfpb200_opts *opts, uint32_t pfbwt_flags,
                                   int keep_files, pfpb200_stats *stats, pfpb200_bwtparse_result *bp_out,
                                   pfpb200_pfbwt_result *res) {
    if (!ctx || !opts || !res) return PFPB200_E_ARG;
    if (opts->flags & PFPB200_F_COMPRESS) return pfp_fail(ctx, PFPB200_E_ARG, "bigbwt: -c stops after the parse, use pfpb200_parse_file");
    pfpb200_opts o = *opts;
    o.flags |= PFPB200_F_SAI;                                  // the later stages take .sai whenever a suffix array is wanted
    o.nseg = 0;
    pfpb200_stats st;
    pfpb200_outputs dv;
    PFP_TRY(parse_file_impl(ctx, path, &o, &st, keep_files != 0, &dv));
    if (stats) *stats = st;
    const double t0 = wall_sec();
    pfpb200_bwtparse_result bp;
    PFP_TRY(pfpb200_bwtparse_device(ctx, dv.parse, dv.n_phrases, dv.last, dv.sai, &bp));
    if (bp_out) *bp_out = bp;
    PFP_TRY(pfpb200_pfbwt_device(ctx, dv.dict, dv.dict_bytes, dv.occ, dv.n_distinct, bp.ilist, bp.bwlast, bp.bwsai,
                                 bp.n_out, o.w, pfbwt_flags, res));
    char name[4096];
    auto put = [&](const char *ext, const void *p, u64 bytes) -> int {
        snprintf(name, sizeof(name), "%s.%s", path, ext);
        return pfp_device_to_file(ctx, name, p, bytes);
    };
    if (keep_files) {
        PFP_TRY(put("ilist", bp.ilist, bp.n_out * 4));
        PFP_TRY(put("bwlast", bp.bwlast, bp.n_out));
        PFP_TRY(put("bwsai", bp.bwsai, bp.n_out * PFP_IBYTES));
    }
    PFP_TRY(put("bwt", res->bwt, res->n_bwt));
    if (pfbwt_flags & PFPB200_PFBWT_SA) PFP_TRY(put("sa", res->sa, res->n_sa * PFP_IBYTES));
    if (pfbwt_flags & PFPB200_PFBWT_SSA) PFP_TRY(put("ssa", res->ssa, res->n_ssa * 2 * PFP_IBYTES));
    if (pfbwt_flags & PFPB200_PFBWT_ESA) PFP_TRY(put("esa", res->esa, res->n_esa * 2 * PFP_IBYTES));
    if (stats) stats->sec_write += (float)(wall_sec() - t0);     // (includes the two later stages: they are milliseconds to a second)
    pfp_release_scratch(ctx);
    return PFPB200_OK;
}

static int parse_file_impl(pfpb200_ctx *ctx, const char *path, const pfpb200_opts *opts, pfpb200_stats *stats,
                           bool write_files, pfpb200_outputs *dv_out) {
    PFP_TRY(check_opts(ctx, opts));
    if (!path) return pfp_fail(ctx, PFPB200_E_ARG, "null path");
    if (stats) memset(stats, 0, sizeof(*stats));
    const double t0 = wall_sec();
    const bool fasta = (opts->flags & PFPB200_F_FASTA) != 0;
    int fd = open(path, O_RDONLY);
    if (fd < 0) return pfp_fail(ctx, PFPB200_E_IO, "%s: %s", path, strerror(errno));
    struct stat sb;
    if (fstat(fd, &sb) != 0) { close(fd); return pfp_fail(ctx, PFPB200_E_IO, "%s: %s", path, strerror(errno)); }
    const u64 fsize = (u64)sb.st_size;
    bool gz = false;
    if (fasta && fsize >= 2) {       // gzip input, as the reference's gzread takes it (newscan.cpp:332-336)
        unsigned char mg[2] = {0, 0};
        if (pread(fd, mg, 2, 0) == 2) gz = mg[0] == 0x1f && mg[1] == 0x8b;
    }
    PFP_TRY(begin_call(ctx));
    pfpb200_outputs dv;
    memset(&dv, 0, sizeof(dv));
    double t1 = t0;
    int rc = PFPB200_OK;
    auto run = [&]() -> int {
        u8 *d_text = nullptr;
        u64 n_text = 0;
        bool on_device = false;
        if (!gz) {
            // the file goes to HBM through the pinned ring; it is never held in host memory
            // (scratch: the text lives until the parse is done, the raw FASTA bytes until K0 is)
            u8 *d_file = nullptr;
            PFP_TRY(pfp_alloc(ctx, (void **)&d_file, fsize + 16));
            PFP_TRY(pfp_file_to_device(ctx, fd, 0, fsize, d_file));
            if (!fasta) { d_text = d_file; n_text = fsize; on_device = true; }
            else {
                int supported = 0;
                PFP_TRY(pfp_fasta_device(ctx, d_file, fsize, &d_text, &n_text, &supported, false));    // K0
                on_device = supported != 0;
                PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
                PFP_TRY(pfp_free_now(ctx, d_file));
            }
        }
        if (!on_device) {
            // gzip, FASTQ, CRLF, ...: the host reader with all of kseq's corner cases (pfp_io.c)
            uint8_t *text = nullptr;
            uint64_t n = 0;
            int trunc = 0;
            if (pfpb200_read_input(path, opts->flags, &text, &n, &trunc) != PFPB200_OK)
                return pfp_fail(ctx, PFPB200_E_IO, "%s: cannot read", path);
            if (trunc) fprintf(stderr, "Invalid char found in input file: no additional chars will be read\n");
            int r2 = pfp_alloc(ctx, (void **)&d_text, n + 16);
            if (r2 == PFPB200_OK && n && cudaMemcpyAsync(d_text, text, n, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess)
                r2 = pfp_fail(ctx, PFPB200_E_CUDA, "host-to-device copy of the input failed");
            if (r2 == PFPB200_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess)
                r2 = pfp_fail(ctx, PFPB200_E_CUDA, "host-to-device copy of the input failed");
            pfpb200_free_host(text);
            PFP_TRY(r2);
            n_text = n;
        }
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        t1 = wall_sec();
        PFP_TRY(cut_and_parse_device(ctx, d_text, n_text, opts, &dv, stats));
        return PFPB200_OK;
    };
    rc = run();
    close(fd);
    if (rc != PFPB200_OK) { pfp_release_scratch(ctx); return rc; }
    const double t2 = wall_sec();
    if (write_files) PFP_TRY(write_outputs_from_device(ctx, path, opts, dv));
    if (stats) {
        stats->sec_read = (float)(t1 - t0);
        stats->sec_write = (float)(wall_sec() - t2);
    }
    pfp_release_scratch(ctx);
    if (dv_out) *dv_out = dv;                                  // device pointers, held by the context
    return PFPB200_OK;
}

// K0 alone, for tests and callers that hold FASTA bytes in HBM: *d_text (context-owned, valid until
// the next parse) = the text of `-f` mode; *supported = 0 when the bytes need the host reader
// (pfpb200_fasta_extract) -- FASTQ, '\r', bytes <= 0x02 / 0xFF, no '>' at offset 0.
extern "C" int pfpb200_fasta_extract_device(pfpb200_ctx *ctx, const uint8_t *d_file, uint64_t n,
                                            const uint8_t **d_text, uint64_t *n_text, int *supported) {
    if (!ctx || !d_text || !n_text || !supported || (n && !d_file)) return PFPB200_E_ARG;
    PFP_TRY(begin_call(ctx));
    u8 *out = nullptr;                 // null: an arena buffer held by the context
    int rc = pfp_fasta_device(ctx, d_file, n, &out, n_text, supported, true);
    cudaStreamSynchronize(ctx->stream);
    pfp_release_scratch(ctx);
    *d_text = out;
    return rc;
}

extern "C" int pfpb200_scan_triggers(pfpb200_ctx *ctx, const uint8_t *d_buf, uint64_t n_buf,
                                     uint64_t buf_pos0, uint64_t own_lo, uint64_t own_hi, uint32_t w,
                                     uint32_t p, const uint64_t **d_triggers, uint64_t *n_triggers,
                                     float *ms) {
    pfpb200_opts o = {w, p, 0, 0};
    PFP_TRY(check_opts(ctx, &o));
    if (!d_triggers || !n_triggers) return pfp_fail(ctx, PFPB200_E_ARG, "null output");
    PFP_TRY(begin_call(ctx));
    u64 *out = nullptr, k = 0;
    float a = 0, b = 0;
    int rc = pfp_scan_stage(ctx, d_buf, n_buf, buf_pos0, own_lo, own_hi, w, p, 0, true, &out, &k, &a, &b);
    cudaStreamSynchronize(ctx->stream);
    pfp_release_scratch(ctx);
    if (rc != PFPB200_OK) return rc;
    *d_triggers = out;
    *n_triggers = k;
    if (ms) *ms = a;
    return PFPB200_OK;
}

// ------------------------------------------------------------------------------------------------
// sharded parsing (one process per GPU drives these between its collectives)
// ------------------------------------------------------------------------------------------------
struct CallTimer {
    PfpEvents ev;
    cudaStream_t s;
    explicit CallTimer(cudaStream_t st) : ev(2), s(st) { if (ev.ok) cudaEventRecord(ev[0], s); }
    float stop() {
        float t = 0;
        if (!ev.ok) { cudaStreamSynchronize(s); return t; }
        cudaEventRecord(ev[1], s);
        cudaEventSynchronize(ev[1]);
        cudaEventElapsedTime(&t, ev[0], ev[1]);
        return t;
    }
};

// what is still in the scratch list must survive until the next parse: move it to `held`
static void promote_scratch(pfpb200_ctx *ctx) {
    for (void *p : ctx->scratch) ctx->held.push_back(p);
    ctx->scratch.clear();
}

extern "C" int pfpb200_shard_scan(pfpb200_ctx *ctx, const pfpb200_shard *shard, const pfpb200_opts *opts,
                                  uint64_t *n_triggers, uint64_t *first_trigger, uint64_t *last_trigger,
                                  float *ms) {
    PFP_TRY(check_opts(ctx, opts));
    if (!shard || !n_triggers || !first_trigger || !last_trigger) return pfp_fail(ctx, PFPB200_E_ARG, "null argument");
    if (shard->own_lo > shard->own_hi || shard->own_hi > shard->n_global)
        return pfp_fail(ctx, PFPB200_E_ARG, "bad shard range");
    PFP_TRY(begin_call(ctx));
    ctx->sh.desc = *shard;
    ctx->sh.opts = *opts;
    ctx->sh.route_perm = nullptr;
    ctx->sh.route_ooff = nullptr;
    CallTimer tm(ctx->stream);
    u64 *ends = nullptr, k = 0;
    float a = 0;
    ScanBits sb;
    int rc = pfp_scan_bits(ctx, shard->d_buf, shard->n_buf, shard->buf_pos0, shard->own_lo, shard->own_hi,
                           opts->w, opts->p, true, &sb, &a);
    if (rc == PFPB200_OK) {
        k = sb.total;
        rc = pfp_alloc_t(ctx, &ends, k + 1, true);
    }
    // the streaming K2 pass of shard_words writes the positions itself; the seams only need the
    // first and the last trigger now
    const bool stream_k2 = rc == PFPB200_OK && pfp_stream_ok(sb, opts->w) && !ctx->legacy_k2;
    ctx->sh.ends_emitted = !stream_k2;
    if (rc == PFPB200_OK && !stream_k2) rc = pfp_scan_emit(ctx, sb, ends);
    ctx->sh.bits = sb;
    if (rc == PFPB200_OK && k > 0) {
        if (stream_k2) {
            rc = pfp_scan_first_last(ctx, sb, &ctx->d_flags[8]);
            cudaMemcpyAsync(&ctx->h_flags[8], &ctx->d_flags[8], 2 * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream);
        } else {
            cudaMemcpyAsync(&ctx->h_flags[8], ends, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream);
            cudaMemcpyAsync(&ctx->h_flags[9], ends + (k - 1), sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream);
        }
    }
    float t = tm.stop();
    pfp_release_scratch(ctx);
    if (rc != PFPB200_OK) return rc;
    PFP_CUDA(ctx, cudaGetLastError());
    ctx->sh.ends = ends;
    ctx->sh.n_trig = k;
    *n_triggers = k;
    *first_trigger = k ? ctx->h_flags[8] : 0;
    *last_trigger = k ? ctx->h_flags[9] : 0;
    if (ms) *ms = t;
    return PFPB200_OK;
}

extern "C" int pfpb200_shard_words(pfpb200_ctx *ctx, int64_t first_start, pfpb200_words *out, float *ms) {
    if (!ctx || !out) return PFPB200_E_ARG;
    memset(out, 0, sizeof(*out));
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    const pfpb200_shard &sh = ctx->sh.desc;
    const pfpb200_opts &o = ctx->sh.opts;
    const u32 w = o.w;
    const u64 k = ctx->sh.n_trig;
    const u64 P = k + (sh.is_last ? 1 : 0);
    ctx->sh.P = P;
    ctx->sh.d = 0;
    ctx->sh.uid = nullptr;
    if (ms) *ms = 0;
    if (P == 0) return PFPB200_OK;
    if (P >= 0xFFFFFFFFull) return pfp_fail(ctx, PFPB200_E_LIMIT, "the shard's parse has more than 2^32-2 words");
    CallTimer tm(ctx->stream);
    auto run = [&]() -> int {
        u64 *ends = ctx->sh.ends;
        if (sh.is_last) {
            set_u64_k<<<1, 1, 0, ctx->stream>>>(ends + k, sh.n_global + w - 1);
            PFP_LAUNCHED(ctx);
        }
        PhraseArrays ph{};
        ph.ends = ends;
        PFP_TRY(pfp_alloc_t(ctx, &ph.rec, P));
        PFP_TRY(pfp_alloc_t(ctx, &ph.last, P, true));
        if (o.flags & PFPB200_F_SAI) PFP_TRY(pfp_alloc_t(ctx, &ph.sai, P * PFP_IBYTES, true));
        TextView tv{sh.d_buf, sh.n_buf, (i64)sh.buf_pos0, (i64)sh.n_global};
        DictArrays D;
        if (pfp_stream_ok(ctx->sh.bits, w) && !ctx->legacy_k2)
            PFP_TRY(pfp_stream_stage(ctx, ctx->sh.bits, tv, ph, P, first_start, w, !ctx->sh.ends_emitted));
        else PFP_TRY(pfp_hash_stage(ctx, tv, ph, P, first_start, w));
        PFP_TRY(pfp_dedup_stage(ctx, ph, P, first_start, w, &D));
        PFP_TRY(pfp_uid_words(ctx, &D, P));
        u64 *wfpa = nullptr, *wfpb = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &wfpa, D.d));
        PFP_TRY(pfp_alloc_t(ctx, &wfpb, D.d));
        PFP_TRY(pfp_gather_word_fp(ctx, D, ph, wfpa, wfpb));
        PFP_TRY(pfp_free_now(ctx, ph.rec));
        PFP_TRY(pfp_pool_stage(ctx, tv, &D));
        PFP_TRY(pfp_free_now(ctx, D.rep));
        if (o.flags & PFPB200_F_VERIFY) PFP_TRY(pfp_verify_stage(ctx, tv, ends, first_start, w, P, D));
        PFP_CUDA(ctx, cudaMemcpyAsync(ctx->h_flags, ctx->d_flags, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        PFP_CUDA(ctx, cudaGetLastError());
        if (ctx->h_flags[0] & PFP_ERRBIT_COLLISION)
            return pfp_fail(ctx, PFPB200_E_COLLISION, "two different phrases share a fingerprint (found by the verify pass)");
        ctx->sh.d = D.d;
        ctx->sh.uid = D.uid;
        ctx->sh.wfpa = wfpa; ctx->sh.wfpb = wfpb; ctx->sh.pool = D.pool; ctx->sh.uoff = D.uoff;
        ctx->sh.pool_words = D.pool_words;
        ctx->sh.ulen = D.ulen; ctx->sh.count = D.count; ctx->sh.uwords = D.uwords;
        out->n_words = D.d; out->n_phrases = P; out->pool_words = D.pool_words;
        out->fpa = wfpa; out->fpb = wfpb; out->len = D.ulen; out->count = D.count;
        out->uwords = D.uwords; out->pool = D.pool; out->last = ph.last; out->sai = ph.sai;
        return PFPB200_OK;
    };
    int rc = run();
    float t = tm.stop();
    if (rc != PFPB200_OK) { pfp_release_scratch(ctx); return rc; }
    promote_scratch(ctx);
    if (ms) *ms = t;
    return PFPB200_OK;
}

extern "C" int pfpb200_dict_merge(pfpb200_ctx *ctx, uint64_t n_in, const uint64_t *fpa, const uint64_t *fpb,
                                  const uint32_t *len, const uint32_t *count, const uint32_t *uwords,
                                  const uint64_t *pool, uint64_t pool_words, uint32_t w, uint32_t flags,
                                  pfpb200_merged *out, float *ms) {
    if (!ctx || !out) return PFPB200_E_ARG;
    memset(out, 0, sizeof(*out));
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    PFP_CUDA(ctx, cudaMemsetAsync(ctx->d_flags, 0, PFP_FLAG_SLOTS * sizeof(u64), ctx->stream));
    CallTimer tm(ctx->stream);
    auto run = [&]() -> int {
        if (n_in == 0) {
            u8 *dict = nullptr;
            PFP_TRY(pfp_alloc_t(ctx, &dict, 1, true));
            PFP_CUDA(ctx, cudaMemsetAsync(dict, 0, 1, ctx->stream));
            out->dict = dict; out->dict_bytes = 1;
            return PFPB200_OK;
        }
        DictArrays D;
        u32 *uid_of_entry = nullptr;
        StageTimer tm;
        const bool trace = getenv("PFPB200_TRACE") != nullptr && tm.init() == 0;
        if (trace) tm.mark(ctx->stream);
        PFP_TRY(pfp_merge_stage(ctx, n_in, fpa, fpb, len, count, uwords, pool, pool_words,
                                (flags & PFPB200_F_VERIFY) != 0, &D, &uid_of_entry));
        if (trace) tm.mark(ctx->stream);
        u32 *order = nullptr, rounds = 0;
        PFP_TRY(pfp_rank_stage(ctx, D, &order, &rounds));
        if (trace) tm.mark(ctx->stream);
        u8 *dict = nullptr;
        u32 *occ = nullptr, *rank_of_uid = nullptr, *rank_of_entry = nullptr;
        u64 dict_bytes = 0;
        PFP_TRY(pfp_dict_stage(ctx, D, order, (flags & PFPB200_F_COMPRESS) ? w : 0, &dict, &dict_bytes, &occ,
                               &rank_of_uid));
        PFP_TRY(pfp_alloc_t(ctx, &rank_of_entry, n_in, true));
        PFP_TRY(pfp_remap_stage(ctx, uid_of_entry, rank_of_uid, n_in, rank_of_entry));
        if (trace) tm.mark(ctx->stream);
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        PFP_CUDA(ctx, cudaGetLastError());
        if (trace) {
            fprintf(stderr, "[pfpb200 merge] n_in %llu -> d %llu: dedup %.3f ms, rank %.3f ms (%u rounds), dict+remap %.3f ms\n",
                    (unsigned long long)n_in, (unsigned long long)D.d, tm.ms(0, 1), tm.ms(1, 2), rounds, tm.ms(2, 3));
        }
        out->n_distinct = D.d; out->dict_bytes = dict_bytes; out->sum_word_len = D.sum_len;
        out->dict = dict; out->occ = occ; out->rank_of_entry = rank_of_entry;
        return PFPB200_OK;
    };
    int rc = run();
    float t = tm.stop();
    pfp_release_scratch(ctx);
    if (ms) *ms = t;
    return rc;
}

extern "C" int pfp_unpack_words(pfpb200_ctx *ctx, const pfpb200_word *in, u64 n, u64 *fpa, u64 *fpb,
                                u32 *len, u32 *count, u32 *uwords);

// The merge of received words in two halves, so that the exchange of the pool BYTES can overlap the
// dedup, which only needs the 32-byte word records: _begin dedups (table, counts, representative
// entry of every word), _finish ranks the distinct words and writes .dict/.occ once the bytes are there.
extern "C" int pfpb200_dict_merge_begin(pfpb200_ctx *ctx, uint64_t n_in, const pfpb200_word *words, float *ms) {
    if (!ctx || (n_in && !words)) return PFPB200_E_ARG;
    if (ms) *ms = 0;
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    PFP_CUDA(ctx, cudaMemsetAsync(ctx->d_flags, 0, PFP_FLAG_SLOTS * sizeof(u64), ctx->stream));
    ctx->mg.n_in = n_in;
    ctx->mg.d = 0;
    if (n_in == 0) return PFPB200_OK;
    CallTimer tm(ctx->stream);
    auto run = [&]() -> int {
        u64 *fpa = nullptr, *fpb = nullptr;
        u32 *len = nullptr, *count = nullptr, *uwords = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &fpa, n_in));
        PFP_TRY(pfp_alloc_t(ctx, &fpb, n_in));
        PFP_TRY(pfp_alloc_t(ctx, &len, n_in));
        PFP_TRY(pfp_alloc_t(ctx, &count, n_in));
        PFP_TRY(pfp_alloc_t(ctx, &uwords, n_in));
        PFP_TRY(pfp_unpack_words(ctx, words, n_in, fpa, fpb, len, count, uwords));
        DictArrays D;
        u32 *uid_of_entry = nullptr;
        PFP_TRY(pfp_merge_stage(ctx, n_in, fpa, fpb, len, count, uwords, nullptr, 0, false, &D, &uid_of_entry));
        PFP_TRY(pfp_free_now(ctx, fpa));
        PFP_TRY(pfp_free_now(ctx, fpb));
        PFP_TRY(pfp_free_now(ctx, count));
        ctx->mg.d = D.d; ctx->mg.sum_len = D.sum_len; ctx->mg.max_len = D.max_len;
        ctx->mg.uid_of_entry = uid_of_entry; ctx->mg.rep = D.rep; ctx->mg.count = D.count;
        ctx->mg.ulen = D.ulen; ctx->mg.uwords = D.uwords; ctx->mg.uoff = D.uoff;
        ctx->mg.len_in = len; ctx->mg.uwords_in = uwords;
        return PFPB200_OK;
    };
    int rc = run();
    float t = tm.stop();
    if (rc != PFPB200_OK) { pfp_release_scratch(ctx); ctx->mg.n_in = 0; return rc; }
    promote_scratch(ctx);                 // the dictionary arrays live until _finish (and the next parse)
    if (ms) *ms = t;
    return PFPB200_OK;
}

extern "C" int pfpb200_dict_merge_finish(pfpb200_ctx *ctx, const uint64_t *pool, uint64_t pool_words, uint32_t w,
                                         uint32_t flags, pfpb200_merged *out, float *ms) {
    if (!ctx || !out) return PFPB200_E_ARG;
    memset(out, 0, sizeof(*out));
    if (ms) *ms = 0;
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    CallTimer tm(ctx->stream);
    const u64 n_in = ctx->mg.n_in;
    auto run = [&]() -> int {
        if (n_in == 0) {
            u8 *dict = nullptr;
            PFP_TRY(pfp_alloc_t(ctx, &dict, 1, true));
            PFP_CUDA(ctx, cudaMemsetAsync(dict, 0, 1, ctx->stream));
            out->dict = dict; out->dict_bytes = 1;
            return PFPB200_OK;
        }
        if (!pool) return pfp_fail(ctx, PFPB200_E_ARG, "dict_merge_finish: null pool");
        DictArrays D;
        D.d = ctx->mg.d; D.sum_len = ctx->mg.sum_len; D.max_len = ctx->mg.max_len;
        D.uid = ctx->mg.uid_of_entry; D.rep = ctx->mg.rep; D.count = ctx->mg.count; D.ulen = ctx->mg.ulen;
        D.uwords = ctx->mg.uwords; D.uoff = ctx->mg.uoff;
        D.pool = const_cast<u64 *>(pool); D.pool_words = pool_words;
        if (flags & PFPB200_F_VERIFY)
            PFP_TRY(pfp_merge_verify(ctx, n_in, ctx->mg.uid_of_entry, D.rep, ctx->mg.len_in, ctx->mg.uwords_in, pool));
        u32 *order = nullptr, rounds = 0;
        PFP_TRY(pfp_rank_stage(ctx, D, &order, &rounds));
        u8 *dict = nullptr;
        u32 *occ = nullptr, *rank_of_uid = nullptr, *rank_of_entry = nullptr;
        u64 dict_bytes = 0;
        PFP_TRY(pfp_alloc_t(ctx, &rank_of_entry, n_in, true));
        PFP_TRY(pfp_dict_stage(ctx, D, order, (flags & PFPB200_F_COMPRESS) ? w : 0, &dict, &dict_bytes, &occ,
                               &rank_of_uid, ctx->mg.uid_of_entry, n_in, rank_of_entry));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        PFP_CUDA(ctx, cudaGetLastError());
        out->n_distinct = D.d; out->dict_bytes = dict_bytes; out->sum_word_len = D.sum_len;
        out->dict = dict; out->occ = occ; out->rank_of_entry = rank_of_entry;
        return PFPB200_OK;
    };
    int rc = run();
    float t = tm.stop();
    pfp_release_scratch(ctx);
    ctx->mg.n_in = 0;
    if (ms) *ms = t;
    return rc;
}

extern "C" int pfpb200_dict_merge_words(pfpb200_ctx *ctx, uint64_t n_in, const pfpb200_word *words,
                                        const uint64_t *pool, uint64_t pool_words, uint32_t w,
                                        uint32_t flags, pfpb200_merged *out, float *ms) {
    if (!ctx || !out || (n_in && !words)) return PFPB200_E_ARG;
    float a = 0, b = 0;
    PFP_TRY(pfpb200_dict_merge_begin(ctx, n_in, words, &a));
    int rc = pfpb200_dict_merge_finish(ctx, pool, pool_words, w, flags, out, &b);
    if (ms) *ms = a + b;
    return rc;
}

extern "C" int pfpb200_shard_remap(pfpb200_ctx *ctx, const uint32_t *d_rank_of_word, const uint32_t **d_parse,
                                   float *ms) {
    if (!ctx || !d_parse) return PFPB200_E_ARG;
    *d_parse = nullptr;
    if (ms) *ms = 0;
    const u64 P = ctx->sh.P;
    if (P == 0) return PFPB200_OK;
    if (!d_rank_of_word || !ctx->sh.uid) return pfp_fail(ctx, PFPB200_E_ARG, "shard_remap before shard_words");
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    CallTimer tm(ctx->stream);
    u32 *parse = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &parse, P, true));
    PFP_TRY(pfp_remap_stage(ctx, ctx->sh.uid, d_rank_of_word, P, parse));
    float t = tm.stop();
    PFP_CUDA(ctx, cudaGetLastError());
    *d_parse = parse;
    if (ms) *ms = t;
    return PFPB200_OK;
}

// ---- routing of a shard's words to the owners of their lexicographic range -----------------------
struct Splitters { u64 s[PFPB200_MAX_RANKS]; u32 n; };

extern "C" int pfp_route_impl(pfpb200_ctx *ctx, const Splitters &sp, u32 n_ranks, pfpb200_routed *out);
extern "C" int pfp_first_keys_impl(pfpb200_ctx *ctx, u64 **keys);

extern "C" int pfpb200_shard_first_keys(pfpb200_ctx *ctx, const uint64_t **d_keys) {
    if (!ctx || !d_keys) return PFPB200_E_ARG;
    *d_keys = nullptr;
    if (ctx->sh.d == 0) return PFPB200_OK;
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    u64 *keys = nullptr;
    int rc = pfp_first_keys_impl(ctx, &keys);
    if (rc != PFPB200_OK) return rc;
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *d_keys = keys;
    return PFPB200_OK;
}

extern "C" int pfpb200_shard_route(pfpb200_ctx *ctx, const uint64_t *splitters, uint32_t n_ranks,
                                   pfpb200_routed *out, float *ms) {
    if (!ctx || !out || n_ranks < 1 || n_ranks > PFPB200_MAX_RANKS || (n_ranks > 1 && !splitters))
        return PFPB200_E_ARG;
    memset(out, 0, sizeof(*out));
    if (ms) *ms = 0;
    if (ctx->sh.d == 0) return PFPB200_OK;
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    Splitters sp;
    sp.n = n_ranks - 1;
    for (u32 i = 0; i < sp.n; i++) {
        sp.s[i] = splitters[i];
        if (i && sp.s[i] < sp.s[i - 1]) return pfp_fail(ctx, PFPB200_E_ARG, "splitters not ascending");
    }
    CallTimer tm(ctx->stream);
    int rc = pfp_route_impl(ctx, sp, n_ranks, out);
    float t = tm.stop();
    if (rc != PFPB200_OK) { pfp_release_scratch(ctx); return rc; }
    promote_scratch(ctx);
    if (ms) *ms = t;
    return PFPB200_OK;
}

// ---- routing fused with the exchange (peer memory) -------------------------------------------------
extern "C" int pfp_route_plan_impl(pfpb200_ctx *ctx, const Splitters &sp, u32 n_ranks, u64 *words_to, u64 *pool_to,
                                   const u32 **perm_out);
extern "C" int pfp_route_push_impl(pfpb200_ctx *ctx, u32 n_ranks, const u64 *word_dst, const u64 *pool_dst);

extern "C" int pfpb200_shard_route_plan(pfpb200_ctx *ctx, const uint64_t *splitters, uint32_t n_ranks,
                                        uint64_t *words_to, uint64_t *pool_to, const uint32_t **d_perm,
                                        float *ms) {
    if (!ctx || !words_to || !pool_to || !d_perm || n_ranks < 1 || n_ranks > PFPB200_MAX_RANKS ||
        (n_ranks > 1 && !splitters))
        return PFPB200_E_ARG;
    for (u32 q = 0; q < PFPB200_MAX_RANKS; q++) words_to[q] = pool_to[q] = 0;
    *d_perm = nullptr;
    if (ms) *ms = 0;
    if (ctx->sh.d == 0) return PFPB200_OK;
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    Splitters sp;
    sp.n = n_ranks - 1;
    for (u32 i = 0; i < sp.n; i++) {
        sp.s[i] = splitters[i];
        if (i && sp.s[i] < sp.s[i - 1]) return pfp_fail(ctx, PFPB200_E_ARG, "splitters not ascending");
    }
    CallTimer tm(ctx->stream);
    int rc = pfp_route_plan_impl(ctx, sp, n_ranks, words_to, pool_to, d_perm);
    float t = tm.stop();
    if (rc != PFPB200_OK) { pfp_release_scratch(ctx); return rc; }
    promote_scratch(ctx);
    if (ms) *ms = t;
    return PFPB200_OK;
}

extern "C" int pfpb200_shard_route_push(pfpb200_ctx *ctx, uint32_t n_ranks, const uint64_t *word_dst,
                                        const uint64_t *pool_dst, float *ms) {
    if (!ctx || !word_dst || !pool_dst || n_ranks < 1 || n_ranks > PFPB200_MAX_RANKS) return PFPB200_E_ARG;
    if (ms) *ms = 0;
    if (ctx->sh.d == 0) return PFPB200_OK;
    if (!ctx->sh.route_perm) return pfp_fail(ctx, PFPB200_E_ARG, "shard_route_push before shard_route_plan");
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    CallTimer tm(ctx->stream);
    int rc = pfp_route_push_impl(ctx, n_ranks, word_dst, pool_dst);
    float t = tm.stop();
    if (ms) *ms = t;
    return rc;
}
