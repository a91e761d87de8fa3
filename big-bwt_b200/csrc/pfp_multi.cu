// pfp_multi.cu -- several GPUs of one box behind ONE call of the C ABI (pfpb200_multi_*).
//
// Reference analogue: `newscan.x -t T` / `pscan.x -t T` -- one process, T helper threads, each
// parsing a contiguous range of the input and re-synchronising at the seams (newscan.hpp:230-337,
// pscan.hpp:44-165), a shared dictionary behind mutexes (newscan.cpp:252-294, pscan.cpp:137-205),
// complete outputs when the call returns.  Here: one host thread per GPU, each driving the
// stage-level entry points (pfpb200_shard_*) on its own context and stream;
//   * the text is cut into contiguous shards, every rank copies its shard (and up to 1 MB in
//     front of it: window halo + the head of the phrase straddling the seam) from the host text;
//   * the small "collectives" (trigger counts, splitter samples, the count matrix, dictionary
//     sizes) are host arrays published between thread barriers -- the ranks live in one address
//     space, so there is nothing to send;
//   * the dictionary exchange is the range-partitioned merge of big-bwt_b200/shards.py: words are
//     routed to the rank owning their lexicographic range and travel as ONE peer-to-peer DMA per
//     (source, owner, buffer) straight into the owner's receive buffer over NVLink
//     (cudaMemcpyPeerAsync; cudaDeviceEnablePeerAccess makes it a direct copy), ordered by CUDA
//     events across the devices; the ranks inside each range travel back the same way;
//   * every rank writes its pieces of the five output streams into one set of pinned host
//     buffers at the offsets the all-gathered sizes give.
// `gpuscan.x -g 0,1,2,3 file ...` is the command-line face (bigbwt needs no Python / torch).
// The same device may be listed several times (shards time-share it): that is how the
// single-GPU test box exercises this file.
#include "pfp_common.cuh"
#include "pfp_stages.cuh"
#include <errno.h>
#include <fcntl.h>
#include <stdlib.h>
#include <sys/stat.h>
#include <unistd.h>
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <time.h>

extern "C" {
int pfp_io_write_outputs(const char *path, const pfpb200_opts *opts, const pfpb200_outputs *o, char *err,
                         size_t errlen);
}

namespace {

constexpr u64 MULTI_FRONT = 1u << 20;     // bytes kept in front of a shard (grown on demand)
constexpr u32 MULTI_SAMPLE = 1024;        // first keys sampled per rank for the range splitters
constexpr u64 MULTI_MIN_SHARD = 1u << 16; // shorter texts use fewer shards

enum Phase { PH_START = 0, PH_H2D, PH_SCAN, PH_SEAMS, PH_WORDS, PH_SPLIT, PH_ROUTE, PH_EXCHANGE, PH_MERGE,
             PH_BACK, PH_REMAP, PH_D2H, PH_COUNT };
static_assert(PH_COUNT == PFPB200_N_PHASES, "phase table and header disagree");

struct Barrier {
    std::mutex mu;
    std::condition_variable cv;
    int n = 1, count = 0;
    unsigned gen = 0;
    u64 acc = 0, result = 0;
    int fails = 0, fails_result = 0;
    void wait() {
        std::unique_lock<std::mutex> l(mu);
        const unsigned g = gen;
        if (++count == n) { count = 0; gen++; cv.notify_all(); }
        else cv.wait(l, [&] { return gen != g; });
    }
    // a barrier that returns the sum of what every thread brought and whether any thread brought a
    // failure: the same values for all of them
    u64 sum(u64 v, bool failed, bool *any_failed) {
        std::unique_lock<std::mutex> l(mu);
        const unsigned g = gen;
        acc += v;
        fails += failed ? 1 : 0;
        if (++count == n) {
            result = acc; fails_result = fails;
            acc = 0; fails = 0; count = 0; gen++;
            cv.notify_all();
        } else cv.wait(l, [&] { return gen != g; });
        *any_failed = fails_result != 0;
        return result;
    }
};

struct Rank {
    pfpb200_ctx *ctx = nullptr;
    int device = 0;
    // [front | shard] on the device
    u8 *buf = nullptr;
    size_t buf_cap = 0;
    u64 front = 0, pos0 = 0, n_local = 0;
    bool is_last = false;
    // receive buffers of the exchange (written by the peers)
    pfpb200_word *rx_words = nullptr; size_t rx_words_cap = 0;
    u64 *rx_pool = nullptr; size_t rx_pool_cap = 0;
    u32 *rx_ranks = nullptr; size_t rx_ranks_cap = 0;
    cudaEvent_t ev_sent = nullptr, ev_back = nullptr, ev_routed = nullptr, ev_pool = nullptr;
    cudaStream_t side = nullptr;          // the pool bytes travel here while the owners dedup the word records
    cudaEvent_t ev_phase[PH_COUNT] = {nullptr};
    u64 *d_small = nullptr, *h_small = nullptr;   // 16 u64 of device / pinned scratch
    u64 *h_sample = nullptr;              // pinned, MULTI_SAMPLE keys
    // published per parse (read by the other ranks between barriers)
    u64 first_bad = ~0ull;
    u64 n_trig = 0, last_trig = 0;
    u32 n_sample = 0;
    u64 words_to[PFPB200_MAX_RANKS] = {0}, pool_to[PFPB200_MAX_RANKS] = {0};
    u64 n_words = 0, n_phrases = 0, n_distinct = 0, piece_bytes = 0, sum_word_len = 0;
    pfpb200_words wd;
    pfpb200_routed rt;
    pfpb200_merged mg;
    const u32 *d_parse = nullptr;
    float ms_phase[PH_COUNT] = {0};
    u32 launches = 0;
    // the sharded pfbwt (pfpb200_multi_pfbwt_file); published fields are read by the peers between barriers
    PmState pb;
    const void *pb_in[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // .dict .occ .ilist .bwlast .bwsai
    u64 pb_n[5] = {0, 0, 0, 0, 0};
    u64 *pb_rank = nullptr;               // my block of the rank array
    pfpb200_pfbwt_rank pb_stat;
    u32 pb_rounds = 0;
    u64 pb_windows = 0, pb_ssa = 0, pb_esa = 0;   // output windows, run samples after the stitching
};

}  // namespace

struct pfpb200_multi {
    int n = 0;
    std::vector<Rank> r;
    Barrier bar;
    std::atomic<int> failed{0};
    std::mutex err_mu;
    char err[512] = {0};
    char io_err[512] = {0};
    // the current job: where the text comes from
    //   text     : host memory (pfpb200_multi_parse_host)
    //   src_fd   : a plain-text file, every rank reads its own range through its pinned ring
    //   src_dev  : device memory of rank 0 (the FASTA file after K0), shards travel peer to peer
    const u8 *text = nullptr;
    int src_fd = -1;
    const u8 *src_dev = nullptr;
    const char *out_path = nullptr;       // non-null: every rank writes its pieces straight into the five files
    u64 n_text = 0, n_eff = 0;
    int n_active = 0;                     // shards in use (short texts use fewer)
    pfpb200_opts opts{};
    // host outputs (pinned, kept and grown across calls)
    void *pin[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    size_t pin_cap[5] = {0, 0, 0, 0, 0};
    u64 tot_phrases = 0, tot_distinct = 0, tot_dict = 0, tot_sum_len = 0;
    double sec_wall = 0;
    // PFPB200_MULTI_MIN_SHARD / PFPB200_MULTI_FRONT (tests): seams and front growth on small inputs
    u64 min_shard = MULTI_MIN_SHARD, front_cap = MULTI_FRONT;
    // the current pfbwt job; PFPB200_MULTI_SPLIT_KEY=1 (tests): the two-sort key form of the
    // sharded suffix sort even where one 64-bit key would do
    const char *pb_base = nullptr;
    u32 pb_w = 0, pb_flags = 0;
    bool split_key = false;
};

namespace {

double wall_sec() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

void multi_fail(pfpb200_multi *m, int g, int code, const char *what) {
    int expect = 0;
    if (m->failed.compare_exchange_strong(expect, code)) {
        std::lock_guard<std::mutex> l(m->err_mu);
        snprintf(m->err, sizeof(m->err), "rank %d (device %d): %s", g, m->r[g].device, what ? what : "");
    }
}

#define MR_CUDA(call)                                                                           \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            char b_[256];                                                                       \
            snprintf(b_, sizeof(b_), "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            multi_fail(m, g, e_ == cudaErrorMemoryAllocation ? PFPB200_E_NOMEM : PFPB200_E_CUDA, b_);    \
            return;                                                                             \
        }                                                                                       \
    } while (0)

#define MR_LIB(call)                                                                            \
    do {                                                                                        \
        int rc_ = (call);                                                                       \
        if (rc_ != PFPB200_OK) { multi_fail(m, g, rc_, pfpb200_last_error(R.ctx)); return; }    \
    } while (0)

// even shards over [0, n); texts shorter than n_ranks * MULTI_MIN_SHARD use fewer of them, the
// ranks behind get an empty shard at the end of the text
void plan_shards(pfpb200_multi *m, u64 n) {
    const int G = m->n;
    int act = (int)std::min<u64>((u64)G, std::max<u64>(1, n / m->min_shard));
    m->n_active = act;
    m->n_eff = n;
    for (int g = 0; g < G; g++) {
        Rank &R = m->r[g];
        const u64 lo = g < act ? n / (u64)act * (u64)g : n;
        const u64 hi = g + 1 < act ? n / (u64)act * (u64)(g + 1) : n;
        R.pos0 = lo;
        R.n_local = hi - lo;
        R.is_last = g == act - 1;
        // at least w bytes: w-1 for the window ending at the shard's first position, 1 for its `.last`
        R.front = std::min<u64>(std::max<u64>(m->front_cap, (u64)m->opts.w + 64), lo);
    }
}

// global start of the first phrase ending in shard g (previous trigger - w + 1), -1: text start
i64 first_phrase_start(const pfpb200_multi *m, int g, u32 w) {
    for (int q = g - 1; q >= 0; q--)
        if (m->r[q].n_trig > 0) return (i64)m->r[q].last_trig - (i64)w + 1;
    return -1;
}

// ---- files written by all ranks side by side -------------------------------------------------------------
void stream_name(char *name, size_t cap, const char *path, const char *ext, int seg) {
    if (seg < 0) snprintf(name, cap, "%s.%s", path, ext);                  // utils.c:33-41
    else snprintf(name, cap, "%s.%d.%s", path, seg, ext);                  // utils.c:44-54
}

// phrases [a, b) of segment s when the P phrases are cut into T segments (newscan.hpp:274-276)
void segment_range(u64 P, int T, int s, u64 *a, u64 *b) {
    const u64 per = (P + (u64)T - 1) / (u64)T;
    *a = std::min(P, (u64)s * per);
    *b = std::min(P, *a + per);
}

int create_sized(pfpb200_multi *m, const char *name, u64 bytes) {
    int fd = open(name, O_WRONLY | O_CREAT | O_TRUNC, 0666);
    if (fd < 0 || ftruncate(fd, (off_t)bytes) != 0 || close(fd) != 0) {
        snprintf(m->io_err, sizeof(m->io_err), "%.400s: %s", name, strerror(errno));
        return -1;
    }
    return 0;
}

int multi_create_files(pfpb200_multi *m, u64 dict_bytes, u64 d, u64 P) {
    char name[4096];
    const pfpb200_opts &o = m->opts;
    stream_name(name, sizeof(name), m->out_path, (o.flags & PFPB200_F_COMPRESS) ? "dicz" : "dict", -1);
    if (create_sized(m, name, dict_bytes)) return -1;
    stream_name(name, sizeof(name), m->out_path, "occ", -1);
    if (create_sized(m, name, 4 * d)) return -1;
    stream_name(name, sizeof(name), m->out_path, "parse", -1);
    if (create_sized(m, name, 4 * P)) return -1;
    const int T = o.nseg;
    for (int s = (T > 0 ? 0 : -1); s < (T > 0 ? T : 0); s++) {
        u64 a = 0, b = P;
        if (T > 0) segment_range(P, T, s, &a, &b);
        stream_name(name, sizeof(name), m->out_path, "last", s);
        if (create_sized(m, name, b - a)) return -1;
        if (o.flags & PFPB200_F_SAI) {
            stream_name(name, sizeof(name), m->out_path, "sai", s);
            if (create_sized(m, name, PFP_IBYTES * (b - a))) return -1;
        }
    }
    return 0;
}

// device bytes -> [file_off, +bytes) of the named (existing) file
int piece_to_file(Rank &R, const char *name, u64 file_off, const void *d_src, u64 bytes) {
    if (bytes == 0) return PFPB200_OK;
    int fd = open(name, O_WRONLY);
    if (fd < 0) return pfp_fail(R.ctx, PFPB200_E_IO, "%s: %s", name, strerror(errno));
    int rc = pfp_device_to_fd(R.ctx, fd, file_off, d_src, bytes, name);
    if (close(fd) != 0 && rc == PFPB200_OK) rc = pfp_fail(R.ctx, PFPB200_E_IO, "%s: write error", name);
    return rc;
}

// this rank's pieces of the five streams into the files rank 0 created
int multi_write_pieces(pfpb200_multi *m, Rank &R, u64 off_dict, u64 off_d, u64 off_P) {
    char name[4096];
    const pfpb200_opts &o = m->opts;
    stream_name(name, sizeof(name), m->out_path, (o.flags & PFPB200_F_COMPRESS) ? "dicz" : "dict", -1);
    PFP_TRY(piece_to_file(R, name, off_dict, R.mg.dict, R.piece_bytes));
    stream_name(name, sizeof(name), m->out_path, "occ", -1);
    PFP_TRY(piece_to_file(R, name, 4 * off_d, R.mg.occ, 4 * R.n_distinct));
    stream_name(name, sizeof(name), m->out_path, "parse", -1);
    PFP_TRY(piece_to_file(R, name, 4 * off_P, R.d_parse, 4 * R.n_phrases));
    const int T = o.nseg;
    const u64 P = m->tot_phrases, lo = off_P, hi = off_P + R.n_phrases;
    for (int s = (T > 0 ? 0 : -1); s < (T > 0 ? T : 0); s++) {
        u64 a = 0, b = P;
        if (T > 0) segment_range(P, T, s, &a, &b);
        const u64 x = std::max(a, lo), y = std::min(b, hi);               // my phrases inside this segment
        if (x >= y) continue;
        stream_name(name, sizeof(name), m->out_path, "last", s);
        PFP_TRY(piece_to_file(R, name, x - a, R.wd.last + (x - lo), y - x));
        if (R.wd.sai) {
            stream_name(name, sizeof(name), m->out_path, "sai", s);
            PFP_TRY(piece_to_file(R, name, PFP_IBYTES * (x - a), R.wd.sai + PFP_IBYTES * (x - lo), PFP_IBYTES * (y - x)));
        }
    }
    return PFPB200_OK;
}

template <typename T>
bool ensure_dev(T **p, size_t *cap, size_t count) {
    if (count <= *cap && *p) return true;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    const size_t want = count + count / 4 + 1024;
    if (cudaMalloc((void **)p, want * sizeof(T)) != cudaSuccess) { cudaGetLastError(); return false; }
    *cap = want;
    return true;
}

void mark(Rank &R, int ph) { cudaEventRecord(R.ev_phase[ph], R.ctx->stream); }

// one rank's part of one parse; every rank passes the same barriers whatever happens
void rank_main(pfpb200_multi *m, int g) {
    Rank &R = m->r[g];
    const int G = m->n;
    const u32 w = m->opts.w;
    cudaStream_t st = R.ctx->stream;
    auto ok = [&]() { return m->failed.load(std::memory_order_relaxed) == 0; };
    cudaSetDevice(R.device);
    mark(R, PH_START);

    // ---- 1. shard (+front) to the device; first invalid byte of the shard ---------------------------
    auto upload = [&]() {
        // the working set of a shard (trigger bits, positions, records, table, pool, sort buffers,
        // the owned range's dictionary) in one slab, before the stages ask for it piece by piece
        pfp_arena_reserve(R.ctx, (size_t)(R.n_local + R.n_local / 2) + ((size_t)256 << 20));
        if (!ensure_dev(&R.buf, &R.buf_cap, (size_t)(R.front + R.n_local + 64))) {
            multi_fail(m, g, PFPB200_E_NOMEM, "device allocation of the shard failed");
            return;
        }
        const u64 from = R.pos0 - R.front, bytes = R.front + R.n_local;
        if (bytes == 0) return;
        if (m->text) {
            MR_CUDA(cudaMemcpyAsync(R.buf, m->text + from, (size_t)bytes, cudaMemcpyHostToDevice, st));
        } else if (m->src_dev) {
            MR_CUDA(cudaMemcpyPeerAsync(R.buf, R.device, m->src_dev + from, m->r[0].device, (size_t)bytes, st));
        } else {
            MR_LIB(pfp_file_to_device(R.ctx, m->src_fd, from, bytes, R.buf));
        }
    };
    [&]() {
        if (!ok()) return;
        upload();
        if (!ok()) return;
        R.first_bad = ~0ull;
        if (R.n_local) {
            R.h_small[0] = R.n_local;
            MR_CUDA(cudaMemcpyAsync(R.d_small, R.h_small, sizeof(u64), cudaMemcpyHostToDevice, st));
            MR_LIB(pfp_first_invalid(R.ctx, R.buf + R.front, R.n_local, R.d_small));
            MR_CUDA(cudaMemcpyAsync(R.h_small, R.d_small, sizeof(u64), cudaMemcpyDeviceToHost, st));
            MR_CUDA(cudaStreamSynchronize(st));
            if (R.h_small[0] < R.n_local) R.first_bad = R.pos0 + R.h_small[0];
        }
    }();
    m->bar.wait();
    {   // the text ends at the first byte <= 0x02 (newscan.cpp:364): rare, plan again and copy again
        u64 cut = ~0ull;
        for (int q = 0; q < G; q++) cut = std::min(cut, m->r[q].first_bad);
        const bool redo = cut < m->n_eff;
        m->bar.wait();                                    // everybody has read the old plan
        if (redo) {
            if (g == 0) {
                if (m->opts.flags & PFPB200_F_VERBOSE)
                    fprintf(stderr, "Invalid char found in input file: no additional chars will be read\n");
                plan_shards(m, cut);
            }
            m->bar.wait();
            [&]() {
                if (!ok()) return;
                upload();
                if (ok()) MR_CUDA(cudaStreamSynchronize(st));
            }();
        }
    }
    mark(R, PH_H2D);

    // ---- 2. scan --------------------------------------------------------------------------------------
    auto scan = [&]() {
        pfpb200_shard sh;
        memset(&sh, 0, sizeof(sh));
        sh.d_buf = R.buf; sh.n_buf = R.front + R.n_local; sh.buf_pos0 = R.pos0 - R.front;
        sh.own_lo = R.pos0; sh.own_hi = R.pos0 + R.n_local; sh.n_global = m->n_eff;
        sh.is_last = R.is_last ? 1u : 0u;
        u64 first = 0;
        MR_LIB(pfpb200_shard_scan(R.ctx, &sh, &m->opts, &R.n_trig, &first, &R.last_trig, nullptr));
    };
    R.n_trig = 0;
    if (ok()) scan();
    mark(R, PH_SCAN);
    m->bar.wait();

    // ---- 3. seams: the first phrase ending here starts behind the last trigger of a lower rank ------
    i64 fs = -1;
    [&]() {
        if (!ok()) return;
        fs = first_phrase_start(m, g, w);
        const bool has_phrase = R.n_trig > 0 || R.is_last;
        const u64 from = fs < 0 ? 0 : (u64)fs;
        if (g > 0 && has_phrase && from < R.pos0 - R.front) {
            // a phrase that began more than `front` bytes before this shard (a long run without a
            // trigger, possibly covering whole shards): widen the front, copy and scan again
            R.front = std::min<u64>(R.pos0, ((R.pos0 - from) + 4095) / 4096 * 4096);
            upload();
            if (ok()) scan();
        }
    }();
    mark(R, PH_SEAMS);

    // ---- 4. words: K2 + K3 + pool of the shard -------------------------------------------------------
    memset(&R.wd, 0, sizeof(R.wd));
    if (ok()) [&]() { MR_LIB(pfpb200_shard_words(R.ctx, fs, &R.wd, nullptr)); }();
    R.n_words = R.wd.n_words;
    R.n_phrases = R.wd.n_phrases;
    mark(R, PH_WORDS);

    // ---- 5. splitters from a sample of every rank's first keys ----------------------------------------
    R.n_sample = 0;
    [&]() {
        if (!ok() || R.n_words == 0) return;
        u32 k = 0;
        MR_LIB(pfpb200_shard_sample_keys(R.ctx, MULTI_SAMPLE, R.h_sample, &k));
        R.n_sample = k;
    }();
    m->bar.wait();
    u64 splitters[PFPB200_MAX_RANKS] = {0};
    {
        std::vector<u64> all;
        for (int q = 0; q < G; q++) all.insert(all.end(), m->r[q].h_sample, m->r[q].h_sample + m->r[q].n_sample);
        std::sort(all.begin(), all.end());
        for (int q = 0; q + 1 < G; q++)
            splitters[q] = all.empty() ? 0 : all[std::min<size_t>(all.size() - 1, (size_t)(q + 1) * all.size() / (size_t)G)];
    }
    mark(R, PH_SPLIT);

    // ---- 6. route: local words grouped by owner ---------------------------------------------------------
    memset(&R.rt, 0, sizeof(R.rt));
    for (int q = 0; q < PFPB200_MAX_RANKS; q++) R.words_to[q] = R.pool_to[q] = 0;
    [&]() {
        if (!ok() || R.n_words == 0) return;
        MR_LIB(pfpb200_shard_route(R.ctx, splitters, (u32)G, &R.rt, nullptr));
        for (int q = 0; q < G; q++) { R.words_to[q] = R.rt.words_to[q]; R.pool_to[q] = R.rt.pool_to[q]; }
    }();
    mark(R, PH_ROUTE);
    m->bar.wait();

    // ---- 7. receive buffers ------------------------------------------------------------------------------
    u64 recv_w = 0, recv_p = 0;
    for (int src = 0; src < G; src++) { recv_w += m->r[src].words_to[g]; recv_p += m->r[src].pool_to[g]; }
    [&]() {
        if (!ok()) return;
        if (!ensure_dev(&R.rx_words, &R.rx_words_cap, (size_t)recv_w) ||
            !ensure_dev(&R.rx_pool, &R.rx_pool_cap, (size_t)recv_p) ||
            !ensure_dev(&R.rx_ranks, &R.rx_ranks_cap, (size_t)R.n_words))
            multi_fail(m, g, PFPB200_E_NOMEM, "device allocation of the exchange buffers failed");
    }();
    m->bar.wait();

    // ---- 8. exchange: one DMA per (owner, buffer), straight into the owner's memory.  The 32-byte
    //         word records go first on the main stream; the pool bytes follow on a side stream and
    //         are still travelling while the owners dedup the records (step 9a needs nothing else)
    cudaEventRecord(R.ev_routed, st);
    cudaStreamWaitEvent(R.side, R.ev_routed, 0);
    [&]() {
        if (!ok() || R.n_words == 0) return;
        std::vector<u64> sw(G + 1, 0), sp(G + 1, 0);           // my routed segments, in owner order
        for (int q = 0; q < G; q++) { sw[q + 1] = sw[q] + R.words_to[q]; sp[q + 1] = sp[q] + R.pool_to[q]; }
        for (int pass = 0; pass < 2; pass++)
            for (int i = 0; i < G; i++) {
                const int q = (g + i) % G;                  // start with myself, then round the ring
                Rank &O = m->r[q];
                u64 w_off = 0, p_off = 0;                   // my slot: behind the segments of the lower ranks
                for (int src = 0; src < g; src++) { w_off += m->r[src].words_to[q]; p_off += m->r[src].pool_to[q]; }
                if (pass == 0 && R.words_to[q])
                    MR_CUDA(cudaMemcpyPeerAsync(O.rx_words + w_off, O.device, R.rt.words + sw[q], R.device,
                                                (size_t)R.words_to[q] * sizeof(pfpb200_word), st));
                if (pass == 1 && R.pool_to[q])
                    MR_CUDA(cudaMemcpyPeerAsync(O.rx_pool + p_off, O.device, R.rt.pool + sp[q], R.device,
                                                (size_t)R.pool_to[q] * sizeof(u64), R.side));
            }
    }();
    cudaEventRecord(R.ev_sent, st);
    cudaEventRecord(R.ev_pool, R.side);
    m->bar.wait();
    for (int src = 0; src < G; src++)
        if (src != g) cudaStreamWaitEvent(st, m->r[src].ev_sent, 0);
    mark(R, PH_EXCHANGE);

    // ---- 9. merge: (a) dedup of the received records, (b) once the bytes are here: rank + .dict/.occ -----
    memset(&R.mg, 0, sizeof(R.mg));
    [&]() {
        if (!ok()) return;
        MR_LIB(pfpb200_dict_merge_begin(R.ctx, recv_w, R.rx_words, nullptr));
    }();
    for (int src = 0; src < G; src++) cudaStreamWaitEvent(st, m->r[src].ev_pool, 0);
    [&]() {
        if (!ok()) return;
        MR_LIB(pfpb200_dict_merge_finish(R.ctx, R.rx_pool, recv_p, w,
                                         m->opts.flags & (PFPB200_F_COMPRESS | PFPB200_F_VERIFY), &R.mg, nullptr));
    }();
    R.n_distinct = R.mg.n_distinct;
    R.sum_word_len = R.mg.sum_word_len;
    // only the last piece keeps the final 0x00 (newscan.cpp:438)
    R.piece_bytes = R.mg.dict_bytes ? R.mg.dict_bytes - (g == G - 1 ? 0 : 1) : 0;
    mark(R, PH_MERGE);
    m->bar.wait();

    // ---- 10. totals, host buffers, ranks back ---------------------------------------------------------------
    u64 base[PFPB200_MAX_RANKS] = {0};
    u64 off_P = 0, off_d = 0, off_dict = 0;
    for (int q = 0; q < G; q++) {
        base[q] = q ? base[q - 1] + m->r[q - 1].n_distinct : 0;
        if (q < g) { off_P += m->r[q].n_phrases; off_d += m->r[q].n_distinct; off_dict += m->r[q].piece_bytes; }
    }
    if (g == 0 && ok()) {
        u64 tp = 0, td = 0, tb = 0, ts = 0;
        for (int q = 0; q < G; q++) {
            tp += m->r[q].n_phrases; td += m->r[q].n_distinct; tb += m->r[q].piece_bytes; ts += m->r[q].sum_word_len;
        }
        m->tot_phrases = tp; m->tot_distinct = td; m->tot_dict = tb; m->tot_sum_len = ts;
        if (td > 0x7FFFFFFEull) multi_fail(m, g, PFPB200_E_LIMIT, "more than 2^31-2 distinct words");        // newscan.cpp:114
        else if (tp >= 0xFFFFFFFFull) multi_fail(m, g, PFPB200_E_LIMIT, "the parse contains more than 2^32-2 words");  // bigbwt:110-114
        size_t need[5] = {(size_t)tb, (size_t)td * 4, (size_t)tp * 4, (size_t)tp,
                          (m->opts.flags & PFPB200_F_SAI) ? (size_t)tp * PFP_IBYTES : 0};
        if (m->out_path) {                 // files: created here at their final size, filled by all ranks
            for (int k = 0; k < 5; k++) need[k] = 0;
            if (ok() && multi_create_files(m, tb, td, tp) != 0) multi_fail(m, g, PFPB200_E_IO, m->io_err);
        }
        for (int k = 0; k < 5 && ok(); k++) {
            if (need[k] <= m->pin_cap[k]) continue;
            if (m->pin[k]) cudaFreeHost(m->pin[k]);
            m->pin[k] = nullptr;
            m->pin_cap[k] = 0;
            const size_t cap = need[k] + need[k] / 8 + 4096;
            if (cudaHostAlloc(&m->pin[k], cap, cudaHostAllocPortable) != cudaSuccess) {
                cudaGetLastError();
                multi_fail(m, g, PFPB200_E_NOMEM, "pinned host allocation of the outputs failed");
                break;
            }
            m->pin_cap[k] = cap;
        }
    }
    [&]() {
        if (!ok()) return;
        u64 ro = 0;                                          // my received entries are grouped by source
        for (int src = 0; src < G; src++) {
            const u64 cnt = m->r[src].words_to[g];
            u64 back_off = 0;                                // behind what src routed to the owners below me
            for (int q = 0; q < g; q++) back_off += m->r[src].words_to[q];
            if (cnt)
                MR_CUDA(cudaMemcpyPeerAsync(m->r[src].rx_ranks + back_off, m->r[src].device, R.mg.rank_of_entry + ro,
                                            R.device, (size_t)cnt * sizeof(u32), st));
            ro += cnt;
        }
    }();
    cudaEventRecord(R.ev_back, st);
    m->bar.wait();
    for (int src = 0; src < G; src++)
        if (src != g) cudaStreamWaitEvent(st, m->r[src].ev_back, 0);
    mark(R, PH_BACK);

    // ---- 11. remap: .parse of the shard ----------------------------------------------------------------------
    R.d_parse = nullptr;
    [&]() {
        if (!ok() || R.n_phrases == 0) return;
        const u32 *rank_of_word = nullptr;
        MR_LIB(pfpb200_shard_ranks_back(R.ctx, (u32)G, R.rx_ranks, base, &rank_of_word));
        MR_LIB(pfpb200_shard_remap(R.ctx, rank_of_word, &R.d_parse, nullptr));
    }();
    mark(R, PH_REMAP);

    // ---- 12. my pieces of the five streams: into the files, or to the host buffers ---------------------------
    if (m->out_path) {
        [&]() {
            if (!ok()) return;
            MR_CUDA(cudaStreamSynchronize(st));
            MR_LIB(multi_write_pieces(m, R, off_dict, off_d, off_P));
        }();
    } else
    [&]() {
        if (!ok()) return;
        u8 *h_dict = (u8 *)m->pin[0];
        u32 *h_occ = (u32 *)m->pin[1], *h_parse = (u32 *)m->pin[2];
        u8 *h_last = (u8 *)m->pin[3], *h_sai = (u8 *)m->pin[4];
        if (R.piece_bytes)
            MR_CUDA(cudaMemcpyAsync(h_dict + off_dict, R.mg.dict, (size_t)R.piece_bytes, cudaMemcpyDeviceToHost, st));
        if (R.n_distinct)
            MR_CUDA(cudaMemcpyAsync(h_occ + off_d, R.mg.occ, (size_t)R.n_distinct * 4, cudaMemcpyDeviceToHost, st));
        if (R.n_phrases) {
            MR_CUDA(cudaMemcpyAsync(h_parse + off_P, R.d_parse, (size_t)R.n_phrases * 4, cudaMemcpyDeviceToHost, st));
            MR_CUDA(cudaMemcpyAsync(h_last + off_P, R.wd.last, (size_t)R.n_phrases, cudaMemcpyDeviceToHost, st));
            if (R.wd.sai && h_sai)
                MR_CUDA(cudaMemcpyAsync(h_sai + off_P * PFP_IBYTES, R.wd.sai, (size_t)R.n_phrases * PFP_IBYTES,
                                        cudaMemcpyDeviceToHost, st));
        }
    }();
    mark(R, PH_D2H);
    cudaStreamSynchronize(st);
    cudaStreamSynchronize(R.side);
    if (ok()) {
        for (int k = 1; k < PH_COUNT; k++) {
            float t = 0;
            if (cudaEventElapsedTime(&t, R.ev_phase[k - 1], R.ev_phase[k]) == cudaSuccess) R.ms_phase[k] = t;
            else cudaGetLastError();
        }
    }
    R.launches = pfpb200_launch_count(R.ctx);
    m->bar.wait();
}

int check_multi_opts(pfpb200_multi *m, const pfpb200_opts *o) {
    if (!m || !o) return PFPB200_E_ARG;
    m->err[0] = 0;
    if (o->w < 4) { snprintf(m->err, sizeof(m->err), "Windows size must be at least 4"); return PFPB200_E_ARG; }
    if (o->p < 10) { snprintf(m->err, sizeof(m->err), "Modulus must be at least 10"); return PFPB200_E_ARG; }
    if (o->w > 65536) { snprintf(m->err, sizeof(m->err), "window size too large"); return PFPB200_E_ARG; }
    if (o->nseg < 0) { snprintf(m->err, sizeof(m->err), "Number of threads cannot be negative"); return PFPB200_E_ARG; }
    return PFPB200_OK;
}

}  // namespace

extern "C" int pfpb200_multi_create(int n_gpus, const int *gpu_ids, pfpb200_multi **out) {
    if (!out || n_gpus < 1 || n_gpus > PFPB200_MAX_RANKS) return PFPB200_E_ARG;
    *out = nullptr;
    pfpb200_multi *m = new (std::nothrow) pfpb200_multi();
    if (!m) return PFPB200_E_NOMEM;
    m->n = n_gpus;
    { const char *ev = getenv("PFPB200_MULTI_MIN_SHARD"); if (ev && atoll(ev) > 0) m->min_shard = (u64)atoll(ev); }
    { const char *ev = getenv("PFPB200_MULTI_FRONT"); if (ev && atoll(ev) >= 0) m->front_cap = (u64)atoll(ev); }
    { const char *ev = getenv("PFPB200_MULTI_SPLIT_KEY"); m->split_key = ev && atoi(ev) != 0; }
    m->r.resize(n_gpus);
    m->bar.n = n_gpus;
    int rc = PFPB200_OK;
    {   // the CUDA contexts of the devices come up side by side (a third of a second each)
        std::vector<std::thread> th;
        std::vector<int> rcs(n_gpus, PFPB200_OK);
        for (int g = 0; g < n_gpus; g++) m->r[g].device = gpu_ids ? gpu_ids[g] : g;
        for (int g = 0; g < n_gpus; g++) {
            bool first = true;                       // one thread per distinct device; repeats follow in order
            for (int q = 0; q < g; q++) first = first && m->r[q].device != m->r[g].device;
            if (first) th.emplace_back([m, g, n_gpus, &rcs]() {
                for (int q = g; q < n_gpus; q++)
                    if (m->r[q].device == m->r[g].device) rcs[q] = pfpb200_create(m->r[q].device, &m->r[q].ctx);
            });
        }
        for (auto &t : th) t.join();
        for (int g = 0; g < n_gpus; g++) if (rcs[g] != PFPB200_OK && rc == PFPB200_OK) rc = rcs[g];
    }
    for (int g = 0; g < n_gpus && rc == PFPB200_OK; g++) {
        Rank &R = m->r[g];
        bool ok = cudaSetDevice(R.device) == cudaSuccess &&
                  cudaEventCreateWithFlags(&R.ev_sent, cudaEventDisableTiming) == cudaSuccess &&
                  cudaEventCreateWithFlags(&R.ev_back, cudaEventDisableTiming) == cudaSuccess &&
                  cudaEventCreateWithFlags(&R.ev_routed, cudaEventDisableTiming) == cudaSuccess &&
                  cudaEventCreateWithFlags(&R.ev_pool, cudaEventDisableTiming) == cudaSuccess &&
                  cudaStreamCreateWithFlags(&R.side, cudaStreamNonBlocking) == cudaSuccess &&
                  cudaMalloc(&R.d_small, 16 * sizeof(u64)) == cudaSuccess &&
                  cudaHostAlloc(&R.h_small, 16 * sizeof(u64), cudaHostAllocPortable) == cudaSuccess &&
                  cudaHostAlloc(&R.h_sample, MULTI_SAMPLE * sizeof(u64), cudaHostAllocPortable) == cudaSuccess;
        for (int k = 0; k < PH_COUNT && ok; k++) ok = cudaEventCreate(&R.ev_phase[k]) == cudaSuccess;
        if (!ok) { cudaGetLastError(); rc = PFPB200_E_CUDA; }
    }
    // direct peer copies where the hardware allows them (NVLink / NVSwitch); without peer access
    // cudaMemcpyPeerAsync still works, staged by the driver
    for (int a = 0; a < n_gpus && rc == PFPB200_OK; a++)
        for (int b = 0; b < n_gpus; b++) {
            const int da = m->r[a].device, db = m->r[b].device;
            if (da == db) continue;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, da, db) == cudaSuccess && can) {
                cudaSetDevice(da);
                cudaError_t e = cudaDeviceEnablePeerAccess(db, 0);
                if (e != cudaSuccess) cudaGetLastError();      // already enabled is fine
            }
        }
    if (rc != PFPB200_OK) { pfpb200_multi_destroy(m); return rc; }
    *out = m;
    return PFPB200_OK;
}

extern "C" void pfpb200_multi_destroy(pfpb200_multi *m) {
    if (!m) return;
    for (Rank &R : m->r) {
        if (!R.ctx) continue;
        cudaSetDevice(R.device);
        cudaStreamSynchronize(R.ctx->stream);
        if (R.buf) cudaFree(R.buf);
        if (R.rx_words) cudaFree(R.rx_words);
        if (R.rx_pool) cudaFree(R.rx_pool);
        if (R.rx_ranks) cudaFree(R.rx_ranks);
        if (R.d_small) cudaFree(R.d_small);
        if (R.h_small) cudaFreeHost(R.h_small);
        if (R.h_sample) cudaFreeHost(R.h_sample);
        if (R.ev_sent) cudaEventDestroy(R.ev_sent);
        if (R.ev_back) cudaEventDestroy(R.ev_back);
        if (R.ev_routed) cudaEventDestroy(R.ev_routed);
        if (R.ev_pool) cudaEventDestroy(R.ev_pool);
        if (R.side) { cudaStreamSynchronize(R.side); cudaStreamDestroy(R.side); }
        for (int k = 0; k < PH_COUNT; k++)
            if (R.ev_phase[k]) cudaEventDestroy(R.ev_phase[k]);
        pfpb200_destroy(R.ctx);
    }
    for (int k = 0; k < 5; k++)
        if (m->pin[k]) cudaFreeHost(m->pin[k]);
    delete m;
}

extern "C" const char *pfpb200_multi_last_error(const pfpb200_multi *m) { return m ? m->err : ""; }

extern "C" int pfpb200_multi_n_gpus(const pfpb200_multi *m) { return m ? m->n : 0; }

extern "C" int pfpb200_multi_phase_ms(const pfpb200_multi *m, float *out, int cap) {
    if (!m || !out) return PFPB200_E_ARG;
    int k = 0;
    for (int g = 0; g < m->n; g++)
        for (int p = 0; p < PH_COUNT && k < cap; p++) out[k++] = m->r[g].ms_phase[p];
    return k;
}

// one parse of n_text bytes from the source set in m (text / src_fd / src_dev)
static int multi_run(pfpb200_multi *m, uint64_t n_text, const pfpb200_opts *opts, pfpb200_outputs *host_out,
                     pfpb200_stats *stats) {
    int rc;
    memset(host_out, 0, sizeof(*host_out));
    if (stats) memset(stats, 0, sizeof(*stats));
    m->n_text = n_text;
    m->opts = *opts;
    m->failed.store(0);
    plan_shards(m, n_text);
    const double t0 = wall_sec();
    std::vector<std::thread> th;
    for (int g = 1; g < m->n; g++) th.emplace_back(rank_main, m, g);
    rank_main(m, 0);
    for (auto &t : th) t.join();
    m->sec_wall = wall_sec() - t0;
    rc = m->failed.load();
    if (rc != PFPB200_OK) return rc;
    host_out->dict = (const u8 *)m->pin[0]; host_out->dict_bytes = m->tot_dict;
    host_out->occ = (const u32 *)m->pin[1]; host_out->n_distinct = m->tot_distinct;
    host_out->parse = (const u32 *)m->pin[2]; host_out->n_phrases = m->tot_phrases;
    host_out->last = (const u8 *)m->pin[3];
    host_out->sai = (opts->flags & PFPB200_F_SAI) ? (const u8 *)m->pin[4] : nullptr;
    if (stats) {
        const u64 P = m->tot_phrases, d = m->tot_distinct;
        stats->n_text = m->n_eff; stats->n_phrases = P; stats->n_distinct = d;
        stats->sum_word_len = m->tot_sum_len; stats->dict_bytes = m->tot_dict;
        stats->alg_bytes = m->n_eff + 4 * P + P + ((opts->flags & PFPB200_F_SAI) ? 5 * P : 0) + m->tot_dict + 4 * d;
        auto mx = [&](int a, int b) {                  // slowest rank over phases a..b
            float v = 0;
            for (const Rank &R : m->r) { float s = 0; for (int k = a; k <= b; k++) s += R.ms_phase[k]; v = std::max(v, s); }
            return v;
        };
        stats->ms_h2d = mx(PH_H2D, PH_H2D);
        stats->ms_scan = mx(PH_SCAN, PH_SEAMS);
        stats->ms_hash = mx(PH_WORDS, PH_WORDS);
        stats->ms_dedup = mx(PH_SPLIT, PH_EXCHANGE);       // routing + exchange: the shared dictionary's "map update"
        stats->ms_rank = mx(PH_MERGE, PH_MERGE);
        stats->ms_dict = mx(PH_BACK, PH_BACK);
        stats->ms_remap = mx(PH_REMAP, PH_REMAP);
        stats->ms_d2h = mx(PH_D2H, PH_D2H);
        stats->ms_total = mx(PH_SCAN, PH_REMAP);
        for (const Rank &R : m->r) stats->launches += R.launches;
    }
    return PFPB200_OK;
}

extern "C" int pfpb200_multi_parse_host(pfpb200_multi *m, const uint8_t *text, uint64_t n_text,
                                        const pfpb200_opts *opts, pfpb200_outputs *host_out,
                                        pfpb200_stats *stats) {
    int rc = check_multi_opts(m, opts);
    if (rc != PFPB200_OK) return rc;
    if (!host_out || (n_text && !text)) return PFPB200_E_ARG;
    static const u8 empty = 0;
    m->text = n_text ? text : &empty;
    m->src_fd = -1;
    m->src_dev = nullptr;
    return multi_run(m, n_text, opts, host_out, stats);
}

// newscan.x main() on several GPUs.  Plain text: every rank reads its own range of the file through
// its pinned ring.  FASTA: rank 0 streams the file in and runs K0; the shards of the extracted
// text then travel to the other GPUs peer to peer (NVLink).  gzip / FASTQ / CRLF input takes the
// host reader.  The outputs never gather on the host: rank 0 creates the five files at their final
// size and every rank writes its pieces into them (its own pinned ring, D2H overlapped with pwrite).
extern "C" int pfpb200_multi_parse_file(pfpb200_multi *m, const char *path, const pfpb200_opts *opts,
                                        pfpb200_stats *stats) {
    int rc = check_multi_opts(m, opts);
    if (rc != PFPB200_OK) return rc;
    if (!path) return PFPB200_E_ARG;
    const double t0 = wall_sec();
    const bool fasta = (opts->flags & PFPB200_F_FASTA) != 0;
    int fd = open(path, O_RDONLY);
    if (fd < 0) { snprintf(m->err, sizeof(m->err), "%s: %s", path, strerror(errno)); return PFPB200_E_IO; }
    struct stat sb;
    if (fstat(fd, &sb) != 0) { snprintf(m->err, sizeof(m->err), "%s: %s", path, strerror(errno)); close(fd); return PFPB200_E_IO; }
    const u64 fsize = (u64)sb.st_size;
    bool gz = false;
    if (fasta && fsize >= 2) {
        unsigned char mg[2] = {0, 0};
        if (pread(fd, mg, 2, 0) == 2) gz = mg[0] == 0x1f && mg[1] == 0x8b;
    }
    m->text = nullptr;
    m->src_fd = -1;
    m->src_dev = nullptr;
    u64 n = 0;
    u8 *d_text0 = nullptr;                     // rank 0's copy of the extracted text (FASTA)
    uint8_t *host_text = nullptr;
    Rank &R0 = m->r[0];
    if (!fasta) {
        m->src_fd = fd;
        n = fsize;
    } else if (!gz && fsize > 0) {
        cudaSetDevice(R0.device);
        u8 *d_file = nullptr;
        int supported = 0;
        u64 nt = 0;
        if (cudaMalloc(&d_file, fsize + 16) != cudaSuccess || cudaMalloc(&d_text0, fsize + 32) != cudaSuccess) {
            cudaGetLastError();
            if (d_file) cudaFree(d_file);
            if (d_text0) cudaFree(d_text0);
            close(fd);
            snprintf(m->err, sizeof(m->err), "device allocation for the FASTA file failed");
            return PFPB200_E_NOMEM;
        }
        rc = pfp_file_to_device(R0.ctx, fd, 0, fsize, d_file);
        u8 *out = d_text0;
        if (rc == PFPB200_OK) rc = pfp_fasta_device(R0.ctx, d_file, fsize, &out, &nt, &supported, false);   // K0
        cudaStreamSynchronize(R0.ctx->stream);
        pfp_release_scratch(R0.ctx);
        cudaFree(d_file);
        if (rc != PFPB200_OK) {
            snprintf(m->err, sizeof(m->err), "%s", pfpb200_last_error(R0.ctx));
            cudaFree(d_text0);
            close(fd);
            return rc;
        }
        if (supported) { m->src_dev = d_text0; n = nt; }
        else { cudaFree(d_text0); d_text0 = nullptr; }
    }
    if (fasta && !m->src_dev && !(fsize == 0)) {             // gzip, FASTQ, CRLF, ...: the host reader (pfp_io.c)
        int trunc = 0;
        rc = pfpb200_read_input(path, opts->flags, &host_text, &n, &trunc);
        if (rc != PFPB200_OK) { snprintf(m->err, sizeof(m->err), "cannot read %s", path); close(fd); return rc; }
        if (trunc) fprintf(stderr, "Invalid char found in input file: no additional chars will be read\n");
        m->text = host_text;
    }
    static const u8 empty = 0;
    if (n == 0 && !m->text) { m->text = &empty; m->src_fd = -1; m->src_dev = nullptr; }
    const double t1 = wall_sec();
    pfpb200_outputs ho;
    m->out_path = path;                   // every rank writes its pieces of the five files itself
    rc = multi_run(m, n, opts, &ho, stats);
    m->out_path = nullptr;
    close(fd);
    if (host_text) pfpb200_free_host(host_text);
    if (d_text0) { cudaSetDevice(R0.device); cudaFree(d_text0); }
    m->text = nullptr; m->src_fd = -1; m->src_dev = nullptr;
    if (rc != PFPB200_OK) return rc;
    if (stats) {
        stats->sec_read = (float)(t1 - t0);
        stats->sec_write = stats->ms_d2h * 1e-3f;       // the writes are the ranks' last phase
    }
    return PFPB200_OK;
}

// ---- the sharded pfbwt: pfpb200_multi_pfbwt_file ----------------------------------------------------------
// One host thread per rank runs pfbwt_rank_main.  Every decision that changes the sequence of barriers
// is taken on a value all ranks agree on (Barrier::sum), so a rank that fails keeps passing the same
// barriers as the others; nobody frees memory a peer may still read before the last barrier.
namespace {

// rank 0: the input files into HBM, checked as pfpb200_pfbwt_file checks them
int pb_inputs_rank0(pfpb200_multi *m, Rank &R) {
    void *p[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    PFP_TRY(pb_read_inputs(R.ctx, m->pb_base, m->pb_flags, p, R.pb_n));
    const u64 N = R.pb_n[0], psize = R.pb_n[2];
    if (N <= 1 + (u64)m->pb_w) return pfp_fail(R.ctx, PFPB200_E_ARG, "invalid dictionary file");
    if (psize >= 0xFFFFFFFEull)
        return pfp_fail(R.ctx, PFPB200_E_LIMIT, "more than 2^32-2 words in the parsing (.ilist is 32-bit)");
    for (int k = 0; k < 5; k++) R.pb_in[k] = p[k];
    return PFPB200_OK;
}

// the other ranks: rank 0's buffers when they share its device, otherwise copies peer to peer
int pb_inputs_peer(pfpb200_multi *m, Rank &R) {
    const Rank &R0 = m->r[0];
    for (int k = 0; k < 5; k++) {
        R.pb_n[k] = R0.pb_n[k];
        R.pb_in[k] = R0.pb_in[k];
        if (R.device == R0.device || !R0.pb_in[k]) continue;
        const u64 bytes = R0.pb_n[k] * PB_UNIT[k];
        void *d = nullptr;
        PFP_TRY(pfp_alloc(R.ctx, &d, bytes, true));
        if (bytes) PFP_CUDA(R.ctx, cudaMemcpyPeerAsync(d, R.device, R0.pb_in[k], R0.device, (size_t)bytes, R.ctx->stream));
        R.pb_in[k] = d;
    }
    PFP_CUDA(R.ctx, cudaStreamSynchronize(R.ctx->stream));
    return PFPB200_OK;
}

void pfbwt_rank_main(pfpb200_multi *m, int g) {
    Rank &R = m->r[g];
    const int G = m->n;
    pfpb200_ctx *ctx = R.ctx;
    PmState &S = R.pb;
    cudaSetDevice(R.device);
    auto ok = [&]() { return m->failed.load() == 0; };
    auto agree = [&]() { bool f; m->bar.sum(0, !ok(), &f); return !f; };    // a barrier: true when no rank has failed
    auto run = [&](int rc) { if (rc != PFPB200_OK) multi_fail(m, g, rc, pfpb200_last_error(ctx)); };
    const double t0 = wall_sec();
    double t_read = t0, t_sort = t0, t_plan = t0, t_write = t0;
    char part[2][4096] = {{0}, {0}};                        // my part files of .ssa / .esa (empty: none)
    const u32 launches0 = ctx->launches;
    memset(&R.pb_stat, 0, sizeof(R.pb_stat));
    R.pb_rounds = 0;
    R.pb_windows = R.pb_ssa = R.pb_esa = 0;
    R.pb_rank = nullptr;
    S = PmState();
    pfp_release_scratch(ctx);
    pfp_release_held(ctx);
    ctx->arena.peak = ctx->arena.in_use;                    // the peak reported is this call's
    // the shard and exchange buffers of an earlier parse go back to the driver (a parse grows them again)
    if (R.buf) { cudaFree(R.buf); R.buf = nullptr; R.buf_cap = 0; }
    if (R.rx_words) { cudaFree(R.rx_words); R.rx_words = nullptr; R.rx_words_cap = 0; }
    if (R.rx_pool) { cudaFree(R.rx_pool); R.rx_pool = nullptr; R.rx_pool_cap = 0; }
    if (R.rx_ranks) { cudaFree(R.rx_ranks); R.rx_ranks = nullptr; R.rx_ranks_cap = 0; }
    ctx->err[0] = 0;
    cudaMemsetAsync(ctx->d_flags, 0, 12 * sizeof(u64), ctx->stream);
    const bool want_sa = (m->pb_flags & (PFPB200_PFBWT_SA | PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA)) != 0;
    do {
        // ---- 1. inputs: read once by rank 0, to the other GPUs peer to peer ---------------------------------
        for (int k = 0; k < 5; k++) { R.pb_in[k] = nullptr; R.pb_n[k] = 0; }
        if (g == 0) run(pb_inputs_rank0(m, R));
        if (!agree()) break;
        if (g > 0) run(pb_inputs_peer(m, R));
        S.in = PbInput{(const u8 *)R.pb_in[0], R.pb_n[0], (const u32 *)R.pb_in[1], R.pb_n[1], (const u32 *)R.pb_in[2],
                       (const u8 *)R.pb_in[3], want_sa ? (const u8 *)R.pb_in[4] : nullptr, R.pb_n[2], m->pb_w, m->pb_flags};
        if (ok()) run(pb_words(ctx, S.in, &S.wd));
        t_read = wall_sec();
        if (!agree()) break;
        // ---- 2. partition by first key: splitters from a sample of every rank's block of positions ----------
        const u64 N = S.in.N, per = (N + (u64)G - 1) / (u64)G;
        R.n_sample = 0;
        {
            const u64 lo = std::min(N, per * (u64)g), hi = std::min(N, per * (u64)(g + 1));
            u32 got = 0;
            run(pm_sample(ctx, S, lo, hi, MULTI_SAMPLE, R.h_sample, &got));
            R.n_sample = got;
        }
        if (!agree()) break;
        u64 spl[PFPB200_MAX_RANKS] = {0};
        {
            std::vector<u64> all;
            for (int q = 0; q < G; q++) all.insert(all.end(), m->r[q].h_sample, m->r[q].h_sample + m->r[q].n_sample);
            std::sort(all.begin(), all.end());
            for (int q = 0; q + 1 < G; q++) spl[q] = all[std::min<size_t>(all.size() - 1, (size_t)(q + 1) * all.size() / (size_t)G)];
        }
        u64 M0 = 0;
        run(pm_count(ctx, S, g > 0 ? spl[g - 1] : 0, g + 1 < G ? spl[g] : 0, g > 0, g + 1 < G, &M0));
        S.M0 = M0;
        if (ok() && M0 >= 0xFFFFFFFFull) {
            char b[200];
            snprintf(b, sizeof(b), "%llu dictionary suffixes on one GPU, 2^32 or more: list more GPUs",
                     (unsigned long long)M0);
            multi_fail(m, g, PFPB200_E_LIMIT, b);
        }
        if (!agree()) break;
        S.base = 0;
        for (int q = 0; q < g; q++) S.base += m->r[q].pb.M0;
        if (ok()) run(pfp_alloc_t(ctx, &R.pb_rank, per));
        if (ok()) {
            u64 mx = 0;                                      // one key layout for every rank: the largest share decides
            for (int q = 0; q < G; q++) mx = std::max(mx, m->r[q].pb.M0);
            run(pm_collect(ctx, S, (m->split_key || pb_bits(mx) + pb_bits(N) + 1 > 64) ? 1 : 0));
        }
        if (!agree()) break;
        // ---- 3. prefix doubling in lockstep -------------------------------------------------------------------
        PmRanks ranks;
        memset(&ranks, 0, sizeof(ranks));
        for (int q = 0; q < G; q++) ranks.blk[q] = m->r[q].pb_rank;
        ranks.per = per;
        bool alive = true;
        u32 rounds = 1;
        for (u64 h = (u64)S.wd.h0;; h *= 2, rounds++) {
            u64 active = 0;
            if (ok()) run(pm_update(ctx, S, ranks, h, rounds == 1 ? 1 : 0, &active));   // stores changed ranks
            bool failed = false;
            const u64 tot = m->bar.sum(active, !ok(), &failed);
            if (failed) { alive = false; break; }
            if (tot == 0) {                                 // every rank's kernels are done: no peer reads my block any more
                run(pfp_free_now(ctx, R.pb_rank));
                break;
            }
            if (h >= 2 * N) {
                if (g == 0) multi_fail(m, g, PFPB200_E_INTERNAL, "pfbwt: prefix doubling did not converge");
                alive = false;
                break;
            }
            if (ok()) run(pm_gather(ctx, S, ranks, h));                                 // loads rank(i+h)
            if (!agree()) { alive = false; break; }
            if (ok()) run(pm_sort(ctx, S));
        }
        R.pb_rounds = rounds;
        if (!alive) break;
        if (ok()) run(pm_sort_done(ctx, S));
        t_sort = wall_sec();
        // ---- 4. the plan of my slice: once every rank has one, every offset is known ---------------------------
        if (ok()) run(pm_plan(ctx, S));
        pfp_arena_trim(ctx);                                // the sort's memory goes back for the others' windows
        t_plan = wall_sec();
        if (!agree()) break;
        const u32 flags = m->pb_flags;
        u64 off = 0, n_bwt = 0;
        int share = 0;                                      // ranks listed on my device
        for (int q = 0; q < G; q++) {
            if (q < g) off += m->r[q].pb.plan.chars;
            n_bwt += m->r[q].pb.plan.chars;
            share += m->r[q].device == R.device ? 1 : 0;
        }
        u64 budget = 0;                                     // read now: the other ranks' plans are allocated and
                                                            // their sorts' slabs released
        run(pb_budget(ctx, share, &budget));
        const u64 cap = pb_window_chars(S.plan, flags, budget);
        // ---- 5. files: rank 0 creates them, every rank writes its piece in windows ----------------------------
        char name[4096];
        auto fname = [&](const char *ext) { snprintf(name, sizeof(name), "%s.%s", m->pb_base, ext); return name; };
        if (g == 0) {
            int bad = create_sized(m, fname("bwt"), n_bwt);
            if (!bad && (flags & PFPB200_PFBWT_SA)) bad = create_sized(m, fname("sa"), (n_bwt - 1) * PFP_IBYTES);
            if (!bad && (flags & PFPB200_PFBWT_SSA)) bad = create_sized(m, fname("ssa"), 0);
            if (!bad && (flags & PFPB200_PFBWT_ESA)) bad = create_sized(m, fname("esa"), 0);
            if (bad) multi_fail(m, g, PFPB200_E_IO, m->io_err);
        }
        if (!agree()) break;
        // ranks sharing the device take their window's memory in one piece now that all have read their
        // budgets, before any of them allocates a window
        if (share > 1 && S.plan.n) pfp_arena_reserve(ctx, ctx->arena.total + pb_window_bytes(S.plan, flags, cap));
        {
            PbOutFiles F;
            static const char *const ext[4] = {"bwt", "sa", "ssa", "esa"};
            const u32 want[4] = {0, PFPB200_PFBWT_SA, PFPB200_PFBWT_SSA, PFPB200_PFBWT_ESA};
            for (int i = 0; i < 4 && ok() && S.plan.n; i++) {   // a rank that owns nothing writes nothing
                if (want[i] && !(flags & want[i])) continue;
                if (i < 2) {
                    snprintf(F.name[i], sizeof(F.name[i]), "%s.%s", m->pb_base, ext[i]);
                    F.fd[i] = open(F.name[i], O_WRONLY);
                } else {                                    // the run samples go to a part file of my own first
                    snprintf(part[i - 2], sizeof(part[i - 2]), "%s.%s.%d", m->pb_base, ext[i], g);
                    snprintf(F.name[i], sizeof(F.name[i]), "%s", part[i - 2]);
                    F.fd[i] = open(F.name[i], O_RDWR | O_CREAT | O_TRUNC, 0666);
                    if (F.fd[i] < 0) part[i - 2][0] = 0;
                }
                if (F.fd[i] < 0) run(pfp_fail(ctx, PFPB200_E_IO, "%s: %s", F.name[i], strerror(errno)));
            }
            if (ok() && S.plan.n) run(pb_write_windows(ctx, S.in, S.wd, S.plan, cap, F, off, &S.piece));
            R.pb_windows = S.piece.windows;
            for (int i = 0; i < 2; i++) {
                const int fd = F.fd[i];
                F.fd[i] = -1;
                if (fd >= 0 && close(fd) != 0 && ok())
                    run(pfp_fail(ctx, PFPB200_E_IO, "%s: write error: %s", F.name[i], strerror(errno)));
            }
            if (!agree()) break;
            // ---- 6. run samples across the rank borders: a piece's first -s record goes when the previous
            // non-empty piece ends with the same char, its last -e record when the next one starts with it
            const u64 S2 = 2 * PFP_IBYTES;
            u64 ns[PFPB200_MAX_RANKS], ne[PFPB200_MAX_RANKS], drop_s[PFPB200_MAX_RANKS], off_s = 0, off_e = 0;
            for (int q = 0, prev = -1; q < G; q++) {
                const PbPiece &pq = m->r[q].pb.piece;
                drop_s[q] = (flags & PFPB200_PFBWT_SSA) && pq.c_first >= 0 && pq.c_first == prev ? 1 : 0;
                ns[q] = pq.n_ssa - drop_s[q];
                if (pq.c_last >= 0) prev = pq.c_last;
            }
            for (int q = G - 1, next = -1; q >= 0; q--) {
                const PbPiece &pq = m->r[q].pb.piece;
                ne[q] = pq.n_esa - ((flags & PFPB200_PFBWT_ESA) && pq.c_last >= 0 && pq.c_last == next ? 1 : 0);
                if (pq.c_first >= 0) next = pq.c_first;
            }
            for (int q = 0; q < g; q++) { off_s += ns[q]; off_e += ne[q]; }
            R.pb_ssa = ns[g];
            R.pb_esa = ne[g];
            const u64 from[2] = {drop_s[g] * S2, 0}, bytes[2] = {ns[g] * S2, ne[g] * S2}, to[2] = {off_s * S2, off_e * S2};
            std::vector<u8> buf;
            for (int i = 0; i < 2 && ok(); i++) {
                if (F.fd[2 + i] < 0 || bytes[i] == 0) continue;
                buf.resize((size_t)std::min<u64>(bytes[i], (u64)64 << 20));
                const int fd = open(fname(ext[2 + i]), O_WRONLY);
                if (fd < 0) { run(pfp_fail(ctx, PFPB200_E_IO, "%s: %s", name, strerror(errno))); break; }
                for (u64 done = 0; done < bytes[i] && ok();) {
                    const u64 k = std::min<u64>(bytes[i] - done, buf.size());
                    const ssize_t r = pread(F.fd[2 + i], buf.data(), k, (off_t)(from[i] + done));
                    if (r != (ssize_t)k) run(pfp_fail(ctx, PFPB200_E_IO, "%s: read error", F.name[2 + i]));
                    else run(pb_put_host(ctx, fd, to[i] + done, buf.data(), k, name));
                    done += k;
                }
                if (close(fd) != 0 && ok()) run(pfp_fail(ctx, PFPB200_E_IO, "%s: write error: %s", name, strerror(errno)));
            }
        }
        t_write = wall_sec();
    } while (0);
    cudaStreamSynchronize(ctx->stream);
    for (int i = 0; i < 2; i++)                             // the part files go, whatever happened
        if (part[i][0]) unlink(part[i]);
    R.pb_stat.suffixes = S.M0;
    R.pb_stat.chars = S.plan.chars;
    R.pb_stat.hard = S.plan.n_hard;
    R.pb_stat.peak_bytes = ctx->arena.peak;
    R.pb_stat.ms_read = (float)(1e3 * (t_read - t0));
    R.pb_stat.ms_sort = (float)(1e3 * std::max(0.0, t_sort - t_read));
    // the plan and the windows' device work; the files, the barriers between them and the stitching
    R.pb_stat.ms_emit = (float)(1e3 * std::max(0.0, t_plan - t_sort) + S.piece.ms_emit);
    R.pb_stat.ms_write = (float)std::max(0.0, 1e3 * std::max(0.0, t_write - t_plan) - S.piece.ms_emit);
    R.launches = ctx->launches - launches0;
    m->bar.wait();                                          // no peer reads my memory any more
    pfp_release_scratch(ctx);
    m->bar.wait();                                          // rank 0's inputs, shared on its device, go last
    pfp_release_held(ctx);
}

}  // namespace

extern "C" int pfpb200_multi_pfbwt_file(pfpb200_multi *m, const char *basename, uint32_t w, uint32_t flags,
                                        pfpb200_pfbwt_result *res) {
    if (!m || !basename || !res) return PFPB200_E_ARG;
    memset(res, 0, sizeof(*res));
    m->err[0] = 0;
    if (const char *e = pb_arg_error(w, flags)) {
        snprintf(m->err, sizeof(m->err), "%s", e);
        return PFPB200_E_ARG;
    }
    for (int a = 0; a < m->n; a++)                          // the rank array is read and written across the GPUs
        for (int b = 0; b < m->n; b++) {
            const int da = m->r[a].device, db = m->r[b].device;
            int can = 0;
            if (da == db) continue;
            if (cudaDeviceCanAccessPeer(&can, da, db) != cudaSuccess || !can) {
                cudaGetLastError();
                snprintf(m->err, sizeof(m->err),
                         "CUDA devices %d and %d have no peer access: the sharded pfbwt loads and stores its rank "
                         "array across the GPUs directly (NVLink); list devices that reach each other", da, db);
                return PFPB200_E_ARG;
            }
        }
    m->pb_base = basename;
    m->pb_w = w;
    m->pb_flags = flags;
    m->failed.store(0);
    std::vector<std::thread> th;
    for (int g = 1; g < m->n; g++) th.emplace_back(pfbwt_rank_main, m, g);
    pfbwt_rank_main(m, 0);
    for (auto &t : th) t.join();
    m->pb_base = nullptr;
    const int rc = m->failed.load();
    if (rc != PFPB200_OK) return rc;
    const Rank &R0 = m->r[0];
    for (const Rank &R : m->r) {
        const pfpb200_pfbwt_rank &s = R.pb_stat;
        res->n_bwt += s.chars;
        res->n_ssa += R.pb_ssa;
        res->n_esa += R.pb_esa;
        res->hard += s.hard;
        res->launches += R.launches;
        res->ms_sa = std::max(res->ms_sa, s.ms_sort);
        res->ms_fill = std::max(res->ms_fill, s.ms_emit);
    }
    if (flags & PFPB200_PFBWT_SA) res->n_sa = res->n_bwt - 1;
    res->easy = res->n_bwt - res->hard;
    res->dict_bytes = R0.pb_n[0];
    res->dict_words = R0.pb_n[1];
    res->parse_size = R0.pb_n[2];
    res->rounds = R0.pb_rounds;
    res->ms_total = res->ms_sa + res->ms_fill;
    return PFPB200_OK;
}

extern "C" int pfpb200_multi_pfbwt_ranks(const pfpb200_multi *m, pfpb200_pfbwt_rank *out, int cap) {
    if (!m || !out) return PFPB200_E_ARG;
    int k = 0;
    for (; k < m->n && k < cap; k++) out[k] = m->r[k].pb_stat;
    return k;
}

extern "C" int pfpb200_multi_pfbwt_windows(const pfpb200_multi *m, uint64_t *windows, int cap) {
    if (!m || !windows) return PFPB200_E_ARG;
    int k = 0;
    for (; k < m->n && k < cap; k++) windows[k] = m->r[k].pb_windows;
    return k;
}
