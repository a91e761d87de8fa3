// pfp_ingest.cu -- the host I/O path of the scanner, overlapped, and K0: FASTA text extraction on
// the device.
//
// Reference: newscan reads its input through ifstream::get() / gzread() byte by byte and never
// holds the file in memory (newscan.cpp:332-374); its outputs go out through fwrite per phrase
// (:290-301) and per word (:416-433); the text of `-f` mode is what kseq_read() returns record
// after record (kseq.h:177-218, newscan.cpp:338-349).  Here:
//   * file -> HBM: a few reader threads pread() 8 MB chunks into a ring of pinned slots and send
//     each chunk with ONE cudaMemcpyAsync on the thread's own stream -- read, copy and the next
//     read overlap; the file is never held in host memory;
//   * K0 (fasta_sum_k / fasta_scan_k / fasta_emit_k): the FASTA file bytes in HBM become the
//     text T: header lines and newlines dropped, a-z upper-cased, records concatenated.  "Is
//     this byte inside a header line" is a three-state automaton over the bytes (in a header
//     line / in a sequence line / at a line start); a run of bytes maps to a small summary that
//     composes associatively, so it is a scan: per 16 KB tile, over the tiles, and again inside
//     every tile to place the kept bytes.  Files with anything beyond plain multi-line FASTA
//     (FASTQ records, '\r', bytes <= 0x02 or 0xFF, junk in front of the first '>') are reported
//     as unsupported and take the host reader of pfp_io.c, which has all of kseq's corner cases;
//   * HBM -> files: the mirror image, D2H chunks through the same ring into pwrite().
#include "pfp_common.cuh"
#include "pfp_stages.cuh"
#include <errno.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <thread>
#include <unistd.h>

// ------------------------------------------------------------------------------------------------
// pinned ring + worker threads
// ------------------------------------------------------------------------------------------------
constexpr int IO_THREADS = PFP_IO_THREADS;
constexpr size_t IO_CHUNK = PFP_IO_CHUNK;

static int io_ensure(pfpb200_ctx *ctx) {
    PfpIo &io = ctx->io;
    if (io.ready) return PFPB200_OK;
    for (int t = 0; t < IO_THREADS; t++) {
        PFP_CUDA(ctx, cudaStreamCreateWithFlags(&io.stream[t], cudaStreamNonBlocking));
        for (int s = 0; s < 2; s++) {
            if (cudaHostAlloc(&io.slot[t][s], IO_CHUNK, cudaHostAllocPortable) != cudaSuccess) {
                cudaGetLastError();
                return pfp_fail(ctx, PFPB200_E_NOMEM, "pinned I/O ring: allocation failed");
            }
            PFP_CUDA(ctx, cudaEventCreateWithFlags(&io.ev[t][s], cudaEventDisableTiming));
        }
    }
    io.ready = true;
    return PFPB200_OK;
}

void pfp_io_destroy(pfpb200_ctx *ctx) {
    PfpIo &io = ctx->io;
    for (int t = 0; t < IO_THREADS; t++) {
        for (int s = 0; s < 2; s++) {
            if (io.slot[t][s]) cudaFreeHost(io.slot[t][s]);
            if (io.ev[t][s]) cudaEventDestroy(io.ev[t][s]);
            io.slot[t][s] = nullptr;
            io.ev[t][s] = nullptr;
        }
        if (io.stream[t]) cudaStreamDestroy(io.stream[t]);
        io.stream[t] = nullptr;
    }
    io.ready = false;
}

static ssize_t pread_all(int fd, void *buf, size_t n, off_t off) {
    size_t got = 0;
    while (got < n) {
        ssize_t r = pread(fd, (char *)buf + got, n - got, off + (off_t)got);
        if (r < 0) { if (errno == EINTR) continue; return -1; }
        if (r == 0) break;
        got += (size_t)r;
    }
    return (ssize_t)got;
}

static int pwrite_all(int fd, const void *buf, size_t n, off_t off) {
    size_t done = 0;
    while (done < n) {
        ssize_t r = pwrite(fd, (const char *)buf + done, n - done, off + (off_t)done);
        if (r < 0) { if (errno == EINTR) continue; return -1; }
        done += (size_t)r;
    }
    return 0;
}

// bytes [off, off+bytes) of fd -> d_dst.  Blocks until the data is in device memory.
int pfp_file_to_device(pfpb200_ctx *ctx, int fd, u64 off, u64 bytes, u8 *d_dst) {
    if (bytes == 0) return PFPB200_OK;
    PFP_TRY(io_ensure(ctx));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));       // d_dst may still be in use by earlier work
    PfpIo &io = ctx->io;
    const u64 nchunks = (bytes + IO_CHUNK - 1) / IO_CHUNK;
    int err[IO_THREADS] = {0};
    auto worker = [&](int t) {
        cudaSetDevice(ctx->device);
        u64 k = 0;
        for (u64 c = (u64)t; c < nchunks; c += IO_THREADS, k++) {
            const int s = (int)(k & 1);
            if (k >= 2 && cudaEventSynchronize(io.ev[t][s]) != cudaSuccess) { err[t] = 2; break; }
            const u64 o = c * IO_CHUNK;
            const size_t len = (size_t)((bytes - o) < IO_CHUNK ? (bytes - o) : IO_CHUNK);
            if (pread_all(fd, io.slot[t][s], len, (off_t)(off + o)) != (ssize_t)len) { err[t] = 1; break; }
            if (cudaMemcpyAsync(d_dst + o, io.slot[t][s], len, cudaMemcpyHostToDevice, io.stream[t]) != cudaSuccess ||
                cudaEventRecord(io.ev[t][s], io.stream[t]) != cudaSuccess) { err[t] = 2; break; }
        }
        if (cudaStreamSynchronize(io.stream[t]) != cudaSuccess && !err[t]) err[t] = 2;
    };
    std::thread th[IO_THREADS];
    const int nt = (int)(nchunks < (u64)IO_THREADS ? nchunks : (u64)IO_THREADS);
    for (int t = 1; t < nt; t++) th[t] = std::thread(worker, t);
    worker(0);
    for (int t = 1; t < nt; t++) th[t].join();
    for (int t = 0; t < nt; t++) {
        if (err[t] == 1) return pfp_fail(ctx, PFPB200_E_IO, "short read or read error: %s", strerror(errno));
        if (err[t] == 2) { cudaGetLastError(); return pfp_fail(ctx, PFPB200_E_CUDA, "host-to-device copy of the input failed"); }
    }
    return PFPB200_OK;
}

// d_src[0..bytes) -> file `name` (created / truncated).  The data must be complete on ctx->stream.
int pfp_device_to_file(pfpb200_ctx *ctx, const char *name, const void *d_src, u64 bytes) {
    int fd = open(name, O_WRONLY | O_CREAT | O_TRUNC, 0666);
    if (fd < 0) return pfp_fail(ctx, PFPB200_E_IO, "%s: %s", name, strerror(errno));
    if (bytes && ftruncate(fd, (off_t)bytes) != 0) { /* the writers extend the file themselves then */ }
    int rc = pfp_device_to_fd(ctx, fd, 0, d_src, bytes, name);
    if (close(fd) != 0 && rc == PFPB200_OK) rc = pfp_fail(ctx, PFPB200_E_IO, "%s: write error: %s", name, strerror(errno));
    return rc;
}

// d_src[0..bytes) -> bytes [file_off, file_off + bytes) of the open file fd (several GPUs write
// their pieces of one file side by side)
int pfp_device_to_fd(pfpb200_ctx *ctx, int fd, u64 file_off, const void *d_src, u64 bytes, const char *name) {
    if (bytes == 0) return PFPB200_OK;
    int rc = io_ensure(ctx);
    if (rc != PFPB200_OK) return rc;
    PfpIo &io = ctx->io;
    const u64 nchunks = (bytes + IO_CHUNK - 1) / IO_CHUNK;
    int err[IO_THREADS] = {0};
    auto worker = [&](int t) {
        cudaSetDevice(ctx->device);
        // chunk k+1 is on its way to the host while chunk k is written
        u64 mine[2] = {0, 0};
        size_t mlen[2] = {0, 0};
        u64 k = 0;
        auto issue = [&](u64 c, int s) {
            const u64 o = c * IO_CHUNK;
            mine[s] = o;
            mlen[s] = (size_t)((bytes - o) < IO_CHUNK ? (bytes - o) : IO_CHUNK);
            return cudaMemcpyAsync(io.slot[t][s], (const u8 *)d_src + o, mlen[s], cudaMemcpyDeviceToHost, io.stream[t]) == cudaSuccess &&
                   cudaEventRecord(io.ev[t][s], io.stream[t]) == cudaSuccess;
        };
        u64 c = (u64)t;
        if (c < nchunks && !issue(c, 0)) { err[t] = 2; return; }
        for (; c < nchunks; c += IO_THREADS, k++) {
            const int s = (int)(k & 1);
            const u64 nxt = c + IO_THREADS;
            if (nxt < nchunks && !issue(nxt, s ^ 1)) { err[t] = 2; break; }
            if (cudaEventSynchronize(io.ev[t][s]) != cudaSuccess) { err[t] = 2; break; }
            if (pwrite_all(fd, io.slot[t][s], mlen[s], (off_t)(file_off + mine[s])) != 0) { err[t] = 1; break; }
        }
        cudaStreamSynchronize(io.stream[t]);
    };
    std::thread th[IO_THREADS];
    const int nt = (int)(nchunks < (u64)IO_THREADS ? nchunks : (u64)IO_THREADS);
    for (int t = 1; t < nt; t++) th[t] = std::thread(worker, t);
    worker(0);
    for (int t = 1; t < nt; t++) th[t].join();
    int bad = 0;
    for (int t = 0; t < nt; t++) bad |= err[t];
    if (bad & 2) { cudaGetLastError(); return pfp_fail(ctx, PFPB200_E_CUDA, "%s: device-to-host copy failed", name); }
    if (bad & 1) return pfp_fail(ctx, PFPB200_E_IO, "%s: write error: %s", name, strerror(errno));
    return PFPB200_OK;
}

// ------------------------------------------------------------------------------------------------
// K0: FASTA on the device
// ------------------------------------------------------------------------------------------------
// States of the line automaton BEFORE a byte: H = inside a header line, S = inside a sequence
// line, L = at a line start.  Byte b:  L: '>' -> H, '\n' -> L, else -> S and b is kept;
// H: '\n' -> L, else H;  S: '\n' -> L, else S and b is kept.  (kseq.h:177-218: a record's header
// runs to the end of its line; then lines are appended without their newline until a line starts
// with '>', '@' or '+'.)
enum : u32 { FS_H = 0, FS_S = 1, FS_L = 2 };
static_assert(FS_L == PFP_FASTA_LINE_START, "the streamed parse starts a file in state L");

// Summary of a run of bytes.  Up to its first newline a run behaves according to the state it is
// entered in (all kept or all dropped); behind the first newline everything is fixed.
struct FaSum {
    u32 head;      // bytes in front of the first newline (all bytes if there is none)
    u32 rest;      // kept bytes behind the first newline
    u32 flags;     // bit 0: has a newline; bit 1: the run's first byte is '>' (head > 0); bits 2-3: state
                   // behind the run if it has a newline
};

__device__ __forceinline__ u32 fa_head_kept(const FaSum &b, u32 s) {
    if (s == FS_H) return 0u;
    if (s == FS_S) return b.head;
    return (b.head > 0 && !(b.flags & 2u)) ? b.head : 0u;
}
__device__ __forceinline__ u32 fa_out(const FaSum &b, u32 s) {
    if (b.flags & 1u) return (b.flags >> 2) & 3u;
    if (s != FS_L) return s;
    return b.head > 0 ? ((b.flags & 2u) ? FS_H : FS_S) : FS_L;
}
// a followed by b
__device__ __forceinline__ FaSum fa_join(const FaSum &a, const FaSum &b) {
    FaSum r;
    if (!(a.flags & 1u)) {                         // a has no newline: the heads join
        r.head = a.head + b.head;
        r.rest = b.rest;
        const u32 gt = a.head > 0 ? (a.flags & 2u) : (b.flags & 2u);
        r.flags = (b.flags & 1u) | gt | (b.flags & 12u);
    } else {
        const u32 s = (a.flags >> 2) & 3u;
        r.head = a.head;
        r.rest = a.rest + fa_head_kept(b, s) + b.rest;
        r.flags = 1u | (a.flags & 2u) | (fa_out(b, s) << 2);
    }
    return r;
}
__device__ __forceinline__ FaSum fa_identity() { FaSum r; r.head = 0; r.rest = 0; r.flags = 0; return r; }

constexpr int K0_T = 256;
constexpr int K0_RUN = 64;                         // bytes per thread
constexpr int K0_TILE = K0_T * K0_RUN;             // 16 KB per CTA
constexpr u32 K0_BAD = 1u;                         // flag word: input needs the host reader

// the 64 bytes of thread t of tile `tile` (zero beyond the end of the file: n is handled by len)
__device__ __forceinline__ void k0_load(const u8 *__restrict__ f, u64 n, u64 base, u32 w[16], u32 &len) {
    len = base >= n ? 0u : (u32)((n - base) < (u64)K0_RUN ? (n - base) : (u64)K0_RUN);
    if (len == K0_RUN && (((uintptr_t)(f + base)) & 15) == 0) {
        const uint4 *p = reinterpret_cast<const uint4 *>(f + base);
#pragma unroll
        for (int i = 0; i < 4; i++) { const uint4 v = __ldg(p + i); w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w; }
    } else {
#pragma unroll
        for (int i = 0; i < 16; i++) {
            u32 v = 0;
            for (int b = 0; b < 4; b++) {
                const u32 k = 4 * i + b;
                if (k < len) v |= (u32)f[base + k] << (8 * b);
            }
            w[i] = v;
        }
    }
}

// summary of the run held in w[] (len bytes) and whether it holds a byte the device path does
// not handle
__device__ __forceinline__ FaSum k0_summarise(const u32 w[16], u32 len, u32 &bad) {
    FaSum s = fa_identity();
    u32 st = FS_L;                                 // state behind the first newline is L
    bool seen_nl = false;
    u32 head = 0, rest = 0;
    bool first_gt = false;
#pragma unroll
    for (int i = 0; i < K0_RUN; i++) {
        if ((u32)i < len) {
            const u32 b = (w[i >> 2] >> (8 * (i & 3))) & 255u;
            if (b <= 2u || b == 255u || b == '\r') bad = 1;
            if (!seen_nl) {
                if (b == '\n') seen_nl = true;
                else { if (head == 0) first_gt = b == '>'; head++; }
            } else {
                if (st == FS_L) {
                    if (b == '>') st = FS_H;
                    else if (b == '@' || b == '+') { bad = 1; st = FS_S; rest++; }
                    else if (b != '\n') { st = FS_S; rest++; }
                } else if (b == '\n') st = FS_L;
                else if (st == FS_S) rest++;
            }
        }
    }
    s.head = head;
    s.rest = rest;
    s.flags = (seen_nl ? 1u : 0u) | (first_gt ? 2u : 0u) | (st << 2);
    return s;
}

__device__ __forceinline__ FaSum fa_shfl_up(const FaSum &v, int o) {
    FaSum r;
    r.head = __shfl_up_sync(0xffffffffu, v.head, o);
    r.rest = __shfl_up_sync(0xffffffffu, v.rest, o);
    r.flags = __shfl_up_sync(0xffffffffu, v.flags, o);
    return r;
}

// inclusive scan of the thread summaries over the CTA; *total = the whole tile
__device__ __forceinline__ FaSum k0_block_scan(FaSum v, FaSum *total, FaSum *sm /* 9 */) {
    const u32 lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const FaSum u = fa_shfl_up(v, o);
        if (lane >= (u32)o) v = fa_join(u, v);
    }
    __syncthreads();
    if (lane == 31) sm[wp] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        FaSum acc = fa_identity();
        for (int k = 0; k < K0_T / 32; k++) { const FaSum x = sm[k]; sm[k] = acc; acc = fa_join(acc, x); }
        sm[8] = acc;
    }
    __syncthreads();
    *total = sm[8];
    return fa_join(sm[wp], v);
}

// pass A: one summary per tile
__global__ void __launch_bounds__(K0_T) fasta_sum_k(const u8 *__restrict__ f, u64 n, FaSum *__restrict__ tsum,
                                                    u32 *__restrict__ flags) {
    __shared__ FaSum sm[9];
    const u64 base = (u64)blockIdx.x * K0_TILE + (u64)threadIdx.x * K0_RUN;
    u32 w[16], len, bad = 0;
    k0_load(f, n, base, w, len);
    const FaSum mine = k0_summarise(w, len, bad);
    FaSum tot;
    k0_block_scan(mine, &tot, sm);
    if (threadIdx.x == 0) tsum[blockIdx.x] = tot;
    if (__syncthreads_or((int)bad) && threadIdx.x == 0) atomicOr(flags, K0_BAD);
}

// scan over the tiles (one CTA): state and kept bytes in front of every tile, total kept bytes.
// Counters are 64 bit here: a slice of tiles, or a single line, may hold more than 4 GB.
struct FaSum64 { u64 head, rest; u32 flags; };
__device__ __forceinline__ u64 fa_head_kept64(u64 head, u32 flags, u32 s) {
    if (s == FS_H) return 0ull;
    if (s == FS_S) return head;
    return (head > 0 && !(flags & 2u)) ? head : 0ull;
}
__device__ __forceinline__ u32 fa_out64(u64 head, u32 flags, u32 s) {
    if (flags & 1u) return (flags >> 2) & 3u;
    if (s != FS_L) return s;
    return head > 0 ? ((flags & 2u) ? FS_H : FS_S) : FS_L;
}
__device__ __forceinline__ FaSum64 fa_join64(const FaSum64 &a, const FaSum &b) {
    FaSum64 r;
    if (!(a.flags & 1u)) {
        r.head = a.head + b.head;
        r.rest = b.rest;
        const u32 gt = a.head > 0 ? (a.flags & 2u) : (b.flags & 2u);
        r.flags = (b.flags & 1u) | gt | (b.flags & 12u);
    } else {
        const u32 s = (a.flags >> 2) & 3u;
        r.head = a.head;
        r.rest = a.rest + fa_head_kept64(b.head, b.flags, s) + b.rest;
        r.flags = 1u | (a.flags & 2u) | (fa_out64(b.head, b.flags, s) << 2);
    }
    return r;
}

__global__ void __launch_bounds__(1024) fasta_scan_k(const FaSum *__restrict__ tsum, u32 ntiles, u32 start,
                                                     u32 *__restrict__ tstate, u64 *__restrict__ toff,
                                                     u64 *__restrict__ total, u32 *__restrict__ end_state) {
    __shared__ u32 s_state[1024];
    __shared__ u64 s_kept[1024];
    __shared__ FaSum64 s_sum[1024];
    const u32 t = threadIdx.x;
    const u32 per = (ntiles + 1023) / 1024;
    const u32 lo = min(ntiles, t * per), hi = min(ntiles, lo + per);
    FaSum64 acc;
    acc.head = 0; acc.rest = 0; acc.flags = 0;
    for (u32 i = lo; i < hi; i++) acc = fa_join64(acc, tsum[i]);
    s_sum[t] = acc;
    __syncthreads();
    if (t == 0) {                                  // chain the 1024 slices from the entry state
        u32 st = start;
        u64 kept = 0;
        for (u32 k = 0; k < 1024; k++) {
            const FaSum64 b = s_sum[k];
            s_state[k] = st;
            s_kept[k] = kept;
            kept += fa_head_kept64(b.head, b.flags, st) + b.rest;
            st = fa_out64(b.head, b.flags, st);
        }
        *total = kept;
        *end_state = st;
    }
    __syncthreads();
    u32 st = s_state[t];
    u64 kept = s_kept[t];
    for (u32 i = lo; i < hi; i++) {
        const FaSum b = tsum[i];
        tstate[i] = st;
        toff[i] = kept;
        kept += (u64)fa_head_kept(b, st) + (u64)b.rest;
        st = fa_out(b, st);
    }
}

// pass B: kept bytes of the tile, upper-cased, to out[toff[tile] ..)
__global__ void __launch_bounds__(K0_T) fasta_emit_k(const u8 *__restrict__ f, u64 n, const u32 *__restrict__ tstate,
                                                     const u64 *__restrict__ toff, u8 *__restrict__ out,
                                                     u32 *__restrict__ flags) {
    __shared__ FaSum sm[9];
    __shared__ __align__(16) u8 stage[K0_TILE + 32];
    const u64 base = (u64)blockIdx.x * K0_TILE + (u64)threadIdx.x * K0_RUN;
    u32 w[16], len, bad = 0;
    k0_load(f, n, base, w, len);
    const FaSum mine = k0_summarise(w, len, bad);
    FaSum tot;
    const FaSum incl = k0_block_scan(mine, &tot, sm);
    // exclusive prefix = everything in front of my run inside the tile, entered in the tile's state
    const u32 s_tile = tstate[blockIdx.x];
    // (re-derive the exclusive summary: join of the runs before mine)
    FaSum excl;
    {
        const FaSum up = fa_shfl_up(incl, 1);
        const u32 lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
        excl = lane ? up : sm[wp];                 // sm[wp] = the warps in front (exclusive), still valid
    }
    const u32 my_state = fa_out(excl, s_tile);
    u32 pos = fa_head_kept(excl, s_tile) + ((excl.flags & 1u) ? excl.rest : 0u);
    const u64 o0 = toff[blockIdx.x];
    const u32 mis = (u32)((uintptr_t)(out + o0) & 15);          // stage so that 16-byte vectors line up
    u32 st = my_state;
#pragma unroll
    for (int i = 0; i < K0_RUN; i++) {
        if ((u32)i < len) {
            u32 b = (w[i >> 2] >> (8 * (i & 3))) & 255u;
            bool keep = false;
            if (st == FS_L) {
                if (b == '>') st = FS_H;
                else if (b != '\n') { st = FS_S; keep = true; if (b == '@' || b == '+') bad = 1; }   // FASTQ: host reader
            } else if (b == '\n') st = FS_L;
            else keep = st == FS_S;
            if (keep) {
                if (b - 'a' < 26u) b -= 32u;                    // toupper (newscan.cpp:340)
                stage[mis + pos++] = (u8)b;
            }
        }
    }
    if (__syncthreads_or((int)bad) && threadIdx.x == 0) atomicOr(flags, K0_BAD);
    const u32 kept = fa_head_kept(tot, s_tile) + ((tot.flags & 1u) ? tot.rest : 0u);
    if (kept == 0) return;
    u8 *dst = out + o0;
    const u32 head = min(kept, (16u - mis) & 15u);
    for (u32 i = threadIdx.x; i < head; i += K0_T) dst[i] = stage[mis + i];
    const u32 nvec = (kept - head) >> 4;
    const uint4 *sv = reinterpret_cast<const uint4 *>(stage + mis + head);      // mis + head is a multiple of 16
    uint4 *dv = reinterpret_cast<uint4 *>(dst + head);
    for (u32 i = threadIdx.x; i < nvec; i += K0_T) dv[i] = sv[i];
    const u32 done = head + 16 * nvec;
    for (u32 i = done + threadIdx.x; i < kept; i += K0_T) dst[i] = stage[mis + i];
}

__global__ void fasta_first_byte_k(const u8 *__restrict__ f, u32 *__restrict__ flags) {
    if (f[0] != '>') atomicOr(flags, K0_BAD);      // kseq skips junk in front of the first '>' / '@'
}

// d_file[0..n) (FASTA bytes in HBM) -> *d_text, *n_text.  *d_text non-null on entry: the caller's
// buffer (>= n + 16 bytes) is filled; else an arena buffer of ctx (held or scratch).
// *supported = 0: the file needs the host reader, nothing was produced.
// state: null = d_file is the whole file.  Otherwise d_file is a piece of it: *state holds the
// automaton state in front of it (FS_L at the file start) and receives the state behind it, and the
// leading '>' is required only of the piece that starts the file.
int pfp_fasta_device(pfpb200_ctx *ctx, const u8 *d_file, u64 n, u8 **d_text, u64 *n_text, int *supported,
                     bool held, u32 *state, bool file_start) {
    u8 *const user_out = *d_text;
    *d_text = nullptr;
    *n_text = 0;
    *supported = 1;
    if (n == 0) return PFPB200_OK;
    const u64 nt64 = (n + K0_TILE - 1) / K0_TILE;
    if (nt64 > 0x7FFFFFFFull) { *supported = 0; return PFPB200_OK; }
    const u32 ntiles = (u32)nt64;
    FaSum *tsum = nullptr;
    u32 *tstate = nullptr, *flags = nullptr;
    u64 *toff = nullptr, *total = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &tsum, ntiles));
    PFP_TRY(pfp_alloc_t(ctx, &tstate, ntiles));
    PFP_TRY(pfp_alloc_t(ctx, &toff, ntiles));
    PFP_TRY(pfp_alloc_t(ctx, &flags, 4));
    total = reinterpret_cast<u64 *>(flags + 2);
    PFP_CUDA(ctx, cudaMemsetAsync(flags, 0, 4 * sizeof(u32), ctx->stream));
    if (file_start) {
        fasta_first_byte_k<<<1, 1, 0, ctx->stream>>>(d_file, flags);
        PFP_LAUNCHED(ctx);
    }
    fasta_sum_k<<<ntiles, K0_T, 0, ctx->stream>>>(d_file, n, tsum, flags);
    PFP_LAUNCHED(ctx);
    fasta_scan_k<<<1, 1024, 0, ctx->stream>>>(tsum, ntiles, state ? *state : (u32)FS_L, tstate, toff, total, flags + 1);
    PFP_LAUNCHED(ctx);
    u32 h[4];
    PFP_CUDA(ctx, cudaMemcpyAsync(h, flags, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    u64 kept;
    memcpy(&kept, &h[2], sizeof(u64));
    if (h[0] & K0_BAD) {
        *supported = 0;
    } else {
        u8 *out = user_out;
        if (!out) PFP_TRY(pfp_alloc(ctx, (void **)&out, kept + 16, held));
        fasta_emit_k<<<ntiles, K0_T, 0, ctx->stream>>>(d_file, n, tstate, toff, out, flags);
        PFP_LAUNCHED(ctx);
        // a line starting with '@' or '+' (FASTQ) is only recognised now that the states are known
        PFP_CUDA(ctx, cudaMemcpyAsync(h, flags, sizeof(u32), cudaMemcpyDeviceToHost, ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (h[0] & K0_BAD) { *supported = 0; if (!user_out) PFP_TRY(pfp_free_now(ctx, out)); }
        else { *d_text = out; *n_text = kept; if (state) *state = h[1]; }
    }
    PFP_TRY(pfp_free_now(ctx, tsum));
    PFP_TRY(pfp_free_now(ctx, tstate));
    PFP_TRY(pfp_free_now(ctx, toff));
    PFP_TRY(pfp_free_now(ctx, flags));
    return PFPB200_OK;
}
