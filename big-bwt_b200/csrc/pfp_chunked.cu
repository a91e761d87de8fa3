// pfp_chunked.cu -- the streamed parse of pfpb200_parse_file: a text larger than the device memory
// passes through HBM in chunks against ONE dictionary that lives across them.
//
// Reference: newscan streams its input byte by byte and keeps only the dictionary in RAM
// (newscan.cpp:332-374); the std::map lives across the whole input, the per-phrase hashes go to
// .parse_old, and remapParse() turns them into ranks at the end (:443-466).  Here:
//   * a chunk's device buffer is a CARRY (the text from the previous chunk's last trigger - w + 1
//     on, or everything from position 0 while no trigger has been seen) followed by new text; the
//     chunk owns the phrases that end in its new bytes and runs the shard stages on them (K1 with
//     a left halo, K2 with a first_start for the straddling phrase, K3 local dedup, pool);
//   * the chunk's distinct words go into the GLOBAL dictionary: a device table keyed by the
//     128-bit fingerprint (gdict_insert_k: plain load first, CAS on an empty slot), global word ids
//     d, d+1, .. for the new words in chunk-word order from one scan, their bytes appended to a
//     global pool (gdict_append_k), the table rehashed (gdict_rehash_k) before it passes half full;
//   * the chunk's phrases leave as global word ids, u32, into .parse at their offset (the
//     reference's .parse_old), .last and .sai straight to their files;
//   * after the last chunk the global dictionary is ranked and written as .dict/.occ, and .parse is
//     read back in pieces and rewritten in place with the ranks.
// Only the last chunk has the virtual 0x02^w final phrase.  Memory: the chunk pipeline is bounded
// by the budget; the global dictionary comes on top (DESIGN.md §6b).
#include "pfp_common.cuh"
#include "pfp_stages.cuh"
#include "pfp_fp.cuh"
#include <errno.h>
#include <fcntl.h>
#include <stdlib.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>
#include <algorithm>

namespace {

// device bytes per byte of new text a chunk may take: the two text buffers, the raw FASTA bytes
// and the parse scratch of the chunk (<= 4.5 B per byte at p = 10) fit with room to spare
constexpr u64 STREAM_BYTES_PER_BYTE = 8;
constexpr u64 STREAM_MIN_CHUNK = 256;
constexpr int STREAM_RESTART = 1;            // K0 met bytes it does not handle: start again from the host reader

struct __align__(16) GSlot { u64 key; u32 gid; u32 chk; };   // key 0: empty
constexpr int G_T = 256;
constexpr u32 G_MAX_PROBES = 4096;

double wall() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

// the fingerprint as the dictionary table sees it (PFPB200_TEST_WEAK_FP keeps 2 bits, as K3 does)
__device__ __forceinline__ PhraseFp table_fp(u64 fa, u64 fb, u32 weak) {
    PhraseFp r;
    r.fpa = weak ? (fa & 3ull) : fa;
    r.fpb = weak ? 0ull : fb;
    return r;
}

// Local word u of the chunk into the global table.  A word seen in an earlier chunk gets its global
// id and its count added (the words of one chunk have distinct keys, so one thread per global word
// and chunk touches its count); a new word claims an empty slot with a CAS and is numbered by
// gdict_assign_k.  new_words[u] = its pool words if new, else 0 (the scan of it places the bytes).
__global__ void __launch_bounds__(G_T) gdict_insert_k(const u64 *__restrict__ wfpa, const u64 *__restrict__ wfpb,
                                                      const u32 *__restrict__ lcount, const u32 *__restrict__ luwords,
                                                      u64 dl, GSlot *__restrict__ tab, u64 cap, u32 weak,
                                                      u32 *__restrict__ gcount, u32 *__restrict__ gmap,
                                                      u64 *__restrict__ lslot, u32 *__restrict__ is_new,
                                                      u32 *__restrict__ new_words, u64 *__restrict__ flags) {
    const u64 u = (u64)blockIdx.x * G_T + threadIdx.x;
    if (u >= dl) return;
    const PhraseFp r = table_fp(wfpa[u], wfpb[u], weak);
    const u64 k = sort_key_of(r.fpa, r.fpb);
    const u32 chk = check_of(r);
    u64 s = __umul64hi(k, cap);
    is_new[u] = 0;
    new_words[u] = 0;
    for (u32 probes = 0; probes <= G_MAX_PROBES; probes++) {
        const uint4 sv = __ldcg(reinterpret_cast<const uint4 *>(tab + s));
        const u64 key = ((u64)sv.y << 32) | sv.x;
        if (key == 0ull) {
            const u64 prev = atomicCAS((unsigned long long *)&tab[s].key, 0ull, (unsigned long long)k);
            if (prev == 0ull) {
                tab[s].chk = chk;
                lslot[u] = s;
                is_new[u] = 1;
                new_words[u] = luwords[u];
                return;
            }
            if (prev == k) {                           // two words of one chunk with one key: K3 rules it out
                atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_INTERNAL);
                return;
            }
        } else if (key == k) {
            if (sv.w != chk) atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_COLLISION);
            const u32 g = sv.z;
            gmap[u] = g;
            const u32 old = gcount[g], c = lcount[u];
            if (old + c < old) atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_LIMIT);   // newscan.cpp:613-617
            gcount[g] = old + c;
            return;
        }
        s = (s + 1 == cap) ? 0 : s + 1;
    }
    atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_TABLE_FULL);
}

// new words: global id d0 + (new words in front of u), into the table slot and the per-word arrays;
// acc[0] / acc[1] = largest / total length of the new words
__global__ void __launch_bounds__(G_T) gdict_assign_k(const u32 *__restrict__ is_new, const u32 *__restrict__ new_idx,
                                                      const u64 *__restrict__ new_off, u64 dl, u64 d0, u64 pw0,
                                                      const u64 *__restrict__ lslot, const u64 *__restrict__ wfpa,
                                                      const u64 *__restrict__ wfpb, const u32 *__restrict__ lcount,
                                                      const u32 *__restrict__ lulen, const u32 *__restrict__ luwords,
                                                      GSlot *__restrict__ tab, PhraseFp *__restrict__ gfp,
                                                      u32 *__restrict__ gcount, u32 *__restrict__ glen,
                                                      u32 *__restrict__ guw, u64 *__restrict__ goff,
                                                      u32 *__restrict__ gmap, u64 *__restrict__ acc) {
    const u64 u = (u64)blockIdx.x * G_T + threadIdx.x;
    const bool mine = u < dl && is_new[u];
    u32 len = 0;
    if (mine) {
        const u64 g = d0 + new_idx[u];
        len = lulen[u];
        tab[lslot[u]].gid = (u32)g;
        gmap[u] = (u32)g;
        store_rec(gfp, g, wfpa[u], wfpb[u]);
        gcount[g] = lcount[u];
        glen[g] = len;
        guw[g] = luwords[u];
        goff[g] = pw0 + new_off[u];
    }
    const u32 mx = __reduce_max_sync(0xffffffffu, len);
    u64 sum64 = len;                                         // 64 bit: 32 lengths may pass 2^32
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum64 += __shfl_xor_sync(0xffffffffu, sum64, o);
    if ((threadIdx.x & 31) == 0 && sum64) {
        atomicMax((unsigned long long *)&acc[0], (unsigned long long)mx);
        atomicAdd((unsigned long long *)&acc[1], (unsigned long long)sum64);
    }
}

// the bytes of the new words, from the chunk's pool to the end of the global pool: one warp per word
__global__ void __launch_bounds__(G_T) gdict_append_k(const u32 *__restrict__ is_new, const u32 *__restrict__ gmap,
                                                      const u32 *__restrict__ luwords, const u64 *__restrict__ luoff,
                                                      const u64 *__restrict__ lpool, u64 dl,
                                                      const u64 *__restrict__ goff, u64 *__restrict__ gpool) {
    const u32 lane = threadIdx.x & 31;
    for (u64 u = (u64)blockIdx.x * (G_T / 32) + (threadIdx.x >> 5); u < dl; u += (u64)gridDim.x * (G_T / 32)) {
        if (!is_new[u]) continue;
        const u64 *src = lpool + luoff[u];
        u64 *dst = gpool + goff[gmap[u]];
        const u32 n = luwords[u];
        for (u32 k = lane; k < n; k += 32) dst[k] = src[k];
    }
}

// PFPB200_F_VERIFY: every local word that met a word of an earlier chunk is compared byte for byte
// with the global copy (as pfp_merge_verify does for merged entries)
__global__ void __launch_bounds__(G_T) gdict_verify_k(const u32 *__restrict__ is_new, const u32 *__restrict__ gmap,
                                                      const u32 *__restrict__ lulen, const u64 *__restrict__ luoff,
                                                      const u64 *__restrict__ lpool, u64 dl,
                                                      const u32 *__restrict__ glen, const u64 *__restrict__ goff,
                                                      const u64 *__restrict__ gpool, u64 *__restrict__ flags) {
    const u32 lane = threadIdx.x & 31;
    for (u64 u = (u64)blockIdx.x * (G_T / 32) + (threadIdx.x >> 5); u < dl; u += (u64)gridDim.x * (G_T / 32)) {
        if (is_new[u]) continue;
        const u32 g = gmap[u];
        bool bad = lulen[u] != glen[g];
        if (!bad) {
            const u64 *a = lpool + luoff[u], *b = gpool + goff[g];
            const u32 n = (lulen[u] + 7) >> 3;
            for (u32 k = lane; k < n; k += 32) bad |= a[k] != b[k];
        }
        if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_COLLISION);
    }
}

// the d global words into an empty table of cap slots (their keys are distinct)
__global__ void __launch_bounds__(G_T) gdict_rehash_k(const PhraseFp *__restrict__ gfp, u64 d, u32 weak,
                                                      GSlot *__restrict__ tab, u64 cap, u64 *__restrict__ flags) {
    const u64 g = (u64)blockIdx.x * G_T + threadIdx.x;
    if (g >= d) return;
    const uint4 a = __ldg(reinterpret_cast<const uint4 *>(gfp + g));
    const PhraseFp r = table_fp(((u64)a.y << 32) | a.x, ((u64)a.w << 32) | a.z, weak);
    const u64 k = sort_key_of(r.fpa, r.fpb);
    u64 s = __umul64hi(k, cap);
    for (u32 probes = 0; probes <= G_MAX_PROBES; probes++) {
        if (atomicCAS((unsigned long long *)&tab[s].key, 0ull, (unsigned long long)k) == 0ull) {
            tab[s].gid = (u32)g;
            tab[s].chk = check_of(r);
            return;
        }
        s = (s + 1 == cap) ? 0 : s + 1;
    }
    atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_TABLE_FULL);
}

__global__ void set_u64_one_k(u64 *p, u64 v) { *p = v; }

// ---- host side -----------------------------------------------------------------------------------

// the global dictionary: per-word arrays indexed by global word id, the pool, the table
struct GDict {
    u64 d = 0, wcap = 0;
    PhraseFp *fp = nullptr;
    u32 *count = nullptr, *len = nullptr, *uw = nullptr;
    u64 *off = nullptr;
    u64 *pool = nullptr, pool_words = 0, pool_cap = 0;
    GSlot *tab = nullptr;
    u64 cap = 0;
    u32 max_len = 0;
    u64 sum_len = 0;
};

// where the new text of a chunk comes from
enum SrcKind { SRC_PLAIN, SRC_FASTA, SRC_HOST };

struct Stream {
    pfpb200_ctx *ctx;
    const char *path;
    pfpb200_opts o;
    u64 chunk = 0;
    // source
    SrcKind kind = SRC_PLAIN;
    int in_fd = -1;
    u64 in_size = 0, in_pos = 0;
    const u8 *host = nullptr;
    u32 fa_state = PFP_FASTA_LINE_START;
    u8 *raw = nullptr;                        // FASTA bytes of the chunk
    // buffers: [carry | new text], two of them so that the carry is one device-to-device copy
    u8 *buf[2] = {nullptr, nullptr};
    u64 bcap[2] = {0, 0};
    int cur = 0;
    u64 carry = 0;                            // bytes at the front of buf[cur]
    i64 pos0 = 0;                             // global position of buf[cur][0]
    i64 fs = -1;                              // start of the first phrase not yet owned
    u64 n_seen = 0;                           // text bytes so far
    u64 P = 0;                                // phrases written
    int chunks = 0;
    GDict G;
    u64 *acc = nullptr;                       // [0] largest new word, [1] their total length
    std::vector<void *> keep;                 // what lives across chunks
    // outputs
    int fd_parse = -1, fd_last = -1, fd_sai = -1;
    char n_parse[4096], n_last[4096], n_sai[4096];
    // timings
    double sec_read = 0, sec_write = 0;
    float ms_scan = 0, ms_hash = 0, ms_dedup = 0, ms_insert = 0, ms_remap = 0;
    bool trace = false;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};

    ~Stream() {
        for (cudaEvent_t e : ev)
            if (e) cudaEventDestroy(e);
        for (int f : {fd_parse, fd_last, fd_sai})
            if (f >= 0) close(f);
    }

    void persist(void *p) { keep.push_back(p); }
    void unpersist(void *p) {
        for (size_t i = 0; i < keep.size(); i++)
            if (keep[i] == p) { keep[i] = keep.back(); keep.pop_back(); return; }
    }
    // the chunk's scratch back to the arena; what lives across chunks stays
    int drop_chunk_scratch() {
        std::vector<void *> drop;
        for (void *p : ctx->scratch)
            if (std::find(keep.begin(), keep.end(), p) == keep.end()) drop.push_back(p);
        for (void *p : drop) PFP_TRY(pfp_free_now(ctx, p));
        return PFPB200_OK;
    }
    template <typename T>
    int grow(T **p, u64 used, u64 newcap) {      // a persistent array to newcap entries, the first `used` kept
        T *q = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &q, newcap));
        if (used) PFP_CUDA(ctx, cudaMemcpyAsync(q, *p, used * sizeof(T), cudaMemcpyDeviceToDevice, ctx->stream));
        if (*p) { unpersist(*p); PFP_TRY(pfp_free_now(ctx, *p)); }
        persist(q);
        *p = q;
        return PFPB200_OK;
    }
    int ensure_buf(int b, u64 bytes) {
        if (bcap[b] >= bytes) return PFPB200_OK;
        if (buf[b]) { unpersist(buf[b]); PFP_TRY(pfp_free_now(ctx, buf[b])); buf[b] = nullptr; }
        const u64 want = std::max(bytes, bcap[b] + bcap[b] / 2);
        PFP_TRY(pfp_alloc(ctx, (void **)&buf[b], want));
        persist(buf[b]);
        bcap[b] = want;
        return PFPB200_OK;
    }

    int open_out(const char *ext, char *name, int *fd, bool part) {
        snprintf(name, 4096, part ? "%s.%s.part" : "%s.%s", path, ext);
        *fd = open(name, O_RDWR | O_CREAT | O_TRUNC, 0666);
        if (*fd < 0) return pfp_fail(ctx, PFPB200_E_IO, "%s: %s", name, strerror(errno));
        return PFPB200_OK;
    }
    int to_file(int fd, u64 off, const void *d, u64 bytes, const char *name) {
        const double t = wall();
        const int rc = pfp_device_to_fd(ctx, fd, off, d, bytes, name);
        sec_write += wall() - t;
        return rc;
    }

    // up to `chunk` bytes of new text to dst; *last: the input ends with them; *restart: K0 refuses
    int next_text(u8 *dst, u64 *got, bool *last, bool *restart) {
        const double t = wall();
        *got = 0;
        *restart = false;
        const u64 take = std::min(chunk, in_size - in_pos);
        if (kind == SRC_HOST) {
            if (take) PFP_CUDA(ctx, cudaMemcpyAsync(dst, host + in_pos, take, cudaMemcpyHostToDevice, ctx->stream));
            *got = take;
        } else if (kind == SRC_PLAIN) {
            PFP_TRY(pfp_file_to_device(ctx, in_fd, in_pos, take, dst));
            *got = take;
            if (take) {   // the text ends at the first byte <= 0x02 (newscan.cpp:364)
                set_u64_one_k<<<1, 1, 0, ctx->stream>>>(&ctx->d_flags[14], take);
                PFP_LAUNCHED(ctx);
                PFP_TRY(pfp_first_invalid(ctx, dst, take, &ctx->d_flags[14]));
                PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[14], &ctx->d_flags[14], sizeof(u64), cudaMemcpyDeviceToHost,
                                              ctx->stream));
                PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
                if (ctx->h_flags[14] < take) {
                    fprintf(stderr, "Invalid char found in input file: no additional chars will be read\n");
                    *got = ctx->h_flags[14];
                    in_pos = in_size - take;                   // nothing behind the cut is read: this chunk is the last
                }
            }
        } else {
            PFP_TRY(pfp_file_to_device(ctx, in_fd, in_pos, take, raw));
            int supported = 1;
            u8 *out = dst;
            PFP_TRY(pfp_fasta_device(ctx, raw, take, &out, got, &supported, false, &fa_state, in_pos == 0));
            if (!supported) { *restart = true; return PFPB200_OK; }
        }
        in_pos += take;
        *last = in_pos == in_size;
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        sec_read += wall() - t;
        return PFPB200_OK;
    }

    // the table holds need words at most half full, the arrays and the pool hold need / pool_need
    int ensure_dict(u64 need) {
        if (need > G.wcap) {
            const u64 c = std::max<u64>({need, 2 * G.wcap, 1024u});
            PFP_TRY(grow(&G.fp, G.d, c));
            PFP_TRY(grow(&G.count, G.d, c));
            PFP_TRY(grow(&G.len, G.d, c));
            PFP_TRY(grow(&G.uw, G.d, c));
            PFP_TRY(grow(&G.off, G.d, c));
            G.wcap = c;
        }
        if (2 * need > G.cap) {
            if (G.tab) { unpersist(G.tab); PFP_TRY(pfp_free_now(ctx, G.tab)); G.tab = nullptr; }
            G.cap = std::max<u64>({4 * need, 2 * G.cap, 1024u});
            PFP_TRY(pfp_alloc_t(ctx, &G.tab, G.cap));
            persist(G.tab);
            PFP_CUDA(ctx, cudaMemsetAsync(G.tab, 0, G.cap * sizeof(GSlot), ctx->stream));
            if (G.d) {
                gdict_rehash_k<<<pfp_blocks(G.d, G_T), G_T, 0, ctx->stream>>>(G.fp, G.d, ctx->weak_fp, G.tab, G.cap,
                                                                           ctx->d_flags);
                PFP_LAUNCHED(ctx);
            }
        }
        return PFPB200_OK;
    }

    // the chunk's local dictionary D (wfpa/wfpb: its fingerprints) into the global one; gmap[u] =
    // global id of local word u
    int insert(const DictArrays &D, const u64 *wfpa, const u64 *wfpb, u32 *gmap, u64 *n_new) {
        const u64 dl = D.d;
        *n_new = 0;
        if (dl == 0) return PFPB200_OK;
        PFP_TRY(ensure_dict(G.d + dl));
        u64 *lslot = nullptr, *new_off = nullptr;
        u32 *is_new = nullptr, *new_words = nullptr, *new_idx = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &lslot, dl));
        PFP_TRY(pfp_alloc_t(ctx, &is_new, dl));
        PFP_TRY(pfp_alloc_t(ctx, &new_words, dl));
        PFP_TRY(pfp_alloc_t(ctx, &new_idx, dl));
        PFP_TRY(pfp_alloc_t(ctx, &new_off, dl));
        gdict_insert_k<<<pfp_blocks(dl, G_T), G_T, 0, ctx->stream>>>(wfpa, wfpb, D.count, D.uwords, dl, G.tab, G.cap,
                                                                  ctx->weak_fp, G.count, gmap, lslot, is_new,
                                                                  new_words, ctx->d_flags);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_exclusive_scan_u32(ctx, is_new, new_idx, dl, reinterpret_cast<u32 *>(&ctx->d_flags[1])));
        PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, new_words, new_off, dl, &ctx->d_flags[2]));
        PFP_CUDA(ctx, cudaMemcpyAsync(ctx->h_flags, ctx->d_flags, 3 * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        const u64 fl = ctx->h_flags[0];
        if (fl & PFP_ERRBIT_COLLISION)
            return pfp_fail(ctx, PFPB200_E_COLLISION, "fingerprint collision between different phrases");
        if (fl & PFP_ERRBIT_LIMIT) return pfp_fail(ctx, PFPB200_E_LIMIT, "a word occurs more than 2^32-1 times");
        if (fl & (PFP_ERRBIT_TABLE_FULL | PFP_ERRBIT_INTERNAL))
            return pfp_fail(ctx, PFPB200_E_INTERNAL, "global dictionary table: insert failed");
        const u64 nn = (u32)ctx->h_flags[1], npw = ctx->h_flags[2];
        if (G.d + nn > 0x7FFFFFFEull)
            return pfp_fail(ctx, PFPB200_E_LIMIT, "%llu distinct words exceed the limit 2^31-2",
                            (unsigned long long)(G.d + nn));                                    // newscan.cpp:114-117
        if (G.pool_words + npw > G.pool_cap) {
            const u64 c = std::max<u64>({G.pool_words + npw, 2 * G.pool_cap, 1024u});
            PFP_TRY(grow(&G.pool, G.pool_words, c));
            G.pool_cap = c;
        }
        gdict_assign_k<<<pfp_blocks(dl, G_T), G_T, 0, ctx->stream>>>(is_new, new_idx, new_off, dl, G.d, G.pool_words,
                                                                  lslot, wfpa, wfpb, D.count, D.ulen, D.uwords, G.tab,
                                                                  G.fp, G.count, G.len, G.uw, G.off, gmap, acc);
        PFP_LAUNCHED(ctx);
        const u64 want = (dl + G_T / 32 - 1) / (G_T / 32), maxb = (u64)ctx->sm_count * 16;
        const u32 nb = (u32)std::max<u64>(1, std::min(want, maxb));
        gdict_append_k<<<nb, G_T, 0, ctx->stream>>>(is_new, gmap, D.uwords, D.uoff, D.pool, dl, G.off, G.pool);
        PFP_LAUNCHED(ctx);
        if (o.flags & PFPB200_F_VERIFY) {
            gdict_verify_k<<<nb, G_T, 0, ctx->stream>>>(is_new, gmap, D.ulen, D.uoff, D.pool, dl, G.len, G.off, G.pool,
                                                        ctx->d_flags);
            PFP_LAUNCHED(ctx);
        }
        G.d += nn;
        G.pool_words += npw;
        *n_new = nn;
        return PFPB200_OK;
    }

    // one chunk: buf[cur][0 .. carry + got), its new bytes [carry, carry + got) owned
    int run_chunk(u64 got, bool last) {
        const u32 w = o.w;
        u8 *const B = buf[cur];
        const u64 n_buf = carry + got;
        const u64 own_lo = n_seen;
        n_seen += got;
        const i64 n_global = last ? (i64)n_seen : INT64_MAX / 4;     // no border behind a chunk that is not the last
        cudaEventRecord(ev[0], ctx->stream);
        ScanBits sb;
        float ms1 = 0;
        PFP_TRY(pfp_scan_bits(ctx, B, n_buf, (u64)pos0, own_lo, n_seen, w, o.p, false, &sb, &ms1));
        ms_scan += ms1;
        const u64 k = sb.total;
        const u64 Pc = k + (last ? 1 : 0);
        if (P + Pc >= 0xFFFFFFFFull)
            return pfp_fail(ctx, PFPB200_E_LIMIT, "the parse contains %llu words, more than 2^32-2",
                            (unsigned long long)(P + Pc));                                      // bigbwt:110-114
        cudaEventRecord(ev[1], ctx->stream);
        u64 dl = 0, nn = 0;
        i64 last_trig = -1;
        if (Pc > 0) {
            u64 *ends = nullptr;
            PFP_TRY(pfp_alloc_t(ctx, &ends, Pc));
            if (last) {
                set_u64_one_k<<<1, 1, 0, ctx->stream>>>(ends + k, (u64)n_global + w - 1);   // final word (:376-377)
                PFP_LAUNCHED(ctx);
            }
            PhraseArrays ph{};
            ph.ends = ends;
            PFP_TRY(pfp_alloc_t(ctx, &ph.rec, Pc));
            PFP_TRY(pfp_alloc_t(ctx, &ph.last, Pc));
            if (o.flags & PFPB200_F_SAI) PFP_TRY(pfp_alloc_t(ctx, &ph.sai, Pc * PFP_IBYTES));
            const TextView tv{B, n_buf, pos0, n_global};
            if (pfp_stream_ok(sb, w) && !ctx->legacy_k2) PFP_TRY(pfp_stream_stage(ctx, sb, tv, ph, Pc, fs, w, true));
            else {
                PFP_TRY(pfp_scan_emit(ctx, sb, ends));
                PFP_TRY(pfp_hash_stage(ctx, tv, ph, Pc, fs, w));
            }
            PFP_TRY(pfp_scan_bits_free(ctx, &sb));
            if (k > 0) {
                PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[13], ends + (k - 1), sizeof(u64), cudaMemcpyDeviceToHost,
                                              ctx->stream));
            }
            cudaEventRecord(ev[2], ctx->stream);
            DictArrays D;
            PFP_TRY(pfp_dedup_stage(ctx, ph, Pc, fs, w, &D));
            if (k > 0) last_trig = (i64)ctx->h_flags[13];                   // the dedup synchronised
            PFP_TRY(pfp_uid_words(ctx, &D, Pc));
            u64 *wfpa = nullptr, *wfpb = nullptr;
            PFP_TRY(pfp_alloc_t(ctx, &wfpa, D.d));
            PFP_TRY(pfp_alloc_t(ctx, &wfpb, D.d));
            PFP_TRY(pfp_gather_word_fp(ctx, D, ph, wfpa, wfpb));
            PFP_TRY(pfp_free_now(ctx, ph.rec));
            PFP_TRY(pfp_pool_stage(ctx, tv, &D));
            if (o.flags & PFPB200_F_VERIFY) PFP_TRY(pfp_verify_stage(ctx, tv, ends, fs, w, Pc, D));
            cudaEventRecord(ev[3], ctx->stream);
            u32 *gmap = nullptr;
            PFP_TRY(pfp_alloc_t(ctx, &gmap, D.d));
            dl = D.d;
            PFP_TRY(insert(D, wfpa, wfpb, gmap, &nn));
            cudaEventRecord(ev[4], ctx->stream);
            // the chunk's phrases as global word ids: the .parse_old of the reference
            u32 *gids = nullptr;
            PFP_TRY(pfp_alloc_t(ctx, &gids, Pc));
            PFP_TRY(pfp_remap_stage(ctx, D.uid, gmap, Pc, gids));
            cudaEventRecord(ev[5], ctx->stream);
            PFP_CUDA(ctx, cudaMemcpyAsync(ctx->h_flags, ctx->d_flags, sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
            PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            PFP_CUDA(ctx, cudaGetLastError());
            if (ctx->h_flags[0] & PFP_ERRBIT_COLLISION)
                return pfp_fail(ctx, PFPB200_E_COLLISION,
                                "two different phrases share a fingerprint (found by the verify pass)");
            float t[5];
            for (int i = 0; i < 5; i++) cudaEventElapsedTime(&t[i], ev[i], ev[i + 1]);
            ms_hash += t[1]; ms_dedup += t[2]; ms_insert += t[3]; ms_remap += t[4];
            const double tw = sec_write;
            PFP_TRY(to_file(fd_parse, 4 * P, gids, 4 * Pc, n_parse));
            PFP_TRY(to_file(fd_last, P, ph.last, Pc, n_last));
            if (ph.sai) PFP_TRY(to_file(fd_sai, PFP_IBYTES * P, ph.sai, PFP_IBYTES * Pc, n_sai));
            if (trace)
                fprintf(stderr, "[pfpb200 stream] chunk %d: new %llu carry %llu phrases %llu words %llu new %llu | "
                                "K1 %.3f K2 %.3f K3 %.3f insert %.3f remap %.3f ms, write %.3f s\n",
                        chunks, (unsigned long long)got, (unsigned long long)carry, (unsigned long long)Pc,
                        (unsigned long long)dl, (unsigned long long)nn, ms1, t[1], t[2], t[3], t[4], sec_write - tw);
        } else {
            PFP_TRY(pfp_scan_bits_free(ctx, &sb));
        }
        P += Pc;
        chunks++;
        if (!last) {
            // the carry: from the last trigger - w + 1 on (the phrase that straddles into the next chunk)
            i64 start = pos0;
            if (k > 0) {
                fs = last_trig - (i64)w + 1;
                start = std::max<i64>(fs, 0);
            }
            const u64 nc = n_seen - (u64)start;
            PFP_TRY(ensure_buf(cur ^ 1, nc + chunk + 64));
            if (nc)
                PFP_CUDA(ctx, cudaMemcpyAsync(buf[cur ^ 1], B + (start - pos0), nc, cudaMemcpyDeviceToDevice, ctx->stream));
            cur ^= 1;
            carry = nc;
            pos0 = start;
        }
        return drop_chunk_scratch();
    }

    int run_chunks() {
        PFP_TRY(ensure_buf(0, chunk + 64));
        if (kind == SRC_FASTA) {
            PFP_TRY(pfp_alloc(ctx, (void **)&raw, chunk + 16));
            persist(raw);
        }
        for (;;) {
            u64 got = 0;
            bool last = false, restart = false;
            PFP_TRY(next_text(buf[cur] + carry, &got, &last, &restart));
            if (restart) return STREAM_RESTART;
            PFP_TRY(run_chunk(got, last));
            if (last) return PFPB200_OK;
        }
    }

    // ranks of the global dictionary, .dict/.occ, and .parse rewritten from global ids to ranks
    int finish(pfpb200_stats *st) {
        // the table and the fingerprints are done with: room for the ranking
        for (void *p : {(void *)G.tab, (void *)G.fp}) { unpersist(p); PFP_TRY(pfp_free_now(ctx, p)); }
        G.tab = nullptr; G.fp = nullptr;
        for (u8 *&b : buf) { unpersist(b); PFP_TRY(pfp_free_now(ctx, b)); b = nullptr; }
        if (raw) { unpersist(raw); PFP_TRY(pfp_free_now(ctx, raw)); raw = nullptr; }
        PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[12], acc, 2 * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        G.max_len = (u32)ctx->h_flags[12];
        G.sum_len = ctx->h_flags[13];
        DictArrays D;
        D.d = G.d;
        D.count = G.count; D.ulen = G.len; D.uwords = G.uw; D.uoff = G.off;
        D.pool = G.pool; D.pool_words = G.pool_words;
        D.max_len = G.max_len; D.sum_len = G.sum_len;
        cudaEventRecord(ev[0], ctx->stream);
        u32 *order = nullptr, rounds = 0;
        PFP_TRY(pfp_rank_stage(ctx, D, &order, &rounds));
        cudaEventRecord(ev[1], ctx->stream);
        u8 *dict = nullptr;
        u32 *occ = nullptr, *rank_of_gid = nullptr;
        u64 dict_bytes = 0;
        PFP_TRY(pfp_dict_stage(ctx, D, order, (o.flags & PFPB200_F_COMPRESS) ? o.w : 0, &dict, &dict_bytes, &occ,
                               &rank_of_gid));
        cudaEventRecord(ev[2], ctx->stream);
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        PFP_CUDA(ctx, cudaGetLastError());
        float ms_rank = 0, ms_dict = 0;
        cudaEventElapsedTime(&ms_rank, ev[0], ev[1]);
        cudaEventElapsedTime(&ms_dict, ev[1], ev[2]);
        char name[4096];
        double tw = wall();
        snprintf(name, sizeof(name), "%s.%s", path, (o.flags & PFPB200_F_COMPRESS) ? "dicz" : "dict");
        PFP_TRY(pfp_device_to_file(ctx, name, dict, dict_bytes));
        snprintf(name, sizeof(name), "%s.occ", path);
        PFP_TRY(pfp_device_to_file(ctx, name, occ, 4 * G.d));
        const double t_dict_write = wall() - tw;
        // .parse: global ids -> ranks, in place, a piece at a time
        tw = wall();
        float ms_rewrite = 0;
        const u64 piece = std::max<u64>(chunk / 4, 1u << 16);
        u32 *pb = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &pb, std::min(piece, std::max<u64>(P, 1))));
        for (u64 a = 0; a < P; a += piece) {
            const u64 m = std::min(piece, P - a);
            PFP_TRY(pfp_file_to_device(ctx, fd_parse, 4 * a, 4 * m, (u8 *)pb));
            cudaEventRecord(ev[3], ctx->stream);
            PFP_TRY(pfp_remap_stage(ctx, pb, rank_of_gid, m, pb));
            cudaEventRecord(ev[4], ctx->stream);
            PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            float t = 0;
            cudaEventElapsedTime(&t, ev[3], ev[4]);
            ms_rewrite += t;
            PFP_TRY(pfp_device_to_fd(ctx, fd_parse, 4 * a, pb, 4 * m, n_parse));
        }
        const double t_rewrite = wall() - tw;
        sec_write += t_dict_write + t_rewrite;
        // -t T: the .last/.sai segments (newscan.hpp:274-276) from the streamed files
        tw = wall();
        if (o.nseg > 0) PFP_TRY(split_segments());
        sec_write += wall() - tw;
        if (trace)
            fprintf(stderr, "[pfpb200 stream] end: %d chunks, %llu phrases, %llu words | rank %.3f ms, dict %.3f ms, "
                            ".dict/.occ write %.3f s, .parse rewrite %.3f s (remap %.3f ms), segments %.3f s\n",
                    chunks, (unsigned long long)P, (unsigned long long)G.d, ms_rank, ms_dict, t_dict_write, t_rewrite,
                    ms_rewrite, wall() - tw);
        if (st) {
            st->n_text = n_seen; st->n_phrases = P; st->n_distinct = G.d;
            st->sum_word_len = G.sum_len; st->dict_bytes = dict_bytes;
            st->alg_bytes = n_seen + 4 * P + P + ((o.flags & PFPB200_F_SAI) ? 5 * P : 0) + dict_bytes + 4 * G.d;
            st->rank_rounds = rounds;
            st->launches = ctx->launches;
            st->ms_scan = ms_scan; st->ms_hash = ms_hash; st->ms_dedup = ms_dedup + ms_insert;
            st->ms_rank = ms_rank; st->ms_dict = ms_dict; st->ms_remap = ms_remap + ms_rewrite;
            st->ms_total = ms_scan + ms_hash + ms_dedup + ms_insert + ms_remap + ms_rank + ms_dict + ms_rewrite;
        }
        return PFPB200_OK;
    }

    int split_segments() {
        const int T = o.nseg;
        const u64 per = (P + (u64)T - 1) / (u64)T;
        std::vector<u8> hb((size_t)64 << 20);
        for (int pass = 0; pass < 2; pass++) {
            const int src = pass == 0 ? fd_last : fd_sai;
            if (src < 0) continue;
            const u64 unit = pass == 0 ? 1 : PFP_IBYTES;
            const char *ext = pass == 0 ? "last" : "sai";
            for (int s = 0; s < T; s++) {
                const u64 a = std::min(P, (u64)s * per), b = std::min(P, a + per);
                char name[4096];
                snprintf(name, sizeof(name), "%s.%d.%s", path, s, ext);              // utils.c:44-54
                const int fd = open(name, O_WRONLY | O_CREAT | O_TRUNC, 0666);
                if (fd < 0) return pfp_fail(ctx, PFPB200_E_IO, "%s: %s", name, strerror(errno));
                for (u64 x = a * unit; x < b * unit;) {
                    const size_t m = (size_t)std::min<u64>(hb.size(), b * unit - x);
                    if (pread(src, hb.data(), m, (off_t)x) != (ssize_t)m ||
                        pwrite(fd, hb.data(), m, (off_t)(x - a * unit)) != (ssize_t)m) {
                        close(fd);
                        return pfp_fail(ctx, PFPB200_E_IO, "%s: %s", name, strerror(errno));
                    }
                    x += m;
                }
                if (close(fd) != 0) return pfp_fail(ctx, PFPB200_E_IO, "%s: write error: %s", name, strerror(errno));
            }
        }
        close(fd_last); fd_last = -1; unlink(n_last);
        if (fd_sai >= 0) { close(fd_sai); fd_sai = -1; unlink(n_sai); }
        return PFPB200_OK;
    }

    int start(SrcKind k) {
        kind = k;
        PFP_TRY(open_out("parse", n_parse, &fd_parse, false));
        PFP_TRY(open_out("last", n_last, &fd_last, o.nseg > 0));
        if (o.flags & PFPB200_F_SAI) PFP_TRY(open_out("sai", n_sai, &fd_sai, o.nseg > 0));
        PFP_TRY(pfp_alloc_t(ctx, &acc, 2));
        persist(acc);
        PFP_CUDA(ctx, cudaMemsetAsync(acc, 0, 2 * sizeof(u64), ctx->stream));
        return run_chunks();
    }
};

}  // namespace

// The streamed form of pfpb200_parse_file (pfp_api.cu routes here when the one-shot footprint does
// not fit `budget` bytes of device memory).  *chunks = the chunks it took.
int pfp_parse_file_streamed(pfpb200_ctx *ctx, const char *path, const pfpb200_opts *opts, pfpb200_stats *stats,
                            u64 budget, u64 *chunks) {
    *chunks = 0;
    const bool fasta = (opts->flags & PFPB200_F_FASTA) != 0;
    int fd = open(path, O_RDONLY);
    if (fd < 0) return pfp_fail(ctx, PFPB200_E_IO, "%s: %s", path, strerror(errno));
    struct stat sbuf;
    if (fstat(fd, &sbuf) != 0) { close(fd); return pfp_fail(ctx, PFPB200_E_IO, "%s: %s", path, strerror(errno)); }
    bool gz = false;
    if (fasta && sbuf.st_size >= 2) {          // gzip input, as the reference's gzread takes it (newscan.cpp:332-336)
        unsigned char mg[2] = {0, 0};
        if (pread(fd, mg, 2, 0) == 2) gz = mg[0] == 0x1f && mg[1] == 0x8b;
    }
    const u64 chunk = std::max<u64>(budget / STREAM_BYTES_PER_BYTE, STREAM_MIN_CHUNK);
    uint8_t *text = nullptr;
    int rc = PFPB200_OK;
    double t_host = 0;
    for (int attempt = 0; attempt < 2; attempt++) {
        const bool host = gz || attempt > 0;
        if (host) {
            // gzip, FASTQ, CRLF, ...: the host reader with all of kseq's corner cases (pfp_io.c), as the
            // one-shot path takes them; the driver streams from its text
            const double t = wall();
            uint64_t n = 0;
            int trunc = 0;
            if (pfpb200_read_input(path, opts->flags, &text, &n, &trunc) != PFPB200_OK) {
                rc = pfp_fail(ctx, PFPB200_E_IO, "%s: cannot read", path);
                break;
            }
            if (trunc) fprintf(stderr, "Invalid char found in input file: no additional chars will be read\n");
            t_host = wall() - t;
            sbuf.st_size = (off_t)n;
        }
        Stream S;
        S.ctx = ctx; S.path = path; S.o = *opts; S.chunk = chunk;
        S.in_fd = fd; S.in_size = (u64)sbuf.st_size; S.host = text;
        S.trace = getenv("PFPB200_TRACE") != nullptr;
        for (cudaEvent_t &e : S.ev)
            if (cudaEventCreate(&e) != cudaSuccess) { rc = pfp_fail(ctx, PFPB200_E_CUDA, "cudaEventCreate failed"); break; }
        if (rc != PFPB200_OK) break;
        rc = S.start(host ? SRC_HOST : (fasta ? SRC_FASTA : SRC_PLAIN));
        if (rc == STREAM_RESTART) {            // K0 refused a later chunk: the host reader's text, from the start
            cudaStreamSynchronize(ctx->stream);
            pfp_release_scratch(ctx);
            ctx->err[0] = 0;
            rc = PFPB200_OK;
            continue;
        }
        if (rc == PFPB200_OK) rc = S.finish(stats);
        *chunks = (u64)S.chunks;
        if (stats) {
            stats->sec_read = (float)(S.sec_read + t_host);
            stats->sec_write = (float)S.sec_write;
        }
        break;
    }
    if (rc != PFPB200_OK) cudaStreamSynchronize(ctx->stream);
    if (text) pfpb200_free_host(text);
    close(fd);
    pfp_release_scratch(ctx);
    return rc;
}
