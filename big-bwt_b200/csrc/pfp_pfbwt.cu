// pfp_pfbwt.cu -- the last stage of the pipeline: the BWT (and suffix array) of the text from the
// dictionary, the inverted list of the parse's BWT and the permuted .last/.sai.  SURVEY.md 8(f) row 2.
//
// Replaces pfbwt.cpp of the reference (bwt(), pfbwt.cpp:109-242; main(), :318-407): there gSACA-K
// sorts the suffixes of the dictionary on one core (compute_dict_bwt_lcp, :483-515), and one loop
// walks them in order: suffixes of length <= w are skipped (:152), a suffix that is a whole word
// emits the .bwlast char of each of its occurrences (:154-203), a group of EQUAL proper suffixes
// of several words emits the chars in front of them, merged by the positions of the words'
// occurrences in the BWT of the parse -- a heap of ilist cursors (fwrite_chars_same_suffix, :521-560).
// Here, with everything resident in HBM:
//   1. word structure of the dictionary bytes (terminator flags -> scan -> word id per byte);
//   2. the dictionary suffixes, each ENDING AT ITS WORD'S TERMINATOR, sorted by prefix doubling on
//      ranks with the library's radix sort: rank = the slot where a suffix's group starts, the key
//      of a round is (rank, rank h bytes on -- or 0 past the terminator), a suffix alone in its
//      group or completely compared (h > length) leaves the active list.  Equal suffixes of
//      different words keep equal keys for ever: they end as one group -- exactly the groups the
//      reference finds through lcp >= suffixLen (:208-219).  No LCP array is needed;
//   3. per suffix in sorted order: occurrences of its word -> a scan gives every group its range of
//      the BWT; a group with one member or one char is filled directly ("easy"), the others go
//      through a radix sort of (group, ilist position) -- the merge of the reference's heap --
//      in batches of at most 2^30 occurrences ("hard");
//   4. with -S / -s / -e the suffix-array value of every BWT position is bwsai[ilist position] -
//      suffix length (:161,:585): written as 5-byte integers; the sampled variants are the
//      entries at the starts / ends of the BWT's runs (:165-193, :628-650).
// Outputs are byte-identical to pfbwtNT.x (.bwt, .sa, .ssa, .esa): tests/test_pfbwt_gpu.py.
#include "pfp_common.cuh"
#include "pfp_stages.cuh"
#include <errno.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

constexpr int PB_T = 256;
constexpr u64 PB_BATCH = (u64)1 << 30;          // occurrences sorted at once in the hard groups
constexpr u32 PB_BIG = 512;                     // easy members with more occurrences get a CTA instead of a thread

__device__ __forceinline__ bool pb_term(u8 c) { return c <= PFP_END_OF_WORD; }   // EndOfWord, EndOfDict

__global__ void __launch_bounds__(PB_T) pb_flags_k(const u8 *__restrict__ d, u64 N, u8 *__restrict__ flag) {
    const u64 t = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (t < N) flag[t] = pb_term(d[t]) ? 1 : 0;
}

// wend[k] = position of the k-th terminator; wid[t] = terminators before t = the word of position t
__global__ void __launch_bounds__(PB_T) pb_wend_k(const u8 *__restrict__ flag, const u32 *__restrict__ wid, u64 N,
                                                  u32 *__restrict__ wend) {
    const u64 t = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (t < N && flag[t]) wend[wid[t]] = (u32)t;
}

// round 1: every position by its first h0 symbols, cut behind the word's terminator (zero padded);
// terminators get key 0 and sort in front.  The symbols are the ORDER-PRESERVING DENSE CODES of the
// byte values that occur in the dictionary (terminators 1, then the text's alphabet from 2 up), bs
// bits each: a DNA dictionary has 7 values, 3 bits, and the first round already sorts by 21 symbols
// instead of 8 -- the doubling then runs at depths 21, 42, 84, ... and a third of its work is gone.
struct PbCodes { u8 code[256]; };

__global__ void __launch_bounds__(PB_T) pb_alpha_k(const u8 *__restrict__ d, u64 N, u32 *__restrict__ present) {
    u32 pm[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (u64 t = (u64)blockIdx.x * PB_T + threadIdx.x; t < N; t += (u64)gridDim.x * PB_T) {
        const u32 c = d[t];
#pragma unroll
        for (int k = 0; k < 8; k++) pm[k] |= ((c >> 5) == (u32)k) ? (1u << (c & 31)) : 0u;
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const u32 o = __reduce_or_sync(0xffffffffu, pm[k]);
        if ((threadIdx.x & 31) == 0 && o) atomicOr(&present[k], o);
    }
}

__global__ void __launch_bounds__(PB_T) pb_init_k(const u8 *__restrict__ d, u64 N, PbCodes cd, int h0, int bs,
                                                  u64 *__restrict__ key, u32 *__restrict__ val, u32 *__restrict__ slot) {
    __shared__ u8 code[256];
    code[threadIdx.x] = cd.code[threadIdx.x];                        // PB_T = 256
    __syncthreads();
    const u64 t = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (t >= N) return;
    u64 k = 0;
    bool live = !pb_term(d[t]);
    for (int i = 0; i < h0; i++) {
        u32 c = 0;
        if (live) {
            const u8 b = t + i < N ? d[t + i] : (u8)0;
            c = code[b];
            if (pb_term(b)) live = false;                            // the terminator itself is part of the key
        }
        k = (k << bs) | c;
    }
    key[t] = k;
    val[t] = (u32)t;
    slot[t] = (u32)t;
}

__global__ void __launch_bounds__(PB_T) pb_gflags_k(const u64 *__restrict__ key, u64 M, u8 *__restrict__ flag) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k < M) flag[k] = (k == 0 || key[k] != key[k - 1]) ? 1 : 0;
}

__global__ void __launch_bounds__(PB_T) pb_heads_k(const u8 *__restrict__ flag, const u32 *__restrict__ escan,
                                                   const u32 *__restrict__ slot, u64 M, u32 *__restrict__ head) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k < M && flag[k]) head[escan[k]] = slot[k];
}

// lim[t] = position of the terminator of t's word (one gather per round instead of two)
__global__ void __launch_bounds__(PB_T) pb_lim_k(const u32 *__restrict__ wid, const u32 *__restrict__ wend, u64 N,
                                                 u32 *__restrict__ lim) {
    const u64 t = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (t < N) lim[t] = wend[wid[t]];
}

// The sorted active suffixes: rank = slot where the group starts; a suffix leaves the active list
// when it is alone in its group or compared to its end (length + terminator <= h) -- only then is it
// written to the suffix array, and its rank only when it changed (both are random 4-byte stores).
// KB > 0: the keys are (old rank << (KB + 1)) | (second rank << 1) | done, written by pb_compact_k;
// KB = 0: the first round (raw bytes as keys) or 32-bit ranks: lengths and old ranks are not in the key.
__global__ void __launch_bounds__(PB_T) pb_update_k(const u8 *__restrict__ flag, const u32 *__restrict__ escan,
                                                    const u32 *__restrict__ slot, const u32 *__restrict__ val,
                                                    const u64 *__restrict__ key, int kb, int first,
                                                    const u32 *__restrict__ head, const u32 *__restrict__ lim, u64 M, u64 h,
                                                    u64 *__restrict__ sa, u32 *__restrict__ rank, u32 *__restrict__ rs,
                                                    u8 *__restrict__ keep) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k >= M) return;
    const u32 f = flag[k], s = val[k];
    const u32 r = head[escan[k] + f - 1u];
    const bool single = f && (k + 1 == M || flag[k + 1]);
    bool done, same = false;
    if (kb > 0 && !first) {
        const u64 kk = key[k];
        done = (kk & 1u) != 0;
        same = (u32)(kk >> (kb + 1)) == r;
    } else {
        done = (u64)lim[s] - s + 1 <= h;                      // bytes of the suffix + its terminator
        if (!first) same = (u32)(key[k] >> 32) == r;
    }
    if (!same) rank[s] = r;
    rs[k] = r;
    const bool stay = !(single || done);
    keep[k] = stay ? 1 : 0;
    if (!stay) sa[slot[k]] = ((u64)r << 32) | s;              // final place: (rank = start of its group, suffix) in one store
}

__global__ void __launch_bounds__(PB_T) pb_compact_k(const u8 *__restrict__ keep, const u32 *__restrict__ kscan,
                                                     const u32 *__restrict__ slot, const u32 *__restrict__ val,
                                                     const u32 *__restrict__ rs, const u32 *__restrict__ rank,
                                                     const u32 *__restrict__ lim, u64 M, u64 h, int kb,
                                                     u32 *__restrict__ slot2, u32 *__restrict__ val2,
                                                     u64 *__restrict__ key2) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k >= M || !keep[k]) return;
    const u32 p = kscan[k], s = val[k], l = lim[s];
    const u64 j = (u64)s + h;
    const u64 r2 = j <= l ? (u64)rank[j] : 0u;                // the terminator's rank is 0
    slot2[p] = slot[k];
    val2[p] = s;
    if (kb > 0) key2[p] = ((u64)rs[k] << (kb + 1)) | (r2 << 1) | (((u64)l - s + 1 <= 2 * h) ? 1u : 0u);
    else key2[p] = ((u64)rs[k] << 32) | r2;
}

// ---- the walk over the sorted suffixes -----------------------------------------------------------
struct PbView {
    const u8 *d;
    const u64 *sa;              // per slot: (rank << 32) | suffix position
    const u32 *wid, *wend, *occ, *istart;
    uint2 *mrec;                // per slot, written by pb_count_k: {word, suffix length}
    u16 *mc;                    // per slot: char in front | whole word << 8 | counts << 9
    u64 N;
    u32 w;
};
// the member record of slot k (pb_count_k wrote it): word, length, char in front; false: terminator or length <= w
__device__ __forceinline__ bool pb_member(const PbView &v, u64 k, u32 &word, u32 &len, bool &full, u8 &c) {
    const u32 m = v.mc[k];
    const uint2 r = v.mrec[k];
    word = r.x; len = r.y;
    full = (m & 0x100u) != 0;
    c = (u8)m;
    return (m & 0x200u) != 0;
}

// occurrences each sorted suffix contributes (0: terminator or length <= w), its member record, group starts
__global__ void __launch_bounds__(PB_T) pb_count_k(PbView v, u32 *__restrict__ cnt, u8 *__restrict__ newgrp) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k >= v.N) return;
    const u64 e = v.sa[k];
    const u32 s = (u32)e;
    newgrp[k] = (k == 0 || (u32)(e >> 32) != (u32)(v.sa[k - 1] >> 32)) ? 1 : 0;
    u32 word = 0, len = 0, n = 0, m = 0;
    if (!pb_term(v.d[s])) {
        word = v.wid[s];
        len = v.wend[word] - s;
        if (len > v.w) {                                             // pfbwt.cpp:152
            const bool full = s == 0 || v.d[s - 1] == PFP_END_OF_WORD;   // :154
            const u32 c = (s <= 1) ? 0u : v.d[s - 1];                // d[0] = 0 is the EOF char of the final BWT (:127)
            m = c | (full ? 0x100u : 0u) | 0x200u;
            n = v.occ[word];
        }
    }
    v.mrec[k] = make_uint2(word, len);
    v.mc[k] = (u16)m;
    cnt[k] = n;
}

__global__ void __launch_bounds__(PB_T) pb_first_k(const u8 *__restrict__ newgrp, const u32 *__restrict__ gscan, u64 N,
                                                   u32 *__restrict__ first) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k < N && newgrp[k]) first[gscan[k]] = (u32)k;
}

// mixed[g] = 1 when the members of group g do not all have the same char in front
__global__ void __launch_bounds__(PB_T) pb_mixed_k(PbView v, const u8 *__restrict__ newgrp, const u32 *__restrict__ gscan,
                                                   const u32 *__restrict__ first, u8 *__restrict__ mixed) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k >= v.N || newgrp[k]) return;
    u32 word, len; bool full; u8 c, c0;
    if (!pb_member(v, k, word, len, full, c)) return;
    const u32 g = gscan[k] + newgrp[k] - 1u;
    pb_member(v, first[g], word, len, full, c0);
    if (c != c0) mixed[g] = 1;
}

// hcnt[k] = occurrences of member k that need the merge: its group has several members and
// (different chars, or suffix-array values are wanted -- they differ even when the chars agree)
__global__ void __launch_bounds__(PB_T) pb_hard_k(const u32 *__restrict__ cnt, const u8 *__restrict__ newgrp,
                                                  const u32 *__restrict__ gscan, const u8 *__restrict__ mixed, u64 N,
                                                  int want_sa, u32 *__restrict__ hcnt) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k >= N) return;
    const bool alone = newgrp[k] && (k + 1 == N || newgrp[k + 1]);
    const u32 g = gscan[k] + newgrp[k] - 1u;
    hcnt[k] = (!alone && (want_sa || mixed[g])) ? cnt[k] : 0u;
}

__device__ __forceinline__ u64 pb_get5(const u8 *__restrict__ a, u64 i) {
    u64 x = 0;
#pragma unroll
    for (int j = PFP_IBYTES - 1; j >= 0; j--) x = (x << 8) | a[i * PFP_IBYTES + j];
    return x;
}
__device__ __forceinline__ void pb_put5(u8 *__restrict__ a, u64 i, u64 x) {
#pragma unroll
    for (int j = 0; j < PFP_IBYTES; j++) a[i * PFP_IBYTES + j] = (u8)(x >> (8 * j));
}

// members that need no merge: a whole word (chars from .bwlast, :155-203), or one char for all
__global__ void __launch_bounds__(PB_T) pb_easy_k(PbView v, const u32 *__restrict__ cnt, const u32 *__restrict__ hcnt,
                                                  const u64 *__restrict__ off, const u32 *__restrict__ ilist,
                                                  const u8 *__restrict__ bwlast, const u8 *__restrict__ bwsai,
                                                  u8 *__restrict__ bwt, u8 *__restrict__ sa5, u32 *__restrict__ big,
                                                  u32 *__restrict__ big_n, u32 big_cap) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k >= v.N || cnt[k] == 0 || hcnt[k] != 0) return;
    u32 word, len; bool full; u8 c;
    pb_member(v, k, word, len, full, c);
    const u32 n = cnt[k];
    if (n > PB_BIG) {                                                // a word with many occurrences: one CTA each, below
        const u32 i = atomicAdd(big_n, 1u);
        if (i < big_cap) big[i] = (u32)k;
        return;
    }
    const u64 o = off[k];
    const u32 is = v.istart[word] + 1u;                              // ilist[0] is the end symbol's entry (:376-383)
    for (u32 j = 0; j < n; j++) {
        const u32 ip = (full || sa5) ? ilist[is + j] : 0u;
        bwt[o + j] = full ? bwlast[ip] : c;
        if (sa5) pb_put5(sa5, o + j, (full && word == 0) ? pb_get5(bwsai, 0) - v.w   // the EOF suffix: the text length (:182)
                                                          : pb_get5(bwsai, ip) - len);
    }
}

// the easy members with more than PB_BIG occurrences: the threads of a CTA share the loop
__global__ void __launch_bounds__(PB_T) pb_easy_big_k(PbView v, const u32 *__restrict__ big, const u32 *__restrict__ big_n,
                                                      u32 big_cap, const u32 *__restrict__ cnt, const u64 *__restrict__ off,
                                                      const u32 *__restrict__ ilist, const u8 *__restrict__ bwlast,
                                                      const u8 *__restrict__ bwsai, u8 *__restrict__ bwt,
                                                      u8 *__restrict__ sa5) {
    const u32 nbig = min(*big_n, big_cap);
    for (u32 b = blockIdx.x; b < nbig; b += gridDim.x) {
        const u64 k = big[b];
        u32 word, len; bool full; u8 c;
        pb_member(v, k, word, len, full, c);
        const u32 n = cnt[k];
        const u64 o = off[k];
        const u32 is = v.istart[word] + 1u;
        for (u32 j = threadIdx.x; j < n; j += PB_T) {
            const u32 ip = (full || sa5) ? ilist[is + j] : 0u;
            bwt[o + j] = full ? bwlast[ip] : c;
            if (sa5) pb_put5(sa5, o + j, (full && word == 0) ? pb_get5(bwsai, 0) - v.w : pb_get5(bwsai, ip) - len);
        }
    }
}

// the occurrences of the hard members of slots [k0, k1), keyed by (group, position in the parse's BWT)
__global__ void __launch_bounds__(PB_T) pb_gen_k(PbView v, const u32 *__restrict__ hcnt, const u64 *__restrict__ hoff,
                                                 const u32 *__restrict__ gscan, const u8 *__restrict__ newgrp,
                                                 const u32 *__restrict__ ilist, u64 k0, u64 k1, u64 e0, u32 g0,
                                                 u64 *__restrict__ key, u32 *__restrict__ val) {
    const u64 k = k0 + (u64)blockIdx.x * PB_T + threadIdx.x;
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

__global__ void __launch_bounds__(PB_T) pb_scatter_k(PbView v, const u64 *__restrict__ key, const u32 *__restrict__ val,
                                                     u64 ne, u64 e0, u32 g0, const u32 *__restrict__ first,
                                                     const u64 *__restrict__ off, const u64 *__restrict__ hoff,
                                                     const u8 *__restrict__ bwsai, u8 *__restrict__ bwt,
                                                     u8 *__restrict__ sa5) {
    const u64 e = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (e >= ne) return;
    const u64 kk = key[e];
    const u32 k = val[e], f = first[(u32)(kk >> 32) + g0];
    const u64 pos = off[f] + (e0 + e - hoff[f]);
    u32 word, len; bool full; u8 c;
    pb_member(v, k, word, len, full, c);
    bwt[pos] = c;
    if (sa5) pb_put5(sa5, pos, pb_get5(bwsai, (u32)kk) - len);
}

// the next batch of hard groups: out = {kb, hoff[kb], group of slot ka, groups in [ka, kb)} with [ka, kb) =
// as many whole groups as fit into `cap` occurrences, at least one (hoff[0..N] is non-decreasing)
__global__ void pb_batch_k(const u64 *__restrict__ hoff, const u32 *__restrict__ gscan, const u8 *__restrict__ newgrp,
                           const u32 *__restrict__ first, u64 ngroups, u64 ka, u64 N, u64 cap, u64 *__restrict__ out) {
    const u64 target = hoff[ka] + cap;
    u64 kb = N;
    if (hoff[N] > target) {
        u64 a = ka, b = N;                                       // first index with hoff > target
        while (a < b) {
            const u64 m = (a + b) >> 1;
            if (hoff[m] <= target) a = m + 1; else b = m;
        }
        const u64 kl = a - 1;                                    // >= ka: hoff[ka] <= target
        const u64 g = gscan[kl] + newgrp[kl] - 1u;
        kb = first[g];
        if (kb <= ka) kb = g + 1 < ngroups ? first[g + 1] : N;   // one group larger than the batch: take it whole
    }
    const u64 ga = gscan[ka] + newgrp[ka] - 1u;
    out[0] = kb;
    out[1] = hoff[kb];
    out[2] = ga;
    out[3] = kb < N ? gscan[kb] + newgrp[kb] - 1u - ga : ngroups - ga;
}

// sampled suffix array: flag[pos] = 1 at the first (start) / last (end) position of every run of the BWT
__global__ void __launch_bounds__(PB_T) pb_runs_k(const u8 *__restrict__ bwt, u64 n, int at_end, u8 *__restrict__ flag) {
    const u64 i = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (i >= n) return;
    flag[i] = at_end ? (i + 1 == n || bwt[i + 1] != bwt[i]) : (i == 0 || bwt[i] != bwt[i - 1]);
}
__global__ void __launch_bounds__(PB_T) pb_sample_k(const u8 *__restrict__ flag, const u64 *__restrict__ fscan,
                                                    const u8 *__restrict__ sa5, u64 n, u8 *__restrict__ out) {
    const u64 i = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (i >= n || !flag[i]) return;
    const u64 o = fscan[i];
    pb_put5(out, 2 * o, i);                                           // (position, suffix-array value), :170-171
    pb_put5(out, 2 * o + 1, pb_get5(sa5, i));
}
__global__ void __launch_bounds__(PB_T) pb_widen_k(const u8 *__restrict__ f, u64 n, u32 *__restrict__ out) {
    const u64 i = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (i < n) out[i] = f[i];
}

int pfp_dict_alphabet(pfpb200_ctx *ctx, const u8 *d, u64 N, u32 *present) {
    PFP_CUDA(ctx, cudaMemsetAsync(present, 0, 8 * sizeof(u32), ctx->stream));
    pb_alpha_k<<<ctx->sm_count * 8, PB_T, 0, ctx->stream>>>(d, N, present);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

static int pb_bits(u64 v) {
    int b = 1;
    while (b < 64 && (v >> b) != 0) b++;
    return b;
}

static void pb_drop_own_outputs(pfpb200_ctx *ctx) {
    pfp_release_scratch(ctx);
    for (int k = 0; k < 4; k++) {
        void *p = ctx->pb_out[k];
        ctx->pb_out[k] = nullptr;
        if (!p) continue;
        for (size_t i = 0; i < ctx->held.size(); i++)
            if (ctx->held[i] == p) {
                ctx->held[i] = ctx->held.back();
                ctx->held.pop_back();
                ctx->scratch.push_back(p);
                break;
            }
    }
    pfp_release_scratch(ctx);
}

static int pfbwt_device_impl(pfpb200_ctx *ctx, const u8 *d_dict, u64 N, const u32 *d_occ, u64 dwords, const u32 *d_ilist,
                             const u8 *d_bwlast, const u8 *d_bwsai, u64 psize, u32 w, u32 flags,
                             pfpb200_pfbwt_result *res) {
    memset(res, 0, sizeof(*res));
    const bool want_sa = (flags & (PFPB200_PFBWT_SA | PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA)) != 0;
    if (w < 4) return pfp_fail(ctx, PFPB200_E_ARG, "Windows size must be at least 4");                  // pfbwt.cpp:301
    if ((flags & PFPB200_PFBWT_SA) && (flags & (PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA)))
        return pfp_fail(ctx, PFPB200_E_ARG, "You can either require the sampled SA or the full SA, not both");   // :297
    if (N <= 1 + (u64)w) return pfp_fail(ctx, PFPB200_E_ARG, "invalid dictionary file");               // :330
    if (want_sa && !d_bwsai) return pfp_fail(ctx, PFPB200_E_ARG, "suffix array output needs the .bwsai stream");
    if (N >= 0xFFFFFFF0ull || psize >= 0xFFFFFFFEull)
        return pfp_fail(ctx, PFPB200_E_LIMIT, "dictionary of 4 GB or more / more than 2^32-2 words in the parsing");
    PfpEvents evs(3);
    if (!evs.ok) return pfp_fail(ctx, PFPB200_E_CUDA, "cudaEventCreate failed");
    const u32 launches0 = ctx->launches;
    const u32 nb = pfp_blocks(N, PB_T);
    PFP_CUDA(ctx, cudaEventRecord(evs[0], ctx->stream));
    // ---- 1. word structure ---------------------------------------------------------------------------
    u8 *flag = nullptr, *keep = nullptr;
    u32 *wid = nullptr, *wend = nullptr, *istart = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &flag, N));
    PFP_TRY(pfp_alloc_t(ctx, &keep, N));
    PFP_TRY(pfp_alloc_t(ctx, &wid, N));
    PFP_TRY(pfp_alloc_t(ctx, &wend, dwords + 2));
    PFP_TRY(pfp_alloc_t(ctx, &istart, dwords + 1));
    pb_flags_k<<<nb, PB_T, 0, ctx->stream>>>(d_dict, N, flag);
    PFP_LAUNCHED(ctx);
    u32 *d_cnt = reinterpret_cast<u32 *>(&ctx->d_flags[1]);
    PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, flag, wid, N, d_cnt));
    PFP_TRY(pfp_exclusive_scan_u32(ctx, d_occ, istart, dwords, reinterpret_cast<u32 *>(&ctx->d_flags[2])));
    PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[1], &ctx->d_flags[1], 2 * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if ((u32)ctx->h_flags[1] != dwords + 1)                           // get_num_words(), :360, + the final EndOfDict
        return pfp_fail(ctx, PFPB200_E_ARG, "the dictionary holds %u words, .occ %llu", (u32)ctx->h_flags[1] - 1,
                        (unsigned long long)dwords);
    if ((u64)(u32)ctx->h_flags[2] + 1 != psize)                       // assert(last==psize), :384
        return pfp_fail(ctx, PFPB200_E_ARG, "sum of .occ + 1 != size of .ilist");
    pb_wend_k<<<nb, PB_T, 0, ctx->stream>>>(flag, wid, N, wend);
    PFP_LAUNCHED(ctx);
    // ---- 2. suffix sort ----------------------------------------------------------------------------------
    u64 *k0 = nullptr, *k1 = nullptr;
    u32 *v0 = nullptr, *v1 = nullptr, *rank = nullptr, *rs = nullptr, *escan = nullptr;
    u64 *sa = nullptr;
    u32 *slot = nullptr, *slot2 = nullptr, *head = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &sa, N));
    PFP_TRY(pfp_alloc_t(ctx, &rank, N));
    PFP_TRY(pfp_alloc_t(ctx, &k0, N));
    PFP_TRY(pfp_alloc_t(ctx, &k1, N));
    PFP_TRY(pfp_alloc_t(ctx, &v0, N));
    PFP_TRY(pfp_alloc_t(ctx, &v1, N));
    PFP_TRY(pfp_alloc_t(ctx, &rs, N));
    PFP_TRY(pfp_alloc_t(ctx, &escan, N));
    PFP_TRY(pfp_alloc_t(ctx, &slot, N));
    PFP_TRY(pfp_alloc_t(ctx, &slot2, N));
    PFP_TRY(pfp_alloc_t(ctx, &head, N));
    u32 *lim = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &lim, N));
    pb_lim_k<<<nb, PB_T, 0, ctx->stream>>>(wid, wend, N, lim);
    PFP_LAUNCHED(ctx);
    // alphabet of the dictionary -> order-preserving dense codes -> symbols per 64-bit key
    u32 *present = reinterpret_cast<u32 *>(&ctx->d_flags[8]);       // 8 x 32 bits = slots 8..11
    PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[8], 0, 4 * sizeof(u64), ctx->stream));
    pb_alpha_k<<<ctx->sm_count * 8, PB_T, 0, ctx->stream>>>(d_dict, N, present);
    PFP_LAUNCHED(ctx);
    PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[8], &ctx->d_flags[8], 4 * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    PbCodes cd;
    memset(&cd, 0, sizeof(cd));
    u32 sigma = 1;                                              // code 1: the terminators 0x00 and 0x01
    cd.code[0] = cd.code[1] = 1;
    {
        const u32 *pm = reinterpret_cast<const u32 *>(&ctx->h_flags[8]);
        for (u32 c = 2; c < 256; c++)
            if (pm[c >> 5] & (1u << (c & 31))) cd.code[c] = (u8)++sigma;
    }
    const int bs = pb_bits(sigma);                             // bits of a code
    const int h0 = 64 / bs > 32 ? 32 : 64 / bs;                // symbols in the first key
    pb_init_k<<<nb, PB_T, 0, ctx->stream>>>(d_dict, N, cd, h0, bs, k0, v0, slot);
    PFP_LAUNCHED(ctx);
    const int b = pb_bits(N);
    const int kb = b <= 31 ? b : 0;                           // 2 b + 1 key bits fit into 64: old rank, second rank, done bit
    const int sort_bits = kb ? 2 * b + 1 : 64;
    u64 *ks = nullptr;
    u32 *vs = nullptr;
    PFP_TRY(pfp_radix_sort_pairs(ctx, k0, v0, k1, v1, N, 0, h0 * bs, &ks, &vs));
    u32 rounds = 1;
    u64 M = N;
    for (u64 h = (u64)h0;; h *= 2, rounds++) {
        const u32 mb = pfp_blocks(M, PB_T);
        pb_gflags_k<<<mb, PB_T, 0, ctx->stream>>>(ks, M, flag);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, flag, escan, M, nullptr));
        pb_heads_k<<<mb, PB_T, 0, ctx->stream>>>(flag, escan, slot, M, head);
        PFP_LAUNCHED(ctx);
        pb_update_k<<<mb, PB_T, 0, ctx->stream>>>(flag, escan, slot, vs, ks, kb, rounds == 1 ? 1 : 0, head, lim, M, h, sa,
                                                  rank, rs, keep);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, keep, escan, M, d_cnt));
        PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[1], &ctx->d_flags[1], sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        const u64 M2 = (u32)ctx->h_flags[1];
        if (M2 == 0) break;
        if (h >= 2 * N) return pfp_fail(ctx, PFPB200_E_INTERNAL, "pfbwt: prefix doubling did not converge");
        u64 *ko = ks == k0 ? k1 : k0;
        u32 *vo = vs == v0 ? v1 : v0;
        pb_compact_k<<<mb, PB_T, 0, ctx->stream>>>(keep, escan, slot, vs, rs, rank, lim, M, h, kb, slot2, vo, ko);
        PFP_LAUNCHED(ctx);
        { u32 *t = slot; slot = slot2; slot2 = t; }
        M = M2;
        PFP_TRY(pfp_radix_sort_pairs(ctx, ko, vo, ks, vs, M, 0, sort_bits, &ks, &vs));
    }
    PFP_TRY(pfp_free_now(ctx, lim));
    PFP_TRY(pfp_free_now(ctx, k0)); PFP_TRY(pfp_free_now(ctx, k1)); PFP_TRY(pfp_free_now(ctx, v0));
    PFP_TRY(pfp_free_now(ctx, v1)); PFP_TRY(pfp_free_now(ctx, rs)); PFP_TRY(pfp_free_now(ctx, slot));
    PFP_TRY(pfp_free_now(ctx, slot2)); PFP_TRY(pfp_free_now(ctx, head)); PFP_TRY(pfp_free_now(ctx, keep));
    PFP_CUDA(ctx, cudaEventRecord(evs[1], ctx->stream));
    // ---- 3. ranges of the BWT, easy members ------------------------------------------------------------------
    PFP_TRY(pfp_free_now(ctx, rank));                        // the ranks travel with the suffix array from here on
    uint2 *mrec = nullptr;
    u16 *mc = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &mrec, N));
    PFP_TRY(pfp_alloc_t(ctx, &mc, N));
    PbView V{d_dict, sa, wid, wend, d_occ, istart, mrec, mc, N, w};
    u32 *cnt = nullptr, *hcnt = nullptr, *gscan = escan, *first = nullptr;
    u8 *newgrp = flag, *mixed = nullptr;
    u64 *off = nullptr, *hoff = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &cnt, N));
    PFP_TRY(pfp_alloc_t(ctx, &hcnt, N));
    PFP_TRY(pfp_alloc_t(ctx, &off, N + 1));
    PFP_TRY(pfp_alloc_t(ctx, &hoff, N + 1));
    pb_count_k<<<nb, PB_T, 0, ctx->stream>>>(V, cnt, newgrp);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, newgrp, gscan, N, d_cnt));
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, cnt, off, N, &ctx->d_flags[2]));
    PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[1], &ctx->d_flags[1], 2 * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const u64 ngroups = (u32)ctx->h_flags[1], n_bwt = ctx->h_flags[2];
    PFP_TRY(pfp_alloc_t(ctx, &first, ngroups + 1));
    PFP_TRY(pfp_alloc_t(ctx, &mixed, ngroups + 1));
    PFP_CUDA(ctx, cudaMemsetAsync(mixed, 0, ngroups + 1, ctx->stream));
    pb_first_k<<<nb, PB_T, 0, ctx->stream>>>(newgrp, gscan, N, first);
    PFP_LAUNCHED(ctx);
    pb_mixed_k<<<nb, PB_T, 0, ctx->stream>>>(V, newgrp, gscan, first, mixed);
    PFP_LAUNCHED(ctx);
    pb_hard_k<<<nb, PB_T, 0, ctx->stream>>>(cnt, newgrp, gscan, mixed, N, want_sa ? 1 : 0, hcnt);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, hcnt, hoff, N, &ctx->d_flags[3]));
    PFP_CUDA(ctx, cudaMemcpyAsync(&hoff[N], &ctx->d_flags[3], sizeof(u64), cudaMemcpyDeviceToDevice, ctx->stream));
    PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[3], &ctx->d_flags[3], sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const u64 n_hard = ctx->h_flags[3];
    u8 *bwt = nullptr, *sa5 = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &bwt, n_bwt, true));
    ctx->pb_out[0] = bwt;
    if (want_sa) {
        PFP_TRY(pfp_alloc_t(ctx, &sa5, n_bwt * PFP_IBYTES, true));
        ctx->pb_out[1] = sa5;
    }
    // (a member with more than PB_BIG occurrences contributes > PB_BIG chars: at most n_bwt / PB_BIG of them)
    const u32 big_cap = (u32)(n_bwt / PB_BIG + 1);
    u32 *big = nullptr, *big_n = reinterpret_cast<u32 *>(&ctx->d_flags[6]);
    PFP_TRY(pfp_alloc_t(ctx, &big, big_cap));
    PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[6], 0, sizeof(u64), ctx->stream));
    pb_easy_k<<<nb, PB_T, 0, ctx->stream>>>(V, cnt, hcnt, off, d_ilist, d_bwlast, d_bwsai, bwt, sa5, big, big_n, big_cap);
    PFP_LAUNCHED(ctx);
    pb_easy_big_k<<<ctx->sm_count * 8, PB_T, 0, ctx->stream>>>(V, big, big_n, big_cap, cnt, off, d_ilist, d_bwlast, d_bwsai, bwt, sa5);
    PFP_LAUNCHED(ctx);
    // ---- 4. hard members: the merge of the ilist cursors as a sort, in batches ------------------------------------
    if (n_hard) {
        const u64 cap = n_hard < PB_BATCH ? n_hard : PB_BATCH;
        u64 *hk0 = nullptr, *hk1 = nullptr;
        u32 *hv0 = nullptr, *hv1 = nullptr;
        u64 ka = 0, ea = 0;                                    // (a single group may exceed the batch: the buffers grow)
        u64 buf = 0;
        while (ka < N && ea < n_hard) {
            pb_batch_k<<<1, 1, 0, ctx->stream>>>(hoff, gscan, newgrp, first, ngroups, ka, N, cap, &ctx->d_flags[4]);
            PFP_LAUNCHED(ctx);
            PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[4], &ctx->d_flags[4], 4 * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
            PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            const u64 kb = ctx->h_flags[4], eb = ctx->h_flags[5], ng = ctx->h_flags[7];
            const u32 g0 = (u32)ctx->h_flags[6];
            const u64 ne = eb - ea;
            if (ne >= 0xFFFFFFFEull) return pfp_fail(ctx, PFPB200_E_LIMIT, "pfbwt: one group of equal suffixes with 2^32 occurrences");
            if (ne) {
                if (ne > buf) {
                    if (hk0) { PFP_TRY(pfp_free_now(ctx, hk0)); PFP_TRY(pfp_free_now(ctx, hk1)); PFP_TRY(pfp_free_now(ctx, hv0)); PFP_TRY(pfp_free_now(ctx, hv1)); }
                    buf = ne > cap ? ne : cap;
                    PFP_TRY(pfp_alloc_t(ctx, &hk0, buf));
                    PFP_TRY(pfp_alloc_t(ctx, &hk1, buf));
                    PFP_TRY(pfp_alloc_t(ctx, &hv0, buf));
                    PFP_TRY(pfp_alloc_t(ctx, &hv1, buf));
                }
                pb_gen_k<<<pfp_blocks(kb - ka, PB_T), PB_T, 0, ctx->stream>>>(V, hcnt, hoff, gscan, newgrp, d_ilist, ka, kb, ea, g0, hk0, hv0);
                PFP_LAUNCHED(ctx);
                u64 *sk = nullptr;
                u32 *sv = nullptr;
                PFP_TRY(pfp_radix_sort_pairs(ctx, hk0, hv0, hk1, hv1, ne, 0, 32 + pb_bits(ng), &sk, &sv));
                pb_scatter_k<<<pfp_blocks(ne, PB_T), PB_T, 0, ctx->stream>>>(V, sk, sv, ne, ea, g0, first, off, hoff, d_bwsai, bwt, sa5);
                PFP_LAUNCHED(ctx);
            }
            ka = kb;
            ea = eb;
        }
    }
    // ---- sampled suffix array: the entries at the starts / ends of the runs ------------------------------------------
    u8 *ssa = nullptr, *esa = nullptr;
    u64 n_ssa = 0, n_esa = 0;
    for (int at_end = 0; at_end < 2; at_end++) {
        if (!(flags & (at_end ? PFPB200_PFBWT_ESA : PFPB200_PFBWT_SSA))) continue;
        u8 *rf = nullptr;
        u32 *rw = nullptr;
        u64 *rscan = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &rf, n_bwt));
        PFP_TRY(pfp_alloc_t(ctx, &rw, n_bwt));
        PFP_TRY(pfp_alloc_t(ctx, &rscan, n_bwt));
        const u32 bb = pfp_blocks(n_bwt, PB_T);
        pb_runs_k<<<bb, PB_T, 0, ctx->stream>>>(bwt, n_bwt, at_end, rf);
        PFP_LAUNCHED(ctx);
        pb_widen_k<<<bb, PB_T, 0, ctx->stream>>>(rf, n_bwt, rw);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, rw, rscan, n_bwt, &ctx->d_flags[5]));
        PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[5], &ctx->d_flags[5], sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        const u64 nr = ctx->h_flags[5];
        u8 *outp = nullptr;
        PFP_TRY(pfp_alloc_t(ctx, &outp, nr * 2 * PFP_IBYTES, true));
        pb_sample_k<<<bb, PB_T, 0, ctx->stream>>>(rf, rscan, sa5, n_bwt, outp);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_free_now(ctx, rf)); PFP_TRY(pfp_free_now(ctx, rw)); PFP_TRY(pfp_free_now(ctx, rscan));
        if (at_end) { esa = outp; n_esa = nr; ctx->pb_out[3] = outp; } else { ssa = outp; n_ssa = nr; ctx->pb_out[2] = outp; }
    }
    PFP_CUDA(ctx, cudaEventRecord(evs[2], ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    res->bwt = bwt;
    res->n_bwt = n_bwt;
    if (flags & PFPB200_PFBWT_SA) {                          // the .sa file has no entry for the first BWT char (:157-163)
        res->sa = sa5 + PFP_IBYTES;
        res->n_sa = n_bwt - 1;
    }
    res->ssa = ssa; res->n_ssa = n_ssa;
    res->esa = esa; res->n_esa = n_esa;
    res->dict_bytes = N; res->dict_words = dwords; res->parse_size = psize;
    res->easy = n_bwt - n_hard; res->hard = n_hard;
    res->rounds = rounds;
    res->launches = ctx->launches - launches0;
    cudaEventElapsedTime(&res->ms_sa, evs[0], evs[1]);
    cudaEventElapsedTime(&res->ms_fill, evs[1], evs[2]);
    res->ms_total = res->ms_sa + res->ms_fill;
    return PFPB200_OK;
}

extern "C" int pfpb200_pfbwt_device(pfpb200_ctx *ctx, const uint8_t *d_dict, uint64_t dict_bytes, const uint32_t *d_occ,
                                    uint64_t n_words, const uint32_t *d_ilist, const uint8_t *d_bwlast,
                                    const uint8_t *d_bwsai, uint64_t parse_size, uint32_t w, uint32_t flags,
                                    pfpb200_pfbwt_result *res) {
    if (!ctx || !d_dict || !d_occ || !d_ilist || !d_bwlast || !res) return PFPB200_E_ARG;
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    pb_drop_own_outputs(ctx);
    ctx->err[0] = 0;
    PFP_CUDA(ctx, cudaMemsetAsync(ctx->d_flags, 0, 8 * sizeof(u64), ctx->stream));
    const int rc = pfbwt_device_impl(ctx, d_dict, dict_bytes, d_occ, n_words, d_ilist, d_bwlast, d_bwsai, parse_size, w,
                                     flags, res);
    pfp_release_scratch(ctx);
    return rc;
}

static int pb_file_to_held(pfpb200_ctx *ctx, const char *base, const char *ext, u64 unit, void **d, u64 *count) {
    char name[4096];
    snprintf(name, sizeof(name), "%s.%s", base, ext);
    const int fd = open(name, O_RDONLY);
    if (fd < 0) return pfp_fail(ctx, PFPB200_E_IO, "cannot open %s: %s", name, strerror(errno));
    struct stat st;
    if (fstat(fd, &st) != 0) { close(fd); return pfp_fail(ctx, PFPB200_E_IO, "cannot stat %s", name); }
    const u64 bytes = (u64)st.st_size;
    if (bytes % unit != 0) { close(fd); return pfp_fail(ctx, PFPB200_E_ARG, "invalid %s file", ext); }   // :348,:366
    int rc = pfp_alloc(ctx, d, bytes, true);
    if (rc == PFPB200_OK && bytes) rc = pfp_file_to_device(ctx, fd, 0, bytes, static_cast<u8 *>(*d));
    close(fd);
    *count = bytes / unit;
    return rc;
}

// `pfbwt.x -w W [-S | -s -e] <basename>`: .dict .occ .ilist .bwlast [.bwsai] -> .bwt [.sa | .ssa .esa]
extern "C" int pfpb200_pfbwt_file(pfpb200_ctx *ctx, const char *basename, uint32_t w, uint32_t flags,
                                  pfpb200_pfbwt_result *res) {
    if (!ctx || !basename || !res) return PFPB200_E_ARG;
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    pfp_release_scratch(ctx);
    pfp_release_held(ctx);
    ctx->err[0] = 0;
    void *dict = nullptr, *occ = nullptr, *ilist = nullptr, *bwlast = nullptr, *bwsai = nullptr;
    u64 N = 0, dwords = 0, psize = 0, nl = 0, ns = 0;
    PFP_TRY(pb_file_to_held(ctx, basename, "dict", 1, &dict, &N));
    PFP_TRY(pb_file_to_held(ctx, basename, "occ", 4, &occ, &dwords));
    PFP_TRY(pb_file_to_held(ctx, basename, "ilist", 4, &ilist, &psize));
    PFP_TRY(pb_file_to_held(ctx, basename, "bwlast", 1, &bwlast, &nl));
    if (nl != psize) return pfp_fail(ctx, PFPB200_E_ARG, ".bwlast holds %llu bytes, .ilist %llu entries",
                                     (unsigned long long)nl, (unsigned long long)psize);
    if (flags & (PFPB200_PFBWT_SA | PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA)) {
        PFP_TRY(pb_file_to_held(ctx, basename, "bwsai", PFP_IBYTES, &bwsai, &ns));
        if (ns != psize) return pfp_fail(ctx, PFPB200_E_ARG, "bwsa info read");
    }
    int rc = pfpb200_pfbwt_device(ctx, static_cast<u8 *>(dict), N, static_cast<u32 *>(occ), dwords, static_cast<u32 *>(ilist),
                                  static_cast<u8 *>(bwlast), static_cast<u8 *>(bwsai), psize, w, flags, res);
    char name[4096];
    auto put = [&](const char *ext, const void *p, u64 bytes) {
        if (rc != PFPB200_OK) return;
        snprintf(name, sizeof(name), "%s.%s", basename, ext);
        rc = pfp_device_to_file(ctx, name, p, bytes);
    };
    put("bwt", res->bwt, res->n_bwt);
    if (flags & PFPB200_PFBWT_SA) put("sa", res->sa, res->n_sa * PFP_IBYTES);
    if (flags & PFPB200_PFBWT_SSA) put("ssa", res->ssa, res->n_ssa * 2 * PFP_IBYTES);
    if (flags & PFPB200_PFBWT_ESA) put("esa", res->esa, res->n_esa * 2 * PFP_IBYTES);
    pfp_release_scratch(ctx);
    return rc;
}
