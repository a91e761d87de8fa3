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
//
// Steps 1, 3 and 4 serve the sharded path too (pfp_pfbwt_multi.cu, pfp_multi.cu): the input reader
// and argument checks, the word structure (pb_words: word ends, no per-position array), the group heads
// of a doubling round, the plan of the emission on a slice of sorted slots (pb_plan), its windows written
// to the files (pb_write_windows) and the run samples (pb_samples).  The emission reads the sort's output
// only through a slot reader.  Step 2 is this file's own: 32-bit packed ranks and positions, N < 2^32 - 16,
// and the word of every position (pb_word_ids); the sharded sort partitions the suffixes, keeps 64-bit
// ranks and finds the words of its own suffixes in the word ends.
#include "pfp_common.cuh"
#include "pfp_stages.cuh"
#include <errno.h>
#include <fcntl.h>
#include <stdlib.h>
#include <sys/stat.h>
#include <time.h>
#include <unistd.h>

constexpr u64 PB_BATCH = (u64)1 << 30;          // occurrences sorted at once in the hard groups
constexpr u32 PB_BIG = 512;                     // easy members with more occurrences get a CTA instead of a thread

// Device bytes that the output of c BWT chars with at most h hard occurrences takes, from the allocations
// of pb_window and pb_samples: per char its byte and, with -S / -s / -e, its 5-byte SA value; then, one
// after the other, the merge of the hard occurrences (u64 key and u32 value, twice for the sort's
// ping-pong: 24, and the sort's digit histograms, 256 u32 per 2048 pairs: 0.5; at most one batch of
// PB_BATCH at a time) and, with -s / -e, the run samples (u32 flag and u64 scan: 12, and at most one
// 10-byte sample per char).  One byte per char on top covers the easy members' CTA list (4 B per 512
// chars) and the scans' tile sums.  A window holds at most min(c, h) hard occurrences.
constexpr u64 PB_MERGE_BYTES = 2 * (8 + 4) + 1;
constexpr u64 PB_SAMPLE_BYTES = 4 + 8 + 2 * PFP_IBYTES;
static u64 pb_out_bytes(u64 c, u64 h, u32 flags) {
    const bool want_sa = (flags & (PFPB200_PFBWT_SA | PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA)) != 0;
    const bool samples = (flags & (PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA)) != 0;
    u64 m = h < c ? h : c;
    if (m > PB_BATCH) m = PB_BATCH;
    const u64 merge = PB_MERGE_BYTES * m, sample = samples ? PB_SAMPLE_BYTES * c : 0;
    return c * (2 + (want_sa ? PFP_IBYTES : 0)) + (merge > sample ? merge : sample);
}

__global__ void __launch_bounds__(PB_T) pb_flags_k(const u8 *__restrict__ d, u64 N, u8 *__restrict__ flag) {
    const u64 t = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (t < N) flag[t] = pb_term(d[t]) ? 1 : 0;
}

// wend[k] = position of the k-th terminator, over the chunk [c0, c0 + n) whose first terminator is
// number k0; scan[t] = terminators of the chunk before t
__global__ void __launch_bounds__(PB_T) pb_wend_k(const u8 *__restrict__ flag, const u32 *__restrict__ scan, u64 n,
                                                  u64 c0, u64 k0, u64 *__restrict__ wend) {
    const u64 t = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (t < n && flag[t]) wend[k0 + scan[t]] = c0 + t;
}

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

// round 1: every position by its first key -- with dense codes the doubling runs at depths 21, 42, 84,
// ... on DNA instead of 8, 16, 32, ..., and a third of its work is gone
__global__ void __launch_bounds__(PB_T) pb_init_k(const u8 *__restrict__ d, u64 N, PbCodes cd, int h0, int bs,
                                                  u64 *__restrict__ key, u32 *__restrict__ val, u32 *__restrict__ slot) {
    __shared__ u8 code[256];
    code[threadIdx.x] = cd.code[threadIdx.x];                        // PB_T = 256
    __syncthreads();
    const u64 t = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (t >= N) return;
    key[t] = pb_first_key(d, N, code, h0, bs, t);
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
__global__ void __launch_bounds__(PB_T) pb_lim_k(const u32 *__restrict__ wid, const u64 *__restrict__ wend, u64 N,
                                                 u32 *__restrict__ lim) {
    const u64 t = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (t < N) lim[t] = (u32)wend[wid[t]];
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

// ---- the walk over the sorted suffixes (both paths) -----------------------------------------------
struct PbView {
    const u8 *d;
    const u32 *occ, *istart;
    const u64 *wend;
    uint2 *mrec;                // per slot, written by pb_count_k: {word, suffix length}
    u16 *mc;                    // per slot: char in front | whole word << 8 | counts << 9
    u64 N;                      // slots
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
template <class Slots>
__global__ void __launch_bounds__(PB_T) pb_count_k(PbView v, Slots sl, u32 *__restrict__ cnt, u8 *__restrict__ newgrp) {
    const u64 k = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k >= v.N) return;
    const auto s = sl.pos(k);
    newgrp[k] = (k == 0 || sl.grp(k) != sl.grp(k - 1)) ? 1 : 0;
    u32 word = 0, len = 0, n = 0, m = 0;
    if (!pb_term(v.d[s])) {
        word = sl.word(k);
        len = (u32)(v.wend[word] - s);
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

// members that need no merge: a whole word (chars from .bwlast, :155-203), or one char for all; slots
// [ka, kb) of a window whose chars start at BWT position base
__global__ void __launch_bounds__(PB_T) pb_easy_k(PbView v, const u32 *__restrict__ cnt, const u32 *__restrict__ hcnt,
                                                  const u64 *__restrict__ off, const u32 *__restrict__ ilist,
                                                  const u8 *__restrict__ bwlast, const u8 *__restrict__ bwsai,
                                                  u64 ka, u64 kb, u64 base, u8 *__restrict__ bwt, u8 *__restrict__ sa5,
                                                  u32 *__restrict__ big, u32 *__restrict__ big_n, u32 big_cap) {
    const u64 k = ka + (u64)blockIdx.x * PB_T + threadIdx.x;
    if (k >= kb || cnt[k] == 0 || hcnt[k] != 0) return;
    u32 word, len; bool full; u8 c;
    pb_member(v, k, word, len, full, c);
    const u32 n = cnt[k];
    if (n > PB_BIG) {                                                // a word with many occurrences: one CTA each, below
        const u32 i = atomicAdd(big_n, 1u);
        if (i < big_cap) big[i] = (u32)k;
        return;
    }
    const u64 o = off[k] - base;
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
                                                      const u8 *__restrict__ bwsai, u64 base, u8 *__restrict__ bwt,
                                                      u8 *__restrict__ sa5) {
    const u32 nbig = min(*big_n, big_cap);
    for (u32 b = blockIdx.x; b < nbig; b += gridDim.x) {
        const u64 k = big[b];
        u32 word, len; bool full; u8 c;
        pb_member(v, k, word, len, full, c);
        const u32 n = cnt[k];
        const u64 o = off[k] - base;
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

// the sorted occurrences of a batch to their BWT positions, less the window's first position base
__global__ void __launch_bounds__(PB_T) pb_scatter_k(PbView v, const u64 *__restrict__ key, const u32 *__restrict__ val,
                                                     u64 ne, u64 e0, u32 g0, const u32 *__restrict__ first,
                                                     const u64 *__restrict__ off, const u64 *__restrict__ hoff,
                                                     const u8 *__restrict__ bwsai, u64 base, u8 *__restrict__ bwt,
                                                     u8 *__restrict__ sa5) {
    const u64 e = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (e >= ne) return;
    const u64 kk = key[e];
    const u32 k = val[e], f = first[(u32)(kk >> 32) + g0];
    const u64 pos = off[f] - base + (e0 + e - hoff[f]);
    u32 word, len; bool full; u8 c;
    pb_member(v, k, word, len, full, c);
    bwt[pos] = c;
    if (sa5) pb_put5(sa5, pos, pb_get5(bwsai, (u32)kk) - len);
}

// The next run of whole groups of slots [ka, end) (end: a group start or the last slot + 1) that fits
// into `cap` items of a scan acc[0..end] (non-decreasing): the hard occurrences of a merge batch (hoff),
// or the chars of a window (off).  out = {kb, acc[kb], group of slot ka, groups in [ka, kb)}, at least one
// group: a group larger than cap is taken whole.
__global__ void pb_batch_k(const u64 *__restrict__ acc, const u32 *__restrict__ gscan, const u8 *__restrict__ newgrp,
                           const u32 *__restrict__ first, u64 ngroups, u64 ka, u64 end, u64 cap, u64 *__restrict__ out) {
    const u64 target = acc[ka] + cap;
    u64 kb = end;
    if (acc[end] > target) {
        u64 a = ka, b = end;                                     // first index with acc > target
        while (a < b) {
            const u64 m = (a + b) >> 1;
            if (acc[m] <= target) a = m + 1; else b = m;
        }
        const u64 kl = a - 1;                                    // >= ka: acc[ka] <= target
        const u64 g = gscan[kl] + newgrp[kl] - 1u;
        kb = first[g];
        if (kb <= ka) kb = g + 1 < ngroups ? first[g + 1] : end;   // one group larger than cap: take it whole
    }
    const u64 ga = gscan[ka] + newgrp[ka] - 1u;
    out[0] = kb;
    out[1] = acc[kb];
    out[2] = ga;
    out[3] = gscan[kb - 1] + newgrp[kb - 1] - ga;                // kb > ka
}

// sampled suffix array: flag[i] = 1 at the first (start) / last (end) position of every run of the BWT;
// prev / next = the chars in front of / behind bwt[0, n) (-1: none)
__global__ void __launch_bounds__(PB_T) pb_runs_k(const u8 *__restrict__ bwt, u64 n, int at_end, int prev, int next,
                                                  u32 *__restrict__ flag) {
    const u64 i = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (i >= n) return;
    bool f;
    if (at_end) f = i + 1 == n ? (next < 0 || bwt[i] != (u8)next) : bwt[i + 1] != bwt[i];
    else f = i == 0 ? (prev < 0 || bwt[0] != (u8)prev) : bwt[i] != bwt[i - 1];
    flag[i] = f ? 1u : 0u;
}
__global__ void __launch_bounds__(PB_T) pb_sample_k(const u32 *__restrict__ flag, const u64 *__restrict__ fscan,
                                                    const u8 *__restrict__ sa5, u64 n, u64 off, u8 *__restrict__ out) {
    const u64 i = (u64)blockIdx.x * PB_T + threadIdx.x;
    if (i >= n || !flag[i]) return;
    const u64 o = fscan[i];
    pb_put5(out, 2 * o, off + i);                                     // (BWT position, suffix-array value), :170-171
    pb_put5(out, 2 * o + 1, pb_get5(sa5, i));
}

// ---- host steps shared by both paths ----------------------------------------------------------------------
const char *pb_arg_error(u32 w, u32 flags) {
    if (w < 4) return "Windows size must be at least 4";                                          // pfbwt.cpp:301
    if ((flags & PFPB200_PFBWT_SA) && (flags & (PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA)))
        return "You can either require the sampled SA or the full SA, not both";                   // :297
    return nullptr;
}

int pb_read_file(pfpb200_ctx *ctx, const char *base, int k, void **d, u64 *count) {
    static const char *const ext[5] = {"dict", "occ", "ilist", "bwlast", "bwsai"};
    char name[4096];
    snprintf(name, sizeof(name), "%s.%s", base, ext[k]);
    const int fd = open(name, O_RDONLY);
    if (fd < 0) return pfp_fail(ctx, PFPB200_E_IO, "cannot open %s: %s", name, strerror(errno));
    struct stat st;
    if (fstat(fd, &st) != 0) { close(fd); return pfp_fail(ctx, PFPB200_E_IO, "cannot stat %s", name); }
    const u64 bytes = (u64)st.st_size;
    if (bytes % PB_UNIT[k] != 0) { close(fd); return pfp_fail(ctx, PFPB200_E_ARG, "invalid %s file", ext[k]); }   // :348,:366
    int rc = pfp_alloc(ctx, d, bytes, true);
    if (rc == PFPB200_OK && bytes) rc = pfp_file_to_device(ctx, fd, 0, bytes, static_cast<u8 *>(*d));
    close(fd);
    *count = bytes / PB_UNIT[k];
    return rc;
}

int pb_read_inputs(pfpb200_ctx *ctx, const char *base, u32 flags, void *in[5], u64 n[5]) {
    for (int k = 0; k < 4; k++) PFP_TRY(pb_read_file(ctx, base, k, &in[k], &n[k]));
    if (n[3] != n[2])
        return pfp_fail(ctx, PFPB200_E_ARG, ".bwlast holds %llu bytes, .ilist %llu entries", (unsigned long long)n[3],
                        (unsigned long long)n[2]);
    if (flags & (PFPB200_PFBWT_SA | PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA)) {
        PFP_TRY(pb_read_file(ctx, base, 4, &in[4], &n[4]));
        if (n[4] != n[2]) return pfp_fail(ctx, PFPB200_E_ARG, "bwsa info read");
    }
    return PFPB200_OK;
}

int pb_sync_read(pfpb200_ctx *ctx, int slot, int n) {
    PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[slot], &ctx->d_flags[slot], n * sizeof(u64), cudaMemcpyDeviceToHost,
                                  ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return PFPB200_OK;
}

// terminator flags -> word ends, chunk by chunk; .occ -> first .ilist entry of every word; the
// dictionary's alphabet -> dense codes, symbols per 64-bit first key
int pb_words(pfpb200_ctx *ctx, const PbInput &in, PbWords *W) {
    const u64 N = in.N, chunk = N < PB_CHUNK ? N : PB_CHUNK;
    PFP_TRY(pfp_alloc_t(ctx, &W->wend, in.dwords + 2));
    PFP_TRY(pfp_alloc_t(ctx, &W->istart, in.dwords + 1));
    u8 *flag = nullptr;
    u32 *scan = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &flag, chunk));
    PFP_TRY(pfp_alloc_t(ctx, &scan, chunk));
    u64 words = 0;                                                    // terminators before the chunk
    for (u64 c0 = 0; c0 < N; c0 += chunk) {
        const u64 n = N - c0 < chunk ? N - c0 : chunk;
        PB_LAUNCH(ctx, n, pb_flags_k, in.d + c0, n, flag);
        PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, flag, scan, n, reinterpret_cast<u32 *>(&ctx->d_flags[1])));
        PFP_TRY(pb_sync_read(ctx, 1, 1));
        const u64 nt = (u32)ctx->h_flags[1];
        if (words + nt <= in.dwords + 1) PB_LAUNCH(ctx, n, pb_wend_k, flag, scan, n, c0, words, W->wend);
        words += nt;                                                  // (too many: reported below)
    }
    PFP_TRY(pfp_free_now(ctx, flag));
    PFP_TRY(pfp_free_now(ctx, scan));
    if (words != in.dwords + 1)                                       // get_num_words(), :360, + the final EndOfDict
        return pfp_fail(ctx, PFPB200_E_ARG, "the dictionary holds %u words, .occ %llu", (u32)words - 1,
                        (unsigned long long)in.dwords);
    PFP_TRY(pfp_exclusive_scan_u32(ctx, in.occ, W->istart, in.dwords, reinterpret_cast<u32 *>(&ctx->d_flags[2])));
    PFP_TRY(pb_sync_read(ctx, 2, 1));
    if ((u64)(u32)ctx->h_flags[2] + 1 != in.psize)                    // assert(last==psize), :384
        return pfp_fail(ctx, PFPB200_E_ARG, "sum of .occ + 1 != size of .ilist");
    u32 *present = reinterpret_cast<u32 *>(&ctx->d_flags[8]);       // 8 x 32 bits = slots 8..11
    PFP_CUDA(ctx, cudaMemsetAsync(present, 0, 8 * sizeof(u32), ctx->stream));
    pb_alpha_k<<<ctx->sm_count * 8, PB_T, 0, ctx->stream>>>(in.d, N, present);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pb_sync_read(ctx, 8, 4));
    memset(&W->cd, 0, sizeof(W->cd));
    u32 sigma = 1;                                              // code 1: the terminators 0x00 and 0x01
    W->cd.code[0] = W->cd.code[1] = 1;
    const u32 *pm = reinterpret_cast<const u32 *>(&ctx->h_flags[8]);
    for (u32 c = 2; c < 256; c++)
        if (pm[c >> 5] & (1u << (c & 31))) W->cd.code[c] = (u8)++sigma;
    W->bs = pb_bits(sigma);
    W->h0 = 64 / W->bs > 32 ? 32 : 64 / W->bs;
    return PFPB200_OK;
}

// wid[t] = terminators before t = the word of position t (N < 2^32 - 16 on the one-GPU path)
int pb_word_ids(pfpb200_ctx *ctx, const PbInput &in, PbWords *W) {
    u8 *flag = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &flag, in.N));
    PFP_TRY(pfp_alloc_t(ctx, &W->wid, in.N));
    PB_LAUNCH(ctx, in.N, pb_flags_k, in.d, in.N, flag);
    PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, flag, W->wid, in.N, nullptr));
    return pfp_free_now(ctx, flag);
}

// the plan over all n slots: count -> scans -> first / mixed / hard
template <class Slots>
int pb_plan(pfpb200_ctx *ctx, const PbInput &in, const PbWords &W, Slots sl, u64 n, u8 *newgrp, u32 *gscan, PbPlan *P) {
    const bool want_sa = (in.flags & (PFPB200_PFBWT_SA | PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA)) != 0;
    P->n = n;
    P->newgrp = newgrp;
    P->gscan = gscan;
    PFP_TRY(pfp_alloc_t(ctx, &P->mrec, n));
    PFP_TRY(pfp_alloc_t(ctx, &P->mc, n));
    PFP_TRY(pfp_alloc_t(ctx, &P->cnt, n));
    PFP_TRY(pfp_alloc_t(ctx, &P->hcnt, n));
    PFP_TRY(pfp_alloc_t(ctx, &P->off, n + 1));
    PFP_TRY(pfp_alloc_t(ctx, &P->hoff, n + 1));
    const PbView V{in.d, in.occ, W.istart, W.wend, P->mrec, P->mc, n, in.w};
    PB_LAUNCH(ctx, n, pb_count_k<Slots>, V, sl, P->cnt, newgrp);
    PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, newgrp, gscan, n, reinterpret_cast<u32 *>(&ctx->d_flags[1])));
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, P->cnt, P->off, n, &ctx->d_flags[2]));
    PFP_CUDA(ctx, cudaMemcpyAsync(&P->off[n], &ctx->d_flags[2], sizeof(u64), cudaMemcpyDeviceToDevice, ctx->stream));
    PFP_TRY(pb_sync_read(ctx, 1, 2));
    const u64 ngroups = P->ngroups = (u32)ctx->h_flags[1];
    P->chars = ctx->h_flags[2];
    PFP_TRY(pfp_alloc_t(ctx, &P->first, ngroups + 1));
    PFP_TRY(pfp_alloc_t(ctx, &P->mixed, ngroups + 1));
    PFP_CUDA(ctx, cudaMemsetAsync(P->mixed, 0, ngroups + 1, ctx->stream));
    PB_LAUNCH(ctx, n, pb_first_k, newgrp, gscan, n, P->first);
    PB_LAUNCH(ctx, n, pb_mixed_k, V, newgrp, gscan, P->first, P->mixed);
    PB_LAUNCH(ctx, n, pb_hard_k, P->cnt, newgrp, gscan, P->mixed, n, want_sa ? 1 : 0, P->hcnt);
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, P->hcnt, P->hoff, n, &ctx->d_flags[3]));
    PFP_CUDA(ctx, cudaMemcpyAsync(&P->hoff[n], &ctx->d_flags[3], sizeof(u64), cudaMemcpyDeviceToDevice, ctx->stream));
    PFP_TRY(pb_sync_read(ctx, 3, 1));
    P->n_hard = ctx->h_flags[3];
    return PFPB200_OK;
}
int pb_window_end(pfpb200_ctx *ctx, const PbPlan &P, u64 ka, u64 cap, u64 *kb, u64 *chars_end) {
    pb_batch_k<<<1, 1, 0, ctx->stream>>>(P.off, P.gscan, P.newgrp, P.first, P.ngroups, ka, P.n, cap, &ctx->d_flags[12]);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pb_sync_read(ctx, 12, 2));
    *kb = ctx->h_flags[12];
    *chars_end = ctx->h_flags[13];
    return PFPB200_OK;
}

// easy / easy-big -> hard batches, over the slots [ka, kb) of one window
int pb_window(pfpb200_ctx *ctx, const PbInput &in, const PbWords &W, const PbPlan &P, u64 ka, u64 kb, u64 hcap,
              bool held, PbEmit *E) {
    const bool want_sa = (in.flags & (PFPB200_PFBWT_SA | PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA)) != 0;
    const PbView V{in.d, in.occ, W.istart, W.wend, P.mrec, P.mc, P.n, in.w};
    // the window's first and last char and hard occurrence
    u64 *h = &ctx->h_flags[12];
    PFP_CUDA(ctx, cudaMemcpyAsync(&h[0], &P.off[ka], sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaMemcpyAsync(&h[1], &P.off[kb], sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaMemcpyAsync(&h[2], &P.hoff[ka], sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaMemcpyAsync(&h[3], &P.hoff[kb], sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const u64 base = h[0], chars = h[1] - h[0], e_end = h[3];
    u64 ea = h[2];
    E->base = base;
    E->chars = chars;
    E->n_hard = e_end - ea;
    E->ngroups = P.ngroups;
    PFP_TRY(pfp_alloc_t(ctx, &E->bwt, chars, held));
    if (held) ctx->pb_out[0] = E->bwt;
    if (want_sa) {
        PFP_TRY(pfp_alloc_t(ctx, &E->sa5, chars * PFP_IBYTES, held));
        if (held) ctx->pb_out[1] = E->sa5;
    }
    u8 *bwt = E->bwt, *sa5 = E->sa5;
    // (a member with more than PB_BIG occurrences contributes > PB_BIG chars: at most chars / PB_BIG of them)
    const u32 big_cap = (u32)(chars / PB_BIG + 1);
    u32 *big = nullptr, *big_n = reinterpret_cast<u32 *>(&ctx->d_flags[6]);
    PFP_TRY(pfp_alloc_t(ctx, &big, big_cap));
    PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[6], 0, sizeof(u64), ctx->stream));
    PB_LAUNCH(ctx, kb - ka, pb_easy_k, V, P.cnt, P.hcnt, P.off, in.ilist, in.bwlast, in.bwsai, ka, kb, base, bwt, sa5, big,
              big_n, big_cap);
    if (kb > ka) {
        pb_easy_big_k<<<ctx->sm_count * 8, PB_T, 0, ctx->stream>>>(V, big, big_n, big_cap, P.cnt, P.off, in.ilist,
                                                                   in.bwlast, in.bwsai, base, bwt, sa5);
        PFP_LAUNCHED(ctx);
    }
    // ---- hard members: the merge of the ilist cursors as a sort, in batches ----
    if (E->n_hard) {
        const u64 lim = hcap < PB_BATCH ? hcap : PB_BATCH;
        const u64 cap = lim ? lim : 1;
        u64 *hk0 = nullptr, *hk1 = nullptr;
        u32 *hv0 = nullptr, *hv1 = nullptr;
        u64 k = ka;                                            // (a single group may exceed the batch: the buffers grow)
        u64 buf = 0;
        while (k < kb && ea < e_end) {
            pb_batch_k<<<1, 1, 0, ctx->stream>>>(P.hoff, P.gscan, P.newgrp, P.first, P.ngroups, k, kb, cap, &ctx->d_flags[4]);
            PFP_LAUNCHED(ctx);
            PFP_TRY(pb_sync_read(ctx, 4, 4));
            const u64 k2 = ctx->h_flags[4], eb = ctx->h_flags[5], ng = ctx->h_flags[7];
            const u32 g0 = (u32)ctx->h_flags[6];
            const u64 ne = eb - ea;
            if (ne >= 0xFFFFFFFEull) return pfp_fail(ctx, PFPB200_E_LIMIT, "pfbwt: one group of equal suffixes with 2^32 occurrences");
            if (ne) {
                if (ne > buf) {
                    if (hk0) { PFP_TRY(pfp_free_now(ctx, hk0)); PFP_TRY(pfp_free_now(ctx, hk1)); PFP_TRY(pfp_free_now(ctx, hv0)); PFP_TRY(pfp_free_now(ctx, hv1)); }
                    buf = ne > cap ? ne : cap;
                    if (buf > E->n_hard) buf = E->n_hard;
                    PFP_TRY(pfp_alloc_t(ctx, &hk0, buf));
                    PFP_TRY(pfp_alloc_t(ctx, &hk1, buf));
                    PFP_TRY(pfp_alloc_t(ctx, &hv0, buf));
                    PFP_TRY(pfp_alloc_t(ctx, &hv1, buf));
                }
                pb_gen_k<<<pfp_blocks(k2 - k, PB_T), PB_T, 0, ctx->stream>>>(V, P.hcnt, P.hoff, P.gscan, P.newgrp, in.ilist, k, k2, ea, g0, hk0, hv0);
                PFP_LAUNCHED(ctx);
                u64 *sk = nullptr;
                u32 *sv = nullptr;
                PFP_TRY(pfp_radix_sort_pairs(ctx, hk0, hv0, hk1, hv1, ne, 0, 32 + pb_bits(ng), &sk, &sv));
                pb_scatter_k<<<pfp_blocks(ne, PB_T), PB_T, 0, ctx->stream>>>(V, sk, sv, ne, ea, g0, P.first, P.off, P.hoff,
                                                                             in.bwsai, base, bwt, sa5);
                PFP_LAUNCHED(ctx);
            }
            k = k2;
            ea = eb;
        }
        PFP_TRY(pfp_free_now(ctx, hk0)); PFP_TRY(pfp_free_now(ctx, hk1));
        PFP_TRY(pfp_free_now(ctx, hv0)); PFP_TRY(pfp_free_now(ctx, hv1));
    }
    PFP_TRY(pfp_free_now(ctx, big));
    return PFPB200_OK;
}

template int pb_plan<PbSplitSlots>(pfpb200_ctx *, const PbInput &, const PbWords &, PbSplitSlots, u64, u8 *, u32 *,
                                   PbPlan *);

int pb_samples(pfpb200_ctx *ctx, const PbEmit &E, int at_end, int prev, int next, u64 off, bool held, u8 **out,
               u64 *n_out) {
    const u64 n = E.chars;
    *n_out = 0;
    if (n == 0) return PFPB200_OK;
    u32 *rf = nullptr;
    u64 *rscan = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &rf, n));
    PFP_TRY(pfp_alloc_t(ctx, &rscan, n));
    PB_LAUNCH(ctx, n, pb_runs_k, E.bwt, n, at_end, prev, next, rf);
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, rf, rscan, n, &ctx->d_flags[5]));
    PFP_TRY(pb_sync_read(ctx, 5, 1));
    *n_out = ctx->h_flags[5];
    PFP_TRY(pfp_alloc_t(ctx, out, *n_out * 2 * PFP_IBYTES, held));
    if (held) ctx->pb_out[2 + at_end] = *out;
    PB_LAUNCH(ctx, n, pb_sample_k, rf, rscan, E.sa5, n, off, *out);
    PFP_TRY(pfp_free_now(ctx, rf));
    PFP_TRY(pfp_free_now(ctx, rscan));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return PFPB200_OK;
}

// ---- the one-GPU path -------------------------------------------------------------------------------------
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

int pb_budget(pfpb200_ctx *ctx, int share, u64 *budget) {
    const char *ev = getenv("PFPB200_PFBWT_BUDGET");
    if (ev && atoll(ev) > 0) {
        *budget = (u64)atoll(ev);
        return PFPB200_OK;
    }
    size_t fr = 0, tot = 0;
    PFP_CUDA(ctx, cudaMemGetInfo(&fr, &tot));
    // a context alone on its device counts its arena's unused part; contexts that share the device do
    // not: a window's arrays do not fit into scattered holes, and the growth of their arenas would then
    // take memory the other contexts count on
    *budget = share > 1 ? (u64)fr / (u64)share : (u64)fr + (u64)(ctx->arena.total - ctx->arena.in_use);
    return PFPB200_OK;
}

u64 pb_window_bytes(const PbPlan &P, u32 flags, u64 cap) {
    return pb_out_bytes(cap < P.chars ? cap : P.chars, P.n_hard, flags);
}

u64 pb_window_chars(const PbPlan &P, u32 flags, u64 budget) {
    if (pb_out_bytes(P.chars, P.n_hard, flags) <= budget) return P.chars;
    u64 lo = 0, hi = P.chars;                                // pb_out_bytes grows with c: the largest c that fits
    while (lo < hi) {
        const u64 mid = lo + (hi - lo + 1) / 2;
        if (pb_out_bytes(mid, P.n_hard, flags) <= budget) lo = mid; else hi = mid - 1;
    }
    return lo;
}

int pb_put_host(pfpb200_ctx *ctx, int fd, u64 file_off, const u8 *p, u64 bytes, const char *name) {
    u64 done = 0;
    while (done < bytes) {
        const ssize_t r = pwrite(fd, p + done, bytes - done, (off_t)(file_off + done));
        if (r <= 0) return pfp_fail(ctx, PFPB200_E_IO, "%s: write error: %s", name, strerror(errno));
        done += (u64)r;
    }
    return PFPB200_OK;
}

static double pb_ms(const struct timespec &a) {
    struct timespec b;
    clock_gettime(CLOCK_MONOTONIC, &b);
    return 1e3 * (double)(b.tv_sec - a.tv_sec) + 1e-6 * (double)(b.tv_nsec - a.tv_nsec);
}

// Samples across a window border: a window's first char knows the char in front of it (-s); the last
// run end of a window (-e) waits on the host until the next window's first char shows whether the run
// goes on.  Across the piece's own borders nothing is known here: its first char starts a run and its
// last char ends one (the sharded path drops those records when a neighbouring piece continues the run).
int pb_write_windows(pfpb200_ctx *ctx, const PbInput &in, const PbWords &W, const PbPlan &P, u64 cap, PbOutFiles &F,
                     u64 off, PbPiece *pc) {
    const u64 S2 = 2 * PFP_IBYTES;                            // one sample: (BWT position, SA value)
    u64 ka = 0, n_s = 0, n_e = 0;
    int prev = -1;                                           // last char of the windows so far (-1: none yet)
    bool pending = false;                                    // the last run end so far, not yet written
    u8 pend[2 * PFP_IBYTES];
    *pc = PbPiece();
    struct timespec t;
    while (ka < P.n) {
        u64 kb = 0, cend = 0;
        clock_gettime(CLOCK_MONOTONIC, &t);
        PFP_TRY(pb_window_end(ctx, P, ka, cap, &kb, &cend));
        PbEmit E;
        PFP_TRY(pb_window(ctx, in, W, P, ka, kb, cap, false, &E));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        pc->ms_emit += pb_ms(t);
        pc->windows++;
        const u64 n = E.chars, gb = off + E.base;             // the window's chars: BWT positions [gb, gb + n)
        if (n) {
            clock_gettime(CLOCK_MONOTONIC, &t);
            u8 *cf = reinterpret_cast<u8 *>(&ctx->h_flags[9]), *cl = reinterpret_cast<u8 *>(&ctx->h_flags[10]);
            PFP_CUDA(ctx, cudaMemcpyAsync(cf, E.bwt, 1, cudaMemcpyDeviceToHost, ctx->stream));
            PFP_CUDA(ctx, cudaMemcpyAsync(cl, E.bwt + n - 1, 1, cudaMemcpyDeviceToHost, ctx->stream));
            PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            const int c_first = *cf, c_last = *cl;
            if (pc->c_first < 0) pc->c_first = c_first;
            PFP_TRY(pfp_device_to_fd(ctx, F.fd[0], gb, E.bwt, n, F.name[0]));
            if (F.fd[1] >= 0) {                              // the .sa file has no entry for BWT position 0
                if (gb == 0) PFP_TRY(pfp_device_to_fd(ctx, F.fd[1], 0, E.sa5 + PFP_IBYTES, (n - 1) * PFP_IBYTES, F.name[1]));
                else PFP_TRY(pfp_device_to_fd(ctx, F.fd[1], (gb - 1) * PFP_IBYTES, E.sa5, n * PFP_IBYTES, F.name[1]));
            }
            u8 *out = nullptr;
            u64 m = 0;
            if (F.fd[2] >= 0) {
                PFP_TRY(pb_samples(ctx, E, 0, prev, -1, gb, false, &out, &m));
                PFP_TRY(pfp_device_to_fd(ctx, F.fd[2], n_s * S2, out, m * S2, F.name[2]));
                PFP_TRY(pfp_free_now(ctx, out));
                n_s += m;
            }
            if (F.fd[3] >= 0) {
                if (pending && c_first != prev) {
                    PFP_TRY(pb_put_host(ctx, F.fd[3], n_e * S2, pend, S2, F.name[3]));
                    n_e++;
                }
                // with no char behind the window its last position ends a run: m >= 1, the last one pending
                PFP_TRY(pb_samples(ctx, E, 1, -1, -1, gb, false, &out, &m));
                PFP_TRY(pfp_device_to_fd(ctx, F.fd[3], n_e * S2, out, (m - 1) * S2, F.name[3]));
                PFP_CUDA(ctx, cudaMemcpyAsync(pend, out + (m - 1) * S2, S2, cudaMemcpyDeviceToHost, ctx->stream));
                PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
                PFP_TRY(pfp_free_now(ctx, out));
                n_e += m - 1;
                pending = true;
            }
            prev = c_last;
            pc->ms_write += pb_ms(t);
        }
        PFP_TRY(pfp_free_now(ctx, E.bwt));
        PFP_TRY(pfp_free_now(ctx, E.sa5));
        ka = kb;
    }
    if (pending) {
        PFP_TRY(pb_put_host(ctx, F.fd[3], n_e * S2, pend, S2, F.name[3]));
        n_e++;
    }
    pc->c_last = prev;
    pc->n_ssa = n_s;
    pc->n_esa = n_e;
    return PFPB200_OK;
}

// the one-GPU file outputs in windows: <base>.bwt / .sa created at their final sizes, .ssa / .esa appended
static int pb_write_files(pfpb200_ctx *ctx, const PbInput &in, const PbWords &W, const PbPlan &P, u64 cap,
                          const char *base, pfpb200_pfbwt_result *res, u64 *windows) {
    static const char *const ext[4] = {"bwt", "sa", "ssa", "esa"};
    const u32 want[4] = {0, PFPB200_PFBWT_SA, PFPB200_PFBWT_SSA, PFPB200_PFBWT_ESA};   // .bwt always
    const u64 size[4] = {P.chars, (P.chars - 1) * PFP_IBYTES, 0, 0};   // .sa: no entry for BWT position 0
    PbOutFiles F;
    for (int i = 0; i < 4; i++) {
        if (want[i] && !(in.flags & want[i])) continue;
        snprintf(F.name[i], sizeof(F.name[i]), "%s.%s", base, ext[i]);
        F.fd[i] = open(F.name[i], O_WRONLY | O_CREAT | O_TRUNC, 0666);
        if (F.fd[i] < 0) return pfp_fail(ctx, PFPB200_E_IO, "%s: %s", F.name[i], strerror(errno));
        if (size[i] && ftruncate(F.fd[i], (off_t)size[i]) != 0)
            return pfp_fail(ctx, PFPB200_E_IO, "%s: %s", F.name[i], strerror(errno));
    }
    PbPiece pc;
    PFP_TRY(pb_write_windows(ctx, in, W, P, cap, F, 0, &pc));
    *windows = pc.windows;
    for (int i = 0; i < 4; i++) {
        const int fd = F.fd[i];
        F.fd[i] = -1;
        if (fd >= 0 && close(fd) != 0) return pfp_fail(ctx, PFPB200_E_IO, "%s: write error: %s", F.name[i], strerror(errno));
    }
    res->n_bwt = P.chars;
    if (in.flags & PFPB200_PFBWT_SA) res->n_sa = P.chars - 1;
    res->n_ssa = pc.n_ssa;
    res->n_esa = pc.n_esa;
    return PFPB200_OK;
}

// out_base == null: the outputs stay in HBM, held by the context (pfpb200_pfbwt_device).  Otherwise they
// are meant for the files <out_base>.*: held as well when they fit the device memory the call has once its
// plan is done (the caller writes them), written here window by window when they do not (res->bwt ...
// stay null).  *windows: windows the output took.
static int pfbwt_device_impl(pfpb200_ctx *ctx, const PbInput &in, const char *out_base, pfpb200_pfbwt_result *res,
                             u64 *windows) {
    memset(res, 0, sizeof(*res));
    const u64 N = in.N, dwords = in.dwords, psize = in.psize;
    const u32 w = in.w, flags = in.flags;
    const bool want_sa = (flags & (PFPB200_PFBWT_SA | PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA)) != 0;
    if (const char *e = pb_arg_error(w, flags)) return pfp_fail(ctx, PFPB200_E_ARG, "%s", e);
    if (N <= 1 + (u64)w) return pfp_fail(ctx, PFPB200_E_ARG, "invalid dictionary file");               // :330
    if (want_sa && !in.bwsai) return pfp_fail(ctx, PFPB200_E_ARG, "suffix array output needs the .bwsai stream");
    if (N >= 0xFFFFFFF0ull || psize >= 0xFFFFFFFEull)
        return pfp_fail(ctx, PFPB200_E_LIMIT, "dictionary of 4 GB or more / more than 2^32-2 words in the parsing");
    PfpEvents evs(3);
    if (!evs.ok) return pfp_fail(ctx, PFPB200_E_CUDA, "cudaEventCreate failed");
    const u32 launches0 = ctx->launches;
    const u32 nb = pfp_blocks(N, PB_T);
    PFP_CUDA(ctx, cudaEventRecord(evs[0], ctx->stream));
    // ---- 1. word structure ---------------------------------------------------------------------------
    PbWords W;
    PFP_TRY(pb_words(ctx, in, &W));
    PFP_TRY(pb_word_ids(ctx, in, &W));
    // ---- 2. suffix sort ----------------------------------------------------------------------------------
    u8 *flag = nullptr, *keep = nullptr;
    u64 *k0 = nullptr, *k1 = nullptr;
    u32 *v0 = nullptr, *v1 = nullptr, *rank = nullptr, *rs = nullptr, *escan = nullptr;
    u64 *sa = nullptr;
    u32 *slot = nullptr, *slot2 = nullptr, *head = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &flag, N));
    PFP_TRY(pfp_alloc_t(ctx, &keep, N));
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
    pb_lim_k<<<nb, PB_T, 0, ctx->stream>>>(W.wid, W.wend, N, lim);
    PFP_LAUNCHED(ctx);
    pb_init_k<<<nb, PB_T, 0, ctx->stream>>>(in.d, N, W.cd, W.h0, W.bs, k0, v0, slot);
    PFP_LAUNCHED(ctx);
    const int b = pb_bits(N);
    const int kb = b <= 31 ? b : 0;                           // 2 b + 1 key bits fit into 64: old rank, second rank, done bit
    const int sort_bits = kb ? 2 * b + 1 : 64;
    u64 *ks = nullptr;
    u32 *vs = nullptr;
    PFP_TRY(pfp_radix_sort_pairs(ctx, k0, v0, k1, v1, N, 0, W.h0 * W.bs, &ks, &vs));
    u32 rounds = 1;
    u64 M = N;
    for (u64 h = (u64)W.h0;; h *= 2, rounds++) {
        const u32 mb = pfp_blocks(M, PB_T);
        pb_gflags_k<<<mb, PB_T, 0, ctx->stream>>>(ks, M, flag);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, flag, escan, M, nullptr));
        pb_heads_k<<<mb, PB_T, 0, ctx->stream>>>(flag, escan, slot, M, head);
        PFP_LAUNCHED(ctx);
        pb_update_k<<<mb, PB_T, 0, ctx->stream>>>(flag, escan, slot, vs, ks, kb, rounds == 1 ? 1 : 0, head, lim, M, h, sa,
                                                  rank, rs, keep);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, keep, escan, M, reinterpret_cast<u32 *>(&ctx->d_flags[1])));
        PFP_TRY(pb_sync_read(ctx, 1, 1));
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
    // ---- 3. emission --------------------------------------------------------------------------------------------
    PFP_TRY(pfp_free_now(ctx, rank));                        // the ranks travel with the suffix array from here on
    PbPlan P;
    PFP_TRY(pb_plan(ctx, in, W, PbPackedSlots{sa, W.wid}, N, flag, escan, &P));
    u64 cap = P.chars;
    if (out_base) {              // one window when the whole output fits, else windows of the most chars that fit
        u64 budget = 0;
        PFP_TRY(pb_budget(ctx, 1, &budget));
        cap = pb_window_chars(P, flags, budget);             // < P.chars: windows; 0: one group per window
    }
    *windows = 1;
    if (cap < P.chars) {
        PFP_TRY(pb_write_files(ctx, in, W, P, cap, out_base, res, windows));
    } else {
        PbEmit E;
        PFP_TRY(pb_window(ctx, in, W, P, 0, N, P.n_hard, true, &E));
        // ---- 4. sampled suffix array: the entries at the starts / ends of the runs ------------------------------------
        u8 *ssa = nullptr, *esa = nullptr;
        u64 n_ssa = 0, n_esa = 0;
        if (flags & PFPB200_PFBWT_SSA) PFP_TRY(pb_samples(ctx, E, 0, -1, -1, 0, true, &ssa, &n_ssa));
        if (flags & PFPB200_PFBWT_ESA) PFP_TRY(pb_samples(ctx, E, 1, -1, -1, 0, true, &esa, &n_esa));
        res->bwt = E.bwt;
        res->n_bwt = E.chars;
        if (flags & PFPB200_PFBWT_SA) {                      // the .sa file has no entry for the first BWT char (:157-163)
            res->sa = E.sa5 + PFP_IBYTES;
            res->n_sa = E.chars - 1;
        }
        res->ssa = ssa; res->n_ssa = n_ssa;
        res->esa = esa; res->n_esa = n_esa;
    }
    PFP_CUDA(ctx, cudaEventRecord(evs[2], ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    res->dict_bytes = N; res->dict_words = dwords; res->parse_size = psize;
    res->easy = P.chars - P.n_hard; res->hard = P.n_hard;
    res->rounds = rounds;
    res->launches = ctx->launches - launches0;
    cudaEventElapsedTime(&res->ms_sa, evs[0], evs[1]);
    cudaEventElapsedTime(&res->ms_fill, evs[1], evs[2]);
    res->ms_total = res->ms_sa + res->ms_fill;
    return PFPB200_OK;
}

// entry of the device and file calls: the outputs of the previous call go, the flags are cleared
static int pb_begin(pfpb200_ctx *ctx) {
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    pb_drop_own_outputs(ctx);
    ctx->err[0] = 0;
    PFP_CUDA(ctx, cudaMemsetAsync(ctx->d_flags, 0, 8 * sizeof(u64), ctx->stream));
    return PFPB200_OK;
}

extern "C" int pfpb200_pfbwt_device(pfpb200_ctx *ctx, const uint8_t *d_dict, uint64_t dict_bytes, const uint32_t *d_occ,
                                    uint64_t n_words, const uint32_t *d_ilist, const uint8_t *d_bwlast,
                                    const uint8_t *d_bwsai, uint64_t parse_size, uint32_t w, uint32_t flags,
                                    pfpb200_pfbwt_result *res) {
    if (!ctx || !d_dict || !d_occ || !d_ilist || !d_bwlast || !res) return PFPB200_E_ARG;
    PFP_TRY(pb_begin(ctx));
    const PbInput in{d_dict, dict_bytes, d_occ, n_words, d_ilist, d_bwlast, d_bwsai, parse_size, w, flags};
    u64 windows = 0;
    const int rc = pfbwt_device_impl(ctx, in, nullptr, res, &windows);
    pfp_release_scratch(ctx);
    return rc;
}

// the inputs (device pointers) -> <base>.bwt [.sa | .ssa .esa]: in one window when they fit, else in windows;
// the plan of the call for pfpb200_pfbwt_plan
int pb_to_files(pfpb200_ctx *ctx, const PbInput &in, const char *base, pfpb200_pfbwt_result *res) {
    PFP_TRY(pb_begin(ctx));
    u64 windows = 0;
    int rc = pfbwt_device_impl(ctx, in, base, res, &windows);
    char name[4096];
    auto put = [&](const char *ext, const void *p, u64 bytes) {
        if (rc != PFPB200_OK) return;
        snprintf(name, sizeof(name), "%s.%s", base, ext);
        rc = pfp_device_to_file(ctx, name, p, bytes);
    };
    if (rc == PFPB200_OK && res->bwt) {                           // held: the one-window run
        put("bwt", res->bwt, res->n_bwt);
        if (in.flags & PFPB200_PFBWT_SA) put("sa", res->sa, res->n_sa * PFP_IBYTES);
        if (in.flags & PFPB200_PFBWT_SSA) put("ssa", res->ssa, res->n_ssa * 2 * PFP_IBYTES);
        if (in.flags & PFPB200_PFBWT_ESA) put("esa", res->esa, res->n_esa * 2 * PFP_IBYTES);
    }
    ctx->pb_windows = windows;
    ctx->pb_peak = ctx->arena.peak;
    pfp_release_scratch(ctx);
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
    ctx->pb_windows = ctx->pb_peak = 0;
    ctx->arena.peak = ctx->arena.in_use;                              // pfpb200_pfbwt_plan reports this call's peak
    void *in[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    u64 n[5] = {0, 0, 0, 0, 0};
    PFP_TRY(pb_read_inputs(ctx, basename, flags, in, n));
    const PbInput pin{static_cast<u8 *>(in[0]), n[0], static_cast<u32 *>(in[1]), n[1], static_cast<u32 *>(in[2]),
                      static_cast<u8 *>(in[3]), static_cast<u8 *>(in[4]), n[2], w, flags};
    return pb_to_files(ctx, pin, basename, res);
}

extern "C" int pfpb200_pfbwt_plan(const pfpb200_ctx *ctx, uint64_t *windows, uint64_t *peak_device_bytes) {
    if (!ctx) return PFPB200_E_ARG;
    if (windows) *windows = ctx->pb_windows;
    if (peak_device_bytes) *peak_device_bytes = ctx->pb_peak;
    return PFPB200_OK;
}
