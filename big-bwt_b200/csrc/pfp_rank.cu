// pfp_rank.cu -- K4 lexicographic ranking of the distinct words, .dict/.occ emission, K5 remap.
//
// Replaces std::sort with pstringCompare (newscan.cpp:387-390,636), writeDictOcc (:394-441)
// and remapParse (:443-466).  Order = unsigned-byte lexicographic, as std::string compares.
//
// The distinct words sit in a pool, each zero-padded to 8-byte words.  Ranking: one global LSD
// radix sort on an alphabet-compacted first key (21 symbols for DNA), then MSD refinement of the
// tie groups on 8-byte big-endian chunks -- by LCP walks along each group's most frequent word,
// inside a warp for groups of up to 32 (rank_small_lcp_k) and 256 words (rank_lcp_k) and in a
// CTA up to 2048 (rank_lcp_cta_k), and by further global radix-sort rounds on (tie group, chunk)
// only for larger groups.  The chunk-pass kernels the walks replaced (rank_window_k / rank_warp_k,
// rank_mid_k / rank_cta_k) stay as A/B paths and for words of 8 MB and more.  A word's padding is 0x00, below every
// text byte (> 0x02), so shorter-is-smaller falls out.  Also here: routing of a shard's words to
// the owners of their lexicographic range (multi-GPU).
#include "pfp_common.cuh"
#include "pfp_stages.cuh"

__device__ __forceinline__ u64 bswap64(u64 v) {
    u32 lo = (u32)v, hi = (u32)(v >> 32);
    return ((u64)__byte_perm(lo, 0, 0x0123) << 32) | (u64)__byte_perm(hi, 0, 0x0123);
}

__device__ __forceinline__ u64 word_key(const u64 *__restrict__ pool, const u64 *__restrict__ uoff,
                                        const u32 *__restrict__ uwords, u32 u, u32 r) {
    return (r < uwords[u]) ? bswap64(__ldg(pool + uoff[u] + r)) : 0ull;
}

// ---- alphabet compaction for the first key ------------------------------------------------------------
// If the words use few distinct byte values in their first 24 bytes (DNA: A C G T N 0x02), an
// order-preserving code of `bits` bits per symbol packs 64/bits symbols into the first 64-bit
// key (21 for DNA) instead of 8, so the one global sort already separates almost everything.
struct AlphaMap {
    u32 bits;     // bits per symbol in the packed first key (8 = raw bytes)
    u32 chars;    // symbols covered by the first key
    u32 depth0;   // whole 8-byte chunks covered by the first key: refinement resumes there
    u32 pad;
    u8 lut[256];  // symbol -> code (1..sigma), order preserving; 0 = past the end of the word
};

constexpr u32 ALPHA_PROBE_WORDS = 3;   // first 24 bytes of every word are inspected

__global__ void alpha_presence_k(const u64 *__restrict__ pool, const u64 *__restrict__ uoff,
                                 const u32 *__restrict__ ulen, u64 d, u32 *__restrict__ gmask) {
    __shared__ u32 sm[8];
    if (threadIdx.x < 8) sm[threadIdx.x] = 0;
    __syncthreads();
    u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < d) {
        u32 len = ulen[u];
        u32 nb = len < 8 * ALPHA_PROBE_WORDS ? len : 8 * ALPHA_PROBE_WORDS;
        u32 m[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (u32 k = 0; k * 8 < nb; k++) {
            u64 v = __ldg(pool + uoff[u] + k);
            for (u32 b = 0; b < 8 && k * 8 + b < nb; b++) {
                u32 c = (u32)(v >> (8 * b)) & 255u;
#pragma unroll
                for (int q = 0; q < 8; q++) m[q] |= ((c >> 5) == (u32)q) ? (1u << (c & 31)) : 0u;
            }
        }
#pragma unroll
        for (int q = 0; q < 8; q++) {
            u32 x = __reduce_or_sync(__activemask(), m[q]);
            if ((threadIdx.x & 31) == (__ffs(__activemask()) - 1) && x) atomicOr(&sm[q], x);
        }
    }
    __syncthreads();
    if (threadIdx.x < 8 && sm[threadIdx.x]) atomicOr(&gmask[threadIdx.x], sm[threadIdx.x]);
}

// from_scan: the byte set comes from the DNA form of K1 over the whole text; the letters its table
// path stands for and the virtual border symbol are added here
__global__ void alpha_build_k(u32 *__restrict__ gmask, AlphaMap *am, int from_scan) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (from_scan) {
        gmask[0] |= 1u << PFP_DOLLAR;
        gmask[2] |= (1u << ('A' & 31)) | (1u << ('C' & 31)) | (1u << ('G' & 31)) | (1u << ('T' & 31));
    }
    u32 sigma = 0;
    for (int q = 0; q < 8; q++) sigma += __popc(gmask[q]);
    u32 bits = 3;            // >= 3 so that the key never reaches past the probed 24 bytes
    while ((1u << bits) < sigma + 1) bits++;
    if (bits > 4) {          // large alphabet: plain big-endian bytes
        am->bits = 8; am->chars = 8; am->depth0 = 1;
        for (int c = 0; c < 256; c++) am->lut[c] = (u8)c;
    } else {
        am->bits = bits; am->chars = 64 / bits; am->depth0 = (64 / bits) / 8;
        u32 code = 0;
        for (int c = 0; c < 256; c++) {
            bool present = (gmask[c >> 5] >> (c & 31)) & 1u;
            if (present) code++;
            am->lut[c] = (u8)(present ? code : 0);
        }
    }
    am->pad = 0;
}

__global__ void rank_keys0_k(const u64 *__restrict__ pool, const u64 *__restrict__ uoff,
                             const u32 *__restrict__ ulen, const u32 *__restrict__ count, u64 d,
                             const AlphaMap *__restrict__ am, u64 *__restrict__ keys, u32 *__restrict__ vals,
                             WordMeta *__restrict__ meta) {
    __shared__ u8 lut[256];
    __shared__ u32 s_bits, s_chars;
    lut[threadIdx.x & 255] = am->lut[threadIdx.x & 255];
    if (threadIdx.x == 0) { s_bits = am->bits; s_chars = am->chars; }
    __syncthreads();
    u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= d) return;
    const u32 bits = s_bits, chars = s_chars, len = ulen[u];
    const u64 off = uoff[u];
    {
        WordMeta wm;
        wm.off = off; wm.len = len; wm.count = count[u];
        meta[u] = wm;
    }
    const u32 nc = len < chars ? len : chars;
    u64 key = 0;
    u64 v = 0;
    for (u32 i = 0; i < nc; i++) {
        if ((i & 7) == 0) v = __ldg(pool + off + (i >> 3));
        u32 c = (u32)(v >> (8 * (i & 7))) & 255u;
        key |= (u64)lut[c] << (64 - bits * (i + 1));
    }
    keys[u] = key;
    vals[u] = (u32)u;
}

// Only the key bits [begin_bit, 64) were sorted (enough to tell d words apart; the rest is left to
// the tie kernels, which compare whole chunks anyway): groups and their known common depth follow
// from those bits alone.
__global__ void rank_heads0_k(const u64 *__restrict__ ks, u64 d, const AlphaMap *__restrict__ am, u32 begin_bit,
                              u8 *__restrict__ head, u32 *__restrict__ depth) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d) return;
    head[i] = (i == 0 || (ks[i] >> begin_bit) != (ks[i - 1] >> begin_bit)) ? 1 : 0;
    const u32 chars = (64u - begin_bit) / am->bits;           // whole symbols inside the sorted bits
    const u32 d0 = chars / 8u;                                // whole 8-byte chunks they cover
    depth[i] = d0 < am->depth0 ? d0 : am->depth0;
}

// ---- tie groups ------------------------------------------------------------------------------------------
constexpr u32 LOCAL_MAX = 2048;   // largest tie group finished inside one CTA
constexpr u32 WARP_MAX = 32;      // largest tie group finished inside one warp

// hp[k] = first position of group k (k < nheads), hp[nheads] = d; gid[i] = group of position i
__global__ void groups_compact_k(const u8 *__restrict__ head, const u32 *__restrict__ hscan, u64 d,
                                 const u32 *__restrict__ nheads, u32 *__restrict__ hp,
                                 u32 *__restrict__ gid) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d) return;
    u32 g = hscan[i] + head[i] - 1;
    gid[i] = g;
    if (head[i]) hp[g] = (u32)i;
    if (i == 0) hp[*nheads] = (u32)d;
}

// positions in groups larger than LOCAL_MAX go through another global round; the other groups were
// finished on chip in this round and become singletons
__global__ void rank_active_k(u8 *__restrict__ head, const u32 *__restrict__ gid,
                              const u32 *__restrict__ hp, u64 d, u8 *__restrict__ act,
                              u8 *__restrict__ gh) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d) return;
    u32 g = gid[i];
    bool big = (hp[g + 1] - hp[g]) > LOCAL_MAX;
    act[i] = big ? 1 : 0;
    gh[i] = (big && head[i]) ? 1 : 0;
    if (!big) head[i] = 1;
}

__global__ void rank_compact_k(const u8 *__restrict__ act, const u8 *__restrict__ gh,
                               const u32 *__restrict__ ascan, const u32 *__restrict__ gscan,
                               const u32 *__restrict__ ord, const u32 *__restrict__ gid,
                               const u32 *__restrict__ hp, const u32 *__restrict__ depth, u64 d,
                               const u64 *pool, const u64 *uoff, const u32 *uwords,
                               u32 *__restrict__ apos, u64 *__restrict__ keys, u32 *__restrict__ vals,
                               u32 *__restrict__ gid_of_u) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d || !act[i]) return;
    u32 j = ascan[i];
    u32 u = ord[i];
    u32 r = depth[hp[gid[i]]];          // chunks this group is known to share
    apos[j] = (u32)i;
    keys[j] = word_key(pool, uoff, uwords, u, r);
    vals[j] = u;
    gid_of_u[u] = gscan[i] + gh[i] - 1;
}

__global__ void rank_gidkeys_k(const u32 *__restrict__ vs, const u32 *__restrict__ gid_of_u, u64 m,
                               u64 *__restrict__ keys2) {
    u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < m) keys2[j] = gid_of_u[vs[j]];
}

// new heads where the chunk changes inside an old group; every (old or new) head of a group that
// took part now shares one more chunk
__global__ void rank_writeback_k(const u32 *__restrict__ apos, const u64 *__restrict__ gk,
                                 const u32 *__restrict__ vs, u64 m, const u32 *__restrict__ gid,
                                 const u32 *__restrict__ hp, const u32 *__restrict__ depth_in,
                                 const u64 *pool, const u64 *uoff, const u32 *uwords,
                                 u32 *__restrict__ ord, u8 *__restrict__ head,
                                 u32 *__restrict__ depth_out) {
    u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    u32 i = apos[j];
    u32 u = vs[j];
    u32 r = depth_in[hp[gid[i]]];
    ord[i] = u;
    bool newhead = false;
    if (j > 0 && gk[j] == gk[j - 1]) {
        u32 up = vs[j - 1];
        newhead = word_key(pool, uoff, uwords, u, r) != word_key(pool, uoff, uwords, up, r);
        if (newhead) head[i] = 1;
    }
    if (newhead || head[i]) depth_out[i] = r + 1;
}

// ---- local refinement of small tie groups inside a warp -----------------------------------------------
// Lanes are words and never move.  A lane knows the tie range it is in as (lo, sz): the rank of
// the range's first word and its size, and the depth r (8-byte chunk index) up to which the
// range is known to agree; lanes with the same lo are the same range (`match.any` finds them).
// One pass is a three-way split of every range around the chunk of its first lane (multikey
// quicksort): smaller | equal | larger, counted with two ballots -- the equal part goes one
// chunk deeper, the others keep their depth.  When every range is a singleton, lo is the rank.
// Nothing in a pass depends on the size of a group, so one warp refines all the groups that lie
// inside a window of 32 consecutive positions at once (rank_window_k); the groups straddling a
// window border get a warp of their own (rank_warp_k).
__device__ __forceinline__ u32 warp_refine(const u64 *__restrict__ wptr, u32 wn, u32 lo, u32 sz, u32 r,
                                           u32 max_chunks, u64 *__restrict__ flags) {
    u64 k0 = 0, k1 = 0, k2 = 0, k3 = 0;
    u32 have = 0;                                   // chunks r .. r+have-1 are in k0..
    for (;;) {
        const bool active = sz > 1;
        if (!__any_sync(0xffffffffu, active)) break;
        if (__any_sync(0xffffffffu, active && r >= max_chunks)) {
            if ((threadIdx.x & 31) == 0) atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_INTERNAL);
            break;
        }
        if (active && have == 0) {                  // four independent loads: one round trip per 32 bytes
            k0 = (r + 0 < wn) ? bswap64(__ldg(wptr + r + 0)) : 0ull;
            k1 = (r + 1 < wn) ? bswap64(__ldg(wptr + r + 1)) : 0ull;
            k2 = (r + 2 < wn) ? bswap64(__ldg(wptr + r + 2)) : 0ull;
            k3 = (r + 3 < wn) ? bswap64(__ldg(wptr + r + 3)) : 0ull;
            have = 4;
        }
        const u64 key = active ? k0 : 0ull;
        const u32 peers = __match_any_sync(0xffffffffu, lo);
        const u64 hk = __shfl_sync(0xffffffffu, key, __ffs(peers) - 1);
        const u32 b0 = __ballot_sync(0xffffffffu, active && key < hk) & peers;
        const u32 b1 = __ballot_sync(0xffffffffu, active && key == hk) & peers;
        if (active) {
            const u32 n0 = __popc(b0), n1 = __popc(b1);
            if (key < hk) sz = n0;
            else if (key == hk) { lo += n0; sz = n1; r++; k0 = k1; k1 = k2; k2 = k3; have--; }
            else { lo += n0 + n1; sz -= n0 + n1; }
        }
    }
    return lo;
}

// all groups of 2..32 words that lie inside one window of 32 consecutive positions
__global__ void __launch_bounds__(256) rank_window_k(const u32 *__restrict__ hp, const u32 *__restrict__ gid,
                                                     const u32 *__restrict__ depth, const u64 *pool,
                                                     const u64 *uoff, const u32 *uwords, u64 d, u32 max_chunks,
                                                     u32 shift /* 0, or 16: the groups pass 0 left over */,
                                                     u32 *__restrict__ ord, u64 *__restrict__ flags) {
    const u32 lane = threadIdx.x & 31;
    const u64 nwin = (d + 31) / 32 + (shift ? 1 : 0);
    const u64 nwarps = (u64)gridDim.x * 8;
    for (u64 k = (u64)blockIdx.x * 8 + (threadIdx.x >> 5); k < nwin; k += nwarps) {
        const i64 w0 = (i64)(k * 32) - (i64)shift;              // first position of the window
        const i64 pos = w0 + lane;
        u32 s = 0, m = 0;
        if (pos >= 0 && (u64)pos < d) {
            const u32 g = gid[pos];
            s = hp[g];
            m = hp[g + 1] - s;
        }
        bool in = m >= 2 && (i64)s >= w0 && (i64)s + m <= w0 + 32;
        if (shift) in = in && (s >> 5) != ((s + m - 1) >> 5);   // inside an unshifted window: done already
        if (!__any_sync(0xffffffffu, in)) continue;
        const u32 uid = in ? ord[pos] : 0;
        const u64 *wptr = pool + (in ? uoff[uid] : 0);
        const u32 wn = in ? uwords[uid] : 0;
        const u32 lo0 = in ? (u32)((i64)s - w0) : 0xFFFF0000u + lane;
        const u32 lo = warp_refine(wptr, wn, lo0, in ? m : 1u, in ? depth[s] : 0u, max_chunks, flags);
        if (in) ord[w0 + lo] = uid;
    }
}

// groups of 2..32 words that straddle a window border: one warp each
__global__ void __launch_bounds__(256) rank_warp_k(const u32 *__restrict__ hp,
                                                   const u32 *__restrict__ list,
                                                   const u32 *__restrict__ count,
                                                   const u32 *__restrict__ depth,
                                                   const u64 *pool, const u64 *uoff, const u32 *uwords,
                                                   u32 max_chunks, u32 *__restrict__ ord,
                                                   u64 *__restrict__ flags) {
    const u32 lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const u32 ng = *count;
    const u32 nwarps = gridDim.x * 8;
    for (u32 q = blockIdx.x * 8 + wp; q < ng; q += nwarps) {
        const u32 g = list[q];
        const u32 s = hp[g], m = hp[g + 1] - s;
        const bool mem = lane < m;
        const u32 uid = mem ? ord[s + lane] : 0;
        const u64 *wptr = pool + (mem ? uoff[uid] : 0);
        const u32 wn = mem ? uwords[uid] : 0;
        const u32 lo = warp_refine(wptr, wn, mem ? 0u : 0xFFFF0000u + lane, mem ? m : 1u, depth[s], max_chunks, flags);
        if (mem) ord[s + lo] = uid;
    }
}

// ---- local refinement of larger tie groups in shared memory ---------------------------------------------
// A group's words sit in shared memory in their current order, worked on by NT threads: NT = 32
// (one warp per group of up to MID_MAX words, eight groups per CTA) or NT = 256 (one CTA per
// group of up to LOCAL_MAX words).  Every word knows the tie range [lo, hi) it is in and the
// depth (8-byte chunk index) up to which that range is known to agree.  One pass:
//   * every word of a range of more than one word loads its chunk at the range's depth;
//   * the range is split three ways around the chunk of its FIRST word: smaller | equal | larger
//     (multikey quicksort).  The equal part moves one chunk deeper, the other two keep their
//     depth and are split again in the next pass;
//   * the position of a word inside its part is its rank among the words of the same class in
//     front of it in the range: one segmented scan over the positions (three 16-bit counters in
//     one 64-bit word), so a pass costs O(m) -- not O(range^2) as counting against every other
//     word of the range did.  Families of near-identical words (a thousand haplotypes' variants
//     of one phrase: long shared prefixes, one or two words leaving per chunk) are exactly the
//     case where that difference is a factor of the family size.
constexpr u32 MID_MAX = 256;
constexpr u32 TIE_EMAX = 8;       // positions per thread at most: CAP / NT

template <u32 CAP>
struct TieSort {
    u64 key[CAP];
    u64 tot[CAP];                 // class totals of a range, stored at its lo
    u32 uid[2][CAP];
    u32 off[2][CAP];              // pool offset of the word (8-byte words)
    u32 wn[2][CAP];               // its length in 8-byte words
    u16 lo[2][CAP];
    u16 hi[2][CAP];
    u32 dep[2][CAP];              // chunks the words of the range are known to share
};

template <int NT>
__device__ __forceinline__ void tie_sync() {
    if (NT == 32) __syncwarp(); else __syncthreads();
}
template <int NT>
__device__ __forceinline__ int tie_any(int x) {
    if (NT == 32) { int r = __any_sync(0xffffffffu, x); __syncwarp(); return r; }
    return __syncthreads_or(x);
}

// exclusive segmented scan across the NT threads: v = sum of my block behind its last segment
// start (or of the whole block), f = my block holds a segment start.  Returns the sum over the
// preceding threads back to the most recent start.
template <int NT>
__device__ __forceinline__ u64 tie_carry(u64 v, bool f, u64 *sm_v, u32 *sm_f) {
    const u32 lane = threadIdx.x & 31;
    u64 iv = v;
    int fl = f ? 1 : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u64 uv = __shfl_up_sync(0xffffffffu, iv, o);
        const int uf = __shfl_up_sync(0xffffffffu, fl, o);
        if (lane >= (u32)o && !fl) { iv += uv; fl = uf; }
    }
    u64 ex = __shfl_up_sync(0xffffffffu, iv, 1);        // inclusive value of the lane in front
    int exf = __shfl_up_sync(0xffffffffu, fl, 1);        // ... and whether it already saw a start
    if (lane == 0) { ex = 0; exf = 0; }
    if (NT == 32) return ex;
    // NT == 256: join the eight warps
    const u32 wp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 31) { sm_v[wp] = iv; sm_f[wp] = (u32)fl; }
    __syncthreads();
    u64 cin = 0;
    for (u32 k = 0; k < wp; k++) {
        if (sm_f[k]) cin = 0;
        cin += sm_v[k];
    }
    return exf ? ex : ex + cin;
}

// TIE_E: compile-time bound of the positions per thread (2, 4 or 8), so that small groups do not
// pay for eight predicated-off copies of every loop body
template <int NT, u32 CAP, u32 TIE_E>
__device__ __noinline__ void tie_refine_e(TieSort<CAP> &S, u64 *sm_v, u32 *sm_f, u32 t, u32 s, u32 m, u32 r0,
                                          const u64 *pool, const u64 *uoff, const u32 *uwords, u32 max_chunks,
                                          u32 *__restrict__ ord, u64 *__restrict__ flags) {
    static_assert(CAP == NT * TIE_EMAX && TIE_E <= TIE_EMAX, "blocked layout: up to TIE_EMAX positions per thread");
    int cur = 0;
    tie_sync<NT>();
    for (u32 i = t; i < m; i += NT) {
        const u32 u = ord[s + i];
        S.uid[0][i] = u; S.off[0][i] = (u32)uoff[u]; S.wn[0][i] = uwords[u];
        S.lo[0][i] = 0; S.hi[0][i] = (u16)m; S.dep[0][i] = r0;
    }
    tie_sync<NT>();
    const u32 E = (m + NT - 1) / NT;                     // positions per thread for this group (<= TIE_E)
    const u32 p0 = t * E;                                // my positions: p0 .. p0 + E - 1
    for (;;) {
        // ---- chunks at the ranges' depths ---------------------------------------------------------------
        int any = 0, bad = 0;
#pragma unroll
        for (u32 e = 0; e < TIE_E; e++) {
            const u32 p = p0 + e;
            if (e < E && p < m) {
                const bool act = (u32)(S.hi[cur][p] - S.lo[cur][p]) > 1;
                const u32 r = S.dep[cur][p];
                S.key[p] = (act && r < S.wn[cur][p]) ? bswap64(__ldg(pool + S.off[cur][p] + r)) : 0ull;
                any |= act ? 1 : 0;
                bad |= (act && r >= max_chunks) ? 1 : 0;
            }
        }
        if (!tie_any<NT>(any | (bad << 1))) break;
        if (tie_any<NT>(bad)) {
            if (t == 0) atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_INTERNAL);
            break;
        }
        // ---- classes and the segmented scan of their counters ----------------------------------------
        u64 incl[TIE_E];
        u32 cls[TIE_E];
        u64 run = 0;
        bool started = false;                            // a range starts inside my block
        int differs = 0;
#pragma unroll
        for (u32 e = 0; e < TIE_E; e++) {
            const u32 p = p0 + e;
            incl[e] = 0; cls[e] = 1;
            if (e < E && p < m) {
                const u32 l = S.lo[cur][p];
                if (l == p) { started = true; run = 0; }
                const bool act = (u32)(S.hi[cur][p] - l) > 1;
                const u64 k = S.key[p], hk = S.key[l];
                cls[e] = !act ? 1u : (k < hk ? 0u : (k == hk ? 1u : 2u));
                differs |= cls[e] != 1u ? 1 : 0;
                run += 1ull << (16 * cls[e]);
                incl[e] = run;
            }
        }
        if (!tie_any<NT>(differs)) {                     // a chunk every range shares: nothing moves
#pragma unroll
            for (u32 e = 0; e < TIE_E; e++) {
                const u32 p = p0 + e;
                if (e < E && p < m && (u32)(S.hi[cur][p] - S.lo[cur][p]) > 1) S.dep[cur][p]++;
            }
            continue;
        }
        // run = my block behind its last range start (or all of it): what the next threads continue
        const u64 carry = tie_carry<NT>(run, started, sm_v, sm_f);
        // ---- totals of every range, left at its lo by its last word ---------------------------------------
        started = false;
#pragma unroll
        for (u32 e = 0; e < TIE_E; e++) {
            const u32 p = p0 + e;
            if (e < E && p < m) {
                const u32 l = S.lo[cur][p];
                if (l == p) started = true;
                if (!started) incl[e] += carry;         // still in the range the previous threads began
                if (p + 1 == S.hi[cur][p]) S.tot[l] = incl[e];
            }
        }
        tie_sync<NT>();
        // ---- move ------------------------------------------------------------------------------------------
#pragma unroll
        for (u32 e = 0; e < TIE_E; e++) {
            const u32 p = p0 + e;
            if (e < E && p < m) {
                const u32 l = S.lo[cur][p], h = S.hi[cur][p], r = S.dep[cur][p];
                u32 np = p, nlo = l, nhi = h, nr = r;
                if (h - l > 1) {
                    const u64 T = S.tot[l];
                    const u32 n0 = (u32)(T & 0xFFFFu), n1 = (u32)((T >> 16) & 0xFFFFu);
                    const u32 idx = (u32)((incl[e] >> (16 * cls[e])) & 0xFFFFu) - 1u;
                    if (cls[e] == 0) { nlo = l; nhi = l + n0; }
                    else if (cls[e] == 1) { nlo = l + n0; nhi = l + n0 + n1; nr = r + 1; }
                    else { nlo = l + n0 + n1; nhi = h; }
                    np = nlo + idx;
                }
                S.uid[cur ^ 1][np] = S.uid[cur][p];
                S.off[cur ^ 1][np] = S.off[cur][p];
                S.wn[cur ^ 1][np] = S.wn[cur][p];
                S.lo[cur ^ 1][np] = (u16)nlo;
                S.hi[cur ^ 1][np] = (u16)nhi;
                S.dep[cur ^ 1][np] = nr;
            }
        }
        tie_sync<NT>();
        cur ^= 1;
    }
    tie_sync<NT>();
    for (u32 i = t; i < m; i += NT) ord[s + i] = S.uid[cur][i];
}

template <int NT, u32 CAP>
__device__ __forceinline__ void tie_refine(TieSort<CAP> &S, u64 *sm_v, u32 *sm_f, u32 t, u32 s, u32 m, u32 r0,
                                           const u64 *pool, const u64 *uoff, const u32 *uwords, u32 max_chunks,
                                           u32 *__restrict__ ord, u64 *__restrict__ flags) {
    const u32 E = (m + NT - 1) / NT;
    if (E <= 2) tie_refine_e<NT, CAP, 2>(S, sm_v, sm_f, t, s, m, r0, pool, uoff, uwords, max_chunks, ord, flags);
    else if (E <= 4) tie_refine_e<NT, CAP, 4>(S, sm_v, sm_f, t, s, m, r0, pool, uoff, uwords, max_chunks, ord, flags);
    else tie_refine_e<NT, CAP, 8>(S, sm_v, sm_f, t, s, m, r0, pool, uoff, uwords, max_chunks, ord, flags);
}

// lists of the groups for the kernels above; warp_list == nullptr: rank_small_lcp_k takes every
// group of 2..32 words.  counts[3] != 0: some group is larger than LOCAL_MAX (another global round).
__global__ void rank_lists_k(const u32 *__restrict__ hp, const u32 *__restrict__ nheads, u64 d,
                             u32 *__restrict__ mid_list, u32 *__restrict__ big_list,
                             u32 *__restrict__ warp_list,
                             u32 *__restrict__ counts /* [0]=mid, [1]=big, [2]=warp, [3]=global */) {
    u64 g = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= d || g >= *nheads) return;
    const u32 s = hp[g], m = hp[g + 1] - s;
    if (m < 2) return;
    if (m <= WARP_MAX) {                      // inside one window of 32 positions: rank_window_k has it
        if (warp_list && (s >> 5) != ((s + m - 1) >> 5)) warp_list[atomicAdd(&counts[2], 1u)] = (u32)g;
    } else if (m <= MID_MAX) mid_list[atomicAdd(&counts[0], 1u)] = (u32)g;
    else if (m <= LOCAL_MAX) big_list[atomicAdd(&counts[1], 1u)] = (u32)g;
    else counts[3] = 1u;
}

__global__ void __launch_bounds__(256) rank_mid_k(const u32 *__restrict__ hp,
                                                  const u32 *__restrict__ list,
                                                  const u32 *__restrict__ count,
                                                  const u32 *__restrict__ depth,
                                                  const u64 *pool, const u64 *uoff, const u32 *uwords,
                                                  u32 max_chunks, u32 *__restrict__ ord,
                                                  u64 *__restrict__ flags) {
    extern __shared__ __align__(16) unsigned char mid_raw[];
    const u32 lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    TieSort<MID_MAX> &S = reinterpret_cast<TieSort<MID_MAX> *>(mid_raw)[wp];
    u64 *sm_v = nullptr;
    u32 *sm_f = nullptr;
    const u32 n = *count;
    for (u32 q = blockIdx.x * 8 + wp; q < n; q += gridDim.x * 8) {
        const u32 g = list[q];
        const u32 s = hp[g], m = hp[g + 1] - s;
        tie_refine<32, MID_MAX>(S, sm_v, sm_f, lane, s, m, depth[s], pool, uoff, uwords, max_chunks, ord, flags);
    }
}

// ---- LCP-aware refinement of mid-size tie groups (33..256 words), one warp per group ----------------------
// The multikey-quicksort passes above advance ONE 8-byte chunk per pass; a family of variants of
// one long phrase (p = 1000: words of a kilobyte, a hundred of them differing in one base each)
// then costs a pass -- a memory round trip, a scan and two moves of the group -- per chunk of
// shared prefix.  Here a round costs one walk per word instead: every word of a range walks along
// the range's FIRST word (its head) until they differ, at chunk c with own chunk v against the
// head's h.  For two words x, y below the head (v < h): c_x < c_y  =>  x[c_x] < head[c_x] = y[c_x],
// so x < y; with equal c the chunks decide; above the head the order in c is reversed.  So
//      (below: c ascending, v ascending) < head < (above: c descending, v ascending)
// is the lexicographic order of the range, up to ties (same c, same v), which agree on c + 1
// chunks and form the ranges of the next round.  One bitonic sort of the group by
// (range, class/c, v) per round; a family is done in two or three rounds whatever its length.
constexpr u32 LCP_MAX = 256;                  // words per group finished by one warp
constexpr u32 LCP_WALK = 4;                   // chunks fetched per memory round trip of a walk
constexpr u32 LCP_HEAD = 1u << 20;            // class-and-depth code of a range's head / a finished word
constexpr u32 LCP_MAX_CHUNKS = LCP_HEAD - 1;  // longer words (8 MB) take the chunk-pass kernels

// sort key of a word inside its group: ka = range start << 21 | code, code = c (left the head at
// chunk c, below it), LCP_HEAD (the head), 2^21 - 1 - c (above it); kb = the word's chunk at c
template <u32 CAP>
struct LcpSort {
    u64 kb[CAP];
    u32 ka[CAP];
    u32 uid[CAP];
    u32 off[CAP];                             // pool offset (8-byte words)
    u32 wn[CAP];                              // length in 8-byte words
    u32 dep[CAP];                             // at a range start: chunks the range is known to share
    u16 lo[CAP];                              // range start of every position
    u16 pay[CAP];                             // position before the sort; then: 1 = a range starts here
    unsigned long long best;                  // occurrences << 32 | position of the group's most frequent word
};

__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ bool lcp_less(u32 a0, u64 b0, u32 a1, u64 b1) { return a0 < a1 || (a0 == a1 && b0 < b1); }

// compare-exchange of the (ka, kb, pay) held by two lanes (partner = lane ^ j), ascending iff `up`
__device__ __forceinline__ void lcp_cx_shfl(u32 &ka, u64 &kb, u32 &pay, u32 j, bool up, bool lower) {
    const u32 oa = __shfl_xor_sync(0xffffffffu, ka, j);
    const u64 ob = __shfl_xor_sync(0xffffffffu, kb, j);
    const u32 op = __shfl_xor_sync(0xffffffffu, pay, j);
    const bool mine_less = lcp_less(ka, kb, oa, ob);
    // the lower lane keeps the smaller key in an ascending block, the larger one in a descending block
    const bool keep = (mine_less == lower) == up;
    if (!keep && !(ka == oa && kb == ob)) { ka = oa; kb = ob; pay = op; }
}

// compare-exchange inside a lane: elements e and e ^ DJ (partner distance DJ * 32 positions)
template <int E, int DJ>
__device__ __forceinline__ void lcp_cx_lane(u32 (&ka)[E], u64 (&kb)[E], u32 (&pay)[E], u32 lane, u32 k) {
#pragma unroll
    for (int e = 0; e < E; e++) {
        const int x = e ^ DJ;
        if (x > e && x < E) {
            const bool up = (((u32)e * 32 + lane) & k) == 0;
            if (lcp_less(ka[x], kb[x], ka[e], kb[e]) == up) {
                const u32 ta = ka[e]; ka[e] = ka[x]; ka[x] = ta;
                const u64 tb = kb[e]; kb[e] = kb[x]; kb[x] = tb;
                const u32 tp = pay[e]; pay[e] = pay[x]; pay[x] = tp;
            }
        }
    }
}

// bitonic sort of E*32 keys held E per lane (position e*32 + lane) entirely in registers: partners
// at distance < 32 are reached by shuffles, the others sit in the same lane.  The (k, j) loops stay
// loops: fully unrolled, the four instantiations are tens of thousands of instructions and the
// kernel stalls on instruction fetch (measured: 69 % of the stall samples).
template <int E>
__device__ __forceinline__ void lcp_bitonic_regs(u32 (&ka)[E], u64 (&kb)[E], u32 (&pay)[E], u32 lane) {
#pragma unroll 1
    for (u32 k = 2; k <= (u32)E * 32; k <<= 1) {
#pragma unroll 1
        for (u32 j = k >> 1; j > 0; j >>= 1) {
            if (j >= 32) {
                const u32 dj = j >> 5;
                if (dj == 1) lcp_cx_lane<E, 1>(ka, kb, pay, lane, k);
                else if (dj == 2) lcp_cx_lane<E, 2>(ka, kb, pay, lane, k);
                else lcp_cx_lane<E, 4>(ka, kb, pay, lane, k);
            } else {
#pragma unroll
                for (int e = 0; e < E; e++) {
                    const bool up = (((u32)e * 32 + lane) & k) == 0;
                    lcp_cx_shfl(ka[e], kb[e], pay[e], j, up, (lane & j) == 0);
                }
            }
        }
    }
}

template <int E>
__device__ __noinline__ void lcp_sort_regs(LcpSort<LCP_MAX> &S, u32 lane) {
    u32 ka[E], pay[E];
    u64 kb[E];
#pragma unroll
    for (int e = 0; e < E; e++) { ka[e] = S.ka[e * 32 + lane]; kb[e] = S.kb[e * 32 + lane]; pay[e] = S.pay[e * 32 + lane]; }
    lcp_bitonic_regs<E>(ka, kb, pay, lane);
    __syncwarp();
#pragma unroll
    for (int e = 0; e < E; e++) { S.ka[e * 32 + lane] = ka[e]; S.kb[e * 32 + lane] = kb[e]; S.pay[e * 32 + lane] = (u16)pay[e]; }
}

// One group of m words (hp range [s, s+m)) by the NT threads of a team (a warp, or a CTA).
template <int NT, u32 CAP>
__device__ __forceinline__ void lcp_refine(LcpSort<CAP> &S, u32 t, u32 s, u32 m, u32 r0, const u64 *__restrict__ pool,
                                           const u64 *__restrict__ uoff, const u32 *__restrict__ uwords,
                                           const u32 *__restrict__ occ_of_word, u32 max_chunks,
                                           u32 *__restrict__ ord, u64 *__restrict__ flags) {
    u32 M = 32;                                               // bitonic size: next power of two
    while (M < m) M <<= 1;
    if (t == 0) S.best = 0ull;
    tie_sync<NT>();
    {   // the words of the group: ids first, then their offsets / lengths (independent loads in flight together)
        constexpr u32 EM = CAP / NT;
        u32 us[EM];
#pragma unroll
        for (u32 e = 0; e < EM; e++) { const u32 p = e * NT + t; us[e] = p < m ? ord[s + p] : 0u; }
#pragma unroll
        for (u32 e = 0; e < EM; e++) {
            const u32 p = e * NT + t;
            if (p < m) {
                const u32 o = (u32)uoff[us[e]];
                S.uid[p] = us[e]; S.off[p] = o; S.wn[p] = uwords[us[e]];
                S.lo[p] = 0;
                prefetch_l2(pool + o + r0);                   // where the first walk starts
                atomicMax(&S.best, ((unsigned long long)occ_of_word[us[e]] << 32) | p);
            }
        }
    }
    if (t == 0) S.dep[0] = r0;
    tie_sync<NT>();
    // The head of the first round is the group's MOST FREQUENT word.  Any member would do for
    // correctness; but a tie group is typically a family -- one consensus phrase and its variants,
    // each differing from the consensus in one place -- and against the consensus every variant
    // leaves at its own place (one round), while against a variant everything that mutates
    // behind the variant's place leaves together and has to be split again, round after round.
    if (t == 0) {
        const u32 b = (u32)(S.best & 0xFFFFFFFFull);
        if (b != 0 && b < m) {
            const u32 u0 = S.uid[0], o0 = S.off[0], w0 = S.wn[0];
            S.uid[0] = S.uid[b]; S.off[0] = S.off[b]; S.wn[0] = S.wn[b];
            S.uid[b] = u0; S.off[b] = o0; S.wn[b] = w0;
        }
    }
    tie_sync<NT>();
    for (u32 round = 0;; round++) {
        // ---- 1. every word of a range of two or more walks along the range's head -------------------------
        // (the chunks where the walks start are requested for ALL of a thread's words first: the walks
        //  of one thread run one after the other, and each would otherwise wait for DRAM on its own)
        if (round > 0)
            for (u32 p = t; p < m; p += NT) {
                const u32 l = S.lo[p];
                if (p != l) prefetch_l2(pool + S.off[p] + S.dep[l]);
            }
        int any = 0, bad = 0;
        u32 na = 0;                                           // words still tied (NT == 32: exact, for all lanes)
        for (u32 p = t; p < M; p += NT) {
            u32 ka = 0xFFFFFFFFu;                             // padding sorts behind everything
            u64 kb = 0;
            bool active = false;
            if (p < m) {
                const u32 l = S.lo[p];
                const bool single = (p == l) && (p + 1 >= m || S.lo[p + 1] != l);
                active = !single;
                u32 code = LCP_HEAD;
                if (active && p != l) {
                    const u64 *mine = pool + S.off[p], *head = pool + S.off[l];
                    const u32 wm = S.wn[p], wh = S.wn[l];
                    u32 c = S.dep[l];
                    u64 v = 0, h = 0;
                    for (;;) {
                        u64 a[LCP_WALK], b[LCP_WALK];
#pragma unroll
                        for (u32 i = 0; i < LCP_WALK; i++) {
                            a[i] = (c + i < wm) ? __ldg(mine + c + i) : 0ull;
                            b[i] = (c + i < wh) ? __ldg(head + c + i) : 0ull;
                        }
                        bool found = false;
#pragma unroll
                        for (u32 i = 0; i < LCP_WALK; i++)
                            if (!found && a[i] != b[i]) { found = true; c += i; v = bswap64(a[i]); h = bswap64(b[i]); }
                        if (found) break;
                        c += LCP_WALK;
                        prefetch_l2(mine + c + LCP_WALK);     // one batch ahead
                        if (c >= max_chunks) { bad = 1; break; }          // two equal words: cannot happen
                    }
                    code = v < h ? c : 2u * LCP_HEAD - 1u - c;
                    kb = v;
                }
                ka = (l << 21) | code;
            }
            if (NT == 32) na += __popc(__ballot_sync(0xffffffffu, active));
            any |= active ? 1 : 0;
            S.ka[p] = ka; S.kb[p] = kb; S.pay[p] = (u16)p;
        }
        if (tie_any<NT>(bad)) {
            if (t == 0) atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_INTERNAL);
            break;
        }
        if (!tie_any<NT>(any)) break;
        // ---- 2. sort the group by (range start, class/depth code, chunk) -------------------------------------
        if (NT == 32 && na <= 48) {
            // few words are still tied (every round but the first): each finds its place among the
            // words of its range by counting the smaller ones
            u16 np[LCP_MAX / 32];
#pragma unroll
            for (u32 e = 0; e < LCP_MAX / 32; e++) {
                const u32 p = e * 32 + t;
                np[e] = (u16)p;
                if (p < m) {
                    const u32 l = S.lo[p];
                    const bool single = (p == l) && (p + 1 >= m || S.lo[p + 1] != l);
                    if (!single) {
                        const u32 a0 = S.ka[p];
                        const u64 b0 = S.kb[p];
                        u32 rank = 0;
                        for (u32 q = l; q < m && S.lo[q] == l; q++) {
                            const u32 a1 = S.ka[q];
                            const u64 b1 = S.kb[q];
                            rank += (lcp_less(a1, b1, a0, b0) || (a1 == a0 && b1 == b0 && q < p)) ? 1u : 0u;
                        }
                        np[e] = (u16)(l + rank);
                    }
                }
            }
            // pay[new position] = old position, keys move along
            u32 ka[LCP_MAX / 32];
            u64 kb[LCP_MAX / 32];
#pragma unroll
            for (u32 e = 0; e < LCP_MAX / 32; e++) {
                const u32 p = e * 32 + t;
                if (p < m) { ka[e] = S.ka[p]; kb[e] = S.kb[p]; }
            }
            __syncwarp();
#pragma unroll
            for (u32 e = 0; e < LCP_MAX / 32; e++) {
                const u32 p = e * 32 + t;
                if (p < m) { S.ka[np[e]] = ka[e]; S.kb[np[e]] = kb[e]; S.pay[np[e]] = (u16)p; }
            }
            __syncwarp();
        } else if (NT == 32) {
            __syncwarp();
            LcpSort<LCP_MAX> &W = reinterpret_cast<LcpSort<LCP_MAX> &>(S);
            if (M == 32) lcp_sort_regs<1>(W, t);
            else if (M == 64) lcp_sort_regs<2>(W, t);
            else if (M == 128) lcp_sort_regs<4>(W, t);
            else lcp_sort_regs<8>(W, t);
            __syncwarp();
        } else {
            tie_sync<NT>();
            for (u32 k = 2; k <= M; k <<= 1) {
                for (u32 j = k >> 1; j > 0; j >>= 1) {
                    for (u32 i = t; i < M; i += NT) {
                        const u32 x = i ^ j;
                        if (x > i) {
                            const u32 a0 = S.ka[i], a1 = S.ka[x];
                            const u64 b0 = S.kb[i], b1 = S.kb[x];
                            if (lcp_less(a1, b1, a0, b0) == ((i & k) == 0)) {
                                S.ka[i] = a1; S.ka[x] = a0; S.kb[i] = b1; S.kb[x] = b0;
                                const u16 tp = S.pay[i]; S.pay[i] = S.pay[x]; S.pay[x] = tp;
                            }
                        }
                    }
                    tie_sync<NT>();
                }
            }
        }
        // ---- 3. move the words; ranges of the next round = runs of equal keys ---------------------------------
        {
            constexpr u32 EM = CAP / NT;
            u32 mu[EM], mo[EM], mw[EM];
#pragma unroll
            for (u32 e = 0; e < EM; e++) {
                const u32 p = e * NT + t;
                if (p < m) { const u32 q = S.pay[p]; mu[e] = S.uid[q]; mo[e] = S.off[q]; mw[e] = S.wn[q]; }
            }
            tie_sync<NT>();
#pragma unroll
            for (u32 e = 0; e < EM; e++) {
                const u32 p = e * NT + t;
                if (p < m) {
                    S.uid[p] = mu[e]; S.off[p] = mo[e]; S.wn[p] = mw[e];
                    const bool start = p == 0 || S.ka[p] != S.ka[p - 1] || S.kb[p] != S.kb[p - 1];
                    S.pay[p] = start ? 1 : 0;
                    if (start) {                              // depth of a new range: its members left their old
                        const u32 code = S.ka[p] & (2u * LCP_HEAD - 1u);    // head at the same chunk c
                        const u32 c = code < LCP_HEAD ? code : 2u * LCP_HEAD - 1u - code;
                        S.dep[p] = code == LCP_HEAD ? 0u : c + 1;
                    }
                }
            }
            tie_sync<NT>();
            if (t < 32) {                                     // range start of every position: one warp, ballots
                u32 carry = 0;
                for (u32 b0 = 0; b0 < m; b0 += 32) {
                    const u32 p = b0 + t;
                    const u32 sm = __ballot_sync(0xffffffffu, p < m && S.pay[p] != 0);
                    if (p < m) {
                        const u32 below = sm & (0xFFFFFFFFu >> (31 - t));
                        S.lo[p] = (u16)(below ? b0 + (31 - __clz(below)) : carry);
                    }
                    if (sm) carry = b0 + (31 - __clz(sm));
                }
            }
            tie_sync<NT>();
        }
    }
    tie_sync<NT>();
    for (u32 p = t; p < m; p += NT) ord[s + p] = S.uid[p];
}

// groups of 33..256 words: one warp each
__global__ void __launch_bounds__(256, 3) rank_lcp_k(const u32 *__restrict__ hp, const u32 *__restrict__ list,
                                                  const u32 *__restrict__ count, const u32 *__restrict__ depth,
                                                  const u64 *__restrict__ pool, const u64 *__restrict__ uoff,
                                                  const u32 *__restrict__ uwords, const u32 *__restrict__ occ_of_word,
                                                  u32 max_chunks, u32 *__restrict__ ord, u64 *__restrict__ flags) {
    extern __shared__ __align__(16) unsigned char lcp_raw[];
    const u32 lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    LcpSort<LCP_MAX> &S = reinterpret_cast<LcpSort<LCP_MAX> *>(lcp_raw)[wp];
    const u32 n = *count;
    for (u32 gq = blockIdx.x * 8 + wp; gq < n; gq += gridDim.x * 8) {
        const u32 g = list[gq];
        const u32 s = hp[g], m = hp[g + 1] - s;
        lcp_refine<32, LCP_MAX>(S, lane, s, m, depth[s], pool, uoff, uwords, occ_of_word, max_chunks, ord, flags);
    }
}

// groups of 257..2048 words: one CTA each
__global__ void __launch_bounds__(256) rank_lcp_cta_k(const u32 *__restrict__ hp, const u32 *__restrict__ list,
                                                      const u32 *__restrict__ count, const u32 *__restrict__ depth,
                                                      const u64 *__restrict__ pool, const u64 *__restrict__ uoff,
                                                      const u32 *__restrict__ uwords, const u32 *__restrict__ occ_of_word,
                                                      u32 max_chunks, u32 *__restrict__ ord, u64 *__restrict__ flags) {
    extern __shared__ __align__(16) unsigned char lcp_cta_raw[];
    LcpSort<LOCAL_MAX> &S = *reinterpret_cast<LcpSort<LOCAL_MAX> *>(lcp_cta_raw);
    const u32 n = *count;
    for (u32 gq = blockIdx.x; gq < n; gq += gridDim.x) {
        const u32 g = list[gq];
        const u32 s = hp[g], m = hp[g + 1] - s;
        lcp_refine<256, LOCAL_MAX>(S, threadIdx.x, s, m, depth[s], pool, uoff, uwords, occ_of_word, max_chunks, ord, flags);
    }
}

// ---- LCP walks for the small tie groups (2..32 words), one warp per window of 32 group starts -------------
// Warp k owns every group of 2..32 words whose first position lies in [32k, 32k + 32): they cover at
// most the 63 positions [32k, 32k + 63), so a lane holds up to two words (entries e = 0, 1 at
// positions 32k + 32e + lane; entry id = 32e + lane).  Entries never move: each knows its position
// inside the warp's span, the range [lo, lo + sz) it is tied in and the chunks dep its range shares.
// A round is lcp_refine's: the range's most frequent word is the head, every other word walks along
// it to the first chunk c where they differ (own chunk v), and the range is ordered by
// (code, v) with code = c below the head, LCP_HEAD for the head, 2 LCP_HEAD - 1 - c above it;
// equal keys are the ranges of the next round, at depth c + 1.  Families of variants of one
// consensus phrase are done in one or two rounds, whatever their depth.
constexpr u32 SMALL_WALK = 4;                 // 16-byte loads per word per memory round trip: 8 chunks

// Walk the word at `mine` (wm chunks) along `head` (wh chunks) from chunk c; returns the first chunk
// where they differ, with both chunks there (big-endian) in v, h.  Chunks past a word's end are 0.
// The loads are 16-byte aligned: a block that starts inside a word stays in its 16-byte line.
__device__ __forceinline__ u32 small_walk(const u64 *mine, u32 wm, const u64 *head, u32 wh, u32 c, u32 max_chunks,
                                          u64 &v, u64 &h, bool &bad) {
    constexpr u32 NC = 2 * SMALL_WALK;
    for (;;) {
        const u32 sa = (u32)((uintptr_t)(mine + c) >> 3) & 1u, sb = (u32)((uintptr_t)(head + c) >> 3) & 1u;
        const ulonglong2 *A = reinterpret_cast<const ulonglong2 *>(mine + c - sa);
        const ulonglong2 *B = reinterpret_cast<const ulonglong2 *>(head + c - sb);
        u64 a[NC], b[NC];
#pragma unroll
        for (u32 i = 0; i < SMALL_WALK; i++) {
            ulonglong2 x = make_ulonglong2(0ull, 0ull), y = make_ulonglong2(0ull, 0ull);
            if (c + 2 * i < wm + sa) x = __ldg(A + i);
            if (c + 2 * i < wh + sb) y = __ldg(B + i);
            a[2 * i] = x.x; a[2 * i + 1] = x.y;
            b[2 * i] = y.x; b[2 * i + 1] = y.y;
        }
        const u32 n = NC - (sa | sb);                 // chunks c .. c + n - 1 are in a, b
        bool found = false;
#pragma unroll
        for (u32 i = 0; i < NC; i++) {
            u64 x = (i + 1 < NC && sa) ? a[i + 1] : a[i];
            u64 y = (i + 1 < NC && sb) ? b[i + 1] : b[i];
            if (c + i >= wm) x = 0ull;
            if (c + i >= wh) y = 0ull;
            if (!found && i < n && x != y) { found = true; v = bswap64(x); h = bswap64(y); c += i; }
        }
        if (found) return c;
        c += n;
        if (c >= max_chunks) { bad = true; return c; }   // two equal words: cannot happen
    }
}

__global__ void __launch_bounds__(256, 4) rank_small_lcp_k(const u32 *__restrict__ hp, const u32 *__restrict__ gid,
                                                           const u32 *__restrict__ depth, const u64 *__restrict__ pool,
                                                           const u64 *__restrict__ uoff, const u32 *__restrict__ uwords,
                                                           const u32 *__restrict__ occ_of_word, u64 d, u32 max_chunks,
                                                           u32 *__restrict__ ord, u64 *__restrict__ flags) {
    __shared__ const u64 *s_ptr[8][64];        // per entry id: the word in the pool
    __shared__ u32 s_wn[8][64];                // ... its length in chunks
    __shared__ u32 s_uid[8][64];               // ... its id
    __shared__ u32 s_hkey[8][64];              // ... occurrences << 6 | entry id: the most frequent word heads its range
    __shared__ u32 s_best[8][64];              // per range start: (occurrences << 6 | entry id) of its head
    __shared__ u32 s_ka[8][64];                // per position: class/depth code of this round
    __shared__ u64 s_kb[8][64];                // ... and the chunk where the word left its head
    const u32 lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const u64 nwin = (d + 31) / 32;
    const u64 nwarps = (u64)gridDim.x * 8;
    for (u64 k = (u64)blockIdx.x * 8 + wp; k < nwin; k += nwarps) {
        const u64 w0 = k * 32;
        // entry 0: a group that starts inside the window; entry 1: the rest of the one group that crosses its end
        u32 s = 0, m = 0;
        if (w0 + lane < d) {
            const u32 g = gid[w0 + lane];
            s = hp[g];
            m = hp[g + 1] - s;
        }
        const bool in0 = m >= 2 && m <= WARP_MAX && s >= w0;
        const u32 end31 = __shfl_sync(0xffffffffu, in0 ? s + m : 0u, 31);   // end of the group at position 31
        const bool in1 = (u64)end31 > w0 + 32 + lane;
        if (!__any_sync(0xffffffffu, in0)) continue;
        const u32 s31 = __shfl_sync(0xffffffffu, s, 31), m31 = __shfl_sync(0xffffffffu, m, 31);
        u32 pos[2], lo[2], sz[2], dep[2];
#pragma unroll
        for (u32 e = 0; e < 2; e++) {
            const bool in = e ? in1 : in0;
            const u32 gs = e ? s31 : s, gm = e ? m31 : m;
            pos[e] = 32 * e + lane;
            s_uid[wp][pos[e]] = in ? ord[w0 + pos[e]] : 0u;
            lo[e] = in ? (u32)(gs - w0) : pos[e];
            sz[e] = in ? gm : 1u;
            dep[e] = in ? depth[gs] : 0u;
        }
#pragma unroll
        for (u32 e = 0; e < 2; e++) {
            const bool in = sz[e] > 1;
            const u32 u = s_uid[wp][pos[e]];
            const u32 c = in ? occ_of_word[u] : 0u;
            s_hkey[wp][pos[e]] = ((c < (1u << 26) ? c : (1u << 26) - 1) << 6) | pos[e];
            if (in) {
                s_ptr[wp][pos[e]] = pool + uoff[u];
                s_wn[wp][pos[e]] = uwords[u];
            }
        }
        for (;;) {
            const bool act0 = sz[0] > 1, act1 = sz[1] > 1;
            if (!__any_sync(0xffffffffu, act0 || act1)) break;
            // ---- head of every range: its most frequent word ----------------------------------------------
            if (act0 && pos[0] == lo[0]) s_best[wp][lo[0]] = 0;
            if (act1 && pos[1] == lo[1]) s_best[wp][lo[1]] = 0;
            __syncwarp();
            if (act0) atomicMax(&s_best[wp][lo[0]], s_hkey[wp][lane]);
            if (act1) atomicMax(&s_best[wp][lo[1]], s_hkey[wp][32 + lane]);
            __syncwarp();
            // ---- every other word of the range walks along the head -------------------------------------------
            // (one call site for both entries: the walk's loads take most of the registers)
            bool bad = false;
#pragma unroll 1
            for (u32 e = 0; e < 2; e++) {
                const u32 esz = e ? sz[1] : sz[0], elo = e ? lo[1] : lo[0], epos = e ? pos[1] : pos[0];
                if (esz > 1) {
                    const u32 hid = s_best[wp][elo] & 63u, me = 32 * e + lane;
                    u32 code = LCP_HEAD;
                    u64 v = 0, h = 0;
                    if (hid != me) {
                        const u32 c = small_walk(s_ptr[wp][me], s_wn[wp][me], s_ptr[wp][hid], s_wn[wp][hid],
                                                 e ? dep[1] : dep[0], max_chunks, v, h, bad);
                        code = v < h ? c : 2u * LCP_HEAD - 1u - c;
                    }
                    s_ka[wp][epos] = code;
                    s_kb[wp][epos] = v;
                }
            }
            if (__any_sync(0xffffffffu, bad)) {
                if (lane == 0) atomicOr((unsigned long long *)&flags[0], PFP_ERRBIT_INTERNAL);
                break;
            }
            __syncwarp();
            // ---- place every word among the words of its range; equal keys tie in the next round -------------
            u32 nlo[2], nsz[2], npos[2];
#pragma unroll
            for (u32 e = 0; e < 2; e++) {
                nlo[e] = lo[e]; nsz[e] = sz[e]; npos[e] = pos[e];
                if (sz[e] > 1) {
                    const u32 code = s_ka[wp][pos[e]];
                    const u64 kv = s_kb[wp][pos[e]];
                    u32 less = 0, eq = 0, eq_before = 0;
                    for (u32 q = lo[e]; q < lo[e] + sz[e]; q++) {
                        const u32 a1 = s_ka[wp][q];
                        const u64 b1 = s_kb[wp][q];
                        const bool same = a1 == code && b1 == kv;
                        less += lcp_less(a1, b1, code, kv) ? 1u : 0u;
                        eq += same ? 1u : 0u;
                        eq_before += (same && q < pos[e]) ? 1u : 0u;
                    }
                    nlo[e] = lo[e] + less;
                    nsz[e] = eq;
                    npos[e] = nlo[e] + eq_before;
                    if (code != LCP_HEAD) dep[e] = (code < LCP_HEAD ? code : 2u * LCP_HEAD - 1u - code) + 1;
                }
            }
            __syncwarp();
#pragma unroll
            for (u32 e = 0; e < 2; e++) { lo[e] = nlo[e]; sz[e] = nsz[e]; pos[e] = npos[e]; }
        }
        if (in0) ord[w0 + pos[0]] = s_uid[wp][lane];
        if (in1) ord[w0 + pos[1]] = s_uid[wp][32 + lane];
        __syncwarp();
    }
}

__global__ void __launch_bounds__(256) rank_cta_k(const u32 *__restrict__ hp,
                                                  const u32 *__restrict__ list,
                                                  const u32 *__restrict__ count,
                                                  const u32 *__restrict__ depth,
                                                  const u64 *pool, const u64 *uoff, const u32 *uwords,
                                                  u32 max_chunks, u32 *__restrict__ ord,
                                                  u64 *__restrict__ flags) {
    extern __shared__ __align__(16) unsigned char cta_raw[];
    TieSort<LOCAL_MAX> &S = *reinterpret_cast<TieSort<LOCAL_MAX> *>(cta_raw);
    __shared__ u64 sm_v[8];
    __shared__ u32 sm_f[8];
    const u32 n = *count;
    for (u32 q = blockIdx.x; q < n; q += gridDim.x) {
        const u32 g = list[q];
        const u32 s = hp[g], m = hp[g + 1] - s;
        tie_refine<256, LOCAL_MAX>(S, sm_v, sm_f, threadIdx.x, s, m, depth[s], pool, uoff, uwords, max_chunks, ord,
                                   flags);
    }
}

int pfp_rank_init(pfpb200_ctx *ctx) {
    PFP_CUDA(ctx, cudaFuncSetAttribute(rank_cta_k, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)sizeof(TieSort<LOCAL_MAX>)));
    PFP_CUDA(ctx, cudaFuncSetAttribute(rank_mid_k, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(8 * sizeof(TieSort<MID_MAX>))));
    PFP_CUDA(ctx, cudaFuncSetAttribute(rank_lcp_k, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)(8 * sizeof(LcpSort<LCP_MAX>))));
    PFP_CUDA(ctx, cudaFuncSetAttribute(rank_lcp_cta_k, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)sizeof(LcpSort<LOCAL_MAX>)));
    return PFPB200_OK;
}

int pfp_rank_stage(pfpb200_ctx *ctx, DictArrays &D, u32 **order, u32 *rounds, bool alpha_from_scan) {
    const int TB = 256;
    const u64 d = D.d;
    const u32 nbd = pfp_blocks(d, TB);
    const u32 max_chunks = (D.max_len + 7) / 8 + 1;
    u64 *k0 = nullptr, *k1 = nullptr, *ks = nullptr;
    u32 *v0 = nullptr, *v1 = nullptr, *vs = nullptr;
    u32 *ord = nullptr, *depth = nullptr, *hscan = nullptr, *hp = nullptr, *gid = nullptr;
    u8 *head = nullptr;
    AlphaMap *am = nullptr;
    u32 *amask = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &k0, d));
    PFP_TRY(pfp_alloc_t(ctx, &k1, d));
    PFP_TRY(pfp_alloc_t(ctx, &v0, d));
    PFP_TRY(pfp_alloc_t(ctx, &v1, d));
    PFP_TRY(pfp_alloc_t(ctx, &ord, d));
    PFP_TRY(pfp_alloc_t(ctx, &depth, d));
    PFP_TRY(pfp_alloc_t(ctx, &hscan, d));
    PFP_TRY(pfp_alloc_t(ctx, &hp, d + 1));
    PFP_TRY(pfp_alloc_t(ctx, &gid, d));
    PFP_TRY(pfp_alloc_t(ctx, &head, d));
    PFP_TRY(pfp_alloc_t(ctx, &am, 1));
    PFP_TRY(pfp_alloc_t(ctx, &amask, 8));
    // first key: alphabet-compacted prefix, one global sort
    if (alpha_from_scan) {             // K1 saw every byte of the text these words come from
        PFP_CUDA(ctx, cudaMemcpyAsync(amask, ctx->d_alpha, 8 * sizeof(u32), cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
        PFP_CUDA(ctx, cudaMemsetAsync(amask, 0, 8 * sizeof(u32), ctx->stream));
        alpha_presence_k<<<nbd, TB, 0, ctx->stream>>>(D.pool, D.uoff, D.ulen, d, amask);
        PFP_LAUNCHED(ctx);
    }
    alpha_build_k<<<1, 32, 0, ctx->stream>>>(amask, am, alpha_from_scan ? 1 : 0);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pfp_alloc_t(ctx, &D.meta, d));
    rank_keys0_k<<<nbd, TB, 0, ctx->stream>>>(D.pool, D.uoff, D.ulen, D.count, d, am, k0, v0, D.meta);
    PFP_LAUNCHED(ctx);
    // LSD passes only over the top 2 log2(d) + 2 key bits (whole bytes): with fewer, unrelated
    // words start to collide by chance (measured on 8 GB of random text: sorting 40 of 64 bits
    // saved 3 ms of sort passes and cost 9 ms of tie groups); with these, 6 or 7 passes instead
    // of 8 for 4 M .. 100 M words.  Words that agree on the sorted bits form the tie groups; the
    // tie kernels compare whole chunks, so nothing is lost.
    int lg = 1;
    while (lg < 32 && (1ull << lg) < d) lg++;
    int sort_bits = (2 * lg + 2 + 7) / 8 * 8;
    if (sort_bits > 64) sort_bits = 64;
    const int begin_bit = 64 - sort_bits;
    PFP_TRY(pfp_radix_sort_pairs(ctx, k0, v0, k1, v1, d, begin_bit, 64, &ks, &vs));
    rank_heads0_k<<<nbd, TB, 0, ctx->stream>>>(ks, d, am, (u32)begin_bit, head, depth);
    PFP_LAUNCHED(ctx);
    PFP_CUDA(ctx, cudaMemcpyAsync(ord, vs, d * sizeof(u32), cudaMemcpyDeviceToDevice, ctx->stream));

    u8 *act = nullptr, *gh = nullptr;
    u32 *ascan = nullptr, *gscan = nullptr, *apos = nullptr, *gid_of_u = nullptr, *depth2 = nullptr;
    u32 *d_nheads = reinterpret_cast<u32 *>(&ctx->d_flags[4]);
    // A/B (and words of 8 MB and more): the kernels the LCP walks replaced, one 8-byte chunk per pass
    const bool chunk_passes = ctx->rank_chunk_passes || max_chunks >= LCP_MAX_CHUNKS;
    const bool warp_passes = ctx->rank_warp_passes || max_chunks >= LCP_MAX_CHUNKS;
    u32 r = 1;
    bool big_bufs = false;
    for (;; r++) {
        // group table from the head flags
        PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[1], 0, 4 * sizeof(u64), ctx->stream));
        PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, head, hscan, d, d_nheads));
        groups_compact_k<<<nbd, TB, 0, ctx->stream>>>(head, hscan, d, d_nheads, hp, gid);
        PFP_LAUNCHED(ctx);
        if (d < 2) break;
        // finish every tie group of up to LOCAL_MAX words on chip; the larger ones (none, unless a
        // family has thousands of members) go through a global round and come back here split
        u32 *mid_list = v1, *big_list = v0;      // sort buffers are free until the global round
        u32 *counts = reinterpret_cast<u32 *>(&ctx->d_flags[5]);
        PFP_CUDA(ctx, cudaMemsetAsync(counts, 0, 4 * sizeof(u32), ctx->stream));
        rank_lists_k<<<nbd, TB, 0, ctx->stream>>>(hp, d_nheads, d, mid_list, big_list,
                                                  warp_passes ? reinterpret_cast<u32 *>(k1) : nullptr, counts);
        PFP_LAUNCHED(ctx);
        u64 want = (d / 2 + 7) / 8;
        u64 maxb = (u64)ctx->sm_count * 16;
        u32 nbw = (u32)(want < maxb ? want : maxb);
        if (nbw == 0) nbw = 1;
        if (warp_passes) {
            rank_window_k<<<nbw, 256, 0, ctx->stream>>>(hp, gid, depth, D.pool, D.uoff, D.uwords, d, max_chunks, 0,
                                                        ord, ctx->d_flags);
            PFP_LAUNCHED(ctx);
            // (a second pass over windows shifted by 16 for the groups straddling a border was measured:
            //  it costs what it saves -- the kernels are bound by their chains of dependent loads)
            rank_warp_k<<<nbw, 256, 0, ctx->stream>>>(hp, reinterpret_cast<u32 *>(k1), counts + 2, depth, D.pool,
                                                      D.uoff, D.uwords, max_chunks, ord, ctx->d_flags);
        } else {
            rank_small_lcp_k<<<nbw, 256, 0, ctx->stream>>>(hp, gid, depth, D.pool, D.uoff, D.uwords, D.count, d,
                                                           max_chunks, ord, ctx->d_flags);
        }
        PFP_LAUNCHED(ctx);
        if (chunk_passes)
            rank_mid_k<<<ctx->sm_count * 4, 256, 8 * sizeof(TieSort<MID_MAX>), ctx->stream>>>(
                hp, mid_list, counts, depth, D.pool, D.uoff, D.uwords, max_chunks, ord, ctx->d_flags);
        else
            rank_lcp_k<<<ctx->sm_count * 6, 256, 8 * sizeof(LcpSort<LCP_MAX>), ctx->stream>>>(
                hp, mid_list, counts, depth, D.pool, D.uoff, D.uwords, D.count, max_chunks, ord, ctx->d_flags);
        PFP_LAUNCHED(ctx);
        if (chunk_passes)
            rank_cta_k<<<ctx->sm_count * 4, 256, sizeof(TieSort<LOCAL_MAX>), ctx->stream>>>(
                hp, big_list, counts + 1, depth, D.pool, D.uoff, D.uwords, max_chunks, ord, ctx->d_flags);
        else
            rank_lcp_cta_k<<<ctx->sm_count * 3, 256, sizeof(LcpSort<LOCAL_MAX>), ctx->stream>>>(
                hp, big_list, counts + 1, depth, D.pool, D.uoff, D.uwords, D.count, max_chunks, ord, ctx->d_flags);
        PFP_LAUNCHED(ctx);
        PFP_CUDA(ctx, cudaMemcpyAsync(ctx->h_flags, ctx->d_flags, 7 * sizeof(u64), cudaMemcpyDeviceToHost,
                                      ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (ctx->h_flags[0] & PFP_ERRBIT_INTERNAL)
            return pfp_fail(ctx, PFPB200_E_INTERNAL, "ranking found words that never differ (duplicates?)");
        if (reinterpret_cast<const u32 *>(&ctx->h_flags[5])[3] == 0) break;
        if (!big_bufs) {
            PFP_TRY(pfp_alloc_t(ctx, &act, d));
            PFP_TRY(pfp_alloc_t(ctx, &gh, d));
            PFP_TRY(pfp_alloc_t(ctx, &ascan, d));
            PFP_TRY(pfp_alloc_t(ctx, &gscan, d));
            big_bufs = true;
        }
        rank_active_k<<<nbd, TB, 0, ctx->stream>>>(head, gid, hp, d, act, gh);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, act, ascan, d, reinterpret_cast<u32 *>(&ctx->d_flags[1])));
        PFP_TRY(pfp_exclusive_scan_u8_u32(ctx, gh, gscan, d, reinterpret_cast<u32 *>(&ctx->d_flags[2])));
        PFP_CUDA(ctx, cudaMemcpyAsync(ctx->h_flags, ctx->d_flags, 3 * sizeof(u64),
                                      cudaMemcpyDeviceToHost, ctx->stream));
        PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        u64 m = (u32)ctx->h_flags[1], ng = (u32)ctx->h_flags[2];
        if (r > max_chunks + 1)
            return pfp_fail(ctx, PFPB200_E_INTERNAL,
                            "ranking did not separate %llu words after %u rounds (duplicate words?)",
                            (unsigned long long)m, r);
        if (!apos) {
            PFP_TRY(pfp_alloc_t(ctx, &apos, d));
            PFP_TRY(pfp_alloc_t(ctx, &gid_of_u, d));
            PFP_TRY(pfp_alloc_t(ctx, &depth2, d));
        }
        rank_compact_k<<<nbd, TB, 0, ctx->stream>>>(act, gh, ascan, gscan, ord, gid, hp, depth, d, D.pool,
                                                    D.uoff, D.uwords, apos, k0, v0, gid_of_u);
        PFP_LAUNCHED(ctx);
        PFP_TRY(pfp_radix_sort_pairs(ctx, k0, v0, k1, v1, m, 0, 64, &ks, &vs));
        // second key: the tie group, stable, only as many bits as there are groups
        u64 *g_in = (ks == k0) ? k1 : k0;
        u32 *v_other = (vs == v0) ? v1 : v0;
        const u32 nbm = pfp_blocks(m, TB);
        rank_gidkeys_k<<<nbm, TB, 0, ctx->stream>>>(vs, gid_of_u, m, g_in);
        PFP_LAUNCHED(ctx);
        int bits = 1;
        while (bits < 32 && (1ull << bits) < ng) bits++;
        u64 *gs = nullptr;
        u32 *vs2 = nullptr;
        PFP_TRY(pfp_radix_sort_pairs(ctx, g_in, vs, ks, v_other, m, 0, bits, &gs, &vs2));
        PFP_CUDA(ctx, cudaMemcpyAsync(depth2, depth, d * sizeof(u32), cudaMemcpyDeviceToDevice, ctx->stream));
        rank_writeback_k<<<nbm, TB, 0, ctx->stream>>>(apos, gs, vs2, m, gid, hp, depth, D.pool, D.uoff,
                                                      D.uwords, ord, head, depth2);
        PFP_LAUNCHED(ctx);
        u32 *tdp = depth; depth = depth2; depth2 = tdp;
    }
    *rounds = r;
    *order = ord;
    void *to_free[] = {k0, k1, v0, v1, depth, depth2, hscan, hp, gid, head, am, amask, act, gh, ascan,
                       gscan, apos, gid_of_u};
    for (void *q : to_free) PFP_TRY(pfp_free_now(ctx, q));
    return PFPB200_OK;
}

// ---- .dict / .occ -----------------------------------------------------------------------------------
__device__ __forceinline__ void out_span(const u64 *pool, u64 off, u32 len, u32 strip_w, u32 *skip,
                                         u32 *outlen) {
    // -c mode (newscan.cpp:410-413): drop the last w bytes and a leading 0x02
    *skip = 0;
    *outlen = len;
    if (strip_w) {
        u32 l = len - strip_w;
        if ((u8)(pool[off] & 0xFF) == PFP_DOLLAR) { *skip = 1; l -= 1; }
        *outlen = l;
    }
}

__global__ void dict_layout_k(const u32 *__restrict__ ord, u64 d, const DictArrays D, u32 strip_w,
                              u32 *__restrict__ rank_of_uid, u32 *__restrict__ occ,
                              u32 *__restrict__ dl) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d) return;
    u32 u = ord[i];
    rank_of_uid[u] = (u32)i + 1;                     // 1-based (newscan.cpp:405,436)
    const uint4 mv = __ldg(reinterpret_cast<const uint4 *>(D.meta + u));     // one sector: offset, length, count
    occ[i] = mv.w;                                   // newscan.cpp:433
    u32 skip, outlen;
    out_span(D.pool, ((u64)mv.y << 32) | mv.x, mv.z, strip_w, &skip, &outlen);
    dl[i] = outlen + 1;                              // + EndOfWord (newscan.cpp:416)
}

// the ranks laid out by dictionary-table slot, for the records that hold a slot instead of a word
// id (DictArrays::slot_of_word): only words met more than once have such records
__global__ void rank_of_slot_k(const u32 *__restrict__ slot_of_word, const u32 *__restrict__ count,
                               const u32 *__restrict__ rank_of_uid, u64 d, u32 *__restrict__ rank_of_slot) {
    u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < d && count[u] > 1) rank_of_slot[slot_of_word[u]] = rank_of_uid[u];
}

constexpr int DC_T = 256;
constexpr int DC_GROUP = 8;

// One 8-lane group per word.  The source (pool) is 8-byte aligned, the destination is not: the
// bytes up to the destination's next 8-byte boundary and the last <8 bytes go out as byte
// stores, everything between as aligned 8-byte stores of funnel-shifted pool words.
__global__ void __launch_bounds__(DC_T) dict_copy_k(const u32 *__restrict__ ord,
                                                    const u64 *__restrict__ doff, u64 d,
                                                    const DictArrays D, u32 strip_w, u64 total,
                                                    u8 *__restrict__ dict) {
    const u32 li = threadIdx.x & (DC_GROUP - 1);
    if (blockIdx.x == 0 && threadIdx.x == 0) dict[total] = (u8)PFP_END_OF_DICT;   // :438
    for (u64 i = (u64)blockIdx.x * (DC_T / DC_GROUP) + (threadIdx.x / DC_GROUP); i < d;
         i += (u64)gridDim.x * (DC_T / DC_GROUP)) {
        const u32 u = ord[i];
        u32 skip, outlen;
        const uint4 mv = __ldg(reinterpret_cast<const uint4 *>(D.meta + u));
        const u64 off = ((u64)mv.y << 32) | mv.x;
        out_span(D.pool, off, mv.z, strip_w, &skip, &outlen);
        const u64 *src64 = D.pool + off;
        const u8 *src = reinterpret_cast<const u8 *>(src64) + skip;
        u8 *dst = dict + doff[i];
        u32 head = (u32)((8 - ((uintptr_t)dst & 7)) & 7);
        if (head > outlen) head = outlen;
        if (li < head) dst[li] = src[li];
        const u32 nbody = (outlen - head) >> 3;
        u64 *dst64 = reinterpret_cast<u64 *>(dst + head);
        for (u32 k = li; k < nbody; k += DC_GROUP) {
            u32 so = skip + head + 8 * k;
            u32 sh = (so & 7) * 8;
            u64 w0 = __ldg(src64 + (so >> 3));
            u64 v = w0;
            if (sh) v = (w0 >> sh) | (__ldg(src64 + (so >> 3) + 1) << (64 - sh));
            dst64[k] = v;
        }
        const u32 done = head + 8 * nbody;
        if (li < outlen - done) dst[done + li] = src[done + li];
        if (li == DC_GROUP - 1) dst[outlen] = (u8)PFP_END_OF_WORD;                 // :416
    }
}

__global__ void remap_k(const u32 *__restrict__ uid, const u32 *__restrict__ rank_of_uid, u64 P,
                        u32 *__restrict__ parse, const u32 *__restrict__ rank_of_slot);

// remap_uid / remap_out non-null: K5 (remap_out[j] = rank of remap_uid[j], j < remap_n) is launched
// on the context's aux stream as soon as the ranks exist and runs beside the .dict gather; the
// main stream waits for it before this function returns.  With D.slot_of_word, remap_uid holds
// table slots for most records (DictArrays): the ranks are then also laid out by slot, for the remap.
int pfp_dict_stage(pfpb200_ctx *ctx, const DictArrays &D, const u32 *order, u32 strip_w, u8 **dict,
                   u64 *dict_bytes, u32 **occ, u32 **rank_of_uid, const u32 *remap_uid, u64 remap_n,
                   u32 *remap_out) {
    const int TB = 256;
    const u64 d = D.d;
    u32 *dl = nullptr;
    u64 *doff = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, occ, d, true));
    PFP_TRY(pfp_alloc_t(ctx, rank_of_uid, d));
    PFP_TRY(pfp_alloc_t(ctx, &dl, d));
    PFP_TRY(pfp_alloc_t(ctx, &doff, d));
    const bool side_remap = remap_uid && remap_out && remap_n;
    u32 *rank_of_slot = nullptr;
    if (side_remap && D.slot_of_word) PFP_TRY(pfp_alloc_t(ctx, &rank_of_slot, D.slots));
    dict_layout_k<<<pfp_blocks(d, TB), TB, 0, ctx->stream>>>(order, d, D, strip_w, *rank_of_uid, *occ, dl);
    PFP_LAUNCHED(ctx);
    if (side_remap) {
        PFP_CUDA(ctx, cudaEventRecord(ctx->ev_aux0, ctx->stream));
        PFP_CUDA(ctx, cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_aux0, 0));
        if (rank_of_slot) {
            rank_of_slot_k<<<pfp_blocks(d, TB), TB, 0, ctx->aux_stream>>>(D.slot_of_word, D.count, *rank_of_uid, d,
                                                                          rank_of_slot);
            PFP_LAUNCHED(ctx);
        }
        remap_k<<<pfp_blocks((remap_n + 3) / 4, 256), 256, 0, ctx->aux_stream>>>(remap_uid, *rank_of_uid, remap_n,
                                                                                 remap_out, rank_of_slot);
        PFP_LAUNCHED(ctx);
        PFP_CUDA(ctx, cudaEventRecord(ctx->ev_aux1, ctx->aux_stream));
    }
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, dl, doff, d, &ctx->d_flags[1]));
    PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[1], &ctx->d_flags[1], sizeof(u64),
                                  cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    u64 total = ctx->h_flags[1];
    *dict_bytes = total + 1;
    PFP_TRY(pfp_alloc_t(ctx, dict, (size_t)(total + 1), true));
    u64 want = (d + (DC_T / DC_GROUP) - 1) / (DC_T / DC_GROUP);
    u64 maxb = (u64)ctx->sm_count * 32;
    u32 nb = (u32)(want < maxb ? want : maxb);
    if (nb == 0) nb = 1;
    dict_copy_k<<<nb, DC_T, 0, ctx->stream>>>(order, doff, d, D, strip_w, total, *dict);
    PFP_LAUNCHED(ctx);
    if (side_remap) PFP_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_aux1, 0));
    PFP_TRY(pfp_free_now(ctx, rank_of_slot));
    PFP_TRY(pfp_free_now(ctx, dl));
    PFP_TRY(pfp_free_now(ctx, doff));
    return PFPB200_OK;
}

// ---- K5 -----------------------------------------------------------------------------------------------
// rank_of_slot non-null: uid[] as DictArrays::slot_of_word describes it
__device__ __forceinline__ u32 rank_of(u32 v, const u32 *__restrict__ rank_of_uid, const u32 *__restrict__ rank_of_slot) {
    if (rank_of_slot && !(v & UID_CREATOR)) return __ldg(rank_of_slot + v);
    return __ldg(rank_of_uid + (v & ~UID_CREATOR));                                  // newscan.cpp:456-458
}

// four phrases per thread: four independent gathers in flight
__global__ void remap_k(const u32 *__restrict__ uid, const u32 *__restrict__ rank_of_uid, u64 P,
                        u32 *__restrict__ parse, const u32 *__restrict__ rank_of_slot) {
    const u64 q = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 j = 4 * q;
    if (j + 4 <= P && (((uintptr_t)uid | (uintptr_t)parse) & 15) == 0) {
        const uint4 v = __ldcs(reinterpret_cast<const uint4 *>(uid) + q);
        uint4 r;
        r.x = rank_of(v.x, rank_of_uid, rank_of_slot); r.y = rank_of(v.y, rank_of_uid, rank_of_slot);
        r.z = rank_of(v.z, rank_of_uid, rank_of_slot); r.w = rank_of(v.w, rank_of_uid, rank_of_slot);
        reinterpret_cast<uint4 *>(parse)[q] = r;
    } else {
        for (u64 i = j; i < P && i < j + 4; i++) parse[i] = rank_of(uid[i], rank_of_uid, rank_of_slot);
    }
}

int pfp_remap_stage(pfpb200_ctx *ctx, const u32 *uid, const u32 *rank_of_uid, u64 P, u32 *parse) {
    remap_k<<<pfp_blocks((P + 3) / 4, 256), 256, 0, ctx->stream>>>(uid, rank_of_uid, P, parse, nullptr);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

// ---- routing (range-partitioned dictionary merge) ----------------------------------------------------
struct Splitters { u64 s[PFPB200_MAX_RANKS]; u32 n; };

__global__ void first_keys_k(const u64 *__restrict__ pool, const u64 *__restrict__ uoff,
                             const u32 *__restrict__ uwords, u64 d, u64 *__restrict__ keys) {
    u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < d) keys[u] = word_key(pool, uoff, uwords, (u32)u, 0);
}

__global__ void route_dest_k(const u64 *__restrict__ pool, const u64 *__restrict__ uoff,
                             const u32 *__restrict__ uwords, u64 d, Splitters sp,
                             u64 *__restrict__ keys, u32 *__restrict__ vals,
                             unsigned long long *__restrict__ cnt /* [2*MAX_RANKS] */) {
    __shared__ unsigned long long sc[2 * PFPB200_MAX_RANKS];
    for (int i = threadIdx.x; i < 2 * PFPB200_MAX_RANKS; i += blockDim.x) sc[i] = 0;
    __syncthreads();
    u64 u = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < d) {
        u64 k = word_key(pool, uoff, uwords, (u32)u, 0);
        u32 dest = 0;
        for (u32 i = 0; i < sp.n; i++) dest += (sp.s[i] <= k) ? 1u : 0u;
        keys[u] = dest;
        vals[u] = (u32)u;
        atomicAdd(&sc[dest], 1ull);
        atomicAdd(&sc[PFPB200_MAX_RANKS + dest], (unsigned long long)uwords[u]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * PFPB200_MAX_RANKS; i += blockDim.x)
        if (sc[i]) atomicAdd(&cnt[i], sc[i]);
}

__global__ void route_gather_k(const u32 *__restrict__ perm, u64 d, const u64 *__restrict__ fpa,
                               const u64 *__restrict__ fpb, const u32 *__restrict__ len,
                               const u32 *__restrict__ count, const u32 *__restrict__ uwords,
                               pfpb200_word *__restrict__ out, u32 *__restrict__ ouwords) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d) return;
    u32 u = perm[i];
    u64 a = fpa[u], b = fpb[u];
    u32 uw = uwords[u];
    uint4 *q = reinterpret_cast<uint4 *>(out + i);
    q[0] = make_uint4((u32)a, (u32)(a >> 32), (u32)b, (u32)(b >> 32));
    q[1] = make_uint4(len[u], count[u], uw, 0u);
    ouwords[i] = uw;
}

__global__ void gather_u32_k(const u32 *__restrict__ perm, const u32 *__restrict__ in, u64 d, u32 *__restrict__ out) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < d) out[i] = in[perm[i]];
}

// wire records -> the separate arrays the merge stage works on
__global__ void unpack_words_k(const pfpb200_word *__restrict__ in, u64 n, u64 *__restrict__ fpa,
                               u64 *__restrict__ fpb, u32 *__restrict__ len, u32 *__restrict__ count,
                               u32 *__restrict__ uwords) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint4 *q = reinterpret_cast<const uint4 *>(in + i);
    uint4 a = __ldg(q), b = __ldg(q + 1);
    fpa[i] = ((u64)a.y << 32) | a.x;
    fpb[i] = ((u64)a.w << 32) | a.z;
    len[i] = b.x; count[i] = b.y; uwords[i] = b.z;
}

extern "C" int pfp_unpack_words(pfpb200_ctx *ctx, const pfpb200_word *in, u64 n, u64 *fpa, u64 *fpb,
                                u32 *len, u32 *count, u32 *uwords) {
    unpack_words_k<<<pfp_blocks(n, 256), 256, 0, ctx->stream>>>(in, n, fpa, fpb, len, count, uwords);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

__global__ void __launch_bounds__(256) route_pool_k(const u32 *__restrict__ perm, u64 d,
                                                    const u64 *__restrict__ pool,
                                                    const u64 *__restrict__ uoff,
                                                    const u32 *__restrict__ uwords,
                                                    const u64 *__restrict__ ooff,
                                                    u64 *__restrict__ opool) {
    const u32 li = threadIdx.x & 7;
    for (u64 i = (u64)blockIdx.x * 32 + (threadIdx.x >> 3); i < d; i += (u64)gridDim.x * 32) {
        u32 u = perm[i];
        const u64 *src = pool + uoff[u];
        u64 *dst = opool + ooff[i];
        u32 nw = uwords[u];
        for (u32 k = li; k < nw; k += 8) dst[k] = __ldg(src + k);
    }
}

// keys of every step-th word only: what the splitter sample needs
__global__ void sample_keys_k(const u64 *__restrict__ pool, const u64 *__restrict__ uoff,
                              const u32 *__restrict__ uwords, u64 d, u64 step, u32 n, u64 *__restrict__ keys) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 u = (u64)i * step;
    keys[i] = u < d ? word_key(pool, uoff, uwords, (u32)u, 0) : 0ull;
}

extern "C" int pfpb200_shard_sample_keys(pfpb200_ctx *ctx, uint32_t max_samples, uint64_t *h_keys, uint32_t *n_keys) {
    if (!ctx || !h_keys || !n_keys || max_samples == 0) return PFPB200_E_ARG;
    *n_keys = 0;
    const u64 d = ctx->sh.d;
    if (d == 0) return PFPB200_OK;
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    const u64 step = d / max_samples ? d / max_samples : 1;
    const u32 n = (u32)((d + step - 1) / step < max_samples ? (d + step - 1) / step : max_samples);
    u64 *keys = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &keys, n));
    sample_keys_k<<<pfp_blocks(n, 256), 256, 0, ctx->stream>>>(ctx->sh.pool, ctx->sh.uoff, ctx->sh.uwords, d, step, n, keys);
    PFP_LAUNCHED(ctx);
    PFP_CUDA(ctx, cudaMemcpyAsync(h_keys, keys, (size_t)n * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    PFP_TRY(pfp_free_now(ctx, keys));
    *n_keys = n;
    return PFPB200_OK;
}

extern "C" int pfp_first_keys_impl(pfpb200_ctx *ctx, u64 **keys) {
    const u64 d = ctx->sh.d;
    PFP_TRY(pfp_alloc_t(ctx, keys, d, true));
    first_keys_k<<<pfp_blocks(d, 256), 256, 0, ctx->stream>>>(ctx->sh.pool, ctx->sh.uoff, ctx->sh.uwords, d, *keys);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

// ---- routing fused with the exchange: store straight into the owners' buffers (NVLink peer memory) ----
struct RouteDst {
    u64 so[PFPB200_MAX_RANKS + 1];        // routed positions [so[q], so[q+1]) go to owner q
    u64 pso[PFPB200_MAX_RANKS + 1];       // the same in pool words
    u64 word_dst[PFPB200_MAX_RANKS];      // address of this rank's first record in owner q's buffer
    u64 pool_dst[PFPB200_MAX_RANKS];      // ... and of its first pool word
    u32 n;
};

__device__ __forceinline__ u32 route_owner(const RouteDst &R, u64 i) {
    u32 q = 0;
    while (q + 1 < R.n && i >= R.so[q + 1]) q++;
    return q;
}

// eight lanes per word (one warp per word, 256-byte stores, was slower: 1.73 vs 1.39 ms on 2 GPUs)
__global__ void __launch_bounds__(256) route_push_k(const u32 *__restrict__ perm, u64 d,
                                                    const u64 *__restrict__ fpa, const u64 *__restrict__ fpb,
                                                    const u32 *__restrict__ len, const u32 *__restrict__ count,
                                                    const u64 *__restrict__ pool, const u64 *__restrict__ uoff,
                                                    const u32 *__restrict__ uwords, const u64 *__restrict__ ooff,
                                                    const RouteDst R) {
    const u32 li = threadIdx.x & 7;
    for (u64 i = (u64)blockIdx.x * 32 + (threadIdx.x >> 3); i < d; i += (u64)gridDim.x * 32) {
        const u32 u = perm[i];
        const u32 q = route_owner(R, i);
        const u32 nw = uwords[u];
        if (li == 0) {                                       // the 32-byte wire record
            const u64 a = fpa[u], b = fpb[u];
            uint4 *rec = reinterpret_cast<uint4 *>(R.word_dst[q]) + 2 * (i - R.so[q]);
            rec[0] = make_uint4((u32)a, (u32)(a >> 32), (u32)b, (u32)(b >> 32));
            rec[1] = make_uint4(len[u], count[u], nw, 0u);
        }
        const u64 *src = pool + uoff[u];
        u64 *dst = reinterpret_cast<u64 *>(R.pool_dst[q]) + (ooff[i] - R.pso[q]);
        for (u32 k = li; k < nw; k += 8) dst[k] = __ldg(src + k);
    }
}

// plan: owner of every word, routed order (perm), per-owner counts; kept in the context for the push
extern "C" int pfp_route_plan_impl(pfpb200_ctx *ctx, const Splitters &sp, u32 n_ranks, u64 *words_to, u64 *pool_to,
                                   const u32 **perm_out) {
    const u64 d = ctx->sh.d;
    const u32 nbd = pfp_blocks(d, 256);
    u64 *k0 = nullptr, *k1 = nullptr, *ks = nullptr, *ooff = nullptr;
    u32 *v0 = nullptr, *v1 = nullptr, *perm = nullptr, *ouwords = nullptr;
    unsigned long long *cnt = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &k0, d));
    PFP_TRY(pfp_alloc_t(ctx, &k1, d));
    PFP_TRY(pfp_alloc_t(ctx, &v0, d));
    PFP_TRY(pfp_alloc_t(ctx, &v1, d));
    PFP_TRY(pfp_alloc_t(ctx, &cnt, 2 * PFPB200_MAX_RANKS));
    PFP_CUDA(ctx, cudaMemsetAsync(cnt, 0, 2 * PFPB200_MAX_RANKS * sizeof(unsigned long long), ctx->stream));
    route_dest_k<<<nbd, 256, 0, ctx->stream>>>(ctx->sh.pool, ctx->sh.uoff, ctx->sh.uwords, d, sp, k0, v0, cnt);
    PFP_LAUNCHED(ctx);
    int bits = 1;
    while ((1u << bits) < n_ranks) bits++;
    PFP_TRY(pfp_radix_sort_pairs(ctx, k0, v0, k1, v1, d, 0, bits, &ks, &perm));
    PFP_TRY(pfp_alloc_t(ctx, &ouwords, d));
    PFP_TRY(pfp_alloc_t(ctx, &ooff, d));
    gather_u32_k<<<nbd, 256, 0, ctx->stream>>>(perm, ctx->sh.uwords, d, ouwords);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, ouwords, ooff, d, nullptr));
    unsigned long long hc[2 * PFPB200_MAX_RANKS];
    PFP_CUDA(ctx, cudaMemcpyAsync(hc, cnt, sizeof(hc), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (u32 r = 0; r < PFPB200_MAX_RANKS; r++) {
        words_to[r] = hc[r];
        pool_to[r] = hc[PFPB200_MAX_RANKS + r];
        ctx->sh.route_words_to[r] = hc[r];
        ctx->sh.route_pool_to[r] = hc[PFPB200_MAX_RANKS + r];
    }
    ctx->sh.route_perm = perm;
    ctx->sh.route_ooff = ooff;
    *perm_out = perm;
    u32 *perm_other = (perm == v0) ? v1 : v0;
    PFP_TRY(pfp_free_now(ctx, k0));
    PFP_TRY(pfp_free_now(ctx, k1));
    PFP_TRY(pfp_free_now(ctx, perm_other));
    PFP_TRY(pfp_free_now(ctx, cnt));
    PFP_TRY(pfp_free_now(ctx, ouwords));
    return PFPB200_OK;
}

extern "C" int pfp_route_push_impl(pfpb200_ctx *ctx, u32 n_ranks, const u64 *word_dst, const u64 *pool_dst) {
    const u64 d = ctx->sh.d;
    RouteDst R;
    memset(&R, 0, sizeof(R));
    R.n = n_ranks;
    for (u32 q = 0; q < n_ranks; q++) {
        R.so[q + 1] = R.so[q] + ctx->sh.route_words_to[q];
        R.pso[q + 1] = R.pso[q] + ctx->sh.route_pool_to[q];
        R.word_dst[q] = word_dst[q];
        R.pool_dst[q] = pool_dst[q];
    }
    u64 want = (d + 31) / 32, maxb = (u64)ctx->sm_count * 32;
    u32 nb = (u32)(want < maxb ? want : maxb);
    route_push_k<<<nb ? nb : 1, 256, 0, ctx->stream>>>(ctx->sh.route_perm, d, ctx->sh.wfpa, ctx->sh.wfpb, ctx->sh.ulen,
                                                       ctx->sh.count, ctx->sh.pool, ctx->sh.uoff, ctx->sh.uwords,
                                                       ctx->sh.route_ooff, R);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

extern "C" int pfp_route_impl(pfpb200_ctx *ctx, const Splitters &sp, u32 n_ranks, pfpb200_routed *out) {
    const u64 d = ctx->sh.d;
    const u32 nbd = pfp_blocks(d, 256);
    u64 *k0 = nullptr, *k1 = nullptr, *ks = nullptr, *ooff = nullptr;
    u32 *v0 = nullptr, *v1 = nullptr, *perm = nullptr;
    unsigned long long *cnt = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &k0, d));
    PFP_TRY(pfp_alloc_t(ctx, &k1, d));
    PFP_TRY(pfp_alloc_t(ctx, &v0, d));
    PFP_TRY(pfp_alloc_t(ctx, &v1, d));
    PFP_TRY(pfp_alloc_t(ctx, &cnt, 2 * PFPB200_MAX_RANKS));
    PFP_CUDA(ctx, cudaMemsetAsync(cnt, 0, 2 * PFPB200_MAX_RANKS * sizeof(unsigned long long), ctx->stream));
    route_dest_k<<<nbd, 256, 0, ctx->stream>>>(ctx->sh.pool, ctx->sh.uoff, ctx->sh.uwords, d, sp, k0, v0, cnt);
    PFP_LAUNCHED(ctx);
    int bits = 1;
    while ((1u << bits) < n_ranks) bits++;
    PFP_TRY(pfp_radix_sort_pairs(ctx, k0, v0, k1, v1, d, 0, bits, &ks, &perm));
    u64 *opool = nullptr;
    pfpb200_word *owords = nullptr;
    u32 *ouwords = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &owords, d));
    PFP_TRY(pfp_alloc_t(ctx, &ouwords, d));
    PFP_TRY(pfp_alloc_t(ctx, &ooff, d));
    PFP_TRY(pfp_alloc_t(ctx, &opool, (size_t)ctx->sh.pool_words));
    route_gather_k<<<nbd, 256, 0, ctx->stream>>>(perm, d, ctx->sh.wfpa, ctx->sh.wfpb, ctx->sh.ulen, ctx->sh.count,
                                                 ctx->sh.uwords, owords, ouwords);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, ouwords, ooff, d, nullptr));
    u64 want = (d + 31) / 32, maxb = (u64)ctx->sm_count * 32;
    u32 nb = (u32)(want < maxb ? want : maxb);
    route_pool_k<<<nb ? nb : 1, 256, 0, ctx->stream>>>(perm, d, ctx->sh.pool, ctx->sh.uoff, ctx->sh.uwords, ooff, opool);
    PFP_LAUNCHED(ctx);
    unsigned long long hc[2 * PFPB200_MAX_RANKS];
    PFP_CUDA(ctx, cudaMemcpyAsync(hc, cnt, sizeof(hc), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (u32 r = 0; r < PFPB200_MAX_RANKS; r++) {
        out->words_to[r] = hc[r];
        out->pool_to[r] = hc[PFPB200_MAX_RANKS + r];
    }
    out->words = owords;
    out->pool = opool; out->perm = perm;
    for (u32 q = 0; q < PFPB200_MAX_RANKS; q++) {
        ctx->sh.route_words_to[q] = hc[q];
        ctx->sh.route_pool_to[q] = hc[PFPB200_MAX_RANKS + q];
    }
    ctx->sh.route_perm = perm;
    // free what the caller does not need; the rest is promoted to `held` by the caller
    u32 *perm_other = (perm == v0) ? v1 : v0;
    PFP_TRY(pfp_free_now(ctx, k0));
    PFP_TRY(pfp_free_now(ctx, k1));
    PFP_TRY(pfp_free_now(ctx, perm_other));
    PFP_TRY(pfp_free_now(ctx, cnt));
    PFP_TRY(pfp_free_now(ctx, ooff));
    PFP_TRY(pfp_free_now(ctx, ouwords));
    return PFPB200_OK;
}

// ---- ranks travelling back (range-partitioned merge) ------------------------------------------------------
// back[i] = rank, inside its owner's range, of the word this shard routed to position i; the
// global rank adds the number of distinct words in the ranges below that owner.
struct OwnerBase {
    u64 so[PFPB200_MAX_RANKS + 1];        // routed positions [so[q], so[q+1]) went to owner q
    u32 base[PFPB200_MAX_RANKS];
    u32 n;
};

__global__ void ranks_unroute_k(const u32 *__restrict__ perm, const u32 *__restrict__ back, u64 d,
                                const OwnerBase B, u32 *__restrict__ rank_of_word) {
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d) return;
    u32 q = 0;
    while (q + 1 < B.n && i >= B.so[q + 1]) q++;
    rank_of_word[perm[i]] = back[i] + B.base[q];
}

extern "C" int pfpb200_shard_ranks_back(pfpb200_ctx *ctx, uint32_t n_ranks, const uint32_t *d_back,
                                        const uint64_t *rank_base, const uint32_t **d_rank_of_word) {
    if (!ctx || !d_rank_of_word || n_ranks < 1 || n_ranks > PFPB200_MAX_RANKS || !rank_base) return PFPB200_E_ARG;
    *d_rank_of_word = nullptr;
    const u64 d = ctx->sh.d;
    if (d == 0) return PFPB200_OK;
    if (!ctx->sh.route_perm || !d_back) return pfp_fail(ctx, PFPB200_E_ARG, "shard_ranks_back before shard_route");
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    OwnerBase B;
    memset(&B, 0, sizeof(B));
    B.n = n_ranks;
    for (u32 q = 0; q < n_ranks; q++) {
        B.so[q + 1] = B.so[q] + ctx->sh.route_words_to[q];
        if (rank_base[q] > 0x7FFFFFFFull) return pfp_fail(ctx, PFPB200_E_LIMIT, "more than 2^31-2 distinct words");
        B.base[q] = (u32)rank_base[q];
    }
    u32 *out = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &out, d, true));
    ranks_unroute_k<<<pfp_blocks(d, 256), 256, 0, ctx->stream>>>(ctx->sh.route_perm, d_back, d, B, out);
    PFP_LAUNCHED(ctx);
    *d_rank_of_word = out;
    return PFPB200_OK;
}

// ---- self-check: the dictionary is strictly increasing (std::sort order, newscan.cpp:387-390,636) ---------
// One thread per adjacent pair of a .dict byte stream (words end in 0x01): word i must be
// strictly smaller than word i+1 in unsigned-byte order, a proper prefix counting as smaller.
__global__ void dict_order_check_k(const u8 *__restrict__ dict, const u64 *__restrict__ seps, u64 d,
                                   unsigned long long *__restrict__ bad) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i + 1 >= d) return;
    const u64 a0 = i ? seps[i - 1] + 1 : 0, a1 = seps[i];          // word i   = dict[a0, a1)
    const u64 b0 = a1 + 1, b1 = seps[i + 1];                        // word i+1 = dict[b0, b1)
    const u64 la = a1 - a0, lb = b1 - b0;
    const u64 m = la < lb ? la : lb;
    u64 k = 0;
    while (k < m && dict[a0 + k] == dict[b0 + k]) k++;
    const bool less = k < m ? dict[a0 + k] < dict[b0 + k] : la < lb;
    if (!less) atomicAdd(bad, 1ull);
}

extern "C" int pfpb200_check_dict_order(pfpb200_ctx *ctx, const uint8_t *d_dict, const uint64_t *d_seps,
                                        uint64_t n_words, uint64_t *n_bad) {
    if (!ctx || !n_bad || (n_words && (!d_dict || !d_seps))) return PFPB200_E_ARG;
    *n_bad = 0;
    if (n_words < 2) return PFPB200_OK;
    PFP_CUDA(ctx, cudaSetDevice(ctx->device));
    PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[13], 0, sizeof(u64), ctx->stream));
    dict_order_check_k<<<pfp_blocks(n_words - 1, 256), 256, 0, ctx->stream>>>(
        d_dict, d_seps, n_words, reinterpret_cast<unsigned long long *>(&ctx->d_flags[13]));
    PFP_LAUNCHED(ctx);
    PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[13], &ctx->d_flags[13], sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *n_bad = ctx->h_flags[13];
    return PFPB200_OK;
}
