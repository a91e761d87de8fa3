// pfp_stream.cu -- K2, streaming form: phrase records and fingerprints in ONE pass over the text.
//
// Replaces save_update_word() + kr_hash() of the reference (newscan.cpp:229-304) for all phrases
// at once.  Input: the text and the trigger bits of K1a (one bit per position).  A CTA takes the
// same 32 KB tile as K1 and stages its text (+32 B left halo, +4 KB to the right) and trigger
// bits in shared memory.  It then
//   1. compacts the trigger bits into tile-local positions and writes, per trigger, its global
//      position (ends[]), the `.last` byte (newscan.cpp:296) and the `.sai` value (:299-301) --
//      one thread per trigger, coalesced stores;
//   2. owns every phrase that STARTS at one of its triggers (phrase j = text from e_{j-1}-w+1 to
//      e_j); its end is the next trigger, in the tile or in the 4 KB behind it;
//   3. counting-sorts those phrases by their number of 16-byte chunks, longest first, so that the
//      32 phrases of a warp have (almost) the same length -- phrase lengths are geometric, and
//      giving lanes arbitrary phrases leaves two thirds of a warp idle;
//   4. fingerprints them: one lane per phrase for up to 32 chunks (aligned 32-bit shared loads
//      + funnel shift to the phrase's own alignment, one key load per chunk, the previous
//      chunk's last word and second key carried in registers), one warp per longer phrase.
// Every phrase is hashed by exactly one lane or warp, so there are no partial sums to join.
// Left to the list kernel (phrase_hash_long_k): the buffer's first phrase, a final phrase ending
// at the virtual text border, phrases that do not end within 4 KB of their tile or are longer
// than one key segment (8 KB).  Tiles with more triggers than K2_CAP (p < ~40) are not handled
// here at all: pfp_stream_stage reports them and the caller uses the per-phrase kernels.
#include "pfp_common.cuh"
#include "pfp_stages.cuh"
#include "pfp_fp.cuh"
#include "pfp_tma.cuh"

constexpr int K2_T = PFP_TILE_T;
constexpr int K2_TILE = PFP_TILE;
constexpr int K2_HALO = 32;                                   // >= w (w <= 32 on this path)
constexpr int K2_EXT = 4096;                                  // text staged behind the tile
constexpr int K2_TEXT = K2_HALO + K2_TILE + K2_EXT + 32;      // staged text bytes
constexpr int K2_MWORDS = (K2_TILE + K2_EXT) / 32;            // staged trigger-bit words
constexpr int K2_CAP = 1024;                                  // triggers per tile handled here
constexpr int K2_NBIN = 34;                                   // bins 1..32 = chunks, 33 = warp path
constexpr int K2_LANE_MAX = 32;                               // chunks hashed by a single lane
constexpr int K2_OFF_M = K2_TEXT;
constexpr int K2_OFF_K = K2_OFF_M + K2_MWORDS * 4;
constexpr int K2_OFF_SE = K2_OFF_K + NH_KEY_WORDS * 4;
constexpr int K2_OFF_PERM = K2_OFF_SE + (K2_CAP + 8) * 2;
constexpr int K2_SMEM = K2_OFF_PERM + K2_CAP * 2;
constexpr u32 K2_NONE = 0xFFFFu;
static_assert(K2_T == 256, "block scan below is written for 256 threads");
static_assert(K2_TEXT % 16 == 0 && K2_MWORDS % 4 == 0 && NH_KEY_WORDS % 4 == 0, "16-byte staging");
static_assert(K2_OFF_SE % 16 == 0 && K2_TILE + K2_EXT < 0xFFFF, "tile-local positions are 16 bit");

struct StreamArgs {
    const uint4 *A;            // 16-byte aligned base of the buffer (q = 0)
    u64 q_end;
    u64 pos_bias;              // global position of q = 0
    const uint4 *mask;         // trigger bits
    u32 ntiles;
    const u64 *tile_off;
    u32 w;
    u64 *ends_out;             // null: positions are already there
    u8 *last;
    u8 *sai;                   // may be null
    PhraseFp *rec;
    const u32 *keytab;
    u32 *long_list, *long_count;
    u64 n_regular;             // phrases 1 .. n_regular-1 are hashed here (all end at a trigger)
    u64 *flags;                // [0] errors
};

__device__ __noinline__ uint4 k2_partial_chunk(const unsigned char *b, int nb) {
    u32 wds[4] = {0, 0, 0, 0};
    for (int i = 0; i < nb; i++) wds[i >> 2] |= (u32)b[i] << ((i & 3) * 8);
    return make_uint4(wds[0], wds[1], wds[2], wds[3]);
}

// zero the bytes of a 16-byte chunk at and behind byte `rem` (1 <= rem <= 16)
__device__ __forceinline__ void mask_tail(u32 &x0, u32 &x1, u32 &x2, u32 &x3, int rem) {
    const int t = 8 * rem;
    // word j keeps min(max(t - 32 j, 0), 32) low bits: ~(all ones << n), n clamped to 32
    x0 &= ~__funnelshift_lc(0u, 0xFFFFFFFFu, (u32)t);
    x1 &= ~__funnelshift_lc(0u, 0xFFFFFFFFu, (u32)max(t - 32, 0));
    x2 &= ~__funnelshift_lc(0u, 0xFFFFFFFFu, (u32)max(t - 64, 0));
    x3 &= ~__funnelshift_lc(0u, 0xFFFFFFFFu, (u32)max(t - 96, 0));
}

__device__ __forceinline__ void nh_add(u64 &pa, u64 &pb, u32 x0, u32 x1, u32 x2, u32 x3, const uint4 &k0,
                                       const uint4 &k1) {
    pa += (u64)(x0 + k0.x) * (u64)(x1 + k0.y);
    pa += (u64)(x2 + k0.z) * (u64)(x3 + k0.w);
    pb += (u64)(x0 + k1.x) * (u64)(x1 + k1.y);
    pb += (u64)(x2 + k1.z) * (u64)(x3 + k1.w);
}

__global__ void __launch_bounds__(K2_T, 4) phrase_stream_k(const StreamArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    u8 *sT = smem;
    u32 *sM = reinterpret_cast<u32 *>(smem + K2_OFF_M);
    u32 *sk = reinterpret_cast<u32 *>(smem + K2_OFF_K);
    u16 *se = reinterpret_cast<u16 *>(smem + K2_OFF_SE);      // tile-local trigger positions
    u16 *perm = reinterpret_cast<u16 *>(smem + K2_OFF_PERM);  // phrases, longest first
    __shared__ u32 s_scan[9];
    __shared__ u32 s_hist[K2_NBIN], s_cur[K2_NBIN];
    const u32 t = threadIdx.x, lane = t & 31, wp = t >> 5;
    const u64 tile = blockIdx.x;
    const i64 q0 = (i64)(tile * (u64)K2_TILE);
    const u32 w = a.w;

    // ---- stage text (+halos), trigger bits and keys ----------------------------------------------------
    // interior tiles: three bulk copies (TMA) on one mbarrier; the first/last tiles of the buffer
    // (halo before the buffer, partial 16-byte chunk at its end) take the explicit path
    __shared__ __align__(8) u64 s_bar;
    const i64 qs = q0 - K2_HALO;
    const bool bulk = qs >= 0 && (u64)qs + K2_TEXT <= (a.q_end & ~(u64)15) &&
                      (tile * (u64)K2_T + K2_MWORDS / 4) <= (u64)a.ntiles * K2_T;
    if (bulk) {
        if (t == 0) { mbar_init(&s_bar, 1); mbar_init_fence(); }
        __syncthreads();
        if (t == 0) {
            mbar_expect_tx(&s_bar, (u32)(K2_TEXT + K2_MWORDS * 4 + NH_KEY_WORDS * 4));
            bulk_copy_g2s(sT, a.A + (qs >> 4), K2_TEXT, &s_bar);
            bulk_copy_g2s(sM, a.mask + tile * (u64)K2_T, K2_MWORDS * 4, &s_bar);
            bulk_copy_g2s(sk, a.keytab, NH_KEY_WORDS * 4, &s_bar);
        }
        if (t < K2_NBIN) { s_hist[t] = 0; }
        mbar_wait(&s_bar, 0);
    } else {
        for (int i = t; i < NH_KEY_WORDS / 4; i += K2_T)
            reinterpret_cast<uint4 *>(sk)[i] = __ldg(reinterpret_cast<const uint4 *>(a.keytab) + i);
        for (int c = t; c < K2_TEXT / 16; c += K2_T) {
            const i64 qc = qs + 16 * (i64)c;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (qc >= 0 && (u64)qc + 16 <= a.q_end) v = __ldg(a.A + (qc >> 4));
            else if (qc >= 0 && (u64)qc < a.q_end)
                v = k2_partial_chunk(reinterpret_cast<const unsigned char *>(a.A) + qc, (int)(a.q_end - (u64)qc));
            reinterpret_cast<uint4 *>(sT)[c] = v;
        }
        for (int i = t; i < K2_MWORDS / 4; i += K2_T) {
            const u64 gi = tile * (u64)K2_T + (u64)i;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (gi < (u64)a.ntiles * K2_T) v = __ldg(a.mask + gi);
            reinterpret_cast<uint4 *>(sM)[i] = v;
        }
        if (t < K2_NBIN) { s_hist[t] = 0; }
    }
    __syncthreads();

    // ---- trigger bits -> tile-local positions se[0..tot), se[tot] = first trigger behind the tile ----
    const uint4 mv = reinterpret_cast<const uint4 *>(sM)[t];
    u32 tot;
    const u32 ex = block_excl_scan_256(__popc(mv.x) + __popc(mv.y) + __popc(mv.z) + __popc(mv.w), &tot, s_scan);
    if (tot == 0) return;
    if (tot > (u32)K2_CAP) {            // dense tile: the caller falls back to the per-phrase kernels
        if (t == 0) atomicOr((unsigned long long *)&a.flags[0], PFP_ERRBIT_INTERNAL);
        return;
    }
    {
        u32 o = ex;
        const u32 mw[4] = {mv.x, mv.y, mv.z, mv.w};
#pragma unroll
        for (int k = 0; k < 4; k++) {
            u32 x = mw[k];
            while (x) {
                const int b = __ffs(x) - 1;
                x &= x - 1;
                se[o++] = (u16)(t * 128 + k * 32 + b);
            }
        }
    }
    if (wp == 0) {                      // first trigger in the K2_EXT / 32 words behind the tile
        u32 found = K2_NONE;
        for (int b0 = 0; b0 < K2_EXT / 32 && found == K2_NONE; b0 += 32) {
            const u32 x = sM[K2_TILE / 32 + b0 + lane];
            const u32 nz = __ballot_sync(0xffffffffu, x != 0);
            if (nz) {
                const int fl = __ffs(nz) - 1;
                const u32 xf = __shfl_sync(0xffffffffu, x, fl);
                found = (u32)(K2_TILE + 32 * (b0 + fl) + __ffs(xf) - 1);
            }
        }
        if (lane == 0) se[tot] = (u16)found;
    }
    __syncthreads();

    // ---- per trigger: position, .last, .sai (newscan.cpp:296-301) ---------------------------------------
    const u64 tile_first = a.tile_off[tile];
    for (u32 li = t; li < tot; li += K2_T) {
        const int e = se[li];
        const u64 idx = tile_first + li;
        const u64 g = (u64)(q0 + e) + a.pos_bias;
        if (a.ends_out) a.ends_out[idx] = g;
        a.last[idx] = (g < (u64)w) ? (u8)PFP_DOLLAR : sT[K2_HALO + e - (int)w];
        if (a.sai) {
            const u64 pos = g + 1;
            u8 *d = a.sai + idx * PFP_IBYTES;
#pragma unroll
            for (int k = 0; k < PFP_IBYTES; k++) d[k] = (u8)(pos >> (8 * k));
        }
    }

    // ---- the phrases starting at my triggers: chunk counts, counting sort (longest first) ----------
    // phrase q (1 <= q <= tot) runs from se[q-1] - w + 1 to se[q]
    u32 mybin[K2_CAP / K2_T];
#pragma unroll
    for (int r = 0; r < K2_CAP / K2_T; r++) {
        const u32 q = t + 1 + r * K2_T;
        u32 bin = 0;
        if (q <= tot && tile_first + q < a.n_regular) {
            const u32 e = se[q];
            const u32 len = e - se[q - 1] + w;                  // e - s + 1
            const u32 nch = (len + 15) >> 4;
            if (e == K2_NONE || nch > NH_SEG_BYTES / 16) {      // open behind the tile, or too long
                a.long_list[atomicAdd(a.long_count, 1u)] = (u32)(tile_first + q);
            } else {
                bin = nch > (u32)K2_LANE_MAX ? (u32)K2_NBIN - 1 : nch;
                atomicAdd(&s_hist[bin], 1u);
            }
        }
        mybin[r] = bin;
    }
    __syncthreads();
    if (wp == 0) {                      // descending offsets: bin 33 first, then 32, 31, .., 1
        const u32 rb = K2_NBIN - 1 - lane;                      // lanes 0..31 <-> bins 33..2
        const u32 h = s_hist[rb];
        const u32 inc = warp_incl_scan(h);
        s_cur[rb] = inc - h;
        const u32 above1 = __shfl_sync(0xffffffffu, inc, 31);   // phrases in bins 2..33
        if (lane == 0) { s_cur[1] = above1; s_scan[0] = above1 + s_hist[1]; }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < K2_CAP / K2_T; r++) {
        if (mybin[r]) perm[atomicAdd(&s_cur[mybin[r]], 1u)] = (u16)(t + 1 + r * K2_T);
    }
    const u32 nvalid = s_scan[0];
    const u32 nwarp = s_hist[K2_NBIN - 1];
    __syncthreads();

    // ---- phrases of more than 32 chunks: one warp each ----------------------------------------------------
    for (u32 i = wp; i < nwarp; i += K2_T / 32) {
        const u32 q = perm[i];
        const int s = (int)se[q - 1] - (int)w + 1;
        const u32 len = (u32)se[q] - (u32)se[q - 1] + w;
        const u32 nch = (len + 15) >> 4;
        u64 pa = 0, pb = 0;
        for (u32 c = lane; c < nch; c += 32) {
            const int ad = s + K2_HALO + 16 * (int)c;
            const u32 *p4 = reinterpret_cast<const u32 *>(sT + (ad & ~3));
            const u32 sh = (u32)(ad & 3) * 8u;
            const u32 W0 = p4[0], W1 = p4[1], W2 = p4[2], W3 = p4[3], W4 = p4[4];
            u32 x0 = __funnelshift_r(W0, W1, sh), x1 = __funnelshift_r(W1, W2, sh);
            u32 x2 = __funnelshift_r(W2, W3, sh), x3 = __funnelshift_r(W3, W4, sh);
            if (c == nch - 1) mask_tail(x0, x1, x2, x3, (int)(len - 16 * c));
            const uint4 k0 = *reinterpret_cast<const uint4 *>(sk + 4 * c);
            const uint4 k1 = *reinterpret_cast<const uint4 *>(sk + 4 * c + 4);
            nh_add(pa, pb, x0, x1, x2, x3, k0, k1);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            pa += __shfl_xor_sync(0xffffffffu, pa, o);
            pb += __shfl_xor_sync(0xffffffffu, pb, o);
        }
        if (lane == 0) store_rec(a.rec, tile_first + q, pa, pb);
    }

    // ---- all other phrases: one lane each, warps hold phrases of (almost) equal length ---------------
    for (u32 i = nwarp + t; i < nvalid; i += K2_T) {
        const u32 q = perm[i];
        const int s = (int)se[q - 1] - (int)w + 1;
        const u32 len = (u32)se[q] - (u32)se[q - 1] + w;
        const u32 nch = (len + 15) >> 4;
        const int ad = s + K2_HALO;
        const u32 *p4 = reinterpret_cast<const u32 *>(sT + (ad & ~3));
        const u32 sh = (u32)(ad & 3) * 8u;
        const u32 *kp = sk;
        uint4 k0 = *reinterpret_cast<const uint4 *>(kp);
        u32 W0 = p4[0];
        u64 pa = 0, pb = 0;
        for (u32 c = 1; c < nch; c++) {                          // full chunks
            const u32 W1 = p4[1], W2 = p4[2], W3 = p4[3], W4 = p4[4];
            const uint4 k1 = *reinterpret_cast<const uint4 *>(kp + 4);
            nh_add(pa, pb, __funnelshift_r(W0, W1, sh), __funnelshift_r(W1, W2, sh),
                   __funnelshift_r(W2, W3, sh), __funnelshift_r(W3, W4, sh), k0, k1);
            W0 = W4;
            k0 = k1;
            p4 += 4;
            kp += 4;
        }
        {                                                        // last chunk: zero padding behind the end
            const u32 W1 = p4[1], W2 = p4[2], W3 = p4[3], W4 = p4[4];
            const uint4 k1 = *reinterpret_cast<const uint4 *>(kp + 4);
            u32 x0 = __funnelshift_r(W0, W1, sh), x1 = __funnelshift_r(W1, W2, sh);
            u32 x2 = __funnelshift_r(W2, W3, sh), x3 = __funnelshift_r(W3, W4, sh);
            mask_tail(x0, x1, x2, x3, (int)(len - 16 * (nch - 1)));
            nh_add(pa, pb, x0, x1, x2, x3, k0, k1);
        }
        store_rec(a.rec, tile_first + q, pa, pb);
    }
}

// the buffer's first phrase, and a final phrase ending at the virtual border (no trigger of its own)
__global__ void special_list_k(u32 *list, u32 *count, u64 P, u64 total) {
    u32 n = *count;
    if (P > 0) list[n++] = 0u;
    if (P > total && total > 0) list[n++] = (u32)total;
    *count = n;
}

int pfp_stream_stage(pfpb200_ctx *ctx, const ScanBits &sb, const TextView &tv, const PhraseArrays &ph,
                     u64 P, i64 first_start, u32 w, bool emit_ends) {
    if (!pfp_stream_ok(sb, w)) return pfp_fail(ctx, PFPB200_E_INTERNAL, "stream stage: unsupported shape");
    u32 *list = nullptr;
    const u64 cap = 8ull * sb.ntiles + 8;
    PFP_TRY(pfp_alloc_t(ctx, &list, cap + 1));
    u32 *count = list + cap;
    PFP_CUDA(ctx, cudaMemsetAsync(count, 0, sizeof(u32), ctx->stream));
    if (sb.ntiles > 0 && sb.total > 0) {
        StreamArgs a{};
        a.A = sb.A; a.q_end = sb.q_end; a.pos_bias = sb.pos_bias;
        a.mask = sb.mask; a.ntiles = sb.ntiles; a.tile_off = sb.tile_off;
        a.w = w;
        a.ends_out = emit_ends ? ph.ends : nullptr;
        a.last = ph.last; a.sai = ph.sai; a.rec = ph.rec;
        a.keytab = ctx->d_keys; a.flags = ctx->d_flags;
        a.long_list = list; a.long_count = count;
        a.n_regular = sb.total;
        phrase_stream_k<<<sb.ntiles, K2_T, K2_SMEM, ctx->stream>>>(a);
        PFP_LAUNCHED(ctx);
    }
    special_list_k<<<1, 1, 0, ctx->stream>>>(list, count, P, sb.total);
    PFP_LAUNCHED(ctx);
    PFP_TRY(pfp_hash_list(ctx, tv, ph, first_start, w, list, count, cap));
    PFP_TRY(pfp_records_range(ctx, tv, ph, sb.total, P, w));
    PFP_TRY(pfp_free_now(ctx, list));
    return PFPB200_OK;
}

int pfp_stream_init(pfpb200_ctx *ctx) {
    PFP_CUDA(ctx, cudaFuncSetAttribute(phrase_stream_k, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM));
    return PFPB200_OK;
}

bool pfp_stream_ok(const ScanBits &sb, u32 w) {
    return w <= (u32)K2_HALO && sb.max_tile_cnt <= (u32)K2_CAP;
}
