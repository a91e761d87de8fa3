// pfp_scan.cu -- K1: Karp-Rabin rolling-window trigger scan + compaction of trigger positions.
//
// Replaces KR_window::addchar + `hash % p == 0` of the reference (newscan.cpp:194-202,344,367;
// pscan.cpp:239-247) for a whole shard at once.  The window hash depends only on the last w
// bytes, so every thread owns a run of K1_RUN consecutive positions, rebuilds the hash of the
// w bytes in front of its run and then rolls.  A CTA stages a 32 KB tile (+32 B left halo)
// in shared memory with coalesced 16-byte loads; threads read their run back with
// conflict-free LDS.128 (slots padded to 144 B).  Output of K1a is one bit per text position;
// K1c turns bits into ascending 64-bit positions using per-tile offsets from a device scan.
//
// Measured alternatives that lost (B200, 4 GB, w=10): reading the bytes as LDS.U8 from 33-word
// slots (moves the PRMT extractions from the ALU pipe, 63 % busy, to the idle LSU pipe) with a
// predicated OR for the mask: 3.05 ms vs 2.86 ms for this version (56 registers, fewer CTAs).
#include "pfp_common.cuh"
#include "pfp_stages.cuh"
#include <stdlib.h>

constexpr int K1_T = PFP_TILE_T;             // threads per CTA
constexpr int K1_RUN = PFP_TILE_RUN;         // positions per thread
constexpr int K1_TILE = PFP_TILE;            // 32768 positions per CTA
constexpr int K1_SLOT = K1_RUN + 16;         // padded slot: LDS.128 of 8 lanes hits 32 banks
constexpr int K1_SMEM = (K1_T + 1) * K1_SLOT;
constexpr int K1_CHUNKS = K1_TILE / 16;
constexpr int K1_MAXW_FAST = 32;             // halo of two 16-byte chunks

// byte j (-32 <= j < 16) of the 48-byte register window {prev2, prev1, cur}
#define WIN_BYTE(win, j) (__byte_perm((win)[((j) + 32) >> 2], 0u, 0x4440u | (((j) + 32) & 3)))

__device__ __forceinline__ u32 range_mask32(u64 q0, u64 lo, u64 hi) {
    // bits i with lo <= q0+i < hi
    u32 m = 0xFFFFFFFFu;
    if (lo > q0) m = (lo - q0 >= 32) ? 0u : (0xFFFFFFFFu << (u32)(lo - q0));
    if (hi <= q0) return 0u;
    if (hi - q0 < 32) m &= (1u << (u32)(hi - q0)) - 1u;
    return m;
}

// last, partial 16-byte chunk of the buffer: byte loads (rare; kept out of line)
__device__ __noinline__ uint4 k1_partial_chunk(const unsigned char *b, int nb) {
    u32 wds[4] = {0, 0, 0, 0};
    for (int i = 0; i < nb; i++) wds[i >> 2] |= (u32)b[i] << ((i & 3) * 8);
    return make_uint4(wds[0], wds[1], wds[2], wds[3]);
}

// stage tile `tile` (+ halo) of the 16-byte-aligned stream A into padded shared memory
__device__ __forceinline__ void k1_stage_tile(const uint4 *__restrict__ A, u64 q_end, u64 tile,
                                              unsigned char *sm) {
    const i64 q0 = (i64)(tile * (u64)K1_TILE);
#pragma unroll
    for (int it = 0; it < (K1_CHUNKS + 2 + K1_T - 1) / K1_T; it++) {
        int c = (int)threadIdx.x + it * K1_T - 2;     // chunk index, -2 and -1 are the halo
        if (c < K1_CHUNKS) {
            i64 qc = q0 + (i64)c * 16;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (qc >= 0 && (u64)qc + 16 <= q_end) {
                v = __ldg(A + (qc >> 4));
            } else if (qc >= 0 && (u64)qc < q_end) {
                v = k1_partial_chunk(reinterpret_cast<const unsigned char *>(A) + qc, (int)(q_end - (u64)qc));
            }
            int cc = c + 8;
            *reinterpret_cast<uint4 *>(sm + (cc >> 3) * K1_SLOT + (cc & 7) * 16) = v;
        }
    }
}

template <int W>
__global__ void __launch_bounds__(K1_T) kr_scan_k(const uint4 *__restrict__ A, u64 q_end, u64 q_lo,
                                                  u64 q_hi, pfp_scan_consts C,
                                                  uint4 *__restrict__ mask,
                                                  u32 *__restrict__ tile_cnt) {
    extern __shared__ __align__(16) unsigned char sm[];
    __shared__ u32 s_cnt;
    const u32 t = threadIdx.x;
    const u64 tile = blockIdx.x;
    if (t == 0) s_cnt = 0;
    k1_stage_tile(A, q_end, tile, sm);
    __syncthreads();

    const u32 negw = C.negw, pinv = C.pinv, pshift = C.pshift, plimit = C.plimit;
    u32 win[12];
    {   // the two chunks in front of this thread's run: tail of the previous slot
        uint4 p2 = *reinterpret_cast<const uint4 *>(sm + t * K1_SLOT + 96);
        uint4 p1 = *reinterpret_cast<const uint4 *>(sm + t * K1_SLOT + 112);
        win[0] = p2.x; win[1] = p2.y; win[2] = p2.z; win[3] = p2.w;
        win[4] = p1.x; win[5] = p1.y; win[6] = p1.z; win[7] = p1.w;
    }
    // hash of the w bytes in front of the run (the window ending just before it); its first
    // byte is the one the first roll removes
    u32 h = 0;
#pragma unroll
    for (int j = -W; j < 0; j++) h = pfp_push(h, WIN_BYTE(win, j));

    unsigned char *slot = sm + (t + 1) * K1_SLOT;
    const u64 qrun = tile * (u64)K1_TILE + (u64)t * K1_RUN;
    u32 cnt = 0;
#pragma unroll 1
    for (int kk = 0; kk < K1_RUN / 32; kk++) {
        u32 m = 0;
#pragma unroll
        for (int half = 0; half < 2; half++) {
            uint4 cur = *reinterpret_cast<const uint4 *>(slot + kk * 32 + half * 16);
            win[8] = cur.x; win[9] = cur.y; win[10] = cur.z; win[11] = cur.w;
#pragma unroll
            for (int i = 0; i < 16; i++) {
                u32 c_in = WIN_BYTE(win, i);
                u32 c_out = WIN_BYTE(win, i - W);
                h = pfp_roll(h, c_in, c_out, negw);
                if (pfp_is_trigger(h, pinv, pshift, plimit)) m |= 1u << (half * 16 + i);
            }
#pragma unroll
            for (int i = 0; i < 4; i++) { win[i] = win[4 + i]; win[4 + i] = win[8 + i]; }
        }
        m &= range_mask32(qrun + (u64)kk * 32, q_lo, q_hi);
        cnt += __popc(m);
        *reinterpret_cast<u32 *>(slot + K1_RUN + kk * 4) = m;   // own slot padding
    }
    mask[tile * (u64)K1_T + t] = *reinterpret_cast<const uint4 *>(slot + K1_RUN);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((t & 31) == 0 && cnt) atomicAdd(&s_cnt, cnt);
    __syncthreads();
    if (t == 0) tile_cnt[tile] = s_cnt;
}

// Any window size: bytes straight from global memory (L1-cached byte loads).  Slow path.
__global__ void __launch_bounds__(K1_T) kr_scan_generic_k(const unsigned char *__restrict__ A8,
                                                          u64 q_end, u64 q_lo, u64 q_hi,
                                                          pfp_scan_consts C,
                                                          uint4 *__restrict__ mask,
                                                          u32 *__restrict__ tile_cnt) {
    __shared__ u32 s_cnt;
    const u32 t = threadIdx.x;
    const u64 tile = blockIdx.x;
    if (t == 0) s_cnt = 0;
    __syncthreads();
    const i64 w = C.w;
    const i64 qrun = (i64)(tile * (u64)K1_TILE + (u64)t * K1_RUN);
    u32 h = 0;
    for (i64 q = qrun - w; q < qrun; q++) {
        u32 c = (q >= 0 && (u64)q < q_end) ? A8[q] : 0u;
        h = pfp_push(h, c);
    }
    u32 mw[4];
    u32 cnt = 0;
#pragma unroll
    for (int kk = 0; kk < 4; kk++) {
        u32 m = 0;
        for (int i = 0; i < 32; i++) {
            i64 q = qrun + kk * 32 + i;
            u32 c_in = ((u64)q < q_end) ? A8[q] : 0u;
            i64 qo = q - w;
            u32 c_out = (qo >= 0 && (u64)qo < q_end) ? A8[qo] : 0u;
            h = pfp_roll(h, c_in, c_out, C.negw);
            if (pfp_is_trigger(h, C.pinv, C.pshift, C.plimit)) m |= 1u << i;
        }
        m &= range_mask32((u64)qrun + (u64)kk * 32, q_lo, q_hi);
        cnt += __popc(m);
        mw[kk] = m;
    }
    mask[tile * (u64)K1_T + t] = make_uint4(mw[0], mw[1], mw[2], mw[3]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((t & 31) == 0 && cnt) atomicAdd(&s_cnt, cnt);
    __syncthreads();
    if (t == 0) tile_cnt[tile] = s_cnt;
}

// ------------------------------------------------------------------------------------------------
// K1a on DNA text: what the interval form (kr_scan_ivf_k) and its row kernel (kr_scan_rows_k)
// share.  A warp takes 1 KB rows of the text, a lane 32 consecutive positions: two coalesced
// 16-byte loads (kd_load_unit at the buffer's ends), 2-bit codes ((c >> 1) & 3: A=0 C=1 T=2 G=3)
// packed four at a time with one multiply (dna_pack4 / dna_pack16).  Exactness: every loaded byte
// is checked against the letter its code stands for (PRMT decode + compare); a row with any other
// byte (N, lower case, text that is not DNA at all) is redone with the rolling arithmetic of
// kr_scan_k (kd_row_by_arithmetic) -- same trigger set for every input, DNA or not.
// ------------------------------------------------------------------------------------------------
constexpr int KD_T = 1024;                    // threads per CTA (one CTA per SM)
constexpr int KD_MAXW = 10;
constexpr u32 KD_LETTERS = 0x47544341u;       // code -> letter: 0 'A', 1 'C', 2 'T', 3 'G'

// Powers of two kept in constant memory on purpose: a shift by a compile-time amount written as
// a multiplication by an operand the compiler cannot see through is issued on the FMA pipe
// (IMAD / IMAD.HI), which has room, instead of the ALU pipe (SHF), which bounds these kernels.
__constant__ u32 kd_pow2[33];
__device__ __forceinline__ u32 shr_fma(u32 x, int s) { return s ? __umulhi(x, kd_pow2[32 - s]) : x; }
// four text bytes -> their four 2-bit codes in bits 0..7 (first byte lowest); `bad` collects
// every bit in which a byte differs from the letter of its code
// returns a word whose TOP byte holds the four codes
__device__ __forceinline__ u32 dna_pack4(u32 x, u32 &bad) {
    const u32 y = shr_fma(x, 1) & 0x03030303u;
    const u32 z = y | shr_fma(y, 4);                          // nibbles: (c0,c1) in byte 0, (c2,c3) in byte 2
    const u32 sel = __byte_perm(z, 0u, 0x4420u);              // c0,c1,c2,c3 as the low four nibbles
    u32 dec;                                                  // raw PRMT: every selector nibble is < 4, nothing to mask
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(dec) : "r"(KD_LETTERS), "r"(0u), "r"(sel));
    bad |= dec ^ x;
    return y * 0x01041040u;
}
__device__ __forceinline__ u32 dna_pack16(const uint4 &v, u32 &bad) {
    const u32 a = __byte_perm(dna_pack4(v.x, bad), dna_pack4(v.y, bad), 0x0073u);   // top bytes of both
    const u32 b = __byte_perm(dna_pack4(v.z, bad), dna_pack4(v.w, bad), 0x0073u);
    return __byte_perm(a, b, 0x5410u);
}

__device__ __forceinline__ uint4 kd_load_unit(const uint4 *__restrict__ A, u64 q_end, i64 qc) {
    if (qc >= 0 && (u64)qc + 16 <= q_end) return __ldg(A + (qc >> 4));
    if (qc >= 0 && (u64)qc < q_end)
        return k1_partial_chunk(reinterpret_cast<const unsigned char *>(A) + qc, (int)(q_end - (u64)qc));
    return make_uint4(0, 0, 0, 0);
}

// the byte values of a lane's 32 positions into the 256-bit set `alpha` (kept out of line)
__device__ __noinline__ void kd_note_alphabet(uint4 u0, uint4 u1, u64 q, u64 q_text0, u64 q_end, u32 lane,
                                               u32 *__restrict__ alpha) {
    const u32 xs[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
    u32 pm[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int i = 0; i < 32; i++) {
        const u32 c = (xs[i >> 2] >> (8 * (i & 3))) & 255u;
        const bool in_text = q + i >= q_text0 && q + i < q_end;     // bytes in front of / behind the text are not text
#pragma unroll
        for (int k = 0; k < 8; k++) pm[k] |= (in_text && (c >> 5) == (u32)k) ? (1u << (c & 31)) : 0u;
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const u32 o = __reduce_or_sync(0xffffffffu, pm[k]);
        if (lane == 0 && o) atomicOr(&alpha[k], o);
    }
}

// byte j (-16 <= j < 32) of {four words in front, eight words of the lane}
#define KD_BYTE(wd, j) (__byte_perm((wd)[((j) + 16) >> 2], 0u, 0x4440u | (((j) + 16) & 3)))

// A row that holds something besides A C G T, or a clipped row at the buffer's ends: the trigger
// bits of the lane's 32 positions by the rolling arithmetic of kr_scan_k, exact for any bytes; and,
// when `note` is set, the row's byte values go into the alphabet set.
template <int W>
__device__ __noinline__ u32 kd_row_by_arithmetic(uint4 u0, uint4 u1, u32 lane, pfp_scan_consts C, u64 q, u64 q_text0,
                                                 u64 q_end, bool note, u32 *__restrict__ alpha) {
    if (note) kd_note_alphabet(u0, u1, q, q_text0, q_end, lane, alpha);
    u32 wd[12];
    wd[0] = __shfl_up_sync(0xffffffffu, u1.x, 1);
    wd[1] = __shfl_up_sync(0xffffffffu, u1.y, 1);
    wd[2] = __shfl_up_sync(0xffffffffu, u1.z, 1);
    wd[3] = __shfl_up_sync(0xffffffffu, u1.w, 1);
    if (lane == 0) { wd[0] = 0; wd[1] = 0; wd[2] = 0; wd[3] = 0; }   // only used by word 0: nothing in front
    wd[4] = u0.x; wd[5] = u0.y; wd[6] = u0.z; wd[7] = u0.w;
    wd[8] = u1.x; wd[9] = u1.y; wd[10] = u1.z; wd[11] = u1.w;
    u32 h = 0, m = 0;
#pragma unroll
    for (int j = -W; j < 0; j++) h = pfp_push(h, KD_BYTE(wd, j));
#pragma unroll
    for (int i = 0; i < 32; i++) {
        h = pfp_roll(h, KD_BYTE(wd, i), KD_BYTE(wd, i - W), C.negw);
        if (pfp_is_trigger(h, C.pinv, C.pshift, C.plimit)) m |= 1u << i;
    }
    return m;
}

// ------------------------------------------------------------------------------------------------
// K1a, interval form (w <= 10, p < PW) -- the default for DNA text since round 2.
//
// Round 1's form, a 4^w-bit trigger table in shared memory, paid 3.6 wavefronts per position (32
// random words in 32 banks; DESIGN.md §3a).  This form needs ONE conflict-free wavefront, from two
// facts about the hash:
//  (1) it is LINEAR: H(window) = (Ah[hi] + Bl[lo]) mod PW, hi / lo = the codes of the w-5 older
//      and the 5 newest symbols; and the hi block of the window ending at i IS the lo block of
//      the window ending at i-5, so ONE table of 4^5 = 1024 entries, indexed by the 5-symbol block
//      ending at a position, serves both halves: one look-up per position, each used twice;
//  (2) "H mod p == 0" becomes an INTERVAL test after multiplying by u = p^-1 mod PW: H = k p with
//      0 <= k <= K = (PW-1)/p  <=>  (H u mod PW) <= K, and H u = Ah u + Bl u (mod PW).
//      Scaled by 2^16/PW the reduction mod PW is the wrap of 16-bit addition: with
//      a16 = floor(Ah u 2^16/PW), b16 = floor(Bl u 2^16/PW), t = (a16 + b16) mod 2^16, the true
//      scaled sum lies in [t, t+2) (mod 2^16), so every trigger has (t + 2) mod 2^16 < theta + 4,
//      theta = (K+1) 2^16/PW.  One entry holds (a16 + 2) in its high and b16 in its low half:
//            T = (E[i] << 16) + E[i-5];   candidate  <=>  T < (floor(theta) + 4) << 16
//      -- one multiply-add and one compare per position.  The table is 4 KB, so it is replicated
//      32 times (word 32 x + lane): every lane reads its own bank.
// Candidates (all triggers + 6e-5 of the positions for p = 100) are then decided EXACTLY from the
// full 32-bit partial hashes {Ah, Bl} (a second, unreplicated 8 KB table) with the same
// pfp_is_trigger() as everywhere else, so the trigger set is identical for every input; rows
// holding anything besides A C G T go to the rolling arithmetic (kr_scan_rows_k).
// tests/test_arith.py::test_interval_form_* models both tables in numpy over all 4^10 windows.
// ------------------------------------------------------------------------------------------------
constexpr u32 KE_ENT = 1024;                                        // 5-symbol blocks
constexpr size_t KE_SMEM = (size_t)KE_ENT * 32 * 4 + (size_t)KE_ENT * 8;   // replicated E + exact {Ah, Bl}

__global__ void dna_etab_k(pfp_scan_consts C, u32 uinv, u32 *__restrict__ etab, uint2 *__restrict__ xtab) {
    const u32 x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= KE_ENT) return;
    u64 bl = 0, ah = 0;
    for (int j = 0; j < 5; j++) {                                    // symbol j of the block, j = 0 oldest
        const u64 c = (KD_LETTERS >> (8 * ((x >> (2 * j)) & 3u))) & 255u;
        if ((int)C.w - 5 + j >= 0) bl = (bl * 256 + c) % PFP_PW;     // as the lo block: window symbol w-5+j
        if ((int)C.w - 10 + j >= 0) ah = (ah * 256 + c) % PFP_PW;    // as the hi block: window symbol w-10+j
    }
    for (int j = 0; j < 5; j++) ah = (ah * 256) % PFP_PW;            // the hi block stands 5 symbols higher
    xtab[x] = make_uint2((u32)ah, (u32)bl);
    const u64 as = (ah * uinv) % PFP_PW, bs = (bl * uinv) % PFP_PW;
    const u32 a16 = (u32)((as << 16) / PFP_PW), b16 = (u32)((bs << 16) / PFP_PW);
    etab[x] = (((a16 + 2u) & 0xFFFFu) << 16) | b16;
}

// (bits [b, b+NB) of the 96-bit stream {S[0], S[1], S[2]}) << 7, other bits undefined
template <int B, int NB = 10>
__device__ __forceinline__ u32 ke_block_x128(const u32 (&S)[3]) {
    constexpr int k = B >> 5, sh = B & 31;
    if constexpr (sh < 7) return S[k] * kd_pow2[7 - sh];                      // IMAD (FMA pipe)
    else if constexpr (sh + NB <= 32) return shr_fma(S[k], sh - 7);           // IMAD.HI
    else return __funnelshift_r(S[k], S[k + 1], sh - 7);                      // SHF (ALU pipe), a few of 16
}

template <int I>
__device__ __forceinline__ u32 ke_lookup(const u32 (&S)[3], const unsigned char *rep_lane) {
    const u32 v = ke_block_x128<2 * (I + 12)>(S);                   // block of the symbols I-4 .. I
    return *reinterpret_cast<const u32 *>(rep_lane + (v & 0x1FF80u));
}

// ---- 11 <= w <= 16: FOUR blocks of 4 symbols (256 entries of 8 bytes, 16 replicas: every lane of a
// half warp reads its own pair of banks).  The block ending at a position serves the windows
// ending 0, 4, 8 and 12 positions later in roles 0..3; entry = {lo: f1 << 16 | f0, hi: f3 << 16 | f2},
//     T = (lo[i] << 16) + lo[i-4] + (hi[i-8] << 16) + hi[i-12]
// (the low halves add up to garbage that may carry once into the high half: with four floors the
// true scaled sum lies in [t-1, t+4), the table carries a bias of 5 and the threshold is
// floor(theta) + 7).  Candidates are decided exactly from the four exact partial hashes.
constexpr u32 K4_ENT = 256;
constexpr size_t K4_SMEM = (size_t)K4_ENT * 16 * 8 + (size_t)K4_ENT * 16;

__global__ void dna_etab4_k(pfp_scan_consts C, u32 uinv, uint2 *__restrict__ etab, uint4 *__restrict__ xtab) {
    const u32 x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= K4_ENT) return;
    u32 F[4], f16[4];
    for (int r = 0; r < 4; r++) {                                    // role r: the block ends 4 r symbols before the window's end
        u64 h = 0;
        for (int j = 0; j < 4; j++) {                                // symbol j of the block, j = 0 oldest
            const u32 dist = 4u * r + (3u - j);                      // distance from the window's last symbol
            if (dist >= C.w) continue;
            u64 c = (KD_LETTERS >> (8 * ((x >> (2 * j)) & 3u))) & 255u;
            for (u32 k = 0; k < dist; k++) c = (c * 256) % PFP_PW;
            h = (h + c) % PFP_PW;
        }
        F[r] = (u32)h;
        f16[r] = (u32)((((h * uinv) % PFP_PW) << 16) / PFP_PW);
    }
    xtab[x] = make_uint4(F[0], F[1], F[2], F[3]);
    etab[x] = make_uint2((f16[1] << 16) | f16[0], (((f16[3] + 5u) & 0xFFFFu) << 16) | f16[2]);
}

template <int I>
__device__ __forceinline__ uint2 k4_lookup(const u32 (&S)[3], const unsigned char *rep_lane) {
    const u32 v = ke_block_x128<2 * (I + 13), 8>(S);                // block of the symbols I-3 .. I
    return *reinterpret_cast<const uint2 *>(rep_lane + (v & 0x7F80u));
}

__device__ __forceinline__ u32 k4_row_bits(const u32 (&S)[3], const unsigned char *rep_lane,
                                           const uint4 *__restrict__ xt, const pfp_scan_consts &C, u32 cthr) {
    u32 L[36], H[44];                                                // L[4 + i], H[12 + i]: block ending at position i
#define K4_L(I) { const uint2 e = k4_lookup<I>(S, rep_lane); L[4 + I] = e.x; H[12 + I] = e.y; }
    K4_L(20) K4_L(21) K4_L(22) K4_L(23) K4_L(24) K4_L(25) K4_L(26) K4_L(27) K4_L(28) K4_L(29) K4_L(30) K4_L(31)
    K4_L(0) K4_L(1) K4_L(2) K4_L(3) K4_L(4) K4_L(5) K4_L(6) K4_L(7) K4_L(8) K4_L(9) K4_L(10) K4_L(11) K4_L(12)
    K4_L(13) K4_L(14) K4_L(15) K4_L(16) K4_L(17) K4_L(18) K4_L(19)
#undef K4_L
#pragma unroll
    for (int j = 0; j < 12; j++) H[j] = __shfl_up_sync(0xffffffffu, H[32 + j], 1);   // blocks ending at -12 .. -1
#pragma unroll
    for (int j = 0; j < 4; j++) L[j] = __shfl_up_sync(0xffffffffu, L[32 + j], 1);    // blocks ending at -4 .. -1
    u32 m = 0;
#pragma unroll
    for (int i = 0; i < 32; i++) {
        const u32 T = (L[4 + i] * kd_pow2[16] + L[i]) + (H[4 + i] * kd_pow2[16] + H[i]);
        asm("{\n\t.reg .pred c;\n\tsetp.lt.u32 c, %1, %2;\n\t@c or.b32 %0, %0, %3;\n\t}"
            : "+r"(m) : "r"(T), "r"(cthr), "r"(1u << i));
    }
    u32 cand = m;
    while (cand) {
        const u32 bit = cand & (0u - cand);
        cand ^= bit;
        const u32 o = 2u * (u32)(31 - __clz(bit)) + 2u;              // first stream bit of the 16 symbols ending here
        const bool k0 = o < 32u, k2 = o >= 64u;
        const u32 lo = k0 ? S[0] : (k2 ? S[2] : S[1]);
        const u32 hi = k0 ? S[1] : S[2];                             // k2: o = 64, shift 0, the upper word is not used
        const u32 v = __funnelshift_r(lo, hi, o);                    // 32 bits: roles 3, 2, 1, 0 from the low byte up
        u32 a = xt[v >> 24].x + xt[(v >> 16) & 255u].y, b = xt[(v >> 8) & 255u].z + xt[v & 255u].w;
        a = min(a, a - PFP_PW);
        b = min(b, b - PFP_PW);
        u32 h = a + b;
        h = min(h, h - PFP_PW);
        if (!pfp_is_trigger(h, C.pinv, C.pshift, C.plimit)) m ^= bit;
    }
    return m;
}

// trigger bits of a lane's 32 positions; S = {16 symbols in front, 32 own symbols}, 2 bits each
__device__ __forceinline__ u32 ke_row_bits(const u32 (&S)[3], const unsigned char *rep_lane,
                                           const uint2 *__restrict__ xt, const pfp_scan_consts &C, u32 cthr) {
    u32 E[37];                                                       // E[5 + i]: block ending at position i
#define KE_L(I) E[5 + I] = ke_lookup<I>(S, rep_lane);
    KE_L(27) KE_L(28) KE_L(29) KE_L(30) KE_L(31)
    KE_L(0) KE_L(1) KE_L(2) KE_L(3) KE_L(4) KE_L(5) KE_L(6) KE_L(7) KE_L(8) KE_L(9) KE_L(10) KE_L(11) KE_L(12)
    KE_L(13) KE_L(14) KE_L(15) KE_L(16) KE_L(17) KE_L(18) KE_L(19) KE_L(20) KE_L(21) KE_L(22) KE_L(23) KE_L(24)
    KE_L(25) KE_L(26)
#undef KE_L
#pragma unroll
    for (int j = 0; j < 5; j++) E[j] = __shfl_up_sync(0xffffffffu, E[32 + j], 1);   // blocks ending at -5 .. -1
    u32 m = 0;
#pragma unroll
    for (int i = 0; i < 32; i++) {
        const u32 T = E[5 + i] * kd_pow2[16] + E[i];
        asm("{\n\t.reg .pred c;\n\tsetp.lt.u32 c, %1, %2;\n\t@c or.b32 %0, %0, %3;\n\t}"
            : "+r"(m) : "r"(T), "r"(cthr), "r"(1u << i));
    }
    // candidates -> triggers, exactly (about one candidate per three lanes and row for p = 100)
    u32 cand = m;
    while (cand) {
        const u32 bit = cand & (0u - cand);
        cand ^= bit;
        const u32 o = 2u * (u32)(31 - __clz(bit)) + 14u;             // first stream bit of the window's hi block
        const bool k0 = o < 32u, k2 = o >= 64u;
        const u32 lo = k0 ? S[0] : (k2 ? S[2] : S[1]);
        const u32 hi = k0 ? S[1] : S[2];                             // k2: o + 20 <= 96, the upper word is not reached
        const u32 v = __funnelshift_r(lo, hi, o);                    // (shift taken mod 32) 20 bits: hi block, lo block
        u32 h = xt[v & 1023u].x + xt[(v >> 10) & 1023u].y;
        h = min(h, h - PFP_PW);
        if (!pfp_is_trigger(h, C.pinv, C.pshift, C.plimit)) m ^= bit;
    }
    return m;
}

// The interior rows of the buffer (every position inside [q_lo, q_hi), whole 16-byte units): one
// persistent 1024-thread CTA per SM, every warp walks a CONTIGUOUS run of rows (a running pointer
// instead of 64-bit index arithmetic; the per-tile trigger counts are kept per lane and flushed
// when the lane's word leaves its tile).  Rows overlap by one lane: row r covers the 32-position
// words 31r .. 31r+31 of the bit array, lane 0 only supplies the symbols in front of lane 1 (its
// word belongs to lane 31 of row r-1) -- 1/32 of redundant work, and no special case for "the
// bytes before my row".
// A row holding anything besides A C G T is not handled here: its number goes to `redo` and
// kr_scan_rows_k does it by the rolling arithmetic -- this loop has no calls and no clipping.
// BLK = 5: two blocks of 5 symbols (w <= 10); BLK = 4: four blocks of 4 symbols (11 <= w <= 16)
template <int BLK>
__global__ void __launch_bounds__(KD_T, 1) kr_scan_ivf_k(const unsigned char *__restrict__ A8, pfp_scan_consts C,
                                                         const void *__restrict__ etab_g,
                                                         const void *__restrict__ xtab_g, u32 cthr,
                                                         u32 *__restrict__ mask32, u32 *__restrict__ tile_cnt,
                                                         u32 row_lo, u32 n_rows,
                                                         u32 *__restrict__ redo, u32 *__restrict__ redo_n) {
    extern __shared__ __align__(16) u32 ke_sm[];
    const u32 lane = threadIdx.x & 31;
    const unsigned char *rep_lane;
    const void *xt_v;
    if constexpr (BLK == 5) {
        u32 *rep = ke_sm;
        uint2 *xt = reinterpret_cast<uint2 *>(ke_sm + KE_ENT * 32);
        for (u32 i = threadIdx.x; i < KE_ENT * 32; i += KD_T) rep[i] = static_cast<const u32 *>(etab_g)[i >> 5];
        for (u32 i = threadIdx.x; i < KE_ENT; i += KD_T) xt[i] = static_cast<const uint2 *>(xtab_g)[i];
        rep_lane = reinterpret_cast<const unsigned char *>(rep) + lane * 4;
        xt_v = xt;
    } else {
        uint2 *rep = reinterpret_cast<uint2 *>(ke_sm);
        uint4 *xt = reinterpret_cast<uint4 *>(ke_sm + K4_ENT * 16 * 2);
        for (u32 i = threadIdx.x; i < K4_ENT * 16; i += KD_T) rep[i] = static_cast<const uint2 *>(etab_g)[i >> 4];
        for (u32 i = threadIdx.x; i < K4_ENT; i += KD_T) xt[i] = static_cast<const uint4 *>(xtab_g)[i];
        rep_lane = reinterpret_cast<const unsigned char *>(rep) + (lane & 15) * 8;
        xt_v = xt;
    }
    __syncthreads();
    const u32 g = blockIdx.x * (KD_T / 32) + (threadIdx.x >> 5), nw = gridDim.x * (KD_T / 32);
    const u32 r0 = row_lo + (u32)((u64)g * n_rows / nw), r1 = row_lo + (u32)((u64)(g + 1) * n_rows / nw);
    if (r0 >= r1) return;
    u32 word = r0 * 31 + lane;                                       // my 32 positions = bit-array word `word`
    const uint4 *p = reinterpret_cast<const uint4 *>(A8 + (u64)word * 32);
    u32 *pm = mask32 + word;
    u32 acc = 0;                                                     // triggers of my words in tile word >> 10
    uint4 u0 = __ldg(p), u1 = __ldg(p + 1);
    for (u32 row = r0; row < r1; row++) {
        u32 bad = 0;
        const u32 S1 = dna_pack16(u0, bad), S2 = dna_pack16(u1, bad);
        // the bytes are packed: their registers take the next row, which has the rest of this one to arrive
        p += 62;
        if (row + 1 < r1) { u0 = __ldg(p); u1 = __ldg(p + 1); }
        const u32 S0 = __shfl_up_sync(0xffffffffu, S2, 1);          // the 16 symbols in front of my run
        if (!__any_sync(0xffffffffu, bad != 0)) {
            const u32 S[3] = {S0, S1, S2};
            u32 m;
            if constexpr (BLK == 5) m = ke_row_bits(S, rep_lane, static_cast<const uint2 *>(xt_v), C, cthr);
            else m = k4_row_bits(S, rep_lane, static_cast<const uint4 *>(xt_v), C, cthr);
            if (lane != 0) {
                *pm = m;
                acc += __popc(m);
            }
        } else if (lane == 0) {
            redo[atomicAdd(redo_n, 1u)] = row;
        }
        const u32 nword = word + 31;
        if (((nword ^ word) >> 10) != 0 && acc) {                    // my next word lies in the next tile
            atomicAdd(&tile_cnt[word >> 10], acc);
            acc = 0;
        }
        word = nword;
        pm += 31;
    }
    if (acc) atomicAdd(&tile_cnt[(word - 31) >> 10], acc);
}

// The rows the loop above does not take: the first and last rows of the buffer (clipped to
// [q_lo, q_hi), partial 16-byte units, the padding words of the last tile) and the rows of the
// `redo` list, by the rolling arithmetic -- exact for any bytes.
template <int W>
__global__ void __launch_bounds__(256) kr_scan_rows_k(const uint4 *__restrict__ A, u64 q_end, u64 q_lo, u64 q_hi,
                                                      pfp_scan_consts C, u32 *__restrict__ mask32,
                                                      u32 *__restrict__ tile_cnt, u32 nwords, u32 nrows,
                                                      u32 fast_lo, u32 fast_n, const u32 *__restrict__ redo,
                                                      const u32 *__restrict__ redo_n, u32 *__restrict__ alpha) {
    const u32 lane = threadIdx.x & 31;
    const u32 nb = nrows - fast_n, total = nb + *redo_n;
    for (u32 idx = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); idx < total; idx += gridDim.x * (blockDim.x / 32)) {
        const u32 row = idx < fast_lo ? idx : idx < nb ? idx + fast_n : redo[idx - nb];
        const u32 word = row * 31 + lane;
        const u64 q = (u64)word * 32;
        const uint4 u0 = kd_load_unit(A, q_end, (i64)q), u1 = kd_load_unit(A, q_end, (i64)q + 16);
        u32 m = kd_row_by_arithmetic<W>(u0, u1, lane, C, q, q_lo >= (u64)(W - 1) ? q_lo - (u64)(W - 1) : 0, q_end, true, alpha);
        const bool mine = (lane != 0 || row == 0) && word < nwords;
        if (q < q_lo || q + 32 > q_hi) m &= range_mask32(q, q_lo, q_hi);
        if (!mine) m = 0;
        if (mine) mask32[word] = m;
        // per-tile counts: the words of a row lie in at most two tiles
        const u32 c = __popc(m);
        const u32 t0 = (row * 31 + 1) >> 10;
        const bool in0 = (word >> 10) == t0 || lane == 0;
        const u32 c0 = __reduce_add_sync(0xffffffffu, in0 ? c : 0u);
        const u32 c1 = __reduce_add_sync(0xffffffffu, in0 ? 0u : c);
        if (lane == 0) {
            if (c0) atomicAdd(&tile_cnt[t0], c0);
            if (c1) atomicAdd(&tile_cnt[t0 + 1], c1);
        }
    }
}

// K1c: bits -> ascending global positions
__global__ void __launch_bounds__(K1_T) kr_emit_k(const uint4 *__restrict__ mask,
                                                  const u64 *__restrict__ tile_off,
                                                  u64 pos_bias /* buf_pos0 - delta */,
                                                  u64 *__restrict__ out) {
    __shared__ u32 sm[9];
    const u32 t = threadIdx.x;
    const u64 tile = blockIdx.x;
    uint4 mv = mask[tile * (u64)K1_T + t];
    u32 m[4] = {mv.x, mv.y, mv.z, mv.w};
    u32 c = __popc(m[0]) + __popc(m[1]) + __popc(m[2]) + __popc(m[3]);
    u32 tot;
    u32 ex = block_excl_scan_256(c, &tot, sm);
    if (tot == 0) return;
    u64 o = tile_off[tile] + ex;
    u64 q = tile * (u64)K1_TILE + (u64)t * K1_RUN + pos_bias;
#pragma unroll
    for (int kk = 0; kk < 4; kk++) {
        u32 x = m[kk];
        while (x) {
            int b = __ffs(x) - 1;
            x &= x - 1;
            out[o++] = q + (u64)(kk * 32 + b);
        }
    }
}

// largest number of triggers in one tile (the streaming K2 pass has a per-tile capacity)
__global__ void __launch_bounds__(256) tile_max_k(const u32 *__restrict__ tile_cnt, u32 ntiles,
                                                  unsigned long long *__restrict__ out) {
    u32 m = 0;
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < ntiles; i += gridDim.x * blockDim.x)
        m = max(m, tile_cnt[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(out, (unsigned long long)m);
}

template <int W>
static void launch_scan(pfpb200_ctx *ctx, u32 ntiles, const uint4 *A, u64 q_end, u64 q_lo, u64 q_hi,
                        const pfp_scan_consts &C, uint4 *mask, u32 *tile_cnt) {
    kr_scan_k<W><<<ntiles, K1_T, K1_SMEM, ctx->stream>>>(A, q_end, q_lo, q_hi, C, mask, tile_cnt);
}

#define K1_CASE(W) case W: launch_scan<W>(ctx, ntiles, A, q_end, q_lo, q_hi, C, mask, tile_cnt); break;

template <int W>
static cudaError_t launch_scan_iv(pfpb200_ctx *ctx, u32 ntiles, const uint4 *A, u64 q_end, u64 q_lo, u64 q_hi,
                                  const pfp_scan_consts &C, uint4 *mask, u32 *tile_cnt, u32 *redo) {
    const u32 nwords = ntiles * (u32)(K1_TILE / 32);      // every word of every tile gets written
    const u32 nrows = (nwords + 30) / 31;
    // rows that need no clipping: all 1024 positions inside [q_lo, q_hi) and inside whole 16-byte units
    const u64 lim = q_hi < (q_end & ~(u64)15) ? q_hi : (q_end & ~(u64)15);
    u64 f_lo = (q_lo + 991) / 992;
    if (f_lo < 1) f_lo = 1;
    const u64 f_hi = lim >= 1024 ? (lim - 1024) / 992 + 1 : 0;
    const u32 fast_lo = f_hi > f_lo ? (u32)f_lo : 0u, fast_n = f_hi > f_lo ? (u32)(f_hi - f_lo) : 0u;
    u32 *redo_n = reinterpret_cast<u32 *>(&ctx->d_flags[3]);
    if (fast_n) {
        if (W <= 10)
            kr_scan_ivf_k<5><<<ctx->sm_count, KD_T, KE_SMEM, ctx->stream>>>(reinterpret_cast<const unsigned char *>(A), C,
                                                                           ctx->iv_etab, ctx->iv_xtab, ctx->iv_cthr,
                                                                           reinterpret_cast<u32 *>(mask), tile_cnt,
                                                                           fast_lo, fast_n, redo, redo_n);
        else
            kr_scan_ivf_k<4><<<ctx->sm_count, KD_T, K4_SMEM, ctx->stream>>>(reinterpret_cast<const unsigned char *>(A), C,
                                                                           ctx->iv_etab, ctx->iv_xtab, ctx->iv_cthr,
                                                                           reinterpret_cast<u32 *>(mask), tile_cnt,
                                                                           fast_lo, fast_n, redo, redo_n);
        ctx->launches++;
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    kr_scan_rows_k<W><<<ctx->sm_count, 256, 0, ctx->stream>>>(A, q_end, q_lo, q_hi, C, reinterpret_cast<u32 *>(mask),
                                                              tile_cnt, nwords, nrows, fast_lo, fast_n, redo, redo_n,
                                                              ctx->d_alpha);
    return cudaGetLastError();
}
#define KE_CASE(W) case W: le = launch_scan_iv<W>(ctx, ntiles, A, q_end, q_lo, q_hi, C, mask, tile_cnt, redo); break;

// dynamic shared memory limits of every scan kernel and the constant powers of two, on ctx's device
int pfp_scan_init(pfpb200_ctx *ctx) {
#define K1_ATTR(W) PFP_CUDA(ctx, cudaFuncSetAttribute(kr_scan_k<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, K1_SMEM));
    K1_ATTR(4) K1_ATTR(5) K1_ATTR(6) K1_ATTR(7) K1_ATTR(8) K1_ATTR(9) K1_ATTR(10)
    K1_ATTR(11) K1_ATTR(12) K1_ATTR(13) K1_ATTR(14) K1_ATTR(15) K1_ATTR(16)
    K1_ATTR(20) K1_ATTR(24) K1_ATTR(28) K1_ATTR(31) K1_ATTR(32)
#undef K1_ATTR
    PFP_CUDA(ctx, cudaFuncSetAttribute(kr_scan_ivf_k<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)KE_SMEM));
    PFP_CUDA(ctx, cudaFuncSetAttribute(kr_scan_ivf_k<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K4_SMEM));
    u32 h[33];
    for (int i = 0; i < 32; i++) h[i] = 1u << i;
    h[32] = 0;
    PFP_CUDA(ctx, cudaMemcpyToSymbol(kd_pow2, h, sizeof(h), 0, cudaMemcpyHostToDevice));
    return PFPB200_OK;
}

// p^-1 modulo the prime PW (extended Euclid); 0 when p is a multiple of PW
static u32 inverse_mod_pw(u32 p) {
    i64 r0 = PFP_PW, r1 = p % PFP_PW, t0 = 0, t1 = 1;
    if (r1 == 0) return 0;
    while (r1) {
        const i64 qq = r0 / r1;
        const i64 r2 = r0 - qq * r1; r0 = r1; r1 = r2;
        const i64 t2 = t0 - qq * t1; t0 = t1; t1 = t2;
    }
    return (u32)(t0 < 0 ? t0 + PFP_PW : t0);
}

// the two 1024-entry tables of the interval form for (w, p), cached in the context
static int ensure_iv_tables(pfpb200_ctx *ctx, const pfp_scan_consts &C) {
    if (ctx->iv_etab && ctx->iv_w == C.w && ctx->iv_p == C.p) return PFPB200_OK;
    if (!ctx->iv_etab) {                                    // room for either scheme: 1024 x 4 / 256 x 8 and 1024 x 8 / 256 x 16 bytes
        PFP_CUDA(ctx, cudaMalloc(&ctx->iv_etab, KE_ENT * sizeof(u32)));
        PFP_CUDA(ctx, cudaMalloc(&ctx->iv_xtab, KE_ENT * sizeof(uint2)));
    }
    const u32 uinv = inverse_mod_pw(C.p);
    // theta = (K + 1) 2^16 / PW, K = (PW - 1) / p: every trigger has T < (floor(theta) + 4) << 16 (+ 7 with four blocks)
    const u64 theta = (((u64)(PFP_PW - 1) / C.p + 1) << 16) / PFP_PW;
    if (C.w <= (u32)KD_MAXW) {
        dna_etab_k<<<KE_ENT / 256, 256, 0, ctx->stream>>>(C, uinv, static_cast<u32 *>(ctx->iv_etab),
                                                          static_cast<uint2 *>(ctx->iv_xtab));
        ctx->iv_cthr = (u32)((theta + 4) << 16);
    } else {
        dna_etab4_k<<<1, K4_ENT, 0, ctx->stream>>>(C, uinv, static_cast<uint2 *>(ctx->iv_etab),
                                                   static_cast<uint4 *>(ctx->iv_xtab));
        ctx->iv_cthr = (u32)((theta + 7) << 16);
    }
    PFP_LAUNCHED(ctx);
    ctx->iv_w = C.w;
    ctx->iv_p = C.p;
    return PFPB200_OK;
}

// K1a + the scan over tiles.  On return sb describes the trigger bits of the buffer, sb->total
// is the number of triggers and sb->max_tile_cnt the largest per-tile count (read back: one
// synchronisation).
int pfp_scan_bits(pfpb200_ctx *ctx, const u8 *d_buf, u64 n_buf, u64 buf_pos0, u64 own_lo, u64 own_hi,
                  u32 w, u32 p, bool held, ScanBits *sb, float *ms_scan) {
    memset(sb, 0, sizeof(*sb));
    pfp_scan_consts C = pfp_make_scan_consts(w, p);
    uintptr_t addr = (uintptr_t)d_buf;
    u64 delta = addr & 15;
    const uint4 *A = reinterpret_cast<const uint4 *>(addr - delta);
    u64 q_end = delta + n_buf;
    sb->A = A;
    sb->q_end = q_end;
    sb->pos_bias = buf_pos0 - delta;
    // first position whose whole window lies in the text and in the buffer
    u64 lo = own_lo;
    if (lo < (u64)w - 1) lo = (u64)w - 1;
    if (lo < buf_pos0 + w - 1) lo = buf_pos0 + w - 1;
    u64 hi = own_hi;
    if (hi > buf_pos0 + n_buf) hi = buf_pos0 + n_buf;
    if (ms_scan) *ms_scan = 0;
    if (!(lo < hi && n_buf > 0)) return PFPB200_OK;
    u64 q_lo = lo - buf_pos0 + delta, q_hi = hi - buf_pos0 + delta;
    u64 nt64 = (q_end + K1_TILE - 1) / K1_TILE;
    if (nt64 > 0x7FFFFFFFull) return pfp_fail(ctx, PFPB200_E_LIMIT, "shard too large");
    u32 ntiles = (u32)nt64;
    uint4 *mask = nullptr;
    u32 *tile_cnt = nullptr;
    u64 *tile_off = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &mask, (size_t)ntiles * K1_T, held));
    PFP_TRY(pfp_alloc_t(ctx, &tile_cnt, ntiles, held));
    PFP_TRY(pfp_alloc_t(ctx, &tile_off, ntiles, held));
    PfpEvents evs(2);
    if (!evs.ok) return pfp_fail(ctx, PFPB200_E_CUDA, "cudaEventCreate failed");
    const cudaEvent_t e0 = evs[0], e1 = evs[1];
    // a text that is not DNA (most rows of the previous scan went to the arithmetic) is scanned by the
    // rolling kernel directly; the interval form is tried again every eighth call
    const bool not_dna = !ctx->k1_rolling && ctx->iv_skip > 0 && ctx->iv_skip-- > 0;
    // interval form (w <= 16): p must be invertible modulo PW and the threshold must leave the 16-bit
    // range alone; otherwise the rolling kernel
    const bool iv = w <= 16 && !ctx->k1_rolling && !not_dna && p >= 10 && p < PFP_PW &&
                    (u64)ntiles * (K1_TILE / 32) < 0xFFFFFF00ull;
    u32 *redo = nullptr;                                   // rows the interval form hands to the arithmetic
    if (iv) {
        PFP_TRY(ensure_iv_tables(ctx, C));
        PFP_TRY(pfp_alloc_t(ctx, &redo, (size_t)ntiles * (K1_TILE / 32) / 31 + 2, false));
    }
    PFP_CUDA(ctx, cudaEventRecord(e0, ctx->stream));
    ctx->alpha_valid = false;
    if (iv) {
        // bits and per-tile counts (added up by the warps) for every row
        PFP_CUDA(ctx, cudaMemsetAsync(tile_cnt, 0, (size_t)ntiles * sizeof(u32), ctx->stream));
        PFP_CUDA(ctx, cudaMemsetAsync(ctx->d_alpha, 0, 8 * sizeof(u32), ctx->stream));
        ctx->alpha_valid = buf_pos0 == 0 && own_lo == 0;       // the whole text of a single-GPU parse
        PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[3], 0, sizeof(u64), ctx->stream));
        cudaError_t le = cudaSuccess;
        switch ((int)w) {
            KE_CASE(4) KE_CASE(5) KE_CASE(6) KE_CASE(7) KE_CASE(8) KE_CASE(9) KE_CASE(10)
            KE_CASE(11) KE_CASE(12) KE_CASE(13) KE_CASE(14) KE_CASE(15) KE_CASE(16)
            default: le = cudaErrorInvalidValue;
        }
        ctx->launches++;
        if (le != cudaSuccess)
            return pfp_fail(ctx, PFPB200_E_CUDA, "kr_scan_ivf_k / kr_scan_rows_k launch: %s", cudaGetErrorString(le));
    } else {
        switch (w <= K1_MAXW_FAST ? (int)w : 0) {
            K1_CASE(4) K1_CASE(5) K1_CASE(6) K1_CASE(7) K1_CASE(8) K1_CASE(9) K1_CASE(10)
            K1_CASE(11) K1_CASE(12) K1_CASE(13) K1_CASE(14) K1_CASE(15) K1_CASE(16)
            K1_CASE(20) K1_CASE(24) K1_CASE(28) K1_CASE(31) K1_CASE(32)
            default:
                kr_scan_generic_k<<<ntiles, K1_T, 0, ctx->stream>>>(
                    reinterpret_cast<const unsigned char *>(A), q_end, q_lo, q_hi, C, mask, tile_cnt);
        }
        PFP_LAUNCHED(ctx);
    }
    PFP_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
    if (redo) PFP_TRY(pfp_free_now(ctx, redo));
    PFP_CUDA(ctx, cudaMemsetAsync(&ctx->d_flags[5], 0, sizeof(u64), ctx->stream));
    PFP_TRY(pfp_exclusive_scan_u32_u64(ctx, tile_cnt, tile_off, ntiles, &ctx->d_flags[1]));
    tile_max_k<<<ctx->sm_count, 256, 0, ctx->stream>>>(tile_cnt, ntiles,
                                                       reinterpret_cast<unsigned long long *>(&ctx->d_flags[5]));
    PFP_LAUNCHED(ctx);
    PFP_CUDA(ctx, cudaMemcpyAsync(&ctx->h_flags[1], &ctx->d_flags[1], 5 * sizeof(u64),
                                  cudaMemcpyDeviceToHost, ctx->stream));
    PFP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float a = 0;
    cudaEventElapsedTime(&a, e0, e1);
    if (ms_scan) *ms_scan = a;
    sb->ntiles = ntiles;
    sb->mask = mask; sb->tile_cnt = tile_cnt; sb->tile_off = tile_off;
    sb->total = ctx->h_flags[1];
    sb->max_tile_cnt = (u32)ctx->h_flags[5];
    if (iv && (u64)(u32)ctx->h_flags[3] * 4 > (u64)ntiles * (K1_TILE / 32) / 31) ctx->iv_skip = 7;
    return PFPB200_OK;
}

int pfp_scan_bits_free(pfpb200_ctx *ctx, ScanBits *sb) {
    PFP_TRY(pfp_free_now(ctx, sb->mask));
    PFP_TRY(pfp_free_now(ctx, sb->tile_cnt));
    PFP_TRY(pfp_free_now(ctx, sb->tile_off));
    sb->mask = nullptr; sb->tile_cnt = nullptr; sb->tile_off = nullptr;
    return PFPB200_OK;
}

// first and last trigger of the buffer straight from the bits (global positions; total > 0)
__global__ void __launch_bounds__(1024) first_last_trigger_k(const u32 *__restrict__ mask32,
                                                             const u32 *__restrict__ tile_cnt, u32 ntiles,
                                                             u64 pos_bias, u64 *__restrict__ out2) {
    __shared__ u32 s_first, s_last;
    __shared__ u32 s_wf, s_wl;
    const u32 t = threadIdx.x;
    if (t == 0) { s_first = 0xFFFFFFFFu; s_last = 0; s_wf = 0xFFFFFFFFu; s_wl = 0; }
    __syncthreads();
    u32 lo = 0xFFFFFFFFu, hi = 0;
    for (u32 i = t; i < ntiles; i += 1024)
        if (tile_cnt[i]) { lo = min(lo, i); hi = max(hi, i + 1); }
    if (lo != 0xFFFFFFFFu) { atomicMin(&s_first, lo); atomicMax(&s_last, hi); }
    __syncthreads();
    if (s_first == 0xFFFFFFFFu) return;
    const u32 tf = s_first, tl = s_last - 1;
    const u32 wf = mask32[(u64)tf * 1024 + t], wl = mask32[(u64)tl * 1024 + t];    // 1024 words per tile
    if (wf) atomicMin(&s_wf, t);
    if (wl) atomicMax(&s_wl, t + 1);
    __syncthreads();
    if (t == s_wf) out2[0] = ((u64)tf * 1024 + t) * 32 + (u64)(__ffs(wf) - 1) + pos_bias;
    if (t + 1 == s_wl) out2[1] = ((u64)tl * 1024 + t) * 32 + (u64)(31 - __clz(wl)) + pos_bias;
}

int pfp_scan_first_last(pfpb200_ctx *ctx, const ScanBits &sb, u64 *d_out2) {
    if (sb.ntiles == 0 || sb.total == 0) return PFPB200_OK;
    first_last_trigger_k<<<1, 1024, 0, ctx->stream>>>(reinterpret_cast<const u32 *>(sb.mask), sb.tile_cnt, sb.ntiles,
                                                      sb.pos_bias, d_out2);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

// K1c alone: bits -> ascending positions in out[0..total)
int pfp_scan_emit(pfpb200_ctx *ctx, const ScanBits &sb, u64 *out) {
    if (sb.ntiles == 0 || sb.total == 0) return PFPB200_OK;
    kr_emit_k<<<sb.ntiles, K1_T, 0, ctx->stream>>>(sb.mask, sb.tile_off, sb.pos_bias, out);
    PFP_LAUNCHED(ctx);
    return PFPB200_OK;
}

// Runs K1a+scan+K1c.  On return *d_out (scratch, or held when `held`) holds *n_out positions;
// `extra_slots` more u64 are allocated behind them for the caller (final virtual trigger).
int pfp_scan_stage(pfpb200_ctx *ctx, const u8 *d_buf, u64 n_buf, u64 buf_pos0, u64 own_lo,
                   u64 own_hi, u32 w, u32 p, u64 extra_slots, bool held, u64 **d_out, u64 *n_out,
                   float *ms_scan, float *ms_emit) {
    *d_out = nullptr;
    *n_out = 0;
    ScanBits sb;
    PFP_TRY(pfp_scan_bits(ctx, d_buf, n_buf, buf_pos0, own_lo, own_hi, w, p, false, &sb, ms_scan));
    u64 *out = nullptr;
    PFP_TRY(pfp_alloc_t(ctx, &out, (size_t)(sb.total + extra_slots), held));
    PfpEvents evs(2);
    if (!evs.ok) return pfp_fail(ctx, PFPB200_E_CUDA, "cudaEventCreate failed");
    const cudaEvent_t e1 = evs[0], e2 = evs[1];
    PFP_CUDA(ctx, cudaEventRecord(e1, ctx->stream));
    PFP_TRY(pfp_scan_emit(ctx, sb, out));
    PFP_CUDA(ctx, cudaEventRecord(e2, ctx->stream));
    PFP_TRY(pfp_scan_bits_free(ctx, &sb));
    PFP_CUDA(ctx, cudaEventSynchronize(e2));
    float b = 0;
    cudaEventElapsedTime(&b, e1, e2);
    if (ms_emit) *ms_emit = b;
    *d_out = out;
    *n_out = sb.total;
    return PFPB200_OK;
}
