// pfp_stages.cuh -- data layout in HBM shared by the stages, and the stage entry points.
#pragma once
#include "pfp_common.cuh"

// ---- text view ---------------------------------------------------------------------------------
// A shard buffer T[0..n_buf) whose first byte is global text position pos0.  Global positions
// -1 and >= n_global are the reference's virtual 0x02 borders (newscan.cpp:329,376).
struct TextView {
    const u8 *T;
    u64 n_buf;
    i64 pos0;
    i64 n_global;
};

__device__ __forceinline__ u8 tv_byte(const TextView &tv, i64 g) {
    if (g < 0 || g >= tv.n_global) return (u8)PFP_DOLLAR;
    return tv.T[g - tv.pos0];
}

// ---- per-phrase arrays (P entries, text order) ----------------------------------------------------
// 16-byte fingerprint record of a phrase, written once by K2, read once by K3: both 64-bit NH
// sums in full (128 bits).  The length is NOT carried: text bytes are never zero, so the zero
// padded chunks determine it, and the one thread per word that needs it (the word's creator in
// K3) recomputes it from ends[].  The table key and the check digest are derived from the 128
// bits by K3.
struct __align__(16) PhraseFp {
    u64 fpa;        // first NH sum
    u64 fpb;        // second NH sum (Toeplitz-shifted keys)
};

struct PhraseArrays {
    u64 *ends;      // inclusive global END position of the phrase (trigger position; n+w-1 for the last)
    PhraseFp *rec;  // fingerprint records
    u8 *last;       // .last stream
    u8 *sai;        // .sai stream (5 bytes per phrase) or null
};

// ---- dictionary arrays (d entries, in fingerprint-key order = "uid" order) ---------------------------
// what the .dict/.occ emission needs of a word, in one 16-byte record: a gather by rank then
// touches one sector per word instead of three (written by the ranking's key pass, which reads
// these fields of every word anyway)
struct __align__(16) WordMeta { u64 off; u32 len; u32 count; };

constexpr u32 UID_CREATOR = 0x80000000u;   // uid[j] with slot_of_word: marks the word id held by the word's creator

struct DictArrays {
    u64 d = 0;
    WordMeta *meta = nullptr;   // [d] filled by pfp_rank_stage
    u32 *uid = nullptr;     // [P] phrase -> uid
    u32 *slot_of_word = nullptr;   // [d] non-null: uid[j] is word id | UID_CREATOR on the record that
                                   // created a word (won its table slot), and the word's slot in a
                                   // table of `slots` entries on the others; word u lives in slot
                                   // slot_of_word[u] (pfp_dedup_stage; pfp_uid_words makes every
                                   // uid[j] a word id)
    u64 slots = 0;
    u32 *rep = nullptr;     // [d] index of the phrase that created the word (won its table slot)
    i64 *ustart = nullptr;  // [d] global text position of that phrase's first byte (may be -1: virtual border)
    u32 *count = nullptr;   // [d] occurrences
    u32 *ulen = nullptr;    // [d] length in bytes
    u32 *uwords = nullptr;  // [d] length in 8-byte pool words
    u64 *uoff = nullptr;    // [d] offset into the pool (8-byte words)
    u64 *pool = nullptr;    // the words, zero padded to 8 bytes
    u64 pool_words = 0;
    u32 max_len = 0;
    u64 sum_len = 0;
};

// ---- fingerprint parameters ---------------------------------------------------------------------------
constexpr u32 NH_SEG_BYTES = 8192;                 // NH key table covers one segment
constexpr u32 NH_KEY_WORDS = NH_SEG_BYTES / 4 + 8; // + Toeplitz shift for the second sum
constexpr u64 NH_FOLD_A = 0x9E3779B97F4A7C15ULL;   // odd multipliers folding segment sums
constexpr u64 NH_FOLD_B = 0xD6E8FEB86659FD93ULL;

// ---- stages -----------------------------------------------------------------------------------------------
int pfp_scan_stage(pfpb200_ctx *ctx, const u8 *d_buf, u64 n_buf, u64 buf_pos0, u64 own_lo,
                   u64 own_hi, u32 w, u32 p, u64 extra_slots, bool held, u64 **d_out, u64 *n_out,
                   float *ms_scan, float *ms_emit);
int pfp_scan_bits(pfpb200_ctx *ctx, const u8 *d_buf, u64 n_buf, u64 buf_pos0, u64 own_lo, u64 own_hi,
                  u32 w, u32 p, bool held, ScanBits *sb, float *ms_scan);
int pfp_scan_emit(pfpb200_ctx *ctx, const ScanBits &sb, u64 *out);
int pfp_scan_first_last(pfpb200_ctx *ctx, const ScanBits &sb, u64 *d_out2);   // global positions of the first / last trigger
int pfp_scan_bits_free(pfpb200_ctx *ctx, ScanBits *sb);
int pfp_hash_stage(pfpb200_ctx *ctx, const TextView &tv, const PhraseArrays &ph, u64 P,
                   i64 first_start, u32 w);
int pfp_hash_list(pfpb200_ctx *ctx, const TextView &tv, const PhraseArrays &ph, i64 first_start, u32 w,
                  const u32 *long_list, const u32 *long_count, u64 max_count, PhraseFp *rec_compact);
int pfp_insert_list(pfpb200_ctx *ctx, const TextView &tv, const PhraseFp *rec_small, const u32 *list,
                    const u32 *list_count, u64 list_cap, void *tab, u64 cap, const u64 *ends, i64 first_start,
                    u32 w, const DictArrays &D, u64 pool_cap, PhraseFp *rec_full);
int pfp_table_pending(pfpb200_ctx *ctx, const void *tab, u64 P, u32 *uid, u32 *count);
// K2 + K3 + pool in one pass (the table insert fused into the streaming kernel); D is complete on
// return.  ph.rec may be null (only sharded parsing keeps the creators' fingerprints).
int pfp_words_fused_stage(pfpb200_ctx *ctx, const ScanBits &sb, const TextView &tv, const PhraseArrays &ph,
                          u64 P, i64 first_start, u32 w, bool emit_ends, DictArrays *D);
int pfp_records_range(pfpb200_ctx *ctx, const TextView &tv, const PhraseArrays &ph, u64 j0, u64 P, u32 w);
// K2 streaming: one pass over text + trigger bits writes ends (optional), .last, .sai and the
// fingerprint records of all P phrases (ph.ends[P-1] must already hold a final virtual end, if any)
bool pfp_stream_ok(const ScanBits &sb, u32 w);   // false: w > 32 or a tile too dense -> per-phrase kernels
int pfp_stream_stage(pfpb200_ctx *ctx, const ScanBits &sb, const TextView &tv, const PhraseArrays &ph,
                     u64 P, i64 first_start, u32 w, bool emit_ends);
int pfp_dedup_stage(pfpb200_ctx *ctx, const PhraseArrays &ph, u64 P, i64 first_start, u32 w, DictArrays *D);
int pfp_uid_words(pfpb200_ctx *ctx, DictArrays *D, u64 n);   // uid[0..n) -> word ids, if D->slot_of_word is set
int pfp_pool_stage(pfpb200_ctx *ctx, const TextView &tv, const u64 *ends, i64 first_start, u32 w,
                   DictArrays *D);
// Lexicographic order of the d pool words: order[i] = uid of the word of rank i+1.
int pfp_rank_stage(pfpb200_ctx *ctx, DictArrays &D, u32 **order, u32 *rounds, bool alpha_from_scan = false);
// .dict / .occ bytes and rank-per-uid from the order; outputs are `held` device buffers.
int pfp_dict_stage(pfpb200_ctx *ctx, const DictArrays &D, const u32 *order, u32 strip_w,
                   u8 **dict, u64 *dict_bytes, u32 **occ, u32 **rank_of_uid,
                   const u32 *remap_uid = nullptr, u64 remap_n = 0, u32 *remap_out = nullptr);
int pfp_remap_stage(pfpb200_ctx *ctx, const u32 *uid, const u32 *rank_of_uid, u64 P, u32 *parse);

int pfp_first_invalid(pfpb200_ctx *ctx, const u8 *d_text, u64 n, u64 *d_first);

// ---- overlapped file I/O and K0 (pfp_ingest.cu) ------------------------------------------------------------
int pfp_file_to_device(pfpb200_ctx *ctx, int fd, u64 off, u64 bytes, u8 *d_dst);
int pfp_device_to_file(pfpb200_ctx *ctx, const char *name, const void *d_src, u64 bytes);
int pfp_device_to_fd(pfpb200_ctx *ctx, int fd, u64 file_off, const void *d_src, u64 bytes, const char *name);
void pfp_io_destroy(pfpb200_ctx *ctx);
// FASTA bytes in HBM -> the text T of `-f` mode (kseq.h:177-218); *supported = 0: host reader needed
int pfp_fasta_device(pfpb200_ctx *ctx, const u8 *d_file, u64 n, u8 **d_text, u64 *n_text, int *supported,
                     bool held);

// ---- sharded parsing building blocks ------------------------------------------------------------------------
int pfp_gather_word_fp(pfpb200_ctx *ctx, const DictArrays &D, const PhraseArrays &ph, u64 *wfpa,
                       u64 *wfpb);
int pfp_merge_stage(pfpb200_ctx *ctx, u64 n, const u64 *fpa, const u64 *fpb, const u32 *len,
                    const u32 *count_in, const u32 *uwords_in, const u64 *pool, u64 pool_words,
                    bool verify, DictArrays *D, u32 **uid_of_entry);
int pfp_merge_verify(pfpb200_ctx *ctx, u64 n, const u32 *uid_of_entry, const u32 *rep, const u32 *len_in,
                     const u32 *uwords_in, const u64 *pool);
int pfp_verify_stage(pfpb200_ctx *ctx, const TextView &tv, const u64 *ends, i64 first_start, u32 w, u64 P,
                     const DictArrays &D);

// ---- the last stage (pfp_pfbwt.cu) and its sharded form (pfp_pfbwt_multi.cu) ---------------------------------
// present[0..8): bit c set when byte value c occurs in d[0..N)
int pfp_dict_alphabet(pfpb200_ctx *ctx, const u8 *d, u64 N, u32 *present);

// the rank array of the sharded suffix sort, stored by position: block o = [o * per, (o + 1) * per)
// lives on rank o; kernels load and store it through the peers' block pointers
struct PmRanks {
    u64 *blk[PFPB200_MAX_RANKS];
    u64 per;
};

// one rank's state of a sharded pfbwt call (pfpb200_multi_pfbwt_file)
struct PmState {
    // inputs: the whole dictionary and parse-side streams (device pointers valid on this rank)
    const u8 *d = nullptr; u64 N = 0;
    const u32 *occ = nullptr; u64 dwords = 0;
    const u32 *ilist = nullptr; const u8 *bwlast = nullptr, *bwsai = nullptr; u64 psize = 0;
    u32 w = 0, flags = 0;
    // word structure and first-key coding
    u8 *tflag = nullptr; u32 *wid = nullptr, *istart = nullptr; u64 *wend = nullptr;
    u8 code[256]; int bs = 0, h0 = 0;
    // the owned first-key range and suffixes
    u64 rg_lo = 0, rg_hi = 0; int rg_has_lo = 0, rg_has_hi = 0;
    u64 M0 = 0, base = 0, M = 0, M2 = 0;
    int bn = 0, bm = 0, split = 0;                  // key layout: bits of N, bits of M0, two sorts
    u64 *pos = nullptr, *lo = nullptr; u32 *sl = nullptr, *hi = nullptr;   // per element (hi, lo: split key form)
    u64 *k0 = nullptr, *k1 = nullptr, *ks = nullptr, *ko = nullptr;
    u32 *v0 = nullptr, *v1 = nullptr, *vs = nullptr, *vo = nullptr;
    u32 *slot = nullptr, *slot2 = nullptr, *head = nullptr, *escan = nullptr, *rs = nullptr;
    u8 *flag = nullptr, *keep = nullptr;
    u64 *sa_pos = nullptr; u32 *sa_grp = nullptr;  // per local slot
    // emission
    uint2 *mrec = nullptr; u16 *mc = nullptr; u32 *cnt = nullptr, *gscan = nullptr; u8 *newgrp = nullptr;
    u64 *off = nullptr; u64 ngroups = 0, chars = 0, n_hard = 0;
    u8 *bwt = nullptr, *sa5 = nullptr, *ssa = nullptr, *esa = nullptr;
    u64 n_ssa = 0, n_esa = 0;
    int c_first = -1, c_last = -1;                  // first / last char of the piece (-1: empty)
};
int pm_words(pfpb200_ctx *ctx, PmState &S);
int pm_sample(pfpb200_ctx *ctx, PmState &S, u64 lo, u64 hi, u32 want, u64 *h_out, u32 *got);
int pm_count(pfpb200_ctx *ctx, PmState &S, u64 klo, u64 khi, int has_lo, int has_hi, u64 *count);
int pm_collect(pfpb200_ctx *ctx, PmState &S, int split);
int pm_update(pfpb200_ctx *ctx, PmState &S, const PmRanks &R, u64 h, int first, u64 *active);
int pm_gather(pfpb200_ctx *ctx, PmState &S, const PmRanks &R, u64 h);
int pm_sort(pfpb200_ctx *ctx, PmState &S);
int pm_sort_done(pfpb200_ctx *ctx, PmState &S);
int pm_count_chars(pfpb200_ctx *ctx, PmState &S);
int pm_fill(pfpb200_ctx *ctx, PmState &S);
int pm_samples(pfpb200_ctx *ctx, PmState &S, int at_end, int prev, int next, u64 off);
