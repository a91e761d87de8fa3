// pfp_stages.cuh -- data layout in HBM shared by the stages, and the stage entry points.
#pragma once
#include "pfp_common.cuh"
#include <unistd.h>

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
                  const u32 *long_list, const u32 *long_count, u64 max_count);
int pfp_records_range(pfpb200_ctx *ctx, const TextView &tv, const PhraseArrays &ph, u64 j0, u64 P, u32 w);
// K2 streaming: one pass over text + trigger bits writes ends (optional), .last, .sai and the
// fingerprint records of all P phrases (ph.ends[P-1] must already hold a final virtual end, if any)
bool pfp_stream_ok(const ScanBits &sb, u32 w);   // false: w > 32 or a tile too dense -> per-phrase kernels
int pfp_stream_stage(pfpb200_ctx *ctx, const ScanBits &sb, const TextView &tv, const PhraseArrays &ph,
                     u64 P, i64 first_start, u32 w, bool emit_ends);
int pfp_dedup_stage(pfpb200_ctx *ctx, const PhraseArrays &ph, u64 P, i64 first_start, u32 w, DictArrays *D);
int pfp_uid_words(pfpb200_ctx *ctx, DictArrays *D, u64 n);   // uid[0..n) -> word ids, if D->slot_of_word is set
int pfp_pool_stage(pfpb200_ctx *ctx, const TextView &tv, DictArrays *D);
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
// FASTA bytes in HBM -> the text T of `-f` mode (kseq.h:177-218); *supported = 0: host reader needed.
constexpr u32 PFP_FASTA_LINE_START = 2;   // state of the K0 line automaton at the start of a file
// state / file_start: a piece of a file streamed in order (the automaton state carried across pieces)
int pfp_fasta_device(pfpb200_ctx *ctx, const u8 *d_file, u64 n, u8 **d_text, u64 *n_text, int *supported,
                     bool held, u32 *state = nullptr, bool file_start = true);

// ---- the streamed parse of a file larger than the device (pfp_chunked.cu) -------------------------------------
// pfpb200_parse_file in chunks of budget / 8 new bytes against one dictionary; *chunks = how many
int pfp_parse_file_streamed(pfpb200_ctx *ctx, const char *path, const pfpb200_opts *opts, pfpb200_stats *stats,
                            u64 budget, u64 *chunks);

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
// pfp_pfbwt.cu holds what both paths compute the same way: the word structure and first-key coding,
// the group heads of a doubling round, the emission and the sampled suffix array.  The two suffix
// sorts stay apart; the emission reads a sort's output only through a slot reader (PbPackedSlots,
// PbSplitSlots).
constexpr int PB_T = 256;

__device__ __forceinline__ bool pb_term(u8 c) { return c <= PFP_END_OF_WORD; }   // EndOfWord, EndOfDict

// The ORDER-PRESERVING DENSE CODES of the byte values that occur in the dictionary (terminators 1,
// then the text's alphabet from 2 up), bs bits each: a DNA dictionary has 7 values, 3 bits, and the
// first round of a doubling already sorts by 21 symbols instead of 8.
struct PbCodes { u8 code[256]; };

// the first key of position t: its first h0 symbols as dense codes, cut behind the word's terminator
// (zero padded); terminators get key 0 and sort in front.  code[]: PbCodes in shared memory
__device__ __forceinline__ u64 pb_first_key(const u8 *__restrict__ d, u64 N, const u8 *code, int h0, int bs, u64 t) {
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
    return k;
}

static inline int pb_bits(u64 v) {
    int b = 1;
    while (b < 64 && (v >> b) != 0) b++;
    return b;
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

// launches a PB_T-thread kernel over n items, none when n = 0 (a rank of the sharded path may own nothing)
#define PB_LAUNCH(ctx, n, kernel, ...)                                                          \
    do {                                                                                        \
        if ((n) > 0) {                                                                          \
            kernel<<<pfp_blocks((n), PB_T), PB_T, 0, (ctx)->stream>>>(__VA_ARGS__);              \
            PFP_LAUNCHED(ctx);                                                                  \
        }                                                                                       \
    } while (0)

// group starts of a sorted key array, and head[group] = slot of its first member (escan: the scan of flag)
__global__ void __launch_bounds__(PB_T) pb_gflags_k(const u64 *__restrict__ key, u64 M, u8 *__restrict__ flag);
__global__ void __launch_bounds__(PB_T) pb_heads_k(const u8 *__restrict__ flag, const u32 *__restrict__ escan,
                                                   const u32 *__restrict__ slot, u64 M, u32 *__restrict__ head);

// the inputs of a pfbwt call: the dictionary and the parse-side streams (device pointers)
struct PbInput {
    const u8 *d = nullptr; u64 N = 0;
    const u32 *occ = nullptr; u64 dwords = 0;
    const u32 *ilist = nullptr; const u8 *bwlast = nullptr, *bwsai = nullptr; u64 psize = 0;
    u32 w = 0, flags = 0;
};

// the word structure of the dictionary and the coding of the first key (pb_words)
struct PbWords {
    u32 *wid = nullptr;         // [N] word of every position (terminators before it): pb_word_ids, one-GPU path only
    u64 *wend = nullptr;        // [words + 1] position of every word's terminator
    u32 *istart = nullptr;      // [words] first .ilist entry of every word, less one
    PbCodes cd;
    int bs = 0, h0 = 0;         // bits of a code, symbols in the first key
};

// slot k of the sorted dictionary suffixes -> its position, its group (the slot where the group
// starts) and its word.  The one-GPU sort leaves (group << 32) | position in one u64 and reads the word
// from the per-position word ids; the sharded sort leaves three arrays per slot.
struct PbPackedSlots {
    const u64 *sa;
    const u32 *wid;
    __device__ __forceinline__ u32 pos(u64 k) const { return (u32)sa[k]; }
    __device__ __forceinline__ u32 grp(u64 k) const { return (u32)(sa[k] >> 32); }
    __device__ __forceinline__ u32 word(u64 k) const { return wid[pos(k)]; }
};
struct PbSplitSlots {
    const u64 *sa_pos;
    const u32 *sa_grp, *sa_word;
    __device__ __forceinline__ u64 pos(u64 k) const { return sa_pos[k]; }
    __device__ __forceinline__ u32 grp(u64 k) const { return sa_grp[k]; }
    __device__ __forceinline__ u32 word(u64 k) const { return sa_word[k]; }
};

// what the emission leaves: the BWT chars of the slots (of one window: chars [base, base + chars) of the
// slice) and, with -S / -s / -e, their suffix-array values
struct PbEmit {
    u8 *bwt = nullptr, *sa5 = nullptr;
    u64 chars = 0, n_hard = 0, ngroups = 0, base = 0;
};

// The plan of the emission over all n slots (pb_plan): per slot its member record, occurrences, and
// the start of its range in the BWT (off) and in the hard merge (hoff); per group its first slot and
// whether its chars are mixed.  Every group owns one contiguous range of the BWT, so the output can be
// produced for any run of whole groups [ka, kb) on its own: chars [off[ka], off[kb]) (pb_window).
struct PbPlan {
    uint2 *mrec = nullptr;      // [n] {word, suffix length}
    u16 *mc = nullptr;          // [n] char in front | whole word << 8 | counts << 9
    u32 *cnt = nullptr, *hcnt = nullptr;   // [n] occurrences, of them to merge
    u64 *off = nullptr, *hoff = nullptr;   // [n + 1] exclusive scans of cnt / hcnt
    u32 *first = nullptr;       // [ngroups + 1] first slot of every group
    u8 *mixed = nullptr;        // [ngroups + 1]
    u8 *newgrp = nullptr;       // [n] caller's scratch
    u32 *gscan = nullptr;       // [n] caller's scratch: groups before the slot
    u64 n = 0, ngroups = 0, chars = 0, n_hard = 0;
};


// the argument checks of pfbwt.x: the message of the first one that fails, or null
const char *pb_arg_error(u32 w, u32 flags);
// .dict .occ .ilist .bwlast [.bwsai when flags want a suffix array] into held buffers (in[k], n[k] entries
// of PB_UNIT[k] bytes), their sizes checked against each other
constexpr u64 PB_UNIT[5] = {1, 4, 4, 1, PFP_IBYTES};
int pb_read_file(pfpb200_ctx *ctx, const char *base, int k, void **d, u64 *count);   // one of them
int pb_read_inputs(pfpb200_ctx *ctx, const char *base, u32 flags, void *in[5], u64 n[5]);
int pb_sync_read(pfpb200_ctx *ctx, int slot, int n);   // h_flags[slot, slot + n) <- d_flags, then synchronise
// word ends, first .ilist entries and first-key coding; the word ends are found in chunks of at most
// PB_CHUNK positions, so the scratch does not grow with the dictionary
constexpr u64 PB_CHUNK = (u64)1 << 30;
int pb_words(pfpb200_ctx *ctx, const PbInput &in, PbWords *W);
int pb_word_ids(pfpb200_ctx *ctx, const PbInput &in, PbWords *W);   // W->wid[N] (the one-GPU sort reads it)
// the plan of the emission over n sorted slots; newgrp / gscan: scratch of n entries
template <class Slots>
int pb_plan(pfpb200_ctx *ctx, const PbInput &in, const PbWords &W, Slots sl, u64 n, u8 *newgrp, u32 *gscan, PbPlan *P);
// the end of the window of whole groups that starts at slot ka and holds at most cap chars (at least
// one group: a larger group gets a window of its own); *chars_end = off[*kb]
int pb_window_end(pfpb200_ctx *ctx, const PbPlan &P, u64 ka, u64 cap, u64 *kb, u64 *chars_end);
// the BWT chars (and SA values) of the slots [ka, kb), a run of whole groups, into buffers of the window:
// E->bwt[0, E->chars) = chars [off[ka], off[kb]); hard merge batches of at most min(PB_BATCH, hcap)
// occurrences; held: the outputs are held buffers recorded in ctx->pb_out[0..1], otherwise scratch
int pb_window(pfpb200_ctx *ctx, const PbInput &in, const PbWords &W, const PbPlan &P, u64 ka, u64 kb, u64 hcap,
              bool held, PbEmit *E);
// The device memory a pfbwt output call may use once its plan is done: PFPB200_PFBWT_BUDGET=<bytes> if
// set; otherwise, for a context alone on its device, the free memory plus what its arena holds unused,
// and for one of `share` > 1 contexts on the device, its share of the free memory.
int pb_budget(pfpb200_ctx *ctx, int share, u64 *budget);
// the device bytes of a window of at most cap chars (pb_out_bytes)
u64 pb_window_bytes(const PbPlan &P, u32 flags, u64 cap);
// the most chars of a window whose output fits the budget: P.chars when the whole output fits, else the
// largest c with pb_out_bytes(c) <= budget (0: one group per window)
u64 pb_window_chars(const PbPlan &P, u32 flags, u64 budget);
// the output files of one piece: .bwt, .sa (positioned writes), .ssa, .esa (appended from offset 0)
struct PbOutFiles {
    int fd[4] = {-1, -1, -1, -1};
    char name[4][4096];
    ~PbOutFiles() {
        for (int i = 0; i < 4; i++)
            if (fd[i] >= 0) close(fd[i]);
    }
};
// what writing a piece left: its windows, its run samples, its first / last char (-1: empty) and times
struct PbPiece {
    u64 windows = 0, n_ssa = 0, n_esa = 0;
    int c_first = -1, c_last = -1;
    double ms_emit = 0, ms_write = 0;
};
// The outputs of a plan, whose chars are BWT positions [off, off + P.chars), in windows of whole groups
// of at most cap chars, into the files F (DESIGN.md §6c, §6d).  The run samples are those of the piece
// on its own: the run start at its first char and the run end at its last char are always written.
int pb_write_windows(pfpb200_ctx *ctx, const PbInput &in, const PbWords &W, const PbPlan &P, u64 cap, PbOutFiles &F,
                     u64 off, PbPiece *pc);
// host bytes to [file_off, + bytes) of an open file
int pb_put_host(pfpb200_ctx *ctx, int fd, u64 file_off, const u8 *p, u64 bytes, const char *name);
// pfpb200_pfbwt_file from the inputs in HBM: the outputs to <base>.bwt [.sa | .ssa .esa], in windows when they
// do not fit the device memory left once the plan is done; records the plan for pfpb200_pfbwt_plan
int pb_to_files(pfpb200_ctx *ctx, const PbInput &in, const char *base, pfpb200_pfbwt_result *res);
// (BWT position + off, SA value) at the starts (at_end = 0) / ends of the runs of E's chars; prev / next:
// the chars on either side of them (-1: none); held: the output is recorded in ctx->pb_out[2 + at_end]
int pb_samples(pfpb200_ctx *ctx, const PbEmit &E, int at_end, int prev, int next, u64 off, bool held, u8 **out,
               u64 *n_out);

// the rank array of the sharded suffix sort, stored by position: block o = [o * per, (o + 1) * per)
// lives on rank o; kernels load and store it through the peers' block pointers
struct PmRanks {
    u64 *blk[PFPB200_MAX_RANKS];
    u64 per;
};

// one rank's state of a sharded pfbwt call (pfpb200_multi_pfbwt_file)
struct PmState {
    PbInput in;                                     // the whole dictionary and parse-side streams, on this rank
    PbWords wd;                                     // without wid: words come from the word ends
    // the owned first-key range and suffixes
    u64 rg_lo = 0, rg_hi = 0; int rg_has_lo = 0, rg_has_hi = 0;
    u64 M0 = 0, base = 0, M = 0, M2 = 0;
    int bn = 0, bm = 0, split = 0;                  // key layout: bits of N, bits of M0, two sorts
    u64 *pos = nullptr, *lo = nullptr; u32 *sl = nullptr, *we = nullptr, *hi = nullptr;   // per element (hi, lo: split key form)
    u64 *k0 = nullptr, *k1 = nullptr, *ks = nullptr, *ko = nullptr;
    u32 *v0 = nullptr, *v1 = nullptr, *vs = nullptr, *vo = nullptr;
    u32 *slot = nullptr, *slot2 = nullptr, *head = nullptr, *escan = nullptr, *rs = nullptr;
    u8 *flag = nullptr, *keep = nullptr;
    u64 *sa_pos = nullptr; u32 *sa_grp = nullptr, *sa_word = nullptr;   // per local slot
    // emission: the plan over the slice, then the piece in windows
    PbPlan plan;
    PbPiece piece;
};
int pm_sample(pfpb200_ctx *ctx, PmState &S, u64 lo, u64 hi, u32 want, u64 *h_out, u32 *got);
int pm_count(pfpb200_ctx *ctx, PmState &S, u64 klo, u64 khi, int has_lo, int has_hi, u64 *count);
int pm_collect(pfpb200_ctx *ctx, PmState &S, int split);
int pm_update(pfpb200_ctx *ctx, PmState &S, const PmRanks &R, u64 h, int first, u64 *active);
int pm_gather(pfpb200_ctx *ctx, PmState &S, const PmRanks &R, u64 h);
int pm_sort(pfpb200_ctx *ctx, PmState &S);
int pm_sort_done(pfpb200_ctx *ctx, PmState &S);
int pm_plan(pfpb200_ctx *ctx, PmState &S);
