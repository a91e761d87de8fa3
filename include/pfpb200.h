/* pfpb200.h -- C ABI of libpfpb200.so: B200-native prefix-free parsing (PFP).
 *
 * This library replaces ONE stage of alshai/Big-BWT: the scanner that `bigbwt` runs first
 * (reference newscan.cpp / newscan.hpp / pscan.cpp).  The reference has no library API for
 * that stage -- its interface is the newscan.x command line plus five output files
 * (bigbwt:71-86, utils.h:14-26) -- so the entry points below are what a C / ctypes / cgo
 * binding of that stage binds: one call per reference function group, plain pointers and
 * sizes only.  The bundled `gpuscan.x` is a newscan.x-compatible main() over
 * pfpb200_parse_file(); INTEGRATION.md shows the ctypes stub for `bigbwt`.
 *
 * All work runs in hand-written CUDA kernels for sm_100a.  There is NO CPU fallback:
 * every entry point returns PFPB200_E_CUDA when no device / kernel image is usable.
 */
#ifndef PFPB200_H
#define PFPB200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PFPB200_ABI_VERSION 2

/* ---- error codes (reference behaviour: message + exit(1), utils.c:12-16) ------------------ */
#define PFPB200_OK            0
#define PFPB200_E_ARG        -1  /* w < 4, p < 10 (newscan.cpp:537-544), null pointers, ...      */
#define PFPB200_E_IO         -2  /* cannot open / read / write a file (utils.c:33-41)            */
#define PFPB200_E_CUDA       -3  /* no usable GPU, kernel launch or runtime failure              */
#define PFPB200_E_NOMEM      -4  /* host or device allocation failed (newscan.cpp:603-606)       */
#define PFPB200_E_LIMIT      -5  /* > 2^31-2 distinct words, > 2^32-1 occurrences (newscan.cpp:114-117,
                                    613-617), a phrase > 2^32-1 bytes, or >= 2^31-2 phrases on ONE
                                    GPU (the reference allows 2^32-2 phrases, bigbwt:110-114; here
                                    bit 31 of the per-phrase word id marks ids still being created,
                                    so a text with more phrases needs two or more shards, or the
                                    chunks of a streamed pfpb200_parse_file, where the limit applies
                                    per chunk and the total may reach 2^32-2)                    */
#define PFPB200_E_COLLISION  -6  /* fingerprint collision detected (newscan.cpp:282-286)         */
#define PFPB200_E_INTERNAL   -7  /* an invariant of the pipeline was violated                    */

/* ---- options: the newscan.x command line (newscan.cpp:500-555) ---------------------------- */
#define PFPB200_F_SAI       1u   /* -s : also produce .sai (newscan.cpp:320-321)                 */
#define PFPB200_F_FASTA     2u   /* -f : input is FASTA/FASTQ, kseq semantics (newscan.cpp:332)  */
#define PFPB200_F_COMPRESS  4u   /* -c : write .dicz instead of .dict (newscan.cpp:410-413)      */
#define PFPB200_F_VERBOSE   8u   /* -v                                                           */
#define PFPB200_F_VERIFY   16u   /* compare every phrase byte for byte with the dictionary word it
                                    was given, as the reference does on every map hit
                                    (newscan.cpp:282-286): the parse is exact or fails with
                                    PFPB200_E_COLLISION, whatever the 128-bit fingerprints say      */

typedef struct pfpb200_opts {
    uint32_t w;       /* -w window size, >= 4, default 10 (newscan.cpp:155)                     */
    uint32_t p;       /* -p modulus,     >= 10, default 100 (newscan.cpp:156)                   */
    uint32_t flags;   /* PFPB200_F_*                                                             */
    int32_t  nseg;    /* -t : 0 = single .last/.sai files, T>0 = T segment files
                         <file>.<i>.last|sai as bwtparse -t T expects (newscan.hpp:274-276)     */
} pfpb200_opts;

/* ---- counters the reference prints (newscan.cpp:609-611,633-634) + device timings --------- */
typedef struct pfpb200_stats {
    uint64_t n_text;        /* "Total input symbols"                                            */
    uint64_t n_phrases;     /* "Total number of words"                                          */
    uint64_t n_distinct;    /* "Found .. distinct words"                                        */
    uint64_t sum_word_len;  /* "Sum of lenghts of dictionary words"                             */
    uint64_t dict_bytes;    /* size of .dict = sum_word_len + n_distinct + 1                    */
    uint64_t alg_bytes;     /* algorithmic bytes: text read once + every output written once    */
    uint32_t rank_rounds;   /* refinement rounds of the lexicographic ranking                   */
    uint32_t launches;      /* kernels launched by the last call                                */
    float ms_total;         /* CUDA-event time, text resident in HBM -> all outputs in HBM      */
    float ms_scan;          /* K1 trigger scan (KR_window::addchar + hash%p, newscan.cpp:194,344)*/
    float ms_emit;          /* K1 compaction of trigger positions                               */
    float ms_hash;          /* K2 phrase records + fingerprints (save_update_word :245-304)     */
    float ms_dedup;         /* K3 dictionary build (std::map update :256-288)                   */
    float ms_rank;          /* K4 lexicographic ranking (std::sort :636)                        */
    float ms_dict;          /* K4 epilogue: .dict/.occ bytes (writeDictOcc :394-441)            */
    float ms_remap;         /* K5 parse remap (remapParse :443-466)                             */
    float ms_h2d, ms_d2h;   /* host<->device copies (host entry points only)                    */
    float sec_read, sec_write; /* file I/O wall time (file entry point only)                    */
} pfpb200_stats;

/* The five output streams (utils.h:14-26).  Pointers are owned by the context and stay valid
 * until the next parse call on it, pfpb200_set_stream() or pfpb200_destroy().  `sai` is NULL without PFPB200_F_SAI. */
typedef struct pfpb200_outputs {
    const uint8_t  *dict;   uint64_t dict_bytes;   /* words + 0x01 each, final 0x00             */
    const uint32_t *occ;    uint64_t n_distinct;   /* u32 LE occurrences in rank order          */
    const uint32_t *parse;  uint64_t n_phrases;    /* u32 LE 1-based ranks in text order        */
    const uint8_t  *last;                          /* n_phrases bytes                           */
    const uint8_t  *sai;                           /* 5 * n_phrases bytes (IBYTES, utils.h:10)  */
} pfpb200_outputs;

typedef struct pfpb200_ctx pfpb200_ctx;

/* Create / destroy a context bound to one CUDA device.  The context owns a stream, the
 * device scratch and the output buffers.  Not thread-safe; one context per host thread. */
int  pfpb200_create(int device, pfpb200_ctx **ctx);
void pfpb200_destroy(pfpb200_ctx *ctx);
/* Run on a caller-owned cudaStream_t (e.g. a torch stream); NULL restores the own stream.
 * Synchronises the current stream and RELEASES the outputs of the previous parse: pointers
 * obtained before the call are invalid afterwards. */
int  pfpb200_set_stream(pfpb200_ctx *ctx, void *cuda_stream);

/* Replaces process_file() + sort + writeDictOcc() + remapParse() (newscan.cpp:310-466,
 * 581-646) for text already resident in HBM.  d_text: device pointer to n_text bytes, every
 * byte > 0x02.  Outputs are device pointers. */
int pfpb200_parse_device(pfpb200_ctx *ctx, const uint8_t *d_text, uint64_t n_text,
                         const pfpb200_opts *opts, pfpb200_outputs *dev_out,
                         pfpb200_stats *stats);

/* Copy `bytes` of a device-resident output to host memory (synchronous on the context's
 * stream); for callers of pfpb200_parse_device / pfpb200_scan_triggers without a CUDA runtime
 * of their own. */
int pfpb200_memcpy_d2h(pfpb200_ctx *ctx, void *dst_host, const void *src_device, uint64_t bytes);

/* Same for text in host memory (pageable or pinned): input is cut at the first byte <= 0x02
 * (newscan.cpp:364), copied to the device, parsed; outputs are host pointers (pinned memory
 * owned by the context). */
int pfpb200_parse_host(pfpb200_ctx *ctx, const uint8_t *text, uint64_t n_text,
                       const pfpb200_opts *opts, pfpb200_outputs *host_out,
                       pfpb200_stats *stats);

/* newscan.x main() (newscan.cpp:569-650): reads `path` (plain or FASTA per opts->flags),
 * parses on the GPU and writes <path>.dict|.dicz .occ .parse .last [.sai] (segmented
 * .last/.sai when opts->nseg > 0).  The file streams into HBM through a ring of pinned chunks
 * (reads, copies and the FASTA extraction on the device overlap; it is never held in host
 * memory, like the reference's byte-wise reader, newscan.cpp:332-374) and the outputs stream
 * back into the files the same way. */
int pfpb200_parse_file(pfpb200_ctx *ctx, const char *path, const pfpb200_opts *opts,
                       pfpb200_stats *stats);

/* How the last pfpb200_parse_file call ran.  An input whose one-shot footprint (about 1.5 to 4 device
 * bytes per input byte, DESIGN.md §6b) exceeds the device memory available to the call is parsed in
 * chunks instead: the text streams through HBM against one dictionary that lives across the chunks,
 * .parse is written as global word ids and rewritten with ranks at the end, like the reference's
 * .parse_old and remapParse (newscan.cpp:443-466).  The outputs are the same bytes; the text is then
 * bounded by the disk, the dictionary (as the reference's std::map by RAM) by one GPU.  The per-GPU
 * limit of 2^31-2 phrases applies per chunk, so a streamed parse reaches the reference's 2^32-2.
 * PFPB200_PARSE_BUDGET=<bytes> in the environment replaces the available-memory figure (routing and
 * chunk size: budget / 8 new bytes per chunk).  *chunks = 0 for the one-shot path; *peak_device_bytes
 * = the high-water mark of the context's device arena during the call. */
int pfpb200_parse_plan(const pfpb200_ctx *ctx, uint64_t *chunks, uint64_t *peak_device_bytes);

/* kseq-equivalent FASTA/FASTQ extraction + toupper + validity cut (kseq.h:177-218,
 * newscan.cpp:338-349), host side.  `out` must hold n bytes; returns text length and sets
 * *truncated when an invalid byte ended the input. */
uint64_t pfpb200_fasta_extract(const uint8_t *file, uint64_t n, uint8_t *out, int *truncated);

/* K0: the same extraction on the device, for FASTA bytes already in HBM (what pfpb200_parse_file
 * runs after streaming the file in).  *d_text is owned by the context (valid until its next
 * call).  *supported = 0: the bytes hold something beyond plain multi-line FASTA (FASTQ records,
 * '\r', bytes <= 0x02 or 0xFF, junk in front of the first '>') and need pfpb200_fasta_extract. */
int pfpb200_fasta_extract_device(pfpb200_ctx *ctx, const uint8_t *d_file, uint64_t n,
                                 const uint8_t **d_text, uint64_t *n_text, int *supported);

/* The text T that pfpb200_parse_file() parses for `path`, in host memory (release it with
 * pfpb200_free_host): the file bytes, or with PFPB200_F_FASTA the extraction above of a plain or
 * gzip-compressed FASTA/FASTQ file (the reference reads -f input through zlib's gzread,
 * newscan.cpp:332-336, kseq.h).  Host only, no GPU needed. */
int pfpb200_read_input(const char *path, uint32_t flags, uint8_t **text, uint64_t *n_text, int *truncated);
void pfpb200_free_host(void *p);

/* ---- stage-level entry points (device pointers) ------------------------------------------ *
 * The scan stage alone: KR_window::addchar + `hash % p == 0` over a shard of the text
 * (newscan.cpp:194-202,344,367; sharding as pscan.hpp:44-108).  d_buf holds n_buf text bytes
 * whose first byte is global position buf_pos0; trigger END positions e (global) with
 * own_lo <= e < own_hi and e >= w-1 are written ascending to a context-owned device array.
 * The caller must have w-1 bytes of left halo in the buffer (buf_pos0 <= own_lo-(w-1)) unless
 * own_lo == 0. */
int pfpb200_scan_triggers(pfpb200_ctx *ctx, const uint8_t *d_buf, uint64_t n_buf,
                          uint64_t buf_pos0, uint64_t own_lo, uint64_t own_hi,
                          uint32_t w, uint32_t p, const uint64_t **d_triggers,
                          uint64_t *n_triggers, float *ms);

/* ---- sharded parsing: the building blocks big-bwt_b200/shards.py drives, one process per GPU ---- *
 * Reference analogue: the per-thread input ranges of pscan.hpp:114-165 / newscan.hpp:230-337 and
 * the shared dictionary of pscan.cpp:137-205, with NCCL collectives between the calls.
 *   1. pfpb200_shard_scan   : triggers owned by this shard (needs w bytes of left halo in d_buf)
 *   2. (all-gather of last triggers -> first_start; fetch of the straddling phrase's head bytes)
 *   3. pfpb200_shard_words  : phrase records + this shard's local dictionary (words, counts, pool)
 *   4. (exchange of words)  -> pfpb200_dict_merge : global dedup + lexicographic ranks + .dict/.occ
 *   5. pfpb200_shard_remap  : .parse of the shard from the global rank of each local word        */
typedef struct pfpb200_shard {
    const uint8_t *d_buf;   /* device buffer: halo/head bytes followed by the shard              */
    uint64_t n_buf;         /* bytes in d_buf                                                     */
    uint64_t buf_pos0;      /* global text position of d_buf[0]                                   */
    uint64_t own_lo, own_hi;/* this shard owns the phrases whose END position e is in [lo, hi)    */
    uint64_t n_global;      /* length of the whole text                                           */
    uint32_t is_last;       /* 1: also emit the final phrase ending in the virtual 0x02^w         */
    uint32_t reserved;
} pfpb200_shard;

typedef struct pfpb200_words {      /* a shard's local dictionary, device pointers               */
    uint64_t n_words, n_phrases, pool_words;
    const uint64_t *fpa, *fpb;      /* 128-bit fingerprint of each word                          */
    const uint32_t *len, *count;    /* length in bytes, occurrences in this shard                */
    const uint32_t *uwords;         /* length in 8-byte pool words                               */
    const uint64_t *pool;           /* the words back to back, zero padded to 8 bytes            */
    const uint8_t *last, *sai;      /* this shard's .last / .sai streams                         */
} pfpb200_words;

typedef struct pfpb200_merged {
    uint64_t n_distinct, dict_bytes;
    uint64_t sum_word_len;
    const uint8_t *dict;            /* words in rank order + 0x01 each (+ final 0x00, counted)   */
    const uint32_t *occ;
    const uint32_t *rank_of_entry;  /* 1-based rank, inside this merge, of every input entry     */
} pfpb200_merged;

int pfpb200_shard_scan(pfpb200_ctx *ctx, const pfpb200_shard *shard, const pfpb200_opts *opts,
                       uint64_t *n_triggers, uint64_t *first_trigger, uint64_t *last_trigger,
                       float *ms);
/* first_start: global position of the first byte of the first phrase ending in this shard
 * (previous trigger - w + 1), or -1 when that phrase starts at the beginning of the text. */
int pfpb200_shard_words(pfpb200_ctx *ctx, int64_t first_start, pfpb200_words *out, float *ms);
int pfpb200_dict_merge(pfpb200_ctx *ctx, uint64_t n_in, const uint64_t *fpa, const uint64_t *fpb,
                       const uint32_t *len, const uint32_t *count, const uint32_t *uwords,
                       const uint64_t *pool, uint64_t pool_words, uint32_t w, uint32_t flags,
                       pfpb200_merged *out, float *ms);
int pfpb200_shard_remap(pfpb200_ctx *ctx, const uint32_t *d_rank_of_word, const uint32_t **d_parse,
                        float *ms);

/* ---- range-partitioned dictionary merge (mode "partition" of shards.py) -------------------- *
 * Words are routed to the rank that owns their lexicographic range, identified by the big-endian
 * first 8 bytes of the word; equal words have equal keys, so a single exchange serves the global
 * dedup and the global ranking (the reference's analogue: hash % (3*threads) map shards,
 * pscan.cpp:137-205 -- here the partition is by order, so ranks need no second exchange).     */
#define PFPB200_MAX_RANKS 64
/* Device array with the big-endian first 8 bytes (zero padded) of every word of the last
 * pfpb200_shard_words call; used to sample range splitters. */
int pfpb200_shard_first_keys(pfpb200_ctx *ctx, const uint64_t **d_keys);

/* The splitter sample directly: the keys of (up to) max_samples evenly spaced words of the last
 * pfpb200_shard_words call, in HOST memory (h_keys must hold max_samples values). */
int pfpb200_shard_sample_keys(pfpb200_ctx *ctx, uint32_t max_samples, uint64_t *h_keys, uint32_t *n_keys);

typedef struct pfpb200_word {       /* one dictionary word on the wire: 32 bytes                 */
    uint64_t fpa, fpb;              /* 128-bit fingerprint                                       */
    uint32_t len, count, uwords;    /* bytes, occurrences, 8-byte pool words                     */
    uint32_t pad;
} pfpb200_word;

typedef struct pfpb200_routed {     /* the local dictionary regrouped by destination rank        */
    const pfpb200_word *words;      /* n_words records, grouped by destination                   */
    const uint64_t *pool;           /* their bytes in the same order                             */
    const uint32_t *perm;           /* perm[i] = local word stored at routed position i          */
    uint64_t words_to[PFPB200_MAX_RANKS];   /* words / pool words going to each rank             */
    uint64_t pool_to[PFPB200_MAX_RANKS];
} pfpb200_routed;

/* Word u goes to rank  #{ s : splitters[s] <= key(u) }  (n_ranks-1 ascending host keys). */
int pfpb200_shard_route(pfpb200_ctx *ctx, const uint64_t *splitters, uint32_t n_ranks,
                        pfpb200_routed *out, float *ms);

/* The same routing fused with the exchange, for ranks that can store into each other's memory
 * (NVLink peer mappings, e.g. torch symmetric memory).  _plan decides the owner of every word and
 * returns how many words / pool words go to each owner (arrays of PFPB200_MAX_RANKS) and the
 * routed order d_perm; after the ranks have exchanged those counts, _push writes this rank's
 * pfpb200_word records for owner q to word_dst[q] and their pool words to pool_dst[q] -- device
 * addresses inside the owners' receive buffers, as mapped into THIS process -- in routed order.
 * The caller brackets the push with barriers among the ranks. */
int pfpb200_shard_route_plan(pfpb200_ctx *ctx, const uint64_t *splitters, uint32_t n_ranks,
                             uint64_t *words_to, uint64_t *pool_to, const uint32_t **d_perm, float *ms);
int pfpb200_shard_route_push(pfpb200_ctx *ctx, uint32_t n_ranks, const uint64_t *word_dst,
                             const uint64_t *pool_dst, float *ms);

/* pfpb200_dict_merge for words received as pfpb200_word records (the all-to-all payload). */
int pfpb200_dict_merge_words(pfpb200_ctx *ctx, uint64_t n_in, const pfpb200_word *words,
                             const uint64_t *pool, uint64_t pool_words, uint32_t w, uint32_t flags,
                             pfpb200_merged *out, float *ms);

/* Ranks travelling back in the range-partitioned merge: d_back[i] = rank, inside its owner's
 * range, of the word pfpb200_shard_route put at routed position i; rank_base[q] = number of
 * distinct words in the ranges below owner q.  *d_rank_of_word (context-owned) = global 1-based
 * rank of every local word, ready for pfpb200_shard_remap. */
int pfpb200_shard_ranks_back(pfpb200_ctx *ctx, uint32_t n_ranks, const uint32_t *d_back,
                             const uint64_t *rank_base, const uint32_t **d_rank_of_word);

/* ---- several GPUs of one box behind one call ------------------------------------------------ *
 * Reference analogue: `newscan.x -t T` / `pscan.x -t T` -- one process, T helper threads over
 * contiguous ranges of the input, complete outputs at return (newscan.hpp:230-337,
 * pscan.hpp:114-165, bigbwt:71-78).  One host thread per listed GPU drives the pfpb200_shard_*
 * stages; the dictionary words travel between the GPUs as peer-to-peer DMA over NVLink.  gpu_ids
 * NULL = devices 0..n_gpus-1; a device may be listed more than once (its shards time-share it).
 * Outputs: the five whole streams in pinned host memory owned by the handle (valid until the next
 * parse on it), byte-identical to the single-GPU entry points for every n_gpus. */
typedef struct pfpb200_multi pfpb200_multi;
int  pfpb200_multi_create(int n_gpus, const int *gpu_ids, pfpb200_multi **m);
void pfpb200_multi_destroy(pfpb200_multi *m);
int  pfpb200_multi_n_gpus(const pfpb200_multi *m);
int  pfpb200_multi_parse_host(pfpb200_multi *m, const uint8_t *text, uint64_t n_text,
                              const pfpb200_opts *opts, pfpb200_outputs *host_out, pfpb200_stats *stats);
/* newscan.x main() on several GPUs: reads `path`, writes the same files as pfpb200_parse_file. */
int  pfpb200_multi_parse_file(pfpb200_multi *m, const char *path, const pfpb200_opts *opts,
                              pfpb200_stats *stats);
const char *pfpb200_multi_last_error(const pfpb200_multi *m);
/* Per-rank timeline of the last parse: out[rank * PFPB200_N_PHASES + k] = milliseconds rank spent
 * in phase k (start, h2d, scan, seams, words, splitters, route, exchange, merge, ranks-back, remap,
 * d2h; a phase with a barrier includes waiting for the slowest rank).  Returns values written. */
#define PFPB200_N_PHASES 12
int  pfpb200_multi_phase_ms(const pfpb200_multi *m, float *out, int cap);

/* Self-check of a .dict byte stream in device memory: number of adjacent word pairs that are NOT
 * strictly increasing in unsigned-byte order (the std::sort(pstringCompare) order of
 * newscan.cpp:387-390,636; the reference asserts its invariants the same way).  d_seps: ascending
 * positions of the n_words 0x01 terminators. */
int pfpb200_check_dict_order(pfpb200_ctx *ctx, const uint8_t *d_dict, const uint64_t *d_seps,
                             uint64_t n_words, uint64_t *n_bad);

/* pfpb200_dict_merge_words in two halves, so that the exchange of the pool bytes overlaps the
 * dedup: _begin needs only the 32-byte word records (global dedup: table, counts); _finish, called
 * once the pool bytes have arrived, ranks the distinct words and writes .dict/.occ. */
int pfpb200_dict_merge_begin(pfpb200_ctx *ctx, uint64_t n_in, const pfpb200_word *words, float *ms);
int pfpb200_dict_merge_finish(pfpb200_ctx *ctx, const uint64_t *pool, uint64_t pool_words, uint32_t w,
                              uint32_t flags, pfpb200_merged *out, float *ms);

/* Kernels launched on this context since the start of the current parse (the last
 * pfpb200_parse_* / pfpb200_shard_scan call). */
uint32_t pfpb200_launch_count(const pfpb200_ctx *ctx);

/* ---- the stage after the parse: bwtparse (SURVEY.md 8(f) row 3) ---------------------------------- *
 * Replaces main() of bwtparse.c (:218-322): the suffix array of the parse T[0..n] (n symbols of
 * .parse + the end symbol 0, sacak_int(), bwtparse.c:162-174), its BWT, and from them
 *   .ilist  : for every parse symbol in alphabetical order (end symbol first) the BWT positions
 *             where it occurs -- (n+1) u32 (bwtparse.c:276-306)
 *   .bwlast : .last permuted by the suffix array -- n+1 bytes (:243-262)
 *   .bwsai  : .sai permuted the same way -- 5 (n+1) bytes, with -s (:247,:256,:266)
 * exactly as pfbwt*.x reads them.  Limits as the reference: 2 <= n <= 2^32-2 (bwtparse.c:101,241).
 * The result's device pointers are owned by the context and stay valid until its next
 * pfpb200_bwtparse_* or parse call; the outputs of a previous parse on the same context stay valid
 * across this call, so pfpb200_parse_device -> pfpb200_bwtparse_device chains without a copy. */
typedef struct pfpb200_bwtparse_result {
    const uint32_t *ilist;     /* [n_out] device                                                 */
    const uint8_t  *bwlast;    /* [n_out] device                                                 */
    const uint8_t  *bwsai;     /* [5 n_out] device, NULL without .sai input                      */
    uint64_t n_out;            /* n + 1: "ilist positions written"                               */
    uint64_t alphabet;         /* largest parse symbol + 1 (the k+1 of bwtparse.c:233)           */
    uint32_t rounds;           /* prefix-doubling rounds of the suffix sort                      */
    uint32_t launches;         /* kernels launched                                               */
    float ms_sa, ms_lists, ms_total;   /* CUDA-event times: suffix array; BWT + lists; both      */
} pfpb200_bwtparse_result;

int pfpb200_bwtparse_device(pfpb200_ctx *ctx, const uint32_t *d_parse, uint64_t n_phrases,
                            const uint8_t *d_last, const uint8_t *d_sai /* may be NULL */,
                            pfpb200_bwtparse_result *res);
/* host buffers in, host buffers out: ilist[n+1], bwlast[n+1], bwsai[5(n+1)] (NULL iff sai is NULL) */
int pfpb200_bwtparse_host(pfpb200_ctx *ctx, const uint32_t *parse, uint64_t n_phrases,
                          const uint8_t *last, const uint8_t *sai, uint32_t *ilist, uint8_t *bwlast,
                          uint8_t *bwsai, pfpb200_bwtparse_result *res);
/* `bwtparse <basename> [-s] [-t nseg]`: reads <basename>.parse, .last and (sa_info) .sai -- as nseg
 * segment files <basename>.<i>.last|sai when nseg > 0 (utils.c:57-110) -- and writes .ilist,
 * .bwlast and .bwsai (the device copies stay available through res, as above).  That is when the
 * in-HBM suffix sort fits the device memory available to the call (free memory plus what the
 * context's arena holds unused); a larger parse takes the bounded path: a few bytes per phrase stay
 * resident, the sort runs in windows of whole symbol ranges and groups of suffixes, and the outputs
 * are written to the files in windows.  res then carries counts, rounds and CUDA-event times with NULL
 * device pointers.  PFPB200_BWTPARSE_BUDGET=<bytes> in the environment replaces the available-memory
 * figure.  PFPB200_E_NOMEM when even the resident arrays and one window do not fit. */
int pfpb200_bwtparse_file(pfpb200_ctx *ctx, const char *basename, int sa_info, int nseg,
                          pfpb200_bwtparse_result *res);

/* ---- the inverse of the parse: unparse (SURVEY.md 8(f) row 4) ------------------------------------ *
 * Replaces main() of unparse.c (:76-137): the text is the concatenation, over the symbols of
 * .parse, of the words of .dicz (`newscan -c`, newscan.cpp:410-413: words without their last w
 * bytes, the first one without its leading 0x02).  strip_w = 0: d_dict holds .dicz bytes;
 * strip_w = w > 0: d_dict holds plain .dict bytes and the same bytes are skipped on the fly.
 * *d_text is owned by the context (valid until its next unparse or parse call); the outputs of a
 * previous parse on the same context stay valid, so parse -> unparse runs without a copy. */
int pfpb200_unparse_device(pfpb200_ctx *ctx, const uint8_t *d_dict, uint64_t dict_bytes, uint32_t strip_w,
                           const uint32_t *d_parse, uint64_t n_phrases, const uint8_t **d_text,
                           uint64_t *n_text, float *ms);
/* `unparse <basename> [-o outname]`: <basename>.dicz + <basename>.parse -> outname (NULL: <basename>.out) */
int pfpb200_unparse_file(pfpb200_ctx *ctx, const char *basename, const char *outname, uint64_t *n_words,
                         uint64_t *n_text, float *ms);

/* ---- the last stage: pfbwt (SURVEY.md 8(f) row 2) --------------------------------------------------- *
 * Replaces bwt() + main() of pfbwt.cpp (:109-242, :318-407): the BWT of the text -- n + 1 chars, the
 * EOF char is 0 -- from the dictionary (.dict), the occurrences (.occ) and the outputs of bwtparse
 * (.ilist, .bwlast, .bwsai); with PFPB200_PFBWT_SA the suffix array (`-S`: n values of 5 bytes,
 * SABYTES, utils.h:12), with _SSA / _ESA the (position, value) pairs at the starts / ends of the
 * BWT's runs (`-s` / `-e`, pfbwt.cpp:165-193).  Limits: dictionary < 4 GB (the reference's 32-bit
 * build stops at 2 GB, pfbwt.cpp:333), parse < 2^32-2 words (:372).  Device pointers of the result
 * are owned by the context until its next pfbwt or parse call; the outputs of earlier stages on the
 * same context stay valid, so parse -> bwtparse -> pfbwt chains in HBM. */
#define PFPB200_PFBWT_SA   1u   /* -S : full suffix array                                            */
#define PFPB200_PFBWT_SSA  2u   /* -s : sampled suffix array at the starts of the runs (.ssa)        */
#define PFPB200_PFBWT_ESA  4u   /* -e : ... at the ends of the runs (.esa)                           */
typedef struct pfpb200_pfbwt_result {
    const uint8_t *bwt;  uint64_t n_bwt;     /* n_bwt = text length + 1                              */
    const uint8_t *sa;   uint64_t n_sa;      /* 5-byte values, n_bwt - 1 of them (NULL without _SA)  */
    const uint8_t *ssa;  uint64_t n_ssa;     /* pairs of 5-byte values                               */
    const uint8_t *esa;  uint64_t n_esa;
    uint64_t dict_bytes, dict_words, parse_size;
    uint64_t easy, hard;                     /* BWT chars written directly / through the merge       */
    uint32_t rounds, launches;               /* prefix-doubling rounds of the dictionary suffix sort */
    float ms_sa, ms_fill, ms_total;          /* CUDA-event times: suffix sort; BWT/SA emission; both */
} pfpb200_pfbwt_result;

int pfpb200_pfbwt_device(pfpb200_ctx *ctx, const uint8_t *d_dict, uint64_t dict_bytes, const uint32_t *d_occ,
                         uint64_t n_words, const uint32_t *d_ilist, const uint8_t *d_bwlast,
                         const uint8_t *d_bwsai /* NULL without SA flags */, uint64_t parse_size /* n_phrases + 1 */,
                         uint32_t w, uint32_t flags, pfpb200_pfbwt_result *res);
/* `pfbwt.x -w W [-S | -s -e] <basename>`: reads .dict .occ .ilist .bwlast [.bwsai], writes .bwt [.sa | .ssa .esa].
 * Once the suffix sort and the plan of the output are done, the outputs are held in HBM and written
 * as a whole when they fit the device memory left to the call (free memory plus what the context's
 * arena holds unused); res then carries device pointers, as pfpb200_pfbwt_device's does.  Otherwise
 * they are produced in windows of whole groups of equal dictionary suffixes, each written to the files
 * at its offset, and res carries counts and times with NULL device pointers.  The peak then depends on
 * the dictionary, not on the text.  PFPB200_PFBWT_BUDGET=<bytes> in the environment replaces the
 * available-memory figure (windows of the most chars whose output fits it). */
int pfpb200_pfbwt_file(pfpb200_ctx *ctx, const char *basename, uint32_t w, uint32_t flags,
                       pfpb200_pfbwt_result *res);
/* How the last pfpb200_pfbwt_file / pfpb200_bigbwt_file call wrote its outputs: *windows (1: in one
 * piece from HBM) and *peak_device_bytes, the high-water mark of the context's device arena during the
 * pfbwt step.  NULL outputs are skipped; ctx NULL: PFPB200_E_ARG. */
int pfpb200_pfbwt_plan(const pfpb200_ctx *ctx, uint64_t *windows, uint64_t *peak_device_bytes);

/* ---- the last stage on several GPUs ---------------------------------------------------------------- *
 * pfbwt over the ranks of a pfpb200_multi handle, for dictionaries of 4 GB and more: the same files as
 * pfpb200_pfbwt_file, byte for byte, for every number of ranks.  Rank 0 reads the inputs and they
 * travel peer to peer, so every rank holds the dictionary and the parse-side streams; the dictionary
 * suffixes are partitioned by their first symbols, sorted by prefix doubling with the rank array
 * spread over the GPUs (direct peer loads and stores: two different devices in the list need peer
 * access).  No rank holds an array over the whole dictionary other than the dictionary itself: the words
 * of its own suffixes come from the word ends.  Every rank writes its contiguous piece of .bwt / .sa into
 * the files rank 0 created at their final sizes, in windows of whole groups of equal suffixes as
 * pfpb200_pfbwt_file does when its outputs do not fit: one window when the piece's output fits the rank's
 * budget, which is PFPB200_PFBWT_BUDGET=<bytes> per rank if set, else the free memory plus the rank's
 * unused arena for a rank alone on its device, and its share of the free memory for one of several ranks
 * listed on the same device.  The run samples of .ssa / .esa go to part files
 * <basename>.ssa.<g> / .esa.<g> first; once the ranks know each other's first and last chars, every rank
 * copies its part, less a record the run across a rank border makes redundant, into the final file at its
 * offset, and the part files are removed (on failure as well).  res: counts summed over the ranks, device
 * pointers NULL, times the maximum over the ranks; pfpb200_multi_pfbwt_windows gives the windows per rank.
 * Limits: fewer than 2^32 suffixes per rank and fewer than 2^32 occurrences in one group of equal suffixes
 * (PFPB200_E_LIMIT: list more GPUs), parse < 2^32-2 words; a group of equal suffixes is written in one
 * window, whatever the budget. */
int pfpb200_multi_pfbwt_file(pfpb200_multi *m, const char *basename, uint32_t w, uint32_t flags,
                             pfpb200_pfbwt_result *res);
typedef struct pfpb200_pfbwt_rank {
    uint64_t suffixes;                       /* dictionary suffixes this rank sorted (its slice)     */
    uint64_t chars;                          /* BWT chars (and SA values) it wrote                   */
    uint64_t hard;                           /* of those, through the merge of the .ilist cursors    */
    uint64_t peak_bytes;                     /* peak device memory of its context                    */
    float ms_read, ms_sort, ms_emit, ms_write;   /* wall clock: inputs, suffix sort, emission (plan and
                                                    windows), files (with the run samples' stitching) */
} pfpb200_pfbwt_rank;
/* per-rank figures of the last pfpb200_multi_pfbwt_file call: fills up to cap entries, returns how many */
int pfpb200_multi_pfbwt_ranks(const pfpb200_multi *m, pfpb200_pfbwt_rank *out, int cap);
/* output windows each rank of the last pfpb200_multi_pfbwt_file call wrote its piece in (0: the rank owned
 * no dictionary suffix): fills up to cap entries, returns how many; m or windows NULL: PFPB200_E_ARG */
int pfpb200_multi_pfbwt_windows(const pfpb200_multi *m, uint64_t *windows, int cap);

/* ---- the whole pipeline in one call --------------------------------------------------------------------- *
 * What `bigbwt <file> -w W -p P [-f] [-S | -s -e] [-k]` does with three processes and the files between
 * them (bigbwt:66-150): here the input streams into HBM, parse -> bwtparse -> pfbwt run there, and
 * <path>.bwt (and .sa / .ssa / .esa per pfbwt_flags) are written; keep_files != 0 (`-k`) also writes
 * the intermediate .dict .occ .parse .last .sai .ilist .bwlast .bwsai.  stats / bp may be NULL (bp's
 * device pointers stay valid until the next call).  A text that does not fit the device (the routing of
 * pfpb200_parse_file, PFPB200_PARSE_BUDGET) takes the files: the streamed parse writes them, bwtparse
 * reads them, pfbwt reads .dict / .occ, and without keep_files they are deleted at the end.  pfbwt
 * writes as pfpb200_pfbwt_file does, in windows when its outputs do not fit (res then carries no
 * device pointers).  pfpb200_parse_plan and pfpb200_pfbwt_plan report the two steps' plans. */
int pfpb200_bigbwt_file(pfpb200_ctx *ctx, const char *path, const pfpb200_opts *opts, uint32_t pfbwt_flags,
                        int keep_files, pfpb200_stats *stats, pfpb200_bwtparse_result *bp,
                        pfpb200_pfbwt_result *res);

/* How the last pfpb200_bwtparse_file / pfpb200_bigbwt_file call ran bwtparse: *windows (1: the in-HBM
 * path; otherwise the windows of the bounded path's first round) and *peak_device_bytes, the
 * high-water mark of the context's device arena during that step.  NULL outputs are skipped; ctx NULL:
 * PFPB200_E_ARG. */
int pfpb200_bwtparse_plan(const pfpb200_ctx *ctx, uint64_t *windows, uint64_t *peak_device_bytes);

const char *pfpb200_strerror(int code);
/* Message of the last failure on this context (CUDA error string, file name, ...). */
const char *pfpb200_last_error(const pfpb200_ctx *ctx);
int pfpb200_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* PFPB200_H */
