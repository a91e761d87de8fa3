/* gpuscan.c -- newscan.x-compatible command line over libpfpb200 (reference main():
 * newscan.cpp:569-650, options :489-556).  Install it (or symlinks to it) as newscan.x and
 * newscanNT.x next to the unchanged `bigbwt` script, which picks its scanner by path
 * (bigbwt:22-24,71-78) and only looks at the exit status (bigbwt:231-240). */
#define _GNU_SOURCE
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>
#include "../../include/pfpb200.h"

static void usage(const char *exe, const pfpb200_opts *o) {
    printf("Usage: %s <input filename> [options]\n", exe);
    printf("  Options: \n");
    printf("\t-w W\tsliding window size, def. %u\n", o->w);
    printf("\t-p M\tmodulo for defining phrases, def. %u\n", o->p);
    printf("\t-t M\tnumber of .last/.sai segments to write (helper threads of the reference), def. none \n");
    printf("\t-g G\tCUDA device index, or a comma-separated list (e.g. 0,1,2,3): the text is\n"
           "\t    \tsharded over the listed GPUs, def. 0\n");
    printf("\t-h  \tshow help and exit\n");
    printf("\t-s  \tcompute suffix array info\n");
    printf("\t-f  \tread a FASTA/FASTQ file\n");
    printf("\t-P  \taccepted for compatibility (collisions are always detected)\n");
    printf("\t-V  \tverify: compare every phrase with its dictionary word byte for byte\n");
    printf("\t-c  \tcompress the output dictionary\n");
    exit(1);
}

/* the reference reads -w/-p/-t with atoi into ints and rejects what is out of range
 * (newscan.cpp:537-548): parse signed, check, then cast */
static long int_arg(const char *s) {
    char *end = NULL;
    long v = strtol(s, &end, 10);
    if (end == s) return 0;            /* atoi semantics: no digits -> 0, rejected by the range checks */
    return v;
}

int main(int argc, char **argv) {
    pfpb200_opts o = {10, 100, 0, 0};
    int devices[PFPB200_MAX_RANKS] = {0}, n_dev = 1, verbose = 0, c;
    long w = 10, p = 100, nseg = 0;
    puts("==== Command line:");
    for (int i = 0; i < argc; i++) printf(" %s", argv[i]);
    puts("");
    while ((c = getopt(argc, argv, "p:w:fsPcht:vg:V")) != -1) {
        switch (c) {
            case 's': o.flags |= PFPB200_F_SAI; break;
            case 'P': break;
            case 'c': o.flags |= PFPB200_F_COMPRESS; break;
            case 'w': w = int_arg(optarg); break;
            case 'p': p = int_arg(optarg); break;
            case 'V': o.flags |= PFPB200_F_VERIFY; break;
            case 'f': o.flags |= PFPB200_F_FASTA; break;
            case 't': nseg = int_arg(optarg); break;
            case 'g': {
                n_dev = 0;
                for (char *tok = strtok(optarg, ","); tok && n_dev < PFPB200_MAX_RANKS; tok = strtok(NULL, ","))
                    devices[n_dev++] = (int)int_arg(tok);
                if (n_dev == 0) { puts("Invalid device list"); exit(1); }
                break;
            }
            case 'v': verbose++; o.flags |= PFPB200_F_VERBOSE; break;
            case 'h': usage(argv[0], &o); break;
            default: puts("Unknown option. Use -h for help."); exit(1);
        }
    }
    if (argc != optind + 1) { puts("Invalid number of arguments"); usage(argv[0], &o); }
    const char *path = argv[optind];
    if (w < 4) { puts("Windows size must be at least 4"); exit(1); }
    if (p < 10) { puts("Modulus must be at least 10"); exit(1); }
    if (nseg < 0) { puts("Number of threads cannot be negative"); exit(1); }
    if (w > 65536 || p > 0x7FFFFFFFL || nseg > 4096) { puts("Option value too large"); exit(1); }
    o.w = (uint32_t)w; o.p = (uint32_t)p; o.nseg = (int32_t)nseg;
    printf("Windows size: %u\n", o.w);
    printf("Stop word modulus: %u\n", o.p);
    time_t start = time(NULL);
    pfpb200_ctx *ctx = NULL;
    pfpb200_multi *multi = NULL;
    pfpb200_stats st;
    int rc;
    if (n_dev > 1) {           /* one host thread per GPU, complete files at exit (newscan -t T) */
        rc = pfpb200_multi_create(n_dev, devices, &multi);
        if (rc != PFPB200_OK) {
            fprintf(stderr, "gpuscan: cannot use the %d listed CUDA devices: %s\n", n_dev, pfpb200_strerror(rc));
            return 1;
        }
        rc = pfpb200_multi_parse_file(multi, path, &o, &st);
        if (rc != PFPB200_OK) {
            fprintf(stderr, "gpuscan: %s: %s\n", pfpb200_strerror(rc), pfpb200_multi_last_error(multi));
            pfpb200_multi_destroy(multi);
            return 1;
        }
    } else {
        rc = pfpb200_create(devices[0], &ctx);
        if (rc != PFPB200_OK) {
            fprintf(stderr, "gpuscan: cannot use CUDA device %d: %s\n", devices[0], pfpb200_strerror(rc));
            return 1;
        }
        rc = pfpb200_parse_file(ctx, path, &o, &st);
        if (rc != PFPB200_OK) {
            fprintf(stderr, "gpuscan: %s: %s\n", pfpb200_strerror(rc), pfpb200_last_error(ctx));
            pfpb200_destroy(ctx);
            return 1;
        }
    }
    printf("Total input symbols: %llu\n", (unsigned long long)st.n_text);
    printf("Found %llu distinct words\n", (unsigned long long)st.n_distinct);
    printf("Sum of lenghts of dictionary words: %llu\n", (unsigned long long)st.sum_word_len);
    printf("Total number of words: %llu\n", (unsigned long long)st.n_phrases);
    printf("GPU parse: %.3f ms (scan %.3f, emit %.3f, hash %.3f, dict %.3f, rank %.3f [%u rounds], "
           "write-dict %.3f, remap %.3f), h2d %.3f ms, d2h %.3f ms, %u kernel launches\n",
           st.ms_total, st.ms_scan, st.ms_emit, st.ms_hash, st.ms_dedup, st.ms_rank, st.rank_rounds,
           st.ms_dict, st.ms_remap, st.ms_h2d, st.ms_d2h, st.launches);
    printf("File read: %.3f s, file write: %.3f s\n", st.sec_read, st.sec_write);
    if (ctx && verbose) {
        uint64_t chunks = 0, peak = 0;
        pfpb200_parse_plan(ctx, &chunks, &peak);
        if (chunks) printf("Parse plan: streamed in %llu chunks, device peak %llu bytes\n",
                           (unsigned long long)chunks, (unsigned long long)peak);
        else printf("Parse plan: one-shot, device peak %llu bytes\n", (unsigned long long)peak);
    }
    if (multi && verbose) {
        static const char *names[PFPB200_N_PHASES] = {"start", "h2d", "scan", "seams", "words", "splitters", "route",
                                                      "exchange", "merge", "ranks-back", "remap", "d2h"};
        float ms[PFPB200_MAX_RANKS * PFPB200_N_PHASES];
        int k = pfpb200_multi_phase_ms(multi, ms, PFPB200_MAX_RANKS * PFPB200_N_PHASES);
        for (int r = 0; r * PFPB200_N_PHASES < k; r++) {
            printf("GPU %d:", devices[r]);
            for (int ph = 1; ph < PFPB200_N_PHASES; ph++) printf(" %s %.3f", names[ph], ms[r * PFPB200_N_PHASES + ph]);
            printf(" ms\n");
        }
    }
    printf("==== Elapsed time: %.0f wall clock seconds\n", difftime(time(NULL), start));
    pfpb200_destroy(ctx);
    pfpb200_multi_destroy(multi);
    (void)verbose;
    return 0;
}
