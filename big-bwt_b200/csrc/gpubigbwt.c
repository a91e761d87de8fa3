/* gpubigbwt.c -- the `bigbwt` driver (bigbwt:35-150) as ONE process on the GPU: the input file streams
 * into HBM, the parse, the BWT of the parse and the final BWT are computed there
 * (pfpb200_bigbwt_file), and only <file>.bwt (and .sa / .ssa / .esa) are written -- the reference
 * runs newscan, bwtparse and pfbwt as three processes that hand each other files.  Options as
 * bigbwt's: -w -p -f -s -e -S -k; ours: -g (CUDA device). */
#define _GNU_SOURCE
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>
#include "../../include/pfpb200.h"

static void usage(const char *exe) {
    printf("Usage: %s <input filename> [options]\n", exe);
    printf("  Options: \n");
    printf("\t-w W\tsliding window size, def. 10\n");
    printf("\t-p M\thash modulus, def. 100\n");
    printf("\t-f  \tread fasta\n");
    printf("\t-s  \tcompute the start of run-length encoded BWT intervals of the sampled SA (.ssa)\n");
    printf("\t-e  \tcompute the end of run-length encoded BWT intervals of the sampled SA (.esa)\n");
    printf("\t-S  \tcompute the full suffix array (.sa)\n");
    printf("\t-k  \tkeep the intermediate files of the three stages\n");
    printf("\t-t T\taccepted for compatibility (helper threads of the reference's stages)\n");
    printf("\t-g G\tCUDA device index, def. 0, or a comma-separated list (e.g. 0,1,2,3): parse and pfbwt\n"
           "\t    \tsharded over those GPUs, bwtparse on the first, through files\n");
    exit(1);
}

static double since(const struct timespec *t0) {
    struct timespec t1;
    clock_gettime(CLOCK_MONOTONIC, &t1);
    return (double)(t1.tv_sec - t0->tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0->tv_nsec);
}

/* the three stages through files, as bigbwt runs them: newscan -> bwtparse -> pfbwt; the parse and
 * pfbwt on all listed GPUs, bwtparse (about a tenth of the parse's size) on the first one */
static int multi_bigbwt(const char *path, const pfpb200_opts *opts, unsigned flags, int keep, const int *devices,
                        int n_dev, const struct timespec *t0) {
    static const char *inter[] = {"dict", "occ", "parse", "last", "sai", "ilist", "bwlast", "bwsai"};
    pfpb200_opts o = *opts;
    o.flags |= PFPB200_F_SAI;                     /* the later stages take .sai whenever a suffix array is wanted */
    pfpb200_multi *multi = NULL;
    pfpb200_ctx *ctx = NULL;
    pfpb200_stats st;
    pfpb200_bwtparse_result bp;
    pfpb200_pfbwt_result r;
    int rc = pfpb200_multi_create(n_dev, devices, &multi);
    if (rc != PFPB200_OK) {
        fprintf(stderr, "gpubigbwt: cannot use the %d listed CUDA devices: %s\n", n_dev, pfpb200_strerror(rc));
        return 1;
    }
    const char *stage = "parse";
    rc = pfpb200_multi_parse_file(multi, path, &o, &st);
    if (rc == PFPB200_OK) {
        stage = "bwtparse";
        rc = pfpb200_create(devices[0], &ctx);
        if (rc == PFPB200_OK) rc = pfpb200_bwtparse_file(ctx, path, 1, 0, &bp);
        if (rc == PFPB200_OK) {
            pfpb200_destroy(ctx);                 /* its HBM goes back before the last stage */
            ctx = NULL;
            stage = "pfbwt";
            rc = pfpb200_multi_pfbwt_file(multi, path, o.w, flags, &r);
        }
    }
    if (rc != PFPB200_OK) {
        fprintf(stderr, "gpubigbwt: %s: %s: %s\n", stage, pfpb200_strerror(rc),
                ctx ? pfpb200_last_error(ctx) : pfpb200_multi_last_error(multi));
    } else {
        printf("Total input symbols: %llu\n", (unsigned long long)st.n_text);
        printf("Found %llu distinct words\n", (unsigned long long)st.n_distinct);
        printf("Total number of words: %llu\n", (unsigned long long)st.n_phrases);
        printf("Easy bwt chars: %llu\n", (unsigned long long)r.easy);
        printf("Hard bwt chars: %llu\n", (unsigned long long)r.hard);
        printf("GPU: parse %.3f ms, bwtparse %.3f ms (%u rounds), pfbwt %.3f ms (suffix sort %.3f in %u rounds, BWT%s %.3f)\n",
               st.ms_total, bp.ms_total, bp.rounds, r.ms_total, r.ms_sa, r.rounds, flags ? " + SA" : "", r.ms_fill);
        pfpb200_pfbwt_rank pr[PFPB200_MAX_RANKS];
        int k = pfpb200_multi_pfbwt_ranks(multi, pr, PFPB200_MAX_RANKS);
        for (int g = 0; g < k; g++)
            printf("GPU %d (rank %d): pfbwt %llu suffixes, %llu chars, sort %.3f ms, emit %.3f ms, write %.3f ms\n",
                   devices[g], g, (unsigned long long)pr[g].suffixes, (unsigned long long)pr[g].chars, pr[g].ms_sort,
                   pr[g].ms_emit, pr[g].ms_write);
    }
    if (!keep) {
        char name[4096];
        for (size_t i = 0; i < sizeof(inter) / sizeof(inter[0]); i++) {
            snprintf(name, sizeof(name), "%s.%s", path, inter[i]);
            unlink(name);
        }
    }
    pfpb200_destroy(ctx);
    pfpb200_multi_destroy(multi);
    if (rc != PFPB200_OK) return 1;
    printf("==== Elapsed time: %.3f wall clock seconds\n", since(t0));
    return 0;
}

int main(int argc, char **argv) {
    pfpb200_opts o = {10, 100, 0, 0};
    long w = 10, p = 100;
    int c, keep = 0, devices[PFPB200_MAX_RANKS] = {0}, n_dev = 1;
    unsigned flags = 0;
    struct timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    puts("==== Command line:");
    for (int i = 0; i < argc; i++) printf(" %s", argv[i]);
    puts("");
    while ((c = getopt(argc, argv, "w:p:fseSkhg:t:v")) != -1) {
        switch (c) {
            case 'w': w = strtol(optarg, NULL, 10); break;
            case 'p': p = strtol(optarg, NULL, 10); break;
            case 'f': o.flags |= PFPB200_F_FASTA; break;
            case 's': flags |= PFPB200_PFBWT_SSA; break;
            case 'e': flags |= PFPB200_PFBWT_ESA; break;
            case 'S': flags |= PFPB200_PFBWT_SA; break;
            case 'k': keep = 1; break;
            case 't': break;                       /* bigbwt -t T: helper threads of the CPU stages, nothing to do here */
            case 'v': break;
            case 'g': {
                n_dev = 0;
                for (char *tok = strtok(optarg, ","); tok && n_dev < PFPB200_MAX_RANKS; tok = strtok(NULL, ","))
                    devices[n_dev++] = atoi(tok);
                if (n_dev == 0) { puts("Invalid device list"); exit(1); }
                break;
            }
            case 'h': usage(argv[0]); break;
            default: puts("Unknown option. Use -h for help."); exit(1);
        }
    }
    if (argc != optind + 1) { puts("Invalid number of arguments"); usage(argv[0]); }
    if (w < 4) { puts("Windows size must be at least 4"); exit(1); }
    if (p < 10) { puts("Modulus must be at least 10"); exit(1); }
    if ((flags & PFPB200_PFBWT_SA) && (flags & (PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA))) {
        puts("You can either compute the full SA or a sample of it, not both. Exiting...");      /* bigbwt:59-61 */
        exit(1);
    }
    if (w > 65536 || p > 0x7FFFFFFFL) { puts("Option value too large"); exit(1); }
    o.w = (uint32_t)w; o.p = (uint32_t)p;
    if (n_dev > 1) return multi_bigbwt(argv[optind], &o, flags, keep, devices, n_dev, &t0);
    pfpb200_ctx *ctx = NULL;
    int rc = pfpb200_create(devices[0], &ctx);
    if (rc != PFPB200_OK) {
        fprintf(stderr, "gpubigbwt: cannot use CUDA device %d: %s\n", devices[0], pfpb200_strerror(rc));
        return 1;
    }
    pfpb200_stats st;
    pfpb200_bwtparse_result bp;
    pfpb200_pfbwt_result r;
    rc = pfpb200_bigbwt_file(ctx, argv[optind], &o, flags, keep, &st, &bp, &r);
    if (rc != PFPB200_OK) {
        fprintf(stderr, "gpubigbwt: %s: %s\n", pfpb200_strerror(rc), pfpb200_last_error(ctx));
        pfpb200_destroy(ctx);
        return 1;
    }
    clock_gettime(CLOCK_MONOTONIC, &t1);
    printf("Total input symbols: %llu\n", (unsigned long long)st.n_text);
    printf("Found %llu distinct words\n", (unsigned long long)st.n_distinct);
    printf("Total number of words: %llu\n", (unsigned long long)st.n_phrases);
    printf("Easy bwt chars: %llu\n", (unsigned long long)r.easy);
    printf("Hard bwt chars: %llu\n", (unsigned long long)r.hard);
    printf("GPU: parse %.3f ms, bwtparse %.3f ms (%u rounds), pfbwt %.3f ms (suffix sort %.3f in %u rounds, BWT%s %.3f)\n",
           st.ms_total, bp.ms_total, bp.rounds, r.ms_total, r.ms_sa, r.rounds, flags ? " + SA" : "", r.ms_fill);
    printf("File read: %.3f s; stages after the parse + file write: %.3f s\n", st.sec_read, st.sec_write);
    printf("==== Elapsed time: %.3f wall clock seconds\n",
           (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec));
    pfpb200_destroy(ctx);
    return 0;
}
