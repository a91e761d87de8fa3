/* gpupfbwt.c -- pfbwt.x-compatible command line over libpfpb200 (reference main(): pfbwt.cpp:318-407,
 * options :257-315).  Install it as pfbwt.x / pfbwtNT.x (/ pfbwt64.x / pfbwtNT64.x) next to the
 * unchanged `bigbwt` script, which runs `pfbwt*.x -w W [-s] [-e] [-S] [-t T] <file>` and only looks
 * at the exit status (bigbwt:130-150,231-240). */
#define _GNU_SOURCE
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>
#include "../../include/pfpb200.h"

static void print_help(const char *name, int w) {
    printf("Usage: %s <input filename> [options]\n", name);
    printf("  Options: \n");
    printf("\t-w W\tsliding window size, def. %d\n", w);
    printf("\t-t M\taccepted for compatibility (helper threads of the reference)\n");
    printf("\t-g G\tCUDA device index, def. 0, or a comma-separated list (e.g. 0,1,2,3): the stage is\n"
           "\t    \tsharded over those GPUs, each writing its piece of the outputs\n");
    printf("\t-h  \tshow help and exit\n");
    printf("\t-s  \tcompute sampled suffix array\n");
    printf("\t-e  \tcompute sampled suffix array at the ends of the runs\n");
    printf("\t-S  \tcompute full suffix array\n");
    exit(1);
}

int main(int argc, char **argv) {
    int c, w = 10, th = 0, devices[PFPB200_MAX_RANKS] = {0}, n_dev = 1;
    unsigned flags = 0;
    time_t start = time(NULL);
    puts("==== Command line:");
    for (int i = 0; i < argc; i++) printf(" %s", argv[i]);
    puts("");
    while ((c = getopt(argc, argv, "t:w:sehSg:")) != -1) {
        switch (c) {
            case 's': flags |= PFPB200_PFBWT_SSA; break;
            case 'e': flags |= PFPB200_PFBWT_ESA; break;
            case 'S': flags |= PFPB200_PFBWT_SA; break;
            case 'w': w = atoi(optarg); break;
            case 't': th = atoi(optarg); break;
            case 'g': {
                n_dev = 0;
                for (char *tok = strtok(optarg, ","); tok && n_dev < PFPB200_MAX_RANKS; tok = strtok(NULL, ","))
                    devices[n_dev++] = atoi(tok);
                if (n_dev == 0) { puts("Invalid device list"); exit(1); }
                break;
            }
            case 'h': print_help(argv[0], w); break;
            default: puts("Unknown option. Use -h for help."); exit(1);
        }
    }
    if (argc != optind + 1) { puts("Invalid number of arguments"); print_help(argv[0], w); }
    if ((flags & PFPB200_PFBWT_SA) && (flags & (PFPB200_PFBWT_SSA | PFPB200_PFBWT_ESA))) {
        printf("You can either require the sampled SA or the full SA, not both");
        exit(1);
    }
    if (w < 4) { puts("Windows size must be at least 4"); exit(1); }
    if (th < 0) { puts("Number of threads cannot be negative"); exit(1); }
    pfpb200_ctx *ctx = NULL;
    pfpb200_multi *multi = NULL;
    pfpb200_pfbwt_result r;
    int rc;
    if (n_dev > 1) {           /* one host thread per GPU, every rank writes its piece of the files */
        rc = pfpb200_multi_create(n_dev, devices, &multi);
        if (rc != PFPB200_OK) {
            fprintf(stderr, "gpupfbwt: cannot use the %d listed CUDA devices: %s\n", n_dev, pfpb200_strerror(rc));
            return 1;
        }
        rc = pfpb200_multi_pfbwt_file(multi, argv[optind], (uint32_t)w, flags, &r);
        if (rc != PFPB200_OK) {
            fprintf(stderr, "gpupfbwt: %s: %s\n", pfpb200_strerror(rc), pfpb200_multi_last_error(multi));
            pfpb200_multi_destroy(multi);
            return 1;
        }
    } else {
        rc = pfpb200_create(devices[0], &ctx);
        if (rc != PFPB200_OK) {
            fprintf(stderr, "gpupfbwt: cannot use CUDA device %d: %s\n", devices[0], pfpb200_strerror(rc));
            return 1;
        }
        rc = pfpb200_pfbwt_file(ctx, argv[optind], (uint32_t)w, flags, &r);
        if (rc != PFPB200_OK) {
            fprintf(stderr, "gpupfbwt: %s: %s\n", pfpb200_strerror(rc), pfpb200_last_error(ctx));
            pfpb200_destroy(ctx);
            return 1;
        }
    }
    printf("Dictionary file size: %llu\n", (unsigned long long)r.dict_bytes);
    printf("Dictionary words: %llu\n", (unsigned long long)r.dict_words);
    printf("Parsing size: %llu\n", (unsigned long long)r.parse_size);
    printf("bwlast file size: %llu\n", (unsigned long long)r.parse_size);
    printf("Full words: %llu\n", (unsigned long long)r.dict_words);
    printf("Easy bwt chars: %llu\n", (unsigned long long)r.easy);
    printf("Hard bwt chars: %llu\n", (unsigned long long)r.hard);
    printf("GPU pfbwt: %.3f ms (dictionary suffix sort %.3f in %u doubling rounds, BWT%s %.3f), %u kernel launches\n",
           r.ms_total, r.ms_sa, r.rounds, flags ? " + SA" : "", r.ms_fill, r.launches);
    if (ctx) {
        uint64_t windows = 0, peak = 0;
        pfpb200_pfbwt_plan(ctx, &windows, &peak);
        printf("Plan: %llu output windows (1: in one piece), device peak %.3f GB\n", (unsigned long long)windows,
               (double)peak * 1e-9);
    }
    if (multi) {
        pfpb200_pfbwt_rank pr[PFPB200_MAX_RANKS];
        int k = pfpb200_multi_pfbwt_ranks(multi, pr, PFPB200_MAX_RANKS);
        for (int g = 0; g < k; g++)
            printf("GPU %d (rank %d): %llu suffixes, %llu chars (%llu hard), read %.3f ms, sort %.3f ms, emit %.3f ms, "
                   "write %.3f ms, peak %.3f GB\n", devices[g], g, (unsigned long long)pr[g].suffixes,
                   (unsigned long long)pr[g].chars, (unsigned long long)pr[g].hard, pr[g].ms_read, pr[g].ms_sort,
                   pr[g].ms_emit, pr[g].ms_write, (double)pr[g].peak_bytes * 1e-9);
        uint64_t wn[PFPB200_MAX_RANKS];
        k = pfpb200_multi_pfbwt_windows(multi, wn, PFPB200_MAX_RANKS);
        printf("Plan: output windows per rank:");
        for (int g = 0; g < k; g++) printf("%s%llu", g ? "," : " ", (unsigned long long)wn[g]);
        printf("\n");
    }
    printf("==== Elapsed time: %.0f wall clock seconds\n", difftime(time(NULL), start));
    pfpb200_destroy(ctx);
    pfpb200_multi_destroy(multi);
    return 0;
}
