/* gpubwtparse.c -- bwtparse-compatible command line over libpfpb200 (reference main():
 * bwtparse.c:218-322, options :131-160).  Install it as bwtparse (and bwtparse64) next to the
 * unchanged `bigbwt` script, which runs `bwtparse <file> [-s] [-t T]` and only looks at the exit
 * status (bigbwt:106-128,231-240). */
#define _GNU_SOURCE
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <unistd.h>
#include "../../include/pfpb200.h"

static void print_help(const char *name) {
    printf("Usage: %s <basename> [options]\n\n", name);
    puts("Compute the BWT of basename.parse and store its inverted list occurrence");
    puts("Permute the file basename.last according to the same permutation");
    puts("  Options:");
    puts("\t-h  \tshow help and exit");
    puts("\t-s  \tpermute also sa info");
    puts("\t-t M\tthe .last/.sai files are in M segments");
    puts("\t-g G\tCUDA device index, def. 0");
    exit(1);
}

int main(int argc, char **argv) {
    int c, sa_info = 0, nseg = 0, device = 0;
    puts("==== Command line:");
    for (int i = 0; i < argc; i++) printf(" %s", argv[i]);
    puts("\n");
    while ((c = getopt(argc, argv, "sht:g:")) != -1) {
        switch (c) {
            case 's': sa_info = 1; break;
            case 'h': print_help(argv[0]); break;
            case 't': nseg = atoi(optarg); break;
            case 'g': device = atoi(optarg); break;
            default: puts("Unknown option. Use -h for help."); exit(1);
        }
    }
    if (argc != optind + 1) print_help(argv[0]);
    if (nseg < 0) { puts("Number of segments cannot be negative"); exit(1); }
    const char *base = argv[optind];
    time_t start = time(NULL);
    pfpb200_ctx *ctx = NULL;
    int rc = pfpb200_create(device, &ctx);
    if (rc != PFPB200_OK) {
        fprintf(stderr, "gpubwtparse: cannot use CUDA device %d: %s\n", device, pfpb200_strerror(rc));
        return 1;
    }
    pfpb200_bwtparse_result r;
    rc = pfpb200_bwtparse_file(ctx, base, sa_info, nseg, &r);
    if (rc != PFPB200_OK) {
        fprintf(stderr, "gpubwtparse: %s: %s\n", pfpb200_strerror(rc), pfpb200_last_error(ctx));
        pfpb200_destroy(ctx);
        return 1;
    }
    printf("Parse file contains %llu words\n", (unsigned long long)(r.n_out - 1));
    printf("Computing SA of size %llu over an alphabet of size %llu\n", (unsigned long long)r.n_out,
           (unsigned long long)r.alphabet);
    printf("SA computed with depth: %u\n", r.rounds);
    printf("---- %llu bwlast chars written ----\n", (unsigned long long)r.n_out);
    puts("---- computing inverted list ----");
    printf("---- %llu ilist positions written (%llu bytes) ----\n", (unsigned long long)r.n_out,
           (unsigned long long)r.n_out * 4ull);
    printf("GPU bwtparse: %.3f ms (suffix array %.3f in %u doubling rounds, BWT + lists %.3f), %u kernel launches\n",
           r.ms_total, r.ms_sa, r.rounds, r.ms_lists, r.launches);
    uint64_t windows = 0, peak = 0;
    pfpb200_bwtparse_plan(ctx, &windows, &peak);
    printf("Plan: bwtparse %llu windows, peak %.3f GB\n", (unsigned long long)windows, (double)peak * 1e-9);
    printf("==== Elapsed time: %.0f wall clock seconds\n", difftime(time(NULL), start));
    pfpb200_destroy(ctx);
    return 0;
}
