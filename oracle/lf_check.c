/* lf_check.c -- TEST INFRASTRUCTURE ONLY: a linear check of bwtparse's outputs (.ilist, .bwlast,
 * .bwsai) against its inputs (.parse, .last, .sai), for parses too large for the oracle's suffix sort.
 *
 * T = the n parse symbols + the end symbol 0; its suffix array has N = n + 1 rows.  The check:
 *   1. .ilist is a permutation of [0, N) that ascends inside each F-range, where F[0] = 0 and
 *      F[c] = 1 + (occurrences of the symbols below c) (bwtparse.c:294-298).  Row k of the sorted first
 *      column then holds symbol c for k in [F[c], F[c + 1]), and the BWT char at position ilist[k] is c;
 *   2. LF(ilist[k]) = k.  Walking LF from row 0 (the end suffix n) must meet T[n-1], T[n-2], ..., T[0]
 *      in the BWT and reach the suffix 0 at row 1 after n steps, visiting every row once: then the BWT
 *      implied by .ilist is the BWT of T, and the walk knows the suffix-array value s of every row;
 *   3. at every row, bwlast = last[s - 2] (last[n - 1] for s = 1, 0 for s = 0) and bwsai = sai[s - 1]
 *      (0 for s = 0), as bwtparse.c:243-272 writes them.
 * Linear time; memory: 8 bytes per row and 8 per symbol beside the inputs. */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define IBYTES 5

int lf_check(const uint32_t *T, uint64_t n, const uint8_t *last, const uint8_t *sai, const uint32_t *ilist,
             const uint8_t *bwlast, const uint8_t *bwsai, uint64_t rows, char *msg, int msglen) {
    const uint64_t N = n + 1;
    msg[0] = 0;
    if (rows != N) { snprintf(msg, msglen, "%llu rows, %llu expected", (unsigned long long)rows, (unsigned long long)N); return 1; }
    uint32_t kmax = 0;
    for (uint64_t i = 0; i < n; i++) if (T[i] > kmax) kmax = T[i];
    uint64_t *F = calloc((uint64_t)kmax + 2, sizeof(uint64_t));
    uint32_t *bwt = malloc(N * sizeof(uint32_t));
    uint32_t *lf = malloc(N * sizeof(uint32_t));
    int rc = 0;
    if (!F || !bwt || !lf) { snprintf(msg, msglen, "out of memory"); rc = 9; goto done; }
    for (uint64_t i = 0; i < n; i++) F[T[i] + 1]++;
    F[1] += 1;                                        /* the end symbol's row sorts with symbol 0 */
    for (uint64_t c = 1; c <= (uint64_t)kmax + 1; c++) F[c] += F[c - 1];
    memset(lf, 0xff, N * sizeof(uint32_t));
    for (uint64_t c = 0, k = 0; k < N; k++) {
        while (k >= F[c + 1]) c++;
        const uint64_t i = ilist[k];
        if (i >= N || lf[i] != 0xffffffffu) {
            snprintf(msg, msglen, "ilist is not a permutation of [0, %llu): entry %llu", (unsigned long long)N, (unsigned long long)k);
            rc = 2; goto done;
        }
        if (k > F[c] && ilist[k - 1] >= i) {
            snprintf(msg, msglen, "ilist does not ascend inside the range of symbol %llu at entry %llu", (unsigned long long)c, (unsigned long long)k);
            rc = 3; goto done;
        }
        lf[i] = (uint32_t)k;
        bwt[i] = (uint32_t)c;
    }
    uint64_t r = 0, s = n;                            /* row 0 holds the end suffix */
    for (uint64_t step = 0; step <= n; step++) {
        if (lf[r] == 0xffffffffu) {
            snprintf(msg, msglen, "the LF walk meets row %llu twice", (unsigned long long)r);
            rc = 4; goto done;
        }
        const uint32_t want = s ? T[s - 1] : 0u;
        const uint8_t wl = s == 0 ? 0 : (s == 1 ? last[n - 1] : last[s - 2]);
        if (bwt[r] != want) {
            snprintf(msg, msglen, "row %llu (suffix %llu): BWT symbol %u, %u expected", (unsigned long long)r,
                     (unsigned long long)s, bwt[r], want);
            rc = 5; goto done;
        }
        if (bwlast[r] != wl) {
            snprintf(msg, msglen, "row %llu (suffix %llu): bwlast %u, %u expected", (unsigned long long)r,
                     (unsigned long long)s, bwlast[r], wl);
            rc = 6; goto done;
        }
        if (sai && bwsai) {
            for (int j = 0; j < IBYTES; j++) {
                const uint8_t ws = s ? sai[(s - 1) * IBYTES + j] : 0;
                if (bwsai[r * IBYTES + j] != ws) {
                    snprintf(msg, msglen, "row %llu (suffix %llu): bwsai byte %d differs", (unsigned long long)r,
                             (unsigned long long)s, j);
                    rc = 7; goto done;
                }
            }
        }
        const uint64_t next = lf[r];
        lf[r] = 0xffffffffu;                          /* visited */
        if (s == 0) {
            if (r != 1) { snprintf(msg, msglen, "the suffix 0 sits at row %llu, not 1", (unsigned long long)r); rc = 8; goto done; }
            break;
        }
        r = next;
        s--;
    }
done:
    free(F);
    free(bwt);
    free(lf);
    return rc;
}
