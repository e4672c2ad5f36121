/*
 * tandem_report_oracle.c -- TEST INFRASTRUCTURE ONLY: the tandem-repeat report of `--reportTRF` (DESIGN §2, R1-R6) for one
 * run u[0..L), computed literally from its statement with 64-bit counts and no bit planes.
 *
 *   R1  c[d] = #{x : 0 <= x < L - d, u[x] in ACGT, u[x] == u[x+d]}      d = 1..D, D = min(P, L - 1)   (case ignored)
 *   R2  p = the smallest d with 10 c[d] >= 9 max c
 *   R3  n_k[b] over x = k mod p; consensus[k] = the b with the largest count, ties to the earliest of A, C, G, T; N if none
 *   R4  matches = #{x : u[x] in ACGT, u[x] == consensus[x mod p]}
 *   R5  count[b] = sum_k n_k[b]
 *   R6  score = M c[p] - X (L - p - c[p])
 */
#include <stdint.h>
#include <stdlib.h>

static int base(uint8_t c) {
    switch (c) {
        case 'A': case 'a': return 0;
        case 'C': case 'c': return 1;
        case 'G': case 'g': return 2;
        case 'T': case 't': return 3;
        default: return -1;
    }
}

/* out[0..6] = period, score, matches, count A, C, G, T; cons receives period bytes (room for P). Returns 0, or -1 on bad
 * arguments / no memory. */
int tro_report(const uint8_t* u, long L, int M, int X, int P, int64_t* out, char* cons) {
    if (L < 2 || P < 1 || M < 1 || X < 0) return -1;
    const long D = P < L - 1 ? P : L - 1;
    int64_t* c = (int64_t*)calloc((size_t)D + 1, sizeof(int64_t));
    int64_t* n = (int64_t*)calloc((size_t)D * 4, sizeof(int64_t));
    if (!c || !n) { free(c); free(n); return -1; }
    for (long d = 1; d <= D; d++)
        for (long x = 0; x < L - d; x++)
            if (base(u[x]) >= 0 && base(u[x]) == base(u[x + d])) c[d]++;
    int64_t cmax = 0;
    for (long d = 1; d <= D; d++) cmax = c[d] > cmax ? c[d] : cmax;
    long p = 0;
    for (long d = 1; d <= D && !p; d++)
        if (10 * c[d] >= 9 * cmax) p = d;
    for (long x = 0; x < L; x++)
        if (base(u[x]) >= 0) n[(x % p) * 4 + base(u[x])]++;
    int64_t count[4] = {0, 0, 0, 0};
    for (long k = 0; k < p; k++) {
        int best = -1;
        for (int b = 0; b < 4; b++) {
            count[b] += n[k * 4 + b];
            if (n[k * 4 + b] > 0 && (best < 0 || n[k * 4 + b] > n[k * 4 + best])) best = b;
        }
        cons[k] = best < 0 ? 'N' : "ACGT"[best];
    }
    int64_t matches = 0;
    for (long x = 0; x < L; x++)
        if (base(u[x]) >= 0 && "ACGT"[base(u[x])] == cons[x % p]) matches++;
    out[0] = p;
    out[1] = (int64_t)M * c[p] - (int64_t)X * (L - p - c[p]);
    out[2] = matches;
    for (int b = 0; b < 4; b++) out[3 + b] = count[b];
    free(c); free(n);
    return 0;
}
