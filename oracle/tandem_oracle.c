/*
 * tandem_oracle.c -- TEST INFRASTRUCTURE ONLY: the tandem-repeat mask of `mimeo map --maxtandem` (DESIGN §2, T1-T4),
 * computed literally from its statement. No clamping, no anti-diagonal order, 64-bit scores.
 *
 *   sub(a,b)  = +M if toupper(a) == toupper(b) and it is one of A,C,G,T, else -X
 *   strip     = prefix-matrix cells (i,j), 0 <= i,j <= n, with 1 <= j-i <= P; every other cell is -inf
 *   H[i][j]   = max(0, H[i-1][j-1] + sub(s[i-1],s[j-1]), H[i-1][j] - G, H[i][j-1] - G)    (H[0][j] = H[i][0] = 0)
 *   H'[i][j]  = max(0, H'[i+1][j+1] + sub(s[i],s[j]), H'[i+1][j] - G, H'[i][j+1] - G)     (0 at i = n or j = n)
 *   best(p,q) = H[p][q] + sub(s[p],s[q]) + H'[p+1][q+1] for 1 <= q-p <= P; (p,q) qualifies iff best >= T
 *   position x is masked iff some qualifying pair has p <= x <= q
 *
 * Both matrices are stored whole, as (n+1) rows of the P diagonals of the strip.
 */
#include <stdint.h>
#include <stdlib.h>

#define NEG_INF (INT64_MIN / 4)

static int is_acgt(uint8_t c) { return c == 'A' || c == 'C' || c == 'G' || c == 'T'; }
static uint8_t up(uint8_t c) { return (c >= 'a' && c <= 'z') ? (uint8_t)(c - 32) : c; }
static int64_t sub(uint8_t a, uint8_t b, int M, int X) {
    a = up(a); b = up(b);
    return (a == b && is_acgt(a)) ? M : -(int64_t)X;
}
static int64_t max2(int64_t a, int64_t b) { return a > b ? a : b; }

/* cell (i, j) of the strip: i in [0, n], d = j - i in [1, P]; anything else is -inf or the boundary */
#define AT(A, i, j) (A)[(size_t)(i) * (size_t)P + (size_t)((j) - (i) - 1)]

static int64_t fwd(const int64_t* H, long n, int P, long i, long j) {
    if (i < 0 || j < 0 || i > n || j > n) return NEG_INF;
    if (i == 0 || j == 0) return 0;
    if (j - i < 1 || j - i > P) return NEG_INF;
    return AT(H, i, j);
}
static int64_t bwd(const int64_t* B, long n, int P, long i, long j) {
    if (i < 0 || j < 0 || i > n || j > n) return NEG_INF;
    if (i == n || j == n) return 0;
    if (j - i < 1 || j - i > P) return NEG_INF;
    return AT(B, i, j);
}

/* Returns m (the number of masked positions of s[0..n)), or -1 on bad arguments / no memory. The merged masked intervals
 * (maximal runs of masked positions, closed, 0-based) go to iv_start / iv_end, at most cap of them; *niv receives how
 * many there are. */
long tro_mask(const uint8_t* s, long n, int M, int X, int G, int T, int P, int64_t* iv_start, int64_t* iv_end, long cap, long* niv) {
    if (niv) *niv = 0;
    if (n < 0 || P < 1 || M < 1 || X < 0 || G < 0 || T < 1) return -1;
    if (n < 2) return 0;
    int64_t* H = (int64_t*)malloc(sizeof(int64_t) * (size_t)(n + 1) * (size_t)P);
    int64_t* B = (int64_t*)malloc(sizeof(int64_t) * (size_t)(n + 1) * (size_t)P);
    uint8_t* mask = (uint8_t*)calloc((size_t)n, 1);
    if (!H || !B || !mask) { free(H); free(B); free(mask); return -1; }
    for (long i = 1; i <= n; i++)
        for (long j = i + 1; j <= n && j - i <= P; j++) {
            int64_t v = 0;
            v = max2(v, fwd(H, n, P, i - 1, j - 1) + sub(s[i - 1], s[j - 1], M, X));
            v = max2(v, fwd(H, n, P, i - 1, j) - G);
            v = max2(v, fwd(H, n, P, i, j - 1) - G);
            AT(H, i, j) = v;
        }
    for (long i = n - 1; i >= 0; i--)
        for (long j = (i + P < n - 1 ? i + P : n - 1); j >= i + 1; j--) {
            int64_t v = 0;
            v = max2(v, bwd(B, n, P, i + 1, j + 1) + sub(s[i], s[j], M, X));
            v = max2(v, bwd(B, n, P, i + 1, j) - G);
            v = max2(v, bwd(B, n, P, i, j + 1) - G);
            AT(B, i, j) = v;
        }
    for (long p = 0; p < n; p++)
        for (long q = p + 1; q < n && q - p <= P; q++) {
            const int64_t best = fwd(H, n, P, p, q) + sub(s[p], s[q], M, X) + bwd(B, n, P, p + 1, q + 1);
            if (best >= T)
                for (long x = p; x <= q; x++) mask[x] = 1;
        }
    long m = 0, k = 0;
    for (long x = 0; x < n; x++) {
        if (!mask[x]) continue;
        m++;
        if (x == 0 || !mask[x - 1]) {
            long e = x;
            while (e + 1 < n && mask[e + 1]) e++;
            if (k < cap) { iv_start[k] = x; iv_end[k] = e; }
            k++;
        }
    }
    if (niv) *niv = k;
    free(H); free(B); free(mask);
    return m;
}
