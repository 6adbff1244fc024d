/*
 * tests/kb_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * A plain sequential CPU restatement of the kernel-basis extraction (blk_kernel_basis, DESIGN.md section 12),
 * the reference for tests/test_gpu_kernel_basis.py.  The reference program has no such step, so this file is
 * pinned by the defining properties of its result in tests/test_kernel_basis_cpu.py.  It is self-contained:
 * the product and the inverse below restate orc_spmv and orc_invmod of oracle/lanczos_oracle.c.
 * Compiled on demand by tests/kb_oracle.py.  All values are canonical residues in [0,p), p < 2^31.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef uint32_t u32;
typedef uint64_t u64;

/* y <- M x (transpose == 0) or M^T x (transpose != 0) on n-wide row-major blocks, COO input */
static void kbo_spmv(u32 *y, int nrows, int ncols, long nnz, const int *Mi, const int *Mj, const u32 *Mx,
                     const u32 *x, int transpose, int n, u64 p)
{
        long out_rows = transpose ? ncols : nrows;
        memset(y, 0, sizeof(u32) * (size_t)out_rows * (size_t)n);
        for (long e = 0; e < nnz; e++) {
                long r = transpose ? Mj[e] : Mi[e];
                long c = transpose ? Mi[e] : Mj[e];
                u64 a = Mx[e];
                for (int l = 0; l < n; l++)
                        y[r * n + l] = (u32)((y[r * n + l] + a * x[c * n + l]) % p);
        }
}

/* a^-1 mod m, extended Euclid */
static u32 kbo_invmod(u32 a, u32 m)
{
        int64_t r0 = m, r1 = a % m, t0 = 0, t1 = 1;
        while (r1) {
                int64_t q = r0 / r1, w;
                w = r0 - q * r1; r0 = r1; r1 = w;
                w = t0 - q * t1; t0 = t1; t1 = w;
        }
        return (u32)(t0 < 0 ? t0 + m : t0);
}


/* ------------------------------------------------------------------ kernel basis
 * The final Gaussian elimination of block Lanczos (Montgomery 1995), which the
 * reference does not have.  V is the N x n block v, T = S1 V the Mc x n block
 * M^T v (left) or M v (right).  Over GF(p):
 *   1. E_T = RREF of the row space of T, pivot columns P_T, F = the others;
 *   2. a_f = e_f - sum_i E_T[i][f] e_{P_T[i]} for f in F (null basis of T);
 *   3. E_V = RREF of the row space of V, B = E_V [a_f], S = the f whose
 *      column of B is a pivot column of RREF(B);
 *   4. X = V [a_f]_{f in S}, k = |S|.
 * X (N x n, caller-allocated) receives X in columns [0,k), zeros elsewhere.
 * Returns k.  Plain row-by-row elimination, one `%` per product.          */

/* insert row x (w entries, destroyed) into the fully reduced basis b[*rank][w]
 * with pivot columns piv[]: reduce, then (if non-zero) normalise at its first
 * non-zero column and clear that column in the other rows. */
static void rref_absorb(u32 *b, int *piv, int *rank, u32 *x, int w, u64 p)
{
        for (int i = 0; i < *rank; i++) {
                u64 c = x[piv[i]];
                if (!c) continue;
                for (int j = 0; j < w; j++)
                        x[j] = (u32)((x[j] + (p - c) * b[i * w + j]) % p);
        }
        int q = 0;
        while (q < w && !x[q]) q++;
        if (q == w) return;
        u64 inv = kbo_invmod(x[q], (u32)p);
        for (int j = 0; j < w; j++) x[j] = (u32)((x[j] * inv) % p);
        for (int i = 0; i < *rank; i++) {
                u64 f = b[i * w + q];
                if (!f) continue;
                for (int j = 0; j < w; j++)
                        b[i * w + j] = (u32)((b[i * w + j] + (p - f) * x[j]) % p);
        }
        memcpy(b + (size_t)*rank * w, x, sizeof(u32) * (size_t)w);
        piv[(*rank)++] = q;
}

/* RREF of the row space of a[rows][w]: rank rows of e (w wide) by increasing pivot */
static int rref_rows(const u32 *a, long rows, int w, u64 p, u32 *e, int *piv)
{
        u32 *b = malloc(sizeof(u32) * (size_t)w * (size_t)w), *x = malloc(sizeof(u32) * (size_t)w);
        int *bp = malloc(sizeof(int) * (size_t)w), rank = 0;
        for (long r = 0; r < rows && rank < w; r++) {
                memcpy(x, a + r * w, sizeof(u32) * (size_t)w);
                rref_absorb(b, bp, &rank, x, w, p);
        }
        int out = 0;
        for (int q = 0; q < w; q++)
                for (int i = 0; i < rank; i++)
                        if (bp[i] == q) {
                                memcpy(e + (size_t)out * w, b + (size_t)i * w, sizeof(u32) * (size_t)w);
                                piv[out++] = q;
                        }
        free(b); free(x); free(bp);
        return rank;
}

int kbo_kernel_basis(int nrows, int ncols, long nnz, const int *Mi, const int *Mj, const u32 *Mx,
                     const u32 *v, int n, u64 p, int right_kernel, u32 *X)
{
        long N = right_kernel ? ncols : nrows, Mc = right_kernel ? nrows : ncols;
        size_t nn = (size_t)n * (size_t)n;
        u32 *T = malloc(sizeof(u32) * (size_t)Mc * (size_t)n);
        u32 *ET = calloc(nn, 4), *EV = calloc(nn, 4), *A = calloc(nn, 4), *Bm = calloc(nn, 4), *EB = calloc(nn, 4);
        int *pt = malloc(sizeof(int) * (size_t)n), *pv = malloc(sizeof(int) * (size_t)n), *pb = malloc(sizeof(int) * (size_t)n);
        int *F = malloc(sizeof(int) * (size_t)n), *isp = calloc((size_t)n, sizeof(int));
        kbo_spmv(T, nrows, ncols, nnz, Mi, Mj, Mx, v, !right_kernel, n, p);
        int rT = rref_rows(T, Mc, n, p, ET, pt);
        int rV = rref_rows(v, N, n, p, EV, pv);
        for (int i = 0; i < rT; i++) isp[pt[i]] = 1;
        int m = 0;
        for (int f = 0; f < n; f++)
                if (!isp[f]) F[m++] = f;
        /* a_f as column t of A (n x m, row-major with stride n) */
        for (int t = 0; t < m; t++) {
                A[(size_t)F[t] * n + t] = 1;
                for (int i = 0; i < rT; i++)
                        A[(size_t)pt[i] * n + t] = (u32)((p - ET[(size_t)i * n + F[t]]) % p);
        }
        /* B = E_V A (rV x m, stride n) */
        for (int i = 0; i < rV; i++)
                for (int t = 0; t < m; t++) {
                        u64 s = 0;
                        for (int j = 0; j < n; j++)
                                s = (s + (u64)EV[(size_t)i * n + j] * A[(size_t)j * n + t]) % p;
                        Bm[(size_t)i * n + t] = (u32)s;
                }
        int rB = rref_rows(Bm, rV, n, p, EB, pb);
        /* X = V A_S, columns [0, rB) */
        memset(X, 0, sizeof(u32) * (size_t)N * (size_t)n);
        for (long r = 0; r < N; r++)
                for (int s = 0; s < rB; s++) {
                        u64 acc = 0;
                        for (int j = 0; j < n; j++)
                                acc = (acc + (u64)v[r * n + j] * A[(size_t)j * n + pb[s]]) % p;
                        X[r * n + s] = (u32)acc;
                }
        free(T); free(ET); free(EV); free(A); free(Bm); free(EB);
        free(pt); free(pv); free(pb); free(F); free(isp);
        return rB;
}
