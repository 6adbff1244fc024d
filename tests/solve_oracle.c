/*
 * tests/solve_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * A plain sequential CPU restatement of the inhomogeneous solve (blk_create_system + blk_solve, DESIGN.md
 * section 13), the reference for tests/test_gpu_solve.py, pinned by tests/test_solve_cpu.py.  It builds on the
 * kernel-basis restatement of tests/kb_oracle.c.  Compiled on demand by tests/solve_oracle.py.  All values are
 * canonical residues in [0,p), p < 2^31; one `%` per product.
 */
#include "kb_oracle.c"

/* The augmented matrix A^ = [M | -B] (right_kernel) or [M ; -B^T]: the COO of M followed by the non-zeros of -B,
 * B being Mc x r row-major (already reduced mod p).  Returns the number of triplets written. */
static long svo_augment(int nrows, int ncols, long nnz, const int *Mi, const int *Mj, const u32 *Mx, const u32 *B, int r,
                        u64 p, int right_kernel, int *Ai, int *Aj, u32 *Ax)
{
        long N = right_kernel ? ncols : nrows, Mc = right_kernel ? nrows : ncols, t = nnz;
        memcpy(Ai, Mi, sizeof(int) * (size_t)nnz);
        memcpy(Aj, Mj, sizeof(int) * (size_t)nnz);
        memcpy(Ax, Mx, sizeof(u32) * (size_t)nnz);
        for (long i = 0; i < Mc; i++)
                for (int j = 0; j < r; j++) {
                        u32 b = (u32)(B[i * r + j] % p);
                        if (!b)
                                continue;
                        Ai[t] = right_kernel ? (int)i : (int)(N + j);
                        Aj[t] = right_kernel ? (int)(N + j) : (int)i;
                        Ax[t] = (u32)(p - b);
                        t++;
                }
        return t;
}

/* The solve, given the COO of M, the Mc x r block B and the block v of the loop on A^ ((N + r) x n):
 *   1. X = v A_S, the kernel basis of A^ (kbo_kernel_basis), k columns;
 *   2. T = rows N .. N+r-1 of X (r x k); Q = the pivot columns of RREF(T);
 *   3. c_j solves T_Q c = e_j when e_j lies in colspace(T_Q) (found[j] = 1), else c_j = 0;
 *   4. x_j = rows 0 .. N-1 of X c_j.
 * x (N x r, row-major) and found[r] are caller-allocated.  Returns the number of solved right-hand sides. */
int svo_solve(int nrows, int ncols, long nnz, const int *Mi, const int *Mj, const u32 *Mx, const u32 *B, int r,
              const u32 *v, int n, u64 p, int right_kernel, u32 *x, int *found)
{
        long N = right_kernel ? ncols : nrows, Mc = right_kernel ? nrows : ncols, Np = N + r;
        long cap = nnz + Mc * r;
        int *Ai = malloc(sizeof(int) * (size_t)(cap ? cap : 1)), *Aj = malloc(sizeof(int) * (size_t)(cap ? cap : 1));
        u32 *Ax = malloc(sizeof(u32) * (size_t)(cap ? cap : 1));
        long annz = svo_augment(nrows, ncols, nnz, Mi, Mj, Mx, B, r, p, right_kernel, Ai, Aj, Ax);
        u32 *X = malloc(sizeof(u32) * (size_t)Np * (size_t)n);
        int k = kbo_kernel_basis(nrows + (right_kernel ? 0 : r), ncols + (right_kernel ? r : 0), annz, Ai, Aj, Ax, v, n, p,
                                 right_kernel, X);
        /* G = [T | I_r], r x (k + r), Gauss-Jordan on the first k columns */
        int w = k + r;
        u32 *G = calloc((size_t)r * (size_t)(w ? w : 1), sizeof(u32));
        int *Q = malloc(sizeof(int) * (size_t)(k ? k : 1)), q = 0;
        for (int i = 0; i < r; i++) {
                for (int s = 0; s < k; s++)
                        G[(size_t)i * w + s] = X[(size_t)(N + i) * n + s];
                G[(size_t)i * w + k + i] = 1;
        }
        u32 *tmp = malloc(sizeof(u32) * (size_t)(w ? w : 1));
        for (int col = 0; col < k; col++) {
                int pv = -1;
                for (int i = q; i < r; i++)
                        if (G[(size_t)i * w + col]) { pv = i; break; }
                if (pv < 0)
                        continue;
                memcpy(tmp, G + (size_t)pv * w, sizeof(u32) * (size_t)w);
                memcpy(G + (size_t)pv * w, G + (size_t)q * w, sizeof(u32) * (size_t)w);
                u64 inv = kbo_invmod(tmp[col], (u32)p);
                for (int c = 0; c < w; c++)
                        G[(size_t)q * w + c] = (u32)((tmp[c] * inv) % p);
                for (int i = 0; i < r; i++) {
                        u64 f = G[(size_t)i * w + col];
                        if (i == q || !f)
                                continue;
                        for (int c = 0; c < w; c++)
                                G[(size_t)i * w + c] = (u32)((G[(size_t)i * w + c] + (p - f) * G[(size_t)q * w + c]) % p);
                }
                Q[q++] = col;
        }
        /* c_j (k entries) for every j; x_j = rows 0 .. N-1 of X c_j */
        u32 *Cm = calloc((size_t)(k ? k : 1) * (size_t)r, sizeof(u32));
        int solved = 0;
        for (int j = 0; j < r; j++) {
                int ok = 1;
                for (int i = q; i < r; i++)
                        ok &= G[(size_t)i * w + k + j] == 0;
                found[j] = ok;
                solved += ok;
                if (ok)
                        for (int i = 0; i < q; i++)
                                Cm[(size_t)Q[i] * r + j] = G[(size_t)i * w + k + j];
        }
        for (long row = 0; row < N; row++)
                for (int j = 0; j < r; j++) {
                        u64 acc = 0;
                        for (int s = 0; s < k; s++)
                                acc = (acc + (u64)X[(size_t)row * n + s] * Cm[(size_t)s * r + j]) % p;
                        x[row * r + j] = (u32)acc;
                }
        free(Ai); free(Aj); free(Ax); free(X); free(G); free(Q); free(tmp); free(Cm);
        return solved;
}
