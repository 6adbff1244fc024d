// kernel_basis.cu -- the final Gaussian elimination of block Lanczos (Montgomery 1995): the kernel vectors
// inside span(v).  The reference has no such step; the definition (DESIGN.md section 12) is
//
//   T = S1 v (M^T v for --left, M v for --right); E_T = RREF of the row space of T, pivot columns P_T, F the others;
//   a_f = e_f - sum_i E_T[i][f] e_{P_T[i]} (f in F);  E_V = RREF of the row space of v;  B = E_V [a_f];
//   S = the f whose column of B is a pivot column of RREF(B);  X = v [a_f]_{f in S},  k = |S|.
//
// An RREF depends only on the row space, so the tall blocks v and T are reduced in any order, in pieces:
//
//   k_kb_reduce   every CTA streams a slab of rows (of v: blockIdx.y = 0, of T: 1) through an echelon basis of at most
//                 n rows in shared memory and stops once it has rank n; the last CTA to finish merges the partial
//                 bases into this rank's basis of each block (a "record": rank word, then the rows)
//   k_kb_small    one CTA: merges the records of all ranks (gathered), then steps E_T, a_f, B, S above; writes the
//                 n_pad x n_pad matrix A_S (column s = a_f of the s-th f in S, zero columns from k on) and k
//   k_block_apply x = v W for an n_pad x w_pad matrix W, one multiply-add per product: X = v A_S here, x = v (A_S C) for
//                 blk_solve (solve.cu)
//
// Every product is accumulated lazily in u64 (mp_mac / mp_fold of modp.cuh), exact for every 2 <= p < 2^31.
#include "blk_internal.cuh"
#include "small_body.cuh"
#include "dense_body.cuh"

namespace {

constexpr int KB_TB = 256;

// Echelon basis in shared memory: rank rows of NP words, fully reduced (a pivot column is zero in every other
// row) and normalised (pivot entry 1); the pivot of a row is its first non-zero column.  Rows are kept in
// insertion order; k_kb_small sorts them by pivot where the RREF itself is needed.
struct Basis {
        u32 *rows;
        int *piv;
        int *rank;
};

__device__ __forceinline__ int fold_period(const ModP &m) { return m.fold_every ? m.fold_every : 64; }

// One warp: reduce the row x (NP words, shared memory) against the basis and insert it if it stays non-zero.
template <int NP>
__device__ void warp_absorb(Basis b, u32 *x, const ModP &m)
{
        constexpr int PL = NP < 32 ? 1 : NP / 32;        // columns per lane: lane + 32 q
        const int lane = threadIdx.x & 31;
        const int r = *b.rank, fe = fold_period(m);
        u32 xv[PL];
#pragma unroll
        for (int q = 0; q < PL; q++) {
                const int j = lane + 32 * q;
                xv[q] = 0;
                if (j < NP) {
                        u64 acc = x[j];
                        int since = 0;
                        for (int i = 0; i < r; i++) {
                                mp_mac(acc, mp_neg(x[b.piv[i]], m), b.rows[i * NP + j]);
                                if (++since == fe) { mp_fold(acc, m); since = 0; }
                        }
                        xv[q] = mp_reduce(acc, m);
                }
        }
        int col = -1;
#pragma unroll
        for (int q = PL - 1; q >= 0; q--) {
                unsigned bal = __ballot_sync(0xffffffffu, xv[q] != 0);
                if (bal) col = 32 * q + __ffs(bal) - 1;
        }
        __syncwarp();
        if (col < 0) return;                              // uniform over the warp
        u32 lead = 0;
#pragma unroll
        for (int q = 0; q < PL; q++) {
                u32 t = __shfl_sync(0xffffffffu, xv[q], col & 31);
                if (q == col / 32) lead = t;
        }
        const u32 inv = mp_inv(lead, m);
#pragma unroll
        for (int q = 0; q < PL; q++) xv[q] = mp_mul(xv[q], inv, m);
        // clear the new pivot column in the rows already there
        for (int i = 0; i < r; i++) {
                const u32 f = mp_neg(b.rows[i * NP + col], m);
                __syncwarp();
                if (f) {
#pragma unroll
                        for (int q = 0; q < PL; q++) {
                                const int j = lane + 32 * q;
                                if (j < NP) b.rows[i * NP + j] = mp_add(b.rows[i * NP + j], mp_mul(f, xv[q], m), m);
                        }
                }
                __syncwarp();
        }
#pragma unroll
        for (int q = 0; q < PL; q++) {
                const int j = lane + 32 * q;
                if (j < NP) b.rows[r * NP + j] = xv[q];
        }
        if (lane == 0) { b.piv[r] = col; *b.rank = r + 1; }
        __syncwarp();
}

template <int NP> struct RoundShape {
        static constexpr int CW = NP < 4 ? NP : 4;        // columns per thread
        static constexpr int TPR = NP / CW;               // threads per row
        static constexpr int R = KB_TB / TPR;             // rows per round
};

// Whole CTA: absorb `rows` rows of src (leading dimension NP) into the basis, R rows per round: every thread
// reduces CW columns of one row against the basis as it stands (one lazy u64 sum per column: the basis is fully
// reduced, so all coefficients are read from the incoming row), then warp 0 inserts the rows that stayed non-zero.
// Stops early once the basis holds `cap` rows.  COH = 1: src was written by other CTAs of this launch (L2 loads).
template <int NP, int COH>
__device__ void cta_absorb_rows(Basis b, u32 *xs, int *flag, const u32 *src, int64_t rows, int cap, const ModP &m)
{
        using S = RoundShape<NP>;
        constexpr int CW = S::CW, TPR = S::TPR, R = S::R;
        const int row = threadIdx.x / TPR, j0 = (threadIdx.x % TPR) * CW;
        const int fe = fold_period(m);
        for (int64_t r0 = 0; r0 < rows; r0 += R) {
                if (*b.rank >= cap) break;                // uniform: read after the barrier that ended the last round
                const int64_t gr = r0 + row;
                u32 x[CW];
                if (gr < rows) ldv_c<CW, COH>(x, src + gr * NP + j0);
                else {
#pragma unroll
                        for (int c = 0; c < CW; c++) x[c] = 0;
                }
                stv<CW>(xs + row * NP + j0, x);
                __syncthreads();
                const int rk = *b.rank;
                u64 acc[CW];
#pragma unroll
                for (int c = 0; c < CW; c++) acc[c] = x[c];
                int since = 0;
                for (int i = 0; i < rk; i++) {
                        const u32 coef = mp_neg(xs[row * NP + b.piv[i]], m);
                        u32 bb[CW];
                        ldv<CW>(bb, b.rows + i * NP + j0);
#pragma unroll
                        for (int c = 0; c < CW; c++) mp_mac(acc[c], coef, bb[c]);
                        if (++since == fe) {
#pragma unroll
                                for (int c = 0; c < CW; c++) mp_fold(acc[c], m);
                                since = 0;
                        }
                }
                u32 y[CW];
                bool nz = false;
#pragma unroll
                for (int c = 0; c < CW; c++) { y[c] = mp_reduce(acc[c], m); nz |= y[c] != 0; }
                __syncthreads();                          // every coefficient has been read
                stv<CW>(xs + row * NP + j0, y);
                if (nz) flag[row] = 1;
                __syncthreads();
                if (threadIdx.x < 32) {
                        for (int w0 = 0; w0 < R && *b.rank < cap; w0 += 32) {
                                unsigned bal = __ballot_sync(0xffffffffu, w0 + (int)threadIdx.x < R && flag[w0 + threadIdx.x]);
                                while (bal && *b.rank < cap) {
                                        const int rr = w0 + __ffs(bal) - 1;
                                        bal &= bal - 1;
                                        warp_absorb<NP>(b, xs + rr * NP, m);
                                }
                        }
                        __syncwarp();
                        for (int e = threadIdx.x; e < R; e += 32) flag[e] = 0;
                }
                __syncthreads();
        }
}

// shared-memory carve-up of one basis + the round buffers
struct KbSmem {
        static size_t words(int n, int np, int nbases, int R) { return (size_t)nbases * (n * np + 64) + (size_t)R * np + R + 8; }
};

template <int NP>
__device__ Basis carve_basis(u32 *&at, int *rank_slot, int n)
{
        Basis b;
        b.rows = at; at += n * NP;
        b.piv = reinterpret_cast<int *>(at); at += 64;
        b.rank = rank_slot;
        return b;
}

// a record: (n + 1) x NP words, word 0 = rank, rows 1 .. rank = the basis rows
template <int NP>
__device__ void write_record(Basis b, u32 *rec, int n)
{
        const int rk = *b.rank;
        for (int e = threadIdx.x; e < n * NP; e += KB_TB) rec[NP + e] = e < rk * NP ? b.rows[e] : 0u;
        if (threadIdx.x == 0) rec[0] = (u32)rk;
}

template <int NP>
__global__ void __launch_bounds__(KB_TB)
k_kb_reduce(const u32 *v, int64_t vrows, const u32 *t, int64_t trows, int n, u32 *part, int *prank, unsigned *counter,
            u32 *rec, ModP m)
{
        using S = RoundShape<NP>;
        extern __shared__ u32 sm_kb[];
        __shared__ int s_rank;
        u32 *at = sm_kb;
        Basis b = carve_basis<NP>(at, &s_rank, n);
        u32 *xs = at; at += S::R * NP;
        int *flag = reinterpret_cast<int *>(at);
        for (int e = threadIdx.x; e < S::R; e += KB_TB) flag[e] = 0;
        if (threadIdx.x == 0) s_rank = 0;
        __syncthreads();

        const int y = blockIdx.y, C = gridDim.x;
        const u32 *src = y ? t : v;
        const int64_t rows = y ? trows : vrows;
        const int64_t slab = (rows + C - 1) / C, lo = (int64_t)blockIdx.x * slab, hi = lo + slab < rows ? lo + slab : rows;
        if (lo < hi) cta_absorb_rows<NP, 0>(b, xs, flag, src + lo * NP, hi - lo, n, m);
        const int rk = s_rank;
        u32 *dst = part + ((size_t)y * C + blockIdx.x) * n * NP;
        for (int e = threadIdx.x; e < rk * NP; e += KB_TB) dst[e] = b.rows[e];
        if (threadIdx.x == 0) prank[y * C + blockIdx.x] = rk;

        if (!last_block_done(counter, gridDim.x * gridDim.y)) return;
        for (int yy = 0; yy < 2; yy++) {
                __syncthreads();
                if (threadIdx.x == 0) s_rank = 0;
                __syncthreads();
                for (int c = 0; c < C; c++) {
                        const int pr = __ldcg(prank + yy * C + c);
                        cta_absorb_rows<NP, 1>(b, xs, flag, part + ((size_t)yy * C + c) * n * NP, pr, n, m);
                        if (s_rank >= n) break;
                }
                write_record<NP>(b, rec + (size_t)yy * (n + 1) * NP, n);
        }
}

// One CTA: the records of `world` ranks (rank w: v at rec[(2w) (n+1) NP], T at rec[(2w+1) (n+1) NP]) -> A_S, k.
template <int NP>
__global__ void __launch_bounds__(KB_TB)
k_kb_small(const u32 *rec, int world, int n, u32 *A_out, int *k_out, ModP m)
{
        using S = RoundShape<NP>;
        extern __shared__ u32 sm_kb[];
        __shared__ int s_rank[3];
        __shared__ int s_rowof[64], s_F[64], s_S[64], s_m, s_k;
        u32 *at = sm_kb;
        Basis bv = carve_basis<NP>(at, &s_rank[0], n);
        Basis bt = carve_basis<NP>(at, &s_rank[1], n);
        Basis bb = carve_basis<NP>(at, &s_rank[2], n);
        u32 *A = at; at += NP * NP;                       // A[j][t] = entry j of a_{F[t]}
        u32 *Brows = at; at += n * NP;
        u32 *xs = at; at += S::R * NP;
        int *flag = reinterpret_cast<int *>(at);
        for (int e = threadIdx.x; e < S::R; e += KB_TB) flag[e] = 0;
        if (threadIdx.x < 3) s_rank[threadIdx.x] = 0;
        __syncthreads();
        for (int w = 0; w < world; w++) {
                const u32 *rv = rec + (size_t)(2 * w) * (n + 1) * NP, *rt = rv + (size_t)(n + 1) * NP;
                cta_absorb_rows<NP, 0>(bv, xs, flag, rv + NP, (int)rv[0], n, m);
                cta_absorb_rows<NP, 0>(bt, xs, flag, rt + NP, (int)rt[0], n, m);
        }
        __syncthreads();
        const int rV = s_rank[0], rT = s_rank[1];
        // E_T row of pivot column j (-1: j in F), F ascending
        if (threadIdx.x < 64) s_rowof[threadIdx.x] = -1;
        __syncthreads();
        if (threadIdx.x < rT) s_rowof[bt.piv[threadIdx.x]] = threadIdx.x;
        __syncthreads();
        if (threadIdx.x == 0) {
                int mm = 0;
                for (int f = 0; f < n; f++)
                        if (s_rowof[f] < 0) s_F[mm++] = f;
                s_m = mm;
        }
        __syncthreads();
        const int mF = s_m;
        for (int e = threadIdx.x; e < NP * NP; e += KB_TB) {
                const int j = e / NP, tt = e % NP;
                u32 a = 0;
                if (tt < mF && j < n) {
                        const int f = s_F[tt];
                        if (j == f) a = 1;
                        else if (s_rowof[j] >= 0) a = mp_neg(bt.rows[s_rowof[j] * NP + f], m);
                }
                A[e] = a;
        }
        __syncthreads();
        // B = E_V A: rows of the basis of v in any order (only its row space matters)
        const int fe = fold_period(m);
        for (int e = threadIdx.x; e < rV * NP; e += KB_TB) {
                const int i = e / NP, tt = e % NP;
                u64 acc = 0;
                int since = 0;
                for (int j = 0; j < n; j++) {
                        mp_mac(acc, bv.rows[i * NP + j], A[j * NP + tt]);
                        if (++since == fe) { mp_fold(acc, m); since = 0; }
                }
                Brows[e] = mp_reduce(acc, m);
        }
        __syncthreads();
        cta_absorb_rows<NP, 0>(bb, xs, flag, Brows, rV, n, m);
        __syncthreads();
        if (threadIdx.x == 0) {
                // S: the pivot columns of RREF(B), ascending
                int kk = 0;
                for (int tt = 0; tt < NP; tt++)
                        for (int i = 0; i < s_rank[2]; i++)
                                if (bb.piv[i] == tt) s_S[kk++] = tt;
                s_k = kk;
                *k_out = kk;
        }
        __syncthreads();
        for (int e = threadIdx.x; e < NP * NP; e += KB_TB) {
                const int j = e / NP, s = e % NP;
                A_out[e] = s < s_k ? A[j * NP + s_S[s]] : 0u;
        }
}

// x = v W (W: NP x WP, WP <= NP): thread (row, slice) forms OC consecutive outputs of one row from the whole row of v
// (NP words, vector loads) and W in shared memory; every product is one multiply-add into a lazy u64, folded every FOLD
// products (0: never, NP <= 64 products fit).
constexpr int APPLY_TB = 256;

template <int NP, int WP, int FOLD>
__global__ void __launch_bounds__(APPLY_TB)
k_block_apply(int64_t rows, const u32 *__restrict__ v, const u32 *__restrict__ W, u32 *__restrict__ x, ModP m)
{
        constexpr int OC = WP < 8 ? WP : 8;               // outputs per thread
        constexpr int TPR = WP / OC;                      // threads per row
        constexpr int VL = NP < 4 ? NP : 4;               // words per load
        __shared__ u32 Ws[NP * WP];
        for (int e = threadIdx.x; e < NP * WP; e += APPLY_TB) Ws[e] = W[e];
        __syncthreads();
        const int64_t gid = (int64_t)blockIdx.x * APPLY_TB + threadIdx.x;
        const int64_t row = gid / TPR;
        if (row >= rows) return;
        const int o0 = (int)(gid % TPR) * OC;
        u64 acc[OC];
#pragma unroll
        for (int o = 0; o < OC; o++) acc[o] = 0;
        const u32 *vr = v + row * NP;
#pragma unroll
        for (int j0 = 0; j0 < NP; j0 += VL) {
                u32 a[VL];
                ldv<VL>(a, vr + j0);
#pragma unroll
                for (int jj = 0; jj < VL; jj++) {
#pragma unroll
                        for (int o = 0; o < OC; o++) mp_mac(acc[o], a[jj], Ws[(j0 + jj) * WP + o0 + o]);
                        if constexpr (FOLD > 0) {
                                if ((j0 + jj + 1) % FOLD == 0) {
#pragma unroll
                                        for (int o = 0; o < OC; o++) mp_fold(acc[o], m);
                                }
                        }
                }
        }
        u32 out[OC];
#pragma unroll
        for (int o = 0; o < OC; o++) out[o] = mp_reduce(acc[o], m);
        u32 *xr = x + row * WP + o0;
        if constexpr (OC >= 4) {
#pragma unroll
                for (int o = 0; o < OC; o += 4) {
                        u32 w4[4] = {out[o], out[o + 1], out[o + 2], out[o + 3]};
                        stv<4>(xr + o, w4);
                }
        } else {
                stv<OC>(xr, out);
        }
}

template <int NP>
int reduce_go(const KbArgs &a, cudaStream_t st)
{
        using S = RoundShape<NP>;
        const size_t smem = sizeof(u32) * KbSmem::words(a.n, NP, 1, S::R);
        cudaFuncSetAttribute(k_kb_reduce<NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        k_kb_reduce<NP><<<dim3(a.ctas, 2), KB_TB, smem, st>>>(a.v, a.vrows, a.t, a.trows, a.n, a.part, a.prank, a.counter,
                                                              a.rec_own, a.m);
        return 1;
}

template <int NP>
int small_go(const KbArgs &a, cudaStream_t st)
{
        using S = RoundShape<NP>;
        const size_t smem = sizeof(u32) * (KbSmem::words(a.n, NP, 3, S::R) + (size_t)NP * NP + (size_t)a.n * NP);
        cudaFuncSetAttribute(k_kb_small<NP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        k_kb_small<NP><<<1, KB_TB, smem, st>>>(a.rec_all, a.world, a.n, a.A, a.k, a.m);
        return 1;
}

template <int NP, int WP>
int apply_wp(int64_t rows, const u32 *v, const u32 *W, u32 *x, const ModP &m, cudaStream_t st)
{
        constexpr int OC = WP < 8 ? WP : 8, TPR = WP / OC;
        const unsigned blocks = (unsigned)((rows * TPR + APPLY_TB - 1) / APPLY_TB);
        switch (m.fold_every) {
        case 0: k_block_apply<NP, WP, 0><<<blocks, APPLY_TB, 0, st>>>(rows, v, W, x, m); break;
        case 8: k_block_apply<NP, WP, 8><<<blocks, APPLY_TB, 0, st>>>(rows, v, W, x, m); break;
        default: k_block_apply<NP, WP, 2><<<blocks, APPLY_TB, 0, st>>>(rows, v, W, x, m); break;
        }
        return 1;
}

template <int NP>
int apply_np(int wp, int64_t rows, const u32 *v, const u32 *W, u32 *x, const ModP &m, cudaStream_t st)
{
        switch (wp) {
        case 1: return apply_wp<NP, 1>(rows, v, W, x, m, st);
        case 2: if constexpr (NP >= 2) return apply_wp<NP, 2>(rows, v, W, x, m, st); break;
        case 4: if constexpr (NP >= 4) return apply_wp<NP, 4>(rows, v, W, x, m, st); break;
        case 8: if constexpr (NP >= 8) return apply_wp<NP, 8>(rows, v, W, x, m, st); break;
        case 16: if constexpr (NP >= 16) return apply_wp<NP, 16>(rows, v, W, x, m, st); break;
        case 32: if constexpr (NP >= 32) return apply_wp<NP, 32>(rows, v, W, x, m, st); break;
        case 64: if constexpr (NP >= 64) return apply_wp<NP, 64>(rows, v, W, x, m, st); break;
        }
        return -1;
}

}  // namespace

int kb_ctas(int64_t rows)
{
        int64_t c = (rows + 1023) / 1024;
        if (c < 1) c = 1;
        if (c > 2 * blk_sm_count()) c = 2 * blk_sm_count();
        return (int)c;
}

int launch_kb_reduce(int np, const KbArgs &a, cudaStream_t st)
{
        switch (np) {
        case 1: return reduce_go<1>(a, st);
        case 2: return reduce_go<2>(a, st);
        case 4: return reduce_go<4>(a, st);
        case 8: return reduce_go<8>(a, st);
        case 16: return reduce_go<16>(a, st);
        case 32: return reduce_go<32>(a, st);
        case 64: return reduce_go<64>(a, st);
        }
        return -1;
}

int launch_kb_small(int np, const KbArgs &a, cudaStream_t st)
{
        switch (np) {
        case 1: return small_go<1>(a, st);
        case 2: return small_go<2>(a, st);
        case 4: return small_go<4>(a, st);
        case 8: return small_go<8>(a, st);
        case 16: return small_go<16>(a, st);
        case 32: return small_go<32>(a, st);
        case 64: return small_go<64>(a, st);
        }
        return -1;
}

int launch_block_apply(int np, int wp, int64_t rows, const u32 *v, const u32 *W, u32 *x, const ModP &m, cudaStream_t st)
{
        if (rows <= 0) return 0;
        switch (np) {
        case 1: return apply_np<1>(wp, rows, v, W, x, m, st);
        case 2: return apply_np<2>(wp, rows, v, W, x, m, st);
        case 4: return apply_np<4>(wp, rows, v, W, x, m, st);
        case 8: return apply_np<8>(wp, rows, v, W, x, m, st);
        case 16: return apply_np<16>(wp, rows, v, W, x, m, st);
        case 32: return apply_np<32>(wp, rows, v, W, x, m, st);
        case 64: return apply_np<64>(wp, rows, v, W, x, m, st);
        }
        return -1;
}
