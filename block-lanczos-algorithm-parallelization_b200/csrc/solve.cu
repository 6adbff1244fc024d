// solve.cu -- inhomogeneous systems M x = b (--right) and x M = b (--left) mod p (blk_create_system, blk_solve).
// The definition (DESIGN.md section 13): with the Mc x r right-hand-side block B,
//
//   A^ = [M | -B] (--right) or [M ; -B^T] (--left); the loop runs unchanged on A^, whose Lanczos vectors have
//   N' = N + r rows, the RHS coordinates N .. N+r-1.  X = v A_S as in section 12 (k columns).
//   T = rows N .. N+r-1 of X (r x k);  Q = the pivot columns of RREF(T);  c_j solves T_Q c = e_j when e_j lies in
//   colspace(T_Q) (found[j] = 1; zeros outside Q), else c_j = 0;  x_j = rows 0 .. N-1 of X c_j = v (A_S C).
//
// The kernels:
//
//   k_rhs_count / k_rhs_triplets   the non-zeros of -B appended to the device COO of M (count per CTA, scan, write
//                                  in order: the appended triplets do not depend on the launch)
//   k_solve_tail                   the r tail rows of v that this rank owns (an r x n_pad block, zero elsewhere;
//                                  the ranks' blocks are summed by one all-reduce)
//   k_solve_small                  one CTA: T = v_tail A_S, Gauss-Jordan of [T | I_r], C, W = A_S C, found
//
// A_S and k come from k_kb_reduce / k_kb_small of kernel_basis.cu, unchanged; x = v W is its k_block_apply with r_pad
// output columns.
#include <cub/cub.cuh>
#include "blk_internal.cuh"

namespace {

constexpr int RHS_TB = 256;
constexpr int RHS_PER = 8;                 // elements of B per thread and CTA pass
constexpr int64_t RHS_CHUNK = (int64_t)RHS_TB * RHS_PER;

// non-zeros of B (mod p) in every chunk of RHS_CHUNK elements
__global__ void __launch_bounds__(RHS_TB) k_rhs_count(const u32 *__restrict__ B, int64_t total, u32 p, u32 *__restrict__ cnt)
{
        const int64_t base = (int64_t)blockIdx.x * RHS_CHUNK;
        int c = 0;
        for (int q = 0; q < RHS_PER; q++) {
                const int64_t e = base + (int64_t)q * RHS_TB + threadIdx.x;
                c += __syncthreads_count(e < total && B[e] % p != 0);
        }
        if (threadIdx.x == 0) cnt[blockIdx.x] = (u32)c;
}

// element e = i * r + j of B (row i of the Mc dimension, right-hand side j) becomes the triplet
// (i, N + j) for --right, (N + j, i) for --left, with value -B[e] mod p, at slot off[chunk] + (its rank in the chunk)
__global__ void __launch_bounds__(RHS_TB) k_rhs_triplets(const u32 *__restrict__ B, int64_t total, int r, int64_t N, int right,
                                                         u32 p, const u64 *__restrict__ off, int32_t *__restrict__ Mi,
                                                         int32_t *__restrict__ Mj, u32 *__restrict__ Mx)
{
        typedef cub::BlockScan<int, RHS_TB> Scan;
        __shared__ typename Scan::TempStorage ts;
        const int64_t base = (int64_t)blockIdx.x * RHS_CHUNK;
        u64 at = off[blockIdx.x];
        for (int q = 0; q < RHS_PER; q++) {
                const int64_t e = base + (int64_t)q * RHS_TB + threadIdx.x;
                const u32 b = e < total ? B[e] % p : 0u;
                int pos = 0, sum = 0;
                Scan(ts).ExclusiveSum(b != 0 ? 1 : 0, pos, sum);
                if (b) {
                        const int32_t i = (int32_t)(e / r), j = (int32_t)(N + e % r);
                        Mi[at + pos] = right ? i : j;
                        Mj[at + pos] = right ? j : i;
                        Mx[at + pos] = p - b;
                }
                at += (u64)sum;
                __syncthreads();                           // ts is reused by the next pass
        }
}

// tail[j][:] = row N0 + j of v (device row map[N0 + j] under a relabelling) when this rank owns it, else zero
__global__ void k_solve_tail(const u32 *__restrict__ v, int64_t N0, int r, int np, const u32 *__restrict__ map, int64_t n0,
                             int64_t n1, u32 *__restrict__ tail)
{
        const int e = blockIdx.x * blockDim.x + threadIdx.x;
        if (e >= r * np) return;
        const int j = e / np, col = e % np;
        const int64_t pos = map ? (int64_t)map[N0 + j] : N0 + j;
        tail[e] = pos >= n0 && pos < n1 ? v[pos * np + col] : 0u;
}

constexpr int SOLVE_TB = 256;

// One CTA.  A (NP x NP, columns from *k_in on zero), tail (r x NP) -> W (NP x rp, columns from r on zero), found[r].
// [T | I_r] lives in shared memory (r x 2 NP words); A is read from global memory (a few KB, cached).
template <int NP>
__global__ void __launch_bounds__(SOLVE_TB)
k_solve_small(const u32 *__restrict__ A, const int *__restrict__ k_in, const u32 *__restrict__ tail, int r, int rp,
              u32 *__restrict__ W, int *__restrict__ found, ModP m)
{
        constexpr int GW = 2 * NP;                        // k + r <= 2 NP columns
        __shared__ u32 G[NP * GW];
        __shared__ u32 fac[NP];
        __shared__ int s_piv, s_rank, s_Q[NP], s_found[NP];
        __shared__ u32 s_inv;
        const int k = *k_in;
        const int fe = m.fold_every ? m.fold_every : 64;
        // T = tail A_S (r x k), then the identity block
        for (int e = threadIdx.x; e < r * GW; e += SOLVE_TB) {
                const int i = e / GW, c = e % GW;
                u32 val = 0;
                if (c < k) {
                        u64 acc = 0;
                        int since = 0;
                        for (int j = 0; j < NP; j++) {
                                mp_mac(acc, tail[i * NP + j], A[j * NP + c]);
                                if (++since == fe) { mp_fold(acc, m); since = 0; }
                        }
                        val = mp_reduce(acc, m);
                } else if (c < k + r) val = c - k == i ? 1u : 0u;
                G[e] = val;
        }
        if (threadIdx.x == 0) s_rank = 0;
        __syncthreads();
        // Gauss-Jordan on the first k columns: afterwards rows [0, q) of the T part are RREF(T), pivot columns s_Q
        for (int col = 0; col < k; col++) {
                const int rk = s_rank;
                if (threadIdx.x == 0) {
                        int pv = -1;
                        for (int i = rk; i < r; i++)
                                if (G[i * GW + col]) { pv = i; break; }
                        s_piv = pv;
                        if (pv >= 0) s_inv = mp_inv(G[pv * GW + col], m);
                }
                __syncthreads();
                const int pv = s_piv;
                __syncthreads();                           // every thread has read s_piv before thread 0 may rewrite it
                if (pv < 0) continue;                      // uniform
                // swap rows pv and rk, normalise the pivot row
                for (int c = threadIdx.x; c < GW; c += SOLVE_TB) {
                        const u32 a = G[pv * GW + c], b = G[rk * GW + c];
                        G[rk * GW + c] = mp_mul(a, s_inv, m);
                        if (pv != rk) G[pv * GW + c] = b;
                }
                __syncthreads();
                for (int i = threadIdx.x; i < r; i += SOLVE_TB) fac[i] = i == rk ? 0u : mp_neg(G[i * GW + col], m);
                __syncthreads();
                for (int e = threadIdx.x; e < r * GW; e += SOLVE_TB) {
                        const int i = e / GW, c = e % GW;
                        if (fac[i]) G[e] = mp_add(G[e], mp_mul(fac[i], G[rk * GW + c], m), m);
                }
                __syncthreads();
                if (threadIdx.x == 0) { s_Q[rk] = col; s_rank = rk + 1; }
                __syncthreads();
        }
        const int q = s_rank;
        // e_j lies in colspace(T) iff column j of the identity part vanishes below row q (those rows span the left
        // null space of T); then c_j[Q[i]] = row i of that column, i < q, and c_j is zero outside Q
        for (int j = threadIdx.x; j < r; j += SOLVE_TB) {
                int ok = 1;
                for (int i = q; i < r; i++) ok &= G[i * GW + k + j] == 0;
                s_found[j] = ok;
                found[j] = ok;
        }
        __syncthreads();
        // W = A_S C (NP x rp):  W[a][j] = sum_i A[a][Q[i]] c_j[Q[i]]
        for (int e = threadIdx.x; e < NP * rp; e += SOLVE_TB) {
                const int a = e / rp, j = e % rp;
                u32 val = 0;
                if (j < r && s_found[j]) {
                        u64 acc = 0;
                        int since = 0;
                        for (int i = 0; i < q; i++) {
                                mp_mac(acc, A[a * NP + s_Q[i]], G[i * GW + k + j]);
                                if (++since == fe) { mp_fold(acc, m); since = 0; }
                        }
                        val = mp_reduce(acc, m);
                }
                W[e] = val;
        }
}

template <int NP>
int small_np(const SolveArgs &a, cudaStream_t st)
{
        k_solve_small<NP><<<1, SOLVE_TB, 0, st>>>(a.A, a.k, a.tail, a.r, a.rp, a.W, a.found, a.m);
        return 1;
}

}  // namespace

int pad_width(int w)
{
        int p = 1;
        while (p < w) p *= 2;
        return p;
}

// The non-zeros of -B as COO triplets of the augmented matrix.  *count receives their number; with Mi == nullptr
// nothing is written (a first call sizes the buffers, a second one fills them at Mi/Mj/Mx).
std::string rhs_triplets(const u32 *B, int64_t Mc, int r, int64_t N, int right, u32 p, int32_t *Mi, int32_t *Mj, u32 *Mx,
                         int64_t *count, cudaStream_t st)
{
        const int64_t total = Mc * r;
        *count = 0;
        if (total == 0) return "";
        const int64_t chunks = (total + RHS_CHUNK - 1) / RHS_CHUNK;
        if (chunks >= (1ll << 31)) return "right-hand-side block too large";
        u32 *cnt = nullptr;
        u64 *off = nullptr;
        void *tmp = nullptr;
        size_t tb = 0;
        std::string err;
        auto ck = [&](cudaError_t e) {
                if (e != cudaSuccess && err.empty()) err = std::string("right-hand-side triplets: ") + cudaGetErrorString(e);
                return e == cudaSuccess;
        };
        u64 h = 0;
        // per-chunk counts (u32), exclusive sum into u64 offsets: off[chunks] is the total
        if (ck(cudaMalloc(&cnt, sizeof(u32) * (size_t)(chunks + 1))) && ck(cudaMalloc(&off, sizeof(u64) * (size_t)(chunks + 1))) &&
            ck(cudaMemsetAsync(cnt, 0, sizeof(u32) * (size_t)(chunks + 1), st))) {
                k_rhs_count<<<(unsigned)chunks, RHS_TB, 0, st>>>(B, total, p, cnt);
                if (ck(cudaGetLastError()) && ck(cub::DeviceScan::ExclusiveSum(nullptr, tb, cnt, off, chunks + 1, st)) &&
                    ck(cudaMalloc(&tmp, tb ? tb : 4)) && ck(cub::DeviceScan::ExclusiveSum(tmp, tb, cnt, off, chunks + 1, st)) &&
                    ck(cudaMemcpyAsync(&h, off + chunks, sizeof(u64), cudaMemcpyDeviceToHost, st)) && ck(cudaStreamSynchronize(st))) {
                        *count = (int64_t)h;
                        if (Mi) {
                                k_rhs_triplets<<<(unsigned)chunks, RHS_TB, 0, st>>>(B, total, r, N, right, p, off, Mi, Mj, Mx);
                                if (ck(cudaGetLastError())) ck(cudaStreamSynchronize(st));
                        }
                }
        }
        cudaFree(tmp); cudaFree(cnt); cudaFree(off);
        return err;
}

int launch_solve_tail(const SolveArgs &a, int64_t N0, const u32 *v_full, const u32 *map, int64_t n0, int64_t n1, cudaStream_t st)
{
        const int tot = a.r * a.np;
        k_solve_tail<<<(tot + 255) / 256, 256, 0, st>>>(v_full, N0, a.r, a.np, map, n0, n1, a.tail);
        return 1;
}

int launch_solve_small(const SolveArgs &a, cudaStream_t st)
{
        switch (a.np) {
        case 1: return small_np<1>(a, st);
        case 2: return small_np<2>(a, st);
        case 4: return small_np<4>(a, st);
        case 8: return small_np<8>(a, st);
        case 16: return small_np<16>(a, st);
        case 32: return small_np<32>(a, st);
        case 64: return small_np<64>(a, st);
        }
        return -1;
}
