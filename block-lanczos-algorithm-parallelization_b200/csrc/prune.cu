// prune.cu -- removal of empty and singleton constraints before the loop (blk_create_pruned), DESIGN.md section 14.
//
// Unknowns are the coordinates of the Lanczos vectors (rows of M for --left, columns for --right), constraints the
// other dimension.  A triplet counts when x mod p != 0; duplicates are not merged.  cnt(c) is the number of counting
// triplets of constraint c on alive unknowns.  Round r removes D_r = the alive constraints with cnt <= 1 and K_r =
// the lone unknown of each of them with cnt = 1, until D_r is empty.  The kept unknowns and constraints are
// renumbered by rank and M' keeps their counting triplets, in their original order, with the value x mod p.
//
// The kernels:
//
//   k_prune_round0     one pass over the COO: cnt[c] += 1 and lone[c] ^= u for every counting triplet (with cnt = 1,
//                      lone is the one unknown left: removing an unknown is the same XOR again); marks the unknowns
//                      that have a counting triplet (SEEN) and checks the indices
//   k_prune_classify   over the constraints: cnt <= 1 -> cnt = DEAD, killed[lone] = SEEN | r; reports whether any
//                      constraint / unknown died
//   k_prune_decrement  over the triplets: only those whose unknown was stamped in this round and whose constraint is
//                      alive touch the counters
//   k_prune_keep       alive flags (and the free unknowns: never SEEN), turned into new indices by CUB exclusive scans
//   k_prune_index      the original indices of the kept unknowns and constraints
//   k_prune_count / k_prune_select   stable select of the kept triplets, renumbered (count per chunk, scan, write
//                      in order)
#include <cub/cub.cuh>
#include "blk_internal.cuh"

namespace {

constexpr int PR_TB = 256;
constexpr int PR_PER = 8;                         // triplets per thread and chunk of the select
constexpr int64_t PR_CHUNK = (int64_t)PR_TB * PR_PER;
constexpr u32 DEAD = 0xffffffffu;                 // cnt[c] of a removed constraint
constexpr u32 SEEN = 0x80000000u;                 // killed[u]: the unknown has a counting triplet; low bits: round removed

__global__ void __launch_bounds__(PR_TB) k_prune_round0(const int32_t *__restrict__ iu, const int32_t *__restrict__ ic,
                                                        const u32 *__restrict__ x, int64_t nnz, int64_t N, int64_t Mc, u32 p,
                                                        u32 *__restrict__ cnt, u32 *__restrict__ lone, u32 *__restrict__ killed,
                                                        unsigned long long *__restrict__ counting, int *__restrict__ bad)
{
        typedef cub::BlockReduce<unsigned, PR_TB> Reduce;
        __shared__ typename Reduce::TempStorage ts;
        unsigned mine = 0;
        bool oob = false;
        for (int64_t s = (int64_t)blockIdx.x * PR_TB + threadIdx.x; s < nnz; s += (int64_t)gridDim.x * PR_TB) {
                const int32_t u = iu[s], c = ic[s];
                if (u < 0 || u >= N || c < 0 || c >= Mc) { oob = true; continue; }
                if (x[s] % p == 0) continue;
                atomicAdd(&cnt[c], 1u);
                atomicXor(&lone[c], (u32)u);
                killed[u] = SEEN;                 // every writer stores the same word
                mine++;
        }
        const unsigned tot = Reduce(ts).Sum(mine);
        if (__syncthreads_or(oob) && threadIdx.x == 0) *bad = 1;
        if (threadIdx.x == 0 && tot) atomicAdd(counting, (unsigned long long)tot);
}

// flags[0]: some constraint was removed in round r, flags[1]: some unknown
__global__ void __launch_bounds__(PR_TB) k_prune_classify(u32 *__restrict__ cnt, const u32 *__restrict__ lone, int64_t Mc,
                                                          u32 *__restrict__ killed, u32 r, int *__restrict__ flags)
{
        bool died = false, lone_died = false;
        for (int64_t c = (int64_t)blockIdx.x * PR_TB + threadIdx.x; c < Mc; c += (int64_t)gridDim.x * PR_TB) {
                const u32 k = cnt[c];
                if (k > 1) continue;              // alive with two or more, or DEAD
                cnt[c] = DEAD;
                died = true;
                if (k == 1) {
                        killed[lone[c]] = SEEN | r;
                        lone_died = true;
                }
        }
        if (__syncthreads_or(died) && threadIdx.x == 0) flags[0] = 1;
        if (__syncthreads_or(lone_died) && threadIdx.x == 0) flags[1] = 1;
}

__global__ void __launch_bounds__(PR_TB) k_prune_decrement(const int32_t *__restrict__ iu, const int32_t *__restrict__ ic,
                                                           const u32 *__restrict__ x, int64_t nnz, u32 p, u32 *__restrict__ cnt,
                                                           u32 *__restrict__ lone, const u32 *__restrict__ killed, u32 r)
{
        for (int64_t s = (int64_t)blockIdx.x * PR_TB + threadIdx.x; s < nnz; s += (int64_t)gridDim.x * PR_TB) {
                const int32_t u = iu[s];
                if (killed[u] != (SEEN | r)) continue;
                const int32_t c = ic[s];
                if (cnt[c] == DEAD || x[s] % p == 0) continue;
                atomicSub(&cnt[c], 1u);
                atomicXor(&lone[c], (u32)u);
        }
}

// unew[u] = 1 for a kept unknown, cnew[c] = 1 for a kept constraint (one extra zero each for the scan total);
// *nfree counts the unknowns without any counting triplet (they are never removed)
__global__ void __launch_bounds__(PR_TB) k_prune_keep(const u32 *__restrict__ killed, int64_t N, const u32 *__restrict__ cnt,
                                                      int64_t Mc, u32 *__restrict__ unew, u32 *__restrict__ cnew,
                                                      unsigned long long *__restrict__ nfree)
{
        typedef cub::BlockReduce<unsigned, PR_TB> Reduce;
        __shared__ typename Reduce::TempStorage ts;
        unsigned mine = 0;
        const int64_t top = (N > Mc ? N : Mc) + 1;
        for (int64_t e = (int64_t)blockIdx.x * PR_TB + threadIdx.x; e < top; e += (int64_t)gridDim.x * PR_TB) {
                if (e <= N) {
                        const u32 k = e < N ? killed[e] : 1u;
                        unew[e] = e < N && (k & ~SEEN) == 0 ? 1u : 0u;
                        mine += k == 0;
                }
                if (e <= Mc) cnew[e] = e < Mc && cnt[e] != DEAD ? 1u : 0u;
        }
        const unsigned tot = Reduce(ts).Sum(mine);
        if (threadIdx.x == 0 && tot) atomicAdd(nfree, (unsigned long long)tot);
}

// after the scans: unew / cnew are the new indices; the kept ones write their original index there
__global__ void __launch_bounds__(PR_TB) k_prune_index(const u32 *__restrict__ killed, int64_t N, const u32 *__restrict__ cnt,
                                                       int64_t Mc, const u32 *__restrict__ unew, const u32 *__restrict__ cnew,
                                                       int32_t *__restrict__ uidx, int32_t *__restrict__ cidx)
{
        const int64_t top = N > Mc ? N : Mc;
        for (int64_t e = (int64_t)blockIdx.x * PR_TB + threadIdx.x; e < top; e += (int64_t)gridDim.x * PR_TB) {
                if (e < N && (killed[e] & ~SEEN) == 0) uidx[unew[e]] = (int32_t)e;
                if (e < Mc && cnt[e] != DEAD) cidx[cnew[e]] = (int32_t)e;
        }
}

__device__ __forceinline__ bool kept(int64_t s, const int32_t *iu, const int32_t *ic, const u32 *x, u32 p, const u32 *killed,
                                     const u32 *cnt)
{
        return x[s] % p != 0 && (killed[iu[s]] & ~SEEN) == 0 && cnt[ic[s]] != DEAD;
}

__global__ void __launch_bounds__(PR_TB) k_prune_count(const int32_t *__restrict__ iu, const int32_t *__restrict__ ic,
                                                       const u32 *__restrict__ x, int64_t nnz, u32 p, const u32 *__restrict__ killed,
                                                       const u32 *__restrict__ cnt, u32 *__restrict__ per_chunk)
{
        const int64_t base = (int64_t)blockIdx.x * PR_CHUNK;
        int k = 0;
        for (int q = 0; q < PR_PER; q++) {
                const int64_t s = base + (int64_t)q * PR_TB + threadIdx.x;
                k += __syncthreads_count(s < nnz && kept(s, iu, ic, x, p, killed, cnt));
        }
        if (threadIdx.x == 0) per_chunk[blockIdx.x] = (u32)k;
}

// the kept triplets of the chunk at off[chunk] + (their rank in the chunk), renumbered, value x mod p
__global__ void __launch_bounds__(PR_TB) k_prune_select(const int32_t *__restrict__ iu, const int32_t *__restrict__ ic,
                                                        const u32 *__restrict__ x, int64_t nnz, u32 p, const u32 *__restrict__ killed,
                                                        const u32 *__restrict__ cnt, const u32 *__restrict__ unew,
                                                        const u32 *__restrict__ cnew, const u64 *__restrict__ off,
                                                        int32_t *__restrict__ ou, int32_t *__restrict__ oc, u32 *__restrict__ ox)
{
        typedef cub::BlockScan<int, PR_TB> Scan;
        __shared__ typename Scan::TempStorage ts;
        const int64_t base = (int64_t)blockIdx.x * PR_CHUNK;
        u64 at = off[blockIdx.x];
        for (int q = 0; q < PR_PER; q++) {
                const int64_t s = base + (int64_t)q * PR_TB + threadIdx.x;
                const bool keep = s < nnz && kept(s, iu, ic, x, p, killed, cnt);
                int pos = 0, sum = 0;
                Scan(ts).ExclusiveSum(keep ? 1 : 0, pos, sum);
                if (keep) {
                        ou[at + pos] = (int32_t)unew[iu[s]];
                        oc[at + pos] = (int32_t)cnew[ic[s]];
                        ox[at + pos] = x[s] % p;
                }
                at += (u64)sum;
                __syncthreads();                          // ts is reused by the next pass
        }
}

}  // namespace

void PruneResult::release()
{
        cudaFree(Mi); cudaFree(Mj); cudaFree(Mx);
        Mi = Mj = nullptr; Mx = nullptr;
}

std::string prune_coo(const int32_t *Mi, const int32_t *Mj, const u32 *Mx, int64_t nnz, int64_t nrows, int64_t ncols, int right,
                      u32 p, cudaStream_t st, PruneResult *out)
{
        const int64_t N = right ? ncols : nrows, Mc = right ? nrows : ncols;
        const int32_t *iu = right ? Mj : Mi, *ic = right ? Mi : Mj;
        std::vector<void *> bufs;
        std::string err;
        auto ck = [&](cudaError_t e) {
                if (e != cudaSuccess && err.empty()) err = std::string("pruning: ") + cudaGetErrorString(e);
                return e == cudaSuccess;
        };
        auto grab = [&](void **dst, size_t bytes) {
                if (!ck(cudaMalloc(dst, bytes ? bytes : 16))) return false;
                bufs.push_back(*dst);
                return true;
        };
        struct Free {
                std::vector<void *> &b;
                ~Free() { for (void *q : b) cudaFree(q); }
        } free_all{bufs};
        int dev = 0, sms = 148;
        if (!ck(cudaGetDevice(&dev)) || !ck(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev))) return err;
        auto grid = [&](int64_t work) { return (unsigned)std::max<int64_t>(1, std::min<int64_t>((work + PR_TB - 1) / PR_TB, (int64_t)sms * 16)); };

        u32 *cnt = nullptr, *lone = nullptr, *killed = nullptr, *unew = nullptr, *cnew = nullptr;
        unsigned long long *acc = nullptr;       // [0] counting triplets, [1] free unknowns
        int *flags = nullptr;                    // [0] bad index, [1] [2] classify
        if (!grab((void **)&cnt, sizeof(u32) * (size_t)Mc) || !grab((void **)&lone, sizeof(u32) * (size_t)Mc) ||
            !grab((void **)&killed, sizeof(u32) * (size_t)N) || !grab((void **)&acc, 2 * sizeof(unsigned long long)) || !grab((void **)&flags, 3 * sizeof(int)))
                return err;
        if (!ck(cudaMemsetAsync(cnt, 0, sizeof(u32) * (size_t)Mc, st)) || !ck(cudaMemsetAsync(lone, 0, sizeof(u32) * (size_t)Mc, st)) ||
            !ck(cudaMemsetAsync(killed, 0, sizeof(u32) * (size_t)N, st)) || !ck(cudaMemsetAsync(acc, 0, 2 * sizeof(unsigned long long), st)) ||
            !ck(cudaMemsetAsync(flags, 0, 3 * sizeof(int), st)))
                return err;

        // ---- round 0
        if (nnz > 0) k_prune_round0<<<grid(nnz), PR_TB, 0, st>>>(iu, ic, Mx, nnz, N, Mc, p, cnt, lone, killed, acc, flags);
        int hf[3] = {0, 0, 0};
        unsigned long long hacc[2] = {0, 0};
        if (!ck(cudaGetLastError()) || !ck(cudaMemcpyAsync(hf, flags, sizeof(int), cudaMemcpyDeviceToHost, st)) ||
            !ck(cudaMemcpyAsync(hacc, acc, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st)) || !ck(cudaStreamSynchronize(st)))
                return err;
        if (hf[0]) return "matrix entry with row/column index out of range";
        const int64_t counting = (int64_t)hacc[0];

        // ---- rounds: one host synchronisation each
        int64_t rounds = 0;
        for (u32 r = 1;; r++) {
                if (!ck(cudaMemsetAsync(flags + 1, 0, 2 * sizeof(int), st))) return err;
                k_prune_classify<<<grid(Mc), PR_TB, 0, st>>>(cnt, lone, Mc, killed, r, flags + 1);
                if (!ck(cudaGetLastError()) || !ck(cudaMemcpyAsync(hf + 1, flags + 1, 2 * sizeof(int), cudaMemcpyDeviceToHost, st)) ||
                    !ck(cudaStreamSynchronize(st)))
                        return err;
                if (!hf[1]) break;
                rounds = r;
                if (hf[2]) {
                        k_prune_decrement<<<grid(nnz), PR_TB, 0, st>>>(iu, ic, Mx, nnz, p, cnt, lone, killed, r);
                        if (!ck(cudaGetLastError())) return err;
                }
        }

        // ---- compaction: new indices, index maps, renumbered M'
        if (!grab((void **)&unew, sizeof(u32) * (size_t)(N + 1)) || !grab((void **)&cnew, sizeof(u32) * (size_t)(Mc + 1))) return err;
        k_prune_keep<<<grid(std::max(N, Mc) + 1), PR_TB, 0, st>>>(killed, N, cnt, Mc, unew, cnew, acc + 1);
        if (!ck(cudaGetLastError())) return err;
        void *tmp = nullptr;
        size_t tb1 = 0, tb2 = 0;
        if (!ck(cub::DeviceScan::ExclusiveSum(nullptr, tb1, unew, unew, N + 1, st)) ||
            !ck(cub::DeviceScan::ExclusiveSum(nullptr, tb2, cnew, cnew, Mc + 1, st)) || !grab((void **)&tmp, std::max(tb1, tb2)) ||
            !ck(cub::DeviceScan::ExclusiveSum(tmp, tb1, unew, unew, N + 1, st)) ||
            !ck(cub::DeviceScan::ExclusiveSum(tmp, tb2, cnew, cnew, Mc + 1, st)))
                return err;
        u32 nkeep[2] = {0, 0};
        if (!ck(cudaMemcpyAsync(&nkeep[0], unew + N, sizeof(u32), cudaMemcpyDeviceToHost, st)) ||
            !ck(cudaMemcpyAsync(&nkeep[1], cnew + Mc, sizeof(u32), cudaMemcpyDeviceToHost, st)) ||
            !ck(cudaMemcpyAsync(&hacc[1], acc + 1, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st)) ||
            !ck(cudaStreamSynchronize(st)))
                return err;
        out->N = nkeep[0]; out->Mc = nkeep[1]; out->free = (int64_t)hacc[1]; out->rounds = rounds;
        if (out->N == N && out->Mc == Mc) {
                // nothing removed: the index maps are the identity (not stored)
                out->identity = true;
                if (counting == nnz) {
                        // and no triplet vanishes mod p: M' is M (blk_create reduces the values itself)
                        out->nnz = nnz;
                        return err;
                }
        } else {
                out->unknowns.resize((size_t)out->N);
                out->constraints.resize((size_t)out->Mc);
                int32_t *uidx = nullptr, *cidx = nullptr;
                if (!grab((void **)&uidx, sizeof(int32_t) * (size_t)out->N) || !grab((void **)&cidx, sizeof(int32_t) * (size_t)out->Mc))
                        return err;
                k_prune_index<<<grid(std::max(N, Mc)), PR_TB, 0, st>>>(killed, N, cnt, Mc, unew, cnew, uidx, cidx);
                if (!ck(cudaGetLastError()) ||
                    !ck(cudaMemcpyAsync(out->unknowns.data(), uidx, sizeof(int32_t) * (size_t)out->N, cudaMemcpyDeviceToHost, st)) ||
                    !ck(cudaMemcpyAsync(out->constraints.data(), cidx, sizeof(int32_t) * (size_t)out->Mc, cudaMemcpyDeviceToHost, st)))
                        return err;
        }
        const int64_t chunks = (nnz + PR_CHUNK - 1) / PR_CHUNK;
        if (chunks >= (1ll << 31)) return "pruning: too many matrix entries";
        u32 *per_chunk = nullptr;
        u64 *off = nullptr, total = 0;
        size_t tb = 0;
        if (!grab((void **)&per_chunk, sizeof(u32) * (size_t)(chunks + 1)) || !grab((void **)&off, sizeof(u64) * (size_t)(chunks + 1)) ||
            !ck(cudaMemsetAsync(per_chunk, 0, sizeof(u32) * (size_t)(chunks + 1), st)))
                return err;
        if (chunks) k_prune_count<<<(unsigned)chunks, PR_TB, 0, st>>>(iu, ic, Mx, nnz, p, killed, cnt, per_chunk);
        if (!ck(cudaGetLastError()) || !ck(cub::DeviceScan::ExclusiveSum(nullptr, tb, per_chunk, off, chunks + 1, st)))
                return err;
        void *tmp2 = nullptr;
        if (!grab((void **)&tmp2, tb) || !ck(cub::DeviceScan::ExclusiveSum(tmp2, tb, per_chunk, off, chunks + 1, st)) ||
            !ck(cudaMemcpyAsync(&total, off + chunks, sizeof(u64), cudaMemcpyDeviceToHost, st)) || !ck(cudaStreamSynchronize(st)))
                return err;
        out->nnz = (int64_t)total;
        int32_t *oi = nullptr, *oj = nullptr;
        u32 *ox = nullptr;
        if (!ck(cudaMalloc(&oi, sizeof(int32_t) * (size_t)std::max<u64>(total, 1)))) return err;
        out->Mi = oi;
        if (!ck(cudaMalloc(&oj, sizeof(int32_t) * (size_t)std::max<u64>(total, 1)))) return err;
        out->Mj = oj;
        if (!ck(cudaMalloc(&ox, sizeof(u32) * (size_t)std::max<u64>(total, 1)))) return err;
        out->Mx = ox;
        if (chunks)
                k_prune_select<<<(unsigned)chunks, PR_TB, 0, st>>>(iu, ic, Mx, nnz, p, killed, cnt, unew, cnew, off, right ? oj : oi,
                                                                   right ? oi : oj, ox);
        if (ck(cudaGetLastError())) ck(cudaStreamSynchronize(st));
        return err;
}
