// spmv.cu -- y(R x n) <- S x(C x n) over GF(p) on the interleaved chunk stream.
//
// Replaces sparse_matrix_vector_product (sequential/lanczos_modp.c:266-287): the reference
// scatters from unsorted COO with a read-modify-write of y and a 64-bit `%` per multiply-add.
// Here every output row is produced by a gather over its own entries (no atomics), products
// are accumulated lazily in u64 (modp.cuh) and reduced once per row segment.
//
// Mapping: one warp per tile of G chunks; lane-group g (L lanes, V columns each) walks chunk g.
// Per step the warp issues one coalesced 8-byte-per-group load of {col|LAST, val} and one
// gather of the x row (V*4 bytes per lane, n_pad*4 contiguous bytes per group).  U steps are
// software-unrolled so that U independent gathers are in flight per lane.
// HBM bytes per entry: 8 (matrix) + 4*n_pad (x row, when x does not fit L2) -- see DESIGN.md.
//
// Fused all-gather (PUSH = 1, multi-GPU): the product whose result every GPU needs next writes
// its finished rows not only to the local y but also, over NVLink, into the same rows of every
// peer's copy of the block (plain stores through peer-mapped pointers).  Rows of a tile are
// consecutive, so after its tile a warp re-reads the rows it finalised (L2 hits) and stores them
// to each peer as coalesced runs of up to 512 bytes; the one row a tile may leave open is pushed
// by k_spmv_fix when it completes it.  The exchange thus costs no extra kernel, no SMs of its own
// and is spread evenly over the product -- this replaces the reference's per-iteration
// Send/Recv + Gatherv of the product result (mpi/lanczos_modp.c:1108-1147).
#include <algorithm>
#include <cstdlib>
#include "blk_internal.cuh"
#include "spmv_body.cuh"

namespace {

constexpr int WARPS = 8;     // warps (tiles) per thread block

// back / ready (nullable together): complete the rows that cross tile borders by look-back (see SpOp)
template <int L, int V, int FOLD, int HOT, int PUSH, int ACC = 0>
__global__ void __launch_bounds__(WARPS * 32)
k_spmv(const uint2 *__restrict__ ent, const u32 *__restrict__ chunk_row, u32 *__restrict__ whead,
       int64_t tile0, int64_t ntiles, int Q, u32 rows, const u32 *__restrict__ x, u32 *__restrict__ y, ModP m,
       const DevSmall *__restrict__ state, u32 hot, PushTargets push, const u32 *__restrict__ back, u32 *__restrict__ ready,
       const u32 *__restrict__ rowmap)
{
        pdl_prologue();
        u64 pol_hot = 0, pol_cold = 0;
        if (HOT) {
                asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_hot));
                asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_cold));
        }
        if (state && state->halt) return;
        const int lane = threadIdx.x & 31;
        const int64_t t = tile0 + (int64_t)blockIdx.x * WARPS + (threadIdx.x >> 5);      // tiles [tile0, ntiles)
        if (t >= ntiles) return;
        spmv_tile<L, V, FOLD, HOT, PUSH, 0, ACC>(ent, chunk_row, whead, t, Q, rows, x, y, m, pol_hot, pol_cold, push, back, ready, lane, rowmap);
}

// rows that cross tile borders: y[row] (partial left by the tile where the row starts) plus the
// heads of the `span` following tiles.
template <int L, int V>
__global__ void __launch_bounds__(256)
k_spmv_fix(const u32 *__restrict__ tail_row, const u32 *__restrict__ span, const u32 *__restrict__ whead,
           int64_t scan_lo, int64_t tile_lo, int64_t tile_hi, u32 *__restrict__ y, ModP m,
           const DevSmall *__restrict__ state, PushTargets push, const u32 *__restrict__ rowmap)
{
        pdl_prologue();
        // finishes the rows that END in tiles [tile_lo, tile_hi); such a row starts in a tile >= scan_lo
        constexpr int NP = L * V;
        if (state && state->halt) return;
        int64_t gid = scan_lo + ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / L;
        int sub = threadIdx.x % L;
        if (gid >= tile_hi) return;
        spmv_fix_row<L, V, 0>(tail_row, span, whead, gid, sub, tile_lo, tile_hi, y, m, push, rowmap);
}

template <int L, int V, int HOT, int PUSH>
void launch_hot(const SpOp &op, const ModP &m, const u32 *x, u32 *y, const DevSmall *state, cudaStream_t st,
                int64_t t0, int64_t t1, const PushTargets &push)
{
        unsigned blocks = (unsigned)((t1 - t0 + WARPS - 1) / WARPS);
        if (blocks == 0) return;
        const u32 *back = op.lookback ? op.back : nullptr;
        u32 *ready = op.lookback ? op.ready : nullptr;
        switch (m.fold_every) {
        case 0: launch_k(k_spmv<L, V, 0, HOT, PUSH>, blocks, WARPS * 32, 0, st, op.ent, op.chunk_row, op.whead, t0, t1, op.Q, (u32)op.rows, x, y, m, state, op.hot_cols, push, back, ready, (const u32 *)nullptr); break;
        case 8: launch_k(k_spmv<L, V, 8, HOT, PUSH>, blocks, WARPS * 32, 0, st, op.ent, op.chunk_row, op.whead, t0, t1, op.Q, (u32)op.rows, x, y, m, state, op.hot_cols, push, back, ready, (const u32 *)nullptr); break;
        default: launch_k(k_spmv<L, V, 2, HOT, PUSH>, blocks, WARPS * 32, 0, st, op.ent, op.chunk_row, op.whead, t0, t1, op.Q, (u32)op.rows, x, y, m, state, op.hot_cols, push, back, ready, (const u32 *)nullptr); break;
        }
}

// compact column-band operator (SpOp::rowmap): results are added into y[rowmap[row]]
template <int L, int V>
void launch_acc(const SpOp &op, const ModP &m, const u32 *x, u32 *y, const DevSmall *state, cudaStream_t st)
{
        unsigned blocks = (unsigned)((op.ntiles + WARPS - 1) / WARPS);
        if (blocks == 0) return;
        const PushTargets none;
        switch (m.fold_every) {
        case 0: launch_k(k_spmv<L, V, 0, 0, 0, 1>, blocks, WARPS * 32, 0, st, op.ent, op.chunk_row, op.whead, (int64_t)0, op.ntiles, op.Q, (u32)op.rows, x, y, m, state, 0u, none, (const u32 *)nullptr, (u32 *)nullptr, (const u32 *)op.rowmap); break;
        case 8: launch_k(k_spmv<L, V, 8, 0, 0, 1>, blocks, WARPS * 32, 0, st, op.ent, op.chunk_row, op.whead, (int64_t)0, op.ntiles, op.Q, (u32)op.rows, x, y, m, state, 0u, none, (const u32 *)nullptr, (u32 *)nullptr, (const u32 *)op.rowmap); break;
        default: launch_k(k_spmv<L, V, 2, 0, 0, 1>, blocks, WARPS * 32, 0, st, op.ent, op.chunk_row, op.whead, (int64_t)0, op.ntiles, op.Q, (u32)op.rows, x, y, m, state, 0u, none, (const u32 *)nullptr, (u32 *)nullptr, (const u32 *)op.rowmap); break;
        }
}

template <int L, int V>
int launch_lv(const SpOp &op, const ModP &m, const u32 *x, u32 *y, const DevSmall *state, cudaStream_t st, int piece,
              const PushTargets *push)
{
        if (op.rows <= 0) return 0;                    // an empty shard (more ranks than rows): nothing to produce
        if (op.rowmap) {
                launch_acc<L, V>(op, m, x, y, state, st);
                if (op.crossing)
                        launch_k(k_spmv_fix<L, V>, (unsigned)((op.ntiles * L + 255) / 256), 256, 0, st, op.tail_row, op.span, op.whead, (int64_t)0, (int64_t)0,
                                 op.ntiles, y, m, state, PushTargets(), (const u32 *)op.rowmap);
                return op.crossing ? 2 : 1;
        }
        int64_t t0 = 0, t1 = op.ntiles, scan = 0;
        if (piece >= 0) { t0 = op.piece_tile[piece]; t1 = op.piece_tile[piece + 1]; scan = op.piece_scan[piece]; }
        const PushTargets none;
        const bool hot = V == 4 && op.hot_cols > 0;
        if (push && push->n > 0) {
                if (hot) launch_hot<L, V, 1, 1>(op, m, x, y, state, st, t0, t1, *push);
                else launch_hot<L, V, 0, 1>(op, m, x, y, state, st, t0, t1, *push);
        } else {
                if (hot) launch_hot<L, V, 1, 0>(op, m, x, y, state, st, t0, t1, none);
                else launch_hot<L, V, 0, 0>(op, m, x, y, state, st, t0, t1, none);
        }
        if (op.lookback) return 1;                     // rows crossing tile borders were finished inside k_spmv
        int64_t threads = (t1 - scan) * L;
        if (threads > 0)
                launch_k(k_spmv_fix<L, V>, (unsigned)((threads + 255) / 256), 256, 0, st, op.tail_row, op.span, op.whead, scan, t0, t1, y, m, state,
                                                                                   push ? *push : none, (const u32 *)nullptr);
        return 2;
}

// y <- 0 ahead of accumulate-in-place bands (a kernel, not a memset: a halted iteration must leave y alone)
__global__ void __launch_bounds__(256)
k_zero_block(u32 *__restrict__ y, int64_t count, const DevSmall *__restrict__ state)
{
        pdl_prologue();
        if (state && state->halt) return;
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x) y[e] = 0u;
}

// y[e] = (z_0[e] + ... + z_{K-1}[e]) mod p: the partial results of the column bands of one product
__global__ void __launch_bounds__(256)
k_band_combine(u32 *__restrict__ y, const u32 *__restrict__ z, int K, size_t stride, int64_t count4, ModP m, const DevSmall *__restrict__ state)
{
        pdl_prologue();
        if (state && state->halt) return;
        // (stride and the blocks are multiples of 4 words whenever count4 > 0: rows * n_pad with n_pad = 4, or handled by the tail)
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < count4; e += (int64_t)gridDim.x * blockDim.x) {
                u64 a0 = 0, a1 = 0, a2 = 0, a3 = 0;
                for (int q = 0; q < K; q++) {
                        const uint4 t = __ldcs(reinterpret_cast<const uint4 *>(z + (size_t)q * stride) + e);
                        a0 += t.x; a1 += t.y; a2 += t.z; a3 += t.w;
                }
                reinterpret_cast<uint4 *>(y)[e] = make_uint4(mp_reduce(a0, m), mp_reduce(a1, m), mp_reduce(a2, m), mp_reduce(a3, m));
        }
}
__global__ void __launch_bounds__(256)
k_band_combine1(u32 *__restrict__ y, const u32 *__restrict__ z, int K, size_t stride, int64_t first, int64_t count, ModP m,
                const DevSmall *__restrict__ state)
{
        pdl_prologue();
        if (state && state->halt) return;
        for (int64_t e = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x) {
                u64 a = 0;
                for (int q = 0; q < K; q++) a += z[(size_t)q * stride + e];
                y[e] = mp_reduce(a, m);
        }
}

// y[0, stride) <- sum of the K partial blocks z + b * stride, mod p
int launch_combine(u32 *y, const u32 *z, int K, size_t stride, const ModP &m, const DevSmall *state, cudaStream_t st)
{
        int k = 0;
        const int64_t count = (int64_t)stride;
        const bool vec = (stride % 4) == 0 && ((uintptr_t)y % 16) == 0;
        const int64_t count4 = vec ? count / 4 : 0;
        if (count4 > 0) {
                unsigned blocks = (unsigned)std::min<int64_t>((int64_t)blk_sm_count() * 16, (count4 + 255) / 256);
                launch_k(k_band_combine, blocks, 256, 0, st, y, z, K, stride, count4, m, state);
                k++;
        }
        if (count4 * 4 < count) {
                unsigned blocks = (unsigned)std::min<int64_t>((int64_t)blk_sm_count() * 16, (count - count4 * 4 + 255) / 256);
                launch_k(k_band_combine1, blocks, 256, 0, st, y, z, K, stride, count4 * 4, count, m, state);
                k++;
        }
        return k;
}

}  // namespace

int launch_spmv(const SpOp &op, const Geometry &geo, const ModP &m, const u32 *x, u32 *y,
                const DevSmall *state, cudaStream_t st, int piece, const PushTargets *push)
{
        if (!op.split.empty() && (piece < 0 || op.piece_tile.size() <= 2) && !(push && push->n > 0)) {
                // heavy prefix as column bands (one launch, band after band, into the partial blocks; then the pass that adds
                // them into y[0, H)), then the light rows -- one after the other, so that the light product's random gathers
                // do not evict the bands' x slices
                const size_t stride = (size_t)op.heavy_rows * geo.np;
                int k = launch_spmv(op.split[0], geo, m, x, op.zheavy, state, st);
                k += launch_combine(y, op.zheavy, op.heavy_bands, stride, m, state, st);
                return k + launch_spmv(op.split[1], geo, m, x, y + stride, state, st);
        }
        if (!op.bands.empty() && (piece < 0 || op.piece_tile.size() <= 2) && !(push && push->n > 0)) {
                // column bands: K products whose x slices are L2-resident, then one pass that adds the partial results
                const int K = (int)op.bands.size();
                const size_t stride = (size_t)op.rows * geo.np;
                int k = 0;
                if (!op.zband) {
                        // accumulate-in-place bands over their non-empty rows: clear y, then every band adds its part
                        unsigned blocks = (unsigned)std::min<int64_t>((int64_t)blk_sm_count() * 16, ((int64_t)stride + 255) / 256);
                        if (blocks) { launch_k(k_zero_block, blocks, 256, 0, st, y, (int64_t)stride, state); k++; }
                        for (int b = 0; b < K; b++) k += launch_spmv(op.bands[b], geo, m, x, y, state, st);
                        return k;
                }
                for (int b = 0; b < K; b++) k += launch_spmv(op.bands[b], geo, m, x, op.zband + (size_t)b * stride, state, st);
                return k + launch_combine(y, op.zband, K, stride, m, state, st);
        }
        switch (geo.np) {
        case 1: return launch_lv<1, 1>(op, m, x, y, state, st, piece, push);
        case 2: return launch_lv<1, 2>(op, m, x, y, state, st, piece, push);
        case 4: return launch_lv<1, 4>(op, m, x, y, state, st, piece, push);
        case 8: return launch_lv<2, 4>(op, m, x, y, state, st, piece, push);
        case 16: return launch_lv<4, 4>(op, m, x, y, state, st, piece, push);
        case 32: return launch_lv<8, 4>(op, m, x, y, state, st, piece, push);
        case 64: return launch_lv<16, 4>(op, m, x, y, state, st, piece, push);
        }
        return -1;
}
