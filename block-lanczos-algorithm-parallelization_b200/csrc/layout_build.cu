// layout_build.cu -- COO triplets (struct sparsematrix_t, sequential/lanczos_modp.c:55-62)
// -> GPU-resident interleaved chunk stream (see blk_internal.cuh).  Runs once per operator at
// blk_create time, entirely on the device: key build + radix sort (CUB) + scans + scatter.
// The reference never builds a row-ordered layout (it scatters from COO on every product,
// sequential/lanczos_modp.c:277-286); sorting is legal because results are canonical residues
// and therefore independent of summation order (SURVEY.md F8).
#include <cub/cub.cuh>
#include <cstdlib>
#include <cstring>
#include "blk_internal.cuh"

#define CK(call)                                                                                   \
        do {                                                                                       \
                cudaError_t e_ = (call);                                                           \
                if (e_ != cudaSuccess)                                                             \
                        return std::string(#call) + ": " + cudaGetErrorString(e_);                 \
        } while (0)

namespace {

constexpr int TB = 256;
inline unsigned nblk(int64_t n) { return (unsigned)((n + TB - 1) / TB); }

__global__ void k_make_keys(int64_t nnz, const int32_t *__restrict__ row, const int32_t *__restrict__ col,
                            const u32 *__restrict__ val, int64_t row_lo, int64_t rows, int64_t cols, u32 p,
                            u64 *__restrict__ keys, u32 *__restrict__ vals, u32 *__restrict__ cnt,
                            int *__restrict__ bad, const u32 *__restrict__ row_map, const u32 *__restrict__ col_map)
{
        int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (s >= nnz) return;
        int64_t r = (int64_t)row[s] - row_lo;
        int64_t c = col[s];
        if (r < 0 || r >= rows || c < 0 || c >= cols) {
                *bad = 1;
                r = 0; c = 0;
        }
        if (row_map) r = row_map[r];                 // relabelling (single-GPU: row_lo == 0)
        if (col_map) c = col_map[c];
        keys[s] = ((u64)r << 32) | (u64)c;
        vals[s] = val[s] % p;                       // Mx[u] = x % prime, sequential/lanczos_modp.c:243
        atomicAdd(&cnt[r], 1u);
}

__global__ void k_row_lengths(int64_t rows, const u32 *__restrict__ cnt, u64 *__restrict__ len,
                              u32 *__restrict__ empty)
{
        int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (r > rows) return;
        if (r == rows) { len[r] = 0; return; }
        u32 c = cnt[r];
        len[r] = c ? c : 1;
        empty[r] = c ? 0u : 1u;
}

__device__ __forceinline__ int64_t interleave(int64_t pos, int G, int Q)
{
        int64_t tile = (int64_t)G * Q;
        int64_t t = pos / tile;
        int o = (int)(pos - t * tile);
        int g = o / Q, i = o - g * Q;
        return t * tile + (int64_t)i * G + g;
}

// hot (HotCols::per > 0): bit 30 of the column word marks the x rows that belong to the L2-resident hot prefix of
// their owner's block -- column c is hot iff c - off[w] < per for the block w with off[w] <= c < off[w+1].
__global__ void k_scatter(int64_t nnz, const u64 *__restrict__ keys, const u32 *__restrict__ vals,
                          const u32 *__restrict__ empties_before, uint2 *__restrict__ ent, int G, int Q, HotCols hot)
{
        int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (s >= nnz) return;
        u64 k = keys[s];
        u32 r = (u32)(k >> 32);
        bool last = (s == nnz - 1) || ((u32)(keys[s + 1] >> 32) != r);
        int64_t pos = s + (int64_t)empties_before[r];
        u32 c = (u32)k, flag = 0;
        if (hot.per) {
                int w = 0;
                while (w + 1 < hot.blocks && (int64_t)c >= hot.off[w + 1]) w++;
                if ((int64_t)c - hot.off[w] < (int64_t)hot.per) flag = 0x40000000u;
        }
        ent[interleave(pos, G, Q)] = make_uint2(c | flag | (last ? 0x80000000u : 0u), vals[s]);
}

__global__ void k_dummies(int64_t rows, const u32 *__restrict__ cnt, const u64 *__restrict__ rowptr,
                          uint2 *__restrict__ ent, int G, int Q)
{
        int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (r >= rows || cnt[r]) return;
        ent[interleave((int64_t)rowptr[r], G, Q)] = make_uint2(0x80000000u, 0u);
}

// largest r in [0, rows] with rowptr[r] <= pos   (rowptr has rows+1 entries, non-decreasing)
__device__ __forceinline__ int64_t row_of(const u64 *__restrict__ rowptr, int64_t rows, u64 pos)
{
        int64_t lo = 0, hi = rows;          // invariant rowptr[lo] <= pos
        while (lo < hi) {
                int64_t mid = (lo + hi + 1) >> 1;
                if (rowptr[mid] <= pos) lo = mid; else hi = mid - 1;
        }
        return lo;
}

__global__ void k_chunk_rows(int64_t nchunks, int Q, int64_t stored, int64_t rows,
                             const u64 *__restrict__ rowptr, u32 *__restrict__ chunk_row)
{
        int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (k >= nchunks) return;
        u64 pos = (u64)k * (u64)Q;
        if ((int64_t)pos >= stored) { chunk_row[k] = (u32)rows; return; }   // pure padding
        int64_t r = row_of(rowptr, rows, pos);
        // rows has no zero-length rows (dummies), so rowptr is strictly increasing below `rows`
        u32 open = rowptr[r] < pos ? 0x80000000u : 0u;
        chunk_row[k] = (u32)r | open;
}

__global__ void k_tile_tails(int64_t ntiles, int64_t tile, int64_t stored, int64_t rows,
                             const u64 *__restrict__ rowptr, u32 *__restrict__ tail_row,
                             u32 *__restrict__ span, u32 *__restrict__ back, int *__restrict__ any_crossing)
{
        int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (t >= ntiles) return;
        u32 tr = 0xffffffffu, sp = 0;
        int64_t end = (t + 1) * tile;
        if (end < stored) {
                int64_t r = row_of(rowptr, rows, (u64)(end - 1));
                int64_t rs = (int64_t)rowptr[r], re = (int64_t)rowptr[r + 1];
                if (re > end && rs >= t * tile) {           // row starts in this tile and runs past it
                        tr = (u32)r;
                        sp = (u32)((re - 1) / tile - t);
                }
        }
        tail_row[t] = tr;
        span[t] = sp;
        if (sp) {
                back[t + sp] = sp;          // (a tile finishes at most one such row: the one open at its start)
                *any_crossing = 1;
        }
}

}  // namespace

void free_operator(SpOp *op)
{
        cudaFree(op->ent); cudaFree(op->chunk_row); cudaFree(op->tail_row);
        cudaFree(op->span); cudaFree(op->whead); cudaFree(op->back); cudaFree(op->ready);
        for (auto &b : op->bands) free_operator(&b);
        for (auto &s : op->split) free_operator(&s);
        cudaFree(op->zband); cudaFree(op->rowmap); cudaFree(op->zheavy);
        *op = SpOp();
}

namespace {
__global__ void k_mark_rows(int64_t count, const int32_t *__restrict__ row, int64_t row_lo, u32 *__restrict__ flag)
{
        int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (s < count) flag[(int64_t)row[s] - row_lo] = 1u;
}
__global__ void k_renumber_rows(int64_t count, int32_t *__restrict__ row, int64_t row_lo, const u32 *__restrict__ idx)
{
        int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (s < count) row[s] = (int32_t)idx[(int64_t)row[s] - row_lo];
}
__global__ void k_fill_rowmap(int64_t rows, const u32 *__restrict__ flag, const u32 *__restrict__ idx, u32 *__restrict__ rowmap)
{
        int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (r < rows && flag[r]) rowmap[idx[r]] = (u32)r;
}
}  // namespace

std::string compact_rows(int64_t count, int32_t *d_row, int64_t row_lo, int64_t rows, u32 **rowmap_out, int64_t *nrows_out,
                         cudaStream_t st)
{
        *rowmap_out = nullptr; *nrows_out = 0;
        if (count <= 0 || rows <= 0) return "";
        u32 *flag = nullptr, *idx = nullptr;
        void *tmp = nullptr;
        auto cleanup = [&]() { cudaFree(flag); cudaFree(idx); cudaFree(tmp); };
#define CKR(call)                                                                                  \
        do {                                                                                       \
                cudaError_t e_ = (call);                                                           \
                if (e_ != cudaSuccess) {                                                           \
                        std::string err = std::string(#call) + ": " + cudaGetErrorString(e_);      \
                        cleanup(); cudaFree(*rowmap_out); *rowmap_out = nullptr;                   \
                        return err;                                                                \
                }                                                                                  \
        } while (0)
        CKR(cudaMalloc(&flag, sizeof(u32) * (size_t)(rows + 1)));
        CKR(cudaMalloc(&idx, sizeof(u32) * (size_t)(rows + 1)));
        CKR(cudaMemsetAsync(flag, 0, sizeof(u32) * (size_t)(rows + 1), st));
        k_mark_rows<<<nblk(count), TB, 0, st>>>(count, d_row, row_lo, flag);
        CKR(cudaGetLastError());
        size_t tb = 0;
        CKR(cub::DeviceScan::ExclusiveSum(nullptr, tb, flag, idx, rows + 1, st));
        CKR(cudaMalloc(&tmp, tb ? tb : 16));
        CKR(cub::DeviceScan::ExclusiveSum(tmp, tb, flag, idx, rows + 1, st));
        u32 h = 0;
        CKR(cudaMemcpyAsync(&h, idx + rows, sizeof(u32), cudaMemcpyDeviceToHost, st));
        CKR(cudaStreamSynchronize(st));
        *nrows_out = (int64_t)h;
        CKR(cudaMalloc(rowmap_out, sizeof(u32) * (size_t)(h ? h : 1)));
        k_renumber_rows<<<nblk(count), TB, 0, st>>>(count, d_row, row_lo, idx);
        k_fill_rowmap<<<nblk(rows), TB, 0, st>>>(rows, flag, idx, *rowmap_out);
        CKR(cudaGetLastError());
        CKR(cudaStreamSynchronize(st));
        cleanup();
        return "";
#undef CKR
}

static int pick_chunk_len(int64_t stored, int G)
{
        // aim for >= 8 warps on each of the 148 SMs; cap the chunk so that u64 accumulators never
        // chain more than 64 products (modp.cuh)
        // (config 4, n = 16: Q = 64 14.57 it/s, 32 14.42, 16 13.94 -- longer chunks mean fewer tile
        // borders to stitch; small operators need short chunks to fill the SMs)
        if (stored / ((int64_t)G * 64) >= (int64_t)blk_sm_count() * 32) return 64;
        int Q = 32;
        while (Q > 8 && stored / ((int64_t)G * Q) < (int64_t)blk_sm_count() * 8) Q >>= 1;
        return Q;
}

std::string build_operator(SpOp *op, const Geometry &geo, int chunk_len, int64_t rows, int64_t cols,
                           int64_t row_lo, int64_t nnz, const int32_t *d_row, const int32_t *d_col,
                           const u32 *d_val, u32 prime, const u32 *row_map, const u32 *col_map, int pieces,
                           cudaStream_t st, const HotCols *hot)
{
        *op = SpOp();
        op->rows = rows; op->cols = cols; op->nnz = nnz; op->G = geo.G;
        if (rows >= (1ll << 31) || cols >= (1ll << 31)) return "matrix dimension >= 2^31";
        if (chunk_len != 0 && (chunk_len < 8 || chunk_len > 64 || (chunk_len & (chunk_len - 1))))
                return "chunk_len must be a power of two in [8,64]";
        if (rows == 0) {
                // an empty shard (more ranks than rows): no tiles, one empty piece; launch_spmv skips it
                if (nnz != 0) return "entries given for an operator without rows";
                op->Q = chunk_len ? chunk_len : 8;
                op->piece_tile.assign({0, 0}); op->piece_row.assign({0, 0}); op->piece_scan.assign({0, 0});
                return "";
        }

        u32 *cnt = nullptr, *empty = nullptr, *vals[2] = {nullptr, nullptr};
        u64 *keys[2] = {nullptr, nullptr}, *rowptr = nullptr;
        void *tmp = nullptr;
        int *bad = nullptr;
        std::string err;
        auto cleanup = [&]() {
                cudaFree(cnt); cudaFree(empty); cudaFree(vals[0]); cudaFree(vals[1]);
                cudaFree(keys[0]); cudaFree(keys[1]); cudaFree(rowptr); cudaFree(tmp); cudaFree(bad);
        };
#define CKC(call)                                                                                  \
        do {                                                                                       \
                cudaError_t e_ = (call);                                                           \
                if (e_ != cudaSuccess) {                                                           \
                        err = std::string(#call) + ": " + cudaGetErrorString(e_);                  \
                        cleanup(); free_operator(op);                                              \
                        return err;                                                                \
                }                                                                                  \
        } while (0)

        int64_t nn = nnz > 0 ? nnz : 1;
        CKC(cudaMalloc(&cnt, sizeof(u32) * (size_t)(rows + 1)));
        CKC(cudaMalloc(&empty, sizeof(u32) * (size_t)(rows + 1)));
        CKC(cudaMalloc(&rowptr, sizeof(u64) * (size_t)(rows + 1)));
        CKC(cudaMalloc(&bad, sizeof(int)));
        CKC(cudaMemsetAsync(cnt, 0, sizeof(u32) * (size_t)(rows + 1), st));
        CKC(cudaMemsetAsync(empty, 0, sizeof(u32) * (size_t)(rows + 1), st));
        CKC(cudaMemsetAsync(bad, 0, sizeof(int), st));
        for (int b = 0; b < 2; b++) {
                CKC(cudaMalloc(&keys[b], sizeof(u64) * (size_t)nn));
                CKC(cudaMalloc(&vals[b], sizeof(u32) * (size_t)nn));
        }
        if (nnz > 0) {
                k_make_keys<<<nblk(nnz), TB, 0, st>>>(nnz, d_row, d_col, d_val, row_lo, rows, cols, prime,
                                                      keys[0], vals[0], cnt, bad, row_map, col_map);
                CKC(cudaGetLastError());
        }
        int h_bad = 0;
        CKC(cudaMemcpyAsync(&h_bad, bad, sizeof(int), cudaMemcpyDeviceToHost, st));
        CKC(cudaStreamSynchronize(st));
        if (h_bad) {
                cleanup(); free_operator(op);
                return "matrix entry with row/column index out of range";
        }

        // sort by (row, col)
        cub::DoubleBuffer<u64> dk(keys[0], keys[1]);
        cub::DoubleBuffer<u32> dv(vals[0], vals[1]);
        if (nnz > 1) {
                int rbits = 1;
                while ((1ll << rbits) < rows) rbits++;
                size_t tb = 0;
                CKC(cub::DeviceRadixSort::SortPairs(nullptr, tb, dk, dv, nnz, 0, 32 + rbits, st));
                CKC(cudaMalloc(&tmp, tb ? tb : 16));
                CKC(cub::DeviceRadixSort::SortPairs(tmp, tb, dk, dv, nnz, 0, 32 + rbits, st));
                CKC(cudaStreamSynchronize(st));
                cudaFree(tmp); tmp = nullptr;
        }

        // stored row pointers (every row >= 1 entry) and the number of empty rows before each row
        k_row_lengths<<<nblk(rows + 1), TB, 0, st>>>(rows, cnt, rowptr, empty);
        CKC(cudaGetLastError());
        {
                size_t tb1 = 0, tb2 = 0;
                CKC(cub::DeviceScan::ExclusiveSum(nullptr, tb1, rowptr, rowptr, rows + 1, st));
                CKC(cub::DeviceScan::ExclusiveSum(nullptr, tb2, empty, empty, rows + 1, st));
                size_t tb = tb1 > tb2 ? tb1 : tb2;
                CKC(cudaMalloc(&tmp, tb ? tb : 16));
                CKC(cub::DeviceScan::ExclusiveSum(tmp, tb1, rowptr, rowptr, rows + 1, st));
                CKC(cub::DeviceScan::ExclusiveSum(tmp, tb2, empty, empty, rows + 1, st));
        }
        u64 h_stored = 0;
        CKC(cudaMemcpyAsync(&h_stored, rowptr + rows, sizeof(u64), cudaMemcpyDeviceToHost, st));
        CKC(cudaStreamSynchronize(st));
        cudaFree(tmp); tmp = nullptr;
        op->stored = (int64_t)h_stored;

        op->Q = chunk_len ? chunk_len : pick_chunk_len(op->stored, geo.G);
        int64_t tile = (int64_t)op->G * op->Q;
        op->ntiles = (op->stored + tile - 1) / tile;
        if (op->ntiles < 1) op->ntiles = 1;
        int64_t nchunks = op->ntiles * op->G;
        if (op->ntiles * tile >= (1ll << 40)) { cleanup(); free_operator(op); return "operator too large"; }

        size_t ent_b = sizeof(uint2) * (size_t)(op->ntiles * tile);
        CKC(cudaMalloc(&op->ent, ent_b));
        CKC(cudaMalloc(&op->chunk_row, sizeof(u32) * (size_t)nchunks));
        CKC(cudaMalloc(&op->tail_row, sizeof(u32) * (size_t)op->ntiles));
        CKC(cudaMalloc(&op->span, sizeof(u32) * (size_t)op->ntiles));
        CKC(cudaMalloc(&op->whead, sizeof(u32) * (size_t)op->ntiles * geo.np));
        CKC(cudaMalloc(&op->back, sizeof(u32) * (size_t)op->ntiles));
        CKC(cudaMalloc(&op->ready, sizeof(u32) * (size_t)op->ntiles));
        CKC(cudaMemsetAsync(op->back, 0, sizeof(u32) * (size_t)op->ntiles, st));
        CKC(cudaMemsetAsync(op->ready, 0, sizeof(u32) * (size_t)op->ntiles, st));
        {
                // measured (profiles/r02_spmv_lookback.txt): look-back costs every warp a fence and two more
                // dependent L2 round trips -- slower than the separate fix-up kernel on every configuration, so it is
                // an opt-in (BLK_SPMV_FIX=lookback)
                const char *e = getenv("BLK_SPMV_FIX");
                op->lookback = e && !strcmp(e, "lookback");
        }
        op->bytes = ent_b + sizeof(u32) * (size_t)(nchunks + 4 * op->ntiles + op->ntiles * geo.np);
        CKC(cudaMemsetAsync(op->ent, 0, ent_b, st));
        CKC(cudaMemsetAsync(op->whead, 0, sizeof(u32) * (size_t)op->ntiles * geo.np, st));
        if (nnz > 0) {
                HotCols h;
                if (hot && hot->per > 0 && cols < (1ll << 30)) { h = *hot; op->hot_cols = h.per; }
                k_scatter<<<nblk(nnz), TB, 0, st>>>(nnz, dk.Current(), dv.Current(), empty, op->ent, op->G, op->Q, h);
                CKC(cudaGetLastError());
        }
        k_dummies<<<nblk(rows), TB, 0, st>>>(rows, cnt, rowptr, op->ent, op->G, op->Q);
        CKC(cudaGetLastError());
        k_chunk_rows<<<nblk(nchunks), TB, 0, st>>>(nchunks, op->Q, op->stored, rows, rowptr, op->chunk_row);
        CKC(cudaGetLastError());
        CKC(cudaMemsetAsync(bad, 0, sizeof(int), st));
        k_tile_tails<<<nblk(op->ntiles), TB, 0, st>>>(op->ntiles, tile, op->stored, rows, rowptr,
                                                      op->tail_row, op->span, op->back, bad);
        CKC(cudaGetLastError());
        int h_cross = 0;
        CKC(cudaMemcpyAsync(&h_cross, bad, sizeof(int), cudaMemcpyDeviceToHost, st));
        CKC(cudaStreamSynchronize(st));
        op->crossing = h_cross != 0;

        // ---- row pieces (see SpOp): boundaries at tile multiples; the row that straddles a boundary
        // is finished by the fix-up of the piece in which it ends
        int K = pieces > 1 ? pieces : 1;
        if (op->ntiles < 4 * (int64_t)K) K = 1;
        op->piece_tile.assign(K + 1, 0); op->piece_row.assign(K + 1, 0); op->piece_scan.assign(K + 1, 0);
        op->piece_tile[K] = op->ntiles; op->piece_row[K] = rows;
        for (int k = 1; k < K; k++) op->piece_tile[k] = op->ntiles * k / K;
        for (int k = 0; k <= K; k++) op->piece_scan[k] = op->piece_tile[k];
        for (int k = 1; k < K; k++) {
                u32 cr = 0;
                CKC(cudaMemcpy(&cr, op->chunk_row + op->piece_tile[k] * op->G, sizeof(u32), cudaMemcpyDeviceToHost));
                int64_t r = cr & 0x7fffffffu;
                op->piece_row[k] = r < rows ? r : rows;
                if ((cr >> 31) && r < rows) {             // row r is open across the boundary
                        u64 start = 0;
                        CKC(cudaMemcpy(&start, rowptr + r, sizeof(u64), cudaMemcpyDeviceToHost));
                        int64_t ts = (int64_t)(start / (u64)tile);
                        u32 sp = 0;
                        CKC(cudaMemcpy(&sp, op->span + ts, sizeof(u32), cudaMemcpyDeviceToHost));
                        int64_t te = ts + sp;
                        for (int q = k; q < K && op->piece_tile[q] <= te; q++)
                                if (ts < op->piece_scan[q]) op->piece_scan[q] = ts;
                }
        }
        cleanup();
        return "";
#undef CKC
}

// ---------------------------------------------------------------------------------------------
// Degree-sorted relabelling of one dimension: new label 0 = the index that occurs most often.
// The Lanczos vectors can be stored under any row order (dots are order-free, orthogonalize is
// row-wise); putting the high-degree rows first makes the rows that the product S1 gathers most
// often one contiguous prefix that fits L2 (and packs two hot 64-byte rows per 128-byte line).
// ---------------------------------------------------------------------------------------------
namespace {
__global__ void k_count_index(int64_t nnz, const int32_t *__restrict__ idx, int64_t dim, u32 *__restrict__ cnt)
{
        int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (s >= nnz) return;
        int64_t r = idx[s];
        if (r >= 0 && r < dim) atomicAdd(&cnt[r], 1u);
}
__global__ void k_sort_keys(int64_t dim, const u32 *__restrict__ cnt, u32 *__restrict__ key, u32 *__restrict__ val)
{
        int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (r >= dim) return;
        key[r] = ~cnt[r];            // ascending sort of ~cnt = descending degree; radix sort is stable
        val[r] = (u32)r;
}
__global__ void k_invert_perm(int64_t dim, const u32 *__restrict__ new2old, u32 *__restrict__ old2new)
{
        int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (s >= dim) return;
        old2new[new2old[s]] = (u32)s;
}
// sorted position s -> label of block s % W, place s / W; block w starts at off[w] = sum_{q<w} ceil((dim - q) / W)
__global__ void k_deal_labels(int64_t dim, int W, const u32 *__restrict__ sorted2old, u32 *__restrict__ new2old,
                              u32 *__restrict__ old2new)
{
        int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (s >= dim) return;
        const int w = (int)(s % W);
        // off[w] = sum_{q<w} ceil((dim - q)/W) = w * floor(dim / W) + min(w, dim % W)
        const int64_t off = (int64_t)w * (dim / W) + (w < dim % W ? w : dim % W);
        const u32 lab = (u32)(off + s / W);
        const u32 old = sorted2old[s];
        new2old[lab] = old;
        old2new[old] = lab;
}
}  // namespace

std::string degree_sort_maps(int64_t nnz, const int32_t *d_idx, int64_t dim, u32 **old2new, u32 **new2old,
                             cudaStream_t st, int world, int64_t *block_off)
{
        *old2new = *new2old = nullptr;
        u32 *cnt = nullptr, *key[2] = {nullptr, nullptr}, *val[2] = {nullptr, nullptr};
        void *tmp = nullptr;
        auto cleanup = [&]() { cudaFree(cnt); cudaFree(key[0]); cudaFree(key[1]); cudaFree(val[0]); cudaFree(val[1]); cudaFree(tmp); };
#define CKD(call)                                                                                  \
        do {                                                                                       \
                cudaError_t e_ = (call);                                                           \
                if (e_ != cudaSuccess) {                                                           \
                        std::string err = std::string(#call) + ": " + cudaGetErrorString(e_);      \
                        cleanup(); cudaFree(*old2new); cudaFree(*new2old); *old2new = *new2old = nullptr; \
                        return err;                                                                \
                }                                                                                  \
        } while (0)
        size_t b = sizeof(u32) * (size_t)dim;
        CKD(cudaMalloc(&cnt, b));
        for (int q = 0; q < 2; q++) { CKD(cudaMalloc(&key[q], b)); CKD(cudaMalloc(&val[q], b)); }
        CKD(cudaMalloc(old2new, b));
        CKD(cudaMalloc(new2old, b));
        CKD(cudaMemsetAsync(cnt, 0, b, st));
        if (nnz) k_count_index<<<nblk(nnz), TB, 0, st>>>(nnz, d_idx, dim, cnt);
        k_sort_keys<<<nblk(dim), TB, 0, st>>>(dim, cnt, key[0], val[0]);
        CKD(cudaGetLastError());
        cub::DoubleBuffer<u32> dk(key[0], key[1]), dv(val[0], val[1]);
        size_t tb = 0;
        CKD(cub::DeviceRadixSort::SortPairs(nullptr, tb, dk, dv, dim, 0, 32, st));
        CKD(cudaMalloc(&tmp, tb ? tb : 16));
        CKD(cub::DeviceRadixSort::SortPairs(tmp, tb, dk, dv, dim, 0, 32, st));
        if (world > 1) {
                k_deal_labels<<<nblk(dim), TB, 0, st>>>(dim, world, dv.Current(), *new2old, *old2new);
                for (int w = 0; w <= world && block_off; w++)
                        block_off[w] = w == world ? dim : (int64_t)w * (dim / world) + (w < dim % world ? w : dim % world);
        } else {
                CKD(cudaMemcpyAsync(*new2old, dv.Current(), b, cudaMemcpyDeviceToDevice, st));
                k_invert_perm<<<nblk(dim), TB, 0, st>>>(dim, *new2old, *old2new);
                if (block_off) { block_off[0] = 0; block_off[1] = dim; }
        }
        CKD(cudaGetLastError());
        CKD(cudaStreamSynchronize(st));
        cleanup();
        return "";
#undef CKD
}
