// blk_internal.cuh -- shared declarations of the CUDA implementation behind include/blk_lanczos.h
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <cstdlib>
#include <string>
#include <utility>
#include <vector>
#include "modp.cuh"

// ----------------------------------------------------------------------------------------------
// Sparse operator layout ("interleaved chunk stream")
//
// One operator S (R x C) computes y(R x n) <- S x(C x n).  Its entries are stored row by row
// (rows sorted, columns ascending inside a row); an empty row contributes one dummy entry
// (col 0, val 0) so that every row owns at least one stored entry.  Each stored entry is a
// uint2 {col | LAST<<31, val}; LAST marks the final entry of a row.
//
// The stream is cut into chunks of Q consecutive entries.  A lane-group (L lanes, L = n_pad/4
// for n_pad >= 4, each lane owning V = n_pad/L columns) walks one chunk sequentially.  A warp
// holds G = 32/L lane-groups, i.e. a tile of G*Q consecutive entries.  Inside a tile the entries
// are interleaved, entry i of chunk g at offset i*G + g, so that at step i the warp's G groups
// read G consecutive uint2 -- one coalesced request, every byte of the matrix is read exactly
// once and no shared-memory staging is needed.
//
// Work is balanced by entries, not rows (power-law rows cost nothing extra).  Rows that
// cross chunk borders are stitched with warp shuffles; rows that cross tile borders leave a
// partial in y and one n-vector per tile in `whead`, completed by a small fix-up kernel.
// ----------------------------------------------------------------------------------------------
struct SpOp {
        int64_t rows = 0;          // R: output rows (local rows of this rank)
        int64_t cols = 0;          // C: input rows (global)
        int64_t nnz = 0;           // real entries
        int64_t stored = 0;        // nnz + empty-row dummies
        int64_t ntiles = 0;        // warp tiles (stored padded up to ntiles*G*Q)
        int Q = 0, G = 0;
        uint2 *ent = nullptr;      // [ntiles*G*Q]
        u32 *chunk_row = nullptr;  // [ntiles*G]  first row of the chunk | HEAD_OPEN<<31
        u32 *tail_row = nullptr;   // [ntiles]    row left open at the end of the tile (started in it)
        u32 *span = nullptr;       // [ntiles]    number of following tiles that finish that row (0: none)
        u32 *whead = nullptr;      // [ntiles*n_pad] scratch: the tile's contribution to a row opened earlier
        // Look-back completion of rows that cross tile borders (inside k_spmv, no second kernel): the tile in which such a
        // row ENDS adds up the partial left in y by the tile where it started and the whead of the tiles in between.
        u32 *back = nullptr;       // [ntiles]    > 0: the row open at the start of this tile ends in it and started `back` tiles earlier
        u32 *ready = nullptr;      // [ntiles]    flag: the tile's part of the row open at its end is in memory (reset by the finisher)
        bool crossing = false;     // some row crosses a tile border (k_spmv_fix / look-back has work to do)
        bool lookback = false;     // true (BLK_SPMV_FIX=lookback): finish those rows inside k_spmv; default: k_spmv_fix (faster, measured)
        size_t bytes = 0;
        // Row pieces for pipelining a product with the exchange of its result (multi-GPU): piece q is
        // tiles [piece_tile[q], piece_tile[q+1]); after its fix-up, rows [piece_row[q], piece_row[q+1])
        // are final.  piece_scan[q] <= piece_tile[q] is the first tile whose open row ends in piece q.
        std::vector<int64_t> piece_tile, piece_row, piece_scan;
        // Column bands (small n_pad, x block >> L2): the operator is ALSO stored as `bands.size()` operators over all rows, band b
        // holding the entries whose column lies in [band_col[b], band_col[b+1]) -- a slice of x that stays L2-resident while its
        // band runs, so its gathers hit L2 instead of pulling one 128-byte HBM line each.  Every band writes a partial
        // result into zband (rows * n_pad words per band); k_band_combine adds them mod p.  launch_spmv dispatches here.
        // Two forms: (a) every band covers all rows and writes a partial result into zband (rows * n_pad words per band), added up
        // by k_band_combine; (b) zband == nullptr: every band is a COMPACT operator over the rows that have entries in it (rowmap:
        // its row r is row rowmap[r] of y) whose kernel ADDS its result to y, cleared beforehand -- no partial blocks, no dummy
        // entries for rows that are empty inside a band.
        std::vector<SpOp> bands;
        std::vector<int64_t> band_col;
        u32 *zband = nullptr;
        u32 *rowmap = nullptr;     // this operator is a compact band: output row r -> y row rowmap[r], results accumulate
        u32 hot_cols = 0;          // > 0: entries carry a HOT bit (bit 30 of the column word): those x rows are gathered with
                                   // L2 evict_last, the rest evict_first (columns are then limited to 2^30)
        // Heavy/light split (product 2, n_pad >= 8, one GPU, degree-sorted rows): the operator is ALSO stored as two operators.
        // split[0] holds the high-degree row prefix [0, H) cut into heavy_bands = K column bands as ONE stream over K * H
        // virtual rows, row b * H + r = (band b, row r): its output rows are the K band-major partial blocks in zheavy
        // (H * n_pad words each), its tiles run band after band in one launch, and k_band_combine adds the partials into
        // y[0, H).  split[1] is an ordinary operator over rows [H, rows) whose output starts at row H.  A partial costs
        // n_pad words per heavy row and band, while the band's L2-resident x slice saves a line per non-zero.  launch_spmv
        // dispatches here for unpieced, unpushed calls; everything else keeps using the full operator.
        std::vector<SpOp> split;
        int64_t heavy_rows = 0;
        int heavy_bands = 0;
        u32 *zheavy = nullptr;
};

// The heavy prefix of product 2 (SpOp::split): rows whose degree is >= min_deg, run as column bands of band_bytes of x each.
// deg: row degrees under the degree-sorted labels (non-increasing).  force: skip the size and cost checks (tests).
struct HeavyPlan {
        int64_t rows = 0;          // H (0: no split)
        int bands = 0;             // K
};
HeavyPlan plan_heavy(const u32 *deg, int64_t rows, int64_t cols, int np, int64_t l2_bytes, int64_t min_deg, int64_t band_bytes,
                     bool force);

// n x n working set of one iteration, resident on the device.  All matrices are stored with
// leading dimension n_pad (zero padded) so the row kernels can use them directly.
struct DevSmall {
        int iters;        // the reference's n_iterations
        int limit;        // blk_iterate: stop when iters == limit (<=0: no limit)
        int stopped;      // semi_inverse returned 0 pivots
        int halt;         // skip whole iterations (stopped or limit reached)
        int do_ortho;     // set by the small kernel of the current iteration
        int npiv;         // last semi_inverse return value
        int bad_index;    // layout build: COO index out of range
        int check;        // BLK_CHECK=1: evaluate the reference's correctness_tests in the n x n stage
        int check_failed; // bit mask of the violated invariants (the loop halts; blk_iterate reports it)
        int fault_iter;   // BLK_CHECK_FAULT=k (with BLK_CHECK=1): corrupt vtAv in iteration k, to test the self-check
};

struct Geometry {
        int n = 0, np = 0;      // blocking factor and its power-of-two padding
        int L = 0, V = 0, G = 0; // lanes per entry, u32 per lane, groups per warp
};

static inline Geometry make_geometry(int n)
{
        Geometry g;
        g.n = n;
        int np = 1;
        while (np < n) np <<= 1;
        g.np = np;
        g.V = np < 4 ? np : 4;
        g.L = np / g.V;
        g.G = 32 / g.L;
        return g;
}

// number of SMs of the current device (cached per ordinal): grids are sized in multiples of it
static inline int blk_sm_count()
{
        static int cache[64] = {0};
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
        if (!cache[dev]) {
                int n = 0;
                if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
                cache[dev] = n;
        }
        return cache[dev];
}

// ---- programmatic dependent launch -------------------------------------------------------------
// The kernels of one iteration form a chain in one stream (or one CUDA graph).  Every one of them starts with
// pdl_prologue(): "launch_dependents" lets the next kernel of the chain be scheduled -- its blocks become
// resident and run their own prologue -- while this one is still working, and "wait" blocks until the
// previous kernel has finished and its writes are visible.  Nothing is read or written before the wait, so
// the results are those of the serial chain; what disappears is the launch latency between two kernels,
// which is most of an iteration on the L2-resident configurations (BASELINE configs 1-3).
// launch_k() launches with the attribute that allows this overlap when BLK_PDL=1.  Measured on configs 1-3
// (gpurun_out/r2_e_small_pdl*.json, profiles/r02_small_configs.txt): 26.1 / 43.6 / 72.1 us per iteration with it,
// 25.0 / 41.4 / 73.6 without -- inside a CUDA graph the gap between two kernel nodes is already hidden, what an
// iteration pays is the latency chain inside each of its six kernels.  So the overlap is OFF by default.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_prologue()
{
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        asm volatile("griddepcontrol.wait;" ::: "memory");
}

static inline bool blk_pdl_enabled()
{
        static int on = -1;
        if (on < 0) {
                const char *e = getenv("BLK_PDL");
                on = e && e[0] == '1';
        }
        return on != 0;
}

template <class... KArgs, class... Args>
static inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args)
{
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = blk_pdl_enabled() ? 1 : 0;
        cfg.attrs = attr; cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, kernel, KArgs(std::forward<Args>(args))...);
}
#endif

// Which x rows of an operator are "hot" (the high-degree prefix of every rank's block of a degree-sorted dimension):
// column c is hot iff c - off[w] < per, w = the block with off[w] <= c < off[w+1].  per == 0: no hot rows.
struct HotCols {
        static constexpr int MAXB = 64;
        int blocks = 0;
        u32 per = 0;
        int64_t off[MAXB + 1] = {0};
};

// ---- launchers (each returns the number of kernels it launched) ---------------------------
// layout_build.cu
std::string build_operator(SpOp *op, const Geometry &geo, int chunk_len, int64_t rows, int64_t cols,
                           int64_t row_lo, int64_t nnz, const int32_t *d_row, const int32_t *d_col,
                           const u32 *d_val, u32 prime, const u32 *row_map, const u32 *col_map, int pieces,
                           cudaStream_t st, const HotCols *hot = nullptr);
void free_operator(SpOp *op);
// Renumber the row keys of `count` entries (global keys in [row_lo, row_lo + rows)) to 0 .. R-1 over the rows that occur, in
// increasing order; *rowmap_out (device, R words) maps the new numbers back to local rows (key - row_lo).
std::string compact_rows(int64_t count, int32_t *d_row, int64_t row_lo, int64_t rows, u32 **rowmap_out, int64_t *nrows_out,
                         cudaStream_t st);
// old->new / new->old labels of one dimension sorted by decreasing number of entries; world > 1: the sorted
// sequence is then dealt round-robin to `world` contiguous blocks (position s of the sorted order goes to block
// s % world, place s / world), so that every block gets the same share of heavy rows -- equal rows, equal
// non-zeros, and its own hot prefix; block_off[world + 1] receives the block boundaries.
std::string degree_sort_maps(int64_t nnz, const int32_t *d_idx, int64_t dim, u32 **old2new, u32 **new2old,
                             cudaStream_t st, int world = 1, int64_t *block_off = nullptr);

// Peer copies of an output block (multi-GPU, peer-mapped device pointers): y[q] addresses the same
// row origin on peer q as the local output pointer of the launch, so a finished row r goes to
// y[q] + r*n_pad on every peer.
struct PushTargets {
        static constexpr int MAX = 7;
        int n = 0;
        u32 *y[MAX] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

// spmv.cu
// piece < 0: the whole operator; else only tiles (and the fix-up) of that row piece.
// push (nullable): also store every finished row into the peers' copies (fused all-gather).
int launch_spmv(const SpOp &op, const Geometry &geo, const ModP &m, const u32 *x, u32 *y,
                const DevSmall *state, cudaStream_t st, int piece = -1, const PushTargets *push = nullptr);

// dense.cu
int dots_num_blocks(int64_t rows, int np);
// When `counter` is non-null the dot-product kernel's last block to finish also runs the n x n
// stage (k_small mode 0) -- one launch less per iteration (single-GPU loop only).
struct SmallFuse {
        unsigned *counter = nullptr;
        u32 *mats = nullptr;
        DevSmall *state = nullptr;
        int n = 0;
};
// dots adds its per-block results (canonical residues) into the u64 accumulators sums[2*np*np]
int launch_dots(const Geometry &geo, const ModP &m, int64_t rows, const u32 *v, const u32 *Av,
                u64 *sums, int nblocks, const DevSmall *state, const SmallFuse &fuse, cudaStream_t st);
// mats layout (u32, each np*np unless noted): [0] vtAv [1] vtAAv [2] winv [3] c [4] vtAvd [5] d (np)
enum { MAT_VTAV = 0, MAT_VTAAV = 1, MAT_WINV = 2, MAT_C = 3, MAT_VTAVD = 4, MAT_D = 5, MAT_COUNT = 6 };
// One block.  mode 0: full iteration step (reduce sums mod p and clear them, semi_inverse,
// coefficients, loop flags); 1: only reduce sums into MAT_VTAV/MAT_VTAAV; 2: semi_inverse of
// MAT_VTAV only; 3: coefficients from given MAT_D/MAT_WINV/MAT_VTAV/MAT_VTAAV.
int launch_small(const Geometry &geo, const ModP &m, u64 *sums, u32 *mats, DevSmall *state, int mode,
                 cudaStream_t st);
int launch_ortho(const Geometry &geo, const ModP &m, int64_t rows, u32 *v, const u32 *Av, u32 *p,
                 u32 *v_out, u32 *p_out, const u32 *mats, const DevSmall *state, int force,
                 cudaStream_t st);
// dense_mma.cu: int8 tensor-core versions of dots / ortho for n_pad in {8,16,32}.  The ortho
// kernel reads its right-hand operands from `bfrag`, stored behind the MAT_COUNT matrices of
// `mats` in MMA fragment order (written by k_small): word index
//   ((((X*4 + b)*T + t)*S + s)*32 + lane)*2 + h,   X in {c, vtAvd, winv}, T = S = np/8,
// holding, for byte beta = 0..3, limb b of (2^(8 beta) * X[w][j] mod p) with j = 8t + (lane>>2)
// and w = (lane&3)*np/4 + 2s + h.
bool dense_mma_supported(int np);
void dense_mma_prepare(int np);
static inline size_t bfrag_words(int np) { return (np >= 8 && np <= 32) ? (size_t)12 * (np / 8) * (np / 8) * 64 : 0; }
static inline size_t mats_words(int np) { return (size_t)MAT_COUNT * np * np + bfrag_words(np); }
int launch_ortho_mma(int np, const ModP &m, int64_t rows, u32 *v, const u32 *Av, u32 *p, u32 *v_out, u32 *p_out,
                     const u32 *mats, const DevSmall *state, int force, cudaStream_t st);
int launch_dots_mma(int np, const ModP &m, int64_t rows, const u32 *v, const u32 *Av, u64 *sums,
                    const DevSmall *state, const SmallFuse &fuse, cudaStream_t st);
// dense_umma.cu: tcgen05/TMEM/TMA versions for n_pad = 16 (opt-in: BLK_DENSE=umma | umma64).
// `wide` < 0 follows BLK_DENSE; 1: one M = 128 instruction for both products, 0: two M = 64.
bool dense_umma_supported(int np, int64_t rows);
void dense_umma_prepare(int np);
int launch_dots_umma(int np, const ModP &m, int64_t rows, const u32 *v, const u32 *Av, u64 *sums,
                     const DevSmall *state, const SmallFuse &fuse, cudaStream_t st, int wide = -1);
int launch_ortho_umma(int np, const ModP &m, int64_t rows, u32 *v, const u32 *Av, u32 *p, u32 *v_out, u32 *p_out,
                      const u32 *mats, const DevSmall *state, int force, cudaStream_t st, int variant = -1);
// loop_coop.cu: the whole loop as one persistent cooperative kernel (single GPU, L2-resident problems, n_pad <= 16)
struct LoopOp {
        const uint2 *ent = nullptr;
        const u32 *chunk_row = nullptr;
        u32 *whead = nullptr;
        const u32 *tail_row = nullptr, *span = nullptr;
        int64_t ntiles = 0;
        int Q = 0;
        u32 rows = 0;
        int crossing = 0;          // some row crosses a tile border: the fix-up phase (and its barrier) is needed
};
struct LoopArgs {
        LoopOp s1, s2;             // tmp <- S1 v ; Av <- S2 tmp
        u32 *v = nullptr, *tmp = nullptr, *Av = nullptr, *p = nullptr;
        int64_t N = 0;
        unsigned long long *sums = nullptr;
        u32 *mats = nullptr;
        DevSmall *state = nullptr;
        ModP m;
        int n = 0, max_iters = 0;
        unsigned *bar = nullptr;   // two words: arrivals, release word of the serial barrier
        unsigned long long *prof = nullptr;      // nullable: six phase clocks of block 0 (SM cycles, accumulated)
};
bool loop_coop_supported(int np);
// thread blocks of the persistent kernel (0 + *why when it cannot run on the current device)
int loop_coop_grid(int n, int np, const ModP &m, std::string *why);
int launch_loop_coop(const LoopArgs &args, int n, int np, int grid, cudaStream_t st, std::string *err);
// per-device one-time kernel attributes (call with the device current, outside stream capture)
void dense_prepare(const Geometry &geo, const ModP &m);
// n <-> n_pad repacking of row-major blocks (rows x n  <->  rows x np), `rows` rows starting at host row r0.
// `map` (nullable, old label -> new label) relabels rows: pad scatters src row r to dst row map[r0 + r],
// unpad gathers dst row r from src row map[r0 + r]; without a map row r <-> row r of the given pointers.
int launch_pad_rows(const u32 *src, u32 *dst, int64_t rows, int n, int np, const u32 *map, int64_t r0, cudaStream_t st);
int launch_unpad_rows(const u32 *src, u32 *dst, int64_t rows, int n, int np, const u32 *map, int64_t r0, cudaStream_t st);
// kernel_basis.cu: the kernel vectors inside span(v) (blk_kernel_basis).  A record is (n + 1) x n_pad words: word 0 the
// rank r, rows 1 .. r an echelon basis of a block's row space.
struct KbArgs {
        int n = 0, world = 1, ctas = 1;
        ModP m;
        const u32 *v = nullptr;        // this rank's rows of v (vrows x n_pad)
        int64_t vrows = 0;
        const u32 *t = nullptr;        // this rank's rows of T = S1 v (trows x n_pad)
        int64_t trows = 0;
        u32 *part = nullptr;           // [2][ctas][n][n_pad] per-CTA bases
        int *prank = nullptr;          // [2][ctas]
        unsigned *counter = nullptr;   // last-CTA ticket (zero before the launch, re-armed by it)
        u32 *rec_own = nullptr;        // this rank's two records (v, T)
        u32 *rec_all = nullptr;        // [world][2] records
        u32 *A = nullptr;              // n_pad x n_pad: A_S, column s = a_f of the s-th vector
        int *k = nullptr;              // number of kernel vectors
};
int kb_ctas(int64_t rows);
// k_kb_reduce: both blocks -> rec_own
int launch_kb_reduce(int np, const KbArgs &a, cudaStream_t st);
// k_kb_small: rec_all -> A, k
int launch_kb_small(int np, const KbArgs &a, cudaStream_t st);
// k_block_apply: x = v W for `rows` rows of v (n_pad words each), W n_pad x wp (wp a power of two <= n_pad), x wp words a row
int launch_block_apply(int np, int wp, int64_t rows, const u32 *v, const u32 *W, u32 *x, const ModP &m, cudaStream_t st);
// solve.cu: inhomogeneous systems (blk_create_system, blk_solve), DESIGN.md section 13.
// The non-zeros of -B (Mc x r, row-major, device) as COO triplets of the augmented matrix: (i, N + j) for --right,
// (N + j, i) for --left.  *count receives their number; with Mi == nullptr nothing is written (a first call sizes the
// buffers, a second one fills them).  Returns an error message or "".
std::string rhs_triplets(const u32 *B, int64_t Mc, int r, int64_t N, int right, u32 p, int32_t *Mi, int32_t *Mj, u32 *Mx,
                         int64_t *count, cudaStream_t st);
int pad_width(int w);                // smallest power of two >= w
struct SolveArgs {
        int np = 1, r = 1, rp = 1;     // n_pad, right-hand sides, r padded to a power of two (<= n_pad)
        ModP m;
        const u32 *A = nullptr;        // n_pad x n_pad: A_S of k_kb_small
        const int *k = nullptr;        // its number of columns
        u32 *tail = nullptr;           // r x n_pad: the tail rows of v (rows N .. N+r-1 of the augmented problem)
        u32 *W = nullptr;              // n_pad x rp: W = A_S C
        int *found = nullptr;          // [r]
};
// k_solve_tail: the tail rows this rank owns (device rows [n0, n1) of the full-length v_full), zero elsewhere
int launch_solve_tail(const SolveArgs &a, int64_t N0, const u32 *v_full, const u32 *map, int64_t n0, int64_t n1, cudaStream_t st);
// k_solve_small: tail, A, k -> W, found
int launch_solve_small(const SolveArgs &a, cudaStream_t st);
// prune.cu: removal of empty and singleton constraints (blk_create_pruned), DESIGN.md section 14.
struct PruneResult {
        int64_t N = 0, Mc = 0, nnz = 0, free = 0, rounds = 0;    // kept unknowns, constraints, triplets; free unknowns; rounds
        std::vector<int32_t> unknowns, constraints;              // original indices of the kept ones, ascending
        bool identity = false;                                   // nothing removed: both maps are the identity (left empty)
        int32_t *Mi = nullptr, *Mj = nullptr;                     // M' on the device (owned), or all null when M' is the input
        u32 *Mx = nullptr;                                        // itself (nothing removed, no triplet vanishes mod p)
        void release();
        ~PruneResult() { release(); }
};
// The COO (device, values not reduced) of an nrows x ncols matrix, pruned as DESIGN.md section 14 defines it, on the
// current device and stream st.  Returns an error message or "".
std::string prune_coo(const int32_t *Mi, const int32_t *Mj, const u32 *Mx, int64_t nnz, int64_t nrows, int64_t ncols, int right,
                      u32 p, cudaStream_t st, PruneResult *out);
