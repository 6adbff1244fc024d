/*
 * blk_lanczos.h -- C ABI of the B200-native block-Lanczos mod-p hot path.
 *
 * The reference (T-amairi/block-lanczos-algorithm-parallelization) has no
 * plugin/FFI interface: it is one translation unit whose main loop,
 * block_lanczos (sequential/lanczos_modp.c:585-669), calls
 *
 *     sparse_matrix_vector_product   sequential/lanczos_modp.c:266  (x2, :635-636)
 *     block_dot_products             sequential/lanczos_modp.c:443  (:640)
 *     semi_inverse                   sequential/lanczos_modp.c:342  (:644)
 *     orthogonalize                  sequential/lanczos_modp.c:456  (:652)
 *     v <- tmp copy                  sequential/lanczos_modp.c:655-656
 *
 * with the blocking factor `n` and the modulus `prime` as globals (:39-40).
 * This header is the boundary a maintainer binds instead of those calls: an
 * opaque context that owns the GPU-resident matrix and vector blocks, a
 * batched "run K iterations" entry point for the loop body, and one host-
 * pointer entry point per reference function (same argument meaning) used by
 * the parity tests and the SpMV-only sweep.
 *
 * Conventions
 *   - plain C, no torch / C++ types; every pointer is a HOST pointer unless a
 *     parameter says otherwise; all vector blocks are row-major x[i*n + j],
 *     u32 canonical residues in [0,p), exactly the reference's layout.
 *   - every function returns 0 on success and non-zero on failure;
 *     blk_last_error() then returns a message (the reference's behaviour is
 *     errx(1, msg): the driver does errx(1, "%s", blk_last_error())).
 *   - there is NO CPU fallback: without a CUDA device blk_create fails.
 *   - one host thread drives a context (like the reference's single thread).
 *   - 1 <= n <= 64, 2 <= prime < 2^31 (the reference caps at 2^30-35,
 *     sequential/lanczos_modp.c:189; lifted, see DESIGN.md).
 */
#ifndef BLK_LANCZOS_H
#define BLK_LANCZOS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BLK_ABI_VERSION 2
#define BLK_MAX_N 64
#define BLK_NCCL_ID_BYTES 128
/* blk_params.rank value: this process drives ALL `world` GPUs (devices device ... device+world-1) through one
 * context; the library runs one host thread per GPU inside every call (nccl_id is not needed). */
#define BLK_RANK_ALL (-1)

typedef struct blk_ctx blk_ctx;

/* Creation parameters.  Zero-initialise, then fill.  Mirrors what
 * block_lanczos receives: the COO matrix of struct sparsematrix_t
 * (sequential/lanczos_modp.c:55-62) plus the globals n, prime, right_kernel. */
typedef struct blk_params {
        int32_t  abi_version;     /* BLK_ABI_VERSION */
        int32_t  nrows, ncols;    /* matrix dimensions (M.nrows, M.ncols) */
        int64_t  nnz;             /* number of COO triplets */
        const int32_t  *Mi;       /* 0-based row indices    [nnz] */
        const int32_t  *Mj;       /* 0-based column indices [nnz] */
        const uint32_t *Mx;       /* values (reduced mod prime on ingest) [nnz] */
        int32_t  coo_on_device;   /* 0: Mi/Mj/Mx are host pointers; 1: device pointers on `device` */
        int32_t  n;               /* blocking factor (global `n`) */
        uint32_t prime;           /* modulus (global `prime`) */
        int32_t  right_kernel;    /* 0: --left (x*M == 0), 1: --right (M*x == 0) */
        int32_t  device;          /* CUDA device ordinal */
        int32_t  rank, world;     /* this context's row shard of a `world`-GPU job (0,1: single GPU);
                                     rank = BLK_RANK_ALL: one context for the whole job (single process) */
        const void *nccl_id;      /* BLK_NCCL_ID_BYTES from blk_nccl_unique_id (rank 0), if world > 1 */
        void    *stream;          /* cudaStream_t to run on, or NULL for a private stream */
        int32_t  chunk_len;       /* entries per lane-group chunk of the sparse layout; 0 = auto */
        int32_t  use_graph;       /* -1 auto, 0 never, 1 always: CUDA-graph the iteration loop */
} blk_params;

/* ---- lifetime -------------------------------------------------------- */
int  blk_abi_version(void);
const char *blk_last_error(void);
int  blk_device_count(int *count);
/* Rank 0 of a multi-GPU job calls this and ships the bytes to the other ranks. */
int  blk_nccl_unique_id(void *id_out /* BLK_NCCL_ID_BYTES */);
/* Builds the GPU-resident sparse layouts of M and M^T once from the COO arrays and
 * allocates the four vector blocks v, tmp, Av, p (block_lanczos :592-607), zeroed. */
int  blk_create(blk_ctx **out, const blk_params *prm);
/* An inhomogeneous system M*x = b (--right) or x*M = b (--left) for nrhs right-hand sides (DESIGN.md section 13).
 * B holds Mc*nrhs u32, row-major (row i = the coordinate i of the other dimension, column j = right-hand side j),
 * reduced mod prime on ingest; it is a host pointer, or a device pointer on prm->device when b_on_device != 0.
 * 1 <= nrhs <= n.  The context is blk_create's for the augmented matrix [M | -B] (--right) or [M ; -B^T] (--left):
 * every other entry point works on it, the Lanczos vectors have N + nrhs rows (blk_block_pad, blk_get_info().N),
 * the last nrhs of them the coordinates of the right-hand sides.  rank / world / BLK_RANK_ALL as for blk_create. */
int  blk_create_system(blk_ctx **out, const blk_params *prm, const uint32_t *B, int32_t nrhs, int32_t b_on_device);
/* Removal of empty and singleton constraints before the loop (DESIGN.md section 14).  Unknowns are the coordinates of
 * the Lanczos vectors (rows of M for --left, columns for --right), constraints the other dimension.  Rounds remove
 * every constraint with at most one counting triplet (x mod p != 0) on a kept unknown, and that unknown, until none
 * is left; the kernel is unchanged up to zeros on the removed unknowns.  The context is blk_create's for M', the kept
 * counting triplets renumbered by rank (every other entry point works on M': blk_get_info().N / Mc, blk_block_pad,
 * the state blocks, ...).  Same inputs as blk_create (host or device COO, rank / world / BLK_RANK_ALL; with one
 * process per rank every rank prunes the whole COO itself).  Fails when every constraint is removed. */
enum { BLK_PR_N = 0, BLK_PR_MC = 1, BLK_PR_NNZ = 2, BLK_PR_FREE = 3, BLK_PR_ROUNDS = 4, BLK_PR_COUNT = 5 };
/* blk_create on M' (see DESIGN.md section 14); stats (nullable) receives N', Mc', nnz', free unknowns, rounds. */
int  blk_create_pruned(blk_ctx **out, const blk_params *prm, int64_t stats[BLK_PR_COUNT]);
/* Original indices of the kept unknowns [N'] and constraints [Mc'], ascending (either may be NULL);
 * fails on a context not made by blk_create_pruned. */
int  blk_pruned_index(blk_ctx *ctx, int32_t *unknowns, int32_t *constraints);
int  blk_destroy(blk_ctx *ctx);

/* Host-only: the contiguous, weight-balanced row partition blk_create uses for a `world`-GPU job.
 * idx[nnz] are the COO indices along the dimension being split (rows of M for the Lanczos
 * vectors of --left, ...), dim its length; offsets[world+1] receives the block boundaries.
 * The reference's MPI build splits into equal blocks with the remainder on coordinate 0
 * (mpi/lanczos_modp.c:590-620); here blocks are balanced by non-zeros + rows. */
int  blk_plan_shards(const int32_t *idx, int64_t nnz, int64_t dim, int32_t world, int64_t *offsets);

/* Host-only: the P x Q block grid of a `world`-GPU job -- the reference's 2-D decomposition
 * (mpi/lanczos_modp.c:532-547: MPI_Dims_create + row/column communicators; :590-620: rows split over
 * dims[0], columns over dims[1], remainder on coordinate 0), here balanced by non-zeros.
 * N = length of the Lanczos vectors (rows of M for --left, columns for --right), Mc = the other dimension.
 *   grid[2]  in: {P, Q} with P*Q == world, or {0, 0} to choose like MPI_Dims_create (P >= Q, most square);
 *            out: the grid used.  Rank of grid coordinate (a, b) = a*Q + b.
 *   n_off[P+1], m_off[Q+1]   block boundaries along N and along Mc; rank (a,b) stores the non-zeros with
 *            N-index in [n_off[a], n_off[a+1]) and Mc-index in [m_off[b], m_off[b+1]).
 *   n_sub[P*(Q+1)]  row block a cut into Q pieces: rank (a,b) owns rows [n_sub[a*(Q+1)+b], n_sub[a*(Q+1)+b+1])
 *            of v, Av and p (all-gathered / reduce-scattered inside grid row a).
 *   m_sub[Q*(P+1)]  column block b cut into P pieces: rank (a,b) owns rows [m_sub[b*(P+1)+a], ..+1]) of tmp.
 *   block_nnz[P*Q]  (nullable) non-zeros per block.
 * Exchange volume per rank and iteration: 2*[(N/P)(Q-1)/Q + (Mc/Q)(P-1)/P] rows, against 2*(W-1)/W*(N+Mc)/2
 * for the 1-D row sharding of blk_create (DESIGN.md section 6). */
int  blk_plan_grid(const int32_t *Mi, const int32_t *Mj, int64_t nnz, int32_t nrows, int32_t ncols,
                   int32_t right_kernel, int32_t world, int32_t grid[2], int64_t *n_off, int64_t *m_off,
                   int64_t *n_sub, int64_t *m_sub, int64_t *block_nnz);

/* Host-only: the heavy prefix of product 2 that blk_create runs as column bands on one GPU (DESIGN.md section 4).
 * deg[rows] are the row degrees of that product under the degree-sorted labels (non-increasing), cols the length
 * of the block it gathers, l2_bytes the device's L2.  *heavy_rows receives H, the rows with degree >= min_deg, and
 * *bands K = ceil(cols * n_pad * 4 / band_bytes) (<= 256); both 0 when no split pays: n_pad < 8, a gathered block
 * that fits L2, or a predicted saving (lines not fetched minus partial traffic and the bands' gather time) <= 0.
 * force skips the last two checks. */
int  blk_plan_heavy(const uint32_t *deg, int64_t rows, int64_t cols, int32_t n_pad, int64_t l2_bytes, int64_t min_deg,
                    int64_t band_bytes, int32_t force, int64_t *heavy_rows, int32_t *bands);

/* block_size_pad of block_lanczos (:594-597) in u32 elements: the length of the
 * reference's v/tmp/Av/p blocks and of every block in blk_get_state. */
int64_t blk_block_pad(int32_t nrows, int32_t ncols, int32_t n, int32_t right_kernel);

/* ---- the iteration (block_lanczos main loop, :631-659) ---------------- */
/* Load the Lanczos state: v and p hold N*n u32 (N = nrows for --left, ncols for
 * --right); p may be NULL (all zero: fresh start).  n_iterations is the
 * reference's counter (non-zero after --load-checkpoint).  In a multi-GPU job
 * every rank is given the same full-length blocks but reads only the rows it owns
 * (1/world of the PCIe traffic); the rest reaches it from the peers over NVLink. */
int  blk_set_state(blk_ctx *ctx, const uint32_t *v, const uint32_t *p, int32_t n_iterations);
/* Run up to max_iters further iterations entirely on the device (no host
 * round-trip per iteration).  With BLK_CHECK=1 in the environment at blk_create time the n x n stage also
 * evaluates the reference's correctness_tests (:532-557) on every iteration; a violated invariant stops the
 * loop before anything is updated and this call fails (the reference aborts on the assert).  Stops early, exactly like the reference, at the
 * iteration whose semi_inverse returns 0 pivots (:644,:649): v is then left
 * untouched and tmp = M^T v (resp. M v).  *stopped is that condition,
 * *iters_total the reference's n_iterations afterwards.                    */
int  blk_iterate(blk_ctx *ctx, int32_t max_iters, int32_t *iters_total, int32_t *stopped);
/* Copy the four blocks to the host in the reference's padded layout
 * (blk_block_pad u32 each; any pointer may be NULL).  Contents are identical
 * to the reference's v/tmp/Av/p at the same point of the loop.             */
int  blk_get_state(blk_ctx *ctx, uint32_t *v, uint32_t *tmp, uint32_t *Av, uint32_t *p);
/* Multi-GPU jobs with one process per GPU: like blk_get_state for v, Av, p (any may be NULL; same padded
 * layout), but only the rows this rank owns -- [local_N0, local_N1) of blk_get_info -- are written, nothing
 * crosses NVLink and each rank moves 1/world of the data over PCIe (a distributed checkpoint).  On a single
 * GPU, and on a BLK_RANK_ALL context, identical to blk_get_state. */
int  blk_get_state_local(blk_ctx *ctx, uint32_t *v, uint32_t *Av, uint32_t *p);
/* final_check (sequential/lanczos_modp.c:560-582) on the device, without copying the blocks back:
 * *v_nonzero = (v != 0) over the N rows, *vtm_zero = (tmp == 0) over the Mc rows, where tmp is the
 * product M^T v (resp. M v) of the current v -- the state the loop is in after it stopped on
 * "no pivot" (otherwise that product is computed first into a scratch block). */
int  blk_final_check(blk_ctx *ctx, int32_t *v_nonzero, int32_t *vtm_zero);
/* The property checker_modp verifies (checker_modp.c:146-204) for a candidate block x of N*n u32:
 * every entry < prime, x not all zero, and x*M == 0 (M*x == 0 for --right).  *ok = 1 if all hold. */
int  blk_check_kernel_block(blk_ctx *ctx, const uint32_t *x, int32_t *ok);
/* The kernel vectors inside span(v) (the final Gaussian elimination of block Lanczos, Montgomery 1995; the
 * reference has no such step, DESIGN.md section 12): with T = M^T v (resp. M v), X = v A where the columns of A
 * are the standard null basis of T reduced to those that stay independent through v.  x receives N*n u32
 * (row-major, stride n, host order): columns [0,k) hold X, columns [k,n) are zero; *k = rank([T; v]) - rank(T).
 * The columns of X are independent, x*M == 0 (M*x == 0 for --right), and they span every such vector in span(v).
 * Callable at any point of the loop; v, tmp, Av and p are left untouched. */
int  blk_kernel_basis(blk_ctx *ctx, uint32_t *x, int32_t *k);
/* The solutions inside span(v) of a context made by blk_create_system (fails on any other context).  x receives
 * N*nrhs u32 (the original N, row-major, stride nrhs, host order), found[nrhs] the flags: column j satisfies
 * M*x_j == b_j (x_j*M == b_j for --left) when found[j] = 1 and is zero otherwise.  found[j] = 0 means no solution
 * lies in span(v): the system may be inconsistent, or the block did not reach one.  Callable at any point of the
 * loop; v, tmp, Av and p are left untouched. */
int  blk_solve(blk_ctx *ctx, uint32_t *x, int32_t *found);
/* n x n results of the last executed iteration (any may be NULL): vtAv, vtAAv,
 * winv are n*n, d is n; *npiv the value semi_inverse returned.            */
int  blk_get_small(blk_ctx *ctx, uint32_t *vtAv, uint32_t *vtAAv, uint32_t *winv, uint32_t *d,
                   int32_t *npiv);

/* ---- one entry point per reference function (host pointers) ----------- */
/* sparse_matrix_vector_product(y, M, x, transpose) (:266): y <- M x (transpose 0,
 * x has ncols*n, y nrows*n entries) or y <- M^T x (transpose 1).           */
int  blk_spmv(blk_ctx *ctx, uint32_t *y, const uint32_t *x, int32_t transpose);
/* block_dot_products(vtAv, vtAAv, N, Av, v) (:443): N rows of n. */
int  blk_block_dot_products(blk_ctx *ctx, uint32_t *vtAv, uint32_t *vtAAv, int64_t N,
                            const uint32_t *Av, const uint32_t *v);
/* semi_inverse(M_, winv, d) (:342); *npiv is its return value. */
int  blk_semi_inverse(blk_ctx *ctx, const uint32_t *M_, uint32_t *winv, uint32_t *d, int32_t *npiv);
/* orthogonalize(v, tmp, p, d, vtAv, vtAAv, winv, N, Av) (:456): tmp[0..N*n) <- next v,
 * p updated in place; v, Av, d and the three n x n matrices are inputs.    */
int  blk_orthogonalize(blk_ctx *ctx, const uint32_t *v, uint32_t *tmp, uint32_t *p, const uint32_t *d,
                       const uint32_t *vtAv, const uint32_t *vtAAv, const uint32_t *winv, int64_t N,
                       const uint32_t *Av);

/* ---- measurement ------------------------------------------------------ */
enum {
        BLK_PH_SPMV1 = 0,      /* tmp <- S1 v   (+ its carry fix-up) */
        BLK_PH_SPMV2 = 1,      /* Av  <- S2 tmp (+ its carry fix-up) */
        BLK_PH_DOTS = 2,       /* block_dot_products */
        BLK_PH_SMALL = 3,      /* reduction of partials + semi_inverse + n x n bookkeeping */
        BLK_PH_ORTHO = 4,      /* orthogonalize (v, p updated in place) */
        BLK_PH_EXCHANGE = 5,   /* multi-GPU all-gathers / all-reduce */
        BLK_PH_COUNT = 6
};
/* When on, blk_iterate brackets every phase with CUDA events on the context's stream
 * (graphs off) and accumulates device milliseconds and launch counts per phase. */
int  blk_set_profiling(blk_ctx *ctx, int32_t on);
int  blk_get_phase_times(blk_ctx *ctx, double ms[BLK_PH_COUNT], int64_t launches[BLK_PH_COUNT]);
/* Run the SpMV kernel `reps` times on the resident blocks (transpose as in blk_spmv) and
 * return the average device time of one product in ms (CUDA events, context stream). */
int  blk_time_spmv(blk_ctx *ctx, int32_t transpose, int32_t reps, double *ms_avg);
/* Kernels launched by this context so far (all phases, fix-ups included). */
int64_t blk_kernel_launches(blk_ctx *ctx);
/* Static facts about the resident layout, for roofline arithmetic. */
typedef struct blk_info {
        int64_t N, Mc;                 /* Lanczos vector length and the other dimension */
        int64_t local_N0, local_N1;    /* this rank's rows of v/Av/p */
        int64_t local_M0, local_M1;    /* this rank's rows of tmp */
        int64_t nnz_local[2];          /* real entries of S1 (rows of tmp) and S2 (rows of Av) on this rank */
        int64_t stored_local[2];       /* stored entries incl. padding and empty-row dummies */
        int64_t tiles[2];              /* warp tiles */
        int32_t n, n_pad, chunk_len[2], groups_per_warp;
        int64_t device_bytes;          /* resident bytes (matrix layouts + blocks) */
        int32_t loop_mode;             /* how blk_iterate runs the loop: 0 chain of kernels / CUDA graph, 1 one persistent
                                          cooperative kernel (L2-resident problems on one GPU, BLK_LOOP) */
        int32_t nrhs;                  /* right-hand sides of a blk_create_system context (counted in N), else 0 */
        int32_t bands[2];              /* column bands of S1 / S2 (0: none): n_pad <= 4 with an x block far larger than L2 */
        int64_t heavy_rows;            /* rows of S2's heavy prefix run as column bands (0: no split, blk_plan_heavy) */
        int32_t heavy_bands;           /* its column bands */
} blk_info;
int  blk_get_info(blk_ctx *ctx, blk_info *info);

#ifdef __cplusplus
}
#endif
#endif /* BLK_LANCZOS_H */
