// context.cu -- implementation of the C ABI in include/blk_lanczos.h.
//
// The context owns what block_lanczos (sequential/lanczos_modp.c:585-669) owns on the host:
// the matrix (as two GPU-resident operators S1, S2 instead of COO arrays) and the four vector
// blocks v, tmp, Av, p.  blk_iterate enqueues the loop body (:635-656) as kernels on one
// stream; the stop decision (:644,:649) and the iteration counter live on the device, so a
// batch of iterations (optionally one CUDA graph per 16 iterations) runs without any host
// round trip and freezes exactly at the iteration where semi_inverse finds no pivot.
//
// Multi-GPU (world > 1, one context per GPU/process): rows of the Lanczos vectors and of both
// operators are sharded in contiguous, weight-balanced blocks.  Per iteration: all-gather v,
// local S1, all-gather tmp, local S2, local dots, all-reduce of 2 n^2 u64 sums, redundant
// semi_inverse, local orthogonalize.  Collectives go through NCCL (resolved with dlopen so the
// library loads on machines without it); the reference's MPI version does the same steps with
// hand-rolled Send/Recv reductions on a root (mpi/lanczos_modp.c:1088-1125, 1209-1256).
#include <dlfcn.h>
#include <nccl.h>
#include <unistd.h>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>
#include "../../include/blk_lanczos.h"
#include "blk_internal.cuh"

static thread_local std::string g_err;

static int fail(const std::string &msg)
{
        g_err = msg;
        return 1;
}

#define CU(call)                                                                                   \
        do {                                                                                       \
                cudaError_t e_ = (call);                                                           \
                if (e_ != cudaSuccess)                                                             \
                        return fail(std::string(#call) + ": " + cudaGetErrorString(e_));           \
        } while (0)

// ---------------------------------------------------------------------------------- NCCL (dlopen)
namespace {
struct NcclApi {
        void *lib = nullptr;
        ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
        ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
        ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
        ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
        ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
        ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
        ncclResult_t (*GroupStart)() = nullptr;
        ncclResult_t (*GroupEnd)() = nullptr;
        const char *(*GetErrorString)(ncclResult_t) = nullptr;
        // only needed by the P x Q grid mode (BLK_GRID); resolved lazily, may be null
        ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
        ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
        ncclResult_t (*CommSplit)(ncclComm_t, int, int, ncclComm_t *, void *) = nullptr;
};
NcclApi g_nccl;

bool nccl_load(std::string *why)
{
        if (g_nccl.lib) return true;
        void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) { *why = std::string("cannot load NCCL: ") + dlerror(); return false; }
#define SYM(field, name)                                                                           \
        *(void **)(&g_nccl.field) = dlsym(h, name);                                                \
        if (!g_nccl.field) { *why = std::string("NCCL symbol missing: ") + name; return false; }
        SYM(GetUniqueId, "ncclGetUniqueId")
        SYM(CommInitRank, "ncclCommInitRank")
        SYM(CommDestroy, "ncclCommDestroy")
        SYM(AllReduce, "ncclAllReduce")
        SYM(Broadcast, "ncclBroadcast")
        SYM(AllGather, "ncclAllGather")
        SYM(GroupStart, "ncclGroupStart")
        SYM(GroupEnd, "ncclGroupEnd")
        SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
        *(void **)(&g_nccl.Send) = dlsym(h, "ncclSend");
        *(void **)(&g_nccl.Recv) = dlsym(h, "ncclRecv");
        *(void **)(&g_nccl.CommSplit) = dlsym(h, "ncclCommSplit");
        g_nccl.lib = h;
        return true;
}
}  // namespace

#define NC(call)                                                                                   \
        do {                                                                                       \
                ncclResult_t r_ = (call);                                                          \
                if (r_ != ncclSuccess)                                                             \
                        return fail(std::string(#call) + ": " + g_nccl.GetErrorString(r_));        \
        } while (0)

// ---------------------------------------------------------------------------------- context
struct blk_ctx {
        Geometry geo;
        ModP m;
        int device = 0, rank = 0, world = 1, right = 0;
        int32_t nrows = 0, ncols = 0;
        int64_t N = 0, Mc = 0;
        int nrhs = 0;                           // blk_create_system: right-hand sides appended to M (N counts them too)
        bool pruned = false;                    // blk_create_pruned: original indices of the kept unknowns / constraints
        bool pr_identity = false;               // (nothing removed: the identity, not stored)
        std::vector<int32_t> pr_unknowns, pr_constraints;
        std::vector<int64_t> n_off, m_off;      // row partition of the N and Mc dimensions
        SpOp S1, S2;                            // tmp <- S1 v ; Av <- S2 tmp
        u32 *v = nullptr, *tmp = nullptr;       // full length: N*np, Mc*np
        u32 *Av = nullptr, *p = nullptr;        // local rows [n0,n1) * np
        u32 *mats = nullptr;
        u64 *sums = nullptr;                   // 2*np*np dot-product accumulators (zero between iterations)
        u32 *n_old2new = nullptr, *n_new2old = nullptr;   // degree-sorted relabelling of the N dimension (or null)
        int64_t hot_rows = 0;
        unsigned *dots_counter = nullptr;      // last-block-done ticket of the fused dots + small kernel
        bool fuse_small = false;
        DevSmall *state = nullptr, *h_state = nullptr;
        int dots_blocks = 1;
        cudaStream_t stream = nullptr;
        bool own_stream = false;
        ncclComm_t comm = nullptr;
        // pipelined product 1 (multi-GPU): S1 runs in row pieces; each finished piece is broadcast on
        // comm_stream while the next one is computed
        int pieces = 1;
        cudaStream_t comm_stream = nullptr;
        std::vector<cudaEvent_t> ev_piece;
        cudaEvent_t ev_comm = nullptr;
        std::vector<int64_t> piece_rows_all;     // [world][pieces+1] local row boundaries of every rank's S1
        std::vector<int64_t> piece_rows_all2;    // same for S2
        int pieces2 = 1;
        // "tmp recurrence" (multi-GPU): the next S1*v is obtained from S1*Av, so the vector that has to
        // be exchanged is Av (hidden behind product 2) instead of the new v (which nothing could hide)
        bool mg_recur = false, ran_since_set = false;
        u32 *Av_full = nullptr;                  // gather target of Av; c->Av points at the local rows inside it
        u32 *Tp = nullptr, *U = nullptr;         // local rows of S1*p and of S1*Av
        u32 *tmp_prev = nullptr;                 // local rows of the previous tmp (only when Mc > N, for checkpoints)
        // How the two full-length vectors of an iteration (Av, new tmp) reach the other GPUs:
        //   XCH_NCCL  grouped ncclBroadcast of every finished row piece on comm_stream (round-1 default)
        //   XCH_CE    the copy engines push finished pieces into the peers' buffers (cudaMemcpyAsync on peer pointers)
        //   XCH_PUSH  stores over NVLink from our own kernels through peer-mapped pointers: product 2 writes every
        //             finished row of Av into all copies itself (k_spmv PUSH, a fused all-gather), the pieces of the new
        //             tmp are pushed by k_push_rows, a copy kernel of a few CTAs on comm_stream; a tiny all-reduce
        //             that follows is the barrier
        enum { XCH_NCCL = 0, XCH_CE = 1, XCH_PUSH = 2 };
        int xch = XCH_NCCL;
        bool push_av_in_spmv = true;             // XCH_PUSH: Av from inside k_spmv (else k_push_rows per piece)
        bool push_bulk = false;                  // XCH_PUSH: pieces travel by k_push_bulk (bulk-copy engine) instead of k_push_rows
        int push_ctas = 32;
        int bulk_stages = 4;                     // k_push_bulk: ring of bulk_stages x bulk_chunk bytes of shared memory per CTA
        unsigned bulk_chunk = 32768;
        std::vector<u32 *> peer_tmp, peer_av;    // [world] peer mappings of every rank's tmp / Av_full (own = local)
        std::vector<char> peer_ipc;              // [world] mapping came from cudaIpcOpenMemHandle (must be closed)
        std::vector<cudaStream_t> copy_streams;  // one per peer offset so that the copies use several copy engines
        std::vector<cudaEvent_t> ev_copies;
        u64 *barrier_word = nullptr;
        ncclResult_t (*nccl_allgather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
        // column-blocked products (experimental, BLK_COLBLOCKS=K; see ColOps below): the consumer of a pieced
        // exchange starts on the columns whose piece has arrived instead of waiting for the whole vector
        int colblocks = 0;
        struct ColOps {
                int K = 0;
                std::vector<SpOp> col;           // [K-1] all local rows x the columns of input piece q (of every rank)
                std::vector<SpOp> last;          // [K]   output row piece i x the columns of input piece K-1
                std::vector<int64_t> prow;       // [K+1] local row boundaries of the output pieces
        } cb1, cb2;
        u32 *zbuf = nullptr;                     // K partial results of one product, zstride elements apart
        size_t zstride = 0;
        std::vector<cudaEvent_t> ev_arrived;     // [2K] piece q of tmp (0..K-1) / of Av (K..2K-1) has landed on this rank
        cudaEvent_t ev_aux = nullptr;
        // P x Q block grid (experimental, BLK_GRID=PxQ | auto; the reference's 2-D decomposition, blk_plan_grid):
        // rank (a,b) = a*Q + b holds block (a,b) of the operator in both orientations and owns piece (a,b) of
        // v, Av, p and piece (b,a) of tmp.  The 1-D operators and blocks above stay in place for everything
        // outside the loop (get_state, final_check, ...): grid_export() copies the distributed state into them.
        struct Grid {
                int P = 0, Q = 0, a = 0, b = 0;
                std::vector<int64_t> n_off, m_off, n_sub, m_sub;     // as returned by blk_plan_grid
                int64_t pieceN = 0, pieceM = 0;                      // padded piece rows inside my block row / column
                int64_t pieceNmax = 0, pieceMmax = 0;                // over all blocks (world-wide gathers)
                ncclComm_t row_comm = nullptr, col_comm = nullptr;
                SpOp S1, S2;                                         // (P*pieceM) x (Q*pieceN) and its transpose
                u32 *vblk = nullptr, *tblk = nullptr;                // v_a (Q pieces), tmp_b (P pieces), piece-padded
                u32 *part1 = nullptr, *part2 = nullptr;              // partial tmp_b / partial Av_a (separate: a halted iteration
                                                                     // skips the products and must find its own partial again)
                u32 *recv = nullptr;                                 // pieces received in a reduce-scatter
                u32 *Av = nullptr, *p = nullptr;                     // owned piece
                bool dirty = false;                                  // the 1-D copies are stale
        } grid;
        bool grid_on = false;
        // resident staging buffer of upload_rows / download_rows (host <-> device repacking, chunk by chunk)
        static constexpr size_t STAGE_BYTES = 32u << 20;
        u32 *stage = nullptr;
        long long l2_persist_before = -1;       // cudaLimitPersistingL2CacheSize found at create time (restored on destroy)
        int bands1 = 0, bands2 = 0;             // column bands of S1 / S2 (0: none), see SpOp::bands
        bool bands_acc = false;                 // BLK_BAND_ACC=1: compact accumulate-in-place bands (measured slower than partial results + combine)
        bool check = false;                     // BLK_CHECK=1: the n x n stage asserts the reference's correctness_tests
        int check_fault = 0;                    // BLK_CHECK_FAULT=k: corrupt vtAv in iteration k (tests the self-check)
        // Single-process multi-GPU job (blk_params.rank == BLK_RANK_ALL): this context owns one member context
        // per GPU and fans every call out to them, one host thread per member (the reference's MPI build is one
        // process per rank, mpi/lanczos_modp.c:1829-1863; here one process can drive the whole box).
        std::vector<blk_ctx *> members;
        bool is_group() const { return !members.empty(); }
        // loop bookkeeping
        int iters = 0, stopped = 0;
        bool tmp_is_spmv = false;               // tmp rows [0,Mc) hold S1*v of the current v (stop case)
        bool any_ortho = false;
        // Persistent cooperative loop kernel (loop_coop.cu): single GPU, n_pad <= 16, operators + blocks L2-sized.
        // One launch runs up to COOP_BATCH iterations; replaces the CUDA graph of six kernel nodes per iteration.
        bool coop = false;
        int coop_grid = 0;
        unsigned *loop_bar = nullptr;            // 2 barrier words, then (8 bytes further) 6 u64 phase clocks
        bool coop_prof = false;                  // BLK_LOOP_PROF=1: profiling mode keeps the persistent kernel and reads its phase clocks
        static constexpr int COOP_BATCH = 1024;
        // graphs
        int use_graph = -1;
        cudaGraphExec_t graph = nullptr;
        static constexpr int GRAPH_ITERS = 16;
        // profiling
        bool profiling = false;
        double ph_ms[BLK_PH_COUNT] = {0};
        int64_t ph_launch[BLK_PH_COUNT] = {0};
        int64_t launches = 0;
        size_t block_bytes = 0;

        // With relabelled rows on several GPUs a rank's rows are scattered over the caller's (host-order) blocks, so
        // host <-> device copies are split by HOST rows instead: rank r moves host rows [h0, h1) over PCIe and the
        // rows find their owners (or their readers) over NVLink.
        bool relabel_mg() const { return n_old2new != nullptr && world > 1; }
        int64_t h0() const { return relabel_mg() ? N * rank / world : n_off[rank]; }
        int64_t h1() const { return relabel_mg() ? N * (rank + 1) / world : n_off[rank + 1]; }
        int64_t n0() const { return n_off[rank]; }
        int64_t n1() const { return n_off[rank + 1]; }
        int64_t m0() const { return m_off[rank]; }
        int64_t m1() const { return m_off[rank + 1]; }
};

namespace {

// run f(member, rank) for every member of a group context, one host thread per member (collectives inside the
// library need all ranks in flight at once); the first failure becomes the group's error
template <class F> int group_run(blk_ctx *g, F f)
{
        const int W = (int)g->members.size();
        std::vector<int> rc((size_t)W, 0);
        std::vector<std::string> why((size_t)W);
        std::vector<std::thread> th;
        auto body = [&](int r) {
                rc[(size_t)r] = f(g->members[(size_t)r], r);
                if (rc[(size_t)r]) why[(size_t)r] = g_err;
        };
        for (int r = 1; r < W; r++) th.emplace_back(body, r);
        body(0);
        for (auto &t : th) t.join();
        for (int r = 0; r < W; r++)
                if (rc[(size_t)r]) return fail("GPU " + std::to_string(g->members[(size_t)r]->device) + ": " + why[(size_t)r]);
        return 0;
}

struct EventTimer {
        // records (phase, start, stop) triples on the stream; resolved after a sync
        struct Rec { int ph; cudaEvent_t a, b; int launches; };
        std::vector<Rec> recs;
        void begin(blk_ctx *c, int ph)
        {
                Rec r; r.ph = ph; r.launches = 0;
                cudaEventCreate(&r.a); cudaEventCreate(&r.b);
                cudaEventRecord(r.a, c->stream);
                recs.push_back(r);
        }
        void end(blk_ctx *c, int launches)
        {
                recs.back().launches = launches;
                cudaEventRecord(recs.back().b, c->stream);
        }
        void resolve(blk_ctx *c)
        {
                for (auto &r : recs) {
                        float ms = 0;
                        cudaEventElapsedTime(&ms, r.a, r.b);
                        c->ph_ms[r.ph] += ms;
                        c->ph_launch[r.ph] += r.launches;
                        cudaEventDestroy(r.a); cudaEventDestroy(r.b);
                }
                recs.clear();
        }
};

// Contiguous partition of `dim` rows into `world` blocks.  Equal blocks (ceil(dim/world) rows, the
// last one short) are preferred because the exchange is then a true in-place ncclAllGather; when
// that would leave some rank more than 5% heavier (weight = non-zeros + 8 per row) than a
// weight-balanced split, the weight-balanced boundaries are used and the all-gather becomes a
// group of broadcasts.
std::vector<int64_t> partition_rows(const std::vector<u32> &cnt, int world)
{
        int64_t dim = (int64_t)cnt.size();
        std::vector<int64_t> off(world + 1, 0), eq(world + 1, 0);
        long double total = 0;
        for (int64_t r = 0; r < dim; r++) total += (long double)cnt[r] + 8.0L;
        long double run = 0;
        int k = 1;
        for (int64_t r = 0; r < dim && k < world; r++) {
                run += (long double)cnt[r] + 8.0L;
                while (k < world && run >= total * k / world) off[k++] = r + 1;
        }
        while (k < world) off[k++] = dim;
        off[world] = dim;
        int64_t R = (dim + world - 1) / world;
        for (int q = 0; q <= world; q++) eq[q] = std::min<int64_t>(dim, (int64_t)q * R);
        auto heaviest = [&](const std::vector<int64_t> &o) {
                long double worst = 0;
                for (int q = 0; q < world; q++) {
                        long double w = 0;
                        for (int64_t r = o[q]; r < o[q + 1]; r++) w += (long double)cnt[r] + 8.0L;
                        worst = std::max(worst, w);
                }
                return worst;
        };
        if (world > 1 && heaviest(eq) <= 1.05L * heaviest(off)) return eq;
        return off;
}

// rows a buffer must hold to be the target of allgather_rows (equal blocks are padded)
int64_t gather_cap(const std::vector<int64_t> &off)
{
        int world = (int)off.size() - 1;
        int64_t dim = off[world], R = off[1] - off[0];
        return std::max<int64_t>(dim, R * world);
}

bool equal_blocks(const std::vector<int64_t> &off)
{
        int world = (int)off.size() - 1;
        int64_t dim = off[world], R = off[1] - off[0];
        if (R <= 0) return false;
        for (int q = 0; q <= world; q++)
                if (off[q] != std::min<int64_t>(dim, (int64_t)q * R)) return false;
        return true;
}

// `map` (nullable): count under the relabelled index map[idx]
__global__ void k_count_rows(int64_t nnz, const int32_t *__restrict__ idx, int64_t dim, u32 *__restrict__ cnt,
                             const u32 *__restrict__ map)
{
        int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (s >= nnz) return;
        int64_t r = idx[s];
        if (r < 0 || r >= dim) return;
        if (map) r = map[r];
        atomicAdd(&cnt[r], 1u);
}

// entries whose (relabelled) key lies in [lo, hi); key_map / other_map (nullable, key_dim / other_dim entries): the
// relabelling of the two index spaces, applied here so that the layout builder sees final labels
__global__ void k_select_range(int64_t nnz, const int32_t *__restrict__ key, const int32_t *__restrict__ other,
                               const u32 *__restrict__ val, int64_t lo, int64_t hi, int32_t *__restrict__ okey,
                               int32_t *__restrict__ oother, u32 *__restrict__ oval,
                               unsigned long long *__restrict__ counter, const u32 *__restrict__ key_map, int64_t key_dim,
                               const u32 *__restrict__ other_map, int64_t other_dim)
{
        int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (s >= nnz) return;
        int64_t k = key[s], o = other[s];
        if (key_map) { if (k < 0 || k >= key_dim) return; k = key_map[k]; }
        if (k < lo || k >= hi) return;
        if (other_map && o >= 0 && o < other_dim) o = other_map[o];
        unsigned long long pos = atomicAdd(counter, 1ull);
        okey[pos] = (int32_t)k; oother[pos] = (int32_t)o; oval[pos] = val[s];
}

inline unsigned nb(int64_t n) { return (unsigned)((n + 255) / 256); }

// ---- column-blocked products -------------------------------------------------------------------
// Piece q of rank r along a dimension with block boundaries off[]: rows off[r] + len_r*q/K .. off[r] + len_r*(q+1)/K.
// The same formula gives the output pieces of the product that writes the dimension and the input pieces of the
// product that reads it, on every rank, without any exchange.
static inline int64_t piece_bound(const std::vector<int64_t> &off, int r, int q, int K)
{
        return off[r] + (off[r + 1] - off[r]) * q / K;
}

// select the entries with row key in [rlo, rhi) whose column key lies in piece q of some rank
// (cb[r*(K+1) + q] <= c < cb[r*(K+1) + q + 1]); okey == nullptr: count only
__global__ void k_select_colblock(int64_t count, const int32_t *__restrict__ rkey, const int32_t *__restrict__ ckey,
                                  const u32 *__restrict__ val, int64_t rlo, int64_t rhi, int W, int K, int q,
                                  const int64_t *__restrict__ cb, int32_t *__restrict__ okey, int32_t *__restrict__ ocol,
                                  u32 *__restrict__ oval, unsigned long long *__restrict__ counter)
{
        int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (s >= count) return;
        int64_t r = rkey[s], c = ckey[s];
        if (r < rlo || r >= rhi) return;
        bool in = false;
        for (int w = 0; w < W && !in; w++)
                in = c >= cb[(size_t)w * (K + 1) + q] && c < cb[(size_t)w * (K + 1) + q + 1];
        if (!in) return;
        unsigned long long pos = atomicAdd(counter, 1ull);
        if (okey) { okey[pos] = (int32_t)r; ocol[pos] = (int32_t)c; oval[pos] = val[s]; }
}

// entries of grid block (a,b) with block-local, piece-padded indices: piece k of the block starts at k*piece rows
__global__ void k_select_grid(int64_t nnz, const int32_t *__restrict__ iN, const int32_t *__restrict__ iM,
                              const u32 *__restrict__ val, int Q, const int64_t *__restrict__ nsub, int64_t pieceN, int P,
                              const int64_t *__restrict__ msub, int64_t pieceM, int32_t *__restrict__ oN,
                              int32_t *__restrict__ oM, u32 *__restrict__ oval, unsigned long long *__restrict__ counter)
{
        int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (s >= nnz) return;
        const int64_t g = iN[s], h = iM[s];
        if (g < nsub[0] || g >= nsub[Q] || h < msub[0] || h >= msub[P]) return;
        int bq = 0, ap = 0;
        while (bq + 1 < Q && g >= nsub[bq + 1]) bq++;
        while (ap + 1 < P && h >= msub[ap + 1]) ap++;
        unsigned long long pos = atomicAdd(counter, 1ull);
        if (oN) {
                oN[pos] = (int32_t)(bq * pieceN + (g - nsub[bq]));
                oM[pos] = (int32_t)(ap * pieceM + (h - msub[ap]));
                oval[pos] = val[s];
        }
}

// out[e] = (own[e] + recv_0[e] + ... + recv_{K-1}[e]) mod p   (the local half of a reduce-scatter)
__global__ void k_sum_pieces(u32 *__restrict__ out, const u32 *__restrict__ own, const u32 *__restrict__ recv, int K,
                             size_t stride, int64_t count, ModP m)
{
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x) {
                u64 acc = own[e];
                for (int q = 0; q < K; q++) acc += recv[(size_t)q * stride + e];
                out[e] = mp_reduce(acc, m);
        }
}

// y[e] = (z_0[e] + ... + z_{K-1}[e]) mod p
__global__ void k_combine_blocks(u32 *__restrict__ y, const u32 *__restrict__ z, int K, size_t stride, int64_t count, ModP m,
                                 const DevSmall *__restrict__ state)
{
        if (state && state->halt) return;
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x) {
                u64 acc = 0;
                for (int q = 0; q < K; q++) acc += z[(size_t)q * stride + e];
                y[e] = mp_reduce(acc, m);
        }
}



// flags[0] |= any element non-zero; flags[1] |= any element >= p
__global__ void k_scan_block(const u32 *__restrict__ a, int64_t count, u32 p, int *__restrict__ flags)
{
        int nz = 0, big = 0;
        for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (int64_t)gridDim.x * blockDim.x) {
                u32 x = a[e];
                nz |= x != 0;
                big |= x >= p;
        }
        if (__any_sync(0xffffffffu, nz) && (threadIdx.x & 31) == 0) atomicOr(&flags[0], 1);
        if (__any_sync(0xffffffffu, big) && (threadIdx.x & 31) == 0) atomicOr(&flags[1], 1);
}

// scan `rows` rows (leading dimension np) and return (any non-zero, any >= p), summed over the ranks
int scan_rows(blk_ctx *c, const u32 *a, int64_t rows, int *any_nonzero, int *any_big)
{
        unsigned long long *d = nullptr, h[2] = {0, 0};
        int *flags = nullptr, hf[2] = {0, 0};
        CU(cudaMalloc(&flags, 2 * sizeof(int)));
        CU(cudaMalloc(&d, 2 * sizeof(unsigned long long)));
        CU(cudaMemsetAsync(flags, 0, 2 * sizeof(int), c->stream));
        int64_t count = rows * c->geo.np;
        if (count > 0) {
                unsigned blocks = (unsigned)std::min<int64_t>(blk_sm_count() * 8, (count + 255) / 256);
                k_scan_block<<<blocks, 256, 0, c->stream>>>(a, count, c->m.p, flags);
                c->launches++;
        }
        CU(cudaMemcpyAsync(hf, flags, sizeof(hf), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        if (c->world > 1) {
                h[0] = hf[0]; h[1] = hf[1];
                CU(cudaMemcpyAsync(d, h, sizeof(h), cudaMemcpyHostToDevice, c->stream));
                NC(g_nccl.AllReduce(d, d, 2, ncclUint64, ncclSum, c->comm, c->stream));
                CU(cudaMemcpyAsync(h, d, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
                CU(cudaStreamSynchronize(c->stream));
                hf[0] = h[0] != 0; hf[1] = h[1] != 0;
        }
        cudaFree(flags); cudaFree(d);
        *any_nonzero = hf[0]; *any_big = hf[1];
        return 0;
}

// buf holds gather_cap(off) rows; every rank contributes rows [off[rank], off[rank+1]) in place.
// wp: words per row (0: n_pad)
int allgather_rows(blk_ctx *c, u32 *buf, const std::vector<int64_t> &off, int wp = 0)
{
        const int np = wp ? wp : c->geo.np;
        if (c->nccl_allgather && equal_blocks(off)) {
                size_t cnt = (size_t)(off[1] - off[0]) * np;
                NC(c->nccl_allgather(buf + (size_t)c->rank * cnt, buf, cnt, ncclUint32, c->comm, c->stream));
                return 0;
        }
        NC(g_nccl.GroupStart());
        for (int r = 0; r < c->world; r++) {
                size_t cnt = (size_t)(off[r + 1] - off[r]) * np;
                u32 *ptr = buf + (size_t)off[r] * np;
                if (cnt) NC(g_nccl.Broadcast(ptr, ptr, cnt, ncclUint32, r, c->comm, c->stream));
        }
        NC(g_nccl.GroupEnd());
        return 0;
}

// broadcast piece q of a row-sharded block from every owner (grouped): rows_all = [world][K+1]
int piece_broadcast(blk_ctx *c, u32 *buf, const std::vector<int64_t> &off, const std::vector<int64_t> &rows_all,
                    int K, int q, cudaStream_t st)
{
        NC(g_nccl.GroupStart());
        for (int r = 0; r < c->world; r++) {
                int64_t lo = rows_all[(size_t)r * (K + 1) + q], hi = rows_all[(size_t)r * (K + 1) + q + 1];
                size_t cnt = (size_t)(hi - lo) * c->geo.np;
                u32 *ptr = buf + (size_t)(off[r] + lo) * c->geo.np;
                if (cnt) NC(g_nccl.Broadcast(ptr, ptr, cnt, ncclUint32, r, c->comm, st));
        }
        NC(g_nccl.GroupEnd());
        return 0;
}

// push my rows of piece q (finished when `ready` fires) into every peer's copy of the block: one copy
// stream per peer offset (several copy engines), staggered so every receiver has one sender at a time
int piece_push(blk_ctx *c, const std::vector<u32 *> &peers, const std::vector<int64_t> &off,
               const std::vector<int64_t> &rows_all, int K, int q, cudaEvent_t ready)
{
        int64_t lo = rows_all[(size_t)c->rank * (K + 1) + q], hi = rows_all[(size_t)c->rank * (K + 1) + q + 1];
        size_t bytes = sizeof(u32) * (size_t)(hi - lo) * c->geo.np;
        size_t at = (size_t)(off[c->rank] + lo) * c->geo.np;
        for (int s = 1; s < c->world; s++) {
                int d = (c->rank + s) % c->world;
                CU(cudaStreamWaitEvent(c->copy_streams[s - 1], ready, 0));
                if (bytes) CU(cudaMemcpyAsync(peers[d] + at, peers[c->rank] + at, bytes, cudaMemcpyDeviceToDevice, c->copy_streams[s - 1]));
        }
        return 0;
}

// the main stream waits until all of this rank's pushes have left
int pushes_done(blk_ctx *c)
{
        for (size_t s = 0; s < c->copy_streams.size(); s++) {
                CU(cudaEventRecord(c->ev_copies[s], c->copy_streams[s]));
                CU(cudaStreamWaitEvent(c->stream, c->ev_copies[s], 0));
        }
        return 0;
}

// Build the column-blocked form of one product.  rkey/ckey/val: `count` entries on the device (global
// indices, a superset of this rank's rows); [lo, hi): this rank's output rows; cols: stored length of the
// input vector; in_off: block boundaries of the input dimension.  Block q < K-1 covers all local rows and
// the columns of input piece q of every rank; the last column block is cut into K output row pieces, so
// that output piece i is final -- and can travel -- as soon as its slice of the last block is done.
int build_colops(blk_ctx *c, blk_ctx::ColOps *ops, int K, int chunk_len, int64_t count, const int32_t *rkey,
                 const int32_t *ckey, const u32 *val, int64_t lo, int64_t hi, int64_t cols, const std::vector<int64_t> &in_off)
{
        const int W = c->world;
        ops->K = K;
        ops->col.assign((size_t)K - 1, SpOp());
        ops->last.assign((size_t)K, SpOp());
        ops->prow.assign((size_t)K + 1, 0);
        for (int i = 0; i <= K; i++) ops->prow[i] = (hi - lo) * i / K;
        std::vector<int64_t> hb((size_t)W * (K + 1));
        for (int r = 0; r < W; r++)
                for (int q = 0; q <= K; q++) hb[(size_t)r * (K + 1) + q] = piece_bound(in_off, r, q, K);
        int64_t *db = nullptr;
        unsigned long long *cnt = nullptr;
        CU(cudaMalloc(&db, sizeof(int64_t) * hb.size()));
        CU(cudaMalloc(&cnt, sizeof(unsigned long long)));
        CU(cudaMemcpyAsync(db, hb.data(), sizeof(int64_t) * hb.size(), cudaMemcpyHostToDevice, c->stream));
        int rc = 0;
        auto one = [&](SpOp *op, int q, int64_t rlo, int64_t rhi) -> int {
                unsigned long long h = 0;
                int32_t *sr = nullptr, *sc = nullptr;
                u32 *sx = nullptr;
                CU(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), c->stream));
                if (count) k_select_colblock<<<nb(count), 256, 0, c->stream>>>(count, rkey, ckey, val, rlo, rhi, W, K, q, db, nullptr, nullptr, nullptr, cnt);
                CU(cudaMemcpyAsync(&h, cnt, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
                CU(cudaStreamSynchronize(c->stream));
                const size_t cap = h ? (size_t)h : 1;
                CU(cudaMalloc(&sr, sizeof(int32_t) * cap));
                CU(cudaMalloc(&sc, sizeof(int32_t) * cap));
                CU(cudaMalloc(&sx, sizeof(u32) * cap));
                CU(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), c->stream));
                if (count) k_select_colblock<<<nb(count), 256, 0, c->stream>>>(count, rkey, ckey, val, rlo, rhi, W, K, q, db, sr, sc, sx, cnt);
                CU(cudaStreamSynchronize(c->stream));
                std::string err = build_operator(op, c->geo, chunk_len, rhi - rlo, cols, rlo, (int64_t)h, sr, sc, sx, c->m.p,
                                                 nullptr, nullptr, 1, c->stream);
                cudaFree(sr); cudaFree(sc); cudaFree(sx);
                if (!err.empty()) return fail("column block: " + err);
                return 0;
        };
        for (int q = 0; q < K - 1 && !rc; q++)
                if (hi > lo) rc = one(&ops->col[q], q, lo, hi);
        for (int i = 0; i < K && !rc; i++)
                if (ops->prow[i + 1] > ops->prow[i]) rc = one(&ops->last[i], K - 1, lo + ops->prow[i], lo + ops->prow[i + 1]);
        cudaFree(db); cudaFree(cnt);
        return rc;
}

void free_colops(blk_ctx::ColOps *ops)
{
        for (auto &o : ops->col) free_operator(&o);
        for (auto &o : ops->last) free_operator(&o);
        ops->col.clear(); ops->last.clear(); ops->K = 0;
}

// y (local rows) <- S x through the column blocks.  arrived[q] (nullable array) gates column block q;
// before_last() runs after the first K-1 blocks; after_piece(i) runs when output rows prow[i] .. prow[i+1] are final.  Returns the kernels launched, < 0 on error.
template <class B, class F>
int colblock_product(blk_ctx *c, blk_ctx::ColOps &ops, const u32 *x, u32 *y, const DevSmall *state, cudaEvent_t *arrived,
                     B before_last, F after_piece)
{
        const int K = ops.K, np = c->geo.np;
        int k = 0;
        for (int q = 0; q < K - 1; q++) {
                if (arrived && cudaStreamWaitEvent(c->stream, arrived[q], 0) != cudaSuccess) return -1;
                if (ops.col[q].rows > 0) k += launch_spmv(ops.col[q], c->geo, c->m, x, c->zbuf + (size_t)q * c->zstride, state, c->stream);
        }
        {
                int kb = before_last();        // work that must precede the first finished piece (returns kernels launched)
                if (kb < 0) return -1;
                k += kb;
        }
        if (arrived && cudaStreamWaitEvent(c->stream, arrived[K - 1], 0) != cudaSuccess) return -1;
        for (int i = 0; i < K; i++) {
                const int64_t lo = ops.prow[i], hi = ops.prow[i + 1];
                if (hi > lo) {
                        k += launch_spmv(ops.last[i], c->geo, c->m, x, c->zbuf + (size_t)(K - 1) * c->zstride + (size_t)lo * np, state, c->stream);
                        const int64_t cnt = (hi - lo) * np;
                        unsigned blocks = (unsigned)std::min<int64_t>(blk_sm_count() * 8, (cnt + 255) / 256);
                        k_combine_blocks<<<blocks, 256, 0, c->stream>>>(y + (size_t)lo * np, c->zbuf + (size_t)lo * np, K, c->zstride, cnt, c->m, state);
                        k += 1;
                }
                if (after_piece(i)) return -1;
        }
        return k;
}

// Copy rows [first16, first16 + count16) (in 16-byte units) of a block into the same place of every peer's copy:
// the exchange of a finished row piece over NVLink with plain coalesced stores.  A few CTAs saturate the
// link; running on the high-priority side stream they slip in between the blocks of the sparse product.
__global__ void __launch_bounds__(512)
k_push_rows(const uint4 *__restrict__ src, PushTargets push, size_t first16, size_t count16, const DevSmall *__restrict__ state)
{
        if (state && !state->do_ortho) return;            // the piece was not rewritten (halted iteration)
        const uint4 *s4 = src + first16;
        const size_t stride = (size_t)gridDim.x * blockDim.x;
        size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
        for (; i + 3 * stride < count16; i += 4 * stride) {
                uint4 a = __ldcg(s4 + i), b = __ldcg(s4 + i + stride), c = __ldcg(s4 + i + 2 * stride), d = __ldcg(s4 + i + 3 * stride);
                for (int q = 0; q < push.n; q++) {
                        uint4 *dst = reinterpret_cast<uint4 *>(push.y[q]) + first16;
                        dst[i] = a; dst[i + stride] = b; dst[i + 2 * stride] = c; dst[i + 3 * stride] = d;
                }
        }
        for (; i < count16; i += stride) {
                uint4 a = __ldcg(s4 + i);
                for (int q = 0; q < push.n; q++) (reinterpret_cast<uint4 *>(push.y[q]) + first16)[i] = a;
        }
}

// The same exchange with the bulk-copy (TMA) engine instead of load/store instructions: ONE thread per CTA streams
// 32 KB chunks of the piece through a ring in shared memory -- cp.async.bulk global -> shared (mbarrier completion),
// then one cp.async.bulk shared -> peer memory per peer (a bulk group per chunk).  No registers, no LSU slots and no
// warps to speak of: a CTA is 32 threads and 128 KB of shared memory, so it shares an SM with the resident blocks of
// the sparse product (which use no shared memory) instead of displacing one of them.
constexpr int PB_MAX_STAGES = 8;
#ifndef BLK_BULK_TIMEOUT_CYCLES
#define BLK_BULK_TIMEOUT_CYCLES 20000000000ll          // ~10 s of SM clock: trap instead of hanging the GPU
#endif

__global__ void __launch_bounds__(32)
k_push_bulk(const unsigned char *__restrict__ src, PushTargets push, size_t first, size_t bytes, const DevSmall *__restrict__ state,
            const int PB_STAGES, const unsigned PB_BYTES)
{
        extern __shared__ __align__(128) unsigned char pb_ring[];
        __shared__ __align__(8) unsigned long long pb_full[PB_MAX_STAGES];
        if (state && !state->do_ortho) return;            // the piece was not rewritten (halted iteration)
        if (threadIdx.x != 0) return;
        const size_t nchunks = (bytes + PB_BYTES - 1) / PB_BYTES;
        const size_t mine = nchunks > blockIdx.x ? (nchunks - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;      // chunks blockIdx.x + k * gridDim.x
        if (mine == 0) return;
        const uint32_t ring0 = (uint32_t)__cvta_generic_to_shared(pb_ring), bar0 = (uint32_t)__cvta_generic_to_shared(pb_full);
        for (int s = 0; s < PB_STAGES; s++) asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar0 + 8 * s), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        auto load = [&](size_t k) {
                const size_t off = ((size_t)blockIdx.x + k * gridDim.x) * PB_BYTES;
                const uint32_t len = (uint32_t)(bytes - off < PB_BYTES ? bytes - off : PB_BYTES);
                const uint32_t bar = bar0 + 8 * (uint32_t)(k % PB_STAGES), dst = ring0 + PB_BYTES * (uint32_t)(k % PB_STAGES);
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(len) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(dst), "l"(src + first + off), "r"(len), "r"(bar) : "memory");
        };
        for (size_t k = 0; k < mine && k < PB_STAGES - 1; k++) load(k);
        for (size_t k = 0; k < mine; k++) {
                const size_t off = ((size_t)blockIdx.x + k * gridDim.x) * PB_BYTES;
                const uint32_t len = (uint32_t)(bytes - off < PB_BYTES ? bytes - off : PB_BYTES);
                const uint32_t bar = bar0 + 8 * (uint32_t)(k % PB_STAGES), stage = ring0 + PB_BYTES * (uint32_t)(k % PB_STAGES);
                const uint32_t parity = (uint32_t)(k / PB_STAGES) & 1u;
                const long long t0 = clock64();
                for (;;) {
                        uint32_t ok;
                        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
                        if (ok) break;
                        if (clock64() - t0 > BLK_BULK_TIMEOUT_CYCLES) __trap();
                }
                for (int q = 0; q < push.n; q++)
                        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                                     ::"l"(reinterpret_cast<unsigned char *>(push.y[q]) + first + off), "r"(stage), "r"(len) : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                if (k + PB_STAGES - 1 < mine) {
                        // the stage chunk k + STAGES - 1 will land in was last read by the stores of chunk k - 1
                        asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                        load(k + PB_STAGES - 1);
                }
        }
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        __threadfence_system();
}

// peers' copies of a block, addressed from row `row0` on (see PushTargets)
PushTargets push_targets(const blk_ctx *c, const std::vector<u32 *> &peers, int64_t row0)
{
        PushTargets t;
        for (int s = 1; s < c->world && t.n < PushTargets::MAX; s++) {
                const int d = (c->rank + s) % c->world;             // staggered: rank r starts with peer r+1
                t.y[t.n++] = peers[d] + (size_t)row0 * c->geo.np;
        }
        return t;
}

// piece q of my rows of a row-sharded block -> every peer (one of the three exchange modes); `ready` fires when the
// piece is final.  state != null: the piece may be unchanged (k_push_rows then returns at once).
int exchange_piece(blk_ctx *c, u32 *buf, const std::vector<u32 *> &peers, const std::vector<int64_t> &off,
                   const std::vector<int64_t> &rows_all, int K, int q, cudaEvent_t ready, const DevSmall *state)
{
        if (c->xch == blk_ctx::XCH_CE) return piece_push(c, peers, off, rows_all, K, q, ready);
        CU(cudaStreamWaitEvent(c->comm_stream, ready, 0));
        if (c->xch == blk_ctx::XCH_NCCL) return piece_broadcast(c, buf, off, rows_all, K, q, c->comm_stream);
        const int64_t lo = rows_all[(size_t)c->rank * (K + 1) + q], hi = rows_all[(size_t)c->rank * (K + 1) + q + 1];
        const size_t per_row = (size_t)c->geo.np * sizeof(u32);
        // blocks start on 16-byte boundaries: row counts times np*4 bytes with np*4 a multiple of 16 for np >= 4;
        // for np < 4 the piece boundaries are rounded by the caller of this mode (see blk_create)
        const size_t first = (size_t)(off[c->rank] + lo) * per_row, bytes = (size_t)(hi - lo) * per_row;
        if (bytes == 0) return 0;
        if ((first | bytes) & 15) return fail("push exchange: piece not 16-byte aligned");
        PushTargets t = push_targets(c, peers, 0);
        if (c->push_bulk) {
                unsigned blocks = (unsigned)std::min<size_t>((size_t)c->push_ctas, (bytes + c->bulk_chunk - 1) / c->bulk_chunk);
                k_push_bulk<<<blocks, 32, (size_t)c->bulk_stages * c->bulk_chunk, c->comm_stream>>>(reinterpret_cast<const unsigned char *>(buf), t, first, bytes,
                                                                                                state, c->bulk_stages, c->bulk_chunk);
                c->launches++;
                return 0;
        }
        const size_t count16 = bytes / 16;
        unsigned blocks = (unsigned)std::min<size_t>((size_t)c->push_ctas, (count16 + 511) / 512);
        k_push_rows<<<blocks, 512, 0, c->comm_stream>>>(reinterpret_cast<const uint4 *>(buf), t, first / 16, count16, state);
        c->launches++;
        return 0;
}

// everything this rank has sent in the current exchange has left, and -- after the all-reduce that every rank
// enters only then -- everything sent to this rank has landed
int exchange_done(blk_ctx *c, bool have_allreduce_next)
{
        if (c->xch == blk_ctx::XCH_CE) {
                if (pushes_done(c)) return 1;
                if (!have_allreduce_next)
                        NC(g_nccl.AllReduce(c->barrier_word, c->barrier_word, 1, ncclUint64, ncclSum, c->comm, c->stream));
                return 0;
        }
        if (c->xch == blk_ctx::XCH_PUSH && !have_allreduce_next)
                NC(g_nccl.AllReduce(c->barrier_word, c->barrier_word, 1, ncclUint64, ncclSum, c->comm, c->comm_stream));
        CU(cudaEventRecord(c->ev_comm, c->comm_stream));
        CU(cudaStreamWaitEvent(c->stream, c->ev_comm, 0));
        return 0;
}

// Multi-GPU iteration.  Invariant at entry: tmp (full length, on every rank) = S1 v for the current
// v, Tp (local rows) = S1 p.  Because S1 is linear and the n x n factors act on the right,
//     S1 v' = sel(d, S1 Av, S1 v) + (S1 v) c + (S1 p) vtAvd,      S1 p' = sel(d, 0, S1 p) + (S1 v) winv
// i.e. exactly orthogonalize() applied to (tmp, S1 Av, Tp).  All values are canonical residues, so
// this is bit-identical to recomputing S1 v'.  What it buys: the only full-length vectors that
// cross NVLink are Av and the new tmp.  Av leaves from inside the product that computes it (XCH_PUSH:
// k_spmv stores every finished row into all copies, nothing is left to wait for but a barrier); the new tmp is
// produced in row pieces (product piece -> row-wise update -> exchange of the piece while the next one is
// computed); the new v is never gathered.
int enqueue_iteration_mg(blk_ctx *c, EventTimer *tm)
{
        const Geometry &g = c->geo;
        const int np = g.np;
        int k = 0;
        const int64_t lrows = c->n1() - c->n0();
        u32 *vloc = c->v + (size_t)c->n0() * np;
        u32 *tloc = c->tmp + (size_t)c->m0() * np;
        const bool fused_av = c->xch == blk_ctx::XCH_PUSH && c->push_av_in_spmv;

        // Av <- S2 tmp
        if (tm) tm->begin(c, BLK_PH_SPMV2);
        if (fused_av) {
                PushTargets t = push_targets(c, c->peer_av, c->n0());
                k += launch_spmv(c->S2, g, c->m, c->tmp, c->Av, c->state, c->stream, -1, &t);
        } else {
                // piece by piece; every finished piece travels while the next one runs
                for (int q = 0; q < c->pieces2; q++) {
                        k += launch_spmv(c->S2, g, c->m, c->tmp, c->Av, c->state, c->stream, q);
                        CU(cudaEventRecord(c->ev_piece[q], c->stream));
                        if (exchange_piece(c, c->Av_full, c->peer_av, c->n_off, c->piece_rows_all2, c->pieces2, q, c->ev_piece[q], nullptr)) return 1;
                }
        }
        c->launches += k;
        if (tm) tm->end(c, k);

        // dots on the local rows do not need the remote part of Av: they overlap the tail of the exchange
        if (tm) tm->begin(c, BLK_PH_DOTS);
        k = launch_dots(g, c->m, lrows, vloc, c->Av, c->sums, c->dots_blocks, c->state, SmallFuse(), c->stream);
        c->launches += k;
        if (tm) tm->end(c, k);
        if (tm) tm->begin(c, BLK_PH_EXCHANGE);
        // the all-reduce below completes only after every rank has reached it, i.e. (stream order) after every
        // rank's product 2 and its pushes: it is the barrier of the Av exchange
        if (!fused_av && exchange_done(c, true)) return 1;
        NC(g_nccl.AllReduce(c->sums, c->sums, (size_t)2 * np * np, ncclUint64, ncclSum, c->comm, c->stream));
        if (tm) tm->end(c, 0);
        if (tm) tm->begin(c, BLK_PH_SMALL);
        k = launch_small(g, c->m, c->sums, c->mats, c->state, 0, c->stream);
        c->launches += k;
        if (tm) tm->end(c, k);
        if (tm) tm->begin(c, BLK_PH_ORTHO);
        k = launch_ortho(g, c->m, lrows, vloc, c->Av, c->p, vloc, c->p, c->mats, c->state, 0, c->stream);
        c->launches += k;
        if (tm) tm->end(c, k);

        // tmp <- S1 v' through the recurrence: U = S1 Av (never skipped: the limit may just have been
        // reached), then orthogonalize(tmp, U, Tp) on the finished rows (skipped exactly when the real
        // orthogonalize is), then the exchange of the piece
        if (c->tmp_prev)
                CU(cudaMemcpyAsync(c->tmp_prev, tloc, sizeof(u32) * (size_t)(c->m1() - c->m0()) * np,
                                   cudaMemcpyDeviceToDevice, c->stream));
        if (tm) tm->begin(c, BLK_PH_SPMV1);
        k = 0;
        for (int q = 0; q < c->pieces; q++) {
                k += launch_spmv(c->S1, g, c->m, c->Av_full, c->U, nullptr, c->stream, q);
                int64_t lo = c->S1.piece_row[q], hi = c->S1.piece_row[q + 1];
                if (hi > lo)
                        k += launch_ortho(g, c->m, hi - lo, tloc + (size_t)lo * np, c->U + (size_t)lo * np, c->Tp + (size_t)lo * np,
                                          tloc + (size_t)lo * np, c->Tp + (size_t)lo * np, c->mats, c->state, 0, c->stream);
                CU(cudaEventRecord(c->ev_piece[q], c->stream));
                if (exchange_piece(c, c->tmp, c->peer_tmp, c->m_off, c->piece_rows_all, c->pieces, q, c->ev_piece[q], c->state)) return 1;
        }
        c->launches += k;
        if (tm) tm->end(c, k);
        if (tm) tm->begin(c, BLK_PH_EXCHANGE);
        if (exchange_done(c, false)) return 1;
        if (tm) tm->end(c, 0);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail(std::string("kernel launch: ") + cudaGetErrorString(e));
        return 0;
}

// Multi-GPU iteration with column-blocked consumers (BLK_COLBLOCKS=K, experimental; not yet measured).
// Same invariant and recurrence as enqueue_iteration_mg.  What changes is when work may start: a product
// begins with the column blocks whose input pieces have already landed, so the exchange of one product's
// result also hides behind the first K-1 blocks of the next product, and a product's last column block is
// computed in output-row pieces that are broadcast one by one.  Nothing on the main stream waits for a whole
// exchange except the n x n stage (its all-reduce is queued behind the Av broadcasts on the communicator's stream).
int enqueue_iteration_mg_arrival(blk_ctx *c, EventTimer *tm)
{
        const Geometry &g = c->geo;
        const int np = g.np, K = c->colblocks;
        const int64_t lrows = c->n1() - c->n0();
        u32 *vloc = c->v + (size_t)c->n0() * np;
        u32 *tloc = c->tmp + (size_t)c->m0() * np;
        cudaEvent_t *tmp_in = c->ev_arrived.data(), *av_in = tmp_in + K;
        auto nothing = []() -> int { return 0; };

        // Av <- S2 tmp
        if (tm) tm->begin(c, BLK_PH_SPMV2);
        int k = colblock_product(c, c->cb2, c->tmp, c->Av, c->state, tmp_in, nothing, [&](int i) -> int {
                CU(cudaEventRecord(c->ev_piece[i], c->stream));
                CU(cudaStreamWaitEvent(c->comm_stream, c->ev_piece[i], 0));
                if (piece_broadcast(c, c->Av_full, c->n_off, c->piece_rows_all2, K, i, c->comm_stream)) return 1;
                CU(cudaEventRecord(av_in[i], c->comm_stream));
                return 0;
        });
        if (k < 0) return g_err.empty() ? fail("column-blocked product 2") : 1;
        c->launches += k;
        if (tm) tm->end(c, k);

        if (tm) tm->begin(c, BLK_PH_DOTS);
        k = launch_dots(g, c->m, lrows, vloc, c->Av, c->sums, c->dots_blocks, c->state, SmallFuse(), c->stream);
        c->launches += k;
        if (tm) tm->end(c, k);
        CU(cudaEventRecord(c->ev_aux, c->stream));
        CU(cudaStreamWaitEvent(c->comm_stream, c->ev_aux, 0));
        NC(g_nccl.AllReduce(c->sums, c->sums, (size_t)2 * np * np, ncclUint64, ncclSum, c->comm, c->comm_stream));
        CU(cudaEventRecord(c->ev_comm, c->comm_stream));

        // U <- S1 Av, then tmp <- orthogonalize(tmp, U, Tp) piece by piece (the recurrence), each piece broadcast at once
        if (tm) tm->begin(c, BLK_PH_SPMV1);
        k = colblock_product(c, c->cb1, c->Av_full, c->U, nullptr, av_in,
                [&]() -> int {
                        // the n x n stage needs the all-reduce, which sits behind the last Av broadcast
                        if (cudaStreamWaitEvent(c->stream, c->ev_comm, 0) != cudaSuccess) return -1;
                        int kk = launch_small(g, c->m, c->sums, c->mats, c->state, 0, c->stream);
                        kk += launch_ortho(g, c->m, lrows, vloc, c->Av, c->p, vloc, c->p, c->mats, c->state, 0, c->stream);
                        if (c->tmp_prev &&
                            cudaMemcpyAsync(c->tmp_prev, tloc, sizeof(u32) * (size_t)(c->m1() - c->m0()) * np, cudaMemcpyDeviceToDevice,
                                            c->stream) != cudaSuccess)
                                return -1;
                        return kk;
                },
                [&](int i) -> int {
                        const int64_t lo = c->cb1.prow[i], hi = c->cb1.prow[i + 1];
                        if (hi > lo)
                                c->launches += launch_ortho(g, c->m, hi - lo, tloc + (size_t)lo * np, c->U + (size_t)lo * np, c->Tp + (size_t)lo * np,
                                                            tloc + (size_t)lo * np, c->Tp + (size_t)lo * np, c->mats, c->state, 0, c->stream);
                        CU(cudaEventRecord(c->ev_piece[i], c->stream));
                        CU(cudaStreamWaitEvent(c->comm_stream, c->ev_piece[i], 0));
                        if (piece_broadcast(c, c->tmp, c->m_off, c->piece_rows_all, K, i, c->comm_stream)) return 1;
                        CU(cudaEventRecord(tmp_in[i], c->comm_stream));
                        return 0;
                });
        if (k < 0) return g_err.empty() ? fail("column-blocked product 1") : 1;
        c->launches += k;
        if (tm) tm->end(c, k);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail(std::string("kernel launch: ") + cudaGetErrorString(e));
        return 0;
}

// the exchange of the last pieces may still be running on the communicator's stream
int drain_exchange(blk_ctx *c)
{
        if (c->colblocks && c->comm_stream) {
                CU(cudaEventRecord(c->ev_comm, c->comm_stream));
                CU(cudaStreamWaitEvent(c->stream, c->ev_comm, 0));
        }
        return 0;
}

// establish the invariant of enqueue_iteration_mg from v (full, on every rank) and p_full (may be null)
int mg_prepare(blk_ctx *c, const u32 *p_full_dev)
{
        const int np = c->geo.np;
        u32 *tloc = c->tmp + (size_t)c->m0() * np;
        c->launches += launch_spmv(c->S1, c->geo, c->m, c->v, tloc, nullptr, c->stream);
        if (allgather_rows(c, c->tmp, c->m_off)) return 1;
        int64_t lm = c->m1() - c->m0();
        if (p_full_dev) c->launches += launch_spmv(c->S1, c->geo, c->m, p_full_dev, c->Tp, nullptr, c->stream);
        else CU(cudaMemsetAsync(c->Tp, 0, sizeof(u32) * (size_t)(lm > 0 ? lm : 1) * np, c->stream));
        if (c->tmp_prev) CU(cudaMemsetAsync(c->tmp_prev, 0, sizeof(u32) * (size_t)(lm > 0 ? lm : 1) * np, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        return 0;
}

int grid_iteration(blk_ctx *c, EventTimer *tm);

// one iteration of the loop body, sequential/lanczos_modp.c:635-656
int enqueue_iteration(blk_ctx *c, EventTimer *tm)
{
        if (c->grid_on) return grid_iteration(c, tm);
        if (c->mg_recur) return c->colblocks ? enqueue_iteration_mg_arrival(c, tm) : enqueue_iteration_mg(c, tm);
        const Geometry &g = c->geo;
        const int np = g.np;
        int k;
        if (c->world > 1) {
                if (tm) tm->begin(c, BLK_PH_EXCHANGE);
                if (allgather_rows(c, c->v, c->n_off)) return 1;
                if (tm) tm->end(c, 0);
        }
        if (tm) tm->begin(c, BLK_PH_SPMV1);
        if (c->world > 1 && c->pieces > 1) {
                // product 1 in row pieces; piece q is broadcast by its owners while piece q+1 is computed
                const int K = c->pieces;
                k = 0;
                for (int q = 0; q < K; q++) {
                        k += launch_spmv(c->S1, g, c->m, c->v, c->tmp + (size_t)c->m0() * np, c->state, c->stream, q);
                        CU(cudaEventRecord(c->ev_piece[q], c->stream));
                        CU(cudaStreamWaitEvent(c->comm_stream, c->ev_piece[q], 0));
                        if (piece_broadcast(c, c->tmp, c->m_off, c->piece_rows_all, K, q, c->comm_stream)) return 1;
                }
                c->launches += k;
                if (tm) tm->end(c, k);
                if (tm) tm->begin(c, BLK_PH_EXCHANGE);          // only the part of the exchange that is not hidden
                CU(cudaEventRecord(c->ev_comm, c->comm_stream));
                CU(cudaStreamWaitEvent(c->stream, c->ev_comm, 0));
                if (tm) tm->end(c, 0);
        } else {
                if (c->colblocks && c->world == 1) {
                        k = colblock_product(c, c->cb1, c->v, c->tmp, c->state, nullptr, []() -> int { return 0; }, [](int) -> int { return 0; });
                        if (k < 0) return fail("column-blocked product 1");
                } else
                        k = launch_spmv(c->S1, g, c->m, c->v, c->tmp + (size_t)c->m0() * np, c->state, c->stream);
                c->launches += k;
                if (tm) tm->end(c, k);
                if (c->world > 1) {
                        if (tm) tm->begin(c, BLK_PH_EXCHANGE);
                        if (allgather_rows(c, c->tmp, c->m_off)) return 1;
                        if (tm) tm->end(c, 0);
                }
        }
        if (tm) tm->begin(c, BLK_PH_SPMV2);
        if (c->colblocks && c->world == 1) {
                k = colblock_product(c, c->cb2, c->tmp, c->Av, c->state, nullptr, []() -> int { return 0; }, [](int) -> int { return 0; });
                if (k < 0) return fail("column-blocked product 2");
        } else
                k = launch_spmv(c->S2, g, c->m, c->tmp, c->Av, c->state, c->stream);
        c->launches += k;
        if (tm) tm->end(c, k);

        int64_t lrows = c->n1() - c->n0();
        u32 *vloc = c->v + (size_t)c->n0() * np;
        if (tm) tm->begin(c, BLK_PH_DOTS);
        SmallFuse fuse;
        if (c->fuse_small) { fuse.counter = c->dots_counter; fuse.mats = c->mats; fuse.state = c->state; fuse.n = g.n; }
        k = launch_dots(g, c->m, lrows, vloc, c->Av, c->sums, c->dots_blocks, c->state, fuse, c->stream);
        c->launches += k;
        if (tm) tm->end(c, k);
        if (c->world > 1) {
                if (tm) tm->begin(c, BLK_PH_EXCHANGE);
                NC(g_nccl.AllReduce(c->sums, c->sums, (size_t)2 * np * np, ncclUint64, ncclSum, c->comm, c->stream));
                if (tm) tm->end(c, 0);
        }
        if (!c->fuse_small) {
                if (tm) tm->begin(c, BLK_PH_SMALL);
                k = launch_small(g, c->m, c->sums, c->mats, c->state, 0, c->stream);
                c->launches += k;
                if (tm) tm->end(c, k);
        }
        if (tm) tm->begin(c, BLK_PH_ORTHO);
        k = launch_ortho(g, c->m, lrows, vloc, c->Av, c->p, vloc, c->p, c->mats, c->state, 0, c->stream);
        c->launches += k;
        if (tm) tm->end(c, k);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail(std::string("kernel launch: ") + cudaGetErrorString(e));
        return 0;
}

// up to `iters` iterations in one launch of the persistent cooperative kernel (it stops by itself on `halt`)
int enqueue_loop_coop(blk_ctx *c, int iters)
{
        auto op = [](const SpOp &s) {
                LoopOp o;
                o.ent = s.ent; o.chunk_row = s.chunk_row; o.whead = s.whead; o.tail_row = s.tail_row; o.span = s.span;
                o.ntiles = s.ntiles; o.Q = s.Q; o.rows = (u32)s.rows; o.crossing = s.crossing ? 1 : 0;
                return o;
        };
        LoopArgs a;
        a.s1 = op(c->S1); a.s2 = op(c->S2);
        a.v = c->v; a.tmp = c->tmp; a.Av = c->Av; a.p = c->p;
        a.N = c->N;
        a.sums = (unsigned long long *)c->sums; a.mats = c->mats; a.state = c->state; a.m = c->m;
        a.n = c->geo.n; a.max_iters = iters; a.bar = c->loop_bar;
        unsigned long long *clocks = reinterpret_cast<unsigned long long *>(c->loop_bar + 2);
        const bool prof = c->profiling && c->coop_prof;
        if (prof) { a.prof = clocks; CU(cudaMemsetAsync(clocks, 0, 6 * sizeof(unsigned long long), c->stream)); }
        std::string err;
        if (launch_loop_coop(a, c->geo.n, c->geo.np, c->coop_grid, c->stream, &err)) return fail(err);
        c->launches += 1;
        if (prof) {
                // SM cycles of block 0 -> ms at the SM clock the driver reports (phases include the barrier that ends them)
                unsigned long long h[6];
                int khz = 0;
                CU(cudaMemcpyAsync(h, clocks, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
                CU(cudaStreamSynchronize(c->stream));
                CU(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, c->device));
                const double ms = khz > 0 ? 1.0 / khz : 0.0;
                c->ph_ms[BLK_PH_SPMV1] += (double)(h[0] + h[1]) * ms; c->ph_ms[BLK_PH_SPMV2] += (double)(h[2] + h[3]) * ms;
                c->ph_ms[BLK_PH_DOTS] += (double)h[4] * ms; c->ph_ms[BLK_PH_ORTHO] += (double)h[5] * ms;
                c->ph_ms[BLK_PH_EXCHANGE] += (double)(h[1] + h[3]) * ms;     // (reported apart: the two fix-up phases)
        }
        return 0;
}

int push_state(blk_ctx *c)
{
        CU(cudaMemcpyAsync(c->state, c->h_state, sizeof(DevSmall), cudaMemcpyHostToDevice, c->stream));
        return 0;
}
int pull_state(blk_ctx *c)
{
        CU(cudaMemcpyAsync(c->h_state, c->state, sizeof(DevSmall), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        return 0;
}

// host block (rows x n, row-major) -> device block with leading dimension np.  `map` (device, nullable: old
// label -> new label, whole dimension): host row r0 + r goes to device row map[r0 + r] of `dst`; without a map to
// row r of `dst`.  Repacking goes through a resident 64 MB staging buffer, chunk by chunk in stream order (the
// PCIe copy dominates; no allocation per call).
int upload_rows(blk_ctx *c, u32 *dst, const u32 *src_host, int64_t rows, const u32 *map = nullptr, int64_t r0 = 0)
{
        const int n = c->geo.n, np = c->geo.np;
        if (rows == 0) return 0;
        if (n == np && !map) {
                CU(cudaMemcpyAsync(dst, src_host, sizeof(u32) * (size_t)rows * n, cudaMemcpyHostToDevice, c->stream));
                CU(cudaStreamSynchronize(c->stream));
                return 0;
        }
        const int64_t per = std::max<int64_t>(1, (int64_t)(2 * blk_ctx::STAGE_BYTES / (sizeof(u32) * n)));
        for (int64_t at = 0; at < rows; at += per) {
                const int64_t cnt = std::min(per, rows - at);
                CU(cudaMemcpyAsync(c->stage, src_host + (size_t)at * n, sizeof(u32) * (size_t)cnt * n, cudaMemcpyHostToDevice, c->stream));
                c->launches += launch_pad_rows(c->stage, map ? dst : dst + (size_t)at * np, cnt, n, np, map, r0 + at, c->stream);
        }
        CU(cudaStreamSynchronize(c->stream));
        return 0;
}
// `map` (device, nullable): host row r0 + r comes from device row map[r0 + r] of `src` (else row r of `src`).
// w / wp: words per host / device row (0: n / n_pad)
int download_rows(blk_ctx *c, u32 *dst_host, const u32 *src, int64_t rows, const u32 *map = nullptr, int64_t r0 = 0,
                  int w = 0, int wp = 0)
{
        const int n = w ? w : c->geo.n, np = wp ? wp : c->geo.np;
        if (rows == 0) return 0;
        if (n == np && !map) {
                CU(cudaMemcpyAsync(dst_host, src, sizeof(u32) * (size_t)rows * n, cudaMemcpyDeviceToHost, c->stream));
                CU(cudaStreamSynchronize(c->stream));
                return 0;
        }
        const int64_t per = std::max<int64_t>(1, (int64_t)(2 * blk_ctx::STAGE_BYTES / (sizeof(u32) * n)));
        for (int64_t at = 0; at < rows; at += per) {
                const int64_t cnt = std::min(per, rows - at);
                c->launches += launch_unpad_rows(map ? src : src + (size_t)at * np, c->stage, cnt, n, np, map, r0 + at, c->stream);
                CU(cudaMemcpyAsync(dst_host + (size_t)at * n, c->stage, sizeof(u32) * (size_t)cnt * n, cudaMemcpyDeviceToHost, c->stream));
        }
        CU(cudaStreamSynchronize(c->stream));
        return 0;
}

// ---- P x Q block grid ---------------------------------------------------------------------------
// The iteration on the grid is specified, and pinned bit for bit on the CPU, by tests/test_grid_cpu.py; this is
// its device side.  Not yet run on GPUs (no multi-GPU time was left in round 1): BLK_GRID=PxQ|auto.

// Plan (same rules as blk_plan_grid), block extraction, operators, buffers, sub-communicators.
// cntN / cntM: entries per row of the N / Mc dimension (host); iN / iM / val: the COO on the device.
int grid_create(blk_ctx *c, int P, int Q, int chunk_len, int64_t nnz, const int32_t *iN, const int32_t *iM, const u32 *val,
                const std::vector<u32> &cntN, const std::vector<u32> &cntM)
{
        blk_ctx::Grid &G = c->grid;
        const int np = c->geo.np, W = c->world;
        if (!g_nccl.Send || !g_nccl.Recv || !g_nccl.CommSplit) return fail("BLK_GRID needs ncclSend / ncclRecv / ncclCommSplit (NCCL >= 2.18)");
        if (P == 0 && Q == 0) {
                Q = 1;
                for (int q = 1; (int64_t)q * q <= W; q++)
                        if (W % q == 0) Q = q;
                P = W / Q;
        }
        if (P < 1 || Q < 1 || P * Q != W) return fail("BLK_GRID: P x Q must equal the number of ranks");
        G.P = P; G.Q = Q; G.a = c->rank / Q; G.b = c->rank % Q;
        G.n_off = partition_rows(cntN, P);
        G.m_off = partition_rows(cntM, Q);
        G.n_sub.assign((size_t)P * (Q + 1), 0);
        G.m_sub.assign((size_t)Q * (P + 1), 0);
        for (int a = 0; a < P; a++)
                for (int b = 0; b <= Q; b++) G.n_sub[(size_t)a * (Q + 1) + b] = G.n_off[a] + (G.n_off[a + 1] - G.n_off[a]) * b / Q;
        for (int b = 0; b < Q; b++)
                for (int a = 0; a <= P; a++) G.m_sub[(size_t)b * (P + 1) + a] = G.m_off[b] + (G.m_off[b + 1] - G.m_off[b]) * a / P;
        auto ceil_div = [](int64_t x, int64_t y) { return (x + y - 1) / y; };
        G.pieceNmax = G.pieceMmax = 1;
        for (int a = 0; a < P; a++) G.pieceNmax = std::max(G.pieceNmax, ceil_div(G.n_off[a + 1] - G.n_off[a], Q));
        for (int b = 0; b < Q; b++) G.pieceMmax = std::max(G.pieceMmax, ceil_div(G.m_off[b + 1] - G.m_off[b], P));
        G.pieceN = std::max<int64_t>(1, ceil_div(G.n_off[G.a + 1] - G.n_off[G.a], Q));
        G.pieceM = std::max<int64_t>(1, ceil_div(G.m_off[G.b + 1] - G.m_off[G.b], P));
        const int64_t rowsN = G.pieceN * Q, rowsM = G.pieceM * P;

        // ---- block (a,b) with piece-padded local indices
        int64_t *dn = nullptr, *dm = nullptr;
        unsigned long long *cnt = nullptr, h = 0;
        CU(cudaMalloc(&dn, sizeof(int64_t) * (Q + 1)));
        CU(cudaMalloc(&dm, sizeof(int64_t) * (P + 1)));
        CU(cudaMalloc(&cnt, sizeof(unsigned long long)));
        CU(cudaMemcpyAsync(dn, &G.n_sub[(size_t)G.a * (Q + 1)], sizeof(int64_t) * (Q + 1), cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemcpyAsync(dm, &G.m_sub[(size_t)G.b * (P + 1)], sizeof(int64_t) * (P + 1), cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), c->stream));
        if (nnz) k_select_grid<<<nb(nnz), 256, 0, c->stream>>>(nnz, iN, iM, val, Q, dn, G.pieceN, P, dm, G.pieceM, nullptr, nullptr, nullptr, cnt);
        CU(cudaMemcpyAsync(&h, cnt, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        const size_t cap = h ? (size_t)h : 1;
        int32_t *ln = nullptr, *lm = nullptr;
        u32 *lx = nullptr;
        CU(cudaMalloc(&ln, sizeof(int32_t) * cap));
        CU(cudaMalloc(&lm, sizeof(int32_t) * cap));
        CU(cudaMalloc(&lx, sizeof(u32) * cap));
        CU(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), c->stream));
        if (nnz) k_select_grid<<<nb(nnz), 256, 0, c->stream>>>(nnz, iN, iM, val, Q, dn, G.pieceN, P, dm, G.pieceM, ln, lm, lx, cnt);
        CU(cudaStreamSynchronize(c->stream));
        // S1: partial tmp_b (rows: Mc-block b) <- v_a ; S2: partial Av_a (rows: N-block a) <- tmp_b
        std::string err = build_operator(&G.S1, c->geo, chunk_len, rowsM, rowsN, 0, (int64_t)h, lm, ln, lx, c->m.p, nullptr, nullptr, 1, c->stream);
        if (err.empty())
                err = build_operator(&G.S2, c->geo, chunk_len, rowsN, rowsM, 0, (int64_t)h, ln, lm, lx, c->m.p, nullptr, nullptr, 1, c->stream);
        cudaFree(ln); cudaFree(lm); cudaFree(lx); cudaFree(dn); cudaFree(dm); cudaFree(cnt);
        if (!err.empty()) return fail("grid block: " + err);

        // ---- buffers
        const size_t bN = sizeof(u32) * (size_t)rowsN * np, bM = sizeof(u32) * (size_t)rowsM * np;
        const size_t brecv = sizeof(u32) * (size_t)std::max<int64_t>(1, std::max((P - 1) * G.pieceM, (Q - 1) * G.pieceN)) * np;
        const size_t bown = sizeof(u32) * (size_t)G.pieceN * np;
        CU(cudaMalloc(&G.vblk, bN)); CU(cudaMalloc(&G.tblk, bM)); CU(cudaMalloc(&G.part1, bM)); CU(cudaMalloc(&G.part2, bN));
        CU(cudaMalloc(&G.recv, brecv));
        CU(cudaMalloc(&G.Av, bown)); CU(cudaMalloc(&G.p, bown));
        CU(cudaMemsetAsync(G.vblk, 0, bN, c->stream)); CU(cudaMemsetAsync(G.tblk, 0, bM, c->stream));
        CU(cudaMemsetAsync(G.part1, 0, bM, c->stream)); CU(cudaMemsetAsync(G.part2, 0, bN, c->stream));
        CU(cudaMemsetAsync(G.recv, 0, brecv, c->stream));
        CU(cudaMemsetAsync(G.Av, 0, bown, c->stream)); CU(cudaMemsetAsync(G.p, 0, bown, c->stream));
        c->block_bytes += 2 * bN + 2 * bM + brecv + 2 * bown;
        CU(cudaStreamSynchronize(c->stream));

        // ---- communicators of my grid row (ranks a*Q .. a*Q+Q-1, my index b) and column (index a)
        NC(g_nccl.CommSplit(c->comm, G.a, G.b, &G.row_comm, nullptr));
        NC(g_nccl.CommSplit(c->comm, P + G.b, G.a, &G.col_comm, nullptr));
        c->grid_on = true;
        return 0;
}

void grid_destroy(blk_ctx *c)
{
        blk_ctx::Grid &G = c->grid;
        if (G.row_comm && g_nccl.CommDestroy) g_nccl.CommDestroy(G.row_comm);
        if (G.col_comm && g_nccl.CommDestroy) g_nccl.CommDestroy(G.col_comm);
        free_operator(&G.S1); free_operator(&G.S2);
        cudaFree(G.vblk); cudaFree(G.tblk); cudaFree(G.part1); cudaFree(G.part2); cudaFree(G.recv); cudaFree(G.Av); cudaFree(G.p);
}

// all-to-all of the pieces of a partial block inside a group + local sum mod p: out <- my piece of the sum
int grid_reduce_scatter(blk_ctx *c, ncclComm_t comm, int size, int me, const u32 *part, int64_t piece_rows, u32 *out)
{
        blk_ctx::Grid &G = c->grid;
        const size_t cnt = (size_t)piece_rows * c->geo.np;
        if (size > 1) {
                NC(g_nccl.GroupStart());
                for (int k = 0; k < size; k++) {
                        if (k == me) continue;
                        NC(g_nccl.Send(part + (size_t)k * cnt, cnt, ncclUint32, k, comm, c->stream));
                        NC(g_nccl.Recv(G.recv + (size_t)(k < me ? k : k - 1) * cnt, cnt, ncclUint32, k, comm, c->stream));
                }
                NC(g_nccl.GroupEnd());
        }
        unsigned blocks = (unsigned)std::min<int64_t>(blk_sm_count() * 8, ((int64_t)cnt + 255) / 256);
        k_sum_pieces<<<blocks ? blocks : 1, 256, 0, c->stream>>>(out, part + (size_t)me * cnt, G.recv, size - 1, cnt, (int64_t)cnt, c->m);
        c->launches += 1;
        return 0;
}

// one iteration on the grid (steps 1-7 of tests/test_grid_cpu.py)
int grid_iteration(blk_ctx *c, EventTimer *tm)
{
        blk_ctx::Grid &G = c->grid;
        const Geometry &g = c->geo;
        const int np = g.np;
        const size_t cN = (size_t)G.pieceN * np, cM = (size_t)G.pieceM * np;
        u32 *vown = G.vblk + (size_t)G.b * cN;
        int k;
        if (tm) tm->begin(c, BLK_PH_EXCHANGE);
        if (G.Q > 1) NC(g_nccl.AllGather(vown, G.vblk, cN, ncclUint32, G.row_comm, c->stream));
        if (tm) tm->end(c, 0);
        if (tm) tm->begin(c, BLK_PH_SPMV1);
        k = launch_spmv(G.S1, g, c->m, G.vblk, G.part1, c->state, c->stream);
        c->launches += k;
        if (tm) tm->end(c, k);
        if (tm) tm->begin(c, BLK_PH_EXCHANGE);
        if (grid_reduce_scatter(c, G.col_comm, G.P, G.a, G.part1, G.pieceM, G.tblk + (size_t)G.a * cM)) return 1;
        if (G.P > 1) NC(g_nccl.AllGather(G.tblk + (size_t)G.a * cM, G.tblk, cM, ncclUint32, G.col_comm, c->stream));
        if (tm) tm->end(c, 1);
        if (tm) tm->begin(c, BLK_PH_SPMV2);
        k = launch_spmv(G.S2, g, c->m, G.tblk, G.part2, c->state, c->stream);
        c->launches += k;
        if (tm) tm->end(c, k);
        if (tm) tm->begin(c, BLK_PH_EXCHANGE);
        if (grid_reduce_scatter(c, G.row_comm, G.Q, G.b, G.part2, G.pieceN, G.Av)) return 1;
        if (tm) tm->end(c, 1);
        if (tm) tm->begin(c, BLK_PH_DOTS);
        k = launch_dots(g, c->m, G.pieceN, vown, G.Av, c->sums, dots_num_blocks(G.pieceN, np), c->state, SmallFuse(), c->stream);
        c->launches += k;
        if (tm) tm->end(c, k);
        if (tm) tm->begin(c, BLK_PH_EXCHANGE);
        NC(g_nccl.AllReduce(c->sums, c->sums, (size_t)2 * np * np, ncclUint64, ncclSum, c->comm, c->stream));
        if (tm) tm->end(c, 0);
        if (tm) tm->begin(c, BLK_PH_SMALL);
        k = launch_small(g, c->m, c->sums, c->mats, c->state, 0, c->stream);
        c->launches += k;
        if (tm) tm->end(c, k);
        if (tm) tm->begin(c, BLK_PH_ORTHO);
        k = launch_ortho(g, c->m, G.pieceN, vown, G.Av, G.p, vown, G.p, c->mats, c->state, 0, c->stream);
        c->launches += k;
        if (tm) tm->end(c, k);
        G.dirty = true;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail(std::string("kernel launch: ") + cudaGetErrorString(e));
        return 0;
}

// blk_set_state has put the full v into c->v (device); p_host may be null.  Fill the grid's blocks.
int grid_import(blk_ctx *c, const u32 *p_host)
{
        blk_ctx::Grid &G = c->grid;
        const int np = c->geo.np, n = c->geo.n, Q = G.Q, P = G.P;
        const size_t cN = (size_t)G.pieceN * np;
        CU(cudaMemsetAsync(G.vblk, 0, sizeof(u32) * cN * Q, c->stream));
        CU(cudaMemsetAsync(G.tblk, 0, sizeof(u32) * (size_t)G.pieceM * np * P, c->stream));
        CU(cudaMemsetAsync(G.Av, 0, sizeof(u32) * cN, c->stream));
        CU(cudaMemsetAsync(G.p, 0, sizeof(u32) * cN, c->stream));
        for (int b = 0; b < Q; b++) {
                const int64_t lo = G.n_sub[(size_t)G.a * (Q + 1) + b], hi = G.n_sub[(size_t)G.a * (Q + 1) + b + 1];
                if (hi > lo)
                        CU(cudaMemcpyAsync(G.vblk + (size_t)b * cN, c->v + (size_t)lo * np, sizeof(u32) * (size_t)(hi - lo) * np,
                                           cudaMemcpyDeviceToDevice, c->stream));
        }
        if (p_host) {
                const int64_t lo = G.n_sub[(size_t)G.a * (Q + 1) + G.b], hi = G.n_sub[(size_t)G.a * (Q + 1) + G.b + 1];
                if (hi > lo && upload_rows(c, G.p, p_host + (size_t)lo * n, hi - lo)) return 1;
        }
        G.dirty = false;
        return 0;
}

// Copy the distributed state into the 1-D blocks everything outside the loop works on: c->v and c->tmp in
// full on every rank, c->Av and c->p on this rank's 1-D rows [n0, n1).
int grid_export(blk_ctx *c)
{
        blk_ctx::Grid &G = c->grid;
        if (!G.dirty) return 0;
        const int np = c->geo.np, P = G.P, Q = G.Q, W = c->world;
        u32 *stage = nullptr;
        const size_t slotN = (size_t)G.pieceNmax * np, slotM = (size_t)G.pieceMmax * np;
        CU(cudaMalloc(&stage, sizeof(u32) * std::max(slotN, slotM) * W));
        struct Item { const u32 *src; size_t have; bool alongN; u32 *dst; int64_t dlo, dhi; };   // dst covers global rows [dlo, dhi)
        const Item items[4] = {
                {G.vblk + (size_t)G.b * G.pieceN * np, (size_t)G.pieceN * np, true, c->v, 0, c->N},
                {G.tblk + (size_t)G.a * G.pieceM * np, (size_t)G.pieceM * np, false, c->tmp, 0, c->Mc},
                {G.Av, (size_t)G.pieceN * np, true, c->Av, c->n0(), c->n1()},
                {G.p, (size_t)G.pieceN * np, true, c->p, c->n0(), c->n1()},
        };
        for (const Item &it : items) {
                const size_t slot = it.alongN ? slotN : slotM;
                CU(cudaMemsetAsync(stage + (size_t)c->rank * slot, 0, sizeof(u32) * slot, c->stream));
                CU(cudaMemcpyAsync(stage + (size_t)c->rank * slot, it.src, sizeof(u32) * it.have, cudaMemcpyDeviceToDevice, c->stream));
                NC(g_nccl.AllGather(stage + (size_t)c->rank * slot, stage, slot, ncclUint32, c->comm, c->stream));
                for (int r = 0; r < W; r++) {
                        const int a = r / Q, b = r % Q;
                        int64_t lo, hi;
                        if (it.alongN) { lo = G.n_sub[(size_t)a * (Q + 1) + b]; hi = G.n_sub[(size_t)a * (Q + 1) + b + 1]; }
                        else { lo = G.m_sub[(size_t)b * (P + 1) + a]; hi = G.m_sub[(size_t)b * (P + 1) + a + 1]; }
                        const int64_t l2 = std::max(lo, it.dlo), h2 = std::min(hi, it.dhi);
                        if (h2 > l2)
                                CU(cudaMemcpyAsync(it.dst + (size_t)(l2 - it.dlo) * np, stage + (size_t)r * slot + (size_t)(l2 - lo) * np,
                                                   sizeof(u32) * (size_t)(h2 - l2) * np, cudaMemcpyDeviceToDevice, c->stream));
                }
        }
        CU(cudaStreamSynchronize(c->stream));
        cudaFree(stage);
        G.dirty = false;
        return 0;
}

void destroy_graph(blk_ctx *c)
{
        if (c->graph) { cudaGraphExecDestroy(c->graph); c->graph = nullptr; }
}

int build_graph(blk_ctx *c)
{
        cudaGraph_t g = nullptr;
        CU(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
        int64_t before = c->launches;
        int rc = 0;
        for (int i = 0; i < blk_ctx::GRAPH_ITERS && !rc; i++) rc = enqueue_iteration(c, nullptr);
        c->launches = before;       // counted when the graph is launched
        cudaError_t e = cudaStreamEndCapture(c->stream, &g);
        if (rc) { if (g) cudaGraphDestroy(g); return 1; }
        if (e != cudaSuccess) return fail(std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
        e = cudaGraphInstantiate(&c->graph, g, 0);
        cudaGraphDestroy(g);
        if (e != cudaSuccess) return fail(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e));
        return 0;
}

int kernels_per_iteration(const blk_ctx *c)
{
        // two products (+ their k_spmv_fix unless the rows crossing tiles are finished by look-back; banded products: every band
        // plus the pass that adds the partial results), dots, [small], orthogonalize
        auto banded = [](const SpOp &op) {
                if (op.bands.empty()) return op.lookback ? 1 : 2;
                int k = 1;
                for (const SpOp &b : op.bands) k += b.lookback ? 1 : 2;
                return k;
        };
        auto product = [&](const SpOp &op) {
                if (op.split.empty()) return banded(op);
                return banded(op.split[0]) + 1 + (op.split[1].rows > 0 ? banded(op.split[1]) : 0);
        };
        return product(c->S1) + product(c->S2) + 1 + (c->fuse_small ? 0 : 1) + 1;
}

}  // namespace

HeavyPlan plan_heavy(const u32 *deg, int64_t rows, int64_t cols, int np, int64_t l2_bytes, int64_t min_deg, int64_t band_bytes,
                     bool force)
{
        HeavyPlan plan;
        const int64_t x_bytes = cols * np * 4;
        if (np < 8 || rows <= 0 || cols <= 0 || band_bytes <= 0 || (!force && x_bytes <= l2_bytes)) return plan;
        const int64_t K = std::min<int64_t>(256, (x_bytes + band_bytes - 1) / band_bytes);
        if (K < 2) return plan;
        int64_t H = 0, heavy_nnz = 0;
        while (H < rows && (int64_t)deg[H] >= min_deg) heavy_nnz += deg[H++];
        if (H == 0) return plan;
        // Bytes of HBM time per iteration: every heavy non-zero stops fetching its own line from HBM but still gathers from its
        // band's slice (measured on config 4: 71 G gathers/s against ~5.9 TB/s, worth ~83 bytes); every (heavy row, band)
        // writes and reads a partial row of 4 * n_pad bytes and streams one dummy entry when the row has nothing in the band.
        // (At n_pad = 32 this says no, and the split measured slower there: 40.3 against 37.7 ms per product.)
        const double line = std::max(128, 4 * np), l2_gather = 83.0;
        const double saving = (line - l2_gather) * (double)heavy_nnz - (8.0 * np + 8.0) * (double)H * (double)K;
        if (!force && saving <= 0) return plan;
        plan.rows = H;
        plan.bands = (int)K;
        return plan;
}

// ---- blk_create, in pieces ------------------------------------------------------------------------
namespace {

// device allocations that live only during blk_create: freed on every exit path
struct Scratch {
        std::vector<void *> ptrs;
        ~Scratch() { for (void *q : ptrs) cudaFree(q); }
        template <class T> int alloc(T **out, size_t bytes)
        {
                *out = nullptr;
                cudaError_t e = cudaMalloc((void **)out, bytes ? bytes : 16);
                if (e != cudaSuccess) return fail(std::string("cudaMalloc (blk_create scratch): ") + cudaGetErrorString(e));
                ptrs.push_back(*out);
                return 0;
        }
        void release(void *q)
        {
                for (auto &x : ptrs)
                        if (x == q) { cudaFree(q); x = nullptr; }
        }
};

bool env_flag(const char *name)
{
        const char *e = getenv(name);
        return e && e[0] && e[0] != '0';
}

// entries per row of one dimension (host copy)
int count_dimension(blk_ctx *c, int64_t nnz, const int32_t *idx, int64_t dim, std::vector<u32> *out, const u32 *map = nullptr)
{
        Scratch tmp;
        u32 *dc = nullptr;
        if (tmp.alloc(&dc, sizeof(u32) * (size_t)dim)) return 1;
        CU(cudaMemsetAsync(dc, 0, sizeof(u32) * (size_t)dim, c->stream));
        if (nnz) k_count_rows<<<nb(nnz), 256, 0, c->stream>>>(nnz, idx, dim, dc, map);
        out->assign((size_t)dim, 0);
        if (dim) CU(cudaMemcpyAsync(out->data(), dc, sizeof(u32) * (size_t)dim, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        return 0;
}

void single_piece(SpOp *op)
{
        op->piece_tile.assign({0, op->ntiles});
        op->piece_row.assign({0, op->rows});
        op->piece_scan.assign({0, 0});
}

// Every rank needs every rank's piece boundaries of both operators, and all ranks must use the same number
// of pieces: build_operator falls back to one piece on a rank whose shard has too few tiles, so the counts
// are compared here and, on any disagreement, EVERY rank drops to one piece (operator included).
int agree_pieces(blk_ctx *c)
{
        const int world = c->world;
        for (int which = 0; which < 2; which++) {
                SpOp &op = which ? c->S2 : c->S1;
                const int KMAX = 32;
                std::vector<long long> mine(KMAX + 2, 0), all((size_t)(KMAX + 2) * world, 0);
                int K = (int)op.piece_tile.size() - 1;
                mine[0] = K;
                for (int k = 0; k <= K; k++) mine[1 + k] = op.piece_row[k];
                Scratch tmp;
                long long *dbuf = nullptr;
                if (tmp.alloc(&dbuf, sizeof(long long) * all.size())) return 1;
                CU(cudaMemcpyAsync(dbuf + (size_t)c->rank * (KMAX + 2), mine.data(), sizeof(long long) * (KMAX + 2),
                                   cudaMemcpyHostToDevice, c->stream));
                NC(g_nccl.AllGather(dbuf + (size_t)c->rank * (KMAX + 2), dbuf, (size_t)(KMAX + 2), ncclInt64, c->comm, c->stream));
                CU(cudaMemcpyAsync(all.data(), dbuf, sizeof(long long) * all.size(), cudaMemcpyDeviceToHost, c->stream));
                CU(cudaStreamSynchronize(c->stream));
                bool same = true;
                for (int r = 0; r < world; r++) same = same && all[(size_t)r * (KMAX + 2)] == K;
                std::vector<int64_t> &dst = which ? c->piece_rows_all2 : c->piece_rows_all;
                int &Kd = which ? c->pieces2 : c->pieces;
                if (same) {
                        Kd = K;
                        dst.assign((size_t)world * (K + 1), 0);
                        for (int r = 0; r < world; r++)
                                for (int k = 0; k <= K; k++)
                                        dst[(size_t)r * (K + 1) + k] = all[(size_t)r * (KMAX + 2) + 1 + k];
                } else {
                        Kd = 1;
                        single_piece(&op);
                        dst.assign((size_t)world * 2, 0);
                        const std::vector<int64_t> &off = which ? c->n_off : c->m_off;
                        for (int r = 0; r < world; r++) dst[(size_t)r * 2 + 1] = off[r + 1] - off[r];
                }
        }
        return 0;
}

// all ranks take the same path: true only if `mine` holds on every rank
int agree_flag(blk_ctx *c, bool mine, bool *all)
{
        Scratch tmp;
        unsigned long long *flag = nullptr, h = mine ? 1ull : 0ull;
        if (tmp.alloc(&flag, sizeof(h))) return 1;
        CU(cudaMemcpyAsync(flag, &h, sizeof(h), cudaMemcpyHostToDevice, c->stream));
        NC(g_nccl.AllReduce(flag, flag, 1, ncclUint64, ncclSum, c->comm, c->stream));
        CU(cudaMemcpyAsync(&h, flag, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        *all = h == (unsigned long long)c->world;
        return 0;
}

// Map every rank's tmp and Av_full into this rank's address space: raw pointers + peer access when the owner
// lives in this process (one thread per GPU), CUDA IPC handles otherwise (one process per GPU).
int setup_peers(blk_ctx *c, bool *ok_all)
{
        struct Record {
                int32_t pid, device;
                unsigned long long tmp, av;
                cudaIpcMemHandle_t h_tmp, h_av;
        };
        const int world = c->world;
        Record mine;
        memset(&mine, 0, sizeof(mine));
        mine.pid = (int32_t)getpid(); mine.device = c->device;
        mine.tmp = (unsigned long long)(uintptr_t)c->tmp; mine.av = (unsigned long long)(uintptr_t)c->Av_full;
        const bool ipc_ok = cudaIpcGetMemHandle(&mine.h_tmp, c->tmp) == cudaSuccess &&
                            cudaIpcGetMemHandle(&mine.h_av, c->Av_full) == cudaSuccess;
        cudaGetLastError();
        Scratch tmp;
        unsigned char *dh = nullptr;
        if (tmp.alloc(&dh, sizeof(Record) * world)) return 1;
        CU(cudaMemcpyAsync(dh + sizeof(Record) * c->rank, &mine, sizeof(Record), cudaMemcpyHostToDevice, c->stream));
        NC(g_nccl.AllGather(dh + sizeof(Record) * c->rank, dh, sizeof(Record), ncclUint8, c->comm, c->stream));
        std::vector<Record> all(world);
        CU(cudaMemcpyAsync(all.data(), dh, sizeof(Record) * world, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        bool ok = true;
        c->peer_tmp.assign(world, nullptr); c->peer_av.assign(world, nullptr); c->peer_ipc.assign(world, 0);
        c->peer_tmp[c->rank] = c->tmp; c->peer_av[c->rank] = c->Av_full;
        for (int r = 0; r < world && ok; r++) {
                if (r == c->rank) continue;
                if (all[r].pid == mine.pid) {
                        int can = 0;
                        ok = all[r].device != c->device && cudaDeviceCanAccessPeer(&can, c->device, all[r].device) == cudaSuccess && can;
                        if (ok) {
                                cudaError_t e = cudaDeviceEnablePeerAccess(all[r].device, 0);
                                ok = e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled;
                        }
                        c->peer_tmp[r] = (u32 *)(uintptr_t)all[r].tmp; c->peer_av[r] = (u32 *)(uintptr_t)all[r].av;
                } else {
                        void *a = nullptr, *b = nullptr;
                        ok = ipc_ok && cudaIpcOpenMemHandle(&a, all[r].h_tmp, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
                        if (ok) {
                                c->peer_tmp[r] = (u32 *)a; c->peer_ipc[r] = 1;
                                ok = cudaIpcOpenMemHandle(&b, all[r].h_av, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
                                if (ok) c->peer_av[r] = (u32 *)b;
                        }
                }
        }
        cudaGetLastError();            // a refused mapping must not poison later calls
        return agree_flag(c, ok, ok_all);
}

void close_peers(blk_ctx *c)
{
        for (int r = 0; r < (int)c->peer_ipc.size(); r++) {
                if (r == c->rank || !c->peer_ipc[r]) continue;
                if (c->peer_tmp[r]) cudaIpcCloseMemHandle(c->peer_tmp[r]);
                if (c->peer_av[r]) cudaIpcCloseMemHandle(c->peer_av[r]);
        }
        c->peer_tmp.clear(); c->peer_av.clear(); c->peer_ipc.clear();
}

// Column bands of one operator (SpOp::bands): the entries (rkey, ckey, val)[count] -- row keys global, in [lo, hi) -- are
// split by column into K equal ranges and each range becomes an operator of its own over all rows.
int build_bands(blk_ctx *c, SpOp *op, int K, int chunk_len, int64_t count, const int32_t *rkey, const int32_t *ckey, const u32 *val,
                int64_t lo, int64_t hi, int64_t cols, bool acc)
{
        if (K < 2 || hi <= lo || count <= 0) return 0;
        {
                // bands are an optimisation: when the device cannot hold them next to what is already resident, the operator
                // simply stays unbanded (upper bounds: one dummy entry per row and band, the partial blocks, the builder's scratch)
                size_t free_b = 0, total_b = 0;
                const double rows = (double)(hi - lo);
                const double need = 8.0 * ((double)count + rows * K) + (acc ? 4.0 * rows * K : 4.0 * K * rows * c->geo.np) +
                                    48.0 * (double)count / K + 16.0 * rows;
                if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || need > 0.85 * (double)free_b) {
                        cudaGetLastError();
                        return 0;
                }
        }
        std::vector<u32> hc;
        if (count_dimension(c, count, ckey, cols, &hc)) return 1;
        op->band_col.assign((size_t)K + 1, 0);
        for (int b = 0; b <= K; b++) op->band_col[(size_t)b] = cols * b / K;
        op->bands.assign((size_t)K, SpOp());
        Scratch tmp;
        unsigned long long *cnt = nullptr;
        if (tmp.alloc(&cnt, sizeof(unsigned long long))) return 1;
        for (int b = 0; b < K; b++) {
                const int64_t c0 = op->band_col[(size_t)b], c1 = op->band_col[(size_t)b + 1];
                int64_t sel = 0;
                for (int64_t q = c0; q < c1; q++) sel += hc[(size_t)q];
                Scratch buf;
                int32_t *sr = nullptr, *sc = nullptr; u32 *sx = nullptr;
                unsigned long long h = 0;
                if (buf.alloc(&sr, sizeof(int32_t) * (size_t)sel) || buf.alloc(&sc, sizeof(int32_t) * (size_t)sel) || buf.alloc(&sx, sizeof(u32) * (size_t)sel))
                        return 1;
                CU(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), c->stream));
                // (selection by column: the column array is the key, the row array rides along)
                k_select_range<<<nb(count), 256, 0, c->stream>>>(count, ckey, rkey, val, c0, c1, sc, sr, sx, cnt, nullptr, 0, nullptr, 0);
                CU(cudaMemcpyAsync(&h, cnt, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
                CU(cudaStreamSynchronize(c->stream));
                if ((int64_t)h != sel) return fail("column band selection count mismatch");
                std::string err;
                if (acc) {
                        // compact form: only the rows that have entries in this band, results accumulated into y
                        u32 *rowmap = nullptr;
                        int64_t nrows = 0;
                        err = compact_rows(sel, sr, lo, hi - lo, &rowmap, &nrows, c->stream);
                        if (err.empty()) err = build_operator(&op->bands[(size_t)b], c->geo, chunk_len, nrows, cols, 0, sel, sr, sc, sx, c->m.p, nullptr,
                                                              nullptr, 1, c->stream, nullptr);
                        if (!err.empty()) { cudaFree(rowmap); return fail("column band: " + err); }
                        op->bands[(size_t)b].rowmap = rowmap;
                        op->bands[(size_t)b].bytes += sizeof(u32) * (size_t)nrows;
                } else {
                        err = build_operator(&op->bands[(size_t)b], c->geo, chunk_len, hi - lo, cols, lo, sel, sr, sc, sx, c->m.p, nullptr, nullptr,
                                             1, c->stream, nullptr);
                        if (!err.empty()) return fail("column band: " + err);
                }
                op->bytes += op->bands[(size_t)b].bytes;
        }
        if (acc) return 0;
        const size_t zb = sizeof(u32) * (size_t)K * (size_t)(hi - lo) * c->geo.np;
        CU(cudaMalloc(&op->zband, zb));
        CU(cudaMemsetAsync(op->zband, 0, zb, c->stream));
        op->bytes += zb;
        return 0;
}

// row r of an entry in column c -> virtual row b * H + r of the band-major heavy operator, b = the band holding c
// (band b covers the columns [cols * b / K, cols * (b + 1) / K))
__global__ void k_band_rows(int64_t count, int32_t *__restrict__ row, const int32_t *__restrict__ col, int64_t cols, int K, int64_t H)
{
        int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (s >= count) return;
        const int64_t c = col[s];
        int64_t b = c * K / cols;
        while (b + 1 < K && cols * (b + 1) / K <= c) b++;
        while (b > 0 && cols * b / K > c) b--;
        row[s] = (int32_t)(b * H + row[s]);
}

// Heavy/light split of product 2 (SpOp::split, plan_heavy): S2's rows are the degree-sorted N dimension, so its H heaviest
// rows are the label prefix [0, H).  The entries (rkey, ckey, val)[nnz] carry the ORIGINAL labels; n_old2new relabels the
// rows.  Like bands, the split is an optimisation: skipped (return 0, no split) when the device cannot hold it.
int build_heavy_split(blk_ctx *c, SpOp *op, int chunk_len, int64_t nnz, const int32_t *rkey, const int32_t *ckey, const u32 *val)
{
        const int np = c->geo.np;
        const char *e = getenv("BLK_HEAVY"), *ed = getenv("BLK_HEAVY_MIN_DEG"), *eb = getenv("BLK_HEAVY_BAND_BYTES");
        if ((e && e[0] == '0') || !c->n_old2new || c->world != 1 || np < 8 || nnz <= 0) return 0;
        // defaults: the fastest point of the sweep on the config-4 matrix (DESIGN.md section 4, profiles/r05_heavy_bands.json)
        const int64_t min_deg = ed ? atoll(ed) : 200;
        const int64_t band_bytes = eb ? std::max(4096ll, atoll(eb)) : 48ll << 20;
        int l2 = 0;
        if (cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, c->device) != cudaSuccess) { cudaGetLastError(); return 0; }
        std::vector<u32> deg;
        if (count_dimension(c, nnz, rkey, c->N, &deg, c->n_old2new)) return 1;
        const HeavyPlan plan = plan_heavy(deg.data(), c->N, c->Mc, np, l2, min_deg, band_bytes, env_flag("BLK_HEAVY_FORCE"));
        if (plan.rows == 0) return 0;
        const int64_t H = plan.rows, K = plan.bands;
        if (H * K >= (1ll << 31)) return 0;
        int64_t cnt_part[2] = {0, 0};
        for (int64_t r = 0; r < c->N; r++) cnt_part[r < H ? 0 : 1] += deg[(size_t)r];
        std::vector<u32>().swap(deg);

        op->split.assign(2, SpOp());
        SpOp &heavy = op->split[0], &light = op->split[1];
        auto give_up = [&]() {
                for (auto &s : op->split) free_operator(&s);
                op->split.clear();
                cudaFree(op->zheavy); op->zheavy = nullptr;
                return 0;
        };
        Scratch tmp;
        unsigned long long *cnt = nullptr;
        if (tmp.alloc(&cnt, sizeof(unsigned long long))) return 1;
        for (int part = 0; part < 2; part++) {
                const int64_t lo = part ? H : 0, hi = part ? c->N : H, sel = cnt_part[part];
                const int64_t rows = part ? hi - lo : K * H;
                {
                        // selection (12 B), the builder's sort (24 B) and the stream (8 B) per entry, one dummy entry and the
                        // builder's row arrays per (virtual) row, the partial blocks
                        size_t free_b = 0, total_b = 0;
                        const double need = 44.0 * sel + 32.0 * rows + (part ? 0.0 : 4.0 * np * rows);
                        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || need > 0.85 * (double)free_b) {
                                cudaGetLastError();
                                return give_up();
                        }
                }
                Scratch buf;
                int32_t *sr = nullptr, *sc = nullptr; u32 *sx = nullptr;
                unsigned long long h = 0;
                if (buf.alloc(&sr, sizeof(int32_t) * (size_t)sel) || buf.alloc(&sc, sizeof(int32_t) * (size_t)sel) ||
                    buf.alloc(&sx, sizeof(u32) * (size_t)sel))
                        return 1;
                CU(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), c->stream));
                k_select_range<<<nb(nnz), 256, 0, c->stream>>>(nnz, rkey, ckey, val, lo, hi, sr, sc, sx, cnt, c->n_old2new, c->N, nullptr, c->Mc);
                CU(cudaMemcpyAsync(&h, cnt, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
                CU(cudaStreamSynchronize(c->stream));
                if ((int64_t)h != sel) return fail("heavy split selection count mismatch");
                if (part == 0 && sel) k_band_rows<<<nb(sel), 256, 0, c->stream>>>(sel, sr, sc, c->Mc, (int)K, H);
                std::string err = build_operator(part ? &light : &heavy, c->geo, chunk_len, rows, c->Mc, lo, sel, sr, sc, sx, c->m.p,
                                                 nullptr, nullptr, 1, c->stream, nullptr);
                if (!err.empty()) return fail(std::string("heavy split, ") + (part ? "light rows: " : "heavy rows: ") + err);
        }
        const size_t zb = sizeof(u32) * (size_t)(K * H) * np;
        CU(cudaMalloc(&op->zheavy, zb));
        CU(cudaMemsetAsync(op->zheavy, 0, zb, c->stream));
        op->heavy_rows = H;
        op->heavy_bands = (int)K;
        op->bytes += heavy.bytes + light.bytes + zb;
        return 0;
}

// the multi-GPU part of blk_create: communicator, pieces, side stream, the recurrence blocks, the exchange mode
int create_multi(blk_ctx *c, const blk_params *prm, bool grid_req)
{
        const int world = c->world, np = c->geo.np;
        std::string why;
        if (!nccl_load(&why)) return fail(why);
        ncclUniqueId id;
        memcpy(&id, prm->nccl_id, sizeof(id));
        NC(g_nccl.CommInitRank(&c->comm, world, id, c->rank));
        const char *e = getenv("BLK_ALLGATHER");
        if (!(e && e[0] == 'b')) c->nccl_allgather = g_nccl.AllGather;     // BLK_ALLGATHER=bcast forces broadcasts
        if (agree_pieces(c)) return 1;
        if (c->colblocks) {
                // arrival-order mode: pieces are equal row counts, known on every rank without an exchange
                const int K = c->colblocks;
                c->pieces = c->pieces2 = K;
                c->piece_rows_all.assign((size_t)world * (K + 1), 0);
                c->piece_rows_all2.assign((size_t)world * (K + 1), 0);
                for (int r = 0; r < world; r++)
                        for (int q = 0; q <= K; q++) {
                                c->piece_rows_all[(size_t)r * (K + 1) + q] = (c->m_off[r + 1] - c->m_off[r]) * q / K;
                                c->piece_rows_all2[(size_t)r * (K + 1) + q] = (c->n_off[r + 1] - c->n_off[r]) * q / K;
                        }
                c->ev_arrived.resize((size_t)2 * K);
                for (auto &ev : c->ev_arrived) CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
                CU(cudaEventCreateWithFlags(&c->ev_aux, cudaEventDisableTiming));
        }
        {
                // highest priority: the block scheduler then places the exchange's few CTAs ahead of the thousands
                // of queued SpMV blocks instead of after them
                int pr_least = 0, pr_greatest = 0;
                CU(cudaDeviceGetStreamPriorityRange(&pr_least, &pr_greatest));
                CU(cudaStreamCreateWithPriority(&c->comm_stream, cudaStreamNonBlocking, pr_greatest));
                c->ev_piece.resize(std::max(c->pieces, c->pieces2));
                for (auto &ev : c->ev_piece) CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
                CU(cudaEventCreateWithFlags(&c->ev_comm, cudaEventDisableTiming));
        }
        const char *er = getenv("BLK_RECUR");
        if ((er && er[0] == '0') || grid_req) return 0;

        c->mg_recur = true;
        const int64_t lm = c->m1() - c->m0();
        const size_t bav = sizeof(u32) * (size_t)gather_cap(c->n_off) * np;
        const size_t blm = sizeof(u32) * (size_t)(lm > 0 ? lm : 1) * np;
        CU(cudaMalloc(&c->Av_full, bav));
        CU(cudaMemsetAsync(c->Av_full, 0, bav, c->stream));
        cudaFree(c->Av);
        c->Av = c->Av_full + (size_t)c->n0() * np;
        CU(cudaMalloc(&c->Tp, blm)); CU(cudaMalloc(&c->U, blm));
        CU(cudaMemsetAsync(c->Tp, 0, blm, c->stream));
        CU(cudaMemsetAsync(c->U, 0, blm, c->stream));
        if (c->Mc > c->N) { CU(cudaMalloc(&c->tmp_prev, blm)); CU(cudaMemsetAsync(c->tmp_prev, 0, blm, c->stream)); }
        c->block_bytes += bav + 3 * blm;
        CU(cudaStreamSynchronize(c->stream));

        // ---- how Av and the new tmp travel (DESIGN.md section 6).  Default: our own stores over NVLink
        // (XCH_PUSH) when every rank could map every peer's blocks; BLK_EXCHANGE=nccl | ce | push selects.
        // Measured on 8 x B200, config 4 (profiles/): see DESIGN.md.
        int want = blk_ctx::XCH_PUSH;
        if (const char *ex = getenv("BLK_EXCHANGE")) {
                if (!strcmp(ex, "nccl")) want = blk_ctx::XCH_NCCL;
                else if (!strcmp(ex, "ce")) want = blk_ctx::XCH_CE;
                else if (!strcmp(ex, "push")) want = blk_ctx::XCH_PUSH;
                else return fail("BLK_EXCHANGE must be nccl, ce or push");
        } else if (env_flag("BLK_P2P")) want = blk_ctx::XCH_CE;           // round-1 spelling
        if (np < 4 || c->colblocks || c->bands1 > 1 || c->bands2 > 1) want = blk_ctx::XCH_NCCL;   // rows shorter than 16 bytes / arrival-order mode / banded products
        if (want != blk_ctx::XCH_NCCL) {
                bool ok = false;
                if (setup_peers(c, &ok)) return 1;
                if (!ok) { close_peers(c); want = blk_ctx::XCH_NCCL; }
        }
        c->xch = want;
        if (const char *ea = getenv("BLK_PUSH_AV")) c->push_av_in_spmv = strcmp(ea, "kernel") != 0;     // kernel | spmv
        if (const char *eb = getenv("BLK_PUSH_COPY")) {
                if (!strcmp(eb, "bulk")) c->push_bulk = true;
                else if (strcmp(eb, "rows")) return fail("BLK_PUSH_COPY must be rows or bulk");
        }
        if (c->push_bulk) {
                c->push_ctas = 16;
                if (const char *es = getenv("BLK_BULK_STAGES")) c->bulk_stages = std::max(2, std::min(PB_MAX_STAGES, atoi(es)));
                if (const char *ek = getenv("BLK_BULK_CHUNK")) c->bulk_chunk = (unsigned)std::max(1024, std::min(65536, atoi(ek))) & ~127u;
                if ((size_t)c->bulk_stages * c->bulk_chunk > 200 * 1024) return fail("BLK_BULK_STAGES x BLK_BULK_CHUNK exceeds the shared memory of an SM");
                CU(cudaFuncSetAttribute(k_push_bulk, cudaFuncAttributeMaxDynamicSharedMemorySize, c->bulk_stages * (int)c->bulk_chunk));
        }
        if (const char *ec = getenv("BLK_PUSH_CTAS")) c->push_ctas = std::max(1, std::min(1024, atoi(ec)));
        if (c->xch != blk_ctx::XCH_NCCL) {
                CU(cudaMalloc(&c->barrier_word, sizeof(u64)));
                CU(cudaMemsetAsync(c->barrier_word, 0, sizeof(u64), c->stream));
        }
        if (c->xch == blk_ctx::XCH_CE) {
                c->copy_streams.resize(world - 1); c->ev_copies.resize(world - 1);
                for (auto &st : c->copy_streams) CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
                for (auto &ev : c->ev_copies) CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        }
        CU(cudaStreamSynchronize(c->stream));
        return 0;
}

int create_impl(blk_ctx *c, const blk_params *prm)
{
        const int world = c->world, np = c->geo.np;
        const ModP &m = c->m;
        // Paths that have been validated on GPUs but are not the default need an explicit opt-in next to
        // their own switch, so that a stray environment variable cannot reroute a production run.
        const bool experimental = env_flag("BLK_EXPERIMENTAL");
        {
                // column-blocked products (world == 1: a test mode that exercises the blocks and the combine kernel
                // under the whole single-GPU test suite; world > 1: arrival-order exchange)
                const char *e = getenv("BLK_COLBLOCKS");
                int K = e ? atoi(e) : 0;
                if (K != 0 && !experimental) return fail("BLK_COLBLOCKS is an experimental mode: set BLK_EXPERIMENTAL=1 as well");
                const char *er = getenv("BLK_RECUR");
                if (K >= 2 && K <= 16 && !(world > 1 && er && er[0] == '0')) c->colblocks = K;
        }
        // BLK_GRID=PxQ or BLK_GRID=auto runs the loop on the P x Q block grid (world > 1 only)
        bool grid_req = false;
        int gridP = 0, gridQ = 0;
        {
                const char *e = getenv("BLK_GRID");
                if (e && e[0] && world > 1) {
                        if (!experimental) return fail("BLK_GRID is an experimental mode: set BLK_EXPERIMENTAL=1 as well");
                        grid_req = true;
                        if (sscanf(e, "%dx%d", &gridP, &gridQ) != 2) gridP = gridQ = 0;      // "auto": like MPI_Dims_create
                        c->colblocks = 0;
                }
        }
        std::vector<u32> grid_cntN, grid_cntM;
        if (prm->stream) c->stream = (cudaStream_t)prm->stream;
        else { CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)); c->own_stream = true; }

        dense_prepare(c->geo, c->m);

        // ---- COO on the device
        const int64_t nnz = prm->nnz;
        Scratch coo;
        int32_t *di = nullptr, *dj = nullptr;
        u32 *dx = nullptr;
        if (prm->coo_on_device || nnz == 0) {
                di = (int32_t *)prm->Mi; dj = (int32_t *)prm->Mj; dx = (u32 *)prm->Mx;
        } else {
                if (coo.alloc(&di, sizeof(int32_t) * (size_t)nnz) || coo.alloc(&dj, sizeof(int32_t) * (size_t)nnz) ||
                    coo.alloc(&dx, sizeof(u32) * (size_t)nnz))
                        return 1;
                CU(cudaMemcpyAsync(di, prm->Mi, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, c->stream));
                CU(cudaMemcpyAsync(dj, prm->Mj, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, c->stream));
                CU(cudaMemcpyAsync(dx, prm->Mx, sizeof(u32) * (size_t)nnz, cudaMemcpyHostToDevice, c->stream));
        }

        // Lanczos-dimension index array and the other one
        const int32_t *idxN = c->right ? dj : di;     // indexes rows of v/Av/p
        const int32_t *idxM = c->right ? di : dj;     // indexes rows of tmp

        // ---- row partitions
        c->n_off.assign(world + 1, 0); c->m_off.assign(world + 1, 0);
        c->n_off[world] = c->N; c->m_off[world] = c->Mc;
        if (world > 1) {
                for (int pass = 0; pass < 2; pass++) {
                        std::vector<u32> hc;
                        if (count_dimension(c, nnz, pass ? idxM : idxN, pass ? c->Mc : c->N, &hc)) return 1;
                        (pass ? c->m_off : c->n_off) = partition_rows(hc, world);
                        if (grid_req) (pass ? grid_cntM : grid_cntN).swap(hc);
                }
        }

        // ---- column bands (n_pad <= 4): with 4 ... 16-byte rows the x block is still far larger than L2 (config 4: 200 ... 800 MB)
        // and every gather still costs a whole 128-byte HBM line -- 32 ... 8 times the bytes it uses.  Cutting the columns into
        // bands whose slice of x stays in L2 turns those line fetches into L2 hits at the price of one partial result per band
        // (rows * n_pad * 4 bytes written and read again), which is cheap exactly when n_pad is small.  BLK_BANDS=0 disables,
        // BLK_BAND_BYTES sets the slice size.  Measured on the config-4 matrix (profiles/r02_column_bands.txt), ms per product:
        // n = 1: 20.1 -> 6.6, n = 2: 26.8 -> 8.8, n = 4: 29.8 -> 15.9 with the default 48 MB (slices of 16 / 32 / 112 MB are slower).
        {
                const char *e = getenv("BLK_BANDS"), *eb = getenv("BLK_BAND_BYTES");
                const long long band_bytes = eb ? std::max(4096ll, atoll(eb)) : 48ll << 20;
                const long long min_bytes = 96ll << 20;
                if (const char *ea = getenv("BLK_BAND_ACC")) c->bands_acc = ea[0] != '0';
                // (the partial-result form pays rows * n_pad * 8 bytes per band: only for n_pad <= 4.  The accumulate form -- compact
                // bands that add into y, allowed up to n_pad = 8 -- avoids the partial blocks and the dummy entries but its
                // read-modify-write of scattered y rows costs a line per row again: 8.6 / 13.0 / 20.8 ms against 6.6 / 8.8 / 15.9 for
                // n = 1 / 2 / 4 and 39.9 against 31.5 ms unbanded at n = 8, profiles/r02_column_bands.txt; it stays an opt-in)
                if (np <= (c->bands_acc ? 8 : 4) && !c->colblocks && !grid_req && !(e && e[0] == '0') && nnz > 0) {
                        auto bands_for = [&](int64_t cols) -> int {
                                const long long x_bytes = (long long)cols * np * 4;
                                if (!eb && x_bytes <= min_bytes) return 0;           // fits L2 well enough as it is
                                long long K = (x_bytes + band_bytes - 1) / band_bytes;
                                return K < 2 ? 0 : (int)std::min(64ll, K);
                        };
                        c->bands1 = bands_for(c->N);          // S1 gathers rows of v
                        c->bands2 = bands_for(c->Mc);         // S2 gathers rows of tmp
                }
        }
        const bool banded = c->bands1 > 1 || c->bands2 > 1;

        // ---- degree-sorted labels for the N dimension + L2-resident hot prefix.  The rows of the Lanczos vectors can
        // be stored under any labels (dots are order-free, orthogonalize is row-wise); sorting them by decreasing
        // number of entries makes the rows product 1 gathers most often a contiguous prefix that L2 can keep.  With
        // several GPUs the sorted sequence is dealt round-robin to the ranks' blocks: every rank owns the same
        // number of rows and of non-zeros (to within one giant row) and its own share of the hot rows.
        HotCols hot;
        {
                const char *e = getenv("BLK_HOT"), *emin = getenv("BLK_HOT_MIN_BYTES"), *eb = getenv("BLK_HOT_BYTES");
                cudaDeviceProp prop;
                CU(cudaGetDeviceProperties(&prop, c->device));
                long long min_bytes = emin ? atoll(emin) : 96ll << 20;
                long long hot_bytes = eb ? atoll(eb) : 24ll << 20;
                bool on = !c->colblocks && !grid_req && !banded && !(e && e[0] == '0') && np >= 4 && nnz > 0 && world <= HotCols::MAXB &&
                          c->N < (1ll << 30) && (long long)c->N * np * 4 > min_bytes && hot_bytes > 0;
                if (world > 1 && env_flag("BLK_HOT_SINGLE_ONLY")) on = false;       // A/B switch: round-1 behaviour
                if (on) {
                        std::vector<int64_t> off((size_t)world + 1, 0);
                        std::string err = degree_sort_maps(nnz, idxN, c->N, &c->n_old2new, &c->n_new2old, c->stream, world, off.data());
                        if (!err.empty()) return fail(err);
                        c->hot_rows = std::min<int64_t>(c->N, hot_bytes / (4 * np));
                        hot.blocks = world;
                        hot.per = (u32)((c->hot_rows + world - 1) / world);
                        for (int w = 0; w <= world; w++) hot.off[w] = off[(size_t)w];
                        if (world > 1) c->n_off = off;          // the dealt blocks replace the weight-balanced partition
                        // B200's L2 is two halves (one per die) and lines gathered by SMs of both dies live
                        // in both, so the set-aside has to hold the hot prefix twice.  (A device-wide limit: the
                        // one piece of process state this library changes; restored by blk_destroy.)
                        const char *ep = getenv("BLK_L2_PERSIST");
                        long long persist = ep ? atoll(ep) : std::min<long long>(prop.persistingL2CacheMaxSize, 2 * hot_bytes);
                        size_t before = 0;
                        if (cudaDeviceGetLimit(&before, cudaLimitPersistingL2CacheSize) == cudaSuccess) {
                                c->l2_persist_before = (long long)before;
                                cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)persist);
                        }
                        cudaGetLastError();
                }
        }

        // ---- the two operators.  S1: rows = my block of the Mc dimension, columns = N dimension;
        //      S2: rows = my block of the N dimension, columns = Mc dimension.
        int want_pieces = 1;
        if (world > 1) {
                const char *e = getenv("BLK_PIECES");
                // a piece should be worth >= ~0.5 ms of product time (about 25M entries); <= 4 pieces by default
                long long per_rank = (long long)(nnz / world);
                want_pieces = e ? atoi(e) : (int)std::max(1ll, std::min(4ll, per_rank / 25000000ll));
                if (want_pieces < 1) want_pieces = 1;
                if (want_pieces > 32) want_pieces = 32;
                if (banded) want_pieces = 1;          // banded products run whole (launch_spmv)
        }
        for (int which = 0; which < 2; which++) {
                SpOp *op = which ? &c->S2 : &c->S1;
                const int32_t *rk = which ? idxN : idxM, *ck = which ? idxM : idxN;
                int64_t lo = which ? c->n0() : c->m0(), hi = which ? c->n1() : c->m1();
                int64_t cols = which ? c->Mc : c->N;
                std::string err;
                if (world == 1) {
                        err = build_operator(op, c->geo, prm->chunk_len, hi - lo, cols, lo, nnz, rk, ck, dx, m.p,
                                             which ? c->n_old2new : nullptr, which ? nullptr : c->n_old2new, 1, c->stream,
                                             which ? nullptr : &hot);
                        if (err.empty() && build_bands(c, op, which ? c->bands2 : c->bands1, prm->chunk_len, nnz, rk, ck, dx, lo, hi, cols, c->bands_acc)) return 1;
                        if (err.empty() && c->colblocks &&
                            build_colops(c, which ? &c->cb2 : &c->cb1, c->colblocks, prm->chunk_len, nnz, rk, ck, dx, lo, hi, cols,
                                         which ? c->m_off : c->n_off))
                                return 1;
                        if (err.empty() && which && !c->colblocks && build_heavy_split(c, op, prm->chunk_len, nnz, rk, ck, dx)) return 1;
                } else {
                        Scratch sel_buf;
                        int32_t *sr = nullptr, *sc = nullptr; u32 *sx = nullptr;
                        unsigned long long *cnt = nullptr, hcnt = 0;
                        // upper bound of the selection is not known: count first
                        // (the N dimension may be relabelled: S2 selects its rows, S1 gathers its columns, under the new labels)
                        const u32 *key_map = which ? c->n_old2new : nullptr, *other_map = which ? nullptr : c->n_old2new;
                        std::vector<u32> hc;
                        if (count_dimension(c, nnz, rk, which ? c->N : c->Mc, &hc, key_map)) return 1;
                        int64_t sel = 0;
                        for (int64_t r = lo; r < hi; r++) sel += hc[(size_t)r];
                        std::vector<u32>().swap(hc);
                        if (sel_buf.alloc(&cnt, sizeof(unsigned long long)) || sel_buf.alloc(&sr, sizeof(int32_t) * (size_t)sel) ||
                            sel_buf.alloc(&sc, sizeof(int32_t) * (size_t)sel) || sel_buf.alloc(&sx, sizeof(u32) * (size_t)sel))
                                return 1;
                        CU(cudaMemsetAsync(cnt, 0, sizeof(unsigned long long), c->stream));
                        if (nnz)
                                k_select_range<<<nb(nnz), 256, 0, c->stream>>>(nnz, rk, ck, dx, lo, hi, sr, sc, sx, cnt, key_map,
                                                                               which ? c->N : c->Mc, other_map, which ? c->Mc : c->N);
                        CU(cudaMemcpyAsync(&hcnt, cnt, sizeof(hcnt), cudaMemcpyDeviceToHost, c->stream));
                        CU(cudaStreamSynchronize(c->stream));
                        if ((int64_t)hcnt != sel) err = "shard selection count mismatch";
                        else err = build_operator(op, c->geo, prm->chunk_len, hi - lo, cols, lo, sel, sr, sc, sx, m.p, nullptr, nullptr,
                                                       want_pieces, c->stream, which ? nullptr : &hot);
                        if (err.empty() && build_bands(c, op, which ? c->bands2 : c->bands1, prm->chunk_len, sel, sr, sc, sx, lo, hi, cols, c->bands_acc)) return 1;
                        if (err.empty() && c->colblocks &&
                            build_colops(c, which ? &c->cb2 : &c->cb1, c->colblocks, prm->chunk_len, sel, sr, sc, sx, lo, hi, cols,
                                         which ? c->m_off : c->n_off))
                                return 1;
                }
                if (!err.empty()) return fail(err);
        }
        CU(cudaStreamSynchronize(c->stream));
        if (!grid_req) { coo.release(di); coo.release(dj); coo.release(dx); }     // the grid mode extracts its block later

        // ---- vector blocks and the small working set
        int64_t ln = c->n1() - c->n0();
        size_t bv = sizeof(u32) * (size_t)gather_cap(c->n_off) * np, bt = sizeof(u32) * (size_t)gather_cap(c->m_off) * np;
        size_t bl = sizeof(u32) * (size_t)(ln > 0 ? ln : 1) * np;
        CU(cudaMalloc(&c->v, bv)); CU(cudaMalloc(&c->tmp, bt));
        CU(cudaMalloc(&c->Av, bl)); CU(cudaMalloc(&c->p, bl));
        CU(cudaMemsetAsync(c->v, 0, bv, c->stream)); CU(cudaMemsetAsync(c->tmp, 0, bt, c->stream));
        CU(cudaMemsetAsync(c->Av, 0, bl, c->stream)); CU(cudaMemsetAsync(c->p, 0, bl, c->stream));
        c->block_bytes = bv + bt + 2 * bl;
        if (c->colblocks) {
                int64_t lm_ = c->m1() - c->m0();
                c->zstride = (size_t)std::max<int64_t>(1, std::max(ln, lm_)) * np;
                CU(cudaMalloc(&c->zbuf, sizeof(u32) * c->zstride * c->colblocks));
                CU(cudaMemsetAsync(c->zbuf, 0, sizeof(u32) * c->zstride * c->colblocks, c->stream));
                c->block_bytes += sizeof(u32) * c->zstride * c->colblocks;
        }
        // staging for host <-> device block copies that need repacking (n < n_pad, relabelled rows): two slots
        // so that the PCIe copy of one chunk overlaps the repacking kernel of the other
        CU(cudaMalloc(&c->stage, 2 * blk_ctx::STAGE_BYTES));
        c->block_bytes += 2 * blk_ctx::STAGE_BYTES;
        c->dots_blocks = dots_num_blocks(ln, np);
        CU(cudaMalloc(&c->mats, sizeof(u32) * mats_words(np)));
        CU(cudaMalloc(&c->sums, sizeof(u64) * (size_t)2 * np * np));
        CU(cudaMalloc(&c->state, sizeof(DevSmall)));
        CU(cudaMalloc(&c->dots_counter, sizeof(unsigned)));
        CU(cudaMemsetAsync(c->dots_counter, 0, sizeof(unsigned), c->stream));
        {
                const char *e = getenv("BLK_FUSE_SMALL");
                c->fuse_small = world == 1 && np <= 32 && !(e && e[0] == '0');
        }
        {
                // BLK_LOOP=coop runs the loop as ONE persistent cooperative kernel (loop_coop.cu) instead of a CUDA graph of six
                // kernel nodes per iteration.  Measured on BASELINE configs 1-3 (profiles/r02_loop_coop.txt): 29.9 / 44.3 / 103.8 us
                // per iteration against 26.1 / 41.2 / 75.3 for the graph -- a grid barrier costs what a graph edge costs
                // (~1.5-2 us), and one block of 16 warps per SM hides the latency of the products worse than three blocks
                // of 8 -- so the graph stays the default (BLK_LOOP=graph | auto) and the persistent kernel is an opt-in.
                const char *e = getenv("BLK_LOOP");
                const bool force = e && !strcmp(e, "coop"), off = e && !strcmp(e, "graph");
                if (e && !force && !off && strcmp(e, "auto")) return fail("BLK_LOOP must be graph, coop or auto");
                const size_t working_set = c->S1.bytes + c->S2.bytes + c->block_bytes - 2 * blk_ctx::STAGE_BYTES;
                const bool eligible = world == 1 && !c->colblocks && loop_coop_supported(np) && !c->S1.lookback && !c->S2.lookback &&
                                      !c->S1.hot_cols && c->S1.bands.empty() && c->S2.bands.empty() && c->S2.split.empty() && c->N > 0 && c->Mc > 0;
                if (force && !eligible) return fail("BLK_LOOP=coop: the persistent loop kernel needs one GPU, n <= 16 and the default product kernels");
                (void)working_set;
                if (eligible && force) {
                        std::string why;
                        c->coop_grid = loop_coop_grid(c->geo.n, np, c->m, &why);
                        if (c->coop_grid > 0) {
                                CU(cudaMalloc(&c->loop_bar, 2 * sizeof(unsigned) + 6 * sizeof(unsigned long long)));
                                CU(cudaMemsetAsync(c->loop_bar, 0, 2 * sizeof(unsigned) + 6 * sizeof(unsigned long long), c->stream));
                                c->coop = true;
                                c->coop_prof = env_flag("BLK_LOOP_PROF");
                        } else if (force) return fail("BLK_LOOP=coop: " + why);
                }
        }
        c->check = env_flag("BLK_CHECK");
        if (const char *ef = getenv("BLK_CHECK_FAULT")) c->check_fault = atoi(ef);
        CU(cudaMallocHost(&c->h_state, sizeof(DevSmall)));
        CU(cudaMemsetAsync(c->mats, 0, sizeof(u32) * mats_words(np), c->stream));
        CU(cudaMemsetAsync(c->sums, 0, sizeof(u64) * (size_t)2 * np * np, c->stream));
        memset(c->h_state, 0, sizeof(DevSmall));
        c->h_state->halt = 1;
        c->h_state->check = c->check ? 1 : 0;
        c->h_state->fault_iter = c->check_fault;
        if (push_state(c)) return 1;
        CU(cudaStreamSynchronize(c->stream));

        if (world > 1) {
                if (create_multi(c, prm, grid_req)) return 1;
                if (grid_req && grid_create(c, gridP, gridQ, prm->chunk_len, nnz, idxN, idxM, dx, grid_cntN, grid_cntM)) return 1;
        }
        return 0;
}

}  // namespace

// blk_params.rank == BLK_RANK_ALL: one process, `world` GPUs (devices prm->device ... prm->device + world - 1)
static int group_create(blk_ctx **out, const blk_params *prm, int world, int ndev)
{
        if (prm->device < 0 || prm->device + world > ndev) return fail("not enough CUDA devices for the requested number of GPUs");
        if (world == 1) {
                blk_params one = *prm;
                one.rank = 0; one.world = 1;
                return blk_create(out, &one);
        }
        unsigned char id[BLK_NCCL_ID_BYTES];
        if (blk_nccl_unique_id(id)) return 1;
        blk_ctx *g = new blk_ctx();
        g->geo = make_geometry(prm->n);
        modp_make(&g->m, prm->prime);
        g->device = prm->device; g->rank = BLK_RANK_ALL; g->world = world; g->right = prm->right_kernel ? 1 : 0;
        g->nrows = prm->nrows; g->ncols = prm->ncols;
        g->N = g->right ? prm->ncols : prm->nrows;
        g->Mc = g->right ? prm->nrows : prm->ncols;
        g->members.assign((size_t)world, nullptr);
        int rc = group_run(g, [&](blk_ctx *, int r) -> int {
                blk_params p2 = *prm;
                p2.rank = r; p2.world = world; p2.device = prm->device + r; p2.nccl_id = id; p2.stream = nullptr;
                Scratch coo;
                if (prm->coo_on_device && prm->nnz > 0 && p2.device != prm->device) {
                        // the triplets live on the first GPU: every other member works on its own copy
                        CU(cudaSetDevice(p2.device));
                        int32_t *di = nullptr, *dj = nullptr;
                        u32 *dx = nullptr;
                        const size_t cnt = (size_t)prm->nnz;
                        if (coo.alloc(&di, sizeof(int32_t) * cnt) || coo.alloc(&dj, sizeof(int32_t) * cnt) || coo.alloc(&dx, sizeof(u32) * cnt)) return 1;
                        CU(cudaMemcpyPeer(di, p2.device, prm->Mi, prm->device, sizeof(int32_t) * cnt));
                        CU(cudaMemcpyPeer(dj, p2.device, prm->Mj, prm->device, sizeof(int32_t) * cnt));
                        CU(cudaMemcpyPeer(dx, p2.device, prm->Mx, prm->device, sizeof(u32) * cnt));
                        p2.Mi = di; p2.Mj = dj; p2.Mx = dx;
                }
                return blk_create(&g->members[(size_t)r], &p2);
        });
        if (rc) {
                std::string why = g_err;
                blk_destroy(g);
                return fail(why);
        }
        *out = g;
        return 0;
}

int blk_create(blk_ctx **out, const blk_params *prm)
{
        if (!out) return fail("blk_create: null output pointer");
        *out = nullptr;
        if (!prm || prm->abi_version != BLK_ABI_VERSION) return fail("blk_params.abi_version mismatch");
        if (prm->n < 1 || prm->n > BLK_MAX_N) return fail("blocking factor n must be in [1,64]");
        if (prm->nrows < 1 || prm->ncols < 1 || prm->nnz < 0) return fail("bad matrix dimensions");
        if (prm->nnz > 0 && (!prm->Mi || !prm->Mj || !prm->Mx)) return fail("null COO arrays");
        int world = prm->world > 0 ? prm->world : 1;
        ModP m;
        if (!modp_make(&m, prm->prime)) return fail("prime must satisfy 2 <= p < 2^31");
        int ndev = 0;
        cudaError_t e0 = cudaGetDeviceCount(&ndev);
        if (e0 != cudaSuccess || ndev == 0)
                return fail(std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e0));
        if (prm->rank == BLK_RANK_ALL) return group_create(out, prm, world, ndev);
        if (prm->rank < 0 || prm->rank >= world) return fail("rank out of range");
        if (world > 1 && !prm->nccl_id) return fail("world > 1 needs blk_params.nccl_id");
        if (prm->device < 0 || prm->device >= ndev) return fail("device ordinal out of range");
        CU(cudaSetDevice(prm->device));

        blk_ctx *c = new blk_ctx();
        c->geo = make_geometry(prm->n);
        c->m = m;
        c->device = prm->device; c->rank = prm->rank; c->world = world; c->right = prm->right_kernel ? 1 : 0;
        c->nrows = prm->nrows; c->ncols = prm->ncols;
        c->N = c->right ? prm->ncols : prm->nrows;
        c->Mc = c->right ? prm->nrows : prm->ncols;
        c->use_graph = prm->use_graph;
        if (create_impl(c, prm)) {
                std::string why = g_err;          // blk_destroy must not lose the reason
                blk_destroy(c);
                return fail(why);
        }
        *out = c;
        return 0;
}


// blk_create_system: the COO of M and the non-zeros of -B (rhs_triplets) in one device COO, handed to blk_create as
// the augmented matrix [M | -B] (--right) or [M ; -B^T] (--left)
static int create_system(blk_ctx **out, const blk_params *prm, const uint32_t *B, int32_t nrhs, int32_t b_on_device)
{
        if (!out) return fail("blk_create_system: null output pointer");
        *out = nullptr;
        if (!prm || prm->abi_version != BLK_ABI_VERSION) return fail("blk_params.abi_version mismatch");
        if (prm->n < 1 || prm->n > BLK_MAX_N) return fail("blocking factor n must be in [1,64]");
        if (prm->nrows < 1 || prm->ncols < 1 || prm->nnz < 0) return fail("bad matrix dimensions");
        if (prm->nnz > 0 && (!prm->Mi || !prm->Mj || !prm->Mx)) return fail("null COO arrays");
        if (nrhs < 1 || nrhs > prm->n) return fail("blk_create_system: the number of right-hand sides must be in [1, n]");
        if (!B) return fail("blk_create_system: null right-hand-side block");
        ModP m;
        if (!modp_make(&m, prm->prime)) return fail("prime must satisfy 2 <= p < 2^31");
        const int right = prm->right_kernel ? 1 : 0;
        const int64_t N = right ? prm->ncols : prm->nrows, Mc = right ? prm->nrows : prm->ncols;
        if (N + nrhs > INT32_MAX) return fail("blk_create_system: the matrix is too large for the appended right-hand sides");
        int ndev = 0;
        cudaError_t e0 = cudaGetDeviceCount(&ndev);
        if (e0 != cudaSuccess || ndev == 0)
                return fail(std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e0));
        if (prm->device < 0 || prm->device >= ndev) return fail("device ordinal out of range");
        CU(cudaSetDevice(prm->device));
        struct Bufs {
                std::vector<void *> p;
                cudaStream_t st = nullptr;
                ~Bufs() { for (void *q : p) cudaFree(q); if (st) cudaStreamDestroy(st); }
        } bufs;
        auto grab = [&](void **dst, size_t bytes) {
                cudaError_t e = cudaMalloc(dst, bytes ? bytes : 4);
                if (e == cudaSuccess) bufs.p.push_back(*dst);
                return e;
        };
        CU(cudaStreamCreateWithFlags(&bufs.st, cudaStreamNonBlocking));
        const cudaStream_t st = bufs.st;
        const u32 *dB = B;
        if (!b_on_device) {
                u32 *hb = nullptr;
                CU(grab((void **)&hb, sizeof(u32) * (size_t)Mc * nrhs));
                CU(cudaMemcpyAsync(hb, B, sizeof(u32) * (size_t)Mc * nrhs, cudaMemcpyHostToDevice, st));
                dB = hb;
        }
        int64_t add = 0, added = 0;
        std::string err = rhs_triplets(dB, Mc, nrhs, N, right, m.p, nullptr, nullptr, nullptr, &add, st);
        if (!err.empty()) return fail(err);
        const int64_t nnz = prm->nnz, tot = nnz + add;
        int32_t *di = nullptr, *dj = nullptr;
        u32 *dx = nullptr;
        CU(grab((void **)&di, sizeof(int32_t) * (size_t)tot));
        CU(grab((void **)&dj, sizeof(int32_t) * (size_t)tot));
        CU(grab((void **)&dx, sizeof(u32) * (size_t)tot));
        if (nnz) {
                const cudaMemcpyKind kind = prm->coo_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
                CU(cudaMemcpyAsync(di, prm->Mi, sizeof(int32_t) * (size_t)nnz, kind, st));
                CU(cudaMemcpyAsync(dj, prm->Mj, sizeof(int32_t) * (size_t)nnz, kind, st));
                CU(cudaMemcpyAsync(dx, prm->Mx, sizeof(u32) * (size_t)nnz, kind, st));
        }
        err = rhs_triplets(dB, Mc, nrhs, N, right, m.p, di + nnz, dj + nnz, dx + nnz, &added, st);
        if (!err.empty()) return fail(err);
        if (added != add) return fail("blk_create_system: right-hand-side count mismatch");
        CU(cudaStreamSynchronize(st));
        blk_params p2 = *prm;
        if (right) p2.ncols += nrhs;
        else p2.nrows += nrhs;
        p2.nnz = tot; p2.Mi = di; p2.Mj = dj; p2.Mx = dx; p2.coo_on_device = 1;
        if (blk_create(out, &p2)) return 1;
        blk_ctx *c = *out;
        c->nrhs = nrhs;
        for (blk_ctx *mem : c->members) mem->nrhs = nrhs;
        return 0;
}


// blk_create_pruned: the COO on prm->device (uploaded when it is on the host), pruned by prune_coo, handed to
// blk_create as a device COO.  The upload is freed before blk_create, so that at most one extra copy of the COO
// (M') is resident while the layouts are built.
static int create_pruned(blk_ctx **out, const blk_params *prm, int64_t stats[BLK_PR_COUNT])
{
        if (!out) return fail("blk_create_pruned: null output pointer");
        *out = nullptr;
        if (!prm || prm->abi_version != BLK_ABI_VERSION) return fail("blk_params.abi_version mismatch");
        if (prm->n < 1 || prm->n > BLK_MAX_N) return fail("blocking factor n must be in [1,64]");
        if (prm->nrows < 1 || prm->ncols < 1 || prm->nnz < 0) return fail("bad matrix dimensions");
        if (prm->nnz > 0 && (!prm->Mi || !prm->Mj || !prm->Mx)) return fail("null COO arrays");
        ModP m;
        if (!modp_make(&m, prm->prime)) return fail("prime must satisfy 2 <= p < 2^31");
        const int right = prm->right_kernel ? 1 : 0;
        int ndev = 0;
        cudaError_t e0 = cudaGetDeviceCount(&ndev);
        if (e0 != cudaSuccess || ndev == 0)
                return fail(std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e0));
        if (prm->device < 0 || prm->device >= ndev) return fail("device ordinal out of range");
        CU(cudaSetDevice(prm->device));
        struct Stream {
                cudaStream_t st = nullptr;
                ~Stream() { if (st) cudaStreamDestroy(st); }
        } s;
        CU(cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking));
        const int64_t nnz = prm->nnz;
        Scratch up;
        const int32_t *di = (const int32_t *)prm->Mi, *dj = (const int32_t *)prm->Mj;
        const u32 *dx = (const u32 *)prm->Mx;
        if (!prm->coo_on_device && nnz > 0) {
                int32_t *hi = nullptr, *hj = nullptr;
                u32 *hx = nullptr;
                if (up.alloc(&hi, sizeof(int32_t) * (size_t)nnz) || up.alloc(&hj, sizeof(int32_t) * (size_t)nnz) ||
                    up.alloc(&hx, sizeof(u32) * (size_t)nnz))
                        return 1;
                CU(cudaMemcpyAsync(hi, prm->Mi, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, s.st));
                CU(cudaMemcpyAsync(hj, prm->Mj, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, s.st));
                CU(cudaMemcpyAsync(hx, prm->Mx, sizeof(u32) * (size_t)nnz, cudaMemcpyHostToDevice, s.st));
                di = hi; dj = hj; dx = hx;
        }
        PruneResult pr;
        std::string err = prune_coo(di, dj, dx, nnz, prm->nrows, prm->ncols, right, m.p, s.st, &pr);
        if (!err.empty()) return fail(err);
        if (pr.Mc == 0) {
                if (pr.N == 0) return fail("blk_create_pruned: pruning removed every unknown and every constraint: the kernel is {0}");
                return fail("blk_create_pruned: pruning removed every constraint: every vector on the " + std::to_string(pr.N) +
                            " surviving unknowns is a kernel vector");
        }
        if (stats) {
                stats[BLK_PR_N] = pr.N; stats[BLK_PR_MC] = pr.Mc; stats[BLK_PR_NNZ] = pr.nnz;
                stats[BLK_PR_FREE] = pr.free; stats[BLK_PR_ROUNDS] = pr.rounds;
        }
        blk_params p2 = *prm;
        p2.nrows = (int32_t)(right ? pr.Mc : pr.N);
        p2.ncols = (int32_t)(right ? pr.N : pr.Mc);
        p2.nnz = pr.nnz; p2.coo_on_device = 1;
        if (pr.Mx) {
                for (void *q : up.ptrs) up.release(q);
                p2.Mi = pr.Mi; p2.Mj = pr.Mj; p2.Mx = pr.Mx;
        } else {
                p2.Mi = di; p2.Mj = dj; p2.Mx = dx;
        }
        if (blk_create(out, &p2)) return 1;
        blk_ctx *c = *out;
        c->pruned = true;
        c->pr_identity = pr.identity;
        c->pr_unknowns = std::move(pr.unknowns);
        c->pr_constraints = std::move(pr.constraints);
        return 0;
}


// ---------------------------------------------------------------------------------- C ABI
extern "C" {

int blk_create_pruned(blk_ctx **out, const blk_params *prm, int64_t stats[BLK_PR_COUNT])
{
        return create_pruned(out, prm, stats);
}

int blk_pruned_index(blk_ctx *c, int32_t *unknowns, int32_t *constraints)
{
        if (!c) return fail("blk_pruned_index: null context");
        if (!c->pruned) return fail("blk_pruned_index: the context was not made by blk_create_pruned");
        if (c->pr_identity) {
                if (unknowns) for (int64_t u = 0; u < c->N; u++) unknowns[u] = (int32_t)u;
                if (constraints) for (int64_t m = 0; m < c->Mc; m++) constraints[m] = (int32_t)m;
                return 0;
        }
        if (unknowns) std::copy(c->pr_unknowns.begin(), c->pr_unknowns.end(), unknowns);
        if (constraints) std::copy(c->pr_constraints.begin(), c->pr_constraints.end(), constraints);
        return 0;
}

int blk_abi_version(void) { return BLK_ABI_VERSION; }

int blk_create_system(blk_ctx **out, const blk_params *prm, const uint32_t *B, int32_t nrhs, int32_t b_on_device)
{
        return create_system(out, prm, B, nrhs, b_on_device);
}

const char *blk_last_error(void) { return g_err.c_str(); }

int blk_device_count(int *count)
{
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        if (e != cudaSuccess) { *count = 0; return fail(std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e)); }
        *count = n;
        return 0;
}

int blk_nccl_unique_id(void *id_out)
{
        std::string why;
        if (!nccl_load(&why)) return fail(why);
        ncclUniqueId id;
        NC(g_nccl.GetUniqueId(&id));
        static_assert(sizeof(ncclUniqueId) == BLK_NCCL_ID_BYTES, "ncclUniqueId size");
        memcpy(id_out, &id, sizeof(id));
        return 0;
}

int blk_plan_shards(const int32_t *idx, int64_t nnz, int64_t dim, int32_t world, int64_t *offsets)
{
        if (!offsets || dim < 0 || world < 1 || (nnz > 0 && !idx)) return fail("blk_plan_shards: bad argument");
        std::vector<u32> cnt((size_t)dim, 0);
        for (int64_t s = 0; s < nnz; s++) {
                if (idx[s] < 0 || idx[s] >= dim) return fail("blk_plan_shards: index out of range");
                cnt[(size_t)idx[s]]++;
        }
        std::vector<int64_t> off = partition_rows(cnt, world);
        for (int r = 0; r <= world; r++) offsets[r] = off[r];
        return 0;
}

int blk_plan_heavy(const uint32_t *deg, int64_t rows, int64_t cols, int32_t n_pad, int64_t l2_bytes, int64_t min_deg,
                   int64_t band_bytes, int32_t force, int64_t *heavy_rows, int32_t *bands)
{
        if (!heavy_rows || !bands || rows < 0 || cols < 0 || (rows > 0 && !deg)) return fail("blk_plan_heavy: bad argument");
        const HeavyPlan plan = plan_heavy(deg, rows, cols, n_pad, l2_bytes, min_deg, band_bytes, force != 0);
        *heavy_rows = plan.rows;
        *bands = plan.bands;
        return 0;
}

int blk_plan_grid(const int32_t *Mi, const int32_t *Mj, int64_t nnz, int32_t nrows, int32_t ncols, int32_t right_kernel,
                  int32_t world, int32_t grid[2], int64_t *n_off, int64_t *m_off, int64_t *n_sub, int64_t *m_sub,
                  int64_t *block_nnz)
{
        if (!grid || !n_off || !m_off || !n_sub || !m_sub || world < 1 || nrows < 0 || ncols < 0 || (nnz > 0 && (!Mi || !Mj)))
                return fail("blk_plan_grid: bad argument");
        int P = grid[0], Q = grid[1];
        if (P == 0 && Q == 0) {
                // MPI_Dims_create(world, 2): the most square factorisation, larger factor first
                Q = 1;
                for (int q = 1; (int64_t)q * q <= world; q++)
                        if (world % q == 0) Q = q;
                P = world / Q;
        }
        if (P < 1 || Q < 1 || (int64_t)P * Q != world) return fail("blk_plan_grid: grid does not match world");
        const int64_t N = right_kernel ? ncols : nrows, Mc = right_kernel ? nrows : ncols;
        const int32_t *iN = right_kernel ? Mj : Mi, *iM = right_kernel ? Mi : Mj;
        std::vector<u32> cn((size_t)N, 0), cm((size_t)Mc, 0);
        for (int64_t s = 0; s < nnz; s++) {
                if (iN[s] < 0 || iN[s] >= N || iM[s] < 0 || iM[s] >= Mc) return fail("blk_plan_grid: index out of range");
                cn[(size_t)iN[s]]++; cm[(size_t)iM[s]]++;
        }
        std::vector<int64_t> no = partition_rows(cn, P), mo = partition_rows(cm, Q);
        for (int a = 0; a <= P; a++) n_off[a] = no[a];
        for (int b = 0; b <= Q; b++) m_off[b] = mo[b];
        // owned pieces: dense work and exchange volume go with rows, so blocks are cut into equal row counts
        for (int a = 0; a < P; a++)
                for (int b = 0; b <= Q; b++) n_sub[(size_t)a * (Q + 1) + b] = no[a] + (no[a + 1] - no[a]) * b / Q;
        for (int b = 0; b < Q; b++)
                for (int a = 0; a <= P; a++) m_sub[(size_t)b * (P + 1) + a] = mo[b] + (mo[b + 1] - mo[b]) * a / P;
        if (block_nnz) {
                std::vector<int> bn((size_t)N), bm((size_t)Mc);
                for (int a = 0; a < P; a++) for (int64_t r = no[a]; r < no[a + 1]; r++) bn[(size_t)r] = a;
                for (int b = 0; b < Q; b++) for (int64_t r = mo[b]; r < mo[b + 1]; r++) bm[(size_t)r] = b;
                for (int e = 0; e < P * Q; e++) block_nnz[e] = 0;
                for (int64_t s = 0; s < nnz; s++) block_nnz[(size_t)bn[(size_t)iN[s]] * Q + bm[(size_t)iM[s]]]++;
        }
        grid[0] = P; grid[1] = Q;
        return 0;
}

int64_t blk_block_pad(int32_t nrows, int32_t ncols, int32_t n, int32_t right_kernel)
{
        int64_t N = right_kernel ? ncols : nrows, Mc = right_kernel ? nrows : ncols;
        int64_t a = ((N + n - 1) / n) * n, b = ((Mc + n - 1) / n) * n;
        return (a > b ? a : b) * n;
}

int blk_destroy(blk_ctx *c)
{
        if (!c) return 0;
        if (c->is_group()) {
                group_run(c, [](blk_ctx *mem, int) { return blk_destroy(mem); });
                delete c;
                return 0;
        }
        cudaSetDevice(c->device);
        if (c->stream) cudaStreamSynchronize(c->stream);
        if (c->comm_stream) cudaStreamSynchronize(c->comm_stream);
        destroy_graph(c);
        grid_destroy(c);
        if (!c->peer_tmp.empty()) {
                // peers hold mappings of this rank's blocks (and this rank of theirs): unmap, then meet, then free
                close_peers(c);
                if (c->comm && c->barrier_word && c->stream) {
                        g_nccl.AllReduce(c->barrier_word, c->barrier_word, 1, ncclUint64, ncclSum, c->comm, c->stream);
                        cudaStreamSynchronize(c->stream);
                }
        }
        if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
        free_operator(&c->S1);
        free_operator(&c->S2);
        free_colops(&c->cb1); free_colops(&c->cb2);
        cudaFree(c->zbuf);
        for (auto e : c->ev_arrived) cudaEventDestroy(e);
        if (c->ev_aux) cudaEventDestroy(c->ev_aux);
        cudaFree(c->v); cudaFree(c->tmp); cudaFree(c->p);
        if (c->Av_full) cudaFree(c->Av_full); else cudaFree(c->Av);
        cudaFree(c->Tp); cudaFree(c->U); cudaFree(c->tmp_prev);
        cudaFree(c->mats); cudaFree(c->sums); cudaFree(c->state); cudaFree(c->dots_counter);
        cudaFree(c->n_old2new); cudaFree(c->n_new2old);
        cudaFree(c->stage); cudaFree(c->loop_bar);
        if (c->h_state) cudaFreeHost(c->h_state);
        for (auto e : c->ev_copies) cudaEventDestroy(e);
        for (auto st : c->copy_streams) cudaStreamDestroy(st);
        cudaFree(c->barrier_word);
        for (auto e : c->ev_piece) cudaEventDestroy(e);
        if (c->ev_comm) cudaEventDestroy(c->ev_comm);
        if (c->comm_stream) cudaStreamDestroy(c->comm_stream);
        if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
        if (c->l2_persist_before >= 0) cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)c->l2_persist_before);
        cudaGetLastError();
        delete c;
        return 0;
}


int blk_set_state(blk_ctx *c, const uint32_t *v, const uint32_t *p, int32_t n_iterations)
{
        if (!c || !v) return fail("blk_set_state: null argument");
        if (c->is_group()) return group_run(c, [&](blk_ctx *mem, int) { return blk_set_state(mem, v, p, n_iterations); });
        CU(cudaSetDevice(c->device));
        const int np = c->geo.np, n = c->geo.n;
        // Every rank reads only ITS share of the host blocks (1/world of the PCIe traffic); the rest of v arrives
        // from the peers over NVLink.
        const int64_t n0 = c->n0(), ln = c->n1() - n0;
        const size_t full_rows = (size_t)gather_cap(c->n_off);
        u32 *pfull = nullptr;                      // p under device labels, all rows (only where it is needed)
        struct Free { u32 *&q; ~Free() { cudaFree(q); } } free_pfull{pfull};
        if (c->relabel_mg()) {
                // host rows [h0, h1) scattered to their labels; exactly one rank contributes each element, so a
                // sum over the ranks assembles the block
                const int64_t h0 = c->h0(), hl = c->h1() - h0;
                CU(cudaMemsetAsync(c->v, 0, sizeof(u32) * full_rows * np, c->stream));
                if (upload_rows(c, c->v, v + (size_t)h0 * n, hl, c->n_old2new, h0)) return 1;
                NC(g_nccl.AllReduce(c->v, c->v, (size_t)c->N * np, ncclUint32, ncclSum, c->comm, c->stream));
                if (p) {
                        CU(cudaMalloc(&pfull, sizeof(u32) * full_rows * np));
                        CU(cudaMemsetAsync(pfull, 0, sizeof(u32) * full_rows * np, c->stream));
                        if (upload_rows(c, pfull, p + (size_t)h0 * n, hl, c->n_old2new, h0)) return 1;
                        NC(g_nccl.AllReduce(pfull, pfull, (size_t)c->N * np, ncclUint32, ncclSum, c->comm, c->stream));
                        CU(cudaMemcpyAsync(c->p, pfull + (size_t)n0 * np, sizeof(u32) * (size_t)ln * np, cudaMemcpyDeviceToDevice, c->stream));
                }
        } else {
                if (upload_rows(c, c->n_old2new ? c->v : c->v + (size_t)n0 * np, v + (size_t)n0 * n, ln, c->n_old2new, n0)) return 1;
                if (c->world > 1 && allgather_rows(c, c->v, c->n_off)) return 1;
                if (p && upload_rows(c, c->p, p + (size_t)n0 * n, ln, c->n_old2new, n0)) return 1;
                if (p && c->mg_recur) {
                        CU(cudaMalloc(&pfull, sizeof(u32) * full_rows * np));
                        CU(cudaMemcpyAsync(pfull + (size_t)n0 * np, c->p, sizeof(u32) * (size_t)ln * np, cudaMemcpyDeviceToDevice, c->stream));
                        if (allgather_rows(c, pfull, c->n_off)) return 1;
                }
        }
        if (!p) CU(cudaMemsetAsync(c->p, 0, sizeof(u32) * (size_t)(ln > 0 ? ln : 1) * np, c->stream));
        CU(cudaMemsetAsync(c->tmp, 0, sizeof(u32) * (size_t)c->Mc * np, c->stream));
        if (c->Av_full) CU(cudaMemsetAsync(c->Av_full, 0, sizeof(u32) * full_rows * np, c->stream));
        else CU(cudaMemsetAsync(c->Av, 0, sizeof(u32) * (size_t)(ln > 0 ? ln : 1) * np, c->stream));
        // invariant of the multi-GPU loop: tmp = S1 v (gathered), Tp = S1 p (local rows)
        if (c->mg_recur && mg_prepare(c, p ? pfull : nullptr)) return 1;
        if (c->grid_on && grid_import(c, p)) return 1;
        c->ran_since_set = false;
        c->iters = n_iterations; c->stopped = 0;
        c->tmp_is_spmv = false; c->any_ortho = n_iterations > 0;
        memset(c->h_state, 0, sizeof(DevSmall));
        c->h_state->iters = n_iterations;
        c->h_state->halt = 1;
        c->h_state->check = c->check ? 1 : 0;
        c->h_state->fault_iter = c->check_fault;
        if (push_state(c)) return 1;
        CU(cudaStreamSynchronize(c->stream));
        return 0;
}

int blk_iterate(blk_ctx *c, int32_t max_iters, int32_t *iters_total, int32_t *stopped)
{
        if (!c) return fail("blk_iterate: null context");
        if (c->is_group()) {
                std::vector<int32_t> it(c->members.size(), 0), st(c->members.size(), 0);
                if (group_run(c, [&](blk_ctx *mem, int r) { return blk_iterate(mem, max_iters, &it[(size_t)r], &st[(size_t)r]); })) return 1;
                c->iters = it[0]; c->stopped = st[0];
                if (iters_total) *iters_total = it[0];
                if (stopped) *stopped = st[0];
                return 0;
        }
        CU(cudaSetDevice(c->device));
        if (max_iters > 0 && !c->stopped) {
                c->h_state->iters = c->iters;
                c->h_state->limit = c->iters + max_iters;
                c->h_state->stopped = 0; c->h_state->halt = 0; c->h_state->do_ortho = 0;
                if (push_state(c)) return 1;
                bool graph = c->use_graph == 1 || (c->use_graph < 0 && c->world == 1 && max_iters >= 4);
                if (c->profiling || c->world > 1 || c->colblocks) graph = false;
                // (use_graph == 0 asks for the plain chain of kernels; per-phase profiling needs kernel boundaries)
                const bool coop = c->coop && c->use_graph != 0 && (!c->profiling || c->coop_prof);
                if (coop) graph = false;
                EventTimer tm;
                int done = 0;
                if (graph && !c->graph) {
                        // first iteration runs un-captured so that every kernel is loaded before capture
                        if (enqueue_iteration(c, nullptr)) return 1;
                        done = 1;
                        if (build_graph(c)) return 1;
                }
                const int check_every = coop ? blk_ctx::COOP_BATCH : (graph ? 16 * blk_ctx::GRAPH_ITERS : 64);
                while (done < max_iters) {
                        int batch = std::min(check_every, max_iters - done);
                        if (coop) {
                                if (enqueue_loop_coop(c, batch)) return 1;
                        } else if (graph) {
                                int ng = (batch + blk_ctx::GRAPH_ITERS - 1) / blk_ctx::GRAPH_ITERS;
                                for (int i = 0; i < ng; i++) CU(cudaGraphLaunch(c->graph, c->stream));
                                c->launches += (int64_t)ng * blk_ctx::GRAPH_ITERS * kernels_per_iteration(c);
                        } else {
                                for (int i = 0; i < batch; i++)
                                        if (enqueue_iteration(c, c->profiling ? &tm : nullptr)) return 1;
                        }
                        done += batch;
                        if (drain_exchange(c)) return 1;
                        if (pull_state(c)) return 1;
                        if (c->profiling) tm.resolve(c);
                        if (c->h_state->halt) break;
                }
                if (c->h_state->check_failed) {
                        // the reference aborts on a failed assert of correctness_tests (sequential/lanczos_modp.c:532-557, :647)
                        static const char *what[5] = {"vtAv not symmetric", "vtAAv not symmetric", "winv not symmetric",
                                                      "winv not supported on the pivots", "winv * vtAv * D != D"};
                        std::string msg = "correctness_tests failed in iteration " + std::to_string(c->h_state->iters + 1) + ":";
                        for (int b = 0; b < 5; b++)
                                if (c->h_state->check_failed & (1 << b)) msg += std::string(" ") + what[b] + ";";
                        c->iters = c->h_state->iters;
                        return fail(msg);
                }
                int before = c->iters;
                c->iters = c->h_state->iters;
                c->stopped = c->h_state->stopped;
                if (c->stopped) c->tmp_is_spmv = true;
                else if (c->iters > before) c->tmp_is_spmv = false;
                if (c->iters > before) c->any_ortho = true;
                c->ran_since_set = true;
        }
        if (iters_total) *iters_total = c->iters;
        if (stopped) *stopped = c->stopped;
        return 0;
}

// Host rows [0, lim) of a block along the Lanczos dimension into dst (w words per host row, wp per device row).  `own`
// holds this rank's rows [n0, n1) (device labels); `full` (nullable) is a buffer of gather_cap(n_off) rows holding them
// in place, else a gathered copy is made here when one is needed:
//   relabelled rows on several GPUs: a rank's rows are scattered over the host order, so the block is gathered over
//     NVLink (device labels) and every rank unpermutes its share [h0, h1) of HOST rows (all of them when whole)
//   whole at world > 1 (a rank of a multi-process job must return complete blocks): gather, then every row
//   otherwise: this rank's rows (unpermuted on the way down when one GPU holds a relabelled dimension)
static int download_owned(blk_ctx *c, u32 *dst, int w, int wp, const u32 *own, u32 *full, int64_t lim, bool whole)
{
        const bool all = whole && c->world > 1;
        const int64_t n0 = c->n0(), ln = c->n1() - n0;
        if (!c->relabel_mg() && !all) {
                const int64_t lo = std::min(n0, lim), hi = std::min(n0 + ln, lim);
                return download_rows(c, dst + (size_t)lo * w, own, hi - lo, c->n_old2new, lo, w, wp);
        }
        u32 *copy = nullptr;
        int rc = 0;
        if (!full) {
                CU(cudaMalloc(&copy, sizeof(u32) * (size_t)gather_cap(c->n_off) * wp));
                full = copy;
                if (cudaMemcpyAsync(full + (size_t)n0 * wp, own, sizeof(u32) * (size_t)ln * wp, cudaMemcpyDeviceToDevice,
                                    c->stream) != cudaSuccess)
                        rc = fail("device copy failed");
        }
        const int64_t r0 = all ? 0 : std::min(c->h0(), lim), r1 = all ? lim : std::min(c->h1(), lim);
        if (!rc) rc = allgather_rows(c, full, c->n_off, wp);
        if (!rc) rc = download_rows(c, dst + (size_t)r0 * w, full, r1 - r0, c->n_old2new, r0, w, wp);
        cudaFree(copy);
        return rc;
}

// What one rank contributes to blk_get_state: rows of v / Av / p straight into the caller's blocks (host layout,
// n per row, written at their global row position) and rows of the device's tmp into `ht` (Mc x n).
// whole = false: only this rank's rows (the blocks of a job are then assembled from the ranks' slices: group
// contexts, blk_get_state_local); whole = true: every row (download_owned).
static int download_state(blk_ctx *c, u32 *v, u32 *Av, u32 *p, u32 *ht, bool whole)
{
        CU(cudaSetDevice(c->device));
        const int n = c->geo.n, np = c->geo.np;
        if (c->grid_on && grid_export(c)) return 1;
        const bool all = whole && c->world > 1;
        const int64_t n0 = c->n0(), m0 = c->m0(), lm = c->m1() - c->m0();
        if (v && download_owned(c, v, n, np, c->v + (size_t)n0 * np, c->v, c->N, whole)) return 1;
        if (Av && download_owned(c, Av, n, np, c->Av, nullptr, c->N, whole)) return 1;
        if (p && download_owned(c, p, n, np, c->p, nullptr, c->N, whole)) return 1;
        if (ht) {
                if (c->mg_recur && !c->ran_since_set) {
                        // nothing has run since blk_set_state: the reference's tmp is still all zero there (the
                        // device already holds S1*v for the first iteration); the caller zero-fills
                } else if (c->mg_recur && !c->tmp_is_spmv && c->Mc > c->N) {
                        // the device tmp already belongs to the NEXT iteration; the reference still shows the
                        // previous product in rows [N,Mc): the saved copy
                        if (all) {
                                u32 *full = nullptr;
                                CU(cudaMalloc(&full, sizeof(u32) * (size_t)gather_cap(c->m_off) * np));
                                int rc = 0;
                                if (cudaMemcpyAsync(full + (size_t)m0 * np, c->tmp_prev, sizeof(u32) * (size_t)lm * np, cudaMemcpyDeviceToDevice, c->stream) != cudaSuccess)
                                        rc = fail("blk_get_state: device copy failed");
                                if (!rc) rc = allgather_rows(c, full, c->m_off);
                                if (!rc) rc = download_rows(c, ht, full, c->Mc);
                                cudaFree(full);
                                if (rc) return 1;
                        } else if (download_rows(c, ht + (size_t)m0 * n, c->tmp_prev, lm)) return 1;
                } else if (all || c->world == 1) {
                        if (download_rows(c, ht, c->tmp, c->Mc)) return 1;
                } else if (download_rows(c, ht + (size_t)m0 * n, c->tmp + (size_t)m0 * np, lm)) return 1;
        }
        return 0;
}

// The reference's tmp block from the device's (DESIGN.md "tmp"): the reference's tmp holds the next v in rows
// [0,N) after orthogonalize + copy (:652-656) and S1*v in rows [0,Mc) after the first product (:635).
static void compose_tmp(const blk_ctx *c, u32 *tmp, std::vector<u32> &ht, const u32 *vsrc, int64_t pad)
{
        const int n = c->geo.n;
        const int64_t N = c->N, Mc = c->Mc;
        memset(tmp, 0, sizeof(u32) * (size_t)pad);
        if (c->mg_recur && !c->ran_since_set) std::fill(ht.begin(), ht.end(), 0u);
        if (c->tmp_is_spmv) {
                if (c->any_ortho && N > Mc)
                        memcpy(tmp + (size_t)Mc * n, vsrc + (size_t)Mc * n, sizeof(u32) * (size_t)(N - Mc) * n);
                memcpy(tmp, ht.data(), sizeof(u32) * (size_t)Mc * n);
        } else {
                if (Mc > N)
                        memcpy(tmp + (size_t)N * n, ht.data() + (size_t)N * n, sizeof(u32) * (size_t)(Mc - N) * n);
                if (c->any_ortho) memcpy(tmp, vsrc, sizeof(u32) * (size_t)N * n);
                else memcpy(tmp, ht.data(), sizeof(u32) * (size_t)std::min(N, Mc) * n);
        }
}

int blk_get_state(blk_ctx *c, uint32_t *v, uint32_t *tmp, uint32_t *Av, uint32_t *p)
{
        if (!c) return fail("blk_get_state: null context");
        const int n = c->geo.n;
        const int64_t pad = blk_block_pad(c->nrows, c->ncols, n, c->right);
        const int64_t N = c->N, Mc = c->Mc;
        std::vector<u32> hv, ht;
        u32 *vdst = v;
        if (!v && tmp) { hv.resize((size_t)N * n); vdst = hv.data(); }
        if (tmp) ht.resize((size_t)Mc * n);
        u32 *htp = tmp ? ht.data() : nullptr;
        const blk_ctx *flags = c;
        if (c->is_group()) {
                // one host block, every GPU writes its own rows into it: PCIe traffic is shared, nothing crosses NVLink
                if (group_run(c, [&](blk_ctx *mem, int) { return download_state(mem, vdst, Av, p, htp, false); })) return 1;
                flags = c->members[0];
        } else if (download_state(c, vdst, Av, p, htp, true)) return 1;
        const size_t tail = sizeof(u32) * (size_t)(pad - N * n);
        if (v) memset(v + (size_t)N * n, 0, tail);
        if (Av) memset(Av + (size_t)N * n, 0, tail);
        if (p) memset(p + (size_t)N * n, 0, tail);
        if (tmp) compose_tmp(flags, tmp, ht, vdst, pad);
        return 0;
}

int blk_get_state_local(blk_ctx *c, uint32_t *v, uint32_t *Av, uint32_t *p)
{
        if (!c) return fail("blk_get_state_local: null context");
        if (c->is_group()) return blk_get_state(c, v, nullptr, Av, p);
        return download_state(c, v, Av, p, nullptr, false);
}

// This rank's rows [m0, m1) of T = S1 v of the current v: tmp already holds them when the loop stopped on "no pivot"
// (or, in the multi-GPU recurrence, whenever the loop has run); otherwise S1 v goes into *scratch, allocated here and
// freed by the caller.  v, tmp, Av and p are left as they are.
static int rows_of_T(blk_ctx *c, const u32 **t, u32 **scratch)
{
        const int np = c->geo.np;
        const int64_t lm = c->m1() - c->m0();
        *t = c->tmp + (size_t)c->m0() * np;
        *scratch = nullptr;
        if (c->tmp_is_spmv || (c->mg_recur && c->ran_since_set)) return 0;
        if (c->world > 1 && allgather_rows(c, c->v, c->n_off)) return 1;
        CU(cudaMalloc(scratch, sizeof(u32) * (size_t)std::max<int64_t>(lm, 1) * np));
        c->launches += launch_spmv(c->S1, c->geo, c->m, c->v, *scratch, nullptr, c->stream);
        *t = *scratch;
        return 0;
}

int blk_final_check(blk_ctx *c, int32_t *v_nonzero, int32_t *vtm_zero)
{
        if (!c || !v_nonzero || !vtm_zero) return fail("blk_final_check: null argument");
        if (c->is_group()) {
                std::vector<int32_t> a(c->members.size(), 0), b(c->members.size(), 0);
                if (group_run(c, [&](blk_ctx *mem, int r) { return blk_final_check(mem, &a[(size_t)r], &b[(size_t)r]); })) return 1;
                *v_nonzero = a[0]; *vtm_zero = b[0];
                return 0;
        }
        CU(cudaSetDevice(c->device));
        const int np = c->geo.np;
        int nz = 0, big = 0;
        if (c->grid_on && grid_export(c)) return 1;
        // v: every rank scans its own rows (padding columns are zero)
        if (scan_rows(c, c->v + (size_t)c->n0() * np, c->n1() - c->n0(), &nz, &big)) return 1;
        *v_nonzero = nz;
        // T = S1 v: every rank scans its own rows
        const u32 *t = nullptr;
        u32 *scratch = nullptr;
        if (rows_of_T(c, &t, &scratch)) return 1;
        int rc = scan_rows(c, t, c->m1() - c->m0(), &nz, &big);
        cudaFree(scratch);
        if (rc) return 1;
        *vtm_zero = !nz;
        return 0;
}

int blk_check_kernel_block(blk_ctx *c, const uint32_t *x, int32_t *ok)
{
        if (!c || !x || !ok) return fail("blk_check_kernel_block: null argument");
        if (c->is_group()) {
                std::vector<int32_t> o(c->members.size(), 0);
                if (group_run(c, [&](blk_ctx *mem, int r) { return blk_check_kernel_block(mem, x, &o[(size_t)r]); })) return 1;
                *ok = o[0];
                return 0;
        }
        CU(cudaSetDevice(c->device));
        const int np = c->geo.np;
        const int64_t lm = c->m1() - c->m0();
        u32 *dx = nullptr, *dy = nullptr;
        CU(cudaMalloc(&dx, sizeof(u32) * (size_t)c->N * np));
        CU(cudaMalloc(&dy, sizeof(u32) * (size_t)(lm > 0 ? lm : 1) * np));
        int rc = upload_rows(c, dx, x, c->N, c->n_old2new);
        int nz = 0, big = 0, ynz = 0, ybig = 0;
        if (!rc) rc = scan_rows(c, dx + (size_t)c->n0() * np, c->n1() - c->n0(), &nz, &big);
        if (!rc && !big) {
                // entries >= p are rejected before the product, as in checker_modp.c:150-153
                c->launches += launch_spmv(c->S1, c->geo, c->m, dx, dy, nullptr, c->stream);
                rc = scan_rows(c, dy, lm, &ynz, &ybig);
        }
        cudaFree(dx); cudaFree(dy);
        if (rc) return 1;
        *ok = nz && !big && !ynz;
        return 0;
}

// One rank of blk_kernel_basis (found == nullptr) or blk_solve: its rows of v and T reduced to two records, the records
// of all ranks gathered (one NCCL all-gather) and the n x n stage run redundantly on every rank, giving A_S and k.  The
// kernel basis is X = v A_S.  A solve takes the r tail rows of v from their owners (one NCCL all-reduce: every entry
// has one owner, the others add zero), runs the r x k stage redundantly on every rank for W = A_S C and found, and
// forms x = v W; rows from N0 = N - r on (the right-hand-side coordinates) are not part of x.  Every rank forms the
// rows it owns.  whole: write every row of the output (a rank of a multi-process job), else only this rank's rows
// (group members).
static int extract_rank(blk_ctx *c, uint32_t *x, int32_t *k, int32_t *found, bool whole)
{
        CU(cudaSetDevice(c->device));
        const int n = c->geo.n, np = c->geo.np;
        const int r = found ? c->nrhs : 0, w = found ? r : n, wp = found ? pad_width(r) : np;
        if (c->grid_on && grid_export(c)) return 1;
        const int64_t n0 = c->n0(), ln = c->n1() - n0, lm = c->m1() - c->m0();
        struct Bufs {
                std::vector<void *> p;
                ~Bufs() { for (void *q : p) cudaFree(q); }
        } bufs;
        auto grab = [&](void **dst, size_t bytes) {
                cudaError_t e = cudaMalloc(dst, bytes ? bytes : 4);
                if (e == cudaSuccess) bufs.p.push_back(*dst);
                return e;
        };
        KbArgs a;
        a.n = n; a.world = c->world; a.m = c->m;
        a.v = c->v + (size_t)n0 * np; a.vrows = ln;
        a.trows = lm;
        a.ctas = kb_ctas(std::max(ln, lm));
        u32 *scratch = nullptr, *xf = nullptr;
        const int trc = rows_of_T(c, &a.t, &scratch);
        if (scratch) bufs.p.push_back(scratch);
        if (trc) return 1;
        const size_t rec_words = (size_t)(n + 1) * np;
        CU(grab((void **)&a.part, sizeof(u32) * (size_t)2 * a.ctas * n * np));
        CU(grab((void **)&a.prank, sizeof(int) * (size_t)2 * a.ctas));
        CU(grab((void **)&a.counter, sizeof(unsigned)));
        CU(grab((void **)&a.rec_all, sizeof(u32) * (size_t)c->world * 2 * rec_words));
        CU(grab((void **)&a.A, sizeof(u32) * (size_t)np * np));
        CU(grab((void **)&a.k, sizeof(int)));
        CU(grab((void **)&xf, sizeof(u32) * (size_t)gather_cap(c->n_off) * wp));
        a.rec_own = a.rec_all + (size_t)c->rank * 2 * rec_words;
        CU(cudaMemsetAsync(a.counter, 0, sizeof(unsigned), c->stream));
        c->launches += launch_kb_reduce(np, a, c->stream);
        if (c->world > 1)
                NC(g_nccl.AllGather(a.rec_own, a.rec_all, 2 * rec_words, ncclUint32, c->comm, c->stream));
        c->launches += launch_kb_small(np, a, c->stream);
        SolveArgs s;
        s.W = a.A;
        if (found) {
                s.np = np; s.r = r; s.rp = wp; s.m = c->m; s.A = a.A; s.k = a.k;
                CU(grab((void **)&s.tail, sizeof(u32) * (size_t)r * np));
                CU(grab((void **)&s.W, sizeof(u32) * (size_t)np * wp));
                CU(grab((void **)&s.found, sizeof(int) * (size_t)r));
                c->launches += launch_solve_tail(s, c->N - r, c->v, c->n_old2new, n0, n0 + ln, c->stream);
                if (c->world > 1)
                        NC(g_nccl.AllReduce(s.tail, s.tail, (size_t)r * np, ncclUint32, ncclSum, c->comm, c->stream));
                c->launches += launch_solve_small(s, c->stream);
        }
        c->launches += launch_block_apply(np, wp, ln, a.v, s.W, xf + (size_t)n0 * wp, c->m, c->stream);
        std::vector<int> h((size_t)(found ? r : 1), 0);
        CU(cudaMemcpyAsync(h.data(), found ? s.found : a.k, sizeof(int) * h.size(), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        CU(cudaGetLastError());
        if (download_owned(c, x, w, wp, xf + (size_t)n0 * wp, xf, c->N - r, whole)) return 1;
        std::copy(h.begin(), h.end(), found ? found : k);
        return 0;
}

int blk_kernel_basis(blk_ctx *c, uint32_t *x, int32_t *k)
{
        if (!c || !x || !k) return fail("blk_kernel_basis: null argument");
        if (c->is_group()) {
                // every GPU writes its own rows into the one host block
                std::vector<int32_t> kk(c->members.size(), 0);
                if (group_run(c, [&](blk_ctx *mem, int r) { return extract_rank(mem, x, &kk[(size_t)r], nullptr, false); })) return 1;
                *k = kk[0];
                return 0;
        }
        return extract_rank(c, x, k, nullptr, true);
}

int blk_solve(blk_ctx *c, uint32_t *x, int32_t *found)
{
        if (!c || !x || !found) return fail("blk_solve: null argument");
        if (c->nrhs < 1) return fail("blk_solve: the context has no right-hand sides (create it with blk_create_system)");
        if (c->is_group()) {
                // every GPU writes its own rows into the one host block
                std::vector<std::vector<int32_t>> ff(c->members.size(), std::vector<int32_t>((size_t)c->nrhs, 0));
                if (group_run(c, [&](blk_ctx *mem, int r) { return extract_rank(mem, x, nullptr, ff[(size_t)r].data(), false); })) return 1;
                for (int j = 0; j < c->nrhs; j++) found[j] = ff[0][(size_t)j];
                return 0;
        }
        return extract_rank(c, x, nullptr, found, true);
}

int blk_get_small(blk_ctx *c, uint32_t *vtAv, uint32_t *vtAAv, uint32_t *winv, uint32_t *d, int32_t *npiv)
{
        if (!c) return fail("blk_get_small: null context");
        if (c->is_group()) return blk_get_small(c->members[0], vtAv, vtAAv, winv, d, npiv);
        CU(cudaSetDevice(c->device));
        const int n = c->geo.n, np = c->geo.np;
        std::vector<u32> h((size_t)MAT_COUNT * np * np);
        CU(cudaMemcpyAsync(h.data(), c->mats, sizeof(u32) * h.size(), cudaMemcpyDeviceToHost, c->stream));
        if (pull_state(c)) return 1;
        auto take = [&](uint32_t *dst, int which) {
                if (!dst) return;
                for (int i = 0; i < n; i++)
                        for (int j = 0; j < n; j++) dst[i * n + j] = h[(size_t)which * np * np + i * np + j];
        };
        take(vtAv, MAT_VTAV); take(vtAAv, MAT_VTAAV); take(winv, MAT_WINV);
        if (d) for (int j = 0; j < n; j++) d[j] = h[(size_t)MAT_D * np * np + j];
        if (npiv) *npiv = c->h_state->npiv;
        return 0;
}

// ---- per-function entry points -----------------------------------------------------------
static SpOp *op_for(blk_ctx *c, int transpose, bool *is_s1)
{
        // S1 is M^T for --left and M for --right (sequential/lanczos_modp.c:635)
        bool s1 = (transpose != 0) == (c->right == 0);
        *is_s1 = s1;
        return s1 ? &c->S1 : &c->S2;
}

int blk_spmv(blk_ctx *c, uint32_t *y, const uint32_t *x, int32_t transpose)
{
        if (!c || !y || !x) return fail("blk_spmv: null argument");
        if (c->is_group()) {
                // every member returns the whole product (gathered over NVLink); only the first one's goes to y
                const size_t out = (size_t)((transpose != 0) == (c->right == 0) ? c->Mc : c->N) * c->geo.n;
                return group_run(c, [&](blk_ctx *mem, int r) {
                        if (r == 0) return blk_spmv(mem, y, x, transpose);
                        std::vector<u32> scratch(out);
                        return blk_spmv(mem, scratch.data(), x, transpose);
                });
        }
        CU(cudaSetDevice(c->device));
        const int np = c->geo.np;
        bool s1;
        SpOp *op = op_for(c, transpose, &s1);
        const std::vector<int64_t> &off = s1 ? c->m_off : c->n_off;
        int64_t out_rows = s1 ? c->Mc : c->N, in_rows = s1 ? c->N : c->Mc;
        u32 *dx = nullptr, *dy = nullptr;
        CU(cudaMalloc(&dx, sizeof(u32) * (size_t)in_rows * np));
        CU(cudaMalloc(&dy, sizeof(u32) * (size_t)gather_cap(off) * np));
        int rc = upload_rows(c, dx, x, in_rows, s1 ? c->n_old2new : nullptr);
        if (!rc) {
                // poison the output: every row must be written by the kernels
                cudaMemsetAsync(dy, 0xff, sizeof(u32) * (size_t)out_rows * np, c->stream);
                int k = launch_spmv(*op, c->geo, c->m, dx, dy + (size_t)off[c->rank] * np, nullptr, c->stream);
                c->launches += k;
                if (c->world > 1) rc = allgather_rows(c, dy, off);
        }
        if (!rc) rc = download_rows(c, y, dy, out_rows, s1 ? nullptr : c->n_old2new);
        cudaError_t e = cudaGetLastError();
        cudaFree(dx); cudaFree(dy);
        if (!rc && e != cudaSuccess) return fail(std::string("blk_spmv: ") + cudaGetErrorString(e));
        return rc;
}

int blk_block_dot_products(blk_ctx *c, uint32_t *vtAv, uint32_t *vtAAv, int64_t N, const uint32_t *Av,
                           const uint32_t *v)
{
        if (!c || !vtAv || !vtAAv || !Av || !v || N < 0) return fail("blk_block_dot_products: bad argument");
        if (c->is_group()) return blk_block_dot_products(c->members[0], vtAv, vtAAv, N, Av, v);
        CU(cudaSetDevice(c->device));
        const int np = c->geo.np, n = c->geo.n;
        u32 *dv = nullptr, *da = nullptr, *mats = nullptr;
        u64 *sums = nullptr;
        int64_t rows = N > 0 ? N : 1;
        int nblocks = dots_num_blocks(N, np);
        CU(cudaMalloc(&dv, sizeof(u32) * (size_t)rows * np));
        CU(cudaMalloc(&da, sizeof(u32) * (size_t)rows * np));
        CU(cudaMalloc(&sums, sizeof(u64) * (size_t)2 * np * np));
        CU(cudaMalloc(&mats, sizeof(u32) * mats_words(np)));
        CU(cudaMemsetAsync(sums, 0, sizeof(u64) * (size_t)2 * np * np, c->stream));
        int rc = upload_rows(c, dv, v, N) || upload_rows(c, da, Av, N);
        if (!rc) {
                c->launches += launch_dots(c->geo, c->m, N, dv, da, sums, nblocks, nullptr, SmallFuse(), c->stream);
                c->launches += launch_small(c->geo, c->m, sums, mats, c->state, 1, c->stream);
                std::vector<u32> h((size_t)2 * np * np);
                cudaMemcpyAsync(h.data(), mats, sizeof(u32) * h.size(), cudaMemcpyDeviceToHost, c->stream);
                cudaError_t e = cudaStreamSynchronize(c->stream);
                if (e != cudaSuccess) rc = fail(std::string("blk_block_dot_products: ") + cudaGetErrorString(e));
                else
                        for (int i = 0; i < n; i++)
                                for (int j = 0; j < n; j++) {
                                        vtAv[i * n + j] = h[(size_t)MAT_VTAV * np * np + i * np + j];
                                        vtAAv[i * n + j] = h[(size_t)MAT_VTAAV * np * np + i * np + j];
                                }
        }
        cudaFree(dv); cudaFree(da); cudaFree(sums); cudaFree(mats);
        return rc;
}

static void put_small(std::vector<u32> &h, int which, const uint32_t *src, int n, int np)
{
        for (int i = 0; i < n; i++)
                for (int j = 0; j < n; j++) h[(size_t)which * np * np + i * np + j] = src[i * n + j];
}

int blk_semi_inverse(blk_ctx *c, const uint32_t *M_, uint32_t *winv, uint32_t *d, int32_t *npiv)
{
        if (!c || !M_ || !winv || !d) return fail("blk_semi_inverse: null argument");
        if (c->is_group()) return blk_semi_inverse(c->members[0], M_, winv, d, npiv);
        CU(cudaSetDevice(c->device));
        const int np = c->geo.np, n = c->geo.n;
        std::vector<u32> h((size_t)MAT_COUNT * np * np, 0);
        put_small(h, MAT_VTAV, M_, n, np);
        u32 *mats = nullptr;
        DevSmall *st = nullptr;
        CU(cudaMalloc(&mats, sizeof(u32) * mats_words(np)));
        CU(cudaMalloc(&st, sizeof(DevSmall)));
        CU(cudaMemsetAsync(st, 0, sizeof(DevSmall), c->stream));
        CU(cudaMemcpyAsync(mats, h.data(), sizeof(u32) * h.size(), cudaMemcpyHostToDevice, c->stream));
        c->launches += launch_small(c->geo, c->m, nullptr, mats, st, 2, c->stream);
        DevSmall hs;
        CU(cudaMemcpyAsync(h.data(), mats, sizeof(u32) * h.size(), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaMemcpyAsync(&hs, st, sizeof(DevSmall), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        cudaFree(mats); cudaFree(st);
        for (int i = 0; i < n; i++)
                for (int j = 0; j < n; j++) winv[i * n + j] = h[(size_t)MAT_WINV * np * np + i * np + j];
        for (int j = 0; j < n; j++) d[j] = h[(size_t)MAT_D * np * np + j];
        if (npiv) *npiv = hs.npiv;
        return 0;
}

int blk_orthogonalize(blk_ctx *c, const uint32_t *v, uint32_t *tmp, uint32_t *p, const uint32_t *d,
                      const uint32_t *vtAv, const uint32_t *vtAAv, const uint32_t *winv, int64_t N,
                      const uint32_t *Av)
{
        if (!c || !v || !tmp || !p || !d || !vtAv || !vtAAv || !winv || !Av || N < 0)
                return fail("blk_orthogonalize: bad argument");
        if (c->is_group()) return blk_orthogonalize(c->members[0], v, tmp, p, d, vtAv, vtAAv, winv, N, Av);
        CU(cudaSetDevice(c->device));
        const int np = c->geo.np, n = c->geo.n;
        std::vector<u32> h((size_t)MAT_COUNT * np * np, 0);
        put_small(h, MAT_VTAV, vtAv, n, np);
        put_small(h, MAT_VTAAV, vtAAv, n, np);
        put_small(h, MAT_WINV, winv, n, np);
        for (int j = 0; j < n; j++) h[(size_t)MAT_D * np * np + j] = d[j];
        int64_t rows = N > 0 ? N : 1;
        u32 *mats = nullptr, *dv = nullptr, *da = nullptr, *dp = nullptr, *dvo = nullptr;
        CU(cudaMalloc(&mats, sizeof(u32) * mats_words(np)));
        CU(cudaMalloc(&dv, sizeof(u32) * (size_t)rows * np));
        CU(cudaMalloc(&dvo, sizeof(u32) * (size_t)rows * np));
        CU(cudaMalloc(&da, sizeof(u32) * (size_t)rows * np));
        CU(cudaMalloc(&dp, sizeof(u32) * (size_t)rows * np));
        CU(cudaMemcpyAsync(mats, h.data(), sizeof(u32) * h.size(), cudaMemcpyHostToDevice, c->stream));
        int rc = upload_rows(c, dv, v, N) || upload_rows(c, da, Av, N) || upload_rows(c, dp, p, N);
        if (!rc && N > 0) {
                c->launches += launch_small(c->geo, c->m, nullptr, mats, c->state, 3, c->stream);
                c->launches += launch_ortho(c->geo, c->m, N, dv, da, dp, dvo, dp, mats, c->state, 1, c->stream);
                rc = download_rows(c, tmp, dvo, N) || download_rows(c, p, dp, N);
                cudaError_t e = cudaGetLastError();
                if (!rc && e != cudaSuccess) rc = fail(std::string("blk_orthogonalize: ") + cudaGetErrorString(e));
        }
        cudaFree(mats); cudaFree(dv); cudaFree(dvo); cudaFree(da); cudaFree(dp);
        return rc;
}

// ---- measurement ---------------------------------------------------------------------------
int blk_set_profiling(blk_ctx *c, int32_t on)
{
        if (!c) return fail("null context");
        if (c->is_group()) {
                for (blk_ctx *mem : c->members) blk_set_profiling(mem, on);
                return 0;
        }
        c->profiling = on != 0;
        for (int i = 0; i < BLK_PH_COUNT; i++) { c->ph_ms[i] = 0; c->ph_launch[i] = 0; }
        return 0;
}

int blk_get_phase_times(blk_ctx *c, double ms[BLK_PH_COUNT], int64_t launches[BLK_PH_COUNT])
{
        if (!c) return fail("null context");
        if (c->is_group()) return blk_get_phase_times(c->members[0], ms, launches);
        for (int i = 0; i < BLK_PH_COUNT; i++) {
                if (ms) ms[i] = c->ph_ms[i];
                if (launches) launches[i] = c->ph_launch[i];
        }
        return 0;
}

int blk_time_spmv(blk_ctx *c, int32_t transpose, int32_t reps, double *ms_avg)
{
        if (!c || reps < 1 || !ms_avg) return fail("blk_time_spmv: bad argument");
        if (c->is_group()) {
                std::vector<double> ms(c->members.size(), 0.0);
                if (group_run(c, [&](blk_ctx *mem, int r) { return blk_time_spmv(mem, transpose, reps, &ms[(size_t)r]); })) return 1;
                *ms_avg = *std::max_element(ms.begin(), ms.end());        // the slowest shard is the product's time
                return 0;
        }
        CU(cudaSetDevice(c->device));
        const int np = c->geo.np;
        bool s1;
        SpOp *op = op_for(c, transpose, &s1);
        const u32 *x = s1 ? c->v : c->tmp;
        u32 *y = s1 ? c->tmp + (size_t)c->m0() * np : c->Av;
        if (c->mg_recur && s1) {          // keep the loop invariant (tmp = S1 v): time S1 on Av into the scratch block
                x = c->Av_full;
                y = c->U;
        }
        cudaEvent_t a, b;
        CU(cudaEventCreate(&a)); CU(cudaEventCreate(&b));
        c->launches += launch_spmv(*op, c->geo, c->m, x, y, nullptr, c->stream);    // warm-up
        CU(cudaEventRecord(a, c->stream));
        for (int i = 0; i < reps; i++) c->launches += launch_spmv(*op, c->geo, c->m, x, y, nullptr, c->stream);
        CU(cudaEventRecord(b, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, a, b));
        cudaEventDestroy(a); cudaEventDestroy(b);
        *ms_avg = (double)ms / reps;
        if (!c->mg_recur) c->tmp_is_spmv = false;
        return 0;
}

int64_t blk_kernel_launches(blk_ctx *c)
{
        if (!c) return 0;
        int64_t total = c->launches;
        for (blk_ctx *mem : c->members) total += mem->launches;
        return total;
}

int blk_get_info(blk_ctx *c, blk_info *info)
{
        if (!c || !info) return fail("blk_get_info: null argument");
        if (c->is_group()) {
                // the job as a whole: every row is local, sizes summed over the members
                if (blk_get_info(c->members[0], info)) return 1;
                for (size_t r = 1; r < c->members.size(); r++) {
                        blk_info one;
                        if (blk_get_info(c->members[r], &one)) return 1;
                        for (int i = 0; i < 2; i++) {
                                info->nnz_local[i] += one.nnz_local[i]; info->stored_local[i] += one.stored_local[i];
                                info->tiles[i] += one.tiles[i];
                        }
                        info->device_bytes += one.device_bytes;
                }
                info->local_N0 = 0; info->local_N1 = c->N; info->local_M0 = 0; info->local_M1 = c->Mc;
                return 0;
        }
        memset(info, 0, sizeof(*info));
        info->N = c->N; info->Mc = c->Mc;
        info->nrhs = c->nrhs;
        // (with relabelled rows on several GPUs: the HOST rows this rank moves in blk_set_state / blk_get_state_local)
        info->local_N0 = c->h0(); info->local_N1 = c->h1();
        info->local_M0 = c->m0(); info->local_M1 = c->m1();
        const SpOp *ops[2] = {&c->S1, &c->S2};
        for (int i = 0; i < 2; i++) {
                info->nnz_local[i] = ops[i]->nnz;
                info->stored_local[i] = ops[i]->stored;
                info->tiles[i] = ops[i]->ntiles;
                info->chunk_len[i] = ops[i]->Q;
        }
        info->n = c->geo.n; info->n_pad = c->geo.np; info->groups_per_warp = c->geo.G;
        info->device_bytes = (int64_t)(c->S1.bytes + c->S2.bytes + c->block_bytes);
        info->loop_mode = (c->coop && c->use_graph != 0) ? 1 : 0;
        info->bands[0] = (int32_t)c->S1.bands.size(); info->bands[1] = (int32_t)c->S2.bands.size();
        info->heavy_rows = c->S2.heavy_rows; info->heavy_bands = c->S2.heavy_bands;
        return 0;
}

}  // extern "C"
