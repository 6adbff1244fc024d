/*
 * lanczos_modp -- host driver of the B200 block-Lanczos mod-p solver.
 *
 * Same command line, same input/output files and the same console report as
 * the reference program (sequential/lanczos_modp.c, plus the checkpoint
 * options of openMP/lanczos_modp.c:187-257), so that checker_modp validates
 * the result unchanged.  Everything inside the iteration
 * (sequential/lanczos_modp.c:635-656) runs on the GPU through the C ABI of
 * include/blk_lanczos.h; there is no CPU fallback.  This file only parses
 * options, loads the matrix, draws the start block with the reference's
 * generator, reports progress, and reads/writes the text files.
 *
 * USAGE:
 *      $ ./lanczos_modp --prime 65537 --n 4 --matrix random_small.mtx
 *      $ ./lanczos_modp --prime 65537 --n 16 --matrix M.mtx --rhs B.mtx --output-file X.mtx [--right]
 *      $ ./lanczos_modp --prime 2 --n 64 --matrix M.mtx --prune --kernel-basis --output-file K.mtx
 *
 * Deviations from the reference, all documented in DESIGN.md:
 *   - p may be as large as 2^31-1 (the reference stops at 2^30-35);
 *   - n <= 64;
 *   - checkpoint files are formatted into *.tmp and renamed into place together, with a commit
 *     marker (checkpoint.commit) that --load-checkpoint verifies;
 *   - BLK_GPUS=G in the environment shards the job over G GPUs of the box (same files, same output);
 *   - --kernel-basis (new, needs --output-file): after the loop, the final Gaussian elimination of block
 *     Lanczos extracts the independent kernel vectors inside span(v) (blk_kernel_basis); the output file then
 *     holds those k columns instead of the n columns of v.  Without it the output is the reference's;
 *   - --rhs FILE (new, needs --output-file): solve M*X = B (--right) or X*M = B (--left) for the r <= n columns
 *     of the MatrixMarket array B (Mc x r, the format of the output file).  The loop runs on the augmented
 *     matrix [M | -B] (resp. [M ; -B^T]); blk_solve then extracts the solutions and the output file holds the
 *     N x r block X.  Exit status 1 and no file when some right-hand side is not solved;
 *   - --prune (new): empty and singleton constraints are removed on the device before the loop
 *     (blk_create_pruned); the loop, the final check and --kernel-basis run on the smaller matrix M', and the
 *     output file is lifted back to the N rows of M (zeros on the removed unknowns).  Exit status 1 and no file
 *     when every constraint is removed;
 *   - the GPU runs iterations in batches, so progress is reported per batch.
 */
#define _POSIX_C_SOURCE 200809L
#include <err.h>
#include <getopt.h>
#include <inttypes.h>
#include <pthread.h>
#include <stdbool.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/time.h>
#include <time.h>

#include "blk_lanczos.h"
#include "mtx_io.h"

struct options {
        const char *matrix, *output;
        uint64_t prime;
        int n;
        bool right;
        int stop_after;
        bool checkpoint, resume, kernel_basis, prune;
        const char *rhs;
        double checkpoint_every;
        int device;
};

static double wall(void)
{
        struct timeval tv;
        gettimeofday(&tv, NULL);
        return tv.tv_sec + tv.tv_usec * 1e-6;
}

static void usage(const char *argv0)
{
        printf("%s [OPTIONS]\n\n", argv0);
        printf("Options:\n");
        printf("--matrix FILENAME           MatrixMarket file containing the sparse matrix\n");
        printf("--prime P                   compute modulo P\n");
        printf("--n N                       blocking factor [default 1]\n");
        printf("--output-file FILENAME      store the block of kernel vectors\n");
        printf("--right                     compute right kernel vectors\n");
        printf("--left                      compute left kernel vectors [default]\n");
        printf("--stop-after N              stop the algorithm after N iterations\n");
        printf("--checkpoint cp             enable checkpointing every cp seconds [default cp = 60 s]\n");
        printf("--load-checkpoint           load vectors from checkpointing files\n");
        printf("--kernel-basis              store only independent kernel vectors (needs --output-file)\n");
        printf("--rhs FILENAME              solve M*X = B (X*M = B with --left) for the array B (needs --output-file)\n");
        printf("--prune                     remove empty and singleton constraints before the loop\n");
        printf("\n");
        printf("The --matrix and --prime arguments are required\n");
        printf("The --stop-after and --output-file arguments mutually exclusive\n");
        exit(0);
}

static void parse_options(struct options *o, int argc, char **argv)
{
        static const struct option longopts[] = {
                {"matrix", required_argument, NULL, 'm'},
                {"prime", required_argument, NULL, 'p'},
                {"n", required_argument, NULL, 'n'},
                {"output-file", required_argument, NULL, 'o'},
                {"right", no_argument, NULL, 'r'},
                {"left", no_argument, NULL, 'l'},
                {"stop-after", required_argument, NULL, 's'},
                {"checkpoint", optional_argument, NULL, 'c'},
                {"load-checkpoint", no_argument, NULL, 'L'},
                {"kernel-basis", no_argument, NULL, 'K'},
                {"rhs", required_argument, NULL, 'B'},
                {"prune", no_argument, NULL, 'P'},
                {NULL, 0, NULL, 0}};
        memset(o, 0, sizeof(*o));
        o->n = 1;
        o->stop_after = -1;
        o->checkpoint_every = 60;
        const char *dev = getenv("BLK_DEVICE");
        o->device = dev ? atoi(dev) : 0;
        int ch;
        while ((ch = getopt_long(argc, argv, "", longopts, NULL)) != -1) {
                switch (ch) {
                case 'm': o->matrix = optarg; break;
                case 'n': o->n = atoi(optarg); break;
                case 'p': o->prime = (uint64_t)atoll(optarg); break;
                case 'o': o->output = optarg; break;
                case 'r': o->right = true; break;
                case 'l': o->right = false; break;
                case 's': o->stop_after = (int)atoll(optarg); break;
                case 'c':
                        o->checkpoint = true;
                        /* "--checkpoint 30" as well as "--checkpoint=30" (openMP/lanczos_modp.c:225-236) */
                        if (!optarg && optind < argc && argv[optind][0] != '-')
                                optarg = argv[optind++];
                        if (optarg)
                                o->checkpoint_every = atoi(optarg);
                        break;
                case 'L': o->resume = true; break;
                case 'K': o->kernel_basis = true; break;
                case 'B': o->rhs = optarg; break;
                case 'P': o->prune = true; break;
                default: errx(1, "Unknown option\n");
                }
        }
        if (!o->matrix || o->prime == 0)
                usage(argv[0]);
        if (o->rhs) {
                if (!o->output)
                        errx(1, "usage: --rhs needs --output-file");
                if (o->kernel_basis || o->stop_after > 0 || o->checkpoint || o->resume)
                        errx(1, "usage: --rhs cannot be combined with --kernel-basis, --stop-after, --checkpoint or --load-checkpoint");
        }
        if (o->prune && (o->rhs || o->checkpoint || o->resume))
                errx(1, "usage: --prune cannot be combined with --rhs, --checkpoint or --load-checkpoint");
        if (o->output && o->stop_after > 0)
                usage(argv[0]);
        if (o->kernel_basis && !o->output)
                usage(argv[0]);
        if (o->prime > 0x7fffffffull)
                errx(1, "p is capped at 2**31 - 1.");
        if (o->n < 1 || o->n > BLK_MAX_N)
                errx(1, "the blocking factor must be between 1 and %d", BLK_MAX_N);
}

/* xoshiro256+ with the reference's fixed seed (sequential/lanczos_modp.c:64-87): the start
 * block must be the same sequence, drawn row-major on the host (:624-625). */
static uint64_t rng_s[4] = {0x1415926535ull, 0x8979323846ull, 0x2643383279ull, 0x5028841971ull};

static inline uint64_t rol64(uint64_t w, int k) { return (w << k) | (w >> (64 - k)); }

static uint64_t rng_next(void)
{
        uint64_t r = rol64(rng_s[0] + rng_s[3], 23) + rng_s[0];
        uint64_t t = rng_s[1] << 17;
        rng_s[2] ^= rng_s[0]; rng_s[3] ^= rng_s[1]; rng_s[1] ^= rng_s[2]; rng_s[0] ^= rng_s[3];
        rng_s[2] ^= t;
        rng_s[3] = rol64(rng_s[3], 45);
        return r;
}

/* at most six characters, like the reference's human_format */
static void human(char *dst, size_t cap, double x)
{
        static const char *suffix[] = {"", "K", "M", "G", "T", "P"};
        int k = 0;
        if (x < 1000) {
                snprintf(dst, cap, "%.0f", x);
                return;
        }
        while (x >= 1000 && k < 5) {
                x /= 1000;
                k++;
        }
        snprintf(dst, cap, "%.1f%s", x, suffix[k]);
}

struct progress {
        double start, last_print, extra;
        bool announced;
        int expected_total;
};

static void report(struct progress *pg, int n_iterations)
{
        double elapsed = wall() - pg->start + pg->extra;
        if (elapsed - pg->last_print < 1 || n_iterations == 0)
                return;
        pg->last_print = elapsed;
        double per_it = elapsed / n_iterations;
        double total = pg->expected_total * per_it;
        time_t end = (time_t)(pg->start - pg->extra + total);
        if (!pg->announced) {
                double rest = total;
                int d = (int)(rest / 86400); rest -= 86400.0 * d;
                int h = (int)(rest / 3600);  rest -= 3600.0 * h;
                int mi = (int)(rest / 60);   rest -= 60.0 * mi;
                printf("    - Expected duration : ");
                if (d > 0) printf("%d j ", d);
                if (h > 0) printf("%d h ", h);
                if (mi > 0) printf("%d min ", mi);
                printf("%d s\n", (int)rest);
                pg->announced = true;
        }
        char eta[32];
        ctime_r(&end, eta);
        eta[strcspn(eta, "\n")] = 0;
        printf("\r    - iteration %d / %d. %.3fs per iteration. ETA: %s", n_iterations, pg->expected_total,
               per_it, eta);
        fflush(stdout);
}

#define GPU(call)                                                                                  \
        do {                                                                                       \
                if ((call) != 0)                                                                   \
                        errx(1, "%s", blk_last_error());                                           \
        } while (0)

/* Checkpoints (openMP/lanczos_modp.c:1013-1022): the four blocks come back from the GPU in one
 * synchronous blk_get_state into a private set of host buffers; formatting and writing the text
 * files (the slow part: 4 * block_size_pad lines) then runs on a writer thread while the GPU
 * already iterates again.  A new snapshot (or program exit) first joins the previous writer. */
struct snapshot {
        long pad;
        int n_iterations;
        double t_start, t_now;
        uint32_t *blk[4];
        pthread_t thread;
        bool running;
};

/* "checkpoint.commit" -- a sidecar next to the reference's five files: "pending K" while the files of
 * snapshot K are being renamed into place, "complete K" afterwards.  --load-checkpoint refuses a set that
 * is not marked complete for the iteration verbosity.txt names (a crash between two renames would otherwise
 * resume from v of one snapshot and p of another).  Checkpoints written by the reference program have no
 * sidecar and are accepted as they are. */
static void write_commit_marker(const char *state, int n_iterations)
{
        FILE *f = fopen("checkpoint.commit.tmp", "w");
        if (!f)
                err(1, "cannot open %s", "checkpoint.commit");
        fprintf(f, "%s %d\n", state, n_iterations);
        if (fclose(f) != 0 || rename("checkpoint.commit.tmp", "checkpoint.commit") != 0)
                err(1, "cannot write %s", "checkpoint.commit");
}

static void *snapshot_writer(void *arg)
{
        struct snapshot *s = arg;
        static const char *names[4] = {"v.txt", "tmp.txt", "Av.txt", "p.txt"};
        /* all five files are formatted into *.tmp first (the slow part) ... */
        for (int k = 0; k < 4; k++)
                vector_write_tmp(names[k], s->pad, s->blk[k]);
        /* verbosity.txt: n_iterations, start, now (openMP/lanczos_modp.c:591-609) */
        FILE *f = fopen("verbosity.txt.tmp", "w");
        if (!f)
                err(1, "cannot open %s", "verbosity.txt");
        printf("\t\t>> Saving verbosity engine infos in %s\n", "verbosity.txt");
        fprintf(f, "%d\n%f\n%f\n", s->n_iterations, s->t_start, s->t_now);
        if (fclose(f) != 0)
                err(1, "cannot write verbosity.txt");
        /* ... and renamed into place together, verbosity.txt last */
        write_commit_marker("pending", s->n_iterations);
        for (int k = 0; k < 4; k++)
                commit_tmp(names[k]);
        commit_tmp("verbosity.txt");
        write_commit_marker("complete", s->n_iterations);
        return NULL;
}

static void snapshot_join(struct snapshot *s)
{
        if (s->running) {
                pthread_join(s->thread, NULL);
                s->running = false;
        }
}

static void write_checkpoint(blk_ctx *ctx, struct snapshot *s, long pad, int n_iterations, const struct progress *pg)
{
        snapshot_join(s);
        if (!s->blk[0]) {
                for (int k = 0; k < 4; k++) {
                        s->blk[k] = malloc(sizeof(uint32_t) * (size_t)pad);
                        if (!s->blk[k])
                                errx(1, "impossible d'allouer les blocs de vecteur");
                }
        }
        GPU(blk_get_state(ctx, s->blk[0], s->blk[1], s->blk[2], s->blk[3]));
        printf("\n");
        s->pad = pad;
        s->n_iterations = n_iterations;
        s->t_start = pg->start - pg->extra;
        s->t_now = wall();
        if (pthread_create(&s->thread, NULL, snapshot_writer, s) != 0)
                snapshot_writer(s);                      /* no thread: write synchronously */
        else
                s->running = true;
}

static int read_checkpoint_info(double *extra)
{
        FILE *f = fopen("verbosity.txt", "r");
        if (!f)
                err(1, "cannot open %s", "verbosity.txt");
        int it = 0;
        double a = 0, b = 0;
        if (fscanf(f, "%d %lf %lf", &it, &a, &b) != 3)
                errx(1, "verbosity.txt is malformed");
        fclose(f);
        *extra = (double)((int)b - (int)a);     /* the reference truncates both to int (:645-673) */
        f = fopen("checkpoint.commit", "r");
        if (f) {
                char state[32] = "";
                int marked = -1;
                if (fscanf(f, "%31s %d", state, &marked) != 2 || strcmp(state, "complete") != 0 || marked != it)
                        errx(1, "the checkpoint files are not one complete snapshot (checkpoint.commit: \"%s %d\", "
                                "verbosity.txt: iteration %d); refusing to resume", state, marked, it);
                fclose(f);
        }
        return it;
}

/* ---- multi-GPU: BLK_GPUS=G in the environment runs the job on G GPUs of this box (devices BLK_DEVICE ...),
 * all driven by this one process through a single context (blk_params.rank = BLK_RANK_ALL) -- the counterpart
 * of `mpirun -np G` for the reference's MPI build (mpi/lanczos_modp.c:1829-1863).  No new option: the command
 * line stays the reference's. */
static int gpus_from_env(void)
{
        const char *e = getenv("BLK_GPUS");
        if (!e || !e[0])
                return 1;
        int g = atoi(e);
        if (g < 1 || g > 64)
                errx(1, "BLK_GPUS must be a number of GPUs between 1 and 64");
        return g;
}

/* The N x w block x (stride w) as the file of the original matrix: without --prune (kept == NULL) as it is, else
 * lifted to its N_orig rows, zeros on the removed unknowns */
static void save_lifted(const char *path, long N, long N_orig, int w, const uint32_t *x, const int32_t *kept)
{
        if (!kept) {
                kernel_block_save(path, (int)N, w, x);
                return;
        }
        uint32_t *big = calloc((size_t)N_orig * (size_t)w, sizeof(*big));
        if (!big)
                errx(1, "cannot allocate the lifted block");
        for (long r = 0; r < N; r++)
                memcpy(big + (size_t)kept[r] * w, x + (size_t)r * w, sizeof(*big) * (size_t)w);
        kernel_block_save(path, (int)N_orig, w, big);
        free(big);
}

int main(int argc, char **argv)
{
        struct options o;
        parse_options(&o, argc, argv);

        struct coo_matrix M;
        mtx_load(&M, o.matrix, o.prime);

        const int n = o.n;
        /* --rhs: the Mc x r block B; the Lanczos vectors of the augmented matrix have N + r rows */
        int nrhs = 0;
        uint32_t *B = NULL;
        if (o.rhs) {
                int brows = 0;
                B = mtx_load_array(o.rhs, o.prime, &brows, &nrhs);
                const long want = o.right ? M.nrows : M.ncols;
                if (brows != want)
                        errx(1, "%s has %d rows, expected %ld (%s of the matrix)", o.rhs, brows, want, o.right ? "rows" : "columns");
                if (nrhs > n)
                        errx(1, "%s has %d right-hand sides, more than the blocking factor n = %d", o.rhs, nrhs, n);
        }
        int anrows = M.nrows + (o.right ? 0 : nrhs), ancols = M.ncols + (o.right ? nrhs : 0);
        const long orig_N = o.right ? M.ncols : M.nrows, orig_Mc = o.right ? M.nrows : M.ncols, orig_nnz = M.nnz;

        blk_params prm;
        memset(&prm, 0, sizeof(prm));
        prm.abi_version = BLK_ABI_VERSION;
        prm.nrows = M.nrows; prm.ncols = M.ncols; prm.nnz = M.nnz;
        prm.Mi = M.i; prm.Mj = M.j; prm.Mx = M.x;
        prm.n = n; prm.prime = (uint32_t)o.prime; prm.right_kernel = o.right;
        const int gpus = gpus_from_env();
        prm.device = o.device; prm.use_graph = -1;
        prm.world = gpus; prm.rank = gpus > 1 ? BLK_RANK_ALL : 0;
        blk_ctx *ctx = NULL;
        double t_build = wall();
        /* --prune: the context of M' comes first, its sizes are those of the loop */
        int64_t pst[BLK_PR_COUNT] = {0};
        int32_t *kept = NULL;                                /* original indices of the kept unknowns */
        printf("Block Lanczos\n");
        if (o.prune) {
                GPU(blk_create_pruned(&ctx, &prm, pst));
                printf("  - Prune: kept %" PRId64 " of %ld unknowns (%" PRId64 " free), %" PRId64 " of %ld constraints, "
                       "%" PRId64 " of %ld entries in %" PRId64 " rounds, %.2f s\n", pst[BLK_PR_N], orig_N, pst[BLK_PR_FREE],
                       pst[BLK_PR_MC], orig_Mc, pst[BLK_PR_NNZ], orig_nnz, pst[BLK_PR_ROUNDS], wall() - t_build);
                anrows = (int)(o.right ? pst[BLK_PR_MC] : pst[BLK_PR_N]);
                ancols = (int)(o.right ? pst[BLK_PR_N] : pst[BLK_PR_MC]);
                kept = malloc(sizeof(*kept) * (size_t)pst[BLK_PR_N]);
                if (!kept)
                        errx(1, "cannot allocate the index map");
                GPU(blk_pruned_index(ctx, kept, NULL));
        }
        const long N = o.right ? ancols : anrows;            /* length of the Lanczos vectors */
        const long Mc = o.right ? anrows : ancols;
        const long N0 = N - nrhs;                            /* the unknowns of the system */
        const long pad = (long)blk_block_pad(anrows, ancols, n, o.right);

        char hs[16];
        human(hs, sizeof(hs), 4.0 * sizeof(int) * pad);
        printf("  - Extra storage needed: %sB\n", hs);

        uint32_t *v = calloc((size_t)pad, sizeof(*v));
        uint32_t *tmp = calloc((size_t)pad, sizeof(*tmp));
        uint32_t *Av = calloc((size_t)pad, sizeof(*Av));
        uint32_t *p = calloc((size_t)pad, sizeof(*p));
        if (!v || !tmp || !Av || !p)
                errx(1, "impossible d'allouer les blocs de vecteur");

        if (!o.prune)
                t_build = wall();
        if (o.rhs)
                GPU(blk_create_system(&ctx, &prm, B, nrhs, 0));
        else if (!o.prune)
                GPU(blk_create(&ctx, &prm));
        free(B);
        if (gpus > 1)
                printf("  - Matrix resident on GPUs %d-%d (row blocks) in %.2fs\n", o.device, o.device + gpus - 1, wall() - t_build);
        else
                printf("  - Matrix resident on GPU %d in %.2fs\n", o.device, wall() - t_build);
        mtx_free(&M);                                    /* the device owns the matrix now */

        struct progress pg = {0};
        int n_iterations = 0;
        if (o.resume) {
                vector_load("v.txt", pad, v);
                vector_load("p.txt", pad, p);
                n_iterations = read_checkpoint_info(&pg.extra);
        } else {
                for (long t = 0; t < N * n; t++)
                        v[t] = (uint32_t)(rng_next() % o.prime);
        }
        GPU(blk_set_state(ctx, v, o.resume ? p : NULL, n_iterations));

        pg.expected_total = 1 + (int)(Mc / n);
        human(hs, sizeof(hs), (double)(pg.expected_total - (o.resume ? n_iterations : 0)));
        printf("  - Expecting %s iterations\n", hs);

        printf("  - Main loop\n");
        pg.start = wall();
        double last_checkpoint = wall();
        struct snapshot snap;
        memset(&snap, 0, sizeof(snap));
        int stopped = 0;
        int batch = 1;
        while (!stopped) {
                if (o.stop_after > 0 && n_iterations >= o.stop_after)
                        break;
                int todo = batch;
                if (o.stop_after > 0 && todo > o.stop_after - n_iterations)
                        todo = o.stop_after - n_iterations;
                if (o.checkpoint && o.checkpoint_every <= 0)
                        todo = 1;                        /* --checkpoint 0: snapshot after every iteration */
                double t0 = wall();
                int before = n_iterations;
                GPU(blk_iterate(ctx, todo, &n_iterations, &stopped));
                double dt = wall() - t0;
                /* size batches to roughly a quarter of a second so that progress and checkpoint
                 * timers keep their one-second resolution */
                if (n_iterations > before) {
                        double per = dt / (n_iterations - before);
                        double want = 0.25 / (per > 1e-9 ? per : 1e-9);
                        batch = want > 65536 ? 65536 : (want < 1 ? 1 : (int)want);
                }
                report(&pg, n_iterations);
                if (o.checkpoint && !stopped && n_iterations > before &&
                    wall() - last_checkpoint >= o.checkpoint_every) {
                        write_checkpoint(ctx, &snap, pad, n_iterations, &pg);
                        last_checkpoint = wall();
                }
        }
        snapshot_join(&snap);
        printf("\n");

        GPU(blk_get_state(ctx, v, NULL, NULL, NULL));
        if (o.stop_after < 0) {
                /* final_check, sequential/lanczos_modp.c:560-582, evaluated on the device */
                int32_t nonzero = 0, annihilated = 0;
                GPU(blk_final_check(ctx, &nonzero, &annihilated));
                printf("Final check:\n");
                printf(nonzero ? "  - OK:    v != 0\n" : "  - KO:    v == 0\n");
                printf(annihilated ? "  - OK: vt*M == 0\n" : "  - KO: vt*M != 0\n");
        }
        printf("  - Terminated in %.1fs after %d iterations\n", wall() - pg.start, n_iterations);

        if (o.output && o.rhs) {
                /* the solutions inside span(v), checked on the device as the kernel block (x_j ; e_j) of the
                 * augmented matrix */
                uint32_t *x = calloc((size_t)N0 * (size_t)nrhs, sizeof(*x));
                int32_t *found = calloc((size_t)nrhs, sizeof(*found));
                if (!x || !found)
                        errx(1, "cannot allocate the solution block");
                GPU(blk_solve(ctx, x, found));
                int solved = 0;
                for (int j = 0; j < nrhs; j++)
                        solved += found[j] != 0;
                printf("  - Solve: %d of %d right-hand sides solved\n", solved, nrhs);
                if (solved > 0) {
                        int32_t ok = 0;
                        memset(tmp, 0, sizeof(*tmp) * (size_t)pad);      /* (N + r) x n, stride n */
                        for (int j = 0; j < nrhs; j++) {
                                if (!found[j])
                                        continue;
                                for (long r = 0; r < N0; r++)
                                        tmp[r * n + j] = x[r * nrhs + j];
                                tmp[(N0 + j) * n + j] = 1;
                        }
                        GPU(blk_check_kernel_block(ctx, tmp, &ok));
                        if (o.right)
                                printf(ok ? "  - OK: M*X == B\n" : "  - KO: M*X != B\n");
                        else
                                printf(ok ? "  - OK: X*M == B\n" : "  - KO: X*M != B\n");
                }
                if (solved < nrhs) {
                        char list[256] = "";
                        size_t at = 0;
                        for (int j = 0; j < nrhs && at < sizeof(list) - 16; j++)
                                if (!found[j])
                                        at += (size_t)snprintf(list + at, sizeof(list) - at, "%s%d", at ? ", " : "", j + 1);
                        errx(1, "no solution in the final block for right-hand side(s) %s: the system may be inconsistent, "
                                "or the block did not reach a solution; nothing saved", list);
                }
                kernel_block_save(o.output, (int)N0, nrhs, x);
                free(x); free(found);
        } else if (o.output && o.kernel_basis) {
                /* the kernel vectors inside span(v): k independent columns, checked like checker_modp would */
                int32_t k = 0, ok = 0;
                GPU(blk_kernel_basis(ctx, tmp, &k));
                printf("  - Kernel basis: %d independent vectors\n", (int)k);
                if (k == 0)
                        errx(1, "no kernel vector in the final block: nothing to save");
                GPU(blk_check_kernel_block(ctx, tmp, &ok));
                printf(ok ? "  - OK: kernel basis * M == 0\n" : "  - KO: kernel basis * M != 0\n");
                for (long r = 0; r < N; r++)                 /* N x n, stride n -> N x k, stride k */
                        for (int j = 0; j < k; j++)
                                Av[r * k + j] = tmp[r * n + j];
                save_lifted(o.output, N, orig_N, (int)k, Av, kept);
        } else if (o.output)
                save_lifted(o.output, N, orig_N, n, v, kept);
        else
                printf("Not saving result (no --output given)\n");
        blk_destroy(ctx);
        free(v); free(tmp); free(Av); free(p); free(kept);
        return EXIT_SUCCESS;
}
