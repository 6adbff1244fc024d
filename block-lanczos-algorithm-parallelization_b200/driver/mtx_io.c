/* mtx_io.c -- see mtx_io.h */
#define _POSIX_C_SOURCE 200809L
#include "mtx_io.h"
#include <ctype.h>
#include <err.h>
#include <pthread.h>
#include <unistd.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <sys/time.h>

static double now(void)
{
        struct timeval tv;
        gettimeofday(&tv, NULL);
        return tv.tv_sec + tv.tv_usec * 1e-6;
}

static char *slurp(const char *filename, size_t *len)
{
        FILE *f = fopen(filename, "rb");
        if (!f)
                err(1, "impossible d'ouvrir %s", filename);
        struct stat sb;
        if (fstat(fileno(f), &sb) != 0)
                err(1, "stat %s", filename);
        size_t size = (size_t)sb.st_size;
        char *buf = malloc(size + 1);
        if (!buf)
                err(1, "Cannot allocate %zu bytes for %s", size, filename);
        size_t got = 0;
        while (got < size) {
                size_t r = fread(buf + got, 1, size - got, f);
                if (r == 0)
                        break;
                got += r;
        }
        fclose(f);
        buf[got] = 0;
        *len = got;
        return buf;
}

/* next line starting at *pos; returns pointer and sets *linelen; advances *pos */
static const char *next_line(const char *buf, size_t len, size_t *pos, size_t *linelen)
{
        if (*pos >= len)
                return NULL;
        const char *s = buf + *pos;
        const char *e = memchr(s, '\n', len - *pos);
        size_t l = e ? (size_t)(e - s) : len - *pos;
        *pos += l + (e ? 1 : 0);
        *linelen = l;
        return s;
}

/* scan one optionally signed decimal integer, skipping leading white space */
static inline int scan_int(const char **pp, const char *end, long long *out)
{
        const char *p = *pp;
        while (p < end && (*p == ' ' || *p == '\t' || *p == '\n' || *p == '\r'))
                p++;
        if (p >= end)
                return 0;
        int neg = 0;
        if (*p == '-' || *p == '+') {
                neg = (*p == '-');
                p++;
        }
        if (p >= end || *p < '0' || *p > '9')
                return 0;
        long long v = 0;
        while (p < end && *p >= '0' && *p <= '9')
                v = v * 10 + (*p++ - '0');
        *out = neg ? -v : v;
        *pp = p;
        return 1;
}

static int ieq(const char *a, const char *b)
{
        for (; *a && *b; a++, b++)
                if (tolower((unsigned char)*a) != tolower((unsigned char)*b))
                        return 0;
        return *a == *b;
}

/* ---- parallel triplet parser -------------------------------------------------------------
 * The data section is a stream of white-space separated integers; entry k is integers 3k..3k+2
 * (exactly what nnz calls of fscanf("%d %d %d\n") consume, sequential/lanczos_modp.c:236-243).
 * The buffer is cut at white space into one segment per thread; pass 1 counts the integers that
 * start in each segment, a prefix sum gives every segment its first global integer index, pass 2
 * parses and stores each integer at (entry, field) = (index / 3, index % 3). */
struct parse_seg {
        const char *b, *e;
        long long ntok, first;          /* integers starting in [b,e); global index of the first one */
        long long bad;                  /* global index of the first malformed integer, or -1 */
        long long nz;
        uint64_t prime;
        int *Mi, *Mj;
        uint32_t *Mx;
};

static inline int is_space(char c) { return c == ' ' || c == '\n' || c == '\t' || c == '\r'; }

static void *seg_count(void *arg)
{
        struct parse_seg *s = arg;
        long long n = 0;
        int in = 0;
        for (const char *p = s->b; p < s->e; p++) {
                int sp = is_space(*p);
                n += (!sp && !in);
                in = !sp;
        }
        s->ntok = n;
        return NULL;
}

static void *seg_parse(void *arg)
{
        struct parse_seg *s = arg;
        const char *p = s->b;
        long long g = s->first, limit = 3 * s->nz;
        s->bad = -1;
        while (g < limit) {
                while (p < s->e && is_space(*p)) p++;
                if (p >= s->e) break;
                int neg = 0;
                if (*p == '-' || *p == '+') { neg = (*p == '-'); p++; }
                if (p >= s->e || *p < '0' || *p > '9') { s->bad = g; return NULL; }
                long long v = 0;
                while (p < s->e && *p >= '0' && *p <= '9') v = v * 10 + (*p++ - '0');
                if (p < s->e && !is_space(*p)) { s->bad = g; return NULL; }
                if (neg) v = -v;
                long long k = g / 3;
                switch (g % 3) {
                case 0: s->Mi[k] = (int)(v - 1); break;            /* MatrixMarket is 1-based */
                case 1: s->Mj[k] = (int)(v - 1); break;
                /* the reference reads "%d" into a u32 and then reduces: -k becomes 2^32-k (F9) */
                default: s->Mx[k] = (uint32_t)((uint64_t)(uint32_t)(int)v % s->prime); break;
                }
                g++;
        }
        return NULL;
}

static void parse_entries(const char *b, const char *e, long long nz, uint64_t prime, int *Mi, int *Mj, uint32_t *Mx)
{
        enum { MAXT = 64 };
        long ncpu = sysconf(_SC_NPROCESSORS_ONLN);
        const char *env = getenv("BLK_PARSE_THREADS");
        long T = env ? atol(env) : ncpu;
        size_t bytes = (size_t)(e - b);
        if (T > MAXT) T = MAXT;
        if ((size_t)T > bytes / (1u << 20) + 1) T = (long)(bytes / (1u << 20) + 1);      /* >= 1 MiB per thread */
        if (T < 1) T = 1;
        struct parse_seg seg[MAXT];
        pthread_t th[MAXT];
        const char *cut = b;
        for (long t = 0; t < T; t++) {
                const char *next = t == T - 1 ? e : b + bytes * (size_t)(t + 1) / (size_t)T;
                if (next < cut) next = cut;
                while (next < e && !is_space(*next)) next++;            /* never cut inside an integer */
                seg[t] = (struct parse_seg){cut, next, 0, 0, -1, nz, prime, Mi, Mj, Mx};
                cut = next;
        }
        for (long t = 0; t < T; t++)
                if (T == 1 || pthread_create(&th[t], NULL, seg_count, &seg[t]) != 0) { seg_count(&seg[t]); th[t] = 0; }
        for (long t = 0; t < T; t++)
                if (th[t]) pthread_join(th[t], NULL);
        long long total = 0;
        for (long t = 0; t < T; t++) { seg[t].first = total; total += seg[t].ntok; }
        for (long t = 0; t < T; t++)
                if (T == 1 || pthread_create(&th[t], NULL, seg_parse, &seg[t]) != 0) { seg_parse(&seg[t]); th[t] = 0; }
        for (long t = 0; t < T; t++)
                if (th[t]) pthread_join(th[t], NULL);
        long long bad = -1;
        for (long t = 0; t < T; t++)
                if (seg[t].bad >= 0 && (bad < 0 || seg[t].bad < bad)) bad = seg[t].bad;
        if (bad < 0 && total < 3 * nz) bad = total;                      /* file ends early */
        if (bad >= 0 && bad < 3 * nz)
                errx(1, "parse error entry %lld\n", bad / 3);
}

void mtx_load(struct coo_matrix *M, const char *filename, uint64_t prime)
{
        printf("Loading matrix from %s\n", filename);
        fflush(stdout);
        double t0 = now();
        size_t len, pos = 0, ll;
        char *buf = slurp(filename, &len);

        /* banner: %%MatrixMarket object format field symmetry */
        const char *line = next_line(buf, len, &pos, &ll);
        char banner[16] = "", object[64] = "", format[64] = "", field[64] = "", symm[64] = "";
        char first[512];
        if (!line)
                errx(1, "Could not process Matrix Market banner.\n");
        snprintf(first, sizeof(first), "%.*s", (int)(ll < 500 ? ll : 500), line);
        if (sscanf(first, "%15s %63s %63s %63s %63s", banner, object, format, field, symm) != 5 ||
            strcmp(banner, "%%MatrixMarket") != 0)
                errx(1, "Could not process Matrix Market banner.\n");
        if (!ieq(object, "matrix") || !ieq(format, "coordinate"))
                errx(1, "Matrix Market type: [%s %s %s %s] not supported (only sparse matrices are OK)",
                     object, format, field, symm);
        if (!ieq(symm, "general") || !ieq(field, "integer"))
                errx(1, "Matrix type [%s %s %s %s] not supported (only integer general are OK)",
                     object, format, field, symm);

        /* skip comments and blank lines up to the size line */
        long long nr = 0, nc = 0, nz = 0;
        for (;;) {
                line = next_line(buf, len, &pos, &ll);
                if (!line)
                        errx(1, "Cannot read matrix size");
                if (ll == 0 || line[0] == '%')
                        continue;
                const char *p = line, *e = line + ll;
                if (!scan_int(&p, e, &nr) || !scan_int(&p, e, &nc) || !scan_int(&p, e, &nz))
                        continue;        /* mmio keeps scanning until three numbers parse */
                break;
        }
        if (nr <= 0 || nc <= 0 || nz < 0 || nr > 0x7fffffff || nc > 0x7fffffff)
                errx(1, "Cannot read matrix size");
        fprintf(stderr, "  - [matrix coordinate integer general] %lld x %lld with %lld nz\n", nr, nc, nz);
        fprintf(stderr, "  - Allocating %.1f MByte\n", 1e-6 * (12.0 * nz));

        size_t cnt = nz > 0 ? (size_t)nz : 1;
        int *Mi = malloc(cnt * sizeof(*Mi));
        int *Mj = malloc(cnt * sizeof(*Mj));
        uint32_t *Mx = malloc(cnt * sizeof(*Mx));
        if (!Mi || !Mj || !Mx)
                err(1, "Cannot allocate sparse matrix");

        parse_entries(buf + pos, buf + len, nz, prime, Mi, Mj, Mx);
        double dt = now() - t0;
        printf("  - Read %s: %.1f MB in %.2fs (%.1f MB/s)\n", filename, len / 1048576., dt,
               len / 1048576. / (dt > 0 ? dt : 1e-9));
        free(buf);
        M->nrows = (int)nr; M->ncols = (int)nc; M->nnz = (long)nz;
        M->i = Mi; M->j = Mj; M->x = Mx;
}

uint32_t *mtx_load_array(const char *filename, uint64_t prime, int *rows, int *cols)
{
        size_t len, pos = 0, ll;
        char *buf = slurp(filename, &len);
        const char *line = next_line(buf, len, &pos, &ll);
        char banner[16] = "", object[64] = "", format[64] = "", field[64] = "", symm[64] = "";
        char first[512];
        if (!line)
                errx(1, "%s: could not process Matrix Market banner", filename);
        snprintf(first, sizeof(first), "%.*s", (int)(ll < 500 ? ll : 500), line);
        if (sscanf(first, "%15s %63s %63s %63s %63s", banner, object, format, field, symm) != 5 ||
            strcmp(banner, "%%MatrixMarket") != 0)
                errx(1, "%s: could not process Matrix Market banner", filename);
        if (!ieq(object, "matrix") || !ieq(format, "array") || !ieq(field, "integer") || !ieq(symm, "general"))
                errx(1, "%s: [%s %s %s %s] not supported (only matrix array integer general)", filename, object, format,
                     field, symm);
        long long nr = 0, nc = 0;
        for (;;) {
                line = next_line(buf, len, &pos, &ll);
                if (!line)
                        errx(1, "%s: cannot read the array size", filename);
                if (ll == 0 || line[0] == '%')
                        continue;
                const char *p = line, *e = line + ll;
                if (!scan_int(&p, e, &nr) || !scan_int(&p, e, &nc))
                        errx(1, "%s: cannot read the array size", filename);
                break;
        }
        if (nr <= 0 || nc <= 0 || nr > 0x7fffffff || nc > 0x7fffffff)
                errx(1, "%s: bad array size %lld x %lld", filename, nr, nc);
        uint32_t *x = malloc(sizeof(uint32_t) * (size_t)nr * (size_t)nc);
        if (!x)
                err(1, "cannot allocate %lld x %lld values for %s", nr, nc, filename);
        const char *p = buf + pos, *end = buf + len;
        long long val;
        for (long long col = 0; col < nc; col++)            /* column-major, like kernel_block_save */
                for (long long r = 0; r < nr; r++) {
                        if (!scan_int(&p, end, &val))
                                errx(1, "%s: expected %lld values, found fewer", filename, nr * nc);
                        x[r * nc + col] = (uint32_t)((uint64_t)(uint32_t)(int)val % prime);
                }
        while (p < end && is_space(*p))
                p++;
        if (p < end)
                errx(1, "%s: unexpected text after %lld values", filename, nr * nc);
        free(buf);
        *rows = (int)nr;
        *cols = (int)nc;
        return x;
}

void mtx_free(struct coo_matrix *M)
{
        free(M->i); free(M->j); free(M->x);
        M->i = M->j = NULL; M->x = NULL;
}

/* fast "%d\n" formatter for values below 2^31 */
static inline char *put_u32_line(char *w, uint32_t v)
{
        char tmp[12];
        int k = 0;
        int32_t s = (int32_t)v;                 /* the reference prints with %d */
        uint32_t a = s < 0 ? (uint32_t)(-(int64_t)s) : (uint32_t)s;
        if (s < 0)
                *w++ = '-';
        do {
                tmp[k++] = (char)('0' + a % 10);
                a /= 10;
        } while (a);
        while (k)
                *w++ = tmp[--k];
        *w++ = '\n';
        return w;
}

static void write_lines(FILE *f, const char *filename, long count, long stride, const uint32_t *v)
{
        enum { CHUNK = 1 << 16 };
        char *buf = malloc((size_t)CHUNK * 12);
        if (!buf)
                err(1, "cannot allocate output buffer");
        for (long base = 0; base < count; base += CHUNK) {
                long m = count - base < CHUNK ? count - base : CHUNK;
                char *w = buf;
                for (long t = 0; t < m; t++)
                        w = put_u32_line(w, v[(base + t) * stride]);
                if (fwrite(buf, 1, (size_t)(w - buf), f) != (size_t)(w - buf))
                        err(1, "cannot write %s", filename);
        }
        free(buf);
}

void kernel_block_save(const char *filename, int nrows, int n, const uint32_t *v)
{
        printf("Saving result in %s\n", filename);
        FILE *f = fopen(filename, "w");
        if (!f)
                err(1, "cannot open %s", filename);
        fprintf(f, "%%%%MatrixMarket matrix array integer general\n");
        fprintf(f, "%%block of left-kernel vector computed by lanczos_modp\n");
        fprintf(f, "%d %d\n", nrows, n);
        for (int col = 0; col < n; col++)           /* column-major, one value per line */
                write_lines(f, filename, nrows, n, v + col);
        if (fclose(f) != 0)
                err(1, "cannot write %s", filename);
}

void vector_write_tmp(const char *filename, long count, const uint32_t *v)
{
        char tmpname[4096];
        snprintf(tmpname, sizeof(tmpname), "%s.tmp", filename);
        FILE *f = fopen(tmpname, "w");
        if (!f)
                err(1, "cannot open %s", tmpname);
        printf("\t\t>> Making a snapshot of a vector in %s\n", filename);
        write_lines(f, tmpname, count, 1, v);
        if (fclose(f) != 0)
                err(1, "cannot write %s", tmpname);
}

void commit_tmp(const char *filename)
{
        char tmpname[4096];
        snprintf(tmpname, sizeof(tmpname), "%s.tmp", filename);
        if (rename(tmpname, filename) != 0)
                err(1, "cannot rename %s to %s", tmpname, filename);
}

void vector_save(const char *filename, long count, const uint32_t *v)
{
        vector_write_tmp(filename, count, v);
        commit_tmp(filename);
}

void vector_load(const char *filename, long count, uint32_t *v)
{
        size_t len;
        char *buf = slurp(filename, &len);
        const char *p = buf, *end = buf + len;
        long got = 0;
        long long val;
        while (scan_int(&p, end, &val)) {
                if (got >= count)
                        errx(1, "%s holds more than %ld values (matrix, --n or side differ from the checkpoint?)",
                             filename, count);
                v[got++] = (uint32_t)(int)val;
        }
        /* a checkpoint block is exactly block_size_pad lines (openMP/lanczos_modp.c:571-589): anything else is a
         * truncated or foreign file and must not be resumed from */
        while (p < end && (*p == ' ' || *p == '\t' || *p == '\r' || *p == '\n'))
                p++;
        if (p < end)
                errx(1, "%s: unexpected text after %ld values", filename, got);
        if (got != count)
                errx(1, "%s holds %ld values, expected %ld (truncated checkpoint, or matrix / --n / side differ)",
                     filename, got, count);
        free(buf);
}
