/* mtx_io.h -- MatrixMarket text I/O for the lanczos_modp driver.
 *
 * Accepts exactly what the reference's loader accepts (sparsematrix_mm_load,
 * sequential/lanczos_modp.c:199-263, through NIST mmio): a
 * "%%MatrixMarket matrix coordinate integer general" banner, comment lines,
 * a "rows cols nnz" size line and nnz "i j x" triplets (1-based).  Written from
 * scratch: one read of the whole file and a hand-rolled integer scanner
 * instead of fscanf per entry (SURVEY.md section 8(f)1).
 */
#ifndef BLK_MTX_IO_H
#define BLK_MTX_IO_H
#include <stdint.h>

struct coo_matrix {
        int nrows, ncols;
        long nnz;
        int *i, *j;          /* 0-based */
        uint32_t *x;         /* value mod prime, with the reference's %d-into-u32 semantics */
};

/* errx(1, ...) on any failure, like the reference */
void mtx_load(struct coo_matrix *M, const char *filename, uint64_t prime);
void mtx_free(struct coo_matrix *M);

/* dense "array integer general" block of rows x cols (the format kernel_block_save writes, column-major values),
 * returned row-major (rows x cols, malloc'ed), values reduced mod prime with mtx_load's semantics (-k is 2^32 - k).
 * errx(1, ...) on any failure. */
uint32_t *mtx_load_array(const char *filename, uint64_t prime, int *rows, int *cols);

/* kernel block, save_vector_block format (sequential/lanczos_modp.c:673-686):
 * dense "array integer general", "N n", then column-major "%d\n" */
void kernel_block_save(const char *filename, int nrows, int n, const uint32_t *v);

/* checkpoint vectors (openMP/lanczos_modp.c:573-589, 611-635): `count` lines of "%d\n".
 * Saving goes through a temporary file + rename so a crash never leaves a torn file. */
void vector_save(const char *filename, long count, const uint32_t *v);
/* the two halves of vector_save: write "<filename>.tmp", then rename it over <filename> */
void vector_write_tmp(const char *filename, long count, const uint32_t *v);
void commit_tmp(const char *filename);
void vector_load(const char *filename, long count, uint32_t *v);
#endif
