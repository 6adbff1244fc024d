/*
 * prune_oracle.c -- sequential CPU restatement of the pruning of DESIGN.md section 14 (blk_create_pruned).
 * TEST INFRASTRUCTURE: compiled on first use by tests/prune_oracle.py.
 *
 * Unknowns are the rows of M (--left) or its columns (--right), constraints the other dimension.  A triplet counts
 * when x mod p != 0; duplicates are not merged.  Instead of the synchronous rounds of the definition this file runs
 * a worklist: a constraint enters the queue with level L + 1 when the removal of a level-L unknown leaves it with a
 * count <= 1 (level 1: the count is <= 1 from the start), and a removed constraint's lone unknown is removed with the
 * constraint's level.  The levels are the BFS levels of the fixpoint, so `rounds` is the largest level.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* returns 0, or -1 when an allocation fails / an index is out of range.
 * ukeep[N], ckeep[Mc]: 1 for a kept unknown / constraint.  oi/oj/ox (capacity nnz): M', renumbered, original order and
 * orientation, value x mod p.  stats: N', Mc', nnz', free unknowns (kept, no triplet in M'), rounds. */
int pro_prune(int nrows, int ncols, long nnz, const int *Mi, const int *Mj, const uint32_t *Mx, uint64_t p, int right,
              int *ukeep, int *ckeep, long *stats, int *oi, int *oj, uint32_t *ox)
{
        const long N = right ? ncols : nrows, Mc = right ? nrows : ncols;
        const int *iu = right ? Mj : Mi, *ic = right ? Mi : Mj;
        long *cnt = calloc((size_t)Mc + 1, sizeof(long));
        long *cstart = calloc((size_t)Mc + 2, sizeof(long));
        long *ustart = calloc((size_t)N + 2, sizeof(long));
        long *by_c = malloc(sizeof(long) * ((size_t)nnz + 1));    /* counting triplets grouped by constraint */
        long *by_u = malloc(sizeof(long) * ((size_t)nnz + 1));    /* ... by unknown */
        long *level = calloc((size_t)Mc + 1, sizeof(long));       /* 0: not queued */
        long *queue = malloc(sizeof(long) * ((size_t)Mc + 1));
        long *pos = malloc(sizeof(long) * ((size_t)(N > Mc ? N : Mc) + 1));
        long *unew = malloc(sizeof(long) * ((size_t)N + 1)), *cnew = malloc(sizeof(long) * ((size_t)Mc + 1));
        char *used = calloc((size_t)N + 1, 1);
        int rc = -1;
        if (!cnt || !cstart || !ustart || !by_c || !by_u || !level || !queue || !pos || !unew || !cnew || !used)
                goto out;
        for (long s = 0; s < nnz; s++)
                if (iu[s] < 0 || iu[s] >= N || ic[s] < 0 || ic[s] >= Mc)
                        goto out;
        for (long u = 0; u < N; u++) ukeep[u] = 1;
        for (long c = 0; c < Mc; c++) ckeep[c] = 1;
        for (long s = 0; s < nnz; s++) {
                if (Mx[s] % p == 0)
                        continue;
                cnt[ic[s]]++;
                cstart[ic[s] + 1]++;
                ustart[iu[s] + 1]++;
        }
        for (long c = 0; c < Mc; c++) cstart[c + 1] += cstart[c];
        for (long u = 0; u < N; u++) ustart[u + 1] += ustart[u];
        memcpy(pos, cstart, sizeof(long) * (size_t)Mc);
        for (long s = 0; s < nnz; s++)
                if (Mx[s] % p != 0) by_c[pos[ic[s]]++] = s;
        memcpy(pos, ustart, sizeof(long) * (size_t)N);
        for (long s = 0; s < nnz; s++)
                if (Mx[s] % p != 0) by_u[pos[iu[s]]++] = s;

        long head = 0, tail = 0, rounds = 0;
        for (long c = 0; c < Mc; c++)
                if (cnt[c] <= 1) {
                        level[c] = 1;
                        queue[tail++] = c;
                }
        while (head < tail) {
                const long c = queue[head++], L = level[c];
                if (L > rounds) rounds = L;
                ckeep[c] = 0;
                if (cnt[c] != 1)
                        continue;
                long u = -1;                      /* the one counting triplet of c on a kept unknown */
                for (long t = cstart[c]; t < cstart[c + 1]; t++)
                        if (ukeep[iu[by_c[t]]]) { u = iu[by_c[t]]; break; }
                ukeep[u] = 0;
                for (long t = ustart[u]; t < ustart[u + 1]; t++) {
                        const long d = ic[by_u[t]];
                        cnt[d]--;
                        if (ckeep[d] && !level[d] && cnt[d] <= 1) {
                                level[d] = L + 1;
                                queue[tail++] = d;
                        }
                }
        }

        long n1 = 0, m1 = 0, z = 0;
        for (long u = 0; u < N; u++) unew[u] = ukeep[u] ? n1++ : -1;
        for (long c = 0; c < Mc; c++) cnew[c] = ckeep[c] ? m1++ : -1;
        for (long s = 0; s < nnz; s++) {
                if (Mx[s] % p == 0 || !ukeep[iu[s]] || !ckeep[ic[s]])
                        continue;
                (right ? oj : oi)[z] = (int)unew[iu[s]];
                (right ? oi : oj)[z] = (int)cnew[ic[s]];
                ox[z] = (uint32_t)(Mx[s] % p);
                used[unew[iu[s]]] = 1;
                z++;
        }
        long nfree = 0;
        for (long u = 0; u < n1; u++) nfree += !used[u];
        stats[0] = n1; stats[1] = m1; stats[2] = z; stats[3] = nfree; stats[4] = rounds;
        rc = 0;
out:
        free(cnt); free(cstart); free(ustart); free(by_c); free(by_u); free(level); free(queue); free(pos);
        free(unew); free(cnew); free(used);
        return rc;
}
