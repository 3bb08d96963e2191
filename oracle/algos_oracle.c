/*
 * ORACLE (test infrastructure, not product code): plain-C restatement of the
 * reference's Cython preprocessing, /root/reference/graphormer/algos.pyx.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * `--impl reference` legs may load this library; the product path never does.
 *
 * Pinned against the really-compiled reference (oracle/_ref, built by
 * oracle/build_ref.py from algos.pyx unmodified) on the KATs in
 * tests/golden/, and on seeded random and node-510 hub graphs in
 * tests/test_oracle_algos.py: there against oracle/_ref when it is built,
 * else against a Python restatement of algos.pyx pinned to those KATs.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define UNREACH 510

/* algos.pyx:9-54  floyd_warshall(adjacency_matrix) -> (M, path)
 *   :27-32  diag <- 0, zero entries <- 510
 *   :35-45  for k: for i: for j: strict '>' relaxation, path[i][j] = k
 *   :48-52  entries >= 510 -> M = path = 510                              */
void oracle_floyd_warshall(const uint8_t *adj, int n, int64_t *M, int64_t *path)
{
    for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) {
            int64_t v = adj[(size_t)i * n + j] ? 1 : 0;
            if (i == j) v = 0;
            else if (v == 0) v = UNREACH;
            M[(size_t)i * n + j] = v;
            path[(size_t)i * n + j] = 0;
        }
    for (int k = 0; k < n; k++) {
        const int64_t *Mk = M + (size_t)k * n;
        for (int i = 0; i < n; i++) {
            int64_t *Mi = M + (size_t)i * n;
            int64_t Mik = Mi[k];
            for (int j = 0; j < n; j++) {
                int64_t c = Mik + Mk[j];
                if (Mi[j] > c) {
                    Mi[j] = c;
                    path[(size_t)i * n + j] = k;
                }
            }
        }
    }
    for (size_t t = 0; t < (size_t)n * n; t++)
        if (M[t] >= UNREACH) { M[t] = UNREACH; path[t] = UNREACH; }
}

/* algos.pyx:57-62  get_all_edges(path, i, j): in-order expansion, with the
 * k == 0 short-circuit ("0" means direct OR via node 0).  Appends to buf.   */
static void all_edges(const int64_t *path, int n, int i, int j, int *buf, int *len)
{
    int k = (int)path[(size_t)i * n + j];
    if (k == 0) return;
    all_edges(path, n, i, k, buf, len);
    buf[(*len)++] = k;
    all_edges(path, n, k, j, buf, len);
}

/* algos.pyx:65-96  gen_edge_input(max_dist, path, edge_feat)
 *   out[n, n, hops, F] float32, -1 filled; for i != j with path != 510 the
 *   walk [i]+get_all_edges+[j] is laid along the hop axis.
 *   `hops` = min(max_dist, hop_cap): identical to slicing the reference
 *   output [:, :, :hop_cap, :] (collator.py:323) without the 510-deep temp.
 *   A walk longer than the hop axis would raise IndexError in the reference
 *   when hop axis == max_dist; with a cap we simply stop (the slice).       */
int oracle_gen_edge_input(int max_dist, const int64_t *path, const int64_t *edge_feat,
                          int n, int F, int hop_cap, float *out)
{
    int hops = max_dist < hop_cap ? max_dist : hop_cap;
    size_t tot = (size_t)n * n * hops * F;
    for (size_t t = 0; t < tot; t++) out[t] = -1.0f;
    int *walk = (int *)malloc(sizeof(int) * (size_t)(4 * n + 8));
    if (!walk) return -1;
    int rc = 0;
    for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) {
            if (i == j) continue;
            if (path[(size_t)i * n + j] == UNREACH) continue;
            int len = 0;
            walk[len++] = i;
            all_edges(path, n, i, j, walk, &len);
            walk[len++] = j;
            int num_path = len - 1;
            if (num_path > max_dist) rc = 1;     /* reference would IndexError */
            for (int k = 0; k < num_path && k < hops; k++)
                for (int f = 0; f < F; f++)
                    out[(((size_t)i * n + j) * hops + k) * F + f] =
                        (float)edge_feat[((size_t)walk[k] * n + walk[k + 1]) * F + f];
        }
    free(walk);
    return rc;
}
