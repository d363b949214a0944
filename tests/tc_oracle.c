/*
 * tc_oracle.c — TEST INFRASTRUCTURE, not product code: the CPU restatement of triangle counting that
 * tests/test_gpu_tc.py compares vglb_tc against. The test compiles it into a temporary directory (gcc -O2 -fopenmp) and
 * loads it with ctypes; it is pinned there against scipy and against closed forms.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <omp.h>

/* ------------------------------------------------------------------------------------------------------------ */
/* Triangle counting (algorithms/tc): the triangles of the undirected simple graph under the CSR ({u, w} is an edge  */
/* when u != w and u->w or w->u is in the CSR). First each vertex's undirected neighbours, sorted, deduplicated and  */
/* without self loops. Then the forward algorithm over the order "higher degree first, ties by id": N<(u) = the      */
/* neighbours that come before u; for u, mark N<(u), and for every v in N<(u) count the marked w in N<(v). Each       */
/* triangle is found once, at its last vertex u. counts[v] = triangles that contain v (int64).                       */
/* ------------------------------------------------------------------------------------------------------------ */

static int cmp_i32(const void *a, const void *b)
{
    const int32_t x = *(const int32_t *)a, y = *(const int32_t *)b;
    return (x > y) - (x < y);
}

int vglo_tc(int32_t V, const int64_t *row_ptr, const int32_t *adj, int64_t *counts, int64_t *total)
{
    const int64_t E = row_ptr[V];
    int64_t *np = calloc((size_t)V + 1, sizeof(int64_t)), *cur = malloc(((size_t)V + 1) * sizeof(int64_t));
    int32_t *nb = malloc((size_t)(2 * E + 1) * sizeof(int32_t)), *deg = calloc((size_t)V + 1, sizeof(int32_t));
    int64_t *lp = calloc((size_t)V + 1, sizeof(int64_t));
    if (!np || !cur || !nb || !deg || !lp) { free(np); free(cur); free(nb); free(deg); free(lp); return 1; }
    for (int32_t u = 0; u < V; u++)
        for (int64_t p = row_ptr[u]; p < row_ptr[u + 1]; p++)
            if (adj[p] != u) { np[u + 1]++; np[adj[p] + 1]++; }
    for (int32_t u = 0; u < V; u++) np[u + 1] += np[u];
    memcpy(cur, np, ((size_t)V + 1) * sizeof(int64_t));
    for (int32_t u = 0; u < V; u++)
        for (int64_t p = row_ptr[u]; p < row_ptr[u + 1]; p++)
            if (adj[p] != u) { nb[cur[u]++] = adj[p]; nb[cur[adj[p]]++] = u; }
    #pragma omp parallel for schedule(dynamic, 256)
    for (int32_t u = 0; u < V; u++)
    {
        int32_t *l = nb + np[u];
        const int64_t n = np[u + 1] - np[u];
        qsort(l, (size_t)n, sizeof(int32_t), cmp_i32);
        int64_t k = 0;
        for (int64_t i = 0; i < n; i++) if (k == 0 || l[i] != l[k - 1]) l[k++] = l[i];
        deg[u] = (int32_t)k;
    }
    /* N<(u) in place at the front of u's list: neighbours w with (deg[w] > deg[u]) or (deg[w] == deg[u] and w < u) */
    for (int32_t u = 0; u < V; u++)
    {
        int32_t *l = nb + np[u];
        int64_t k = 0;
        for (int64_t i = 0; i < deg[u]; i++)
        {
            const int32_t w = l[i];
            if (deg[w] > deg[u] || (deg[w] == deg[u] && w < u)) l[k++] = w;
        }
        lp[u] = k;
    }
    const int T = omp_get_max_threads();
    int64_t *tcnt = calloc((size_t)T * (size_t)V + 1, sizeof(int64_t));
    int32_t *tmark = malloc(((size_t)T * (size_t)V + 1) * sizeof(int32_t));
    if (!tcnt || !tmark) { free(np); free(cur); free(nb); free(deg); free(lp); free(tcnt); free(tmark); return 1; }
    int64_t tot = 0;
    #pragma omp parallel reduction(+ : tot)
    {
        int64_t *cnt = tcnt + (size_t)omp_get_thread_num() * V;
        int32_t *mark = tmark + (size_t)omp_get_thread_num() * V;
        for (int32_t v = 0; v < V; v++) mark[v] = -1;
        #pragma omp for schedule(dynamic, 64)
        for (int32_t u = 0; u < V; u++)
        {
            const int32_t *lu = nb + np[u];
            for (int64_t i = 0; i < lp[u]; i++) mark[lu[i]] = u;
            for (int64_t i = 0; i < lp[u]; i++)
            {
                const int32_t v = lu[i];
                const int32_t *lv = nb + np[v];
                for (int64_t q = 0; q < lp[v]; q++)
                {
                    const int32_t w = lv[q];
                    if (mark[w] == u) { cnt[u]++; cnt[v]++; cnt[w]++; tot++; }
                }
            }
        }
    }
    #pragma omp parallel for
    for (int32_t v = 0; v < V; v++)
    {
        int64_t s = 0;
        for (int t = 0; t < T; t++) s += tcnt[(size_t)t * V + v];
        counts[v] = s;
    }
    *total = tot;
    free(np); free(cur); free(nb); free(deg); free(lp); free(tcnt); free(tmark);
    return 0;
}

