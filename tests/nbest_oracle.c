/* tests/nbest_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU reference of the k most probable paths of every string, for the
 * N-best tests (tests/nbest_oracle.py compiles and loads it).  Plain C11 + OpenMP, on the descriptors of
 * oracle/wfsa_oracle.h.
 *
 * The forward of tests/maxpath_oracle.c in the (max, +) semiring over the dense log-domain lattice (emissions of any length,
 * empty ones included), with a sorted list of the k largest values per lattice node and a backpointer (transition, emission,
 * source rank) per entry, then a traceback of every rank.  Each node adds (log a + mu) first, then log b, and the end adds
 * log a(u, end) last, so every value is the left-to-right sum of its path's steps.  Candidates are pushed in the order source
 * state (in the order below), transition, emission, source rank; a node keeps the first strictly larger ones, and the ranks
 * of a source stop at the first that is not larger than the node's k-th (the source list is sorted).  The end's list takes
 * mu_T[u][r] + log a(u, end) in the order source state, transition, rank.  With k = 1 this is maxpath_dp of
 * tests/maxpath_oracle.c. */
#include "wfsa_oracle.h"

#include <math.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* states in an order in which empty-emission arcs only go forward (as tests/minpath_oracle.c), and the source state of
 * every transition */
static void state_order(const oracle_fsa* f, int32_t* order, int32_t* src)
{
    const int S = f->n_states;
    char* eps = calloc((size_t)S + 1, 1);
    int* indeg = calloc((size_t)S + 1, sizeof(int));
    for (int u = 0; u < S; ++u) for (int t = f->trans_row[u]; t < f->trans_row[u + 1]; ++t) src[t] = u;
    for (int s = 0; s < S; ++s) {
        if (s == f->start_state || s == f->end_state) continue;
        for (int e = f->emis_row[s]; e < f->emis_row[s + 1]; ++e) if (f->emis_tok_off[e + 1] == f->emis_tok_off[e]) eps[s] = 1;
    }
    for (int u = 0; u < S; ++u) for (int t = f->trans_row[u]; t < f->trans_row[u + 1]; ++t) if (eps[f->trans_dst[t]]) indeg[f->trans_dst[t]]++;
    int head = 0, tail = 0;
    for (int s = 0; s < S; ++s) if (!indeg[s]) order[tail++] = s;
    while (head < tail) {
        const int u = order[head++];
        for (int t = f->trans_row[u]; t < f->trans_row[u + 1]; ++t) { const int v = f->trans_dst[t]; if (eps[v] && --indeg[v] == 0) order[tail++] = v; }
    }
    for (int s = 0; tail < S && s < S; ++s) if (indeg[s] > 0) order[tail++] = s;
    free(eps); free(indeg);
}

static int n_threads(int nthreads)
{
    int nth = nthreads > 0 ? nthreads : 1;
#ifdef _OPENMP
    if (nthreads <= 0) nth = omp_get_max_threads();
#endif
    return nth < 1 ? 1 : nth;
}

/* x into the sorted list v[0..k) after every entry >= x, with its backpointer; x > v[k-1] on entry */
static void kb_insert(double* v, int32_t* bt, int32_t* be, int32_t* br, int k, double x, int t, int e, int r)
{
    int j = k - 1;
    while (j > 0 && x > v[j - 1]) { v[j] = v[j - 1]; bt[j] = bt[j - 1]; be[j] = be[j - 1]; br[j] = br[j - 1]; --j; }
    v[j] = x; bt[j] = t; be[j] = e; br[j] = r;
}

/* one string: best[0..k) and the steps of each rank (room for cap pairs each, at steps + r * cap * 2), n[r] steps written
 * (0: no such path, -1: more than cap) */
static void dp_kbest(const oracle_fsa* f, const int32_t* order, const int32_t* src, const double* ltw, const double* lew,
                     const int32_t* tok, int len, int k, double* best, int32_t* steps, int cap, int64_t* n)
{
    const int S = f->n_states;
    const size_t sz = (size_t)(len + 1) * S * k;
    double* mu = malloc(sizeof(double) * (sz > 0 ? sz : 1));
    int32_t* bt = malloc(sizeof(int32_t) * (sz > 0 ? sz : 1));
    int32_t* be = malloc(sizeof(int32_t) * (sz > 0 ? sz : 1));
    int32_t* br = malloc(sizeof(int32_t) * (sz > 0 ? sz : 1));
    int32_t* ft = malloc(sizeof(int32_t) * (size_t)k);
    int32_t* fe = malloc(sizeof(int32_t) * (size_t)k);
    int32_t* fr = malloc(sizeof(int32_t) * (size_t)k);
    for (size_t i = 0; i < sz; ++i) mu[i] = -INFINITY;
    for (int r = 0; r < k; ++r) best[r] = -INFINITY;
    mu[(size_t)f->start_state * k] = 0.0;
    for (int pos = 0; pos <= len; ++pos)
        for (int oi = 0; oi < S; ++oi) {
            const int u = order[oi];
            const double* au = mu + ((size_t)pos * S + u) * k;
            if (au[0] == -INFINITY || u == f->end_state) continue;
            for (int t = f->trans_row[u]; t < f->trans_row[u + 1]; ++t) {
                if (ltw[t] == -INFINITY) continue;
                const int v = f->trans_dst[t];
                if (v == f->end_state) {
                    if (pos == len)
                        for (int r = 0; r < k; ++r) {
                            const double x = au[r] + ltw[t];
                            if (!(x > best[k - 1])) break;
                            kb_insert(best, ft, fe, fr, k, x, t, -1, r);
                        }
                    continue;
                }
                for (int e = f->emis_row[v]; e < f->emis_row[v + 1]; ++e) {
                    if (lew[e] == -INFINITY) continue;
                    const int e0 = f->emis_tok_off[e], el = f->emis_tok_off[e + 1] - e0;
                    if (pos + el > len) continue;
                    int ok = 1;
                    for (int q = 0; q < el; ++q) if (tok[pos + q] != f->emis_tok[e0 + q]) { ok = 0; break; }
                    if (!ok) continue;
                    const size_t d = ((size_t)(pos + el) * S + v) * k;
                    for (int r = 0; r < k; ++r) {
                        const double x = (au[r] + ltw[t]) + lew[e];
                        if (!(x > mu[d + k - 1])) break;
                        kb_insert(mu + d, bt + d, be + d, br + d, k, x, t, e, r);
                    }
                }
            }
        }
    for (int r = 0; r < k; ++r) {
        n[r] = 0;
        if (!(best[r] > -INFINITY)) continue;
        /* walk back once to count, then again to write from the end */
        int64_t cnt = 1;
        for (int p = len, v = src[ft[r]], rr = fr[r]; v != f->start_state; ++cnt) {
            const size_t d = ((size_t)p * S + v) * k + rr;
            p -= f->emis_tok_off[be[d] + 1] - f->emis_tok_off[be[d]];
            v = src[bt[d]]; rr = br[d];
        }
        if (cnt > cap) { n[r] = -1; continue; }
        n[r] = cnt;
        int32_t* st = steps + (size_t)r * cap * 2;
        int64_t o = cnt - 1;
        st[2 * o] = ft[r]; st[2 * o + 1] = -1;
        for (int p = len, v = src[ft[r]], rr = fr[r]; v != f->start_state;) {
            const size_t d = ((size_t)p * S + v) * k + rr;
            --o;
            st[2 * o] = bt[d]; st[2 * o + 1] = be[d];
            p -= f->emis_tok_off[be[d] + 1] - f->emis_tok_off[be[d]];
            v = src[bt[d]]; rr = br[d];
        }
    }
    free(mu); free(bt); free(be); free(br); free(ft); free(fe); free(fr);
}

/* best[s * k + r], n_steps[s * k + r] and the steps of path s * k + r at steps + (s * k + r) * cap * 2 */
int nbest_kbest(const oracle_fsa* f, const oracle_corpus* c, const double* ltw, const double* lew, int k, double* best,
                  int64_t* n_steps, int32_t* steps, int cap, int nthreads)
{
    if (k < 1) return -1;
    const int S = f->n_states;
    int32_t* order = malloc(sizeof(int32_t) * (size_t)(S > 0 ? S : 1));
    int32_t* src = malloc(sizeof(int32_t) * (size_t)(f->trans_row[S] > 0 ? f->trans_row[S] : 1));
    state_order(f, order, src);
    const int nth = n_threads(nthreads);
#ifdef _OPENMP
#pragma omp parallel for num_threads(nth) schedule(dynamic, 16)
#endif
    for (int64_t s = 0; s < c->n_strings; ++s)
        dp_kbest(f, order, src, ltw, lew, c->tokens + c->offsets[s], (int)(c->offsets[s + 1] - c->offsets[s]), k,
                 best + (size_t)s * k, steps + (size_t)s * k * cap * 2, cap, n_steps + (size_t)s * k);
    (void)nth;
    free(order); free(src);
    return 0;
}
