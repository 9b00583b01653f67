/* tests/minpath_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU reference of the smallest path weight of every string, for
 * the rmin tests (tests/minpath_oracle.py compiles and loads it).  Plain C11 + OpenMP, on the descriptors of
 * oracle/wfsa_oracle.h.
 *
 * m[s] = min over the accepting paths of string s of the summed log-weights of their edges (+inf: not recognised), by a
 * forward pass in the (min, +) semiring over the dense lattice of the oracle's log-domain forward-backward (emissions of
 * any length, empty ones included).  The smallest path posterior of s is exp(m[s] - logq[s]). */
#include "wfsa_oracle.h"

#include <math.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* one string; a -inf edge (trimmed away) is no edge.  (src/QuasiNewtonLearner.cpp:80-84 takes the minimum of the path
 * posteriors over every path.) */
static double dp_minpath(const oracle_fsa* f, const int32_t* order, const double* ltw, const double* lew, const int32_t* tok, int len)
{
    const int S = f->n_states;
    const size_t sz = (size_t)(len + 1) * S;
    double* mu = malloc(sizeof(double) * (sz > 0 ? sz : 1));
    for (size_t i = 0; i < sz; ++i) mu[i] = INFINITY;
    mu[f->start_state] = 0.0;
    double m = INFINITY;
    for (int pos = 0; pos <= len; ++pos)
        for (int oi = 0; oi < S; ++oi) {
            const int u = order[oi];
            const double au = mu[(size_t)pos * S + u];
            if (au == INFINITY || u == f->end_state) continue;
            for (int t = f->trans_row[u]; t < f->trans_row[u + 1]; ++t) {
                if (ltw[t] == -INFINITY) continue;
                const int v = f->trans_dst[t];
                const double wv = au + ltw[t];
                if (v == f->end_state) { if (pos == len && wv < m) m = wv; continue; }
                for (int e = f->emis_row[v]; e < f->emis_row[v + 1]; ++e) {
                    if (lew[e] == -INFINITY) continue;
                    const int e0 = f->emis_tok_off[e], el = f->emis_tok_off[e + 1] - e0;
                    if (pos + el > len) continue;
                    int ok = 1;
                    for (int k = 0; k < el; ++k) if (tok[pos + k] != f->emis_tok[e0 + k]) { ok = 0; break; }
                    if (!ok) continue;
                    double* d = mu + (size_t)(pos + el) * S + v;
                    if (wv + lew[e] < *d) *d = wv + lew[e];
                }
            }
        }
    free(mu);
    return m;
}

int minpath_dp(const oracle_fsa* f, const oracle_corpus* c, const double* ltw, const double* lew, double* m, int nthreads)
{
    const int S = f->n_states;
    /* states in an order in which empty-emission arcs only go forward (as the oracle's dp_build, for every automaton) */
    int32_t* order = malloc(sizeof(int32_t) * (size_t)(S > 0 ? S : 1));
    char* eps = calloc((size_t)S + 1, 1);
    int* indeg = calloc((size_t)S + 1, sizeof(int));
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
    int nth = nthreads > 0 ? nthreads : 1;
#ifdef _OPENMP
    if (nthreads <= 0) nth = omp_get_max_threads();
#endif
    if (nth < 1) nth = 1;
#ifdef _OPENMP
#pragma omp parallel for num_threads(nth) schedule(dynamic, 64)
#endif
    for (int64_t s = 0; s < c->n_strings; ++s)
        m[s] = dp_minpath(f, order, ltw, lew, c->tokens + c->offsets[s], (int)(c->offsets[s + 1] - c->offsets[s]));
    free(order);
    return 0;
}
