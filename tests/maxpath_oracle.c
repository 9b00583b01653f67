/* tests/maxpath_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU reference of the most probable path of every string, for
 * the Viterbi tests (tests/maxpath_oracle.py compiles and loads it).  Plain C11 + OpenMP, on the descriptors of
 * oracle/wfsa_oracle.h.
 *
 * best[s] = max over the accepting paths of string s of the summed log-weights of their edges (-inf: not recognised), by a
 * forward pass in the (max, +) semiring over the dense lattice of the oracle's log-domain forward-backward (emissions of
 * any length, empty ones included), with a backpointer (transition, emission) per lattice node and a traceback.  Each node
 * adds (log a + mu) first, then log b, and the end adds log a(u, end) last, so best[s] is the left-to-right sum of the
 * returned steps. */
#include "wfsa_oracle.h"

#include <math.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* one string; a -inf edge (trimmed away) is no edge.  steps: room for cap (transition, emission) pairs, emission -1 on the
 * final transition; *n = steps written (0: no path, -1: more than cap) */
static double dp_maxpath(const oracle_fsa* f, const int32_t* order, const int32_t* src, const double* ltw, const double* lew,
                         const int32_t* tok, int len, int32_t* steps, int cap, int64_t* n)
{
    const int S = f->n_states;
    const size_t sz = (size_t)(len + 1) * S;
    double* mu = malloc(sizeof(double) * (sz > 0 ? sz : 1));
    int32_t* bt = malloc(sizeof(int32_t) * (sz > 0 ? sz : 1));
    int32_t* be = malloc(sizeof(int32_t) * (sz > 0 ? sz : 1));
    for (size_t i = 0; i < sz; ++i) mu[i] = -INFINITY;
    mu[f->start_state] = 0.0;
    double m = -INFINITY;
    int fin_t = -1, fin_u = -1;
    for (int pos = 0; pos <= len; ++pos)
        for (int oi = 0; oi < S; ++oi) {
            const int u = order[oi];
            const double au = mu[(size_t)pos * S + u];
            if (au == -INFINITY || u == f->end_state) continue;
            for (int t = f->trans_row[u]; t < f->trans_row[u + 1]; ++t) {
                if (ltw[t] == -INFINITY) continue;
                const int v = f->trans_dst[t];
                const double wv = au + ltw[t];
                if (v == f->end_state) { if (pos == len && wv > m) { m = wv; fin_t = t; fin_u = u; } continue; }
                for (int e = f->emis_row[v]; e < f->emis_row[v + 1]; ++e) {
                    if (lew[e] == -INFINITY) continue;
                    const int e0 = f->emis_tok_off[e], el = f->emis_tok_off[e + 1] - e0;
                    if (pos + el > len) continue;
                    int ok = 1;
                    for (int k = 0; k < el; ++k) if (tok[pos + k] != f->emis_tok[e0 + k]) { ok = 0; break; }
                    if (!ok) continue;
                    const size_t d = (size_t)(pos + el) * S + v;
                    if (wv + lew[e] > mu[d]) { mu[d] = wv + lew[e]; bt[d] = t; be[d] = e; }
                }
            }
        }
    *n = 0;
    if (m > -INFINITY) {
        /* walk back once to count, then again to write from the end */
        int64_t cnt = 1;
        for (int p = len, v = fin_u; v != f->start_state; ++cnt) {
            const size_t d = (size_t)p * S + v;
            p -= f->emis_tok_off[be[d] + 1] - f->emis_tok_off[be[d]];
            v = src[bt[d]];
        }
        if (cnt > cap) *n = -1;
        else {
            *n = cnt;
            int64_t o = cnt - 1;
            steps[2 * o] = fin_t; steps[2 * o + 1] = -1;
            for (int p = len, v = fin_u; v != f->start_state;) {
                const size_t d = (size_t)p * S + v;
                --o;
                steps[2 * o] = bt[d]; steps[2 * o + 1] = be[d];
                p -= f->emis_tok_off[be[d] + 1] - f->emis_tok_off[be[d]];
                v = src[bt[d]];
            }
        }
    }
    free(mu); free(bt); free(be);
    return m;
}

int maxpath_dp(const oracle_fsa* f, const oracle_corpus* c, const double* ltw, const double* lew, double* best,
               int64_t* n_steps, int32_t* steps, int cap, int nthreads)
{
    const int S = f->n_states;
    /* states in an order in which empty-emission arcs only go forward (as tests/minpath_oracle.c) */
    int32_t* order = malloc(sizeof(int32_t) * (size_t)(S > 0 ? S : 1));
    int32_t* src = malloc(sizeof(int32_t) * (size_t)(f->trans_row[S] > 0 ? f->trans_row[S] : 1));
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
    int nth = nthreads > 0 ? nthreads : 1;
#ifdef _OPENMP
    if (nthreads <= 0) nth = omp_get_max_threads();
#endif
    if (nth < 1) nth = 1;
#ifdef _OPENMP
#pragma omp parallel for num_threads(nth) schedule(dynamic, 64)
#endif
    for (int64_t s = 0; s < c->n_strings; ++s)
        best[s] = dp_maxpath(f, order, src, ltw, lew, c->tokens + c->offsets[s], (int)(c->offsets[s + 1] - c->offsets[s]),
                             steps + (size_t)s * cap * 2, cap, n_steps + s);
    free(order); free(src);
    return 0;
}
