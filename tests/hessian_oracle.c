/* tests/hessian_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU reference of H_f times a block of directions, for the H_f
 * tests (tests/hessian_oracle.py compiles and loads it).  Plain C11 + OpenMP, on the descriptors of oracle/wfsa_oracle.h.
 *
 *   H_f = - sum_s p_s Cov_s(c_j, c_k),   c_j = how often parameter j occurs on the path (the path posterior of string s)
 *
 * without enumerating paths: a tangent forward-backward in long double, in the log domain, over the dense lattice of the
 * oracle's forward-backward (nodes (position, state), states in an order in which empty emissions only go forward, so
 * emissions of any length, empty ones included).  For a direction v the tangent of edge e is d_e = v[trans param] +
 * v[emis param] (0 for a parameter that is not trimmed in), and
 *   A(u) = E[sum of d over the prefix | the prefix ends at u]   (forward: the softmax-weighted mean over incoming edges)
 *   B(u) = E[sum of d over the suffix | the suffix starts at u] (backward, the same over outgoing edges)
 *   Cov_s(c_j, c.v) = sum_e n_j(e) gamma_e (A(src) + d_e + B(dst) - A(end)),   gamma_e = posterior of edge e,
 * since c_j = sum_e n_j(e) [e on the path] and an edge occurs at most once on a path.  All m directions of V (n x m, row
 * major) are carried together per node; HV[j*m + k] = (H_f v_k)_j.  V = I gives the full H_f. */
#include "wfsa_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

typedef long double ld;

/* running softmax-weighted mean: (lse, mean[m]) absorbs one term of log weight lw and value x[m] (x NULL: d + y) */
static void absorb(ld* lse, ld* mean, ld lw, const ld* d, const ld* y, int m)
{
    if (lw == -INFINITY) return;
    if (*lse == -INFINITY) {
        *lse = lw;
        for (int k = 0; k < m; ++k) mean[k] = d[k] + y[k];
        return;
    }
    const ld hi = *lse > lw ? *lse : lw;
    const ld a = expl(*lse - hi), b = expl(lw - hi), z = a + b;
    *lse = hi + logl(z);
    for (int k = 0; k < m; ++k) mean[k] = (mean[k] * a + (d[k] + y[k]) * b) / z;
}

typedef struct {
    const oracle_fsa* f;
    const int32_t* order;
    const double *ltw, *lew;
    const int32_t* edge_param;      /* [n_trans + n_emis] */
    const double* V;
    int n, m, mc, k0;               /* directions k0 .. k0 + mc - 1 of this pass */
} ctx_t;

static void tangent(const ctx_t* C, int t, int e, ld* d)
{
    const int n_trans = C->f->trans_row[C->f->n_states];
    const int jt = C->edge_param[t], je = e >= 0 ? C->edge_param[n_trans + e] : -1;
    for (int k = 0; k < C->mc; ++k) {
        ld v = 0.0L;
        if (jt >= 0) v += C->V[(size_t)jt * C->m + C->k0 + k];
        if (je >= 0) v += C->V[(size_t)je * C->m + C->k0 + k];
        d[k] = v;
    }
}

/* does emission e of the target state match tok at pos? returns its length, or -1 */
static int emis_len(const oracle_fsa* f, int e, const int32_t* tok, int pos, int len)
{
    const int e0 = f->emis_tok_off[e], el = f->emis_tok_off[e + 1] - e0;
    if (pos + el > len) return -1;
    for (int k = 0; k < el; ++k) if (tok[pos + k] != f->emis_tok[e0 + k]) return -1;
    return el;
}

/* one string, one chunk of directions: adds -p Cov(c_j, c.v_k) to acc[j * mc + k] */
static void dp_string(const ctx_t* C, const int32_t* tok, int len, double p, ld* acc,
                      ld* al, ld* be, ld* A, ld* B, ld* d, ld* x)
{
    const oracle_fsa* f = C->f;
    const int S = f->n_states, mc = C->mc;
    const size_t sz = (size_t)(len + 1) * S;
    for (size_t i = 0; i < sz; ++i) { al[i] = -INFINITY; be[i] = -INFINITY; }
    memset(A, 0, sizeof(ld) * sz * mc);
    memset(B, 0, sizeof(ld) * sz * mc);
    ld a_end = -INFINITY, *A_end = x + mc;                 /* x: scratch [2 mc] */
    for (int k = 0; k < mc; ++k) A_end[k] = 0.0L;
    al[f->start_state] = 0.0L;
    /* forward */
    for (int pos = 0; pos <= len; ++pos)
        for (int oi = 0; oi < S; ++oi) {
            const int u = C->order[oi];
            const size_t iu = (size_t)pos * S + u;
            if (al[iu] == -INFINITY || u == f->end_state) continue;
            for (int t = f->trans_row[u]; t < f->trans_row[u + 1]; ++t) {
                if (C->ltw[t] == -INFINITY) continue;
                const int v = f->trans_dst[t];
                if (v == f->end_state) {
                    if (pos != len) continue;
                    tangent(C, t, -1, d);
                    absorb(&a_end, A_end, al[iu] + C->ltw[t], d, A + iu * mc, mc);
                    continue;
                }
                for (int e = f->emis_row[v]; e < f->emis_row[v + 1]; ++e) {
                    if (C->lew[e] == -INFINITY) continue;
                    const int el = emis_len(f, e, tok, pos, len);
                    if (el < 0) continue;
                    const size_t iv = (size_t)(pos + el) * S + v;
                    tangent(C, t, e, d);
                    absorb(&al[iv], A + iv * mc, al[iu] + (ld)C->ltw[t] + (ld)C->lew[e], d, A + iu * mc, mc);
                }
            }
        }
    if (a_end == -INFINITY) return;                        /* not recognised */
    /* backward, and the covariances of every edge */
    for (int pos = len; pos >= 0; --pos)
        for (int oi = S - 1; oi >= 0; --oi) {
            const int u = C->order[oi];
            const size_t iu = (size_t)pos * S + u;
            if (al[iu] == -INFINITY || u == f->end_state) continue;
            for (int t = f->trans_row[u]; t < f->trans_row[u + 1]; ++t) {
                if (C->ltw[t] == -INFINITY) continue;
                const int v = f->trans_dst[t];
                const int n_trans = f->trans_row[S];
                if (v == f->end_state) {
                    if (pos != len) continue;
                    tangent(C, t, -1, d);
                    for (int k = 0; k < mc; ++k) x[k] = 0.0L;
                    absorb(&be[iu], B + iu * mc, (ld)C->ltw[t], d, x, mc);
                    const ld g = expl(al[iu] + (ld)C->ltw[t] - a_end);
                    const int jt = C->edge_param[t];
                    if (jt >= 0)
                        for (int k = 0; k < mc; ++k) acc[(size_t)jt * mc + k] -= (ld)p * g * (A[iu * mc + k] + d[k] - A_end[k]);
                    continue;
                }
                for (int e = f->emis_row[v]; e < f->emis_row[v + 1]; ++e) {
                    if (C->lew[e] == -INFINITY) continue;
                    const int el = emis_len(f, e, tok, pos, len);
                    if (el < 0) continue;
                    const size_t iv = (size_t)(pos + el) * S + v;
                    if (be[iv] == -INFINITY) continue;             /* does not reach the end */
                    const ld lw = (ld)C->ltw[t] + (ld)C->lew[e];
                    tangent(C, t, e, d);
                    absorb(&be[iu], B + iu * mc, lw + be[iv], d, B + iv * mc, mc);
                    const ld g = expl(al[iu] + lw + be[iv] - a_end);
                    const int js[2] = {C->edge_param[t], C->edge_param[n_trans + e]};
                    for (int q = 0; q < 2; ++q) {
                        if (js[q] < 0) continue;
                        for (int k = 0; k < mc; ++k)
                            acc[(size_t)js[q] * mc + k] -= (ld)p * g * (A[iu * mc + k] + d[k] + B[iv * mc + k] - A_end[k]);
                    }
                }
            }
        }
}

int hessian_oracle_hv(const oracle_fsa* f, const oracle_corpus* c, const double* ltw, const double* lew,
                      const int32_t* edge_param, int32_t n, const double* V, int32_t m, double* HV, int nthreads)
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
    int64_t max_len = 0;
    for (int64_t s = 0; s < c->n_strings; ++s) if (c->offsets[s + 1] - c->offsets[s] > max_len) max_len = c->offsets[s + 1] - c->offsets[s];
    /* directions per pass: the tangents of the longest string in at most 64 MB per thread */
    const size_t nodes = (size_t)(max_len + 1) * (S > 0 ? S : 1);
    int mc = (int)((64u << 20) / (2 * sizeof(ld) * nodes));
    if (mc < 1) mc = 1;
    if (mc > m) mc = m;
    memset(HV, 0, sizeof(double) * (size_t)n * m);
    for (int k0 = 0; k0 < m; k0 += mc) {
        const int mk = m - k0 < mc ? m - k0 : mc;
        const ctx_t C = {f, order, ltw, lew, edge_param, V, n, m, mk, k0};
        ld* total = calloc((size_t)n * mk + 1, sizeof(ld));
#ifdef _OPENMP
#pragma omp parallel num_threads(nth)
#endif
        {
            ld* acc = calloc((size_t)n * mk + 1, sizeof(ld));
            ld *al = malloc(sizeof(ld) * nodes), *be = malloc(sizeof(ld) * nodes);
            ld *A = malloc(sizeof(ld) * nodes * mk), *B = malloc(sizeof(ld) * nodes * mk);
            ld *d = malloc(sizeof(ld) * mk), *x = malloc(sizeof(ld) * 2 * mk);
#ifdef _OPENMP
#pragma omp for schedule(dynamic, 16)
#endif
            for (int64_t s = 0; s < c->n_strings; ++s)
                dp_string(&C, c->tokens + c->offsets[s], (int)(c->offsets[s + 1] - c->offsets[s]), c->p[s], acc, al, be, A, B, d, x);
#ifdef _OPENMP
#pragma omp critical
#endif
            for (size_t i = 0; i < (size_t)n * mk; ++i) total[i] += acc[i];
            free(acc); free(al); free(be); free(A); free(B); free(d); free(x);
        }
        for (int j = 0; j < n; ++j)
            for (int k = 0; k < mk; ++k) HV[(size_t)j * m + k0 + k] = (double)total[(size_t)j * mk + k];
        free(total);
    }
    free(order);
    return 0;
}
