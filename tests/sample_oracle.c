/* tests/sample_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU reference of path sampling, for the sampling tests
 * (tests/sample_oracle.py compiles and loads it).  Plain C11 + OpenMP, on the descriptors of oracle/wfsa_oracle.h.
 *
 * Over the dense log-domain lattice of tests/maxpath_oracle.c (emissions of any length, empty ones included), per string:
 * the forward in (logaddexp, +) gives log q and the nodes the forward reaches, the backward gives beta[pos][u], the log
 * weight of the continuations of node (pos, u), both in the order of the device's generic kernel.  Then every draw walks
 * forward from (0, start): at (pos, u) the entries are, in table order, every transition t of u with every emission e of
 * its target that matches the string at pos, weight exp(((log a + log b) + beta_next) - beta_here), and at pos = len the
 * transitions into the end state, weight exp(log a - beta_here).  The draw takes the first entry whose running sum exceeds
 * u * total (the last entry of positive weight when rounding leaves none), u from its own copy of Philox4x32-10 with the
 * counter (d, r, s, 0), d the step.  This is the device's rule for automata without fast tables, so the device returns
 * these draws. */
#include "wfsa_oracle.h"

#include <math.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

void sample_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
    for (int i = 0; i < 10; ++i) {
        if (i) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c0 = n0; c1 = (uint32_t)p1; c2 = n2; c3 = (uint32_t)p0;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

static double uniform(uint32_t d, uint32_t r, uint32_t s, const uint32_t key[2])
{
    const uint32_t ctr[4] = {d, r, s, 0u};
    uint32_t o[4];
    sample_philox4x32_10(ctr, key, o);
    return (double)((((uint64_t)o[0] << 32) | o[1]) >> 11) * 0x1p-53;
}

static double logaddexp(double a, double b)
{
    if (a == -INFINITY) return b;
    if (b == -INFINITY) return a;
    const double m = fmax(a, b);
    return m + log1p(exp(-fabs(a - b)));
}

/* states in an order in which empty-emission arcs only go forward (the device's eps_order, as tests/maxpath_oracle.c) */
static void state_order(const oracle_fsa* f, int32_t* order)
{
    const int S = f->n_states;
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
}

static int matches(const oracle_fsa* f, const int32_t* tok, int len, int pos, int e, int* el)
{
    const int e0 = f->emis_tok_off[e];
    *el = f->emis_tok_off[e + 1] - e0;
    if (pos + *el > len) return 0;
    for (int q = 0; q < *el; ++q) if (tok[pos + q] != f->emis_tok[e0 + q]) return 0;
    return 1;
}

/* one string: log q, and per draw r its logw, its steps (room for cap pairs at steps + r * cap * 2) and their number
 * (0: no path, -1: more than cap) */
static double sample_string(const oracle_fsa* f, const int32_t* order, const double* ltw, const double* lew, const int32_t* tok,
                            int len, int sid, int n, const uint32_t key[2], double* logw, int32_t* steps, int cap, int64_t* nst)
{
    const int S = f->n_states;
    const size_t sz = (size_t)(len + 1) * S;
    double* la = malloc(sizeof(double) * sz);
    double* lb = malloc(sizeof(double) * sz);
    for (size_t i = 0; i < sz; ++i) { la[i] = -INFINITY; lb[i] = -INFINITY; }
    la[f->start_state] = 0.0;
    double lq = -INFINITY;
    int el;
    for (int pos = 0; pos <= len; ++pos)
        for (int oi = 0; oi < S; ++oi) {
            const int u = order[oi];
            const double au = la[(size_t)pos * S + u];
            if (au == -INFINITY || u == f->end_state) continue;
            for (int t = f->trans_row[u]; t < f->trans_row[u + 1]; ++t) {
                const int v = f->trans_dst[t];
                const double w = au + ltw[t];
                if (w == -INFINITY) continue;
                if (v == f->end_state) { if (pos == len) lq = logaddexp(lq, w); continue; }
                for (int e = f->emis_row[v]; e < f->emis_row[v + 1]; ++e) {
                    if (!matches(f, tok, len, pos, e, &el)) continue;
                    double* dst = la + (size_t)(pos + el) * S + v;
                    *dst = logaddexp(*dst, w + lew[e]);
                }
            }
        }
    for (int r = 0; r < n; ++r) { logw[r] = -INFINITY; nst[r] = 0; }
    if (lq > -INFINITY && isfinite(lq)) {
        for (int pos = len; pos >= 0; --pos)
            for (int oi = S - 1; oi >= 0; --oi) {
                const int u = order[oi];
                if (la[(size_t)pos * S + u] == -INFINITY || u == f->end_state) continue;
                double bu = -INFINITY;
                for (int t = f->trans_row[u]; t < f->trans_row[u + 1]; ++t) {
                    const int v = f->trans_dst[t];
                    const double w = ltw[t];
                    if (w == -INFINITY) continue;
                    if (v == f->end_state) { if (pos == len) bu = logaddexp(bu, w); continue; }
                    for (int e = f->emis_row[v]; e < f->emis_row[v + 1]; ++e) {
                        if (!matches(f, tok, len, pos, e, &el)) continue;
                        const double bv = lb[(size_t)(pos + el) * S + v];
                        if (bv == -INFINITY) continue;
                        const double term = w + lew[e] + bv;
                        if (term == -INFINITY) continue;
                        bu = logaddexp(bu, term);
                    }
                }
                lb[(size_t)pos * S + u] = bu;
            }
        for (int r = 0; r < n; ++r) {
            int32_t* st = steps + (size_t)r * cap * 2;
            int pos = 0, u = f->start_state, cnt = 0;
            uint32_t d = 0;
            double acc = 0.0;
            for (;;) {
                const double bh = lb[(size_t)pos * S + u];
                double tot = 0.0, thr = 0.0, run = 0.0;
                int ct = -1, ce = -1, cv = -1, cl = 0, pt = -1, pe = -1, pv = -1, pl = 0;
                for (int pass = 0; pass < 2 && ct < 0; ++pass) {
                    if (pass) thr = uniform(d++, (uint32_t)r, (uint32_t)sid, key) * tot;
                    for (int t = f->trans_row[u]; t < f->trans_row[u + 1] && ct < 0; ++t) {
                        const int v = f->trans_dst[t];
                        const double a = ltw[t];
                        if (a == -INFINITY) continue;
                        const int fin = v == f->end_state;
                        if (fin && pos != len) continue;
                        for (int e = fin ? -1 : f->emis_row[v]; e < (fin ? 0 : f->emis_row[v + 1]); ++e) {
                            double term = a;
                            el = 0;
                            if (e >= 0) {
                                if (!matches(f, tok, len, pos, e, &el)) continue;
                                const double bv = lb[(size_t)(pos + el) * S + v];
                                if (bv == -INFINITY) continue;
                                term = a + lew[e] + bv;
                                if (term == -INFINITY) continue;
                            }
                            const double w = exp(term - bh);
                            if (!pass) { tot += w; continue; }
                            if (w > 0.0) { pt = t; pe = e; pv = v; pl = el; }
                            run += w;
                            if (run > thr) { ct = t; ce = e; cv = v; cl = el; break; }
                        }
                    }
                }
                if (ct < 0) { ct = pt; ce = pe; cv = pv; cl = pl; }
                if (ct < 0) break;
                if (cnt < cap) { st[2 * cnt] = ct; st[2 * cnt + 1] = ce; }
                ++cnt;
                acc = acc + ltw[ct];
                if (ce < 0) break;
                acc = acc + lew[ce];
                pos += cl;
                u = cv;
            }
            logw[r] = acc;
            nst[r] = cnt > cap ? -1 : cnt;
        }
    }
    free(la); free(lb);
    return lq > -INFINITY && isfinite(lq) ? lq : -INFINITY;
}

/* logq[s], logw[s * n + r], n_steps[s * n + r] and the steps of draw s * n + r at steps + (s * n + r) * cap * 2 */
int sample_draws(const oracle_fsa* f, const oracle_corpus* c, const double* ltw, const double* lew, int n, uint64_t seed,
                 double* logq, double* logw, int64_t* n_steps, int32_t* steps, int cap, int nthreads)
{
    if (n < 1) return -1;
    const int S = f->n_states;
    int32_t* order = malloc(sizeof(int32_t) * (size_t)(S > 0 ? S : 1));
    state_order(f, order);
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    int nth = nthreads > 0 ? nthreads : 1;
#ifdef _OPENMP
    if (nthreads <= 0) nth = omp_get_max_threads();
#pragma omp parallel for num_threads(nth) schedule(dynamic, 16)
#endif
    for (int64_t s = 0; s < c->n_strings; ++s)
        logq[s] = sample_string(f, order, ltw, lew, c->tokens + c->offsets[s], (int)(c->offsets[s + 1] - c->offsets[s]), (int)s, n,
                                key, logw + (size_t)s * n, steps + (size_t)s * n * cap * 2, cap, n_steps + (size_t)s * n);
    (void)nth;
    free(order);
    return 0;
}
