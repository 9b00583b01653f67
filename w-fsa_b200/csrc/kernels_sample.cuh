// w-fsa_b200/csrc/kernels_sample.cuh -- n independent draws from the path posterior of every string (sampling):
//   p(pi | s) = w(pi) / q_s
// by a forward sweep that keeps its lattice, then a walk through it per draw that picks every step in proportion to the
// weight of the paths through it.  Randomness is Philox4x32-10 (philox.hpp), counter (d, r, s, 0) for choice d of draw r of
// string s, so a draw does not depend on the grid, the group or the other draws.  Choice rule at a node: the first entry, in
// table order, whose running sum exceeds u * total; when rounding leaves none, the last entry of positive weight.  logw of a
// draw is the left-to-right sum of the log weights of its steps, in wfsa_dev_viterbi's order, bit for bit.
//   k3_sample<WARP>   every handle with fast tables: K3's alpha recursion (so log q is K3's to the last bit), the scaled
//                     alpha rows kept in a per-group slab, then a walk back from the end per draw
//   kg_sample         automata without fast tables, thread per string: the evaluation's log-domain forward and backward,
//                     then forward sampling from the start state
// (Included last, after kernels_nbest.cuh, for the reason given in kernels_rmin.cuh.)
#pragma once
#include "kernels_nbest.cuh"
#include "philox.hpp"

namespace wfsa {

constexpr int kSampleMax = 256;            // most draws per string and call

// ------------------------------------------------------------------------------------------
// Fast tables: a group of threads per string as k3_viterbi (thread g <-> candidate slot g).  The forward sweep is K3's:
// alpha_t[j] = sw[j] * fma chain of tw * alpha_{t-1}[src] over the fent entries, with K3's lazy power-of-two rescale; every
// row of alpha goes to the group's slab [max_len][pitch] (doubles, reused string by string).  The entries of a row share one
// scale, so the walk needs no exponents.  Draw r runs on thread r mod G: choice 0 picks the last slot j among
// alpha_{T-1}[j] * fw[j] in slot order, choice len - t the fent entry of position t among tw * alpha_{t-1}[src] (alpha_{-1}
// = the start row: 1 at slot 0).  Draw r of string s is written at n * (offs[s] + s) + r * (len + 1).
// ------------------------------------------------------------------------------------------
struct K3SampleParams {
    FastTablesD T;
    EvalWeightsD W;                          // linear weights from the call's x (k_weights)
    const double* __restrict__ vtw;          // [n_trans] log weights, -inf where absent (k_maxplus_weights)
    const double* __restrict__ vew;          // [n_emis]
    const int32_t* __restrict__ slot_emis;   // [n_slots] emission edge of the slot
    const int32_t* __restrict__ slot_final;  // [n_slots] transition edge slot-state -> end, or -1
    CorpusD C;
    double* slab;                            // [groups][max_len][pitch] alpha rows
    int pitch;                               // candidates per slab row: 32 (WARP) or blockDim.x
    int max_len;
    int n;                                   // draws per string
    uint32_t key0, key1;                     // Philox key: seed & 0xffffffff, seed >> 32
    double* logw;                            // [n_strings * n]
    double* logq;                            // [n_strings]
    int32_t* trans_edge;                     // [n * (n_tokens + n_strings)]
    int32_t* emis_edge;
};

template <bool WARP>
__global__ void __launch_bounds__(WARP ? 256 : 1024, WARP ? 3 : 1) k3_sample(const K3SampleParams P)
{
    extern __shared__ unsigned long long smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int g = WARP ? lane : tid;                                          // candidate of this thread
    const int G = WARP ? 32 : (int)blockDim.x;
    double* va = reinterpret_cast<double*>(smem) + (WARP ? warp * 64 : 0);    // [2][G] alpha of the group
    double* red = reinterpret_cast<double*>(smem) + 2 * blockDim.x;           // [32] (CTA) q parts of the warps
    int* ired = reinterpret_cast<int*>(red + 32);                             // [32] their largest exponents
    const FastTablesD& T = P.T;
    const int A = T.n_sym;
    const uint32_t key[2] = {P.key0, P.key1};
    const long long grp = WARP ? (long long)blockIdx.x * nwarps + warp : blockIdx.x;
    const long long n_grp = WARP ? (long long)gridDim.x * nwarps : gridDim.x;
    double* slab = P.slab + (size_t)grp * P.max_len * P.pitch;

    for (long long it = grp; it < P.C.n_order; it += n_grp) {
        const int sid = P.C.order[it];
        const long long off = P.C.offs[sid];
        const int len = (int)(P.C.offs[sid + 1] - off);
        const int32_t* tok = P.C.tokens + off;
        const long long out = (long long)P.n * (off + sid);
        vit_sync<WARP>();                                   // the previous walk has read the slab
        if (len == 0) {                                     // one path: start -> end
            const double q = T.start_final_tid >= 0 ? P.W.tw[T.start_final_tid] : 0.0;
            if (g == 0) P.logq[sid] = log(q);
            if (q > 0.0 && q < INFINITY)
                for (int r = g; r < P.n; r += G) {
                    P.logw[(long long)sid * P.n + r] = 0.0 + P.vtw[T.start_final_tid];
                    P.trans_edge[out + r] = T.start_final_tid; P.emis_edge[out + r] = -1;
                }
            continue;
        }
        // ---------------- forward: K3's alpha recursion, every row to the slab ----------------
        int cur = 0, E = 0, cprev = A;
        bool dead = false;
        va[g] = (g == 0) ? 1.0 : 0.0;
        vit_sync<WARP>();
        uint32_t slot = 0;
        double alpha = 0.0;
        for (int t = 0; t < len; ++t) {
            const int c = tok[t];
            if ((unsigned)c >= (unsigned)A) { dead = true; break; }          // (uniform over the group)
            const uint32_t c0 = T.cand_off[c], ncand = T.cand_off[c + 1] - c0;
            slot = c0 + g;
            alpha = 0.0;
            if ((uint32_t)g < ncand) {
                const uint32_t row = T.frow[(size_t)T.slot_state[slot] * (A + 1) + cprev];
                const int cnt = row & ((1u << kRowCntBitsD) - 1);
                const uint32_t st = row >> kRowCntBitsD;
                const double* src = va + cur * G;
                double s = 0.0;
                for (int k = 0; k < cnt; ++k) {
                    const uint32_t ent = T.fent[st + k];
                    s = fma(P.W.tw[ent >> kSlotBitsD], src[ent & ((1u << kSlotBitsD) - 1)], s);
                }
                alpha = s * P.W.sw[slot];
            }
            const bool chk = (t & (kRescaleEvery - 1)) == kRescaleEvery - 1;
            int emax = __reduce_max_sync(FULL, alpha != 0.0 ? biased_exp(alpha) : -1);
            if (!WARP) {
                if (lane == 0) ired[warp] = emax;
                __syncthreads();
                emax = -1;
                for (int w = 0; w < nwarps; ++w) emax = max(emax, ired[w]);
            }
            if (emax < 0) { dead = true; break; }
            if (chk && (emax < 1023 - kRescaleBand || emax > 1023 + kRescaleBand)) {
                const int shift = 1023 - emax;
                alpha = scalbn(alpha, shift);
                E -= shift;
            }
            va[(cur ^ 1) * G + g] = alpha;
            slab[(size_t)t * P.pitch + g] = alpha;
            cur ^= 1;
            cprev = c;
            vit_sync<WARP>();
        }
        // q in K3's order: the warps' sums of alpha * fw, added in warp order (a warp group is K3's first warp)
        double qh = 0.0;
        if (!dead) {
            const double fin = (alpha != 0.0) ? P.W.fw[slot] : 0.0;
            const double part = warp_sum(alpha * fin);
            if (WARP) qh += part;
            else {
                if (lane == 0) red[warp] = part;
                __syncthreads();
                for (int w = 0; w < nwarps; ++w) qh += red[w];
            }
        }
        const bool ok = !dead && qh > 0.0 && isfinite(qh);
        if (g == 0) P.logq[sid] = ok ? log(qh) + (double)E * 0.69314718055994530942 : -INFINITY;
        if (!ok) continue;
        // ---------------- the walks: draw r on thread r mod G ----------------
        const uint32_t cl = T.cand_off[tok[len - 1]], nl = T.cand_off[tok[len - 1] + 1] - cl;
        const double* last = slab + (size_t)(len - 1) * P.pitch;
        for (int r = g; r < P.n; r += G) {
            const long long o = out + (long long)r * (len + 1);
            uint32_t d = 0;
            // the end: a slot among alpha_{T-1}[j] * fw[j]
            double tot = 0.0;
            for (uint32_t j = 0; j < nl; ++j) tot += last[j] * P.W.fw[cl + j];
            double thr = philox_uniform(d++, (uint32_t)r, (uint32_t)sid, key) * tot, run = 0.0;
            int j = -1, jpos = 0;
            for (uint32_t i = 0; i < nl; ++i) {
                const double w = last[i] * P.W.fw[cl + i];
                if (last[i] > 0.0 && P.W.fw[cl + i] > 0.0) jpos = (int)i;
                run += w;
                if (run > thr) { j = (int)i; break; }
            }
            if (j < 0) j = jpos;
            P.trans_edge[o + len] = P.slot_final[cl + j];
            P.emis_edge[o + len] = -1;
            // position t: a fent entry of the candidate among tw * alpha_{t-1}[src]
            uint32_t c0 = cl;
            for (int t = len - 1; t >= 0; --t) {
                const uint32_t sl = c0 + j;
                const int cp = t ? tok[t - 1] : A;
                const uint32_t row = T.frow[(size_t)T.slot_state[sl] * (A + 1) + cp];
                const int cnt = row & ((1u << kRowCntBitsD) - 1);
                const uint32_t st = row >> kRowCntBitsD;
                const double* prev = slab + (size_t)(t ? t - 1 : 0) * P.pitch;
                auto src = [&](uint32_t ent) {
                    const uint32_t q = ent & ((1u << kSlotBitsD) - 1);
                    return t ? prev[q] : (q == 0 ? 1.0 : 0.0);
                };
                double s = 0.0;
                for (int k = 0; k < cnt; ++k) { const uint32_t ent = T.fent[st + k]; s = fma(P.W.tw[ent >> kSlotBitsD], src(ent), s); }
                thr = philox_uniform(d++, (uint32_t)r, (uint32_t)sid, key) * s;
                run = 0.0;
                int kb = -1, kpos = 0;
                for (int k = 0; k < cnt; ++k) {
                    const uint32_t ent = T.fent[st + k];
                    const double tw = P.W.tw[ent >> kSlotBitsD], a = src(ent);
                    if (tw > 0.0 && a > 0.0) kpos = k;
                    run = fma(tw, a, run);
                    if (run > thr) { kb = k; break; }
                }
                const uint32_t ent = T.fent[st + (kb < 0 ? kpos : kb)];
                P.trans_edge[o + t] = (int32_t)(ent >> kSlotBitsD);
                P.emis_edge[o + t] = P.slot_emis[sl];
                j = (int)(ent & ((1u << kSlotBitsD) - 1));
                c0 = T.cand_off[cp];
            }
            // logw: the steps' log weights left to right, as wfsa_dev_viterbi adds them
            double acc = 0.0;
            for (int t = 0; t < len; ++t) {
                const int32_t e = P.emis_edge[o + t];
                acc = (P.vtw[P.trans_edge[o + t]] + acc) + (e < 0 ? 0.0 : P.vew[e]);
            }
            P.logw[(long long)sid * P.n + r] = acc + P.vtw[P.trans_edge[o + len]];
        }
    }
}

// ------------------------------------------------------------------------------------------
// No fast tables: one thread per string.  The log-domain forward and backward of kg_fwdbwd<MODE_EVAL> in the thread's
// scratch (without accumulators): la gives log q, lb[pos][u] = beta, the log weight of the continuations of node (pos, u).
// Then every draw walks forward from (0, start): at (pos, u) the entries are, in table order, every transition t of u with
// every emission e of its target that matches the string at pos (weight exp(((log a + log b) + beta_next) - beta_here)),
// and at pos = len the transitions into the end state (weight exp(log a - beta_here)); choice d is the d-th step.  As
// kg_fwdbwd<MODE_VITERBI>, a first launch (vit_off == nullptr) writes the step count of draw s * n + r to vit_cnt, a second
// one, which repeats the same draws, writes the steps from vit_off.  logw goes to O.logq[s * n + r], log q to logq[s].
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) kg_sample(const GenericParams P, int n, uint32_t key0, uint32_t key1, double* logq)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.count) return;
    const GenericTablesD& G = P.G;
    const int S = G.n_states;
    const int sid = P.C.order[P.first + i];
    const long long off = P.C.offs[sid];
    const int len = (int)(P.C.offs[sid + 1] - off);
    const int32_t* tok = P.C.tokens + off;
    const size_t lat_sz = (size_t)(P.max_len + 1) * S;
    double* la = P.scratch + (size_t)i * 2 * lat_sz;
    double* lb = la + lat_sz;
    for (size_t k = 0; k < (size_t)(len + 1) * S; ++k) { la[k] = -INFINITY; lb[k] = -INFINITY; }
    la[G.start_state] = 0.0;
    double lq = -INFINITY;
    // forward (kg_fwdbwd<MODE_EVAL>'s order: log q is the evaluation's)
    for (int pos = 0; pos <= len; ++pos) {
        for (int oi = 0; oi < S; ++oi) {
            const int u = G.eps_order[oi];
            const double au = la[(size_t)pos * S + u];
            if (au == -INFINITY || u == G.end_state) continue;
            for (int t = G.trans_row[u]; t < G.trans_row[u + 1]; ++t) {
                const int v = G.trans_dst[t];
                const double w = au + P.ltw[t];
                if (w == -INFINITY) continue;
                if (v == G.end_state) {
                    if (pos == len) lq = logaddexp_d(lq, w);
                    continue;
                }
                for (int e = G.emis_row[v]; e < G.emis_row[v + 1]; ++e) {
                    const int e0 = G.emis_tok_off[e], el = G.emis_tok_off[e + 1] - e0;
                    if (pos + el > len) continue;
                    bool m = true;
                    for (int k = 0; k < el; ++k) if (tok[pos + k] != G.emis_tok[e0 + k]) { m = false; break; }
                    if (!m) continue;
                    double* dst = la + (size_t)(pos + el) * S + v;
                    *dst = logaddexp_d(*dst, w + P.lew[e]);
                }
            }
        }
    }
    const bool ok = lq > -INFINITY && isfinite(lq);
    if (!P.vit_off) logq[sid] = ok ? lq : -INFINITY;
    if (!ok) {
        if (!P.vit_off) for (int r = 0; r < n; ++r) P.vit_cnt[(long long)sid * n + r] = 0;
        return;
    }
    // backward: beta of every node the forward reached (kg_fwdbwd<MODE_EVAL>'s order)
    for (int pos = len; pos >= 0; --pos) {
        for (int oi = S - 1; oi >= 0; --oi) {
            const int u = G.eps_order[oi];
            if (la[(size_t)pos * S + u] == -INFINITY || u == G.end_state) continue;
            double bu = -INFINITY;
            for (int t = G.trans_row[u]; t < G.trans_row[u + 1]; ++t) {
                const int v = G.trans_dst[t];
                const double w = P.ltw[t];
                if (w == -INFINITY) continue;
                if (v == G.end_state) {
                    if (pos == len) bu = logaddexp_d(bu, w);
                    continue;
                }
                for (int e = G.emis_row[v]; e < G.emis_row[v + 1]; ++e) {
                    const int e0 = G.emis_tok_off[e], el = G.emis_tok_off[e + 1] - e0;
                    if (pos + el > len) continue;
                    bool m = true;
                    for (int k = 0; k < el; ++k) if (tok[pos + k] != G.emis_tok[e0 + k]) { m = false; break; }
                    if (!m) continue;
                    const double bv = lb[(size_t)(pos + el) * S + v];
                    if (bv == -INFINITY) continue;
                    const double term = w + P.lew[e] + bv;
                    if (term == -INFINITY) continue;
                    bu = logaddexp_d(bu, term);
                }
            }
            lb[(size_t)pos * S + u] = bu;
        }
    }
    // the draws
    const uint32_t key[2] = {key0, key1};
    for (int r = 0; r < n; ++r) {
        const long long q = (long long)sid * n + r;
        int64_t o = P.vit_off ? P.vit_off[q] : 0;
        int pos = 0, u = G.start_state, cnt = 0;
        uint32_t d = 0;
        double acc = 0.0;
        for (;;) {
            // two passes over the entries of node (pos, u): their total, then the choice
            const double bh = lb[(size_t)pos * S + u];
            double tot = 0.0, thr = 0.0, run = 0.0;
            int ct = -1, ce = -1, cv = -1, cl = 0, pt = -1, pe = -1, pv = -1, pl = 0;
            for (int pass = 0; pass < 2; ++pass) {
                if (pass) thr = philox_uniform(d++, (uint32_t)r, (uint32_t)sid, key) * tot;
                for (int t = G.trans_row[u]; t < G.trans_row[u + 1]; ++t) {
                    const int v = G.trans_dst[t];
                    const double a = P.ltw[t];
                    if (a == -INFINITY || (v == G.end_state && pos != len)) continue;
                    for (int e = v == G.end_state ? -1 : G.emis_row[v]; e < (v == G.end_state ? 0 : G.emis_row[v + 1]); ++e) {
                        int el = 0;
                        double term = a;
                        if (e >= 0) {
                            const int e0 = G.emis_tok_off[e];
                            el = G.emis_tok_off[e + 1] - e0;
                            if (pos + el > len) continue;
                            bool m = true;
                            for (int k = 0; k < el; ++k) if (tok[pos + k] != G.emis_tok[e0 + k]) { m = false; break; }
                            if (!m) continue;
                            const double bv = lb[(size_t)(pos + el) * S + v];
                            if (bv == -INFINITY) continue;
                            term = a + P.lew[e] + bv;
                            if (term == -INFINITY) continue;
                        }
                        const double w = exp(term - bh);
                        if (!pass) { tot += w; continue; }
                        if (w > 0.0) { pt = t; pe = e; pv = v; pl = el; }
                        run += w;
                        if (run > thr) { ct = t; ce = e; cv = v; cl = el; goto chosen; }
                    }
                }
            }
            ct = pt; ce = pe; cv = pv; cl = pl;
        chosen:
            if (ct < 0) break;                       // (no entry of positive weight: cannot happen on a node of a path)
            if (P.vit_off) { P.vit_trans[o] = ct; P.vit_emis[o] = ce; ++o; }
            ++cnt;
            acc = acc + P.ltw[ct];
            if (ce < 0) break;
            acc = acc + P.lew[ce];
            pos += cl;
            u = cv;
        }
        if (!P.vit_off) { P.vit_cnt[q] = cnt; P.O.logq[q] = acc; }
    }
}

}  // namespace wfsa
