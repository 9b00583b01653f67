// w-fsa_b200/csrc/kernels_rmin.cuh -- the smallest path posterior (the rmin column of the optimisers) without enumerating
// paths:
//   r_s = min over paths pi of w(pi) / q_s = exp(m_s - log q_s),   m_s = min over paths of sum of log w,
// m_s by a forward sweep in the (min, +) semiring over the lattice of the evaluation: one forward sweep, no backward sweep,
// no accumulators.  Every sweep writes rterm[s] = m_s - log q_s per string; k_min_exp (kernels.cuh) starts its minimum at
// 0 and so caps rmin at 1.  The sweeps work in the log domain without rescaling, and an absent entry (trimmed edge, padding,
// unreachable candidate) is +inf, never log 0 = -inf, which the minimum would pick.
//   k3_minpath          every handle with fast tables (CTA per string, beside K3's alpha recursion for log q)
//   k7_minfwd2          K7's batches (dense automata), with k7_finish_min
//   kg_fwdbwd<MODE_MINPATH> (kernels.cuh) automata without fast tables, with k_rmin_terms
// (Included after the other kernel headers: its kernels are emitted behind theirs, which keeps the layout of the module's
// shared memory declarations, and with it their code, as it was.)
#pragma once
#include "kernels.cuh"
#include "kernels_k7.cuh"

namespace wfsa {

// weights of the (min, +) sweeps: log weights with +inf for an absent edge (trimmed: weight 0), per transition, emission
// and -- with fast tables -- per candidate slot (its emission, its transition to the end state)
__global__ void k_minplus_weights(int n_trans, int n_emis, int n_slots, const int32_t* __restrict__ trans_tp,
                                  const int32_t* __restrict__ emis_tp, const int32_t* __restrict__ slot_emis,
                                  const int32_t* __restrict__ slot_final, const double* __restrict__ x,
                                  double* mtw, double* mew, double* msw, double* mfw)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    auto mw = [&](int tp) { const double l = logweight_of(tp, x, 0); return l > -INFINITY ? l : INFINITY; };
    if (i < n_trans) mtw[i] = mw(trans_tp[i]);
    else if (i < n_trans + n_emis) mew[i - n_trans] = mw(emis_tp[i - n_trans]);
    else if (i < n_trans + n_emis + n_slots) {
        const int s = i - n_trans - n_emis;
        msw[s] = slot_emis[s] < 0 ? 0.0 : mw(emis_tp[slot_emis[s]]);
        mfw[s] = slot_final[s] < 0 ? INFINITY : mw(trans_tp[slot_final[s]]);
    }
}

// rterm[s] = m_s - log q_s for the strings of an order list whose log q is finite (the generic kernel's two launches)
__global__ void k_rmin_terms(long long n, const int32_t* __restrict__ order, const double* __restrict__ m,
                             const double* __restrict__ logq, double* rterm)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int s = order[i];
    if (isfinite(logq[s]) && m[s] < INFINITY) rterm[s] = m[s] - logq[s];
}

// ------------------------------------------------------------------------------------------
// Smallest path posterior of every string, forward only, one CTA per string (thread i <-> candidate slot i):
//   mu_t[j] = log b(j, c_t) + min_k (log a(src_k, j) + mu_{t-1}[src_k]),   m_s = min_j (mu_T[j] + log a(j, end))
// in the log domain without rescaling (the small entries are the answer: a rescaled linear row would lose them), beside
// K3's alpha recursion in K3's order, so that log q_s is the evaluation's to the last bit.  rterm[sid] = m_s - log q_s;
// strings that are not recognised, have a non-finite log q or no choice (the empty string) keep the 0 of the caller.
// Only the fast tables and the per-evaluation weights are read: no lattice slab, any handle with fast tables can run it.
// ------------------------------------------------------------------------------------------
struct K3MinParams {
    FastTablesD T;
    EvalWeightsD W;                       // linear weights of the alpha recursion
    const double* __restrict__ mtw;       // [n_trans] log weights, +inf where absent (k_minplus_weights)
    const double* __restrict__ msw;       // [n_slots] log emission weight of the slot, +inf where absent
    const double* __restrict__ mfw;       // [n_slots] log weight of slot-state -> end, +inf where absent
    CorpusD C;
    double* rterm;                        // [n_strings] m_s - log q_s
};

__global__ void __launch_bounds__(1024, 1) k3_minpath(const K3MinParams P)
{
    extern __shared__ unsigned long long smem[];
    const int nt = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
    double* va = reinterpret_cast<double*>(smem);        // [2][nt] alpha
    double* vm = va + 2 * nt;                            // [2][nt] mu
    double* red = vm + 2 * nt;                           // [32] q parts, [32] min parts
    int* ired = reinterpret_cast<int*>(red + 64);        // [32]
    const FastTablesD& T = P.T;
    const int A = T.n_sym;

    for (long long it = blockIdx.x; it < P.C.n_order; it += gridDim.x) {
        const int sid = P.C.order[it];
        const long long off = P.C.offs[sid];
        const int len = (int)(P.C.offs[sid + 1] - off);
        const int32_t* tok = P.C.tokens + off;
        __syncthreads();
        if (len == 0) continue;                          // one path (start -> end): r = 1
        int cur = 0, E = 0, cprev = A;
        bool dead = false, valid = false;
        va[tid] = (tid == 0) ? 1.0 : 0.0;
        vm[tid] = (tid == 0) ? 0.0 : INFINITY;
        __syncthreads();
        uint32_t slot = 0;
        double alpha = 0.0, mu = INFINITY;
        for (int t = 0; t < len; ++t) {
            const int c = tok[t];
            if ((unsigned)c >= (unsigned)A) { dead = true; break; }
            const uint32_t c0 = T.cand_off[c], ncand = T.cand_off[c + 1] - c0;
            valid = (uint32_t)tid < ncand;
            slot = c0 + tid;
            alpha = 0.0; mu = INFINITY;
            if (valid) {
                const uint32_t row = T.frow[(size_t)T.slot_state[slot] * (A + 1) + cprev];
                const int cnt = row & ((1u << kRowCntBitsD) - 1);
                const uint32_t st = row >> kRowCntBitsD;
                const double* src = va + cur * nt;
                const double* msrc = vm + cur * nt;
                double s = 0.0, m = INFINITY;
                for (int k = 0; k < cnt; ++k) {
                    const uint32_t ent = T.fent[st + k];
                    const uint32_t tr = ent >> kSlotBitsD, sl = ent & ((1u << kSlotBitsD) - 1);
                    s = fma(P.W.tw[tr], src[sl], s);
                    m = fmin(m, P.mtw[tr] + msrc[sl]);
                }
                alpha = s * P.W.sw[slot];
                mu = m + P.msw[slot];
            }
            const bool chk = (t & (kRescaleEvery - 1)) == kRescaleEvery - 1;
            const int e = alpha != 0.0 ? biased_exp(alpha) : -1;
            const int wmax = __reduce_max_sync(FULL, e);
            if (lane == 0) ired[warp] = wmax;
            __syncthreads();
            int emax = -1;
            for (int w = 0; w < nwarps; ++w) emax = max(emax, ired[w]);
            if (emax < 0) { dead = true; break; }
            if (chk && (emax < 1023 - kRescaleBand || emax > 1023 + kRescaleBand)) {
                const int shift = 1023 - emax;
                alpha = scalbn(alpha, shift);
                E -= shift;
            }
            va[(cur ^ 1) * nt + tid] = alpha;
            vm[(cur ^ 1) * nt + tid] = mu;
            cur ^= 1;
            cprev = c;
            __syncthreads();
        }
        if (dead) continue;
        const double fin = (alpha != 0.0) ? P.W.fw[slot] : 0.0;
        const double part = warp_sum(alpha * fin);
        double mf = (valid && mu < INFINITY) ? mu + P.mfw[slot] : INFINITY;
#pragma unroll
        for (int o = 16; o; o >>= 1) mf = fmin(mf, __shfl_xor_sync(FULL, mf, o));
        if (lane == 0) { red[warp] = part; red[32 + warp] = mf; }
        __syncthreads();
        if (tid == 0) {
            double qh = 0.0, m = INFINITY;
            for (int w = 0; w < nwarps; ++w) { qh += red[w]; m = fmin(m, red[32 + w]); }    // q: K3's order
            if (qh > 0.0 && isfinite(qh) && m < INFINITY) P.rterm[sid] = m - (log(qh) + (double)E * 0.69314718055994530942);
        }
    }
}

// ---- K7: the forward step of k7_fwd2 in (min, +) -------------------------------------------------------------------------
//   mu_t[j] = log b(j, c_t) + min_k (log a(src_k, j) + mu_{t-1}[src_k])
// Log domain and no rescaling (a rescaled linear row keeps its largest entries and lets the small ones, the answer here,
// underflow); absent entries are +inf: trimmed edges, the padding entries kK7Sent, unreachable candidates.  mu needs only
// the previous row: the rows ping-pong in two buffers of k7_nb x V, row r = batch-local string r.
struct K7MinParams {
    FastTablesD T;
    const K7Desc* __restrict__ desc;
    const int32_t* __restrict__ perm;
    const double* src;                       // mu_{t-1} rows [r][V]
    double* dst;                             // mu_t rows
    const double* __restrict__ mtw;          // [n_trans] log weights, +inf where absent (k_minplus_weights)
    const double* __restrict__ msw;          // [n_slots]
    const uint32_t* __restrict__ pe;         // forward pair planes (K7Params::pe)
    const uint32_t* __restrict__ pr;
    int V;
};

template <int MAXV, int MINB>
__global__ void __launch_bounds__(MAXV, MINB) k7_minfwd2(const K7MinParams P)
{
    extern __shared__ double k7_tile[];                     // [kK7Chunk][V]
    __shared__ int s_r[kK7Chunk];
    const FastTablesD& T = P.T;
    const int V = P.V, j = threadIdx.x, A = T.n_sym;
    const K7Desc d = P.desc[blockIdx.x];
    const size_t key = (size_t)d.cp * A + d.c;
    if (j < d.cnt) s_r[j] = P.perm[d.start + j];
    uint32_t ent[kK7Planes];
#pragma unroll
    for (int k = 0; k < kK7Planes; ++k) ent[k] = k < d.kf ? P.pe[(key * kK7Planes + k) * V + j] : kK7Sent;
    const uint32_t row = P.pr[key * V + j];
    const double swj = P.msw[min(d.c0c + j, T.n_slots - 1)];     // (beyond the candidates every entry is padding: +inf)
    __syncthreads();
    if (d.cp == A) {
        for (int i = 0; i < d.cnt; ++i) k7_tile[i * V + j] = j == 0 ? 0.0 : INFINITY;
    } else {
        for (int i = 0; i < d.cnt; ++i) k7_cp_async8(k7_tile + i * V + j, P.src + (size_t)s_r[i] * V + j);
    }
    double w[kK7Planes];
    unsigned int off[kK7Planes];
#pragma unroll
    for (int k = 0; k < kK7Planes; ++k) {
        w[k] = (ent[k] >> kSlotBitsD) != (kK7Sent >> kSlotBitsD) ? P.mtw[ent[k] >> kSlotBitsD] : INFINITY;
        off[k] = (ent[k] & ((1u << kSlotBitsD) - 1)) * 8u;
    }
    const int cnt = row & ((1u << kRowCntBitsD) - 1);
    const uint32_t st = row >> kRowCntBitsD;
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
    const char* tile = reinterpret_cast<const char*>(k7_tile);
    const unsigned int rowb = (unsigned int)V * 8u;
    for (int i = 0; i < d.cnt; ++i) {
        const char* sv = tile + (unsigned int)i * rowb;
        double m = INFINITY;
#pragma unroll
        for (int k = 0; k < kK7Planes; ++k) m = fmin(m, w[k] + k7_lds(sv, off[k]));
        for (int k = kK7Planes; k < cnt; ++k) {
            const uint32_t e = T.fent[st + k];
            m = fmin(m, P.mtw[e >> kSlotBitsD] + k7_lds(sv, (e & ((1u << kSlotBitsD) - 1)) * 8u));
        }
        P.dst[(size_t)s_r[i] * V + j] = m + swj;
    }
}

// strings whose last position is t: m_s = min_u (mu_t[u] + log a(u, end)), rterm[sid] = m_s - log q_s (log q from
// k7_finish_q of the same step); one warp per string
struct K7MinFinParams {
    FastTablesD T;
    const int32_t* __restrict__ sid;
    const int32_t* __restrict__ last_tok;
    const double* __restrict__ mu;           // mu_t rows
    const double* __restrict__ mfw;          // [n_slots] log final weight, +inf where absent
    const double* __restrict__ logq;         // [n_strings]
    double* rterm;                           // [n_strings]
    int r0, r1, V;
};

__global__ void __launch_bounds__(256) k7_finish_min(const K7MinFinParams P)
{
    const int lane = threadIdx.x & 31;
    const int r = P.r0 + (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (r >= P.r1) return;
    const int c = P.last_tok[r], sid = P.sid[r];
    const uint32_t c0 = P.T.cand_off[c], ncand = P.T.cand_off[c + 1] - c0;
    double m = INFINITY;
    for (int jj = lane; (uint32_t)jj < ncand; jj += 32) m = fmin(m, P.mu[(size_t)r * P.V + jj] + P.mfw[c0 + jj]);
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmin(m, __shfl_xor_sync(FULL, m, o));
    if (lane == 0) {
        const double lq = P.logq[sid];
        if (isfinite(lq) && m < INFINITY) P.rterm[sid] = m - lq;
    }
}

}  // namespace wfsa
