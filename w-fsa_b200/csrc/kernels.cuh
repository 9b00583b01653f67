// w-fsa_b200/csrc/kernels.cuh -- sm_100a kernels of the w-fsa evaluation backend.
//
// What they compute (SURVEY.md Appendix A; the reference obtains the same numbers by path
// enumeration + sparse algebra, /root/reference/src/Learner.cpp:515-553,
// src/QuasiNewtonLearner.cpp:93-125):
//   alpha_t[v] = b(v,c_t) * sum_u a(u,v) alpha_{t-1}[u]          forward
//   q          = sum_u alpha_{T-1}[u] a(u,end)
//   beta~_t[u] = b(u,c_t) * sum_v a(u,v) beta~_{t+1}[v]           backward (beta~ carries b)
//   gamma(u->v at t) = alpha_t[u] a(u,v) beta~_{t+1}[v] / q       posterior of a combined arc
//   acc[arc] += p_s * gamma          (64-bit fixed point => order independent, bitwise
//                                     reproducible for any grid size and any number of GPUs)
// All arithmetic is FP64 in the linear domain with lazy power-of-two rescaling (exact),
// so results equal the unscaled computation bit for bit whenever that would not under/overflow.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace wfsa {

constexpr unsigned FULL = 0xffffffffu;
constexpr int kSlotBitsD = 10;
constexpr int kRowCntBitsD = 8;
constexpr int kRescaleEvery = 4;       // positions between exponent checks
constexpr int kRescaleBand = 300;      // rescale when the largest entry leaves 2^(+-300)

enum { MODE_EVAL = 0, MODE_STRUCT = 1, MODE_MINPATH = 2 /* generic kernel: forward only, in (min, +) */,
       MODE_VITERBI = 3 /* generic kernel: forward in (max, +) with backpointers, traceback */ };
enum { ACC_SMEM_CAS = 0, ACC_SMEM_SPLIT = 1, ACC_GLOBAL = 2, ACC_NONE = 3 /* timing experiments only */ };

struct FastTablesD {
    const uint32_t* __restrict__ cand_off;    // [n_sym+2]
    const uint32_t* __restrict__ slot_state;  // [n_slots]
    const uint32_t* __restrict__ frow;        // [n_states*(n_sym+1)]
    const uint32_t* __restrict__ fent;
    const uint32_t* __restrict__ brow;        // [n_states*n_sym]
    const uint32_t* __restrict__ bent;
    int n_sym, n_states, n_arcs, n_slots, start_state, start_final_tid;
};

struct EvalWeightsD {
    const double* __restrict__ tw;   // [n_trans] transition weights
    const double* __restrict__ sw;   // [n_slots] emission weight of the slot
    const double* __restrict__ fw;   // [n_slots] weight of slot-state -> end (0 if none)
};

struct CorpusD {
    const int32_t* __restrict__ tokens;
    const int64_t* __restrict__ offs;     // [n_strings+1]
    const double* __restrict__ p;         // [n_strings]
    const int32_t* __restrict__ order;    // [n_order] string ids, longest first
    int64_t n_order;
};

struct EvalOutD {
    double* logq;                    // [n_strings] (string id order) or nullptr
    double* path_count;              // MODE_STRUCT: [n_strings]
    unsigned long long* acc_global;  // [n_arcs + n_slots] combined-arc / final-transition accumulators
    unsigned long long* red;         // red[0] = fixed-point loglik, red[1] = non-finite strings,
                                     // red[2 + e] = per-edge accumulators
    double fx_scale;                 // 2^k fixed-point scale of the accumulators
    double ll_scale;                 // fixed-point scale of loglik
};

// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
__device__ __forceinline__ int biased_exp(double a) { return (__double2hiint(a) >> 20) & 0x7ff; }

template <int ACC>
__device__ __forceinline__ void acc_add(unsigned long long* acc_s, unsigned long long* acc_g, int idx, long long v)
{
    if (v == 0 || ACC == ACC_NONE) return;
    if (ACC == ACC_GLOBAL) {
        atomicAdd(acc_g + idx, (unsigned long long)v);                       // REDG.E.ADD.64
    } else if (ACC == ACC_SMEM_CAS) {
        atomicAdd(acc_s + idx, (unsigned long long)v);                       // ATOMS.CAS.64 loop
    } else {
        // exact 64-bit add out of two native 32-bit shared atomics (carry from the returned word)
        unsigned* w = reinterpret_cast<unsigned*>(acc_s + idx);
        const unsigned lo = (unsigned)v, hi = (unsigned)((unsigned long long)v >> 32);
        const unsigned old = atomicAdd(w, lo);
        const unsigned add_hi = hi + ((old + lo < old) ? 1u : 0u);
        if (add_hi) atomicAdd(w + 1, add_hi);
    }
}

__device__ __forceinline__ void stack_st(unsigned long long* s, unsigned long long* g, int cap, int i, unsigned long long v)
{
    if (i < cap) s[i] = v; else g[i - cap] = v;
}
__device__ __forceinline__ unsigned long long stack_ld(const unsigned long long* s, const unsigned long long* g, int cap, int i)
{
    return (i < cap) ? s[i] : g[i - cap];
}

struct WarpTablesD {
    const uint16_t* __restrict__ brow;        // [n_states*n_sym + 1] row starts of (state, next symbol)
    const uint8_t* __restrict__ bent;         // [n_arcs] target slot inside E[c_next]
    const uint16_t* __restrict__ slot_state;  // [n_slots]
    const uint32_t* __restrict__ cand_off;    // [n_sym+2]
    const double* __restrict__ aw;            // [n_arcs]  a(u,v) * b(v,c_next), recomputed per evaluation
    const double* __restrict__ fw;            // [n_slots] a(state of slot, end), 0 if none
    int n_sym, n_states, n_arcs, n_slots, start_state, start_final_tid;
};

struct K2Params {
    WarpTablesD T;
    const double* __restrict__ tw;   // only for the empty string (start -> end)
    CorpusD C;
    EvalOutD O;
    int n_acc_smem;                  // accumulators kept in shared memory (0 => ACC_GLOBAL)
    int stack_cap;                   // lattice stack words per warp in shared memory
    unsigned long long* gl_stack;    // overflow of the lattice stacks
    size_t gl_stack_words;           // per warp
    int replicas;                    // copies of the global accumulators (CTA b uses copy b % replicas)
};

// byte layout of the staged tables: aw | fw | cand_off | brow | slot_state | bent  (each 8-byte aligned)
struct K2TableLayout { size_t aw, fw, coff, brow, sstate, bent, total; };
__host__ __device__ inline K2TableLayout k2_table_layout(int n_sym, int n_states, int n_arcs, int n_slots)
{
    K2TableLayout t;
    size_t o = 0;
    auto al = [](size_t v) { return (v + 7) & ~(size_t)7; };
    t.aw = o; o += (size_t)n_arcs * 8;
    t.fw = o; o += (size_t)n_slots * 8;
    t.coff = o; o = al(o + ((size_t)n_sym + 2) * 4);
    t.brow = o; o = al(o + ((size_t)n_states * n_sym + 1) * 2);
    t.sstate = o; o = al(o + (size_t)n_slots * 2);
    t.bent = o; o = al(o + (size_t)n_arcs);
    t.total = o;
    return t;
}

// ------------------------------------------------------------------------------------------
// K2: one warp per string.  Lane j <-> j-th candidate (state emitting the current symbol, at most
// 32 of them); alpha / beta live in registers.
//   forward : the few ACTIVE source lanes (ballot mask, ~2 for config 4) scatter along their
//             (state, next symbol) CSR row; one shuffle pair per source;
//   backward: every active lane gathers beta over its own row through shuffles and adds the arc
//             posteriors to the per-arc accumulators.
// The automaton (16-bit CSR rows, 8-bit targets, per-arc weights, final weights) is staged once
// per CTA into shared memory next to the per-arc accumulators and the per-warp lattice stacks.
// ------------------------------------------------------------------------------------------
template <int MODE, int ACC, int TABS>
__global__ void __launch_bounds__(1024, 1) k2_fwdbwd(const K2Params P)
{
    extern __shared__ unsigned long long smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int A = P.T.n_sym, NA = P.T.n_arcs, NS = P.T.n_slots;
    unsigned long long* acc_s = smem;
    unsigned long long* sp_base = smem + P.n_acc_smem;
    const double* aw = P.T.aw;
    const double* fw = P.T.fw;
    const uint16_t* brow = P.T.brow;
    const uint8_t* bent = P.T.bent;
    const uint16_t* slot_state = P.T.slot_state;
    const uint32_t* cand_off = P.T.cand_off;
    if (TABS) {
        const K2TableLayout tl = k2_table_layout(A, P.T.n_states, NA, NS);
        unsigned char* base = reinterpret_cast<unsigned char*>(sp_base);
        double* s_aw = reinterpret_cast<double*>(base + tl.aw);
        double* s_fw = reinterpret_cast<double*>(base + tl.fw);
        uint32_t* s_coff = reinterpret_cast<uint32_t*>(base + tl.coff);
        uint16_t* s_brow = reinterpret_cast<uint16_t*>(base + tl.brow);
        uint16_t* s_ss = reinterpret_cast<uint16_t*>(base + tl.sstate);
        uint8_t* s_bent = base + tl.bent;
        const int n_row = P.T.n_states * A + 1;
        for (int i = threadIdx.x; i < NA; i += blockDim.x) { s_aw[i] = aw[i]; s_bent[i] = bent[i]; }
        for (int i = threadIdx.x; i < NS; i += blockDim.x) { s_fw[i] = fw[i]; s_ss[i] = slot_state[i]; }
        for (int i = threadIdx.x; i < n_row; i += blockDim.x) s_brow[i] = brow[i];
        for (int i = threadIdx.x; i < A + 2; i += blockDim.x) s_coff[i] = cand_off[i];
        aw = s_aw; fw = s_fw; brow = s_brow; bent = s_bent; slot_state = s_ss; cand_off = s_coff;
        sp_base += tl.total / 8;
    }
    unsigned long long* stack = sp_base + (size_t)warp * P.stack_cap;
    const long long gw = (long long)blockIdx.x * nwarps + warp, GW = (long long)gridDim.x * nwarps;
    unsigned long long* gstack = P.gl_stack + (size_t)gw * P.gl_stack_words;
    const int cap = P.stack_cap;
    unsigned long long* const acc_g = P.O.acc_global + (size_t)(blockIdx.x % P.replicas) * (size_t)(NA + P.T.n_states);
    for (int i = threadIdx.x; i < P.n_acc_smem; i += blockDim.x) acc_s[i] = 0ull;
    __syncthreads();

    const unsigned lt_mask = (1u << lane) - 1u;
    long long ll_fx = 0;
    unsigned long long bad = 0;

    for (long long it = gw; it < P.C.n_order; it += GW) {
        const int sid = P.C.order[it];
        const long long off = P.C.offs[sid];
        const int len = (int)(P.C.offs[sid + 1] - off);
        const double ps = P.C.p[sid];
        const int32_t* tok = P.C.tokens + off;

        if (len == 0) {   // the empty string is accepted iff start -> end exists
            if (lane == 0) {
                const double q = P.T.start_final_tid >= 0 ? P.tw[P.T.start_final_tid] : 0.0;
                if (MODE == MODE_STRUCT) {
                    P.O.path_count[sid] = q;
                    if (q != 0.0) atomicAdd(P.O.red + 2 + P.T.start_final_tid, 1ull);
                } else {
                    const double lq = log(q);
                    if (P.O.logq) P.O.logq[sid] = lq;
                    if (q > 0.0 && isfinite(lq)) {
                        ll_fx += __double2ll_rn(ps * lq * P.O.ll_scale);
                        atomicAdd(P.O.red + 2 + P.T.start_final_tid, (unsigned long long)__double2ll_rn(ps * P.O.fx_scale));
                    } else bad++;
                }
            }
            continue;
        }

        // ---------------- forward ----------------
        double alpha = (lane == 0) ? 1.0 : 0.0;   // START pseudo position: only the start state
        unsigned mask = 1u;                       // active lanes of the previous position
        int my_state = P.T.start_state;           // state of this lane's slot at the previous position
        int E = 0, sp = 0, tokreg = 0, c = 0;
        bool dead = false;
        for (int t = 0; t < len; ++t) {
            if ((t & 31) == 0) tokreg = (t + lane < len) ? __ldcs(tok + t + lane) : -1;
            c = __shfl_sync(FULL, tokreg, t & 31);
            if ((unsigned)c >= (unsigned)A) { dead = true; break; }
            unsigned rc = 0;
            if ((mask >> lane) & 1u) {
                const int r = my_state * A + c;
                const unsigned r0 = brow[r];
                rc = (r0 << 8) | (brow[r + 1] - r0);
            }
            double a_new = 0.0;
            for (unsigned m = mask; m; m &= m - 1) {          // active sources scatter along their row
                const int s = __ffs(m) - 1;
                const unsigned rcs = __shfl_sync(FULL, rc, s);
                const double val = __shfl_sync(FULL, alpha, s);
                const unsigned r0 = rcs >> 8, cnt = rcs & 255u;
                for (unsigned j = r0; j < r0 + cnt; ++j)
                    if (lane == (int)bent[j]) a_new = fma(aw[j], val, a_new);
            }
            alpha = a_new;
            mask = __ballot_sync(FULL, alpha != 0.0);
            if (mask == 0) { dead = true; break; }
            if ((t & (kRescaleEvery - 1)) == kRescaleEvery - 1) {
                const int emax = __reduce_max_sync(FULL, alpha != 0.0 ? biased_exp(alpha) : -1);
                if (emax < 1023 - kRescaleBand || emax > 1023 + kRescaleBand) {
                    const int shift = 1023 - emax;
                    alpha = scalbn(alpha, shift);
                    E -= shift;
                }
            }
            if (alpha != 0.0) my_state = slot_state[cand_off[c] + lane];
            // push [values..., meta] on the lattice stack
            const int n = __popc(mask);
            if (alpha != 0.0) stack_st(stack, gstack, cap, sp + __popc(mask & lt_mask), (unsigned long long)__double_as_longlong(alpha));
            if (lane == 0) stack_st(stack, gstack, cap, sp + n, (unsigned long long)mask | ((unsigned long long)(unsigned)E << 32));
            sp += n + 1;
        }
        double qh = 0.0, fin = 0.0;
        int fstate = 0;
        if (!dead) {
            if (alpha != 0.0) {                           // c = last symbol
                const int fslot = (int)cand_off[c] + lane;
                fin = fw[fslot];
                fstate = slot_state[fslot];
            }
            qh = warp_sum(alpha * fin);
        }
        if (dead || !(qh > 0.0) || !isfinite(qh)) {
            if (lane == 0) {
                if (MODE == MODE_STRUCT) P.O.path_count[sid] = 0.0;
                else { if (P.O.logq) P.O.logq[sid] = -INFINITY; bad++; }
            }
            continue;
        }
        const int EQ = E;
        if (lane == 0) {
            if (MODE == MODE_STRUCT) P.O.path_count[sid] = scalbn(qh, EQ);
            else {
                const double lq = log(qh) + (double)EQ * 0.69314718055994530942;
                if (P.O.logq) P.O.logq[sid] = lq;
                ll_fx += __double2ll_rn(ps * lq * P.O.ll_scale);
            }
        }
        __syncwarp();

        // ---------------- backward ----------------
        const double invq = 1.0 / qh;
        const double sc0 = (MODE == MODE_STRUCT) ? 1.0 : invq * ps * P.O.fx_scale;
        double beta;          // beta of the position processed last (lanes = its candidates)
        int F = 0, cnext = c;
        {   // position len-1: beta = a(v,end); posterior of the final transition
            const unsigned long long meta = stack_ld(stack, gstack, cap, sp - 1);
            sp -= __popc((unsigned)meta) + 1;
            if (alpha != 0.0 && fin != 0.0) {             // alpha (registers) still holds position len-1
                if (MODE == MODE_STRUCT) acc_add<ACC>(acc_s, acc_g, NA + fstate, 1);
                else acc_add<ACC>(acc_s, acc_g, NA + fstate, __double2ll_rn(alpha * fin * sc0));
            }
            beta = (alpha != 0.0) ? fin : 0.0;
        }
        for (int t = len - 2; t >= -1; --t) {
            double al = 0.0; int Et = 0; int cc = A; int st_id = 0; bool on;
            if (t >= 0) {
                if ((t & 31) == 31) tokreg = __ldg(tok + (t - 31) + lane);
                cc = __shfl_sync(FULL, tokreg, t & 31);
                const unsigned long long meta = stack_ld(stack, gstack, cap, sp - 1);
                const unsigned msk = (unsigned)meta;
                Et = (int)(meta >> 32);
                sp -= __popc(msk) + 1;
                on = (msk >> lane) & 1u;
                if (on) {
                    al = __longlong_as_double((long long)stack_ld(stack, gstack, cap, sp + __popc(msk & lt_mask)));
                    st_id = slot_state[cand_off[cc] + lane];
                }
            } else {          // the START pseudo position
                on = (lane == 0);
                if (on) { al = 1.0; st_id = P.T.start_state; }
            }
            unsigned r0 = 0, cnt = 0;
            if (on) { const int r = st_id * A + cnext; r0 = brow[r]; cnt = brow[r + 1] - r0; }
            const unsigned maxcnt = __reduce_max_sync(FULL, cnt);
            const int d = Et + F - EQ;
            double sc = sc0;
            if (MODE != MODE_STRUCT && d != 0) sc = scalbn(sc0, d);
            double b = 0.0;
            for (unsigned k = 0; k < maxcnt; ++k) {
                unsigned dst = 0; double w = 0.0;
                if (k < cnt) { dst = bent[r0 + k]; w = aw[r0 + k]; }
                const double term = w * __shfl_sync(FULL, beta, dst);
                b += term;
                if (k < cnt && term != 0.0) {
                    if (MODE == MODE_STRUCT) acc_add<ACC>(acc_s, acc_g, (int)(r0 + k), 1);
                    else acc_add<ACC>(acc_s, acc_g, (int)(r0 + k), __double2ll_rn(al * term * sc));
                }
            }
            beta = on ? b : 0.0;
            if (t >= 0 && (t & (kRescaleEvery - 1)) == 0) {
                const int emax = __reduce_max_sync(FULL, beta != 0.0 ? biased_exp(beta) : -1);
                if (emax >= 0 && (emax < 1023 - kRescaleBand || emax > 1023 + kRescaleBand)) {
                    const int shift = 1023 - emax;
                    beta = scalbn(beta, shift);
                    F -= shift;
                }
            }
            cnext = cc;
        }
        __syncwarp();
    }

    if (lane == 0) {
        if (ll_fx) atomicAdd(P.O.red, (unsigned long long)ll_fx);
        if (bad) atomicAdd(P.O.red + 1, bad);
    }
    if (ACC != ACC_GLOBAL) {
        __syncthreads();
        for (int i = threadIdx.x; i < P.n_acc_smem; i += blockDim.x) {
            const unsigned long long v = acc_s[i];
            if (v) atomicAdd(acc_g + i, v);
        }
    }
}

// ------------------------------------------------------------------------------------------
// KT: one THREAD per string -- 32 strings per warp instruction instead of one.  For sparse
// automata (config 4: 1.8 active states per position) a warp-per-string mapping leaves 30 lanes
// idle and is issue-bound (profiles/r01_k2_warp_per_string_ncu.json); here every lane advances its
// own string.  Per thread: the active set {(state, alpha)} of the current and the next position
// in shared memory (capacity K entries each, entry-major so lanes hit consecutive banks), the
// automaton tables shared by the CTA in shared memory, and the lattice -- one packed 64-bit word
// per active entry (48 high bits of alpha | last-of-position flag | 15-bit state) -- streamed to
// a private region in global memory and read back in reverse by the backward sweep.  Strings
// whose active set ever exceeds K are reported (path_count = -1 in MODE_STRUCT) and evaluated
// by the warp-per-string / CTA-per-string kernel instead.
// The packed alpha (2^-37 relative rounding) only enters the arc posteriors, never the
// recursions, so log q is exact and gradients carry <= 1e-11 relative error.
// ------------------------------------------------------------------------------------------
struct ThreadTablesD {
    const uint16_t* __restrict__ brow;   // [n_states*n_sym + 1]
    const uint16_t* __restrict__ adst;   // [n_arcs] target state
    const double* __restrict__ aw;       // [n_arcs]
    const double* __restrict__ fws;      // [n_states] a(state, end) or 0
    int n_sym, n_states, n_arcs, start_state, start_final_tid;
};
struct KTParams {
    ThreadTablesD T;
    const double* __restrict__ tw;
    CorpusD C;                           // C.order = strings of this kernel, longest first; 32 consecutive = one warp group
    EvalOutD O;
    const int32_t* __restrict__ tokT;    // tokens of group g, position t, lane l at goff[g] + t*32 + l (coalesced)
    const int64_t* __restrict__ goff;    // [n_groups]
    long long n_groups;
    unsigned long long* lattice;         // per warp: [max_len][K][32] packed (alpha | flag | state) words
    uint32_t* latcnt;                    // per warp: [max_len][32]   entries | exponent << 8
    int max_len, K, replicas;
};
struct KTTableLayout { size_t aw, fws, brow, adst, total; };
__host__ __device__ inline KTTableLayout kt_table_layout(int n_sym, int n_states, int n_arcs)
{
    KTTableLayout t; size_t o = 0;
    auto al = [](size_t v) { return (v + 7) & ~(size_t)7; };
    t.aw = o; o += (size_t)n_arcs * 8;
    t.fws = o; o += (size_t)n_states * 8;
    t.brow = o; o = al(o + ((size_t)n_states * n_sym + 1) * 2);
    t.adst = o; o = al(o + (size_t)n_arcs * 2);
    t.total = o;
    return t;
}
__device__ __forceinline__ unsigned long long lat_pack(double a, int st)
{
    return (((unsigned long long)__double_as_longlong(a) + 0x8000ull) & ~0xFFFFull) | (unsigned long long)st;
}
__device__ __forceinline__ double lat_alpha(unsigned long long w) { return __longlong_as_double((long long)(w & ~0xFFFFull)); }

template <int MODE>
__global__ void __launch_bounds__(768, 1) kt_fwdbwd(const KTParams P)
{
    extern __shared__ unsigned long long smem[];
    const int tid = threadIdx.x, NT = blockDim.x, K = P.K, lane = tid & 31;
    const int A = P.T.n_sym, NA = P.T.n_arcs, S = P.T.n_states;
    const KTTableLayout tl = kt_table_layout(A, S, NA);
    unsigned char* base = reinterpret_cast<unsigned char*>(smem);
    double* aw = reinterpret_cast<double*>(base + tl.aw);
    double* fws = reinterpret_cast<double*>(base + tl.fws);
    uint16_t* brow = reinterpret_cast<uint16_t*>(base + tl.brow);
    uint16_t* adst = reinterpret_cast<uint16_t*>(base + tl.adst);
    double* la = reinterpret_cast<double*>(base + tl.total);                 // [2][K][NT]
    uint16_t* ls = reinterpret_cast<uint16_t*>(la + (size_t)2 * K * NT);     // [2][K][NT]
    for (int i = tid; i < NA; i += NT) { aw[i] = P.T.aw[i]; adst[i] = P.T.adst[i]; }
    for (int i = tid; i < S; i += NT) fws[i] = P.T.fws[i];
    for (int i = tid; i < S * A + 1; i += NT) brow[i] = P.T.brow[i];
    __syncthreads();

    const long long gwarp = ((long long)blockIdx.x * NT + tid) >> 5, GW = ((long long)gridDim.x * NT) >> 5;
    unsigned long long* const lat = P.lattice + (size_t)gwarp * P.max_len * K * 32 + lane;
    uint32_t* const cw = P.latcnt + (size_t)gwarp * P.max_len * 32 + lane;
    unsigned long long* const acc_g = P.O.acc_global + (size_t)(blockIdx.x % P.replicas) * (size_t)(NA + S);
    const int KN = K * NT, K32 = K * 32;
    long long ll_fx = 0;
    unsigned long long bad = 0;

    for (long long g = gwarp; g < P.n_groups; g += GW) {
        const long long it = g * 32 + lane;
        if (it >= P.C.n_order) continue;
        const int sid = P.C.order[it];
        const int len = (int)(P.C.offs[sid + 1] - P.C.offs[sid]);
        const double ps = P.C.p[sid];
        const int32_t* tok = P.tokT + P.goff[g] + lane;        // token t at tok[t*32]
        if (len == 0) {
            const double q = P.T.start_final_tid >= 0 ? P.tw[P.T.start_final_tid] : 0.0;
            if (MODE == MODE_STRUCT) {
                P.O.path_count[sid] = q;
                if (q != 0.0) atomicAdd(P.O.red + 2 + P.T.start_final_tid, 1ull);
            } else {
                const double lq = log(q);
                if (P.O.logq) P.O.logq[sid] = lq;
                if (q > 0.0 && isfinite(lq)) {
                    ll_fx += __double2ll_rn(ps * lq * P.O.ll_scale);
                    atomicAdd(P.O.red + 2 + P.T.start_final_tid, (unsigned long long)__double2ll_rn(ps * P.O.fx_scale));
                } else bad++;
            }
            continue;
        }
        // ---------------- forward ----------------
        int buf = 0, n_cur = 1, E = 0;
        bool dead = false, over = false;
        la[tid] = 1.0; ls[tid] = (uint16_t)P.T.start_state;
        int c = __ldcs(tok);
        for (int t = 0; t < len; ++t) {
            const int cnx = (t + 1 < len) ? __ldcs(tok + (size_t)(t + 1) * 32) : 0;     // prefetch the next token
            if ((unsigned)c >= (unsigned)A) { dead = true; break; }
            const double* ca = la + buf * KN + tid; const uint16_t* cs = ls + buf * KN + tid;
            double* na = la + (buf ^ 1) * KN + tid; uint16_t* ns = ls + (buf ^ 1) * KN + tid;
            int n_new = 0;
            for (int i = 0; i < n_cur; ++i) {
                const int u = cs[i * NT];
                const double a = ca[i * NT];
                const int r = u * A + c;
                const unsigned r1 = brow[r + 1];
                for (unsigned j = brow[r]; j < r1; ++j) {
                    const double x = a * aw[j];
                    if (x == 0.0) continue;
                    const uint16_t v = adst[j];
                    int k = 0;
                    for (; k < n_new; ++k) if (ns[k * NT] == v) break;
                    if (k < n_new) na[k * NT] += x;
                    else if (n_new < K) { ns[n_new * NT] = v; na[n_new * NT] = x; ++n_new; }
                    else over = true;
                }
            }
            if (over) break;
            if (n_new == 0) { dead = true; break; }
            if ((t & 7) == 7) {                       // lazy power-of-two rescaling (exact)
                int emax = 0;
                for (int k = 0; k < n_new; ++k) emax = max(emax, biased_exp(na[k * NT]));
                if (emax < 1023 - kRescaleBand || emax > 1023 + kRescaleBand) {
                    const int shift = 1023 - emax;
                    for (int k = 0; k < n_new; ++k) na[k * NT] = scalbn(na[k * NT], shift);
                    E -= shift;
                }
            }
            unsigned long long* lt = lat + (size_t)t * K32;
            for (int k = 0; k < n_new; ++k) lt[k * 32] = lat_pack(na[k * NT], ns[k * NT]);
            cw[(size_t)t * 32] = (uint32_t)n_new | ((uint32_t)E << 8);
            n_cur = n_new;
            buf ^= 1;
            c = cnx;
        }
        if (over) {                                   // handled by the warp / CTA kernel
            if (MODE == MODE_STRUCT) P.O.path_count[sid] = -1.0;
            else bad++;                               // cannot happen: the structural pass filters these
            continue;
        }
        double qh = 0.0;
        if (!dead)
            for (int i = 0; i < n_cur; ++i) qh = fma(la[buf * KN + i * NT + tid], fws[ls[buf * KN + i * NT + tid]], qh);
        if (dead || !(qh > 0.0) || !isfinite(qh)) {
            if (MODE == MODE_STRUCT) P.O.path_count[sid] = 0.0;
            else { if (P.O.logq) P.O.logq[sid] = -INFINITY; bad++; }
            continue;
        }
        const int EQ = E;
        if (MODE == MODE_STRUCT) P.O.path_count[sid] = scalbn(qh, EQ);
        else {
            const double lq = log(qh) + (double)EQ * 0.69314718055994530942;
            if (P.O.logq) P.O.logq[sid] = lq;
            ll_fx += __double2ll_rn(ps * lq * P.O.ll_scale);
        }
        // ---------------- backward ----------------
        const double sc0 = (MODE == MODE_STRUCT) ? 1.0 : (1.0 / qh) * ps * P.O.fx_scale;
        {   // last position: beta = a(v,end); posterior of the final transition; alpha list becomes beta list
            double* ba = la + buf * KN + tid; const uint16_t* bs = ls + buf * KN + tid;
            for (int i = 0; i < n_cur; ++i) {
                const int st = bs[i * NT];
                const double fin = fws[st], a = ba[i * NT];
                if (fin != 0.0) {
                    if (MODE == MODE_STRUCT) atomicAdd(acc_g + NA + st, 1ull);
                    else { const long long v = __double2ll_rn(a * fin * sc0); if (v) atomicAdd(acc_g + NA + st, (unsigned long long)v); }
                }
                ba[i * NT] = fin;
            }
        }
        int n_b = n_cur, F = 0;
        int cn = tok[(size_t)(len - 1) * 32];
        // software pipeline: count word, first entry and token of the next (earlier) position are in flight
        uint32_t pf_cw = len >= 2 ? cw[(size_t)(len - 2) * 32] : 1u;
        unsigned long long pf_w0 = len >= 2 ? lat[(size_t)(len - 2) * K32] : 0ull;
        int pf_c = len >= 2 ? tok[(size_t)(len - 2) * 32] : 0;
        for (int t = len - 2; t >= -1; --t) {
            const uint32_t cwv = pf_cw; const unsigned long long w0 = pf_w0; const int cthis = pf_c;
            if (t >= 1) { pf_cw = cw[(size_t)(t - 1) * 32]; pf_w0 = lat[(size_t)(t - 1) * K32]; pf_c = tok[(size_t)(t - 1) * 32]; }
            const double* bb = la + buf * KN + tid; const uint16_t* bs = ls + buf * KN + tid;
            double* oa = la + (buf ^ 1) * KN + tid; uint16_t* os = ls + (buf ^ 1) * KN + tid;
            const int n_t = (t >= 0) ? (int)(cwv & 255u) : 1;
            const int Et = (t >= 0) ? ((int)cwv >> 8) : 0;
            const int d = Et + F - EQ;
            double sc = sc0;
            if (MODE != MODE_STRUCT && d != 0) sc = scalbn(sc0, d);
            const unsigned long long* lt = lat + (size_t)(t >= 0 ? t : 0) * K32;
            for (int i = 0; i < n_t; ++i) {
                int u; double a;
                if (t >= 0) { const unsigned long long w = (i == 0) ? w0 : lt[i * 32]; u = (int)(w & 0xFFFFull); a = lat_alpha(w); }
                else { u = P.T.start_state; a = 1.0; }
                const int r = u * A + cn;
                const unsigned r1 = brow[r + 1];
                double b = 0.0;
                for (unsigned j = brow[r]; j < r1; ++j) {
                    const uint16_t v = adst[j];
                    for (int k = 0; k < n_b; ++k)
                        if (bs[k * NT] == v) {
                            const double term = aw[j] * bb[k * NT];
                            if (term != 0.0) {
                                b += term;
                                if (MODE == MODE_STRUCT) atomicAdd(acc_g + j, 1ull);
                                else { const long long vv = __double2ll_rn(a * term * sc); if (vv) atomicAdd(acc_g + j, (unsigned long long)vv); }
                            }
                            break;
                        }
                }
                os[i * NT] = (uint16_t)u; oa[i * NT] = b;
            }
            if (t >= 0 && (t & 7) == 0) {
                int emax = 0;
                for (int k = 0; k < n_t; ++k) emax = max(emax, biased_exp(oa[k * NT]));
                if (emax != 0 && (emax < 1023 - kRescaleBand || emax > 1023 + kRescaleBand)) {
                    const int shift = 1023 - emax;
                    for (int k = 0; k < n_t; ++k) oa[k * NT] = scalbn(oa[k * NT], shift);
                    F -= shift;
                }
            }
            n_b = n_t;
            buf ^= 1;
            cn = cthis;
        }
    }
    // per-warp reduction of the fixed-point log-likelihood, one atomic per warp
    for (int o = 16; o; o >>= 1) { ll_fx += __shfl_xor_sync(FULL, ll_fx, o); bad += __shfl_xor_sync(FULL, bad, o); }
    if (lane == 0) {
        if (ll_fx) atomicAdd(P.O.red, (unsigned long long)ll_fx);
        if (bad) atomicAdd(P.O.red + 1, bad);
    }
}

// ------------------------------------------------------------------------------------------
// K3: one CTA per string for automata where more than 32 states emit one symbol.
// Thread i <-> candidate slot i of the current symbol; alpha / beta~ vectors double-buffered in
// shared memory; the lattice (dense over candidates) goes to a per-CTA slab in global memory
// (L2 resident: 148 x 2 slabs); accumulators are 64-bit REDs into L2.
// ------------------------------------------------------------------------------------------
struct K3Params {
    FastTablesD T;
    EvalWeightsD W;
    CorpusD C;
    EvalOutD O;
    double* lattice;           // [grid][max_len][nt]
    int* lat_exp;              // [grid][max_len]
    int max_len;
};

template <int MODE>
__global__ void __launch_bounds__(1024, 1) k3_fwdbwd(const K3Params P)
{
    extern __shared__ unsigned long long smem[];
    const int nt = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
    double* va = reinterpret_cast<double*>(smem);        // [2][nt] alpha or beta~
    double* red = va + 2 * nt;                           // [32]
    int* ired = reinterpret_cast<int*>(red + 32);        // [34]
    const FastTablesD& T = P.T;
    const int A = T.n_sym;
    double* lat = P.lattice + (size_t)blockIdx.x * P.max_len * nt;
    int* lexp = P.lat_exp + (size_t)blockIdx.x * P.max_len;
    long long ll_fx = 0;
    unsigned long long bad = 0;

    for (long long it = blockIdx.x; it < P.C.n_order; it += gridDim.x) {
        const int sid = P.C.order[it];
        const long long off = P.C.offs[sid];
        const int len = (int)(P.C.offs[sid + 1] - off);
        const double ps = P.C.p[sid];
        const int32_t* tok = P.C.tokens + off;
        __syncthreads();
        if (len == 0) {
            if (tid == 0) {
                const double q = T.start_final_tid >= 0 ? P.W.tw[T.start_final_tid] : 0.0;
                if (MODE == MODE_STRUCT) {
                    P.O.path_count[sid] = q;
                    if (q != 0.0) atomicAdd(P.O.red + 2 + T.start_final_tid, 1ull);
                } else {
                    const double lq = log(q);
                    if (P.O.logq) P.O.logq[sid] = lq;
                    if (q > 0.0 && isfinite(lq)) {
                        ll_fx += __double2ll_rn(ps * lq * P.O.ll_scale);
                        atomicAdd(P.O.red + 2 + T.start_final_tid, (unsigned long long)__double2ll_rn(ps * P.O.fx_scale));
                    } else bad++;
                }
            }
            continue;
        }
        // ---------------- forward ----------------
        int cur = 0, E = 0, cprev = A;
        bool dead = false;
        va[tid] = (tid == 0) ? 1.0 : 0.0;
        __syncthreads();
        uint32_t slot = 0;
        double alpha = 0.0;
        for (int t = 0; t < len; ++t) {
            const int c = tok[t];
            if ((unsigned)c >= (unsigned)A) { dead = true; break; }
            const uint32_t c0 = T.cand_off[c], ncand = T.cand_off[c + 1] - c0;
            const bool valid = (uint32_t)tid < ncand;
            slot = c0 + tid;
            alpha = 0.0;
            if (valid) {
                const uint32_t row = T.frow[(size_t)T.slot_state[slot] * (A + 1) + cprev];
                const int cnt = row & ((1u << kRowCntBitsD) - 1);
                const uint32_t st = row >> kRowCntBitsD;
                const double* src = va + cur * nt;
                double s = 0.0;
                for (int k = 0; k < cnt; ++k) {
                    const uint32_t ent = T.fent[st + k];
                    s = fma(P.W.tw[ent >> kSlotBitsD], src[ent & ((1u << kSlotBitsD) - 1)], s);
                }
                alpha = s * P.W.sw[slot];
            }
            // any nonzero? (and the exponent of the largest entry every few positions)
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
            lat[(size_t)t * nt + tid] = alpha;
            if (tid == 0) lexp[t] = E;
            cur ^= 1;
            cprev = c;
            __syncthreads();
        }
        double qh = 0.0, fin = 0.0;
        if (!dead) {
            fin = (alpha != 0.0) ? P.W.fw[slot] : 0.0;
            const double part = warp_sum(alpha * fin);
            if (lane == 0) red[warp] = part;
            __syncthreads();
            for (int w = 0; w < nwarps; ++w) qh += red[w];    // fixed order
        }
        if (dead || !(qh > 0.0) || !isfinite(qh)) {
            if (tid == 0) {
                if (MODE == MODE_STRUCT) P.O.path_count[sid] = 0.0;
                else { if (P.O.logq) P.O.logq[sid] = -INFINITY; bad++; }
            }
            continue;
        }
        const int EQ = E;
        if (tid == 0) {
            if (MODE == MODE_STRUCT) P.O.path_count[sid] = scalbn(qh, EQ);
            else {
                const double lq = log(qh) + (double)EQ * 0.69314718055994530942;
                if (P.O.logq) P.O.logq[sid] = lq;
                ll_fx += __double2ll_rn(ps * lq * P.O.ll_scale);
            }
        }
        // ---------------- backward ----------------
        const double invq = 1.0 / qh;
        int F = 0, cnext = tok[len - 1];
        if (alpha != 0.0 && fin != 0.0) {
            const uint32_t fst = T.slot_state[slot];
            if (MODE == MODE_STRUCT) atomicAdd(P.O.acc_global + T.n_arcs + fst, 1ull);
            else atomicAdd(P.O.acc_global + T.n_arcs + fst, (unsigned long long)__double2ll_rn(alpha * fin * invq * ps * P.O.fx_scale));
        }
        __syncthreads();
        cur = 0;
        va[tid] = (alpha != 0.0) ? fin * P.W.sw[slot] : 0.0;
        __syncthreads();
        for (int t = len - 2; t >= 0; --t) {
            const int c = tok[t];
            const uint32_t c0 = T.cand_off[c];
            slot = c0 + tid;
            const double al = lat[(size_t)t * nt + tid];
            const int Et = lexp[t];
            const int d = Et + F - EQ;
            double sc = invq * ps * P.O.fx_scale;
            if (d != 0) sc = scalbn(sc, d);
            double bt = 0.0;
            if (al != 0.0) {
                const uint32_t row = T.brow[(size_t)T.slot_state[slot] * A + cnext];
                const int cnt = row & ((1u << kRowCntBitsD) - 1);
                const uint32_t st = row >> kRowCntBitsD;
                const double* src = va + cur * nt;
                double b = 0.0;
                for (int k = 0; k < cnt; ++k) {
                    const uint32_t ent = T.bent[st + k];
                    const double term = P.W.tw[ent >> kSlotBitsD] * src[ent & ((1u << kSlotBitsD) - 1)];
                    b += term;
                    if (term != 0.0) {
                        if (MODE == MODE_STRUCT) atomicAdd(P.O.acc_global + st + k, 1ull);
                        else {
                            const long long v = __double2ll_rn(al * term * sc);
                            if (v) atomicAdd(P.O.acc_global + st + k, (unsigned long long)v);
                        }
                    }
                }
                bt = b * P.W.sw[slot];
            }
            if ((t & (kRescaleEvery - 1)) == 0) {
                const int wmax = __reduce_max_sync(FULL, bt != 0.0 ? biased_exp(bt) : -1);
                if (lane == 0) ired[warp] = wmax;
                __syncthreads();
                int emax = -1;
                for (int w = 0; w < nwarps; ++w) emax = max(emax, ired[w]);
                if (emax >= 0 && (emax < 1023 - kRescaleBand || emax > 1023 + kRescaleBand)) {
                    const int shift = 1023 - emax;
                    bt = scalbn(bt, shift);
                    F -= shift;
                }
            }
            va[(cur ^ 1) * nt + tid] = bt;
            cur ^= 1;
            cnext = c;
            __syncthreads();
        }
        {   // arcs out of the start state
            const uint32_t row = T.brow[(size_t)T.start_state * A + cnext];
            const int cnt = row & ((1u << kRowCntBitsD) - 1);
            const uint32_t st = row >> kRowCntBitsD;
            const int d = F - EQ;
            double sc = invq * ps * P.O.fx_scale;
            if (d != 0) sc = scalbn(sc, d);
            const double* src = va + cur * nt;
            for (int k = tid; k < cnt; k += nt) {
                const uint32_t ent = T.bent[st + k];
                const double term = P.W.tw[ent >> kSlotBitsD] * src[ent & ((1u << kSlotBitsD) - 1)];
                if (term != 0.0) {
                    if (MODE == MODE_STRUCT) atomicAdd(P.O.acc_global + st + k, 1ull);
                    else {
                        const long long v = __double2ll_rn(term * sc);
                        if (v) atomicAdd(P.O.acc_global + st + k, (unsigned long long)v);
                    }
                }
            }
        }
    }
    if (tid == 0) {
        if (ll_fx) atomicAdd(P.O.red, (unsigned long long)ll_fx);
        if (bad) atomicAdd(P.O.red + 1, bad);
    }
}

// ------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------
// Generic path: emissions of any length (0, 1, 2, ... tokens), one thread per string, dense
// log-domain lattice (len+1) x n_states in global scratch.  Correct for every automaton the
// reference accepts (no empty-emission cycles); not tuned.
// ------------------------------------------------------------------------------------------
struct GenericTablesD {
    const int32_t* __restrict__ emis_row;
    const int32_t* __restrict__ emis_tok_off;
    const int32_t* __restrict__ emis_tok;
    const int32_t* __restrict__ trans_row;
    const int32_t* __restrict__ trans_dst;
    const int32_t* __restrict__ eps_order;
    int n_states, n_trans, start_state, end_state;
};
struct GenericParams {
    GenericTablesD G;
    const double* __restrict__ ltw;    // log transition weights (MODE_MINPATH: +inf where absent)
    const double* __restrict__ lew;    // log emission weights
    CorpusD C;
    EvalOutD O;
    double* scratch;                   // [n_threads][2][(max_len+1)*n_states]
    int max_len;
    long long first, count;            // slice of C.order handled by this launch
    // MODE_VITERBI: without vit_off the step count of every string goes to vit_cnt; with vit_off ([n_strings+1] step
    // offsets) the steps go to vit_trans / vit_emis
    int32_t* vit_cnt;
    const int64_t* vit_off;
    int32_t* vit_trans;
    int32_t* vit_emis;
};

__device__ __forceinline__ double logaddexp_d(double a, double b)
{
    if (a == -INFINITY) return b;
    if (b == -INFINITY) return a;
    const double m = fmax(a, b);
    return m + log1p(exp(-fabs(a - b)));
}

// semiring: MODE_EVAL = (logaddexp, +) on log-weights; MODE_STRUCT = (+, *) on path counts
// (linear domain so that counts stay exact integers; every weight is 1); MODE_MINPATH = (min, +) on log-weights whose
// absent edges are +inf (k_minplus_weights), never -inf: the minimum would pick them
template <int MODE> __device__ __forceinline__ double sr_zero() { return MODE == MODE_STRUCT ? 0.0 : (MODE == MODE_MINPATH ? INFINITY : -INFINITY); }
template <int MODE> __device__ __forceinline__ double sr_plus(double a, double b) { return MODE == MODE_STRUCT ? a + b : (MODE == MODE_MINPATH ? fmin(a, b) : logaddexp_d(a, b)); }
template <int MODE> __device__ __forceinline__ double sr_times(double a, double b) { return MODE == MODE_STRUCT ? a * b : a + b; }

template <int MODE>
__global__ void __launch_bounds__(128) kg_fwdbwd(const GenericParams P)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.count) return;
    const GenericTablesD& G = P.G;
    const int S = G.n_states;
    const int sid = P.C.order[P.first + i];
    const long long off = P.C.offs[sid];
    const int len = (int)(P.C.offs[sid + 1] - off);
    const double ps = P.C.p[sid];
    const int32_t* tok = P.C.tokens + off;
    const size_t lat_sz = (size_t)(P.max_len + 1) * S;
    double* la = P.scratch + (size_t)i * 2 * lat_sz;
    double* lb = la + lat_sz;
    const double ZERO = sr_zero<MODE>();
    for (size_t k = 0; k < (size_t)(len + 1) * S; ++k) { la[k] = ZERO; lb[k] = ZERO; }
    la[G.start_state] = (MODE == MODE_STRUCT) ? 1.0 : 0.0;
    double lq = ZERO;
    int fin_t = -1, fin_u = -1;                  // MODE_VITERBI: the winning transition into the end state
    // forward
    for (int pos = 0; pos <= len; ++pos) {
        for (int oi = 0; oi < S; ++oi) {
            const int u = G.eps_order[oi];
            const double au = la[(size_t)pos * S + u];
            if (au == ZERO || u == G.end_state) continue;
            for (int t = G.trans_row[u]; t < G.trans_row[u + 1]; ++t) {
                const int v = G.trans_dst[t];
                const double w = (MODE == MODE_STRUCT) ? au : au + P.ltw[t];
                if (w == ZERO) continue;
                if (v == G.end_state) {
                    if (MODE == MODE_VITERBI) { if (pos == len && w > lq) { lq = w; fin_t = t; fin_u = u; } }
                    else if (pos == len) lq = sr_plus<MODE>(lq, w);
                    continue;
                }
                for (int e = G.emis_row[v]; e < G.emis_row[v + 1]; ++e) {
                    const int e0 = G.emis_tok_off[e], el = G.emis_tok_off[e + 1] - e0;
                    if (pos + el > len) continue;
                    bool m = true;
                    for (int k = 0; k < el; ++k) if (tok[pos + k] != G.emis_tok[e0 + k]) { m = false; break; }
                    if (!m) continue;
                    double* dst = la + (size_t)(pos + el) * S + v;
                    if (MODE == MODE_VITERBI) {          // the first strictly larger candidate wins; backpointer (t, e)
                        const double val = w + P.lew[e];
                        if (val > *dst) {
                            *dst = val;
                            reinterpret_cast<unsigned long long*>(lb)[(size_t)(pos + el) * S + v] = ((unsigned long long)t << 32) | (unsigned)e;
                        }
                    } else *dst = sr_plus<MODE>(*dst, (MODE == MODE_STRUCT) ? w : w + P.lew[e]);
                }
            }
        }
    }
    if (MODE == MODE_MINPATH) {                  // lq = m_s, the smallest log weight of a path (+inf: none); no backward
        P.O.logq[sid] = lq;
        return;
    }
    if (MODE == MODE_VITERBI) {                  // lq = the largest log weight of a path (-inf: none); traceback, no backward
        P.O.logq[sid] = lq;
        const bool found = lq > -INFINITY;
        const unsigned long long* bp = reinterpret_cast<const unsigned long long*>(lb);
        int64_t o = found && P.vit_off ? P.vit_off[sid + 1] - 1 : 0;
        if (found && P.vit_off) { P.vit_trans[o] = fin_t; P.vit_emis[o] = -1; }
        int n = found ? 1 : 0, p = len, v = fin_u;
        while (found && v != G.start_state) {
            const unsigned long long b = bp[(size_t)p * S + v];
            const int t = (int)(b >> 32), e = (int)(unsigned)b;
            if (P.vit_off) { --o; P.vit_trans[o] = t; P.vit_emis[o] = e; }
            p -= G.emis_tok_off[e + 1] - G.emis_tok_off[e];
            int lo = 0, hi = S;                  // source state of t: the last state whose transitions start at or before t
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (G.trans_row[mid] <= t) lo = mid; else hi = mid; }
            v = lo;
            ++n;
        }
        if (!P.vit_off) P.vit_cnt[sid] = n;
        return;
    }
    if (MODE == MODE_STRUCT) {
        P.O.path_count[sid] = lq;
        if (!(lq > 0.0)) return;
    } else {
        if (!(lq > -INFINITY) || !isfinite(lq)) {
            if (P.O.logq) P.O.logq[sid] = -INFINITY;
            atomicAdd(P.O.red + 1, 1ull);
            return;
        }
        if (P.O.logq) P.O.logq[sid] = lq;
        atomicAdd(P.O.red, (unsigned long long)__double2ll_rn(ps * lq * P.O.ll_scale));
    }
    // backward: lb[pos][u] = sum over continuations of (pos,u); posteriors on the way
    unsigned long long* eacc = P.O.red + 2;
    for (int pos = len; pos >= 0; --pos) {
        for (int oi = S - 1; oi >= 0; --oi) {
            const int u = G.eps_order[oi];
            const double au = la[(size_t)pos * S + u];
            if (au == ZERO || u == G.end_state) continue;
            double bu = ZERO;
            for (int t = G.trans_row[u]; t < G.trans_row[u + 1]; ++t) {
                const int v = G.trans_dst[t];
                const double w = (MODE == MODE_STRUCT) ? 1.0 : P.ltw[t];
                if (w == ZERO) continue;
                if (v == G.end_state) {
                    if (pos == len) {
                        bu = sr_plus<MODE>(bu, w);
                        if (MODE == MODE_STRUCT) atomicAdd(eacc + t, 1ull);
                        else {
                            const long long fx = __double2ll_rn(exp(au + w - lq) * ps * P.O.fx_scale);
                            if (fx) atomicAdd(eacc + t, (unsigned long long)fx);
                        }
                    }
                    continue;
                }
                for (int e = G.emis_row[v]; e < G.emis_row[v + 1]; ++e) {
                    const int e0 = G.emis_tok_off[e], el = G.emis_tok_off[e + 1] - e0;
                    if (pos + el > len) continue;
                    bool m = true;
                    for (int k = 0; k < el; ++k) if (tok[pos + k] != G.emis_tok[e0 + k]) { m = false; break; }
                    if (!m) continue;
                    const double bv = lb[(size_t)(pos + el) * S + v];
                    if (bv == ZERO) continue;
                    const double term = (MODE == MODE_STRUCT) ? bv : w + P.lew[e] + bv;
                    if (term == ZERO) continue;
                    bu = sr_plus<MODE>(bu, term);
                    if (MODE == MODE_STRUCT) { atomicAdd(eacc + t, 1ull); atomicAdd(eacc + G.n_trans + e, 1ull); }
                    else {
                        const long long fx = __double2ll_rn(exp(au + term - lq) * ps * P.O.fx_scale);
                        if (fx) { atomicAdd(eacc + t, (unsigned long long)fx); atomicAdd(eacc + G.n_trans + e, (unsigned long long)fx); }
                    }
                }
            }
            lb[(size_t)pos * S + u] = bu;
        }
    }
}

// ------------------------------------------------------------------------------------------
// small kernels around the dominant one
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double weight_of(int tp, const double* x, int unit)
{
    if (unit || tp == -1) return 1.0;
    if (tp < -1) return 0.0;
    return exp(x[tp]);
}
__device__ __forceinline__ double logweight_of(int tp, const double* x, int unit)
{
    if (unit || tp == -1) return 0.0;
    if (tp < -1) return -INFINITY;
    return x[tp];
}

// edge weights from x: replaces the exp(P.x) of src/Learner.cpp:530-533 (per edge, not per path)
__global__ void k_weights(int n_trans, int n_emis, int n_slots, const int32_t* __restrict__ trans_tp,
                          const int32_t* __restrict__ emis_tp, const int32_t* __restrict__ slot_emis,
                          const int32_t* __restrict__ slot_final, const double* __restrict__ x, int unit,
                          double* tw, double* sw, double* fw, double* ltw, double* lew)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_trans) {
        tw[i] = weight_of(trans_tp[i], x, unit);
        ltw[i] = logweight_of(trans_tp[i], x, unit);
    } else if (i < n_trans + n_emis) {
        const int e = i - n_trans;
        lew[e] = logweight_of(emis_tp[e], x, unit);
    } else if (i < n_trans + n_emis + n_slots) {
        const int s = i - n_trans - n_emis;
        sw[s] = slot_emis[s] < 0 ? 1.0 : weight_of(emis_tp[slot_emis[s]], x, unit);
        fw[s] = slot_final[s] < 0 ? 0.0 : weight_of(trans_tp[slot_final[s]], x, unit);
    }
}

// final weight per state: a(state, end) or 0
__global__ void k_state_final_weights(int n_states, const int32_t* __restrict__ state_final, const double* __restrict__ tw, double* fws)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_states) fws[i] = state_final[i] < 0 ? 0.0 : tw[state_final[i]];
}

// per combined arc (bwd-CSR order): aw = a(u,v) * b(v, c_next)
__global__ void k_arc_weights(int n_arcs, const int32_t* __restrict__ arc_tid, const int32_t* __restrict__ arc_eid,
                              const int32_t* __restrict__ emis_tp, const double* __restrict__ tw,
                              const double* __restrict__ x, int unit, double* aw)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_arcs) aw[i] = tw[arc_tid[i]] * (arc_eid[i] < 0 ? 1.0 : weight_of(emis_tp[arc_eid[i]], x, unit));
}

// combined-arc / final accumulators -> per-edge accumulators (integer adds: order independent)
__global__ void k_arcs_to_edges(int n_arcs, int n_slots /* = n_states */, int n_trans, const unsigned long long* __restrict__ acc, int replicas,
                                const int32_t* __restrict__ arc_tid, const int32_t* __restrict__ arc_eid,
                                const int32_t* __restrict__ slot_final /* per state */, unsigned long long* edge_acc)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long v = 0;
    if (i < n_arcs + n_slots)
        for (int r = 0; r < replicas; ++r) v += acc[(size_t)r * (n_arcs + n_slots) + i];
    if (i < n_arcs) {
        if (v) {
            atomicAdd(edge_acc + arc_tid[i], v);
            if (arc_eid[i] >= 0) atomicAdd(edge_acc + n_trans + arc_eid[i], v);
        }
    } else if (i < n_arcs + n_slots) {
        const int f = slot_final[i - n_arcs];
        if (v && f >= 0) atomicAdd(edge_acc + f, v);
    }
}

// out[0] = loglik, out[1] = #non-finite strings, out[2+i] = grad_i = -sum_s p_s E_s[count_i]
__global__ void k_finish_eval(int n_edges, int n, const unsigned long long* __restrict__ red,
                              const int32_t* __restrict__ edge_tp, double inv_fx, double inv_ll, double* out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        const double bad = (double)red[1];
        out[0] = bad > 0 ? -INFINITY : (double)(long long)red[0] * inv_ll;
        out[1] = bad;
    }
    if (i < n_edges) {
        const int tp = edge_tp[i];
        if (tp >= 0 && tp < n) out[2 + tp] = -(double)(long long)red[2 + i] * inv_fx;
    }
}

__global__ void k_finish_struct(int n_edges, const unsigned long long* __restrict__ red,
                                const int32_t* __restrict__ edge_raw, uint8_t* used)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_edges) {
        const int r = edge_raw[i];
        if (r >= 0) used[r] = red[2 + i] ? 1 : 0;
    }
}

// ------------------------------------------------------------------------------------------
// K5: H_f block, one warp per ambiguous string (block of paths x cols counts).
//   r = softmax_l( sum_j P_lj x_j ),  g = P^T r,  H_s = p_s ( g g^T - P^T diag(r) P )
// The contraction P^T diag(r) P runs on the FP64 tensor cores (mma.sync m8n8k4 DMMA):
// tiles of 8x8 outputs, k = paths in chunks of 4.  Results are scattered into the dense n x n
// H with fixed-point REDs (order independent).
// ------------------------------------------------------------------------------------------
struct HessParams {
    int64_t n_blocks;
    const int64_t* __restrict__ path_off;
    const int64_t* __restrict__ col_off;
    const int32_t* __restrict__ cols;
    const int64_t* __restrict__ val_off;
    const double* __restrict__ counts;
    const double* __restrict__ p;
    const double* __restrict__ x;
    double* r_scratch;               // [total paths] posterior of every path
    unsigned long long* H_fx;        // [n*n] fixed point
    double* rmin;                    // [1] smallest path posterior (atomicMin on bits)
    int n;
    double fx_scale;
    const int32_t* __restrict__ blk_slot;   // blocks = region types: type slot of block b (-1: no type), or nullptr
    double* slot_lrmin;              // [type slots] log of the smallest path posterior of the type
};

__device__ __forceinline__ void dmma_m8n8k4(double& d0, double& d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(256) k5_hessian(const HessParams P)
{
    const int lane = threadIdx.x & 31;
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long GW = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long b = gw; b < P.n_blocks; b += GW) {
        const long long p0 = P.path_off[b];
        const int L = (int)(P.path_off[b + 1] - p0);
        const long long c0 = P.col_off[b];
        const int D = (int)(P.col_off[b + 1] - c0);
        const double* M = P.counts + P.val_off[b];    // L x D row major
        const int32_t* cols = P.cols + c0;
        const double ps = P.p[b];
        double* r = P.r_scratch + p0;
        // path log-weights, softmax in a fixed order
        double mx = -INFINITY;
        for (int l = lane; l < L; l += 32) {
            double s = 0.0;
            for (int j = 0; j < D; ++j) s = fma(M[(size_t)l * D + j], P.x[cols[j]], s);
            r[l] = s;
            mx = fmax(mx, s);
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) mx = fmax(mx, __shfl_xor_sync(FULL, mx, o));
        __syncwarp();
        double z = 0.0;
        for (int l = lane; l < L; l += 32) { const double e = exp(r[l] - mx); r[l] = e; z += e; }
        z = warp_sum(z);
        __syncwarp();
        double rm = INFINITY;
        for (int l = lane; l < L; l += 32) { const double v = r[l] / z; r[l] = v; rm = fmin(rm, v); }
#pragma unroll
        for (int o = 16; o; o >>= 1) rm = fmin(rm, __shfl_xor_sync(FULL, rm, o));
        // a block without a type slot (a segment of a string that no region type covers) leaves rmin to the caller's sweep
        const int slot = P.blk_slot ? P.blk_slot[b] : 0;
        if (lane == 0 && P.rmin && slot >= 0) atomicMin(reinterpret_cast<unsigned long long*>(P.rmin), (unsigned long long)__double_as_longlong(rm));
        if (lane == 0 && P.blk_slot && slot >= 0) P.slot_lrmin[slot] = log(rm);
        __syncwarp();
        if (!P.H_fx) continue;                                 // rmin only (QuasiNewtonLearner's diagnostic column)
        // 8x8 output tiles; DMMA fragment layout (m8n8k4): A[row=lane/4][k=lane%4],
        // B[k=lane%4][col=lane/4], C[row=lane/4][col=2*(lane%4)+{0,1}]
        const int gi = lane >> 2, ti = lane & 3;
        for (int jt = 0; jt < D; jt += 8) {
            for (int kt = jt; kt < D; kt += 8) {
                double c0v = 0.0, c1v = 0.0, g_a = 0.0, g_b0 = 0.0, g_b1 = 0.0;
                for (int l0 = 0; l0 < L; l0 += 4) {
                    const int l = l0 + ti;
                    double a = 0.0, bb = 0.0;
                    if (l < L) {
                        const double rl = r[l];
                        if (jt + gi < D) a = M[(size_t)l * D + jt + gi] * rl;    // (P^T diag r)[j][l]
                        if (kt + gi < D) bb = M[(size_t)l * D + kt + gi];        // P[l][k]
                    }
                    dmma_m8n8k4(c0v, c1v, a, bb);
                }
                // g_j for the tile rows / cols: g = P^T r (tiny; recomputed per tile)
                {
                    const int jr = jt + gi;
                    const int k0 = kt + 2 * ti, k1 = k0 + 1;
                    for (int l = 0; l < L; ++l) {
                        const double rl = r[l];
                        if (jr < D) g_a = fma(M[(size_t)l * D + jr], rl, g_a);
                        if (k0 < D) g_b0 = fma(M[(size_t)l * D + k0], rl, g_b0);
                        if (k1 < D) g_b1 = fma(M[(size_t)l * D + k1], rl, g_b1);
                    }
                    const int row = jr;
                    if (row < D) {
                        const int pj = cols[row];
                        if (k0 < D) {
                            const long long v = __double2ll_rn(ps * (g_a * g_b0 - c0v) * P.fx_scale);
                            const int pk = cols[k0];
                            if (v) {
                                atomicAdd(P.H_fx + (size_t)pj * P.n + pk, (unsigned long long)v);
                                if (kt != jt) atomicAdd(P.H_fx + (size_t)pk * P.n + pj, (unsigned long long)v);
                            }
                        }
                        if (k1 < D) {
                            const long long v = __double2ll_rn(ps * (g_a * g_b1 - c1v) * P.fx_scale);
                            const int pk = cols[k1];
                            if (v) {
                                atomicAdd(P.H_fx + (size_t)pj * P.n + pk, (unsigned long long)v);
                                if (kt != jt) atomicAdd(P.H_fx + (size_t)pk * P.n + pj, (unsigned long long)v);
                            }
                        }
                    }
                }
            }
        }
        __syncwarp();
    }
}

// rmin = exp(min over the strings of the summed log rmin of their regions, or of m_s - log q_s); one CTA
__global__ void k_min_exp(long long n, const double* __restrict__ v, double* out)
{
    __shared__ double s_m[32];
    double m = 0.0;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) m = fmin(m, v[i]);
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmin(m, __shfl_xor_sync(FULL, m, o));
    if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) { for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmin(m, s_m[w]); *out = exp(m); }
}

__global__ void k_fx_to_double(size_t n, const unsigned long long* __restrict__ in, double inv, double* out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (double)(long long)in[i] * inv;
}

}  // namespace wfsa
