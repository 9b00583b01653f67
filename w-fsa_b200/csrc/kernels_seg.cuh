// w-fsa_b200/csrc/kernels_seg.cuh -- sm_100a kernels over the SEGMENTED compiled lattices (lattice.hpp).
//
// Every string's trimmed lattice is cut at the nodes all of its accepting paths share.  Between two
// cuts lies either one edge (a bridge) or a small DAG (a region); path weights factor over segments:
//     log q_s = sum_{bridges of s} log w[arc]  +  sum_{regions of s} log q_region
//     E_s[count(arc)] = [arc is a bridge of s]  +  posterior of the arc inside its region
// so one evaluation (Learner::ComputeModeledProbs + ComputeObjective + ComputeGrad,
// /root/reference/src/Learner.cpp:515-553, src/QuasiNewtonLearner.cpp:93-125) becomes
//   KR  kr_regions : forward-backward over every distinct region TYPE once (thread per type):
//                    lq[type] = log q_type,  acc[arc] += W_type * posterior   (64-bit fixed-point REDs),
//                    loglik += W_type * lq[type]
//                    (path form: kr_paths; DAG form: big_fwd / big_bwd / big_red; all shared with k_eval6)
// The bridges need no per-string work: with c[arc] = sum_s p_s * (times arc is a bridge of s), computed when the
// lattices are compiled, their part of the gradient is the constant c and their part of the log-likelihood is
// sum_arc c[arc] * log w[arc] (k_prep6).  Only a caller that wants log q_s of every string runs
//   KS  ks_strings : thread per string: log q_s = sum of log w over its bridge arcs (16-bit ids, table in
//                    shared memory) + sum of lq[type] over its regions.
#pragma once
#include "kernels.cuh"

namespace wfsa {

struct KRParams {
    const double* __restrict__ aw;        // [n_arcs] a(u,v) * b(v,e)
    const uint32_t* __restrict__ words;   // word j of lane l of group g at goff[g] + j*32 + l
    const int64_t* __restrict__ goff;     // [n_groups+1]
    const int32_t* __restrict__ grows;    // [n_groups] 0x10000|paths<<8|length = path form; 4/8/12/16 = small DAG; else big DAG (multiple of 16)
    const double* __restrict__ typeW;     // [n_groups*32]
    const uint32_t* __restrict__ pwords;  // reduction plan of the path-form groups: word r of lane l of group g at pgoff[g] + r*32 + l
    const int64_t* __restrict__ pgoff;    // [n_groups+1] (lattice.hpp, SegmentedCorpus::pwords)
    double* lq;                           // [n_groups*32 + 1] log q per type (last = dummy, stays 0)
    long long n_groups;
    double* xs;                           // big regions: per warp [xs_rows][32]
    size_t xs_rows;
    unsigned int* counter;                // dynamic group scheduler
    unsigned long long* acc;              // [replicas][n_arcs]
    double fx_scale;
    int n_arcs, replicas;
    // log-likelihood: sum_s p_s log q_s = sum_types W_type * lq_type + sum_arcs (bridge count of the arc) * log w[arc].
    // The first sum is accumulated here (fixed point, one RED per CTA), the second one arrives as per-CTA partials of
    // the weight kernel in llpart[n_llpart][2] = (value, non-finite terms) and is added by CTA 0.
    double ll_scale;
    unsigned long long* red;              // red[0] fixed-point loglik, red[1] non-finite terms
    const long long* __restrict__ llpart;
    int n_llpart;
};

// 64-bit add without a return value, spelled as `red` so that ptxas emits REDG in every kernel: in a kernel that also
// holds a grid barrier (k_eval6) it keeps atomicAdd() with an unused result as ATOMG, whose lanes travel the return path
// (measured: 0 RED sectors in ncu, region phase 95 us instead of 55 us).
__device__ __forceinline__ void red_add64(unsigned long long* p, unsigned long long v)
{
    asm volatile("red.relaxed.gpu.global.add.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}

// W * log q of one region type into the thread's fixed-point sum (W = 0: a padding lane)
__device__ __forceinline__ void kr_loglik(const KRParams& P, double W, bool ok, double lq, long long& ll)
{
    if (W > 0.0) {
        if (ok) ll += __double2ll_rn(W * lq * P.ll_scale);
        else atomicAdd(P.red + 1, 1ull);
    }
}

// The pool of a thread: node value of slot s of the thread at shared byte address p + s * ps; trash: where a lane without an
// edge stores (big_fwd, big_bwd).  kr_paths borrows slots 0 .. kPathSlots-1 of the warp's own columns (the pool area has
// at least kPathSlots slots per thread).
struct BigPool { unsigned int p, ps, trash; };
constexpr int kPathSlots = 8;                                  // = kSegMaxPaths of lattice.hpp
constexpr uint32_t kPLast = 1u << 31;                          // = kPlanLast of lattice.hpp
__device__ __forceinline__ double lds_f64(unsigned int a) { double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_f64(unsigned int a, double v) { asm volatile("st.shared.f64 [%0], %1;" :: "r"(a), "d"(v)); }
__device__ __forceinline__ long long lds_s64(unsigned int a) { long long v; asm volatile("ld.shared.s64 %0, [%1];" : "=l"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_s64(unsigned int a, long long v) { asm volatile("st.shared.s64 [%0], %1;" :: "r"(a), "l"(v)); }

// One region in PATH FORM per thread: PP paths (padded with zero-weight paths) of L edges each, arc of edge l of path p at
// row l*PP + p.  q = sum_p prod_l w[arc]; every edge of path p gets the posterior r_p / q.  Registers only: PP independent
// multiply chains, no pool, no flags (the reference's P.x / exp / M algebra, src/Learner.cpp:530-545, for one small segment).
// Levels go in batches of LB = 24 / PP: every batch is ONE round trip (LB*PP loads in flight); a rolled loop pays a round
// trip per level.  One instance per PP serves every length: fully unrolled instances per (PP, L) made k_eval6 26 k
// instructions, and a warp that runs a rarely used instance waits for instruction fetches from the L2 (cold after the flush)
// far longer than for data -- measured 15-40 us for ONE group.
// The REDs follow the group's reduction plan (lattice.cpp, build_path_plans): every lane parks its rounded posteriors v[p]
// in its pool column, and walks its plan entries, each the cells (lane', p) of one arc of the group, summing v[p] of lane'
// (64-bit integers: exact and order independent, so the accumulators get the same bits as with one RED per cell) into ONE
// RED per entry.  reds = false: no REDs (timing experiments).
template <int PP>
__device__ __forceinline__ void kr_paths(const KRParams& P, const double* aw, const BigPool& pl, int L, long long g, long long off,
                                         int lane, unsigned long long* acc_g, long long& ll, bool reds)
{
    constexpr int LB = 24 / PP;
    const uint32_t* wp = P.words + off + lane;
    const long long poff = P.pgoff[g], pend = P.pgoff[g + 1];
    // more than one batch: ask for all rows of the group now (one 128-byte row per lane and round), so that the later
    // batches find them in the L2 instead of paying a DRAM round trip each (an 8 x 16 group took 26 us: twelve batches)
    if (L > LB)
        for (int i = lane; i < L * PP; i += 32) asm volatile("prefetch.global.L2 [%0];" :: "l"(P.words + off + (size_t)i * 32));
    const double W = P.typeW[g * 32 + lane];
    double r[PP];
#pragma unroll
    for (int p = 0; p < PP; ++p) r[p] = 1.0;
    for (int l0 = 0; l0 < L; l0 += LB) {
        uint32_t a[LB * PP];
#pragma unroll
        for (int i = 0; i < LB * PP; ++i) a[i] = l0 * PP + i < L * PP ? __ldg(wp + (size_t)(l0 * PP + i) * 32) : (uint32_t)P.n_arcs;
        // the plan rows are on their way to the L2 while the products are formed
        if (l0 == 0 && reds)
            for (long long i = poff + lane * 32; i < pend; i += 32 * 32) asm volatile("prefetch.global.L2 [%0];" :: "l"(P.pwords + i));
#pragma unroll
        for (int l = 0; l < LB; ++l)
            if (l0 + l < L) {
#pragma unroll
                for (int p = 0; p < PP; ++p) r[p] *= aw[a[l * PP + p]];
            }
    }
    double q = 0.0;
#pragma unroll
    for (int p = 0; p < PP; ++p) q += r[p];
    const bool ok = W > 0.0 && q > 0.0 && isfinite(q);
    if (W > 0.0) {
        const double lq = ok ? log(q) : -INFINITY;
        P.lq[g * 32 + lane] = lq;
        kr_loglik(P, W, ok, lq, ll);
    }
    if (!reds) return;
    const double sc = ok ? W * P.fx_scale / q : 0.0;
#pragma unroll
    for (int p = 0; p < PP; ++p) sts_s64(pl.p + (unsigned int)p * pl.ps, __double2ll_rn(r[p] * sc));
    __syncwarp();
    const unsigned int col0 = pl.p - (unsigned int)lane * 8u;          // the warp's lane 0
    const uint32_t* pp = P.pwords + poff + lane;
    const int prow = (int)((pend - poff) >> 5);
    long long s = 0;
    for (int r0 = 0; r0 < prow; r0 += 8) {
        uint32_t w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) w[j] = r0 + j < prow ? __ldcs(pp + (size_t)(r0 + j) * 32) : 0u;
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (r0 + j < prow) {
                const uint32_t c = (w[j] >> 16) & 0xffu;
                s += lds_s64(col0 + (c >> 3) * 8u + (c & 7u) * pl.ps);
                if (w[j] & kPLast) {
                    if (s) red_add64(acc_g + (w[j] & 0xffffu), (unsigned long long)s);
                    s = 0;
                }
            }
    }
    __syncwarp();                                              // the other lanes are done with this lane's column
}

// ---- big DAG regions: the stream format of lattice.hpp (CHECK words rescale, x values on a stack), one thread per region
// A group is walked by three blocks: big_fwd (forward chain), big_bwd (backward chain) and big_red (the REDs).  One warp
// runs all three (k_eval6 with one warp per group, kr_regions), or two warps split them (k_eval6, a CTA that owns one
// staged group): warp 0 big_fwd, warp 1 big_bwd<false> on its own pool at the same time, then warp 0 big_red<true>.
//
// The chain of a region is serial (every step reads the node value the previous step wrote): what a step costs is the
// latency of its dependent instructions.  Both chain loops are therefore free of branches inside a batch of eight words:
// every lane does the same loads, arithmetic and stores, and a lane whose word is padding, FIN or belongs to a shorter region
// works on slot 0 / arc 0 and stores into `trash` (one double per thread).  The decode and the weight loads of step k + 1
// then overlap the chain of step k.  Measured before (45 instructions with four branches per step): ~300 cycles per step,
// the 96-row group of a 125 k-string shard alone took 31 us of a 37 us region phase.  A lone warp still gets ~4 cycles per
// instruction whatever is done about its dependencies (interleaving the two chains in one instruction stream was measured
// twice: slower), but the chains are independent until the posteriors, so two warps -- two schedulers -- can walk them.
//
// The pool lives in shared memory and is addressed as such: node value of slot s of the lane at byte address p + s * ps.
// (A generic store to the shared window sits in the same in-order LSU queue as the chain's LDS/STS and takes longer to
// resolve.)  No memory clobbers: the pool and the staging area are touched by these volatile statements only, which keep
// their order among themselves; a clobber would pin every other memory access around each of them.
constexpr uint32_t kLEdge = 1u << 31, kLFin = 1u << 30, kLFirstIn = 1u << 29, kLLastOut = 1u << 28;   // = kLat* of lattice.hpp
constexpr int kLBand = 200;
__device__ __forceinline__ int lds_exp(unsigned int a) { int hi; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(hi) : "r"(a + 4u)); return (hi >> 20) & 0x7ff; }

// Where the words (row i: word of the lane) and the x stack (row i: 64 bits of the lane) of a group live.  BigSmem: the
// staging area of shared memory (k_eval6), byte addresses of the lane's column, so that the chain runs at shared-memory
// latency.  BigGmem: streamed from HBM, the stack in HBM, one slab per warp (kr_regions, k_eval6 without staging).
struct BigSmem {
    unsigned int w, x;
    __device__ __forceinline__ uint32_t word(int i) const { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(w + (unsigned int)i * 128u)); return v; }
    __device__ __forceinline__ long long ld(int i) const { long long v; asm volatile("ld.shared.b64 %0, [%1];" : "=l"(v) : "r"(x + (unsigned int)i * 256u)); return v; }
    __device__ __forceinline__ void st(int i, long long v) const { asm volatile("st.shared.b64 [%0], %1;" :: "r"(x + (unsigned int)i * 256u), "l"(v)); }
};
struct BigGmem {
    const uint32_t* w; double* x;
    __device__ __forceinline__ uint32_t word(int i) const { return __ldcs(w + (size_t)i * 32); }
    __device__ __forceinline__ long long ld(int i) const { return reinterpret_cast<const long long*>(x)[(size_t)i * 32]; }
    __device__ __forceinline__ void st(int i, long long v) const { reinterpret_cast<long long*>(x)[(size_t)i * 32] = v; }
};

// A CHECK word with pool slot mask m0: when the largest exponent among those slots has left the band 1023 +- kLBand, they
// are scaled back to exponent 0.  Returns the shift (0: nothing to do), which the chain subtracts from its exponent.
__device__ __forceinline__ int big_rescale(const BigPool& pl, uint32_t m0)
{
    if (!m0) return 0;
    int emax = 0;
    for (uint32_t m = m0; m; m &= m - 1) emax = max(emax, lds_exp(pl.p + (unsigned int)(__ffs(m) - 1) * pl.ps));
    if (emax == 0 || (emax >= 1023 - kLBand && emax <= 1023 + kLBand)) return 0;
    const int shift = 1023 - emax;
    for (uint32_t m = m0; m; m &= m - 1) { const unsigned int a = pl.p + (unsigned int)(__ffs(m) - 1) * pl.ps; sts_f64(a, scalbn(lds_f64(a), shift)); }
    return shift;
}

// The posterior scale below a CHECK word.  x = alpha_src * w carries the forward scale 2^E (E from the x stack), beta_dst
// the backward scale 2^F and q the scale 2^EQ, so posterior = (x * beta_dst) * sc with sc = sc0 * 2^(E + F - EQ),
// sc0 = W * fx_scale / q.  The one-warp backward chain (big_bwd<true>) and the two-warp RED pass (big_red<true>) both round
// (x * beta_dst) * sc once, with sc from here and from the same E, F and EQ: every schedule returns the same bits.
__device__ __forceinline__ double big_sc(double sc0, int E, int F, int EQ) { return scalbn(sc0, E + F - EQ); }

// Forward chain: alpha_src * w of every edge to the x stack, E to the CHECK slots; returns q (its exponent in EQ) and whether
// the lane holds a region at all.
template <class M>
__device__ __forceinline__ void big_fwd(const double* aw, const BigPool& pl, const M& m, int nw, double& qh, int& EQ, bool& any)
{
    sts_f64(pl.p, 1.0);
    int E = 0;
    EQ = 0; qh = 0.0; any = false;
    for (int i0 = 0; i0 < nw; i0 += 8) {
        uint32_t w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) w[j] = m.word(i0 + j);
        const bool chk = (i0 & 8) != 0;                       // word 7 of every second batch is a CHECK word (same index in all lanes)
        const uint32_t m0 = chk ? w[7] & 0xffffu : 0u;
        if (chk) w[7] = 0u;
        // decode first (addresses and weights of the eight steps are independent of the chain), then the chain itself:
        // per step  LDS node -> DMUL -> DADD -> select -> STS  and nothing else
        unsigned int fs[8], fd[8];
        double fw[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t wj = w[j];
            const bool edge = (wj & kLEdge) != 0;
            fs[j] = pl.p + (edge ? (wj >> 19) & 15u : (wj & 15u)) * pl.ps;   // (FIN: the exit node)
            fd[j] = edge ? pl.p + ((wj >> 23) & 15u) * pl.ps : pl.trash;
            fw[j] = aw[edge ? (wj & 0xffffu) : 0u];
            any |= edge;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t wj = w[j];
            const bool fin = (wj & (kLEdge | kLFin)) == kLFin;
            const double a = lds_f64(fs[j]);
            const double xv = a * fw[j];
            const double old = lds_f64(fd[j]);
            sts_f64(fd[j], (wj & kLFirstIn) ? xv : old + xv);
            m.st(i0 + j, __double_as_longlong(xv));
            qh = fin ? a : qh;
            EQ = fin ? E : EQ;
        }
        if (chk) {
            m.st(i0 + 7, (long long)E);
            E -= big_rescale(pl, m0);
        }
    }
}

// Backward chain, beta_dst of every edge, F at the CHECK words.  ROUND (one warp, after big_fwd on the same stack): the
// posterior of every edge, rounded to fixed point, replaces x in the stack (0 for every other word); sc0 = 0 when !ok.
// !ROUND (two warps): beta_dst of every edge and F at the CHECK words go to the stack of m -- the y stack, while the
// partner warp fills the x stack with big_fwd -- and big_red<true> forms the posteriors (ok, sc0, EQ unused).
template <bool ROUND, class M>
__device__ __forceinline__ void big_bwd(const double* aw, const BigPool& pl, const M& m, int nw, bool ok, double sc0, int EQ)
{
    double sc = sc0;
    int F = 0;
    for (int i0 = nw - 8; i0 >= 0; i0 -= 8) {
        uint32_t w[8];
        double xv[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { w[j] = m.word(i0 + j); if (ROUND) xv[j] = __longlong_as_double(m.ld(i0 + j)); }
        const bool chk = (i0 & 8) != 0;
        if (chk) {                                             // the CHECK word comes first in backward order
            const uint32_t m0 = w[7] & 0xffffu;
            F -= big_rescale(pl, m0);
            if (!ROUND) m.st(i0 + 7, (long long)F);
            else if (m0) sc = big_sc(sc0, (int)__double_as_longlong(xv[7]), F, EQ);
            w[7] = 0u;
        }
        unsigned int bd_[8], bs[8];
        double bw[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t wj = w[j];
            const bool edge = (wj & kLEdge) != 0;
            bd_[j] = pl.p + ((wj >> 23) & 15u) * pl.ps;
            bs[j] = (wj & (kLEdge | kLFin)) ? pl.p + (edge ? (wj >> 19) & 15u : (wj & 15u)) * pl.ps : pl.trash;   // (FIN: the exit node, beta = 1)
            bw[j] = aw[edge ? (wj & 0xffffu) : 0u];
        }
#pragma unroll
        for (int j = 7; j >= 0; --j) {
            const uint32_t wj = w[j];
            const bool edge = (wj & kLEdge) != 0;
            const bool fin = (wj & (kLEdge | kLFin)) == kLFin;
            const double bd = lds_f64(bd_[j]);
            const double c = bw[j] * bd;
            const double old = lds_f64(bs[j]);
            sts_f64(bs[j], fin ? 1.0 : ((wj & kLLastOut) ? c : old + c));
            if (ROUND) m.st(i0 + j, (edge && ok) ? __double2ll_rn(xv[j] * bd * sc) : 0ll);
            else if (!(j == 7 && chk)) m.st(i0 + j, __double_as_longlong(bd));
        }
    }
}

// The REDs, without dependencies between the steps.  XY = false: the posteriors the one-warp big_bwd left rounded in the
// stack of x, in word order.  XY = true: formed here as (x * y) * sc from the x stack of big_fwd and the y stack of
// big_bwd<false>, backward, because sc changes at the CHECK words.
template <bool XY, class M>
__device__ __forceinline__ void big_red(const M& x, const M& y, int nw, bool ok, double sc0, int EQ, unsigned long long* acc_g)
{
    double sc = sc0;
    for (int k = 0; k < nw; k += 8) {
        const int i0 = XY ? nw - 8 - k : k;
        uint32_t w[8];
        long long xv[8], yv[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { w[j] = x.word(i0 + j); xv[j] = x.ld(i0 + j); if (XY) yv[j] = y.ld(i0 + j); }
        if (XY && (i0 & 8)) {
            if (w[7] & 0xffffu) sc = big_sc(sc0, (int)xv[7], (int)yv[7], EQ);
            w[7] = 0u;
        }
#pragma unroll
        for (int j = 7; j >= 0; --j) {
            long long v = xv[j];
            if (XY) {
                if (!(w[j] & kLEdge) || !ok) continue;
                v = __double2ll_rn(__longlong_as_double(xv[j]) * __longlong_as_double(yv[j]) * sc);
            }
            if (v) red_add64(acc_g + (w[j] & 0xffff), (unsigned long long)v);
        }
    }
}

// log q of the lane's region from the forward chain into lq[] and the log-likelihood; returns whether q is usable and in
// sc0 the posterior scale W * fx_scale / q (0 if not)
__device__ __forceinline__ bool big_lq(const KRParams& P, double W, long long g, int lane, double qh, int EQ, bool any, long long& ll, double& sc0)
{
    const bool ok = any && qh > 0.0 && isfinite(qh);
    if (any) {
        const double lq = ok ? log(qh) + (double)EQ * 0.69314718055994530942 : -INFINITY;
        P.lq[g * 32 + lane] = lq;
        kr_loglik(P, W, ok, lq, ll);
    }
    sc0 = ok ? W * P.fx_scale / qh : 0.0;
    return ok;
}

// One big group on one warp: forward chain, log q, backward chain rounding the posteriors, REDs (reds = false: none).
template <class M>
__device__ __forceinline__ void big_one(const KRParams& P, const double* aw, const BigPool& pl, const M& m, int nw, long long g, int lane,
                                        unsigned long long* acc_g, long long& ll, bool reds)
{
    const double W = P.typeW[g * 32 + lane];
    double qh, sc0;
    int EQ;
    bool any;
    big_fwd(aw, pl, m, nw, qh, EQ, any);
    const bool ok = big_lq(P, W, g, lane, qh, EQ, any, ll, sc0);
    big_bwd<true>(aw, pl, m, nw, ok, sc0, EQ);
    if (reds) big_red<false>(m, m, nw, ok, sc0, EQ, acc_g);
}

template <int ACC, int MAXNT, bool AWG = false>
__global__ void __launch_bounds__(MAXNT, 1) kr_regions(const KRParams P)
{
    extern __shared__ unsigned long long smem[];
    __shared__ double s_trash[MAXNT];                         // where the lanes without an edge store (big_fwd, big_bwd)
    const int tid = threadIdx.x, NT = blockDim.x, lane = tid & 31;
    // [n_arcs + 1] arc weights, the last entry the zero weight of padding: a copy in shared memory, or (AWG: the table does not
    // fit) P.aw itself, which then has the zero entry behind it
    const double* aw = AWG ? P.aw : reinterpret_cast<const double*>(smem);
    double* pool = (AWG ? reinterpret_cast<double*>(smem) : reinterpret_cast<double*>(smem) + P.n_arcs + 1) + tid;   // slot s of this thread at pool[s*NT]
    if (!AWG) { double* t = reinterpret_cast<double*>(smem); for (int i = tid; i <= P.n_arcs; i += NT) t[i] = i < P.n_arcs ? P.aw[i] : 0.0; }
    __syncthreads();
    const long long gwarp = ((long long)blockIdx.x * NT + tid) >> 5;
    double* const xs = P.xs + (size_t)gwarp * P.xs_rows * 32 + lane;
    unsigned long long* const acc_g = P.acc + (size_t)(blockIdx.x % P.replicas) * (size_t)P.n_arcs;
    const bool reds = ACC != ACC_NONE;                        // ACC_NONE: no REDs at all (timing experiment)
    const BigPool pl{(unsigned int)__cvta_generic_to_shared(pool), (unsigned int)NT * 8u, (unsigned int)__cvta_generic_to_shared(&s_trash[tid])};
    // groups are sorted by cost (DAG regions first, then path form by paths and length) and handed out dynamically, one
    // at a time; the id of the next group is requested while the current one is processed
    long long g = 0, ll = 0;
    if (lane == 0) g = (long long)atomicAdd(P.counter, 1u);
    g = __shfl_sync(FULL, g, 0);
    while (g < P.n_groups) {
        long long gn = 0;
        if (lane == 0) gn = (long long)atomicAdd(P.counter, 1u);
        const int rows = P.grows[g];
        const long long off = P.goff[g];
        if (rows & 0x10000) {                                  // path form: paths << 8 | length
            const int L = rows & 0xff;
            switch ((rows >> 8) & 0xff) {
                case 2: kr_paths<2>(P, aw, pl, L, g, off, lane, acc_g, ll, reds); break;
                case 3: kr_paths<3>(P, aw, pl, L, g, off, lane, acc_g, ll, reds); break;
                case 4: kr_paths<4>(P, aw, pl, L, g, off, lane, acc_g, ll, reds); break;
                case 6: kr_paths<6>(P, aw, pl, L, g, off, lane, acc_g, ll, reds); break;
                default: kr_paths<8>(P, aw, pl, L, g, off, lane, acc_g, ll, reds); break;
            }
        } else big_one(P, aw, pl, BigGmem{P.words + off + lane, xs}, (int)((P.goff[g + 1] - off) >> 5), g, lane, acc_g, ll, reds);
        g = __shfl_sync(FULL, gn, 0);
    }
    // the CTA's share of the log-likelihood: integer sums (exact, order independent), one RED per CTA
#pragma unroll
    for (int o = 16; o; o >>= 1) ll += __shfl_xor_sync(FULL, ll, o);
    __syncthreads();                                           // the pool is free now
    long long* part = reinterpret_cast<long long*>(pool - tid);
    if (lane == 0) part[tid >> 5] = ll;
    __syncthreads();
    if (tid == 0) {
        long long s = 0;
        for (int w = 0; w < (NT >> 5); ++w) s += part[w];
        unsigned long long nf = 0;
        if (blockIdx.x == 0)
            for (int k = 0; k < P.n_llpart; ++k) { s += P.llpart[2 * k]; nf += (unsigned long long)P.llpart[2 * k + 1]; }
        if (s) atomicAdd(P.red, (unsigned long long)s);
        if (nf) atomicAdd(P.red + 1, nf);
    }
}

// ------------------------------------------------------------------------------------------
struct KSParams {
    const double* __restrict__ logaw;     // [n_arcs] log weight of every combined arc
    const uint32_t* __restrict__ words;   // chunk-interleaved super-groups (lattice.hpp, SegmentedCorpus)
    const int64_t* __restrict__ sgoff;    // [n_sgroups+1]
    const int32_t* __restrict__ gref;     // [n_sgroups*16] leading rows of a group that hold region type ids
    const double* __restrict__ lq;        // log q per region type (written by kr_regions)
    const double* __restrict__ p;         // [n_sgroups*16*32] p_s in group order (0 = padding lane)
    double* logq;                         // [n_sgroups*16*32] log q_s in group order
    long long n_sgroups;
    unsigned int* counter;
    int n_arcs;
};

// KS: one CTA of 16 warps per super-group of 16 groups, one warp per group, one thread per string.
//   log q_s = sum over the string's bridge arcs of log w[arc]  (two 16-bit ids per word; 8-byte table in shared
//             memory; the host scheduled the ids so that a half-warp reads 16 different bank pairs)
//           + sum over its regions of lq[type]                  (gathers from L2)
// The words of a super-group are interleaved chunk by chunk, so the 16 warps stream ONE contiguous region
// (DRAM sees long bursts: 5.6 TB/s against 4.3 TB/s with one private block per warp, profiles/microbench_stream.cu).
// Measured dead ends, kept in the history: a cp.async (LDGSTS) ring and a TMA bulk-copy ring per warp were both
// slower than this register double buffer (the limit was DRAM burst locality, not bytes in flight).
constexpr int kKsRows = 8, kKsWarps = 16;      // = kKsChunkRows, kKsSuper of lattice.hpp

// AWG: the table does not fit shared memory and is read from HBM/L2 (P.logaw has n_arcs + 16 entries, the last 16 zero)
template <bool AWG = false>
__global__ void __launch_bounds__(kKsWarps * 32, 2) ks_strings(const KSParams P)
{
    extern __shared__ __align__(128) unsigned long long smem[];
    __shared__ long long s_next[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double* tab = AWG ? P.logaw : reinterpret_cast<const double*>(smem);   // [n_arcs + 16]; ids n_arcs.. (padding, one per bank pair) -> 0
    if (!AWG) { double* t = reinterpret_cast<double*>(smem); for (int i = tid; i < P.n_arcs + 16; i += kKsWarps * 32) t[i] = i < P.n_arcs ? P.logaw[i] : 0.0; }
    if (tid == 0) s_next[0] = (long long)atomicAdd(P.counter, 1u);
    __syncthreads();
    int par = 0;
    for (long long sg = s_next[0]; sg < P.n_sgroups;) {
        if (tid == 0) s_next[par ^ 1] = (long long)atomicAdd(P.counter, 1u);   // the next super-group, fetched early
        const long long o = P.sgoff[sg];
        const int chunks = (int)((P.sgoff[sg + 1] - o) / (kKsWarps * kKsRows * 32));
        const long long g = sg * kKsWarps + warp;
        const int nref = P.gref[g];
        const double ps = P.p[g * 32 + lane];
        const uint32_t* wp = P.words + o + (size_t)warp * (kKsRows * 32) + lane;   // chunk c at wp + c * (16*8*32)
        constexpr size_t CS = (size_t)kKsWarps * kKsRows * 32;
        double s0 = 0.0, s1 = 0.0, r = 0.0, v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
        uint32_t a[kKsRows];
#pragma unroll
        for (int j = 0; j < kKsRows; ++j) a[j] = __ldcs(wp + j * 32);
        for (int c = 0; c < chunks; ++c) {
            uint32_t b[kKsRows];
            if (c + 1 < chunks) {
#pragma unroll
                for (int j = 0; j < kKsRows; ++j) b[j] = __ldcs(wp + (size_t)(c + 1) * CS + j * 32);
            }
            if (c * kKsRows < nref) {                           // chunk with region references (the first one, rarely two)
#pragma unroll
                for (int j = 0; j < kKsRows; ++j) {
                    const int i = c * kKsRows + j;
                    if (i < nref) {
                        const double v = P.lq[a[j]];            // the first four are added at the end (latency overlaps)
                        if (i == 0) v0 = v; else if (i == 1) v1 = v; else if (i == 2) v2 = v; else if (i == 3) v3 = v; else r += v;
                    } else { s0 += tab[a[j] & 0xffffu]; s1 += tab[a[j] >> 16]; }
                }
            } else {
#pragma unroll
                for (int j = 0; j < kKsRows; ++j) { s0 += tab[a[j] & 0xffffu]; s1 += tab[a[j] >> 16]; }
            }
            if (c + 1 < chunks) {
#pragma unroll
                for (int j = 0; j < kKsRows; ++j) a[j] = b[j];
            }
        }
        const double lqs = (s0 + s1) + (r + ((v0 + v1) + (v2 + v3)));
        if (ps != 0.0) P.logq[g * 32 + lane] = lqs;
        __syncthreads();
        par ^= 1;
        sg = s_next[par];
    }
}

// no region types at all: the bridge partials are the whole log-likelihood
__global__ void k_add_llpart(const long long* __restrict__ llpart, int n, unsigned long long* red)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        long long s = 0, nf = 0;
        for (int k = 0; k < n; ++k) { s += llpart[2 * k]; nf += llpart[2 * k + 1]; }
        if (s) atomicAdd(red, (unsigned long long)s);
        if (nf) atomicAdd(red + 1, (unsigned long long)nf);
    }
}

// log q of the strings of the segmented path, group order -> string id order
__global__ void k_scatter_logq(long long n, const int32_t* __restrict__ ksid, const double* __restrict__ logq_k, double* logq)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && ksid[i] >= 0) logq[ksid[i]] = logq_k[i];
}

// The bridge part of the log-likelihood: sum over arcs of (sum_s p_s * times the arc is a bridge of s) * log w[arc].
// const_acc holds the first factor in the fixed point of the gradient accumulators (it is the constant part of the
// gradient as well).  Called by all threads of a CTA with the arc of the thread (c = 0 beyond the last
// arc); CTAs that hold arcs store their partial [value, non-finite terms] to llpart[blockIdx.x] (no reset needed).
__device__ __forceinline__ void bridge_loglik_partial(unsigned long long c, double l, double inv_fx, double ll_scale, long long* llpart)
{
    __shared__ long long s_part[32][2];
    long long v = 0, nf = 0;
    if (c) {
        if (isfinite(l)) v = __double2ll_rn((double)(long long)c * inv_fx * l * ll_scale);
        else nf = 1;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) { v += __shfl_xor_sync(FULL, v, o); nf += __shfl_xor_sync(FULL, nf, o); }
    if ((threadIdx.x & 31) == 0) { s_part[threadIdx.x >> 5][0] = v; s_part[threadIdx.x >> 5][1] = nf; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) { v += s_part[w][0]; nf += s_part[w][1]; }
        llpart[2 * blockIdx.x] = v;
        llpart[2 * blockIdx.x + 1] = nf;
    }
}

// per combined arc: aw = a(u,v) * b(v,e) and its logarithm, straight from x
__global__ void __launch_bounds__(256) k_arc_weights_log(int n_arcs, const int32_t* __restrict__ arc_tid, const int32_t* __restrict__ arc_eid,
                                  const int32_t* __restrict__ trans_tp, const int32_t* __restrict__ emis_tp,
                                  const double* __restrict__ x, double* aw, double* logaw,
                                  const unsigned long long* __restrict__ const_acc, double inv_fx, double ll_scale, long long* llpart)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double l = 0.0;
    if (i < n_arcs) {
        l = logweight_of(trans_tp[arc_tid[i]], x, 0) + (arc_eid[i] < 0 ? 0.0 : logweight_of(emis_tp[arc_eid[i]], x, 0));
        logaw[i] = l;
        aw[i] = exp(l);
    }
    bridge_loglik_partial(i < n_arcs ? const_acc[i] : 0ull, l, inv_fx, ll_scale, llpart);
}


// Device-side barrier over the ranks of the communicator through peer memory (benchmark helper: it lines the ranks
// up between two timed evaluations).  One warp: lane r tells rank r "rank `rank` reached epoch e", then waits for
// rank r's word.  Words of epoch e live at bar[(e & 1) * nranks + sender].  Bounded wait (~2 s).
struct PeerBarrierParams {
    unsigned long long* peers[8];
    size_t bar_off;
    int nranks, rank;
    unsigned long long epoch;
};
__global__ void k_peer_barrier(const PeerBarrierParams P)
{
    const int lane = threadIdx.x;
    if (lane < P.nranks) {
        const size_t slot = P.bar_off + (size_t)(P.epoch & 1ull) * P.nranks;
        *reinterpret_cast<volatile unsigned long long*>(P.peers[lane] + slot + P.rank) = P.epoch;
        const volatile unsigned long long* src = P.peers[P.rank] + slot + lane;
        const long long t0 = clock64();
        while (*src != P.epoch)
            if (clock64() - t0 > 4000000000ll) break;
    }
}

}  // namespace wfsa
