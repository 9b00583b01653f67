// w-fsa_b200/csrc/kernels_eval6.cuh -- ONE launch per objective+gradient evaluation of the segmented path.
//
// k_eval6 is a persistent grid (one CTA per SM, all resident) that runs the whole evaluation
// (Learner::ComputeModeledProbs + ComputeObjective + ComputeGrad, /root/reference/src/Learner.cpp:515-553,
// src/QuasiNewtonLearner.cpp:93-125) in four phases:
//   P0  every CTA builds the table of arc weights in shared memory straight from x
//       (exp(x) once per parameter, then one product per combined arc), adds its share of the bridge part of the
//       log-likelihood (sum_arc c[arc] * log w[arc], kernels_seg.cuh) and re-arms the accumulator buffer and the
//       ticket counter of the NEXT evaluation (two of each, used alternately);
//   P1  region types, 32 to a warp, handed out by a ticket counter (kr_regions' loop).  Path-form types: the rows of a group
//       in batches of one round trip each, one RED per distinct arc of the group from its reduction plan (kr_paths);
//       group descriptors of the regular classes come from a class table in shared memory, not from HBM; big DAG groups are
//       staged in shared memory and, when a CTA owns one, walked by two warps (forward chain on warp 0, backward chain on
//       warp 1, REDs on warp 0: kernels_seg.cuh big_fwd / big_bwd<false> / big_red<true>), else by one (big_one);
//   P2  grid barrier (arrival counter in HBM);
//   P3  fold: one warp per edge gathers the (arc, replica) cells of the edge; with several ranks the per-edge sums are
//       exchanged through NVLink peer memory as self-validating packets (ll_exchange, kernels_seg.cuh) and the warp
//       converts the total to grad[i]; one warp does the same for [loglik, non-finite terms].
// Everything an evaluation needs that changes from call to call lives in device memory (x, the fixed-point scale of
// the log-likelihood behind x, the epoch in ctl[3]), so the launch parameters are constant per parameter map and
// wfsa_dev_eval replays the launch as a CUDA graph of this one kernel: with host buffers CTA 0 fetches x from mapped pinned
// memory (x_host) and the results go straight into mapped pinned memory as well (out, done_flag) -- no copy nodes.
#pragma once
#include "kernels_seg.cuh"

namespace wfsa {

constexpr int kE6MaxCls = 160;
struct Eval6Cls { int first, code; long long off; };        // groups [first, next.first): code = grows value, off = word offset of the first

struct Eval6Params {
    // region types (KR layout, lattice.hpp)
    const uint32_t* __restrict__ words;
    const int64_t* __restrict__ goff;
    const int32_t* __restrict__ grows;
    const double* __restrict__ typeW;
    const uint32_t* __restrict__ pwords;        // reduction plan of the path-form groups
    const int64_t* __restrict__ pgoff;
    double* lq;
    long long n_groups, n_big;                  // groups [0, n_big): big DAG regions (descriptor from goff/grows)
    int static_pct;                             // share of the regular groups dealt out statically per CTA (the rest: ticket counter)
    const Eval6Cls* __restrict__ cls;           // classes of the groups [n_big, n_groups), ascending `first`
    int n_cls;
    double* xs; size_t xs_rows;
    // weights
    const int2* __restrict__ arc_tp;            // per arc: trimmed parameter of its transition / emission; -1 weight 1, -2 weight 0
    const double* x;                            // [n + 1]: x, then log2 of the fixed-point scale of loglik
    const double* x_host; double* x_w;          // host-buffer call: x waits in mapped pinned host memory (x_host); CTA 0 copies it to
                                                // x_w (= x) and publishes the epoch in ctl[5], the other CTAs wait for that word
    int n, n_arcs, direct_exp;                  // direct_exp: exp per arc (x does not fit the scratch area)
    double* aw_g;                               // AWG instance: [n_arcs + 1] arc weights in HBM/L2 (they do not fit shared memory); every CTA
                                                // writes the whole table (identical values) before it reads any of it
    const unsigned long long* __restrict__ const_acc;
    unsigned long long* acc;                    // [2][replicas][n_arcs]
    int replicas;
    double fx_scale, inv_fx;
    unsigned long long* red;                    // [2] fixed-point loglik, non-finite terms; zero between evaluations
    unsigned int* ctl;                          // [0..1] ticket counters, [2] barrier arrivals (monotonic), [3] epoch (starts at 1),
                                                // [4] CTAs of the current host-buffer launch that are through, [5] epoch whose x has been fetched from the host,
                                                // [6] host-buffer launches completed
    unsigned int* done_flag;                    // host-mapped word that receives the count of host-buffer launches when the whole grid has written `out`
                                                // (the host-buffer call polls it instead of waiting for a D2H copy and a stream sync), or nullptr
    // fold
    int n_edges;
    const int32_t* __restrict__ e_off; const int32_t* __restrict__ e_arc; const int32_t* __restrict__ edge_tp;
    double* out;                                // [n + 3]: loglik, non-finite terms, grad[n], epoch of a timed-out exchange
    // ranks
    unsigned long long* peers[8];
    size_t ll_off;
    int nranks, rank, pk_words;
    int debug;                                  // stamps[4] = longest group (ns << 32 | rows code), stamps[5] = latest end of P1 (ns)
    int pool_slots;                             // pool doubles per thread (region-local node values)
    int big_dedicate;                           // few big groups: the other warps of a CTA that owns one wait until it is done
    int big_slots, big_rows;                    // staging areas for big DAG groups in shared memory behind the pool: how many, rows each
    unsigned long long* stamps;                 // [4] profiling: ns spent in P0, P1, P2, P3 by CTA 0 (sums), or nullptr
};

__device__ __forceinline__ unsigned long long e6_timer()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ unsigned int e6_ld_acquire(const unsigned int* p)
{
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Sum of the (arc, replica) cells of one edge by a HALF-warp (hl = lane in the half, hmask = its lanes).  The first
// (up to 16) arc ids of the edge are already in `first`, one per lane.
__device__ __forceinline__ unsigned long long e6_fold_edge(const unsigned long long* __restrict__ acc, int n_arcs, int replicas,
                                                          const int32_t* __restrict__ e_arc, int k0, int na, int first, int hl, unsigned hmask)
{
    unsigned long long s = 0;
    for (int b = 0; b < na; b += 16) {
        const int nb = min(16, na - b);
        const int mine = b == 0 ? first : (hl < nb ? e_arc[k0 + b + hl] : 0);
        const int cells = nb * replicas;
        for (int c0 = 0; c0 < cells; c0 += 64) {
            unsigned long long v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int c = c0 + j * 16 + hl;
                const int a = __shfl_sync(hmask, mine, min(c / replicas, nb - 1), 16);
                v[j] = c < cells ? __ldcg(acc + (size_t)(c % replicas) * n_arcs + a) : 0ull;
            }
            s += (v[0] + v[1]) + (v[2] + v[3]);
        }
    }
#pragma unroll
    for (int o = 8; o; o >>= 1) s += __shfl_xor_sync(hmask, s, o, 16);
    return s;
}

// one payload word across the ranks: lane r sends the local value to rank r as two self-validating 8-byte packets
// {32 data bits, 32-bit epoch} and polls the packets rank r sent (ll_exchange of kernels_seg.cuh with the epoch as flag);
// called by a half-warp (at most 8 ranks)
__device__ __forceinline__ unsigned long long e6_exchange(const Eval6Params& P, unsigned int epoch, int w, unsigned long long s,
                                                          int hl, unsigned hmask, bool& timeout)
{
    unsigned long long v = 0;
    const int parity = (int)(epoch & 1u);
    if (hl < P.nranks) {
        volatile unsigned long long* dst = P.peers[hl] + P.ll_off + (((size_t)parity * P.nranks + P.rank) * P.pk_words + w) * 2;
        const unsigned long long fl = (unsigned long long)epoch << 32;
        dst[0] = (s & 0xffffffffull) | fl;
        dst[1] = (s >> 32) | fl;
        const volatile unsigned long long* src = P.peers[P.rank] + P.ll_off + (((size_t)parity * P.nranks + hl) * P.pk_words + w) * 2;
        const long long t0 = clock64();
        unsigned long long a = src[0], b = src[1];
        while ((unsigned int)(a >> 32) != epoch || (unsigned int)(b >> 32) != epoch) {
            if (clock64() - t0 > 60000000000ll) { timeout = true; break; }       // ~30 s: a peer is gone
            a = src[0]; b = src[1];
        }
        v = (a & 0xffffffffull) | (b << 32);
    }
#pragma unroll
    for (int o = 8; o; o >>= 1) v += __shfl_xor_sync(hmask, v, o, 16);
    return v;
}

// log weight of every combined arc, for ks_strings (k_eval6 keeps the weights in shared memory; log q per string is
// computed on request only, from the x of the last evaluation)
__global__ void __launch_bounds__(256) k_arc_logw(int n_arcs, const int2* __restrict__ arc_tp, const double* __restrict__ x, double* logaw)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_arcs) return;
    const int2 tp = arc_tp[i];
    logaw[i] = (tp.x == -2 || tp.y == -2) ? -INFINITY : (tp.x >= 0 ? x[tp.x] : 0.0) + (tp.y >= 0 ? x[tp.y] : 0.0);
}

template <int NT, bool AWG = false>
__global__ void __launch_bounds__(NT, 1) k_eval6(const Eval6Params P)
{
    extern __shared__ unsigned long long smem[];
    __shared__ Eval6Cls s_cls[kE6MaxCls];
    __shared__ long long s_part[NT / 32][2];
    __shared__ unsigned int s_ticket;                         // next entry of this CTA's static share of the regular groups
    __shared__ int s_bigleft;                                 // warps of this CTA still busy with big DAG groups
    __shared__ double s_trash[NT];                            // where the lanes without an edge store (big_fwd, big_bwd)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double* aw = AWG ? P.aw_g : reinterpret_cast<double*>(smem);   // [n_arcs + 1]; the last entry is the zero weight of padding
    double* const sbase = AWG ? reinterpret_cast<double*>(smem) : aw + P.n_arcs + 1;    // shared memory behind the weight table
    double* pool = sbase + tid;                               // slot s of this thread at pool[s*NT]
    double* ex = sbase;                                       // exp(x), in the pool area until the weights are built
    const bool prof = P.stamps && blockIdx.x == 0 && tid == 0;
    unsigned long long t0 = 0, t1 = 0, t2 = 0, t3 = 0;
    if (prof) { t0 = e6_timer(); if (P.debug) P.stamps[6] = t0; }
    const bool tline = (P.debug & 16) && tid == 0;
    unsigned long long tl0 = 0, tl1 = 0, tl2 = 0, tl3 = 0;
    if (tline) tl0 = e6_timer();
    // Big DAG groups are dealt out statically: big group b to warp b / gridDim.x of CTA b % gridDim.x (see P1).  Warp w
    // owns staging area w behind the pool (if w < big_slots); the words of its first big group are on their way to it
    // before anything else happens.
    const long long big0 = (long long)blockIdx.x + (long long)warp * gridDim.x;
    double* const sxs = sbase + (size_t)P.pool_slots * NT + (size_t)warp * P.big_rows * 48 + lane;    // [rows][32] doubles
    uint32_t* const sw = reinterpret_cast<uint32_t*>(sxs - lane + (size_t)P.big_rows * 32) + lane;                 // [rows][32] words
    auto stage_big = [&](long long g) {                        // true: the rows of group g are being copied to the staging area
        const long long off = P.goff[g];
        const int nw = (int)((P.goff[g + 1] - off) >> 5);
        if (warp >= P.big_slots || nw > P.big_rows) return false;
        const uint32_t* gp = P.words + off + lane;
        for (int i = 0; i < nw; ++i) {
            const unsigned int sa = (unsigned int)__cvta_generic_to_shared(sw + (size_t)i * 32);
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(sa), "l"(gp + (size_t)i * 32) : "memory");
        }
        return true;
    };
    bool staged = big0 < P.n_big && stage_big(big0);
    if (tid == 0) {
        int nbw = 0;
        for (int w = 0; w < NT / 32; ++w) nbw += (long long)blockIdx.x + (long long)w * gridDim.x < P.n_big;
        s_bigleft = P.big_dedicate ? nbw : 0;
        s_ticket = 0u;
    }
    // ---- P0: weights ------------------------------------------------------------------------------------------
    // every load that depends on nothing goes out first: an iteration that waits for its own load costs a round trip each
    const unsigned int epoch = *reinterpret_cast<volatile unsigned int*>(P.ctl + 3);     // bumped by CTA 0 behind the grid barrier
    int2 tpv[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) tpv[j] = tid + j * NT < P.n_arcs ? P.arc_tp[tid + j * NT] : make_int2(-2, -2);
    const int bi = (int)blockIdx.x + tid * (int)gridDim.x;    // bridge part of the log-likelihood: arc i on CTA i % gridDim.x
    const unsigned long long bc = bi < P.n_arcs ? P.const_acc[bi] : 0ull;
    const int2 btp = bi < P.n_arcs ? P.arc_tp[bi] : make_int2(-2, -2);
    for (int i = tid; i < P.n_cls; i += NT) s_cls[i] = P.cls[i];
    if (P.x_host) {                                            // (uniform over the grid)
        if (blockIdx.x == 0) {
            for (int i0 = tid; i0 <= P.n; i0 += 8 * NT) {                          // eight loads per thread in flight: a PCIe round trip per batch
                double hv[8];                                                       // (one load per iteration was measured: 10.5 us for 27 KB)
#pragma unroll
                for (int j = 0; j < 8; ++j) hv[j] = i0 + j * NT <= P.n ? __ldcv(P.x_host + i0 + j * NT) : 0.0;
#pragma unroll
                for (int j = 0; j < 8; ++j) if (i0 + j * NT <= P.n) P.x_w[i0 + j * NT] = hv[j];
            }
            __threadfence();
            __syncthreads();
            if (tid == 0) asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(P.ctl + 5), "r"(epoch) : "memory");
        } else {
            if (tid == 0) while (e6_ld_acquire(P.ctl + 5) != epoch) { }
            __syncthreads();
        }
    }
    if (!P.direct_exp)
        for (int i0 = tid; i0 < P.n; i0 += 8 * NT) {
            double xv[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) xv[j] = i0 + j * NT < P.n ? P.x[i0 + j * NT] : 0.0;
#pragma unroll
            for (int j = 0; j < 8; ++j) if (i0 + j * NT < P.n) ex[i0 + j * NT] = exp(xv[j]);
        }
    const double ll_scale = scalbn(1.0, (int)P.x[P.n]), inv_ll = scalbn(1.0, -(int)P.x[P.n]);
    const int par = (int)(epoch & 1u);
    const size_t acc_words = (size_t)P.replicas * P.n_arcs;
    long long ll = 0;
    unsigned long long nf = 0;
    auto arc_logw = [&](int2 tp) { return (tp.x == -2 || tp.y == -2) ? -INFINITY : (tp.x >= 0 ? P.x[tp.x] : 0.0) + (tp.y >= 0 ? P.x[tp.y] : 0.0); };
    // every term of the bridge sum is rounded once, so the sum does not depend on the grid size
    if (bc) { const double l = arc_logw(btp); if (isfinite(l)) ll += __double2ll_rn((double)(long long)bc * P.inv_fx * l * ll_scale); else ++nf; }
    for (int i = bi + NT * (int)gridDim.x; i < P.n_arcs; i += NT * (int)gridDim.x) {
        const unsigned long long c = P.const_acc[i];
        if (c) { const double l = arc_logw(P.arc_tp[i]); if (isfinite(l)) ll += __double2ll_rn((double)(long long)c * P.inv_fx * l * ll_scale); else ++nf; }
    }
    __syncthreads();                                           // exp(x) complete
    for (int i0 = tid; i0 <= P.n_arcs; i0 += 8 * NT) {
        if (i0 != tid) {
#pragma unroll
            for (int j = 0; j < 8; ++j) tpv[j] = i0 + j * NT < P.n_arcs ? P.arc_tp[i0 + j * NT] : make_int2(-2, -2);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int i = i0 + j * NT;
            if (i > P.n_arcs) continue;
            const int2 tp = tpv[j];
            double w = 0.0;
            if (tp.x != -2 && tp.y != -2) {
                if (P.direct_exp) w = exp((tp.x >= 0 ? P.x[tp.x] : 0.0) + (tp.y >= 0 ? P.x[tp.y] : 0.0));
                else w = (tp.x >= 0 ? ex[tp.x] : 1.0) * (tp.y >= 0 ? ex[tp.y] : 1.0);
            }
            aw[i] = w;                                         // i == n_arcs: the zero weight of padding
        }
    }
    if (AWG) __threadfence();                                  // (the table is in global memory: this CTA's copy is complete before any of its threads reads it)
    __syncthreads();                                           // weights complete; exp(x) scratch is free: the pool starts here
    if (prof) t1 = e6_timer();
    if (tline) tl1 = e6_timer();
    // ---- P1: region types -------------------------------------------------------------------------------------
    KRParams R{};
    R.words = P.words; R.goff = P.goff; R.typeW = P.typeW; R.pwords = P.pwords; R.pgoff = P.pgoff; R.lq = P.lq; R.xs = P.xs; R.xs_rows = P.xs_rows;
    R.fx_scale = P.fx_scale; R.ll_scale = ll_scale; R.red = P.red; R.n_arcs = P.n_arcs;
    const bool path_reds = !(P.debug & 8);                     // timing experiment (debug bit 3): no REDs from path-form types
    const BigPool pl{(unsigned int)__cvta_generic_to_shared(pool), (unsigned int)NT * 8u, (unsigned int)__cvta_generic_to_shared(&s_trash[tid])};
    unsigned int* const counter = P.ctl + par;
    unsigned long long* const acc_g = P.acc + (size_t)par * acc_words + (size_t)(blockIdx.x % P.replicas) * (size_t)P.n_arcs;
    const long long gwarp = (long long)blockIdx.x * (NT / 32) + warp;
    double* const xs = P.xs + (size_t)gwarp * P.xs_rows * 32 + lane;
    // The big DAG groups (one long dependent chain per thread: the stragglers of this phase) are dealt out statically, big
    // group b to warp b / gridDim.x of CTA b % gridDim.x, so that they start first and never share an SM when there are
    // fewer of them than SMs.  (Handed out by the ticket counter, the sixteen warps of the first CTA to finish P0 took
    // sixteen of them at once: 45 us for one CTA while the others idled.)  The regular groups follow by ticket.  When
    // there are few big groups (big_dedicate), the other warps of their CTAs wait for them: a chain that shares the LSU
    // with fifteen warps issuing 32-sector REDs runs at 400 cycles per step instead of ~100.
    // Regular groups: the first `static_pct` per cent are dealt out statically, group n_big + b + k * gridDim.x to CTA b,
    // whose warps take them through a counter in SHARED memory; only the rest goes through the ticket counter in HBM,
    // which evens out the tail.  One global counter for all 18.7 k groups of config 4 was the limit of the whole phase:
    // same-address atomics retire at ~3 ns each in the L2, i.e. 55 us, and the profile showed the warps waiting for
    // their next ticket (the SHFL behind the atomic) more than for anything else.
    // With dedicated CTAs (few big groups, each alone on its SM until it is done) the static share is dealt out among the
    // other CTAs only: a dedicated CTA starts on the regular groups late and takes what the ticket counter has left.
    const long long n_rest = P.n_groups - P.n_big;
    const int n_ded = P.big_dedicate ? (int)(P.n_big < (long long)gridDim.x ? P.n_big : (long long)gridDim.x) : 0;
    const int n_free = (int)gridDim.x - n_ded;
    const bool ded = (int)blockIdx.x < n_ded;
    const long long n_stat = n_free > 0 ? P.n_big + n_rest * P.static_pct / 100 / (long long)n_free * (long long)n_free : P.n_big;
    auto fetch = [&]() -> long long {                          // lane 0 only
        if (!ded) {
            const long long gs = P.n_big + (long long)((int)blockIdx.x - n_ded) + (long long)atomicAdd(&s_ticket, 1u) * n_free;
            if (gs < n_stat) return gs;
        }
        return n_stat + (long long)atomicAdd(counter, 1u);
    };
    unsigned long long dbg_max = 0;
    long long big = big0;
    long long g = 0;
    // At most one big group per CTA (n_big <= grid: group blockIdx.x on warp 0): the CTA walks the two chains of the group on
    // two warps, warp 0 forward, warp 1 backward (kernels_seg.cuh, big_fwd / big_bwd<false> / big_red<true>); warp 1 joins
    // the regular groups afterwards.
    bool two = false;
    int two_nw = 0;
    if (P.n_big <= (long long)gridDim.x && warp < 2 && (long long)blockIdx.x < P.n_big && P.big_slots >= 2 && !(P.debug & (4 | 128))) {
        two_nw = (int)((P.goff[blockIdx.x + 1] - P.goff[blockIdx.x]) >> 5);
        two = two_nw <= P.big_rows && !(P.grows[blockIdx.x] & 0x10000);
    }
    if (two && warp == 1) {
        double* const xs0 = sxs - (size_t)P.big_rows * 48;                                  // warp 0's staging area
        const unsigned int w0_sa = (unsigned int)__cvta_generic_to_shared(reinterpret_cast<uint32_t*>(xs0 - lane + (size_t)P.big_rows * 32) + lane);
        asm volatile("bar.sync 1, 64;" ::: "memory");                                        // warp 0 has the words in place
        big_bwd<false>(aw, pl, BigSmem{w0_sa, (unsigned int)__cvta_generic_to_shared(sxs)}, two_nw, false, 0.0, 0);
        asm volatile("bar.sync 1, 64;" ::: "memory");                                        // the y stack is complete
    }
    if (big >= P.n_big) {
        while (*reinterpret_cast<volatile int*>(&s_bigleft) > 0) __nanosleep(500);
        if (lane == 0) g = fetch();
        g = __shfl_sync(FULL, g, 0);
    } else g = big;
    while (g < P.n_groups) {
        const unsigned long long tg0 = P.debug ? e6_timer() : 0ull;
        long long gn = 0;
        big += (long long)gridDim.x * (NT / 32);
        if (big >= P.n_big && lane == 0) gn = fetch();
        int rows; long long off;
        if ((P.debug & 64) && g >= P.n_big) { g = big < P.n_big ? big : __shfl_sync(FULL, gn, 0); continue; }   // profiling: big groups only
        if (g < P.n_big) { rows = P.grows[g]; off = P.goff[g]; }
        else {
            int ci = 0;                                        // last class with first <= g
            for (int step = 128; step; step >>= 1) if (ci + step < P.n_cls && s_cls[ci + step].first <= g) ci += step;
            rows = s_cls[ci].code;
            const int nrows = (rows & 0x10000) ? ((rows >> 8) & 0xff) * (rows & 0xff) : rows;
            off = s_cls[ci].off + (g - s_cls[ci].first) * (long long)(nrows * 32);
        }
        if (rows & 0x10000) {                                  // path form: paths << 8 | length
            const int L = rows & 0xff;
            switch ((rows >> 8) & 0xff) {
                case 2: kr_paths<2>(R, aw, pl, L, g, off, lane, acc_g, ll, path_reds); break;
                case 3: kr_paths<3>(R, aw, pl, L, g, off, lane, acc_g, ll, path_reds); break;
                case 4: kr_paths<4>(R, aw, pl, L, g, off, lane, acc_g, ll, path_reds); break;
                case 6: kr_paths<6>(R, aw, pl, L, g, off, lane, acc_g, ll, path_reds); break;
                default: kr_paths<8>(R, aw, pl, L, g, off, lane, acc_g, ll, path_reds); break;
            }
        } else {
            {
                // a big DAG group: from the staging area of this warp when its rows fit, else streamed from HBM
                const int nw = (int)((P.goff[g + 1] - off) >> 5);
                if (g != big0) staged = stage_big(g);
                if (staged) {
                    asm volatile("cp.async.wait_all;" ::: "memory");
                    __syncwarp();
                    if (P.debug && lane == 0) atomicMax(P.stamps + 7, e6_timer() - tg0);
                }
                if (two && warp == 0 && g == big0) {
                    // (stage_big succeeded for this group: two == the same conditions)
                    const unsigned int wp_sa = (unsigned int)__cvta_generic_to_shared(sw);
                    const BigSmem mx{wp_sa, (unsigned int)__cvta_generic_to_shared(sxs)};
                    const BigSmem my{wp_sa, (unsigned int)__cvta_generic_to_shared(sxs + (size_t)P.big_rows * 48)};   // warp 1's x-stack area
                    asm volatile("bar.sync 1, 64;" ::: "memory");
                    double qh, sc0; int EQ; bool any;
                    big_fwd(aw, pl, mx, nw, qh, EQ, any);
                    const bool ok = big_lq(R, R.typeW[g * 32 + lane], g, lane, qh, EQ, any, ll, sc0);
                    asm volatile("bar.sync 1, 64;" ::: "memory");
                    big_red<true>(mx, my, nw, ok, sc0, EQ, acc_g);
                } else if (!(P.debug & 4)) {
                    if (staged) big_one(R, aw, pl, BigSmem{(unsigned int)__cvta_generic_to_shared(sw), (unsigned int)__cvta_generic_to_shared(sxs)}, nw, g, lane, acc_g, ll, true);
                    else big_one(R, aw, pl, BigGmem{P.words + off + lane, xs}, nw, g, lane, acc_g, ll, true);
                }
                __syncwarp();
            }
        }
        if (P.debug) { const unsigned long long d = ((e6_timer() - tg0) << 32) | (unsigned int)rows; dbg_max = d > dbg_max ? d : dbg_max; }
        if (g < P.n_big && big >= P.n_big && lane == 0) atomicSub(&s_bigleft, 1);      // this warp's last big group is done
        g = big < P.n_big ? big : __shfl_sync(FULL, gn, 0);
    }
    if (P.debug && lane == 0) { atomicMax(P.stamps + 4, dbg_max); atomicMax(P.stamps + 5, e6_timer() - P.stamps[6]); }
    // the static index loads of the fold (they do not depend on the accumulators) go out before the barrier:
    // half-warp h of global warp gw takes edge 2*gw + h (then + 2*TW ...)
    const int TW = (int)gridDim.x * (NT / 32);
    const int gw = (int)gwarp;
    const int hl = lane & 15;
    const unsigned hmask = (lane & 16) ? 0xffff0000u : 0x0000ffffu;
    const int e_first = 2 * gw + (lane >> 4);
    int k0a = 0, naa = 0, fa = 0, tpa = -1;
    if (e_first < P.n_edges) {
        k0a = P.e_off[e_first]; naa = P.e_off[e_first + 1] - k0a; tpa = P.edge_tp[e_first];
        if (hl < min(16, naa)) fa = P.e_arc[k0a + hl];
    }
    // the CTA's share of the log-likelihood: integer sums (exact, order independent), one RED per CTA
#pragma unroll
    for (int o = 16; o; o >>= 1) { ll += __shfl_xor_sync(FULL, ll, o); nf += __shfl_xor_sync(FULL, nf, o); }
    if (lane == 0) { s_part[warp][0] = ll; s_part[warp][1] = (long long)nf; }
    __syncthreads();
    if (prof) t2 = e6_timer();
    if (tline) tl2 = e6_timer();
    // ---- P2: grid barrier -------------------------------------------------------------------------------------
    if (tid == 0) {
        long long s = 0, f = 0;
        for (int w = 0; w < NT / 32; ++w) { s += s_part[w][0]; f += s_part[w][1]; }
        if (s) red_add64(P.red, (unsigned long long)s);
        if (f) red_add64(P.red + 1, (unsigned long long)f);
        __threadfence();
        atomicAdd(P.ctl + 2, 1u);
        const unsigned int target = epoch * gridDim.x;
        while ((int)(e6_ld_acquire(P.ctl + 2) - target) < 0) { }
        __threadfence();
    }
    __syncthreads();
    if (prof) t3 = e6_timer();
    if (tline) tl3 = e6_timer();
    // ---- P3: fold, exchange, conversion ---------------------------------------------------------------------------
    if (blockIdx.x == 0 && tid == 0) P.ctl[3] = epoch + 1u;    // every CTA has read the epoch (it passed the barrier)
    const unsigned long long* const acc_all = P.acc + (size_t)par * acc_words;
    bool timeout = false;
    for (int e = e_first; e < P.n_edges; e += 2 * TW) {
        int k0 = k0a, na = naa, first = fa, tp = tpa;
        if (e != e_first) {
            k0 = P.e_off[e]; na = P.e_off[e + 1] - k0; tp = P.edge_tp[e];
            first = hl < min(16, na) ? P.e_arc[k0 + hl] : 0;
        }
        unsigned long long s = e6_fold_edge(acc_all, P.n_arcs, P.replicas, P.e_arc, k0, na, first, hl, hmask);
        if (P.nranks > 1) s = e6_exchange(P, epoch, 2 + e, s, hl, hmask, timeout);
        if (hl == 0 && tp >= 0 && tp < P.n) P.out[2 + tp] = -(double)(long long)s * P.inv_fx;
    }
    __syncwarp();
    if (gw == TW - 1 && lane < 16) {                           // [loglik, non-finite terms]: a half-warp of the last warp of the grid
        unsigned long long sl = 0, bad = 0;
        if (lane == 0) { sl = __ldcg(P.red); bad = __ldcg(P.red + 1); P.red[0] = 0ull; P.red[1] = 0ull; }
        sl = __shfl_sync(0xffffu, sl, 0); bad = __shfl_sync(0xffffu, bad, 0);
        if (P.nranks > 1) {
            sl = e6_exchange(P, epoch, 0, sl, lane, 0xffffu, timeout); bad = e6_exchange(P, epoch, 1, bad, lane, 0xffffu, timeout);
        }
        if (lane == 0) {
            P.out[0] = bad > 0 ? -INFINITY : (double)(long long)sl * inv_ll;
            P.out[1] = (double)bad;
        }
    }
    __syncwarp();
    {   // re-arm the accumulators and the ticket counter of the NEXT evaluation (nobody reads them during this one);
        // at the end of the kernel, where the stores overlap the exchange instead of delaying the region phase
        unsigned long long* other = P.acc + (size_t)(par ^ 1) * acc_words;
        for (size_t i = (size_t)blockIdx.x * NT + tid; i < acc_words; i += (size_t)gridDim.x * NT)
            other[i] = i < (size_t)P.n_arcs ? P.const_acc[i] : 0ull;
        if (blockIdx.x == 0 && tid == 0) P.ctl[par ^ 1] = 0u;
    }
    if (__any_sync(FULL, timeout) && lane == 0) P.out[2 + P.n] = (double)epoch;
    if (P.done_flag) {                                         // `out` is host memory here: tell the host when every CTA is through
        __syncthreads();
        if (tid == 0) {
            __threadfence_system();
            // ctl[4] counts the CTAs of THIS host-buffer launch that are through (launches are stream ordered); the last one
            // re-arms it and writes the number of host-buffer launches so far (ctl[6], wraps like the host's counter)
            const unsigned int arrived = atomicAdd(P.ctl + 4, 1u) + 1u;
            if (arrived == gridDim.x) {
                P.ctl[4] = 0u;
                const unsigned int done = P.ctl[6] + 1u;
                P.ctl[6] = done;
                *reinterpret_cast<volatile unsigned int*>(P.done_flag) = done;
                __threadfence_system();
            }
        }
    }
    if (prof) {
        const unsigned long long t4 = e6_timer();
        P.stamps[0] += t1 - t0; P.stamps[1] += t2 - t1; P.stamps[2] += t3 - t2; P.stamps[3] += t4 - t3;
    }
    if (P.stamps && (P.debug & 16) && tid == 0) {              // timeline of the last launch: [start, weights, regions, barrier, end] of every CTA
        unsigned long long* tl = P.stamps + 8 + (size_t)blockIdx.x * 8;
        tl[0] = tl0; tl[1] = tl1; tl[2] = tl2; tl[3] = tl3; tl[4] = e6_timer();
    }
}

}  // namespace wfsa
