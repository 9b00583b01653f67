// w-fsa_b200/csrc/kernels_nbest.cuh -- the k most probable accepting paths of every string (N-best decoding, k <= 16):
// the Viterbi recursion of kernels_viterbi.cuh with a sorted list of the k largest values per lattice node instead of one
// value.  A node's list is the k largest of its candidates (log a + mu_{t-1}[src][r]) over every incoming entry and every
// rank r of the source's list, then log b is added to each; the end takes the k largest (mu_T[u][r] + log a(u, end)).  The
// summation order is Viterbi's, so every value is the left-to-right sum of its path's steps, bit for bit, and rank 0 is the
// Viterbi path.  Ties: the first strictly larger candidate wins, in the order (fent entry, source rank) with fast tables and
// (source state in eps_order, transition, emission, source rank) in the generic kernel; at the end (candidate slot, rank),
// respectively (source state, transition, rank).  A source list is sorted, so its ranks stop at the first candidate that is
// not larger than the current k-th.  k = 1 is served by the Viterbi kernels themselves.
//   k3_nbest<WARP, K>   every handle with fast tables: a warp per string (max_cand <= 32) or a CTA per string; runtime k <= K
//   kg_nbest            automata without fast tables, thread per string
// (Included last, after kernels_viterbi.cuh, for the reason given in kernels_rmin.cuh.)
#pragma once
#include "kernels_viterbi.cuh"

namespace wfsa {

constexpr int kNbestMax = 16;              // largest k; a backpointer keeps the source rank in 4 bits
// most threads (candidates) of the CTA form: at K = 16 the 16 values and backpointers of a list spill at 64 or 72 registers
// a thread (1024 or 896 threads); 768 threads leave 80
constexpr int nbest_cta_threads(int K) { return K >= 16 ? 768 : 1024; }

// ------------------------------------------------------------------------------------------
// Fast tables: as k3_viterbi, thread g <-> candidate slot g of the current symbol.  Thread g builds the sorted list of its
// candidate in registers and stores it to the group's shared lists [2][K][G] (rank-major, so that the stores are
// conflict-free); its backpointers (fent entry << 4 | source rank) go to the group's slab bp[(t * k + r) * pitch + g].  The
// end is k rounds of a group-wide argmax over the heads of the lists (lowest slot among equal values), and threads
// 0..k'-1 then trace back the k' paths found in parallel.  Rank r of string s is written at k * (offs[s] + s) + r * (len + 1).
// ------------------------------------------------------------------------------------------
struct K3NbestParams {
    FastTablesD T;
    const double* __restrict__ vtw;          // [n_trans] log weights, -inf where absent (k_maxplus_weights)
    const double* __restrict__ vsw;          // [n_slots] log emission weight of the slot
    const double* __restrict__ vfw;          // [n_slots] log weight of slot-state -> end, -inf where absent
    const int32_t* __restrict__ slot_emis;   // [n_slots] emission edge of the slot
    const int32_t* __restrict__ slot_final;  // [n_slots] transition edge slot-state -> end, or -1
    CorpusD C;
    uint16_t* bp;                            // [groups][max_len][k][pitch] backpointer slabs
    int pitch;                               // candidates per slab row: 32 (WARP) or blockDim.x
    int max_len;
    int k;                                   // 2..K
    double* logw;                            // [n_strings * k]
    int32_t* trans_edge;                     // [k * (n_tokens + n_strings)]
    int32_t* emis_edge;
};

// x into the sorted list v[0..k) after every entry >= x (the first strictly larger candidate wins); x > v[k-1] on entry
template <int K>
__device__ __forceinline__ void nb_insert(double (&v)[K], uint32_t (&b)[K], int k, double x, uint32_t bx)
{
#pragma unroll
    for (int j = K - 1; j > 0; --j) {
        if (j < k) {
            const bool shift = x > v[j - 1], here = !shift && x > v[j];
            v[j] = shift ? v[j - 1] : (here ? x : v[j]);
            b[j] = shift ? b[j - 1] : (here ? bx : b[j]);
        }
    }
    if (x > v[0]) { v[0] = x; b[0] = bx; }
}

template <int K>
__device__ __forceinline__ double nb_at(const double (&v)[K], int i)
{
    double r = -INFINITY;
#pragma unroll
    for (int j = 0; j < K; ++j) if (j == i) r = v[j];
    return r;
}

template <bool WARP, int K>
__global__ void __launch_bounds__(WARP ? 256 : nbest_cta_threads(K), 1) k3_nbest(const K3NbestParams P)
{
    extern __shared__ unsigned long long smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int g = WARP ? lane : tid;                                          // candidate of this thread
    const int G = WARP ? 32 : (int)blockDim.x;
    const int k = P.k;
    double* vm = reinterpret_cast<double*>(smem) + (WARP ? warp * 2 * K * 32 : 0);   // [2][K][G] lists of the group
    double* red = reinterpret_cast<double*>(smem) + 2 * K * blockDim.x;             // [32] (CTA) heads of the warps
    int* ired = reinterpret_cast<int*>(red + 32);                                   // [32] their slots
    int* sel = ired + 32 + (WARP ? warp * kNbestMax : 0);                           // [16] (slot << 4 | rank) of each path
    const FastTablesD& T = P.T;
    const int A = T.n_sym;
    const long long grp = WARP ? (long long)blockIdx.x * nwarps + warp : blockIdx.x;
    const long long n_grp = WARP ? (long long)gridDim.x * nwarps : gridDim.x;
    uint16_t* bp = P.bp + (size_t)grp * P.max_len * k * P.pitch;

    for (long long it = grp; it < P.C.n_order; it += n_grp) {
        const int sid = P.C.order[it];
        const long long off = P.C.offs[sid];
        const int len = (int)(P.C.offs[sid + 1] - off);
        const int32_t* tok = P.C.tokens + off;
        const long long out = (long long)k * (off + sid);
        vit_sync<WARP>();                                   // the previous traceback has read the slab and sel
        if (len == 0) {                                     // one path: start -> end
            if (g == 0 && T.start_final_tid >= 0) {
                const double w = 0.0 + P.vtw[T.start_final_tid];
                if (w > -INFINITY) { P.logw[(long long)sid * k] = w; P.trans_edge[out] = T.start_final_tid; P.emis_edge[out] = -1; }
            }
            continue;
        }
        int cur = 0, cprev = A;
        bool dead = false, valid = false;
        for (int r = 0; r < k; ++r) vm[r * G + g] = (g == 0 && r == 0) ? 0.0 : -INFINITY;
        vit_sync<WARP>();
        uint32_t slot = 0;
        double v[K];
        uint32_t b[K];
        for (int t = 0; t < len; ++t) {
            const int c = tok[t];
            if ((unsigned)c >= (unsigned)A) { dead = true; break; }          // (uniform over the group)
            const uint32_t c0 = T.cand_off[c], ncand = T.cand_off[c + 1] - c0;
            valid = (uint32_t)g < ncand;
            slot = c0 + g;
#pragma unroll
            for (int j = 0; j < K; ++j) { v[j] = -INFINITY; b[j] = 0; }
            if (valid) {
                const uint32_t row = T.frow[(size_t)T.slot_state[slot] * (A + 1) + cprev];
                const int cnt = row & ((1u << kRowCntBitsD) - 1);
                const uint32_t st = row >> kRowCntBitsD;
                const double* msrc = vm + cur * K * G;
                double kth = -INFINITY;
                for (int e = 0; e < cnt; ++e) {
                    const uint32_t ent = T.fent[st + e];
                    const double a = P.vtw[ent >> kSlotBitsD];
                    const double* ms = msrc + (ent & ((1u << kSlotBitsD) - 1));
                    for (int r = 0; r < k; ++r) {
                        const double x = a + ms[r * G];
                        if (!(x > kth)) break;                               // the source list is sorted
                        nb_insert<K>(v, b, k, x, (uint32_t)(e << 4 | r));
                        kth = nb_at<K>(v, k - 1);
                    }
                }
                const double w = P.vsw[slot];
                uint16_t* bt = bp + (size_t)t * k * P.pitch + g;
#pragma unroll
                for (int j = 0; j < K; ++j)
                    if (j < k) { v[j] = v[j] + w; bt[(size_t)j * P.pitch] = (uint16_t)b[j]; }
            }
            double* mdst = vm + (cur ^ 1) * K * G + g;
#pragma unroll
            for (int j = 0; j < K; ++j) if (j < k) mdst[j * G] = v[j];
            cur ^= 1;
            cprev = c;
            vit_sync<WARP>();
        }
        if (dead) continue;
        // the end: k rounds of the largest head (mu_T[u][h] + log a(u, end)), the lowest slot among equal values
        const double fw = valid ? P.vfw[slot] : -INFINITY;
        int h = 0, found = 0;
        for (; found < k; ++found) {
            double best = (valid && h < k) ? nb_at<K>(v, h) + fw : -INFINITY;
            int bj = g;
#pragma unroll
            for (int o = 16; o; o >>= 1) {
                const double ov = __shfl_xor_sync(FULL, best, o);
                const int oj = __shfl_xor_sync(FULL, bj, o);
                if (ov > best || (ov == best && oj < bj)) { best = ov; bj = oj; }
            }
            if (!WARP) {
                if (lane == 0) { red[warp] = best; ired[warp] = bj; }
                __syncthreads();
                best = red[0]; bj = ired[0];
                for (int w = 1; w < nwarps; ++w) if (red[w] > best) { best = red[w]; bj = ired[w]; }
                __syncthreads();                            // red is read before the next round writes it
            }
            if (!(best > -INFINITY)) break;                 // (uniform over the group)
            if (g == bj) { sel[found] = g << 4 | h; P.logw[(long long)sid * k + found] = best; ++h; }
        }
        vit_sync<WARP>();
        if (g >= found) continue;
        int j = sel[g] >> 4, r = sel[g] & 15;
        const long long o = out + (long long)g * (len + 1);
        uint32_t c0 = T.cand_off[tok[len - 1]];
        P.trans_edge[o + len] = P.slot_final[c0 + j];
        P.emis_edge[o + len] = -1;
        for (int t = len - 1; t >= 0; --t) {
            const uint32_t sl = c0 + j;
            const int cp = t ? tok[t - 1] : A;
            const uint32_t row = T.frow[(size_t)T.slot_state[sl] * (A + 1) + cp];
            const uint32_t pb = bp[((size_t)t * k + r) * P.pitch + j];
            const uint32_t ent = T.fent[(row >> kRowCntBitsD) + (pb >> 4)];
            P.trans_edge[o + t] = (int32_t)(ent >> kSlotBitsD);
            P.emis_edge[o + t] = P.slot_emis[sl];
            j = (int)(ent & ((1u << kSlotBitsD) - 1));
            r = (int)(pb & 15);
            c0 = T.cand_off[cp];
        }
    }
}

// ------------------------------------------------------------------------------------------
// No fast tables: the generic kernel's push loop in (max, +) with a list of k values and k packed backpointers
// (transition << 36 | emission << 4 | source rank) per lattice node, in the thread's scratch [2][(max_len+1) * S][k].  The
// end's list lives in the node (len, end state), which nothing else writes.  As kg_fwdbwd<MODE_VITERBI>: a first launch
// (vit_off == nullptr) writes the step count of every path to vit_cnt[s * k + r], a second one writes the steps from
// vit_off[s * k + r].  logw of string s, rank r goes to O.logq[s * k + r].
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void nbg_insert(double* v, unsigned long long* b, int k, double x, unsigned long long bx)
{
    int j = k - 1;                                  // x > v[k-1]: it goes after every entry >= x
    while (j > 0 && x > v[j - 1]) { v[j] = v[j - 1]; b[j] = b[j - 1]; --j; }
    v[j] = x; b[j] = bx;
}

__global__ void __launch_bounds__(128) kg_nbest(const GenericParams P, int k)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.count) return;
    const GenericTablesD& G = P.G;
    const int S = G.n_states;
    const int sid = P.C.order[P.first + i];
    const long long off = P.C.offs[sid];
    const int len = (int)(P.C.offs[sid + 1] - off);
    const int32_t* tok = P.C.tokens + off;
    const size_t lat_sz = (size_t)(P.max_len + 1) * S * k;
    double* lv = P.scratch + (size_t)i * 2 * lat_sz;
    unsigned long long* lb = reinterpret_cast<unsigned long long*>(lv + lat_sz);
    for (size_t q = 0; q < (size_t)(len + 1) * S * k; ++q) lv[q] = -INFINITY;
    lv[(size_t)G.start_state * k] = 0.0;
    double* fv = lv + ((size_t)len * S + G.end_state) * k;                // the end's list
    unsigned long long* fb = lb + ((size_t)len * S + G.end_state) * k;
    for (int pos = 0; pos <= len; ++pos) {
        for (int oi = 0; oi < S; ++oi) {
            const int u = G.eps_order[oi];
            const double* mu = lv + ((size_t)pos * S + u) * k;
            if (mu[0] == -INFINITY || u == G.end_state) continue;
            for (int t = G.trans_row[u]; t < G.trans_row[u + 1]; ++t) {
                const int v = G.trans_dst[t];
                const double a = P.ltw[t];
                if (a == -INFINITY) continue;
                if (v == G.end_state) {
                    if (pos == len)
                        for (int r = 0; r < k; ++r) {
                            const double x = mu[r] + a;
                            if (!(x > fv[k - 1])) break;
                            nbg_insert(fv, fb, k, x, (unsigned long long)t << 36 | (unsigned)r);
                        }
                    continue;
                }
                for (int e = G.emis_row[v]; e < G.emis_row[v + 1]; ++e) {
                    const int e0 = G.emis_tok_off[e], el = G.emis_tok_off[e + 1] - e0;
                    if (pos + el > len) continue;
                    bool m = true;
                    for (int q = 0; q < el; ++q) if (tok[pos + q] != G.emis_tok[e0 + q]) { m = false; break; }
                    if (!m) continue;
                    const double lw = P.lew[e];
                    double* dv = lv + ((size_t)(pos + el) * S + v) * k;
                    unsigned long long* db = lb + ((size_t)(pos + el) * S + v) * k;
                    for (int r = 0; r < k; ++r) {
                        const double x = (mu[r] + a) + lw;
                        if (!(x > dv[k - 1])) break;
                        nbg_insert(dv, db, k, x, (unsigned long long)t << 36 | (unsigned long long)(unsigned)e << 4 | (unsigned)r);
                    }
                }
            }
        }
    }
    for (int r = 0; r < k; ++r) {
        const long long q = (long long)sid * k + r;
        P.O.logq[q] = fv[r];
        if (!(fv[r] > -INFINITY)) { if (!P.vit_off) P.vit_cnt[q] = 0; continue; }
        int t = (int)(fb[r] >> 36), rr = (int)(fb[r] & 15);
        int64_t o = P.vit_off ? P.vit_off[q + 1] - 1 : 0;
        if (P.vit_off) { P.vit_trans[o] = t; P.vit_emis[o] = -1; }
        int n = 1, p = len;
        for (;;) {
            int lo = 0, hi = S;                      // source state of t: the last state whose transitions start at or before t
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (G.trans_row[mid] <= t) lo = mid; else hi = mid; }
            if (lo == G.start_state) break;
            const unsigned long long bb = lb[((size_t)p * S + lo) * k + rr];
            t = (int)(bb >> 36);
            const int e = (int)(unsigned)(bb >> 4);
            rr = (int)(bb & 15);
            if (P.vit_off) { --o; P.vit_trans[o] = t; P.vit_emis[o] = e; }
            p -= G.emis_tok_off[e + 1] - G.emis_tok_off[e];
            ++n;
        }
        if (!P.vit_off) P.vit_cnt[q] = n;
    }
}

}  // namespace wfsa
