// w-fsa_b200/csrc/kernels_viterbi.cuh -- the most probable accepting path of every string (Viterbi decoding):
//   mu_t[j] = max_k (log a(src_k, j) + mu_{t-1}[src_k]) + log b(j, c_t),   logw_s = max_u (mu_T[u] + log a(u, end))
// one forward sweep in the (max, +) semiring with a backpointer per lattice node, then a traceback.  Summation order: every
// node adds (log a + mu_{t-1}) first, then log b; the end adds log a(u, end) last.  logw_s is therefore the left-to-right sum
// of the log weights of the returned steps, bit for bit.  The sweeps work in the log domain without rescaling; an absent
// entry (trimmed edge, padding, unreachable candidate) is -inf.  Ties: the first strictly larger fent entry (or generic
// transition / emission in table order) wins at a node, and the lowest candidate slot wins at the end.
//   k3_viterbi<WARP>          every handle with fast tables: a warp per string (max_cand <= 32) or a CTA per string
//   kg_fwdbwd<MODE_VITERBI>   (kernels.cuh) automata without fast tables
// (Included last, after kernels_rmin.cuh, for the reason given there.)
#pragma once
#include "kernels.cuh"

namespace wfsa {

// (max, +) weights: log weights with -inf for an absent edge, per transition, emission and -- with fast tables -- per
// candidate slot (its emission, its transition to the end state); logw of every string starts at -inf (no path)
__global__ void k_maxplus_weights(int n_trans, int n_emis, int n_slots, long long n_strings, const int32_t* __restrict__ trans_tp,
                                  const int32_t* __restrict__ emis_tp, const int32_t* __restrict__ slot_emis,
                                  const int32_t* __restrict__ slot_final, const double* __restrict__ x,
                                  double* vtw, double* vew, double* vsw, double* vfw, double* logw)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nw = (long long)n_trans + n_emis + n_slots;
    if (i < n_trans) vtw[i] = logweight_of(trans_tp[i], x, 0);
    else if (i < n_trans + n_emis) vew[i - n_trans] = logweight_of(emis_tp[i - n_trans], x, 0);
    else if (i < nw) {
        const int s = (int)(i - n_trans - n_emis);
        vsw[s] = slot_emis[s] < 0 ? 0.0 : logweight_of(emis_tp[slot_emis[s]], x, 0);
        vfw[s] = slot_final[s] < 0 ? -INFINITY : logweight_of(trans_tp[slot_final[s]], x, 0);
    } else if (i < nw + n_strings) logw[i - nw] = -INFINITY;
}

// ------------------------------------------------------------------------------------------
// Fast tables: a group of threads per string, thread g <-> candidate slot g of the current symbol.  WARP: the group is a
// warp (max_cand <= 32, several strings per CTA, warp-synchronous); else the group is the CTA (one string at a time).
// Thread g keeps the index k of the winning fent entry of its candidate and writes it to the group's backpointer slab
// bp[t * pitch + g] (uint16, reused string by string).  After the forward pass thread 0 of the group walks back: it reads
// frow / fent again for the transition and the source slot, slot_emis gives the emission, slot_final the last transition.
// With fast tables a path has len + 1 steps: string s is written at offs[s] + s.
// ------------------------------------------------------------------------------------------
struct K3VitParams {
    FastTablesD T;
    const double* __restrict__ vtw;          // [n_trans] log weights, -inf where absent (k_maxplus_weights)
    const double* __restrict__ vsw;          // [n_slots] log emission weight of the slot
    const double* __restrict__ vfw;          // [n_slots] log weight of slot-state -> end, -inf where absent
    const int32_t* __restrict__ slot_emis;   // [n_slots] emission edge of the slot
    const int32_t* __restrict__ slot_final;  // [n_slots] transition edge slot-state -> end, or -1
    CorpusD C;
    uint16_t* bp;                            // [groups][max_len][pitch] backpointer slabs
    int pitch;                               // candidates per slab row: 32 (WARP) or blockDim.x
    int max_len;
    double* logw;                            // [n_strings]
    int32_t* trans_edge;                     // [n_tokens + n_strings]
    int32_t* emis_edge;
};

template <bool WARP>
__device__ __forceinline__ void vit_sync() { if (WARP) __syncwarp(); else __syncthreads(); }

template <bool WARP>
__global__ void __launch_bounds__(WARP ? 256 : 1024, 1) k3_viterbi(const K3VitParams P)
{
    extern __shared__ unsigned long long smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int g = WARP ? lane : tid;                                          // candidate of this thread
    const int G = WARP ? 32 : (int)blockDim.x;
    double* vm = reinterpret_cast<double*>(smem) + (WARP ? warp * 64 : 0);    // [2][G] mu of the group
    double* red = reinterpret_cast<double*>(smem) + 2 * blockDim.x;           // [32] (CTA) maxima of the warps
    int* ired = reinterpret_cast<int*>(red + 32);                             // [32] their slots
    const FastTablesD& T = P.T;
    const int A = T.n_sym;
    const long long grp = WARP ? (long long)blockIdx.x * nwarps + warp : blockIdx.x;
    const long long n_grp = WARP ? (long long)gridDim.x * nwarps : gridDim.x;
    uint16_t* bp = P.bp + (size_t)grp * P.max_len * P.pitch;

    for (long long it = grp; it < P.C.n_order; it += n_grp) {
        const int sid = P.C.order[it];
        const long long off = P.C.offs[sid];
        const int len = (int)(P.C.offs[sid + 1] - off);
        const int32_t* tok = P.C.tokens + off;
        const long long out = off + sid;
        vit_sync<WARP>();                                   // the previous traceback has read the slab
        if (len == 0) {                                     // one path: start -> end
            if (g == 0 && T.start_final_tid >= 0) {
                const double w = 0.0 + P.vtw[T.start_final_tid];
                if (w > -INFINITY) { P.logw[sid] = w; P.trans_edge[out] = T.start_final_tid; P.emis_edge[out] = -1; }
            }
            continue;
        }
        int cur = 0, cprev = A;
        bool dead = false, valid = false;
        vm[g] = (g == 0) ? 0.0 : -INFINITY;
        vit_sync<WARP>();
        uint32_t slot = 0;
        double mu = -INFINITY;
        for (int t = 0; t < len; ++t) {
            const int c = tok[t];
            if ((unsigned)c >= (unsigned)A) { dead = true; break; }          // (uniform over the group)
            const uint32_t c0 = T.cand_off[c], ncand = T.cand_off[c + 1] - c0;
            valid = (uint32_t)g < ncand;
            slot = c0 + g;
            mu = -INFINITY;
            if (valid) {
                const uint32_t row = T.frow[(size_t)T.slot_state[slot] * (A + 1) + cprev];
                const int cnt = row & ((1u << kRowCntBitsD) - 1);
                const uint32_t st = row >> kRowCntBitsD;
                const double* msrc = vm + cur * G;
                double m = -INFINITY;
                int kb = 0;
                for (int k = 0; k < cnt; ++k) {
                    const uint32_t ent = T.fent[st + k];
                    const double v = P.vtw[ent >> kSlotBitsD] + msrc[ent & ((1u << kSlotBitsD) - 1)];
                    if (v > m) { m = v; kb = k; }
                }
                mu = m + P.vsw[slot];
                bp[(size_t)t * P.pitch + g] = (uint16_t)kb;
            }
            vm[(cur ^ 1) * G + g] = mu;
            cur ^= 1;
            cprev = c;
            vit_sync<WARP>();
        }
        if (dead) continue;
        // the end: the largest mu_T[u] + log a(u, end), the lowest slot among equal values
        double best = (valid && mu > -INFINITY) ? mu + P.vfw[slot] : -INFINITY;
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
        }
        if (g != 0 || !(best > -INFINITY)) continue;
        P.logw[sid] = best;
        int j = bj;
        uint32_t c0 = T.cand_off[tok[len - 1]];
        P.trans_edge[out + len] = P.slot_final[c0 + j];
        P.emis_edge[out + len] = -1;
        for (int t = len - 1; t >= 0; --t) {
            const uint32_t sl = c0 + j;
            const int cp = t ? tok[t - 1] : A;
            const uint32_t row = T.frow[(size_t)T.slot_state[sl] * (A + 1) + cp];
            const uint32_t ent = T.fent[(row >> kRowCntBitsD) + bp[(size_t)t * P.pitch + j]];
            P.trans_edge[out + t] = (int32_t)(ent >> kSlotBitsD);
            P.emis_edge[out + t] = P.slot_emis[sl];
            j = (int)(ent & ((1u << kSlotBitsD) - 1));
            c0 = T.cand_off[cp];
        }
    }
}

}  // namespace wfsa
