// w-fsa_b200/csrc/wfsa_dev.cu -- C ABI of the B200 evaluation backend (include/wfsa_dev.h).
//
// Host side of the device path: copies the lowered automaton and the packed corpus shard to
// HBM once, then every evaluation is   H2D x  ->  k_weights -> forward-backward kernel
// (K2 warp-per-string | K3 CTA-per-string | generic) -> arc->edge fold -> [ncclAllReduce]
// -> k_finish_eval -> D2H [loglik, grad].   There is no CPU fallback: every entry point fails
// with WFSA_ERR_NO_DEVICE / WFSA_ERR_CUDA when the GPU path cannot run.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <map>
#include <memory>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/wfsa_dev.h"
#include "kernels.cuh"
#include "kernels_seg.cuh"
#include "kernels_eval6.cuh"
#include "kernels_k7.cuh"
#include "kernels_rmin.cuh"
#include "kernels_viterbi.cuh"
#include "kernels_nbest.cuh"
#include "kernels_sample.cuh"
#include "layout.hpp"
#include "lattice.hpp"

using namespace wfsa;

static thread_local std::string g_create_error;

// ---- minimal NCCL binding, resolved at run time (libnccl.so.2 is only needed for n_ranks > 1)
namespace {
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
enum { ncclSuccess = 0 };
enum { ncclInt64 = 4, ncclUint64 = 5, ncclInt32 = 2 };
enum { ncclSum = 0, ncclMax = 2 };
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(ncclUniqueId*) = nullptr;
    int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool load(std::string& err)
    {
        if (lib) return true;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) { lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (lib) break; }
        if (!lib) { err = std::string("cannot load libnccl.so.2: ") + dlerror(); return false; }
        GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
        AllReduce = (decltype(AllReduce))dlsym(lib, "ncclAllReduce");
        CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
        GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
        if (!GetUniqueId || !CommInitRank || !AllReduce || !CommDestroy) { err = "libnccl lacks required symbols"; return false; }
        return true;
    }
};
NcclApi g_nccl;
std::atomic<int64_t> g_held_bytes{0};         // wfsa_dev_held_bytes

// Owns one allocation of n elements: device memory, or with Pinned page-locked host memory (cudaHostAlloc `flags`).
template <class T, bool Pinned> struct Buf {
    T* p = nullptr; size_t n = 0;
    Buf() = default;
    Buf(const Buf&) = delete; Buf& operator=(const Buf&) = delete;
    Buf(Buf&& o) noexcept : p(std::exchange(o.p, nullptr)), n(std::exchange(o.n, 0)) {}
    Buf& operator=(Buf&& o) noexcept { if (this != &o) { release(); p = std::exchange(o.p, nullptr); n = std::exchange(o.n, 0); } return *this; }
    ~Buf() { release(); }
    cudaError_t alloc(size_t count, unsigned flags = 0)
    {
        release();
        void* q = nullptr;
        const cudaError_t e = !count ? cudaSuccess : Pinned ? cudaHostAlloc(&q, count * sizeof(T), flags) : cudaMalloc(&q, count * sizeof(T));
        if (e == cudaSuccess && count) { p = static_cast<T*>(q); n = count; g_held_bytes += (int64_t)(n * sizeof(T)); }
        return e;
    }
    cudaError_t upload(const std::vector<T>& v, cudaStream_t s)
    {
        cudaError_t e = alloc(v.size());
        if (e != cudaSuccess || v.empty()) return e;
        return cudaMemcpyAsync(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, s);
    }
    void release() { if (p) { if (Pinned) cudaFreeHost(p); else cudaFree(p); g_held_bytes -= (int64_t)(n * sizeof(T)); } p = nullptr; n = 0; }
};
template <class T> using DevBuf = Buf<T, false>;
template <class T> using PinnedBuf = Buf<T, true>;

// Owns a stream, event, graph or graph exec; converts to the raw handle.
template <class H, cudaError_t (*Destroy)(H)> struct Handle {
    H raw = nullptr;
    Handle() = default;
    Handle(const Handle&) = delete; Handle& operator=(const Handle&) = delete;
    Handle(Handle&& o) noexcept : raw(std::exchange(o.raw, nullptr)) {}
    ~Handle() { reset(); }
    void reset(H v = nullptr) { if (raw) Destroy(raw); raw = v; }
    operator H() const { return raw; }
};
using Stream = Handle<cudaStream_t, cudaStreamDestroy>;
using Event = Handle<cudaEvent_t, cudaEventDestroy>;
using Graph = Handle<cudaGraph_t, cudaGraphDestroy>;
using GraphExec = Handle<cudaGraphExec_t, cudaGraphExecDestroy>;

// Events of the timers: one slot per timed evaluation, reused from every timer_begin on, at most 8192 per window.
struct TimedSlot { Event begin, end, mid; };
struct EventPool {
    std::vector<TimedSlot> slots; size_t used = 0;
    // the next slot (with `mid` also the event between the two stages of the general pipeline); nullptr when full
    TimedSlot* next(bool mid)
    {
        if (used == slots.size() && used < 8192) { slots.emplace_back(); cudaEventCreate(&slots.back().begin.raw); cudaEventCreate(&slots.back().end.raw); }
        if (used == slots.size()) return nullptr;
        TimedSlot& s = slots[used++];
        if (mid && !s.mid) cudaEventCreate(&s.mid.raw);
        return &s;
    }
};
}  // namespace

struct wfsa_dev {
    Stream stream;                             // first, so that it is destroyed after everything that uses it
    std::string err;
    int device = 0, sm_count = 0, kernel = 0, accum = 0;
    wfsa_dev_options opt{};
    HostFsa fsa;
    FastLayout fast;
    GenericLayout gen;
    // corpus shard
    int64_t n_strings = 0, n_tokens = 0, n_active = 0, n_active_tokens = 0;
    int max_len = 0;
    std::vector<int64_t> h_offs;
    std::vector<int32_t> h_order_all;          // all strings, longest first
    DevBuf<int32_t> d_tokens, d_order;
    DevBuf<int64_t> d_offs;
    DevBuf<double> d_p;
    // automaton tables
    DevBuf<uint32_t> d_cand_off, d_slot_state, d_frow, d_fent, d_brow, d_bent;
    DevBuf<int32_t> d_slot_emis, d_slot_final, d_arc_tid, d_arc_eid;
    DevBuf<uint16_t> d_brow16, d_sstate16;
    DevBuf<uint8_t> d_bent8;
    DevBuf<double> d_aw;
    int tab_smem = 0, replicas = 1;
    long long step_bound = 1;
    DevBuf<int32_t> d_emis_row, d_emis_tok_off, d_emis_tok, d_trans_row, d_trans_dst, d_eps_order;
    DevBuf<int32_t> d_trans_tp, d_emis_tp, d_edge_tp, d_edge_raw;
    // per evaluation
    int n = -1;                                // trimmed parameters (-1: map not set)
    int n_edges = 0;
    DevBuf<double> d_x, d_tw, d_sw, d_fw, d_ltw, d_lew, d_logq, d_pathcnt, d_out;
    DevBuf<unsigned long long> d_acc, d_red, d_glstack;
    DevBuf<uint8_t> d_used;
    DevBuf<double> d_k3lat; DevBuf<int> d_k3exp;
    DevBuf<double> d_gscratch;
    long long g_batch = 0;
    PinnedBuf<double> h_out;                   // [2 + n]
    PinnedBuf<double> h_x;                     // mapped [n + 1]
    double* h_x_dev = nullptr;                 // device address of h_x (the host-buffer call lets the kernel fetch x itself)
    double fx_log2 = 0, ll_log2 = 44;
    int grid = 0, block = 0, stack_cap = 0, n_acc_smem = 0;      // warp-per-string (K2) launch
    size_t smem_bytes = 0, glstack_words = 0, table_bytes = 0;
    int k3_grid = 0, k3_block = 0; size_t k3_smem = 0;
            // CTA-per-string (K3) launch
    int kt_grid = 0, kt_block = 0, kt_K = 0; size_t kt_smem = 0, kt_lat_words = 0;   // thread-per-string (KT)
    int secondary = 0;                                            // kernel that takes KT's / the segmented path's overflow strings
    int skernel = 0;                                              // kernel of the structural pass
    // segmented compiled lattices (KR + KS, kernel 6): launch of k_eval6 / kr_regions, per-arc weights and accumulators
    LatticeArcs larcs;
    int seg_grid = 0, seg_block = 0, seg_slots = 0; size_t seg_smem = 0;
    bool awg = false;                         // segmented path with the arc weights in HBM/L2 (they do not fit shared memory)
    int64_t seg_max_big_rows = 0;
    DevBuf<uint32_t> d_seg_counter;
    DevBuf<int32_t> d_seg_arc_tid, d_seg_arc_eid;
    DevBuf<double> d_seg_aw, d_seg_xs;
    DevBuf<unsigned long long> d_seg_acc, d_seg_const;
    size_t ks_smem = 0; int ks_grid = 0, ks_block = 512, ks_ctas = 2;
    int64_t kr_big_groups = 0;                  // DAG-form groups (they sort first)
    int64_t kr_groups = 0, ks_groups = 0, seg_types = 0, seg_instances = 0, seg_region_edges = 0, seg_type_edges = 0,
            seg_bridges = 0, seg_words = 0;
    double seg_host_ms = 0;
    // the per-string layout of the segmented path (only ks_strings reads it) is built on a background thread started by
    // set_param_map and uploaded by ensure_ks() when log q of every string is asked for the first time
    std::thread ks_thread;
    std::shared_ptr<SegmentedStringsJob> ks_job;
    std::unique_ptr<SegmentedCorpus> ks_sc;
    bool ks_failed = false;
    DevBuf<uint32_t> d_krwords, d_krpwords, d_kswords;
    DevBuf<int64_t> d_krgoff, d_krpgoff, d_ksgoff;
    DevBuf<int32_t> d_krgrows, d_ksgref, d_kssid, d_eoff, d_earc;
    DevBuf<double> d_krW, d_krlq, d_ksp, d_kslogq, d_seg_logaw;
    std::vector<double> h_p;
    int64_t n_overflow = 0, n_active_w = 0;
    DevBuf<int32_t> d_order_w;                                    // overflow strings (secondary kernel)
    DevBuf<uint16_t> d_adst16;
    DevBuf<double> d_fws;
    DevBuf<int32_t> d_state_final;
    DevBuf<unsigned long long> d_ktlat;
    DevBuf<uint32_t> d_ktcnt;
    DevBuf<int32_t> d_tokT; DevBuf<int64_t> d_goff;
    std::vector<int32_t> h_tokens;
    long long kt_groups = 0;
    std::vector<uint8_t> h_overflow;
    int64_t launches = 0;
    bool structure_done = false, lean_finished = false, lean_now = false;
    std::vector<uint8_t> h_recognised;
    // Hessian
    DevBuf<int64_t> d_hb_path_off, d_hb_col_off, d_hb_val_off;
    DevBuf<int32_t> d_hb_cols;
    DevBuf<double> d_hb_counts, d_hb_p, d_hb_r, d_H, d_rmin;
    DevBuf<unsigned long long> d_Hfx;
    int64_t hb_blocks = -1, hb_paths = 0;
    // H_f from the compiled region types (no path enumeration per string): host copy of the KR arrays, kept by set_param_map
    std::vector<uint32_t> hrw; std::vector<int64_t> hrgoff; std::vector<int32_t> hrgrows; std::vector<double> hrW;
    std::vector<int32_t> h_seg_overflow;       // strings that no region type covers: H_f blocks of their own segments
    std::vector<int32_t> h_ttp, h_etp;
    bool hb_from_types = false, hb_user = false;
    bool hb_types_failed = false;              // the region types of this parameter map have too many paths for blocks
    DevBuf<int32_t> d_hb_slot; DevBuf<double> d_type_lrmin, d_zero_logaw;
    int hb_fx_log2 = 40;
    // rmin without path blocks (rmin_sweep): per string m_s - log q_s, log q and (generic kernel) m_s, (min, +) weights, rmin
    DevBuf<double> d_rterm, d_mlq, d_mpath, d_mtw, d_mew, d_msw, d_mfw, d_rsweep;
    // Viterbi and N-best (wfsa_dev_viterbi, wfsa_dev_nbest): their own x and (max, +) weights, so that an evaluation in
    // flight keeps its x; per path (string s, rank r: s * k + r) logw and (generic kernel) step counts and offsets;
    // backpointer slabs; kg_nbest's lists when the generic scratch holds fewer than k strings' lists; the steps of the last call
    DevBuf<double> d_vx, d_vtw, d_vew, d_vsw, d_vfw, d_vlogw, d_nscratch;
    // sampling (wfsa_dev_sample) besides: its linear weights (k_weights of its own x) and k3_sample's alpha slabs; d_vlogw
    // holds the logw of its n_strings * n draws and then log q of every string
    DevBuf<double> d_stw, d_ssw, d_sfw, d_sslab;
    DevBuf<int32_t> d_vcnt, d_vtrans, d_vemis;
    DevBuf<int64_t> d_voff;
    DevBuf<uint16_t> d_vbp;
    std::vector<int64_t> h_vpath_off;          // steps of path i: h_vpath_off[i]..[i+1]
    int v_k = 1;                               // paths per string of the last call (draws for wfsa_dev_sample)
    bool v_done = false, v_padded = false;     // padded: rank r of string s starts at k * (offs[s] + s) + r * (len_s + 1)
                                               // (fast tables), else at h_vpath_off[s * k + r]
    // comm
    ncclComm_t comm = nullptr; int rank = 0, nranks = 1;
    // NVLink peer memory for the exchange inside k_eval6 (and the rank barrier of the benchmark); without it ncclAllReduce
    bool peer_ok = false; int peer_words = 0; size_t peer_ll_off = 0, peer_bar_off = 0; unsigned long long peer_bar_epoch = 0;
    DevBuf<unsigned long long> peer_local; unsigned long long* peer_ptrs[8] = {nullptr};
    // timing
    Event ev_begin, ev_end; bool timing = false;
    EventPool kev;          // around the dominant kernel(s); mid, segmented path: behind kr_regions (what follows: overflow strings)
    cudaEvent_t mid_now = nullptr;
    DevBuf<unsigned char> d_flush; DevBuf<unsigned int> d_flush_sink; int flush_byte = 0;
    DevBuf<unsigned long long> d_bar;          // rank barrier without peer memory: a one-word ncclAllReduce
    EventPool sev;                              // around each whole evaluation
    DevBuf<long long> d_llpart;             // bridge part of the log-likelihood: per-CTA partials of the weight kernel
    int llpart_n = 0;
    bool timing_detail = true;
    bool evaluated = false;                 // an evaluation has been launched since set_param_map
    bool ks_done = false;                   // ks_strings has run for the last evaluation (it runs on demand)
    // K7: position-synchronous, pair-batched forward-backward for dense automata (kernels_k7.cuh)
    struct K7Batch {
        int NB = 0, Tmax = 0;
        std::vector<int> n_t;                   // [Tmax + 1] strings longer than t
        std::vector<size_t> row_off;            // [Tmax + 1] lattice rows (= perm entries) before step t
        std::vector<size_t> desc_off;           // [Tmax + 1]
        DevBuf<K7Desc> d_desc; DevBuf<int32_t> d_perm, d_sid, d_last;
    };
    std::vector<K7Batch> k7;
    int k7_V = 0; size_t k7_rows = 0, k7_nb = 0;
    DevBuf<double> d_k7lat, d_k7bt, d_k7scale; DevBuf<int> d_k7exp, d_k7EQ, d_k7F;
    double k7_host_ms = 0;
    // pair planes of K7 (k7_build_planes): entries and row words per (symbol pair, candidate), forward and backward tables
    DevBuf<uint32_t> d_k7pef, d_k7prf, d_k7peb, d_k7prb;
    std::vector<int> k7_kf, k7_kb;             // planes in use per pair key
    bool k7_planes = false;
    // single-launch evaluation of the segmented path (k_eval6, kernels_eval6.cuh)
    DevBuf<unsigned int> d_e6ctl;           // [0..1] tickets, [2] barrier arrivals, [3] epoch
    DevBuf<unsigned long long> d_e6acc, d_e6red, d_e6stamps;
    DevBuf<int2> d_arc_tp;
    DevBuf<Eval6Cls> d_e6cls;
    int e6_ncls = 0, e6_big_slots = 0, e6_big_rows = 0; size_t e6_smem = 0;
    bool e6_ok = false, any_overflow = false, e6_used = false, comm_failed = false;
    Graph e6_graph; GraphExec e6_exec; bool e6_graph_tried = false;
    // host-buffer call: the graph's kernel writes [loglik, bad, grad, time-out epoch] and a completion word straight into mapped pinned memory
    PinnedBuf<double> hm_out; double* hm_out_dev = nullptr; PinnedBuf<unsigned int> hm_flag; unsigned int* hm_flag_dev = nullptr; size_t hm_n = 0;
    bool out_on_host = false;               // the results of the last evaluation are in h_out only (graph path)
    unsigned int hm_runs = 0;               // host-buffer launches of k_eval6 since the control words were last reset
    double e2e_ns[4] = {0, 0, 0, 0}; long long e2e_calls = 0;   // WFSA_E2E_DEBUG: host time of the host-buffer call [stage x, graph launch, wait, copy out]
    Event ev_x; bool x_in_flight = false;
    // only the steps whose order matters: the members free themselves afterwards (the stream last)
    ~wfsa_dev()
    {
        if (ks_thread.joinable()) ks_thread.join();
        cudaSetDevice(device);
        if (stream) cudaStreamSynchronize(stream);
        for (int r = 0; r < 8; ++r) if (peer_ptrs[r] && r != rank) cudaIpcCloseMemHandle(peer_ptrs[r]);
        if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(comm);
    }
};

#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess) {                                                              \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                      \
            return WFSA_ERR_CUDA;                                                             \
        }                                                                                     \
    } while (0)

static int set_err(wfsa_dev* h, int code, const std::string& m) { if (h) h->err = m; return code; }

static int nccl_allreduce(wfsa_dev* h, void* buf, size_t count, int dtype, int op)
{
    if (!h->comm) return WFSA_OK;
    const int r = g_nccl.AllReduce(buf, buf, count, dtype, op, h->comm, h->stream);
    if (r != ncclSuccess)
        return set_err(h, WFSA_ERR_NCCL, std::string("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "error"));
    return WFSA_OK;
}

extern "C" const char* wfsa_dev_version(void) { return "wfsa_b200 0.1 (sm_100a)"; }

extern "C" const char* wfsa_dev_last_error(const wfsa_dev* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

extern "C" void wfsa_dev_destroy(wfsa_dev* h) { if (h) delete h; }

extern "C" int64_t wfsa_dev_held_bytes(void) { return g_held_bytes.load(); }

// ---------------------------------------------------------------------------------------------
static int setup_k2(wfsa_dev* h)
{
    // K2: 1 CTA per SM; shared memory = [accumulators] [automaton tables] [per-warp lattice stacks]
    const FastLayout& L = h->fast;
    const size_t max_smem = 227 * 1024;
    const size_t n_acc = (size_t)L.n_arcs + h->fsa.n_states;
    const size_t tab = k2_table_layout(h->fsa.n_sym, h->fsa.n_states, L.n_arcs, L.n_slots).total;
    const int warps = 32;
    const size_t min_stack = (size_t)warps * 128 * 8;
    h->tab_smem = (tab + min_stack <= max_smem) ? 1 : 0;
    const size_t tab_used = h->tab_smem ? tab : 0;
    int accum = h->opt.accum_mode;
    const bool fits = h->tab_smem && n_acc * 8 + tab_used + (size_t)warps * 128 * 8 <= max_smem;
    if (accum == 0) accum = 2;                 // measured: global REDs are as fast and leave room for the stacks
    if (accum == 1 && !fits) accum = 2;
    h->accum = accum;
    h->n_acc_smem = accum == 1 ? (int)n_acc : 0;
    const size_t avail = max_smem - (size_t)h->n_acc_smem * 8 - tab_used;
    h->stack_cap = (int)std::min<size_t>(avail / 8 / warps, 1024);
    h->block = warps * 32;
    h->grid = h->sm_count;
    h->smem_bytes = (size_t)h->n_acc_smem * 8 + tab_used + (size_t)warps * h->stack_cap * 8;
    h->glstack_words = (size_t)(h->max_len + 1) * 33 + 8;
    CK(h->d_glstack.alloc((size_t)h->grid * warps * h->glstack_words));
    const int mx = 227 * 1024;
    cudaFuncSetAttribute(k2_fwdbwd<MODE_EVAL, ACC_SMEM_CAS, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    cudaFuncSetAttribute(k2_fwdbwd<MODE_EVAL, ACC_SMEM_SPLIT, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    cudaFuncSetAttribute(k2_fwdbwd<MODE_EVAL, ACC_GLOBAL, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    cudaFuncSetAttribute(k2_fwdbwd<MODE_EVAL, ACC_GLOBAL, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    cudaFuncSetAttribute(k2_fwdbwd<MODE_EVAL, ACC_NONE, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    cudaFuncSetAttribute(k2_fwdbwd<MODE_STRUCT, ACC_GLOBAL, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    cudaFuncSetAttribute(k2_fwdbwd<MODE_STRUCT, ACC_GLOBAL, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
    return WFSA_OK;
}

static int setup_k3(wfsa_dev* h)
{
    const FastLayout& L = h->fast;
    int nt = ((L.max_cand + 31) / 32) * 32;
    nt = std::max(nt, 64);
    h->k3_block = nt;
    h->k3_grid = h->sm_count * std::max(1, std::min(4, 1024 / nt));
    h->k3_smem = (size_t)(2 * nt + 32) * 8 + 40 * 4;
    CK(h->d_k3lat.alloc((size_t)h->k3_grid * std::max(h->max_len, 1) * nt));
    CK(h->d_k3exp.alloc((size_t)h->k3_grid * std::max(h->max_len, 1)));
    return WFSA_OK;
}

// thread-per-string: tables + 2 active lists of K entries per thread must fit 227 KB
static bool kt_possible(const wfsa_dev* h, int K, int& nt, size_t& smem)
{
    if (!h->fast.ok || !h->fast.compact_ok) return false;
    const size_t tab = kt_table_layout(h->fsa.n_sym, h->fsa.n_states, h->fast.n_arcs).total;
    const size_t max_smem = 227 * 1024;
    if (tab + (size_t)128 * K * 20 > max_smem) return false;
    nt = (int)((max_smem - tab) / ((size_t)K * 20) / 32) * 32;
    nt = std::min(nt, 768);
    smem = tab + (size_t)nt * K * 20;
    return nt >= 128;
}

static int setup_kt(wfsa_dev* h)
{
    int K = (h->opt.reserved >> 16) & 0xff;
    if (K == 0) K = 8;
    int nt = 0; size_t smem = 0;
    if (!kt_possible(h, K, nt, smem)) return set_err(h, WFSA_ERR_LIMIT, "thread-per-string kernel: tables do not fit shared memory");
    h->kt_K = K; h->kt_block = nt; h->kt_grid = h->sm_count; h->kt_smem = smem;
    const size_t warps = (size_t)h->kt_grid * nt / 32;
    h->kt_lat_words = (size_t)std::max(h->max_len, 1) * K * 32;      // per warp
    CK(h->d_ktlat.alloc(warps * h->kt_lat_words));
    CK(h->d_ktcnt.alloc(warps * (size_t)std::max(h->max_len, 1) * 32));
    cudaFuncSetAttribute(kt_fwdbwd<MODE_EVAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    cudaFuncSetAttribute(kt_fwdbwd<MODE_STRUCT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    return WFSA_OK;
}

// segmented kernels: per-arc weights + K pool doubles per thread must fit 227 KB
// `awg` (may be null = not allowed): set when the table does not fit but the pool alone does -- the segmented kernels then read
// the weights from HBM/L2 (their AWG instances)
static bool seg_possible(const wfsa_dev* h, int K, int want_nt, int& nt, size_t& smem, bool* awg = nullptr)
{
    const LatticeArcs& A = h->larcs;
    if (awg) *awg = false;
    if (A.n_arcs <= 0 || A.n_arcs >= (1 << kLatArcBits)) return false;
    size_t tab = ((size_t)A.n_arcs + 1) * 8;
    const size_t max_smem = 227 * 1024 - 9216;     // + the zero weight of padding (kr_regions); k_eval6 has 7 KB of static shared memory, kr_regions up to 8
    const int S = std::max(K, kPathSlots);          // pool slots per thread: K for the DAG form, at least kPathSlots (kr_paths)
    if (tab + (size_t)128 * S * 8 > max_smem) {
        if (!awg) return false;
        *awg = true; tab = 0;
    }
    nt = (int)((max_smem - tab) / ((size_t)S * 8) / 32) * 32;
    nt = std::min(nt, 1024);
    if (want_nt > 0) nt = std::min(nt, want_nt);
    smem = tab + (size_t)nt * S * 8;
    return nt >= 128;
}

// K7 pair planes: built on the device from the per-state tables (structure only, once per handle).  If they do not fit
// (alphabets far beyond config 5), K7 keeps walking the per-state tables (k7_fwd / k7_bwd).
static int setup_k7_planes(wfsa_dev* h)
{
    h->k7_planes = false;
    if (getenv("WFSA_K7_NO_PLANES")) return WFSA_OK;
    const FastLayout& L = h->fast;
    const size_t A = (size_t)L.n_sym, V = (size_t)h->k7_V, n_keys = (A + 1) * A;
    const size_t words = n_keys * V * (kK7Planes + 1);
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return WFSA_OK; }
    if (2 * words * 4 > free_b / 8) return WFSA_OK;
    DevBuf<uint32_t> pef, prf, peb, prb; DevBuf<int> d_kmax;       // the planes go to the handle once they are built
    if (pef.alloc(n_keys * V * kK7Planes) != cudaSuccess || prf.alloc(n_keys * V) != cudaSuccess ||
        peb.alloc(n_keys * V * kK7Planes) != cudaSuccess || prb.alloc(n_keys * V) != cudaSuccess ||
        d_kmax.alloc(2 * n_keys) != cudaSuccess) {
        cudaGetLastError();
        return WFSA_OK;
    }
    FastTablesD T{};
    T.cand_off = h->d_cand_off.p; T.slot_state = h->d_slot_state.p;
    T.frow = h->d_frow.p; T.fent = h->d_fent.p; T.brow = h->d_brow.p; T.bent = h->d_bent.p;
    T.n_sym = L.n_sym; T.n_states = h->fsa.n_states; T.n_arcs = L.n_arcs; T.n_slots = L.n_slots;
    k7_build_planes<<<(unsigned)n_keys, (unsigned)V, 0, h->stream>>>(T, (int)V, 1, pef.p, prf.p, d_kmax.p);
    k7_build_planes<<<(unsigned)n_keys, (unsigned)V, 0, h->stream>>>(T, (int)V, 0, peb.p, prb.p, d_kmax.p + n_keys);
    h->k7_kf.assign(n_keys, 0); h->k7_kb.assign(n_keys, 0);
    CK(cudaMemcpyAsync(h->k7_kf.data(), d_kmax.p, n_keys * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(h->k7_kb.data(), d_kmax.p + n_keys, n_keys * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->d_k7pef = std::move(pef); h->d_k7prf = std::move(prf); h->d_k7peb = std::move(peb); h->d_k7prb = std::move(prb);
    h->k7_planes = true;
    return WFSA_OK;
}

static int setup_seg(wfsa_dev* h)
{
    int K = (h->opt.reserved >> 16) & 0xff;
    if (K == 0 || K > kLatMaxSlots) K = kLatMaxSlots;
    int nt = 0; size_t smem = 0;
    int want_nt = ((h->opt.reserved >> 24) & 0x7f) * 32;
    if (want_nt == 0) want_nt = 512;       // measured: 16 warps leave the L1 to the register spills
    bool awg = false;
    if (!seg_possible(h, K, want_nt, nt, smem, &awg))
        return set_err(h, WFSA_ERR_LIMIT, "segmented kernel: the arc weights do not fit shared memory");
    h->awg = awg;
    if (want_nt == 512 || nt > 512 || awg) {   // k_eval6 is compiled for 512, 256 and 128 threads (AWG: 512), kr_regions for up to 512
        nt = awg ? 512 : (nt >= 512 ? 512 : (nt >= 256 ? 256 : 128));
        smem = (awg ? 0 : ((size_t)h->larcs.n_arcs + 1) * 8) + (size_t)nt * std::max(K, kPathSlots) * 8;
    }
    h->seg_slots = K; h->seg_block = nt; h->seg_grid = h->sm_count; h->seg_smem = smem;
    // experiment / test knob: a smaller persistent grid, so that a small shard reaches the schedules of a large one (more big DAG
    // groups than CTAs, several per warp).  Read here, before the per-warp x stacks are sized from seg_grid.
    if (const char* g = getenv("WFSA_E6_GRID")) h->seg_grid = std::min(h->sm_count, std::max(1, atoi(g)));
    const LatticeArcs& A = h->larcs;
    CK(h->d_seg_arc_tid.upload(A.arc_tid, h->stream)); CK(h->d_seg_arc_eid.upload(A.arc_eid, h->stream));
    CK(h->d_seg_aw.alloc((size_t)A.n_arcs + 1)); CK(cudaMemsetAsync(h->d_seg_aw.p, 0, ((size_t)A.n_arcs + 1) * 8, h->stream)); CK(h->d_seg_acc.alloc((size_t)A.n_arcs * h->replicas)); CK(h->d_seg_const.alloc(A.n_arcs));
    CK(h->d_seg_counter.alloc(2));
    CK(h->d_llpart.alloc(2 * (size_t)((std::max(h->larcs.n_arcs, 1) + 255) / 256)));
    CK(h->d_seg_logaw.alloc((size_t)A.n_arcs + 16)); CK(cudaMemsetAsync(h->d_seg_logaw.p, 0, ((size_t)A.n_arcs + 16) * 8, h->stream));   // (+ the zero entries of the padding ids)
    {   // arcs of every edge (transition edges, then emission edges) for the gather in k_fold_finish6
        const int nt = h->fsa.n_trans(), ne = nt + h->fsa.n_emis();
        std::vector<int32_t> off((size_t)ne + 1, 0), arc;
        for (int a = 0; a < A.n_arcs; ++a) { off[A.arc_tid[a] + 1]++; if (A.arc_eid[a] >= 0) off[nt + A.arc_eid[a] + 1]++; }
        for (int e = 0; e < ne; ++e) off[e + 1] += off[e];
        arc.resize((size_t)off[ne]);
        std::vector<int32_t> fill(off.begin(), off.end() - 1);
        for (int a = 0; a < A.n_arcs; ++a) { arc[fill[A.arc_tid[a]]++] = a; if (A.arc_eid[a] >= 0) arc[fill[nt + A.arc_eid[a]]++] = a; }
        CK(h->d_eoff.upload(off, h->stream)); CK(h->d_earc.upload(arc, h->stream));
    }
    {   // single-launch evaluation: control words (tickets, barrier arrivals, epoch = 1), reduction cells, phase stamps
        const std::vector<unsigned int> ctl = {0u, 0u, 0u, 1u, 0u, 0u, 0u, 0u};
        CK(h->d_e6ctl.upload(ctl, h->stream));
        CK(h->d_e6red.alloc(2)); CK(cudaMemsetAsync(h->d_e6red.p, 0, 16, h->stream));
        CK(h->d_e6stamps.alloc(8 + 8 * 1024)); CK(cudaMemsetAsync(h->d_e6stamps.p, 0, (8 + 8 * 1024) * 8, h->stream));
        cudaFuncSetAttribute(k_eval6<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 8192);
        cudaFuncSetAttribute(k_eval6<384>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 8192);
        cudaFuncSetAttribute(k_eval6<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 8192);
        cudaFuncSetAttribute(k_eval6<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 8192);
    }
    h->ks_smem = h->awg ? 0 : ((size_t)A.n_arcs + 16) * 8;
    h->ks_block = kKsWarps * 32;
    h->ks_ctas = h->ks_smem * 2 + 2048 <= 227 * 1024 ? 2 : 1;
    h->ks_grid = h->sm_count * h->ks_ctas;
    cudaFuncSetAttribute(k_eval6<512, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 8192);
    cudaFuncSetAttribute(kr_regions<ACC_GLOBAL, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 8192 - 1024);
    cudaFuncSetAttribute(kr_regions<ACC_NONE, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 8192 - 1024);
    cudaFuncSetAttribute(kr_regions<ACC_GLOBAL, 512, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 8192 - 1024);
    cudaFuncSetAttribute(ks_strings<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->ks_smem);   // it also has static shared memory
    return WFSA_OK;
}

static int setup_generic(wfsa_dev* h)
{
    const size_t per = (size_t)2 * (h->max_len + 1) * h->fsa.n_states;
    const size_t budget = (size_t)1 << 28;   // 2 GiB of doubles at most
    long long batch = (long long)std::max<size_t>(1, budget / std::max<size_t>(per, 1));
    batch = std::min<long long>(batch, std::max<int64_t>(h->n_strings, 1));
    batch = std::min<long long>(batch, 1 << 20);
    h->g_batch = batch;
    CK(h->d_gscratch.alloc((size_t)batch * per));
    return WFSA_OK;
}

static int choose_launch(wfsa_dev* h)
{
    h->replicas = (h->opt.reserved >> 8) & 0xff;
    if (h->replicas <= 0) h->replicas = 16;
    if (h->fast.ok) {
        const size_t n_acc = (size_t)h->fast.n_arcs + h->fsa.n_states;
        CK(h->d_acc.alloc(n_acc * h->replicas));
    }
    int rc = WFSA_OK;
    h->skernel = h->kernel;
    if (h->kernel == 6) {
        h->secondary = h->fast.warp_ok ? 1 : (h->fast.ok ? 2 : 3);
        int nt = 0; size_t sm = 0; int K = (h->opt.reserved >> 16) & 0xff; if (K == 0) K = 8;
        h->skernel = (h->fast.ok && kt_possible(h, K, nt, sm)) ? 4 : h->secondary;
        rc = setup_seg(h);
        if (rc == WFSA_OK && h->skernel == 4) rc = setup_kt(h);
        if (rc == WFSA_OK) rc = h->secondary == 1 ? setup_k2(h) : (h->secondary == 2 ? setup_k3(h) : setup_generic(h));
    } else if (h->kernel == 4) {
        h->secondary = h->fast.warp_ok ? 1 : 2;
        rc = setup_kt(h);
        if (rc == WFSA_OK) rc = h->secondary == 1 ? setup_k2(h) : setup_k3(h);
    } else if (h->kernel == 7) {
        h->secondary = 2; h->skernel = 2;                  // structural pass and strings with unknown symbols: CTA-per-string kernel
        h->k7_V = (h->fast.max_cand + 31) / 32 * 32;
        cudaFuncSetAttribute(k7_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, kK7Chunk * h->k7_V * 8);
        cudaFuncSetAttribute(k7_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, kK7Chunk * h->k7_V * 8);
        {   // up to 320 candidates per symbol (config 5): four forward / three backward CTAs per SM; else two of up to 512 threads
            auto prep = [&](auto kern) {
                cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kK7Chunk * h->k7_V * 8);
                cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            };
            prep(k7_fwd2<320, 4>); prep(k7_fwd2<512, 2>); prep(k7_bwd2<320, 3>); prep(k7_bwd2<512, 2>);
            prep(k7_minfwd2<320, 4>); prep(k7_minfwd2<512, 2>);
        }
        rc = setup_k3(h);
        if (rc == WFSA_OK) rc = setup_k7_planes(h);
    } else if (h->kernel == 1) rc = setup_k2(h);
    else if (h->kernel == 2) rc = setup_k3(h);
    else rc = setup_generic(h);
    h->accum = (h->kernel == 1 || (h->kernel >= 4 && h->secondary == 1)) ? h->accum : 2;
    return rc;
}

extern "C" int wfsa_dev_create(const wfsa_fsa_desc* fd, const wfsa_corpus_desc* cd, const wfsa_dev_options* opt, wfsa_dev** out)
{
    g_create_error.clear();
    if (!out) { g_create_error = "out is NULL"; return WFSA_ERR_INVALID; }
    *out = nullptr;
    std::unique_ptr<wfsa_dev> owner(new wfsa_dev());
    wfsa_dev* const h = owner.get();
    auto bail = [&](int code) { g_create_error = h->err; return code; };
    if (opt) h->opt = *opt;
    int status = WFSA_OK;
    std::string msg = copy_and_validate(fd, h->fsa, status);
    if (status != WFSA_OK) { h->err = msg; return bail(status); }
    if (!cd || cd->n_strings < 0 || (cd->n_strings && (!cd->offsets || !cd->p))) { h->err = "corpus descriptor invalid"; return bail(WFSA_ERR_INVALID); }
    if (cd->n_strings > 0x7fffffff) { h->err = "more than 2^31 strings in one shard"; return bail(WFSA_ERR_LIMIT); }

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        h->err = "no CUDA device visible: the w-fsa B200 backend has no CPU fallback";
        return bail(WFSA_ERR_NO_DEVICE);
    }
    h->device = h->opt.device;
    if (h->device < 0 || h->device >= ndev) { h->err = "device ordinal out of range"; return bail(WFSA_ERR_INVALID); }
    cudaDeviceProp prop;
    if (cudaSetDevice(h->device) != cudaSuccess || cudaGetDeviceProperties(&prop, h->device) != cudaSuccess) {
        h->err = "cudaSetDevice failed"; return bail(WFSA_ERR_NO_DEVICE);
    }
    if (prop.major != 10) {
        h->err = std::string("device ") + prop.name + " is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                 "; this library contains sm_100a code only";
        return bail(WFSA_ERR_NO_DEVICE);
    }
    h->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&h->stream.raw, cudaStreamNonBlocking) != cudaSuccess) { h->err = "cudaStreamCreate failed"; return bail(WFSA_ERR_CUDA); }
    cudaEventCreate(&h->ev_begin.raw); cudaEventCreate(&h->ev_end.raw);

    // ---- layout
    msg = build_fast_layout(h->fsa, h->fast, status);
    if (status != WFSA_OK) { h->err = msg; return bail(status); }
    msg = build_generic_layout(h->fsa, h->gen, status);
    if (status != WFSA_OK) { h->err = msg; return bail(status); }
    build_lattice_arcs(h->fsa, h->gen, h->larcs);
    int kernel = h->opt.force_kernel;
    if (kernel == 0) {
        int nt = 0; size_t sm = 0; int K = (h->opt.reserved >> 16) & 0xff; if (K == 0) K = 8;
        bool awg = false;
        if (h->larcs.n_arcs < 65520 && seg_possible(h, kLatMaxSlots, 0, nt, sm, &awg)) kernel = 6;      // weights in shared memory or in HBM/L2 (16-bit arc ids still fit)
        else kernel = !h->fast.ok ? 3 : (kt_possible(h, K, nt, sm) ? 4 : (h->fast.warp_ok ? 1 : (((h->fast.max_cand + 31) / 32 * 32 <= 512 && cd && cd->n_strings >= 200000) ? 7 : 2)));     // K7 pays off once ~3 strings share a symbol pair per position
    }
    if (kernel == 6 && h->larcs.n_arcs >= 65520) { h->err = "forced segmented kernel but the automaton has 65520 or more combined arcs"; return bail(WFSA_ERR_INVALID); }
    if (kernel == 6) { int nt = 0; size_t sm = 0; bool awg = false; if (!seg_possible(h, kLatMaxSlots, 0, nt, sm, &awg)) { h->err = "forced segmented kernel but the arc weights do not fit shared memory"; return bail(WFSA_ERR_INVALID); } }
    if (kernel == 7 && h->fast.ok && (h->fast.max_cand + 31) / 32 * 32 > 512) { h->err = "forced batched kernel but more than 512 states emit one symbol"; return bail(WFSA_ERR_INVALID); }
    if ((kernel == 1 || kernel == 2 || kernel == 4 || kernel == 7) && !h->fast.ok) { h->err = "forced fast kernel but emissions are not all one token long"; return bail(WFSA_ERR_INVALID); }
    if (kernel == 1 && !h->fast.warp_ok) { h->err = "forced warp-per-string kernel but more than 32 states emit one symbol"; return bail(WFSA_ERR_INVALID); }
    if (kernel == 5) { h->err = "force_kernel 5 (thread-per-string over compiled lattices) was removed: the segmented kernel 6 takes every input it took"; return bail(WFSA_ERR_INVALID); }
    if (kernel < 1 || kernel > 7) { h->err = "force_kernel out of range"; return bail(WFSA_ERR_INVALID); }
    h->kernel = kernel;

    // ---- corpus shard
    h->n_strings = cd->n_strings;
    h->h_offs.assign(cd->offsets ? cd->offsets : nullptr, cd->offsets ? cd->offsets + cd->n_strings + 1 : nullptr);
    if (h->h_offs.empty()) h->h_offs.push_back(0);
    if (h->h_offs[0] != 0) { h->err = "offsets must start at 0"; return bail(WFSA_ERR_INVALID); }
    for (int64_t s = 0; s < h->n_strings; ++s) {
        const int64_t len = h->h_offs[s + 1] - h->h_offs[s];
        if (len < 0 || len > (1 << 24)) { h->err = "string length out of range"; return bail(WFSA_ERR_INVALID); }
        h->max_len = std::max<int>(h->max_len, (int)len);
    }
    h->n_tokens = h->h_offs.back();
    if (h->n_tokens && !cd->tokens) { h->err = "tokens is NULL"; return bail(WFSA_ERR_INVALID); }
    h->h_order_all.resize(h->n_strings);
    std::iota(h->h_order_all.begin(), h->h_order_all.end(), 0);
    std::stable_sort(h->h_order_all.begin(), h->h_order_all.end(), [&](int32_t a, int32_t b) {
        return (h->h_offs[a + 1] - h->h_offs[a]) > (h->h_offs[b + 1] - h->h_offs[b]);
    });
    cudaStream_t st = h->stream;
#define CKB(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { h->err = std::string(#call) + ": " + cudaGetErrorString(e_); return bail(e_ == cudaErrorMemoryAllocation ? WFSA_ERR_NOMEM : WFSA_ERR_CUDA); } } while (0)
    CKB(h->d_tokens.alloc(std::max<int64_t>(h->n_tokens, 1) + 32));
    if (h->n_tokens) CKB(cudaMemcpyAsync(h->d_tokens.p, cd->tokens, (size_t)h->n_tokens * 4, cudaMemcpyHostToDevice, st));
    if (kernel >= 4 && h->n_tokens) h->h_tokens.assign(cd->tokens, cd->tokens + h->n_tokens);
    if (h->n_strings) h->h_p.assign(cd->p, cd->p + h->n_strings);
    CKB(h->d_offs.upload(h->h_offs, st));
    CKB(h->d_p.alloc(std::max<int64_t>(h->n_strings, 1)));
    if (h->n_strings) CKB(cudaMemcpyAsync(h->d_p.p, cd->p, (size_t)h->n_strings * 8, cudaMemcpyHostToDevice, st));
    CKB(h->d_order.alloc(std::max<int64_t>(h->n_strings, 1)));
    CKB(h->d_order_w.alloc(std::max<int64_t>(h->n_strings, 1)));
    CKB(h->d_logq.alloc(std::max<int64_t>(h->n_strings, 1)));
    CKB(h->d_pathcnt.alloc(std::max<int64_t>(h->n_strings, 1)));

    // ---- tables
    const HostFsa& F = h->fsa;
    h->n_edges = F.n_trans() + F.n_emis();
    if (h->fast.ok) {
        const FastLayout& L = h->fast;
        CKB(h->d_cand_off.upload(L.cand_off, st)); CKB(h->d_slot_state.upload(L.slot_state, st));
        CKB(h->d_frow.upload(L.frow, st)); CKB(h->d_fent.upload(L.fent, st));
        CKB(h->d_brow.upload(L.brow, st)); CKB(h->d_bent.upload(L.bent, st));
        CKB(h->d_slot_emis.upload(L.slot_emis, st)); CKB(h->d_slot_final.upload(L.slot_final, st));
        CKB(h->d_arc_tid.upload(L.arc_tid, st)); CKB(h->d_arc_eid.upload(L.arc_eid, st));
        CKB(h->d_state_final.upload(L.state_final, st));
        CKB(h->d_fws.alloc(std::max(F.n_states, 1)));
        if (L.compact_ok) {
            CKB(h->d_brow16.upload(L.brow16, st)); CKB(h->d_adst16.upload(L.arc_dst16, st));
            CKB(h->d_aw.alloc(std::max(L.n_arcs, 1)));
        }
        if (L.warp_ok) { CKB(h->d_bent8.upload(L.bent_dst, st)); CKB(h->d_sstate16.upload(L.slot_state16, st)); }
        CKB(h->d_sw.alloc(L.n_slots)); CKB(h->d_fw.alloc(L.n_slots));
        h->table_bytes = 4 * (L.cand_off.size() + L.slot_state.size() + L.frow.size() + L.fent.size() + L.brow.size() + L.bent.size()) +
                         8 * ((size_t)F.n_trans() + 2 * L.n_slots);
    }
    CKB(h->d_emis_row.upload(F.emis_row, st)); CKB(h->d_emis_tok_off.upload(F.emis_tok_off, st));
    CKB(h->d_emis_tok.upload(F.emis_tok, st)); CKB(h->d_trans_row.upload(F.trans_row, st));
    CKB(h->d_trans_dst.upload(F.trans_dst, st)); CKB(h->d_eps_order.upload(h->gen.eps_order, st));
    CKB(h->d_tw.alloc(std::max(F.n_trans(), 1))); CKB(h->d_ltw.alloc(std::max(F.n_trans(), 1)));
    CKB(h->d_lew.alloc(std::max(F.n_emis(), 1)));
    CKB(h->d_trans_tp.alloc(std::max(F.n_trans(), 1))); CKB(h->d_emis_tp.alloc(std::max(F.n_emis(), 1)));
    CKB(h->d_edge_tp.alloc(std::max(h->n_edges, 1)));
    {
        std::vector<int32_t> raw(F.trans_param);
        raw.insert(raw.end(), F.emis_param.begin(), F.emis_param.end());
        CKB(h->d_edge_raw.upload(raw, st));
    }
    CKB(h->d_red.alloc((size_t)h->n_edges + 2));
    CKB(h->d_used.alloc(std::max(F.n_raw, 1)));
    if (choose_launch(h) != WFSA_OK) return bail(WFSA_ERR_CUDA);
    CKB(cudaStreamSynchronize(st));
#undef CKB
    *out = owner.release();
    return WFSA_OK;
}

// ---------------------------------------------------------------------------------------------
// warp-interleaved copy of the tokens of an order list: group g = 32 consecutive strings, token t of
// lane l at goff[g] + t*32 + l, so that a warp of the thread-per-string kernel reads 128 contiguous bytes
static int upload_transposed_tokens(wfsa_dev* h, const std::vector<int32_t>& order)
{
    const long long n = (long long)order.size();
    const long long groups = (n + 31) / 32;
    std::vector<int64_t> goff((size_t)groups + 1, 0);
    for (long long g = 0; g < groups; ++g) {
        int64_t mx = 0;
        for (long long i = g * 32; i < std::min(n, g * 32 + 32); ++i) mx = std::max<int64_t>(mx, h->h_offs[order[i] + 1] - h->h_offs[order[i]]);
        goff[g + 1] = goff[g] + mx * 32;
    }
    std::vector<int32_t> tokT((size_t)goff[groups] + 32, -1);
    for (long long i = 0; i < n; ++i) {
        const int64_t off = h->h_offs[order[i]], len = h->h_offs[order[i] + 1] - off;
        int32_t* dst = tokT.data() + goff[i / 32] + (i % 32);
        for (int64_t t = 0; t < len; ++t) dst[t * 32] = h->h_tokens[off + t];
    }
    CK(h->d_tokT.upload(tokT, h->stream));
    CK(h->d_goff.upload(goff, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->kt_groups = groups;
    return WFSA_OK;
}

static void launch_main(wfsa_dev* h, int kernel, int mode, const CorpusD& C, const EvalOutD& O)
{
    const HostFsa& F = h->fsa;
    const FastLayout& L = h->fast;
    cudaStream_t st = h->stream;
    if (C.n_order <= 0) return;
    if (kernel == 6) {
        // (the general path: evaluations with overflow strings, or without the single-launch kernel)
        cudaMemsetAsync(h->d_seg_counter.p, 0, 8, st);
        if (h->kr_groups > 0) {
            KRParams P{};
            P.aw = h->d_seg_aw.p; P.words = h->d_krwords.p; P.goff = h->d_krgoff.p; P.grows = h->d_krgrows.p; P.typeW = h->d_krW.p;
            P.pwords = h->d_krpwords.p; P.pgoff = h->d_krpgoff.p;
            P.lq = h->d_krlq.p; P.n_groups = h->kr_groups; P.xs = h->d_seg_xs.p; P.xs_rows = (size_t)std::max<int64_t>(h->seg_max_big_rows, 1);
            P.counter = h->d_seg_counter.p; P.acc = h->d_seg_acc.p; P.fx_scale = O.fx_scale; P.n_arcs = h->larcs.n_arcs; P.replicas = h->replicas;
            P.ll_scale = O.ll_scale; P.red = O.red; P.llpart = h->d_llpart.p; P.n_llpart = h->llpart_n;
            if (h->awg) kr_regions<ACC_GLOBAL, 512, true><<<h->seg_grid, h->seg_block, h->seg_smem, st>>>(P);       // weights read from HBM/L2
            else if (h->opt.reserved & 2) kr_regions<ACC_NONE, 512><<<h->seg_grid, h->seg_block, h->seg_smem, st>>>(P);   // timing experiment
            else kr_regions<ACC_GLOBAL, 512><<<h->seg_grid, h->seg_block, h->seg_smem, st>>>(P);
            h->launches++;
        }
        if (h->mid_now) cudaEventRecord(h->mid_now, st);
        // [loglik, grad] are complete after kr_regions: the bridges of every string are folded into constants
        // (gradient: const_acc; log-likelihood: the llpart partials of the weight kernel).  Per-string log q is
        // only computed when a caller asks for it (wfsa_dev_eval_fetch with logq != NULL launches ks_strings).
        h->ks_done = false;
        if (h->kr_groups == 0 && h->larcs.n_arcs > 0) {          // no region at all (unique paths): the bridge part on its own
            k_add_llpart<<<1, 32, 0, st>>>(h->d_llpart.p, h->llpart_n, O.red);
            h->launches++;
        }
    } else if (kernel == 4) {
        KTParams P{};
        P.T = ThreadTablesD{h->d_brow16.p, h->d_adst16.p, h->d_aw.p, h->d_fws.p, F.n_sym, F.n_states, L.n_arcs, F.start, L.start_final_tid};
        P.tw = h->d_tw.p; P.C = C; P.O = O; P.lattice = h->d_ktlat.p; P.latcnt = h->d_ktcnt.p;
        P.tokT = h->d_tokT.p; P.goff = h->d_goff.p; P.n_groups = h->kt_groups;
        P.max_len = std::max(h->max_len, 1); P.K = h->kt_K; P.replicas = h->replicas;
        if (mode == MODE_STRUCT) kt_fwdbwd<MODE_STRUCT><<<h->kt_grid, h->kt_block, h->kt_smem, st>>>(P);
        else kt_fwdbwd<MODE_EVAL><<<h->kt_grid, h->kt_block, h->kt_smem, st>>>(P);
        h->launches++;
    } else if (kernel == 1) {
        K2Params P{};
        P.T = WarpTablesD{h->d_brow16.p, h->d_bent8.p, h->d_sstate16.p, h->d_cand_off.p, h->d_aw.p, h->d_fw.p,
                          F.n_sym, F.n_states, L.n_arcs, L.n_slots, F.start, L.start_final_tid};
        P.tw = h->d_tw.p; P.C = C; P.O = O;
        P.stack_cap = h->stack_cap; P.gl_stack = h->d_glstack.p; P.gl_stack_words = h->glstack_words;
        P.replicas = h->replicas;
        const size_t tab = h->tab_smem ? k2_table_layout(F.n_sym, F.n_states, L.n_arcs, L.n_slots).total : 0;
        if (mode == MODE_STRUCT || h->accum != 1) {
            P.n_acc_smem = 0;
            const size_t avail = 227 * 1024 - tab;       // without shared accumulators the stacks get the rest
            P.stack_cap = (int)std::min<size_t>(avail / 8 / (h->block / 32), 1024);
            const size_t smem = tab + (size_t)(h->block / 32) * P.stack_cap * 8;
            if (mode == MODE_STRUCT) {
                if (h->tab_smem) k2_fwdbwd<MODE_STRUCT, ACC_GLOBAL, 1><<<h->grid, h->block, smem, st>>>(P);
                else k2_fwdbwd<MODE_STRUCT, ACC_GLOBAL, 0><<<h->grid, h->block, smem, st>>>(P);
            } else if (h->opt.reserved & 2) {
                k2_fwdbwd<MODE_EVAL, ACC_NONE, 1><<<h->grid, h->block, smem, st>>>(P);      // timing experiment
            } else {
                if (h->tab_smem) k2_fwdbwd<MODE_EVAL, ACC_GLOBAL, 1><<<h->grid, h->block, smem, st>>>(P);
                else k2_fwdbwd<MODE_EVAL, ACC_GLOBAL, 0><<<h->grid, h->block, smem, st>>>(P);
            }
        } else {
            P.n_acc_smem = h->n_acc_smem;
            if (h->opt.reserved & 1) k2_fwdbwd<MODE_EVAL, ACC_SMEM_CAS, 1><<<h->grid, h->block, h->smem_bytes, st>>>(P);
            else k2_fwdbwd<MODE_EVAL, ACC_SMEM_SPLIT, 1><<<h->grid, h->block, h->smem_bytes, st>>>(P);
        }
        h->launches++;
    } else if (kernel == 7) {
        FastTablesD T{};
        T.cand_off = h->d_cand_off.p; T.slot_state = h->d_slot_state.p;
        T.frow = h->d_frow.p; T.fent = h->d_fent.p; T.brow = h->d_brow.p; T.bent = h->d_bent.p;
        T.n_sym = F.n_sym; T.n_states = F.n_states; T.n_arcs = L.n_arcs; T.n_slots = L.n_slots;
        T.start_state = F.start; T.start_final_tid = L.start_final_tid;
        const EvalWeightsD Wt{h->d_tw.p, h->d_sw.p, h->d_fw.p};
        const int V = h->k7_V;
        const size_t smem = (size_t)kK7Chunk * V * 8;
        double* const lat = h->d_k7lat.p;
        double* const bt[2] = {h->d_k7bt.p, h->d_k7bt.p + h->k7_nb * (size_t)V};
        for (auto& B : h->k7) {
            K7FinParams Fn{};
            Fn.T = T; Fn.W = Wt; Fn.O = O; Fn.sid = B.d_sid.p; Fn.last_tok = B.d_last.p; Fn.p = h->d_p.p;
            Fn.scale = h->d_k7scale.p; Fn.EQ = h->d_k7EQ.p; Fn.F = h->d_k7F.p; Fn.V = V;
            K7Params P{};
            P.T = T; P.W = Wt; P.O = O; P.V = V; P.F = h->d_k7F.p; P.EQ = h->d_k7EQ.p; P.scale = h->d_k7scale.p;
            for (int t = 0; t < B.Tmax; ++t) {                 // forward: every string of the batch advances one position
                P.desc = B.d_desc.p + B.desc_off[t]; P.perm = B.d_perm.p + B.row_off[t];
                P.src = t ? lat + B.row_off[t - 1] * V : nullptr; P.dst = lat + B.row_off[t] * V;
                P.exp_src = t ? h->d_k7exp.p + B.row_off[t - 1] : nullptr; P.exp_dst = h->d_k7exp.p + B.row_off[t];
                P.rescale = (t & (kRescaleEvery - 1)) == kRescaleEvery - 1;
                const unsigned nd = (unsigned)(B.desc_off[t + 1] - B.desc_off[t]);
                if (nd) {
                    if (h->k7_planes) {
                        P.pe = h->d_k7pef.p; P.pr = h->d_k7prf.p;
                        if (V <= 320) k7_fwd2<320, 4><<<nd, V, smem, st>>>(P); else k7_fwd2<512, 2><<<nd, V, smem, st>>>(P);
                    }
                    else k7_fwd<<<nd, V, smem, st>>>(P);
                    h->launches++;
                }
                if (B.n_t[t + 1] < B.n_t[t]) {                 // strings that end here: q, log q, p_s / q_s
                    Fn.r0 = B.n_t[t + 1]; Fn.r1 = B.n_t[t]; Fn.lat = lat + B.row_off[t] * V; Fn.exp_t = h->d_k7exp.p + B.row_off[t];
                    k7_finish_q<<<(Fn.r1 - Fn.r0 + 7) / 8, 256, 0, st>>>(Fn);
                    h->launches++;
                }
            }
            for (int t = B.Tmax - 1; t >= 0; --t) {             // backward
                if (B.n_t[t + 1] < B.n_t[t]) {
                    Fn.r0 = B.n_t[t + 1]; Fn.r1 = B.n_t[t]; Fn.lat = lat + B.row_off[t] * V; Fn.exp_t = h->d_k7exp.p + B.row_off[t];
                    Fn.bt = bt[t & 1];
                    k7_finish_beta<<<(Fn.r1 - Fn.r0 + 7) / 8, 256, 0, st>>>(Fn);
                    h->launches++;
                }
                if (t + 1 < B.Tmax && B.n_t[t + 1] > 0) {
                    P.desc = B.d_desc.p + B.desc_off[t + 1]; P.perm = B.d_perm.p + B.row_off[t + 1];
                    P.src = bt[(t + 1) & 1]; P.dst = bt[t & 1]; P.lat = lat + B.row_off[t] * V; P.exp_t = h->d_k7exp.p + B.row_off[t];
                    P.rescale = (t & (kRescaleEvery - 1)) == 0;
                    const unsigned nd = (unsigned)(B.desc_off[t + 2] - B.desc_off[t + 1]);
                    if (nd) {
                        if (h->k7_planes) {
                            P.pe = h->d_k7peb.p; P.pr = h->d_k7prb.p;
                            if (V <= 320) k7_bwd2<320, 3><<<nd, V, smem, st>>>(P); else k7_bwd2<512, 2><<<nd, V, smem, st>>>(P);
                        }
                        else k7_bwd<<<nd, V, smem, st>>>(P);
                        h->launches++;
                    }
                }
            }
            {                                                  // the arcs out of the start state (descriptors of step 0: cp = START)
                P.desc = B.d_desc.p + B.desc_off[0]; P.perm = B.d_perm.p + B.row_off[0];
                P.src = bt[0]; P.dst = nullptr; P.lat = nullptr; P.exp_t = nullptr; P.rescale = 0;
                const unsigned nd = (unsigned)(B.desc_off[1] - B.desc_off[0]);
                if (nd) { k7_bwd<<<nd, V, smem, st>>>(P); h->launches++; }
            }
        }
    } else if (kernel == 2) {
        K3Params P{};
        FastTablesD T{};
        T.cand_off = h->d_cand_off.p; T.slot_state = h->d_slot_state.p;
        T.frow = h->d_frow.p; T.fent = h->d_fent.p; T.brow = h->d_brow.p; T.bent = h->d_bent.p;
        T.n_sym = F.n_sym; T.n_states = F.n_states; T.n_arcs = L.n_arcs; T.n_slots = L.n_slots;
        T.start_state = F.start; T.start_final_tid = L.start_final_tid;
        P.T = T; P.W = EvalWeightsD{h->d_tw.p, h->d_sw.p, h->d_fw.p}; P.C = C; P.O = O;
        P.lattice = h->d_k3lat.p; P.lat_exp = h->d_k3exp.p; P.max_len = std::max(h->max_len, 1);
        if (mode == MODE_STRUCT) k3_fwdbwd<MODE_STRUCT><<<h->k3_grid, h->k3_block, h->k3_smem, st>>>(P);
        else k3_fwdbwd<MODE_EVAL><<<h->k3_grid, h->k3_block, h->k3_smem, st>>>(P);
        h->launches++;
    } else {
        GenericParams P{};
        P.G = GenericTablesD{h->d_emis_row.p, h->d_emis_tok_off.p, h->d_emis_tok.p, h->d_trans_row.p, h->d_trans_dst.p,
                             h->d_eps_order.p, F.n_states, F.n_trans(), F.start, F.end};
        P.ltw = h->d_ltw.p; P.lew = h->d_lew.p; P.C = C; P.O = O; P.scratch = h->d_gscratch.p; P.max_len = h->max_len;
        for (long long first = 0; first < C.n_order; first += h->g_batch) {
            P.first = first; P.count = std::min<long long>(h->g_batch, C.n_order - first);
            const int grid = (int)((P.count + 127) / 128);
            if (mode == MODE_STRUCT) kg_fwdbwd<MODE_STRUCT><<<grid, 128, 0, st>>>(P);
            else kg_fwdbwd<MODE_EVAL><<<grid, 128, 0, st>>>(P);
            h->launches++;
        }
    }
}

// CTAs that own a big DAG group wait for it before they take regular groups: few big groups (up to grid / 4 by default)
static int eval6_big_dedicate(const wfsa_dev* h)
{
    const int ded_div = getenv("WFSA_E6_DED_DIV") ? std::max(1, atoi(getenv("WFSA_E6_DED_DIV"))) : 4;
    return (h->kr_big_groups > 0 && h->kr_big_groups * ded_div <= h->seg_grid && !getenv("WFSA_E6_NO_DEDICATE")) ? 1 : 0;
}

// The whole evaluation of the segmented path in one launch (kernels_eval6.cuh).  All launch parameters are constant per
// parameter map: x, the scale of loglik and the epoch are read from device memory.
static void fill_eval6_params(wfsa_dev* h, Eval6Params& P)
{
    P = Eval6Params{};
    P.words = h->d_krwords.p; P.goff = h->d_krgoff.p; P.grows = h->d_krgrows.p; P.typeW = h->d_krW.p; P.lq = h->d_krlq.p;
    P.pwords = h->d_krpwords.p; P.pgoff = h->d_krpgoff.p;
    P.n_groups = h->kr_groups; P.n_big = h->kr_big_groups; P.cls = h->d_e6cls.p; P.n_cls = h->e6_ncls;
    // static share of the regular groups: 70 % measured best for the full corpus; none when CTAs are dedicated to their big
    // groups first (a CTA that starts late cannot give its static share away)
    P.static_pct = getenv("WFSA_E6_STATIC") ? std::min(100, std::max(0, atoi(getenv("WFSA_E6_STATIC")))) : 70;
    P.xs = h->d_seg_xs.p; P.xs_rows = (size_t)std::max<int64_t>(h->seg_max_big_rows, 1);
    P.arc_tp = h->d_arc_tp.p; P.x = h->d_x.p; P.n = h->n; P.n_arcs = h->larcs.n_arcs;
    P.direct_exp = (size_t)h->n > (size_t)h->seg_block * h->seg_slots ? 1 : 0;
    P.aw_g = h->d_seg_aw.p;
    P.const_acc = h->d_seg_const.p; P.acc = h->d_e6acc.p; P.replicas = h->replicas;
    P.fx_scale = std::ldexp(1.0, (int)h->fx_log2); P.inv_fx = std::ldexp(1.0, -(int)h->fx_log2);
    P.red = h->d_e6red.p; P.ctl = h->d_e6ctl.p;
    P.n_edges = h->n_edges; P.e_off = h->d_eoff.p; P.e_arc = h->d_earc.p; P.edge_tp = h->d_edge_tp.p; P.out = h->d_out.p;
    P.nranks = h->comm ? h->nranks : 1; P.rank = h->rank; P.pk_words = 2 + h->n_edges; P.ll_off = h->peer_ll_off;
    for (int r = 0; r < 8; ++r) P.peers[r] = (h->comm && r < h->nranks) ? h->peer_ptrs[r] : nullptr;
    P.stamps = h->d_e6stamps.p;
    P.debug = getenv("WFSA_E6_DEBUG") ? atoi(getenv("WFSA_E6_DEBUG")) : 0;
    P.pool_slots = std::max(h->seg_slots, kPathSlots); P.big_slots = h->e6_big_slots; P.big_rows = h->e6_big_rows;
    P.big_dedicate = eval6_big_dedicate(h);
    // dedicated CTAs: the shard is small (a few regular groups per warp): everything static among the free CTAs; one global
    // ticket counter for ~3.5 k groups costs ~3 ns per ticket in the L2, i.e. ~10 us of a ~14 us phase
    if (P.big_dedicate && !getenv("WFSA_E6_STATIC")) P.static_pct = 100;
}

static cudaError_t launch_eval6(wfsa_dev* h, cudaStream_t st, bool count = true, bool to_host = false, bool x_from_host = false)
{
    Eval6Params P;
    fill_eval6_params(h, P);
    if (to_host) { P.out = h->hm_out_dev; P.done_flag = h->hm_flag_dev; }
    if (x_from_host) { P.x_host = h->h_x_dev; P.x_w = h->d_x.p; }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(h->seg_grid); cfg.blockDim = dim3(h->seg_block); cfg.dynamicSmemBytes = h->e6_smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;             // all CTAs resident: the grid barrier and the exchange rely on it
    at[0].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = getenv("WFSA_E6_PLAIN_LAUNCH") ? 0 : 1;
    cudaError_t e;
    if (h->awg) e = cudaLaunchKernelEx(&cfg, k_eval6<512, true>, P);
    else if (h->seg_block == 512) e = cudaLaunchKernelEx(&cfg, k_eval6<512>, P);
    else if (h->seg_block == 384) e = cudaLaunchKernelEx(&cfg, k_eval6<384>, P);
    else if (h->seg_block == 256) e = cudaLaunchKernelEx(&cfg, k_eval6<256>, P);
    else e = cudaLaunchKernelEx(&cfg, k_eval6<128>, P);
    if (e == cudaSuccess && count) { h->launches++; h->e6_used = true; }
    return e;
}

// weights, then the dominant kernel(s) over the given string lists, then the arc -> edge fold.
// `clear` = false appends to the accumulators of a previous call (structural pass, second stage).
static int launch_pipeline(wfsa_dev* h, int mode, int kernel, const int32_t* d_order, int64_t n_order,
                           int kernel2, const int32_t* d_order2, int64_t n_order2, bool clear, bool fold)
{
    const HostFsa& F = h->fsa;
    cudaStream_t st = h->stream;
    const int unit = (mode == MODE_STRUCT) ? 1 : 0;
    // segmented path without overflow strings: one prep launch, KR, one fold(+all-reduce)+finish launch
    const bool lean6 = kernel == 6 && mode == MODE_EVAL && clear && fold && (kernel2 == 0 || !h->any_overflow);
    if (lean6 && h->e6_ok) {
        if (h->comm_failed) return set_err(h, WFSA_ERR_NCCL, "an earlier exchange over peer memory timed out: the ranks are out of step");
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (h->timing && h->timing_detail)
            if (const TimedSlot* s = h->kev.next(false)) { e0 = s->begin; e1 = s->end; }
        if (e0) cudaEventRecord(e0, st);
        {
            const cudaError_t le = launch_eval6(h, st);
            if (le != cudaSuccess) {
                int nb = -1;
                if (h->seg_block == 512) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_eval6<512>, h->seg_block, h->seg_smem);
                cudaFuncAttributes fa{};
                cudaFuncGetAttributes(&fa, k_eval6<512>);
                h->err = std::string("k_eval6 launch: ") + cudaGetErrorString(le) + " (grid " + std::to_string(h->seg_grid) + ", block " + std::to_string(h->seg_block) +
                         ", dynamic smem " + std::to_string(h->seg_smem) + ", static smem " + std::to_string(fa.sharedSizeBytes) + ", regs " + std::to_string(fa.numRegs) +
                         ", local " + std::to_string(fa.localSizeBytes) + ", max dyn smem " + std::to_string(fa.maxDynamicSharedSizeBytes) + ", occupancy " + std::to_string(nb) + " CTAs/SM)";
                cudaGetLastError();
                return WFSA_ERR_CUDA;
            }
        }
        if (e1) cudaEventRecord(e1, st);
        h->lean_now = true; h->lean_finished = true; h->ks_done = false;
        return WFSA_OK;
    }
    if (mode == MODE_EVAL) h->e6_used = false;
    if (clear) {
        CK(cudaMemsetAsync(h->d_red.p, 0, h->d_red.n * 8, st));
        if (h->fast.ok) CK(cudaMemsetAsync(h->d_acc.p, 0, h->d_acc.n * 8, st));
        const int n_slots = h->fast.ok ? h->fast.n_slots : 0;
        const int total = F.n_trans() + F.n_emis() + n_slots;
        if (total > 0) {
            k_weights<<<(total + 255) / 256, 256, 0, st>>>(F.n_trans(), F.n_emis(), n_slots, h->d_trans_tp.p, h->d_emis_tp.p,
                                                          h->d_slot_emis.p, h->d_slot_final.p, h->d_x.p, unit, h->d_tw.p,
                                                          h->d_sw.p, h->d_fw.p, h->d_ltw.p, h->d_lew.p);
            h->launches++;
        }
        if (h->fast.ok && h->fast.compact_ok && h->fast.n_arcs > 0) {
            k_arc_weights<<<(h->fast.n_arcs + 255) / 256, 256, 0, st>>>(h->fast.n_arcs, h->d_arc_tid.p, h->d_arc_eid.p, h->d_emis_tp.p,
                                                                        h->d_tw.p, h->d_x.p, unit, h->d_aw.p);
            h->launches++;
        }
        if (h->fast.ok) {
            k_state_final_weights<<<(F.n_states + 255) / 256, 256, 0, st>>>(F.n_states, h->d_state_final.p, h->d_tw.p, h->d_fws.p);
            h->launches++;
        }
        if (kernel == 6) {
            const int na = h->larcs.n_arcs;
            k_arc_weights_log<<<(na + 255) / 256, 256, 0, st>>>(na, h->d_seg_arc_tid.p, h->d_seg_arc_eid.p, h->d_trans_tp.p,
                                                              h->d_emis_tp.p, h->d_x.p, h->d_seg_aw.p, h->d_seg_logaw.p, h->d_seg_const.p,
                                                              std::ldexp(1.0, -(int)h->fx_log2), std::ldexp(1.0, (int)h->ll_log2),
                                                              h->d_llpart.p);
            h->llpart_n = (na + 255) / 256;
            h->launches++;
            // replica 0 starts from the constant part (bridge edges: posterior exactly 1), the others from 0
            CK(cudaMemcpyAsync(h->d_seg_acc.p, h->d_seg_const.p, (size_t)na * 8, cudaMemcpyDeviceToDevice, st));
            if (h->replicas > 1) CK(cudaMemsetAsync(h->d_seg_acc.p + na, 0, (size_t)na * (h->replicas - 1) * 8, st));
        }
    }
    EvalOutD O{};
    O.logq = h->d_logq.p; O.path_count = h->d_pathcnt.p; O.acc_global = h->d_acc.p; O.red = h->d_red.p;
    O.fx_scale = (mode == MODE_STRUCT) ? 1.0 : std::ldexp(1.0, (int)h->fx_log2);
    O.ll_scale = std::ldexp(1.0, (int)h->ll_log2);
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (h->timing && h->timing_detail && mode == MODE_EVAL)
        if (const TimedSlot* s = h->kev.next(true)) { e0 = s->begin; e1 = s->end; h->mid_now = s->mid; }
    if (e0) cudaEventRecord(e0, st);
    h->lean_now = false;
    launch_main(h, kernel, mode, CorpusD{h->d_tokens.p, h->d_offs.p, h->d_p.p, d_order, n_order}, O);
    if (kernel2) launch_main(h, kernel2, mode, CorpusD{h->d_tokens.p, h->d_offs.p, h->d_p.p, d_order2, n_order2}, O);
    if (e1) cudaEventRecord(e1, st);
    h->mid_now = nullptr;
    CK(cudaGetLastError());
    h->lean_finished = false;
    if (fold && kernel == 6) {
        const int na = h->larcs.n_arcs;
        k_arcs_to_edges<<<(na + 255) / 256, 256, 0, st>>>(na, 0, F.n_trans(), h->d_seg_acc.p, h->replicas, h->d_seg_arc_tid.p,
                                                         h->d_seg_arc_eid.p, nullptr, h->d_red.p + 2);
        h->launches++;
        CK(cudaGetLastError());
    }
    const bool fast_used = kernel == 6 ? (kernel2 == 1 || kernel2 == 2) && n_order2 > 0 : (kernel != 3);
    if (fold && h->fast.ok && fast_used) {
        const int total = h->fast.n_arcs + F.n_states;
        k_arcs_to_edges<<<(total + 255) / 256, 256, 0, st>>>(h->fast.n_arcs, F.n_states, F.n_trans(), h->d_acc.p, h->replicas,
                                                            h->d_arc_tid.p, h->d_arc_eid.p, h->d_state_final.p, h->d_red.p + 2);
        h->launches++;
        CK(cudaGetLastError());
    }
    return WFSA_OK;
}

extern "C" int wfsa_dev_structure(wfsa_dev* h, uint8_t* recognised, double* path_count, uint8_t* param_used)
{
    if (!h) return WFSA_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    // the structural pass reuses the string-order buffers of the evaluation: a parameter map set earlier is void after it
    // (wfsa_dev_eval returns WFSA_ERR_STATE until wfsa_dev_set_param_map is called again)
    h->n = -1; h->evaluated = false;
    CK(cudaMemcpyAsync(h->d_order.p, h->h_order_all.data(), (size_t)h->n_strings * 4, cudaMemcpyHostToDevice, h->stream));
    std::vector<double> pc((size_t)h->n_strings);
    h->h_overflow.assign((size_t)h->n_strings, 0);
    h->n_overflow = 0;
    if (h->skernel == 4) {
        // stage 1: thread-per-string over everything; strings whose active set exceeds K come back as -1
        int rc = upload_transposed_tokens(h, h->h_order_all);
        if (rc != WFSA_OK) return rc;
        rc = launch_pipeline(h, MODE_STRUCT, 4, h->d_order.p, h->n_strings, 0, nullptr, 0, true, false);
        if (rc != WFSA_OK) return rc;
        if (h->n_strings) CK(cudaMemcpyAsync(pc.data(), h->d_pathcnt.p, (size_t)h->n_strings * 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        std::vector<int32_t> over;
        for (int32_t s : h->h_order_all) if (pc[s] < 0.0) { over.push_back(s); h->h_overflow[s] = 1; }
        h->n_overflow = (int64_t)over.size();
        if (!over.empty()) CK(cudaMemcpyAsync(h->d_order_w.p, over.data(), over.size() * 4, cudaMemcpyHostToDevice, h->stream));
        // stage 2: the overflow strings on the warp / CTA kernel, then fold everything
        rc = launch_pipeline(h, MODE_STRUCT, h->secondary, h->d_order_w.p, h->n_overflow, 0, nullptr, 0, false, true);
        if (rc != WFSA_OK) return rc;
    } else {
        int rc = launch_pipeline(h, MODE_STRUCT, h->skernel, h->d_order.p, h->n_strings, 0, nullptr, 0, true, true);
        if (rc != WFSA_OK) return rc;
    }
    // used flags are per-edge instance counts; combine across ranks before thresholding
    int rc = nccl_allreduce(h, h->d_red.p, h->d_red.n, ncclUint64, ncclSum);
    if (rc != WFSA_OK) return rc;
    CK(cudaMemsetAsync(h->d_used.p, 0, h->d_used.n, h->stream));
    if (h->n_edges) {
        k_finish_struct<<<(h->n_edges + 255) / 256, 256, 0, h->stream>>>(h->n_edges, h->d_red.p, h->d_edge_raw.p, h->d_used.p);
        h->launches++;
    }
    if (h->n_strings) CK(cudaMemcpyAsync(pc.data(), h->d_pathcnt.p, (size_t)h->n_strings * 8, cudaMemcpyDeviceToHost, h->stream));
    std::vector<uint8_t> used((size_t)h->fsa.n_raw);
    if (h->fsa.n_raw) CK(cudaMemcpyAsync(used.data(), h->d_used.p, (size_t)h->fsa.n_raw, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    h->h_recognised.resize((size_t)h->n_strings);
    for (int64_t s = 0; s < h->n_strings; ++s) {
        h->h_recognised[s] = pc[s] > 0.0 ? 1 : 0;
        if (recognised) recognised[s] = h->h_recognised[s];
        if (path_count) path_count[s] = pc[s];
    }
    if (param_used) std::copy(used.begin(), used.end(), param_used);
    h->structure_done = true;
    return WFSA_OK;
}

static int setup_peer_allreduce(wfsa_dev* h);

extern "C" int wfsa_dev_set_param_map(wfsa_dev* h, const int32_t* trimmed, int32_t n, const uint8_t* recognised)
{
    if (!h || n < 0 || (!trimmed && h->fsa.n_raw > 0)) return set_err(h, WFSA_ERR_INVALID, "set_param_map: bad arguments");
    CK(cudaSetDevice(h->device));
    const HostFsa& F = h->fsa;
    std::vector<char> seen((size_t)n, 0);
    for (int i = 0; i < F.n_raw; ++i) {
        const int t = trimmed[i];
        if (t < -2 || t >= n) return set_err(h, WFSA_ERR_INVALID, "set_param_map: trimmed index out of range");
        if (t >= 0) { if (seen[t]) return set_err(h, WFSA_ERR_INVALID, "set_param_map: trimmed index used twice"); seen[t] = 1; }
    }
    for (int i = 0; i < n; ++i) if (!seen[i]) return set_err(h, WFSA_ERR_INVALID, "set_param_map: a trimmed index has no parameter");
    std::vector<int32_t> ttp(F.n_trans()), etp(F.n_emis());
    for (int t = 0; t < F.n_trans(); ++t) ttp[t] = F.trans_param[t] < 0 ? -1 : trimmed[F.trans_param[t]];
    for (int e = 0; e < F.n_emis(); ++e) etp[e] = F.emis_param[e] < 0 ? -1 : trimmed[F.emis_param[e]];
    std::vector<int32_t> edge_tp(ttp);
    edge_tp.insert(edge_tp.end(), etp.begin(), etp.end());
    // pinned (-1) and unused (-2) edges produce no gradient entry
    if (!ttp.empty()) CK(cudaMemcpyAsync(h->d_trans_tp.p, ttp.data(), ttp.size() * 4, cudaMemcpyHostToDevice, h->stream));
    if (!etp.empty()) CK(cudaMemcpyAsync(h->d_emis_tp.p, etp.data(), etp.size() * 4, cudaMemcpyHostToDevice, h->stream));
    if (!edge_tp.empty()) CK(cudaMemcpyAsync(h->d_edge_tp.p, edge_tp.data(), edge_tp.size() * 4, cudaMemcpyHostToDevice, h->stream));
    // strings that take part: recognised ones, longest first
    if (h->kernel == 4 && !h->structure_done)
        return set_err(h, WFSA_ERR_STATE, "set_param_map: the thread-per-string kernel needs wfsa_dev_structure first");
    std::vector<int32_t> order, order_w;
    order.reserve((size_t)h->n_strings);
    const uint8_t* rec = recognised ? recognised : (h->structure_done ? h->h_recognised.data() : nullptr);
    int64_t tokens = 0; int max_len = 0;
    for (int32_t s : h->h_order_all)
        if (!rec || rec[s]) {
            if (h->kernel == 4 && h->h_overflow[s]) order_w.push_back(s); else order.push_back(s);
            const int64_t len = h->h_offs[s + 1] - h->h_offs[s];
            tokens += len; max_len = std::max<int>(max_len, (int)len);
        }
    h->n_active = (int64_t)order.size(); h->n_active_w = (int64_t)order_w.size(); h->n_active_tokens = tokens;
    // (the segmented path reads the list of all its strings only in an rmin sweep without region-type blocks)
    if (!order.empty()) CK(cudaMemcpyAsync(h->d_order.p, order.data(), order.size() * 4, cudaMemcpyHostToDevice, h->stream));
    if (h->kernel != 6 && !order_w.empty()) CK(cudaMemcpyAsync(h->d_order_w.p, order_w.data(), order_w.size() * 4, cudaMemcpyHostToDevice, h->stream));
    if (h->kernel == 4) { const int rc = upload_transposed_tokens(h, order); if (rc != WFSA_OK) return rc; }
    // every logq defaults to -inf (unrecognised strings are never touched by an evaluation)
    {
        std::vector<double> minf((size_t)h->n_strings, -INFINITY);
        if (h->n_strings) CK(cudaMemcpyAsync(h->d_logq.p, minf.data(), minf.size() * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    // fixed-point scale: an accumulator is bounded by sum_s p_s * (steps of a path) <= max steps
    long long bound = ((long long)h->max_len + 2) * (h->gen.n_eps_states + 1);
    if (h->comm) {
        long long* d = reinterpret_cast<long long*>(h->d_red.p);
        CK(cudaMemcpyAsync(d, &bound, 8, cudaMemcpyHostToDevice, h->stream));
        int rc = nccl_allreduce(h, d, 1, ncclInt64, ncclMax);
        if (rc != WFSA_OK) return rc;
        CK(cudaMemcpyAsync(&bound, d, 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    h->step_bound = bound;
    int bits = 1;
    while ((1ll << bits) <= bound && bits < 40) ++bits;
    h->fx_log2 = 62 - bits;
    if (h->kernel == 6) {
        // compile every participating string into bridges + region types (structure is independent of x)
        const LatticeArcs& A = h->larcs;
        std::vector<uint8_t> alive((size_t)A.n_arcs);
        for (int a = 0; a < A.n_arcs; ++a)
            alive[a] = ttp[A.arc_tid[a]] != -2 && (A.arc_eid[a] < 0 || etp[A.arc_eid[a]] != -2);
        if (h->ks_thread.joinable()) h->ks_thread.join();       // the layout job of a previous parameter map
        h->ks_job.reset(); h->ks_sc.reset(); h->ks_failed = false;
        SegmentedCorpus sc;
        h->ks_job = compile_corpus_regions(h->fsa, A, alive.data(), h->h_tokens.data(), h->h_offs.data(), h->h_p.data(), order, h->seg_slots,
                                           std::ldexp(1.0, (int)h->fx_log2), sc);
        h->ks_sc.reset(new SegmentedCorpus());
        {
            std::shared_ptr<SegmentedStringsJob> job = h->ks_job;
            SegmentedCorpus* dst = h->ks_sc.get();
            bool* failed = &h->ks_failed;
            h->ks_thread = std::thread([job, dst, failed] {
                try { job->run(*dst); } catch (...) { *failed = true; }
            });
        }
        order_w = sc.overflow;
        order_w.insert(order_w.end(), sc.rejected.begin(), sc.rejected.end());
        h->n_active = (int64_t)order.size() - (int64_t)order_w.size(); h->n_active_w = (int64_t)order_w.size();
        h->kr_big_groups = 0;
        for (int32_t r : sc.rgrows) if (!(r & 0x10000) && r > kSegSmallMax) h->kr_big_groups++;      // big DAG classes sort first
        h->kr_groups = (int64_t)sc.rgrows.size(); h->ks_groups = 0;                                 // KS: set by ensure_ks()
        h->seg_types = sc.n_types; h->seg_instances = sc.n_region_instances; h->seg_region_edges = sc.n_region_edges;
        h->seg_type_edges = sc.n_type_edges; h->seg_bridges = sc.n_bridge; h->seg_host_ms = sc.host_ms;
        h->seg_words = (int64_t)sc.rwords.size();               // + the per-string words once they are built
        h->seg_max_big_rows = sc.max_big_rows;
        CK(h->d_krwords.upload(sc.rwords, h->stream)); CK(h->d_krgoff.upload(sc.rgoff, h->stream));
        CK(h->d_krgrows.upload(sc.rgrows, h->stream)); CK(h->d_krW.upload(sc.typeW, h->stream));
        CK(h->d_krpwords.upload(sc.pwords, h->stream)); CK(h->d_krpgoff.upload(sc.pgoff, h->stream));
        CK(h->d_krlq.alloc((size_t)h->kr_groups * 32 + 1));
        CK(cudaMemsetAsync(h->d_krlq.p, 0, h->d_krlq.n * 8, h->stream));
        std::vector<unsigned long long> cacc(sc.const_acc.begin(), sc.const_acc.end());
        CK(cudaMemcpyAsync(h->d_seg_const.p, cacc.data(), cacc.size() * 8, cudaMemcpyHostToDevice, h->stream));
        if (!order_w.empty()) CK(cudaMemcpyAsync(h->d_order_w.p, order_w.data(), order_w.size() * 4, cudaMemcpyHostToDevice, h->stream));
        {   // single-launch evaluation (k_eval6): trimmed parameters per arc, class table of the regular groups, two accumulator buffers
            std::vector<int2> atp((size_t)A.n_arcs);
            for (int a = 0; a < A.n_arcs; ++a) atp[a] = make_int2(ttp[A.arc_tid[a]], A.arc_eid[a] < 0 ? -1 : etp[A.arc_eid[a]]);
            CK(h->d_arc_tp.upload(atp, h->stream));
            std::vector<Eval6Cls> cls;
            bool regular = true;
            for (int64_t g = h->kr_big_groups; g < h->kr_groups; ++g) {
                const int code = sc.rgrows[g];
                const int nrows = (code & 0x10000) ? ((code >> 8) & 0xff) * (code & 0xff) : code;
                if (sc.rgoff[g + 1] - sc.rgoff[g] != (int64_t)nrows * 32) regular = false;
                if (cls.empty() || cls.back().code != code) cls.push_back(Eval6Cls{(int)g, code, (long long)sc.rgoff[g]});
            }
            h->e6_ncls = (int)cls.size();
            h->e6_ok = regular && cls.size() <= (size_t)kE6MaxCls && (h->seg_block == 512 || h->seg_block == 384 || h->seg_block == 256 || h->seg_block == 128) && h->kr_groups < (int64_t)0x7fffffff && !getenv("WFSA_EVAL6_OFF");
            if (cls.empty()) cls.push_back(Eval6Cls{0, 4, 0});
            {   // staging areas for the big DAG groups in the shared memory the tables and the pool leave free
                const size_t room = (size_t)(227 * 1024 - 8192) - h->seg_smem;
                int rows = (int)std::max<int64_t>(sc.max_big_rows, 0);
                if (rows > 0 && (size_t)rows * 384 > room) rows = (int)(room / 384 / 16) * 16;      // larger groups stay in HBM
                h->e6_big_rows = rows;
                h->e6_big_slots = rows > 0 ? (int)std::min<size_t>(4, room / ((size_t)rows * 384)) : 0;
                if (getenv("WFSA_E6_NO_STAGING")) h->e6_big_slots = 0;
                h->e6_smem = h->seg_smem + (size_t)h->e6_big_slots * h->e6_big_rows * 384;
            }
            CK(h->d_e6cls.upload(cls, h->stream));
            const size_t cells = (size_t)A.n_arcs * h->replicas;
            CK(h->d_e6acc.alloc(2 * cells));
            CK(cudaMemsetAsync(h->d_e6acc.p, 0, 2 * cells * 8, h->stream));
            for (int b = 0; b < 2; ++b) CK(cudaMemcpyAsync(h->d_e6acc.p + b * cells, cacc.data(), cacc.size() * 8, cudaMemcpyHostToDevice, h->stream));
            CK(cudaMemsetAsync(h->d_e6red.p, 0, 16, h->stream));
            CK(cudaStreamSynchronize(h->stream));
        }
        const size_t warps = (size_t)h->seg_grid * h->seg_block / 32;
        const size_t need = warps * (size_t)std::max<int64_t>(sc.max_big_rows, 1) * 32;
        if (h->d_seg_xs.n < need) {
            const cudaError_t e = h->d_seg_xs.alloc(need);
            if (e != cudaSuccess) return set_err(h, WFSA_ERR_NOMEM, "segmented kernel: cannot allocate the per-warp x stacks");
        }
        CK(cudaStreamSynchronize(h->stream));
        // the region types stay on the host as well: wfsa_dev_hessian derives its path blocks from them
        h->hrw = std::move(sc.rwords); h->hrgoff = std::move(sc.rgoff); h->hrgrows = std::move(sc.rgrows); h->hrW = std::move(sc.typeW);
        h->h_seg_overflow = std::move(sc.overflow);
        h->h_ttp = ttp; h->h_etp = etp;
        if (!h->hb_user) h->hb_blocks = -1;
        h->hb_from_types = false; h->hb_types_failed = false;
    }
    if (h->kernel == 7) {
        // K7: batches of strings (longest first) whose alpha lattices fit the device memory; per batch and position the
        // strings grouped by the symbol pair (c_{t-1}, c_t), in chunks of kK7Chunk
        const auto t_begin = std::chrono::steady_clock::now();
        const int A = F.n_sym, V = h->k7_V;
        std::vector<int32_t> good;
        for (int32_t s : order) {
            bool ok = true;
            for (int64_t i = h->h_offs[s]; i < h->h_offs[s + 1]; ++i) if ((unsigned)h->h_tokens[i] >= (unsigned)A) { ok = false; break; }
            if (h->h_offs[s + 1] == h->h_offs[s]) ok = false;                    // the empty string: the CTA-per-string kernel knows how
            (ok ? good : order_w).push_back(s);
        }
        h->n_active = (int64_t)good.size(); h->n_active_w = (int64_t)order_w.size();
        if (!order_w.empty()) CK(cudaMemcpyAsync(h->d_order_w.p, order_w.data(), order_w.size() * 4, cudaMemcpyHostToDevice, h->stream));
        // the batches and the lattice of a previous map go first: the budget below counts their memory as free
        h->k7.clear();
        h->d_k7lat.release(); h->d_k7bt.release(); h->d_k7exp.release(); h->d_k7scale.release(); h->d_k7EQ.release(); h->d_k7F.release();
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        // per lattice row: V doubles + one exponent + one permutation entry; keep a third of the free memory for everything else
        size_t budget_rows = (size_t)((double)free_b * 0.6) / ((size_t)V * 8 + 8);
        if (getenv("WFSA_K7_ROWS")) budget_rows = (size_t)atoll(getenv("WFSA_K7_ROWS"));
        size_t i0 = 0;
        size_t max_rows = 0, max_nb = 0;
        while (i0 < good.size()) {
            size_t rows = 0, i1 = i0;
            while (i1 < good.size()) {
                const size_t len = (size_t)(h->h_offs[good[i1] + 1] - h->h_offs[good[i1]]);
                if (i1 > i0 && rows + len > budget_rows) break;
                rows += len; ++i1;
            }
            h->k7.emplace_back();
            wfsa_dev::K7Batch& B = h->k7.back();
            B.NB = (int)(i1 - i0);
            B.Tmax = (int)(h->h_offs[good[i0] + 1] - h->h_offs[good[i0]]);
            B.n_t.assign((size_t)B.Tmax + 2, 0);
            for (size_t i = i0; i < i1; ++i) B.n_t[(size_t)(h->h_offs[good[i] + 1] - h->h_offs[good[i]]) - 1]++;     // strings whose last position is t
            for (int t = B.Tmax - 1; t >= 0; --t) B.n_t[t] += B.n_t[t + 1];                                      // -> strings longer than t
            B.row_off.assign((size_t)B.Tmax + 1, 0);
            for (int t = 0; t < B.Tmax; ++t) B.row_off[t + 1] = B.row_off[t] + (size_t)B.n_t[t];
            std::vector<int32_t> perm(rows), sid((size_t)B.NB), last((size_t)B.NB);
            for (int r = 0; r < B.NB; ++r) { sid[r] = good[i0 + r]; last[r] = h->h_tokens[h->h_offs[sid[r] + 1] - 1]; }
            // counting sort of the strings of every step by their pair key, steps dealt out to the host threads
            std::vector<std::vector<K7Desc>> step_desc((size_t)B.Tmax);
            unsigned hw = std::thread::hardware_concurrency();
            const int NT = (int)std::max(1u, std::min(hw ? hw : 4u, 32u));
            auto work = [&](int tid) {
                std::vector<int32_t> cnt((size_t)(A + 1) * A + 1);
                for (int t = tid; t < B.Tmax; t += NT) {
                    std::fill(cnt.begin(), cnt.end(), 0);
                    const int n = B.n_t[t];
                    auto key_of = [&](int r) {
                        const int64_t o = h->h_offs[sid[r]];
                        return (t ? h->h_tokens[o + t - 1] : A) * A + h->h_tokens[o + t];
                    };
                    for (int r = 0; r < n; ++r) cnt[(size_t)key_of(r) + 1]++;
                    std::vector<K7Desc>& D = step_desc[t];
                    int run = 0;
                    for (size_t k = 0; k + 1 < cnt.size(); ++k) {
                        const int c = cnt[k + 1];
                        if (c > 0) {
                            const int cp = (int)(k / A), cc = (int)(k % A);
                            const int kf = h->k7_planes ? h->k7_kf[k] : 0, kb = h->k7_planes ? h->k7_kb[k] : 0;
                            for (int b = 0; b < c; b += kK7Chunk)
                                D.push_back(K7Desc{cp, cc, run + b, std::min(kK7Chunk, c - b), (int)h->fast.cand_off[cc], (int)h->fast.cand_off[cp], kf, kb});
                        }
                        cnt[k + 1] = run; run += c;                                       // becomes the write cursor of key k
                    }
                    int32_t* out = perm.data() + B.row_off[t];
                    for (int r = 0; r < n; ++r) out[cnt[(size_t)key_of(r) + 1]++] = r;
                }
            };
            {
                std::vector<std::thread> th;
                for (int k = 1; k < NT; ++k) th.emplace_back(work, k);
                work(0);
                for (auto& x : th) x.join();
            }
            B.desc_off.assign((size_t)B.Tmax + 1, 0);
            for (int t = 0; t < B.Tmax; ++t) B.desc_off[t + 1] = B.desc_off[t] + step_desc[t].size();
            std::vector<K7Desc> desc(B.desc_off[B.Tmax]);
            for (int t = 0; t < B.Tmax; ++t) std::copy(step_desc[t].begin(), step_desc[t].end(), desc.begin() + B.desc_off[t]);
            CK(B.d_desc.upload(desc, h->stream)); CK(B.d_perm.upload(perm, h->stream));
            CK(B.d_sid.upload(sid, h->stream)); CK(B.d_last.upload(last, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            max_rows = std::max(max_rows, rows); max_nb = std::max(max_nb, (size_t)B.NB);
            i0 = i1;
        }
        h->k7_rows = max_rows; h->k7_nb = max_nb;
        if (max_rows) {
            if (h->d_k7lat.alloc(max_rows * (size_t)V) != cudaSuccess || h->d_k7exp.alloc(max_rows) != cudaSuccess ||
                h->d_k7bt.alloc(2 * max_nb * (size_t)V) != cudaSuccess || h->d_k7scale.alloc(max_nb) != cudaSuccess ||
                h->d_k7EQ.alloc(max_nb) != cudaSuccess || h->d_k7F.alloc(max_nb) != cudaSuccess) {
                cudaGetLastError();
                return set_err(h, WFSA_ERR_NOMEM, "batched kernel: cannot allocate the alpha lattice of a batch");
            }
        }
        h->k7_host_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    }
    if (h->n != n) {
        CK(h->h_out.alloc((size_t)n + 3));                       // [loglik, non-finite terms, grad[n], epoch of a timed-out exchange]
        CK(h->h_x.alloc((size_t)n + 1, cudaHostAllocMapped));    // [x[n], log2 of the fixed-point scale of loglik]
        h->h_x_dev = nullptr;
        if (cudaHostGetDevicePointer(&h->h_x_dev, h->h_x.p, 0) != cudaSuccess) { cudaGetLastError(); h->h_x_dev = nullptr; }
        CK(h->d_x.alloc((size_t)n + 1));
        CK(h->d_out.alloc((size_t)n + 3));
    }
    CK(cudaMemsetAsync(h->d_out.p, 0, h->d_out.n * 8, h->stream));
    h->e6_exec.reset(); h->e6_graph.reset();
    h->e6_graph_tried = false;
    h->n = n;
    h->evaluated = false;
    CK(cudaStreamSynchronize(h->stream));
    h->any_overflow = h->n_active_w > 0;
    if (h->comm) {
        // every rank must take the same route through an evaluation (one launch with the exchange inside, or kernels +
        // ncclAllReduce): agree on "some rank has strings for the secondary kernel" and "some rank cannot run k_eval6"
        long long flags[2] = {h->any_overflow ? 1 : 0, (h->kernel == 6 && !h->e6_ok) ? 1 : 0};
        long long* d = reinterpret_cast<long long*>(h->d_red.p);
        CK(cudaMemcpyAsync(d, flags, 16, cudaMemcpyHostToDevice, h->stream));
        int rc = nccl_allreduce(h, d, 2, ncclInt64, ncclMax);
        if (rc != WFSA_OK) return rc;
        CK(cudaMemcpyAsync(flags, d, 16, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        h->any_overflow = flags[0] != 0;
        if (flags[1]) h->e6_ok = false;
        rc = setup_peer_allreduce(h);
        if (rc != WFSA_OK) return rc;
        if (!h->peer_ok) h->e6_ok = false;                   // the exchange of k_eval6 goes through peer memory
    }
    return WFSA_OK;
}

// x into the pinned staging buffer, followed by log2 of the fixed-point scale of loglik (k_eval6 reads it from there)
static int stage_x(wfsa_dev* h, const double* x)
{
    if (!h || (!x && h->n > 0)) return set_err(h, WFSA_ERR_INVALID, "upload_x: bad arguments");
    if (h->n < 0) return set_err(h, WFSA_ERR_STATE, "upload_x before set_param_map");
    // the staging buffer is reused by every call: wait for the copy of the previous one before overwriting it
    if (h->x_in_flight) { CK(cudaEventSynchronize(h->ev_x)); h->x_in_flight = false; }
    // fixed-point scale of loglik: |sum_s p_s log q_s| <= max steps * (2 max|x| + log(fan-out))
    // (one pass the compiler can vectorise: max of |x| with NaN mapped to +inf, so `finite` falls out of the maximum)
    double mx = 0.0;
    {
        const int n = h->n;
        double* __restrict__ dst = h->h_x.p;
        double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0;
        int i = 0;
        for (; i + 4 <= n; i += 4) {
            const double a = x[i], b = x[i + 1], c = x[i + 2], d = x[i + 3];
            dst[i] = a; dst[i + 1] = b; dst[i + 2] = c; dst[i + 3] = d;
            const double fa = a == a ? std::fabs(a) : HUGE_VAL, fb = b == b ? std::fabs(b) : HUGE_VAL;
            const double fc = c == c ? std::fabs(c) : HUGE_VAL, fd = d == d ? std::fabs(d) : HUGE_VAL;
            m0 = fa > m0 ? fa : m0; m1 = fb > m1 ? fb : m1; m2 = fc > m2 ? fc : m2; m3 = fd > m3 ? fd : m3;
        }
        for (; i < n; ++i) { const double a = x[i]; dst[i] = a; const double fa = a == a ? std::fabs(a) : HUGE_VAL; m0 = fa > m0 ? fa : m0; }
        mx = std::max(std::max(m0, m1), std::max(m2, m3));
    }
    const bool finite = mx < HUGE_VAL;
    if (!finite) {                                             // the largest finite |x| sets the scale, as before
        mx = 0.0;
        for (int i = 0; i < h->n; ++i) if (std::isfinite(x[i])) mx = std::max(mx, std::fabs(x[i]));
    }
    const double B = (double)h->step_bound * (2.0 * mx + std::log((double)h->n_edges + 2.0)) + 1.0;
    int bits = 1;
    while (std::ldexp(1.0, bits) <= B && bits < 40) ++bits;
    h->ll_log2 = finite ? 62 - bits : 22;
    h->h_x.p[h->n] = h->ll_log2;
    return WFSA_OK;
}

extern "C" int wfsa_dev_upload_x(wfsa_dev* h, const double* x)
{
    const int rc = stage_x(h, x);
    if (rc != WFSA_OK) return rc;
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(h->d_x.p, h->h_x.p, ((size_t)h->n + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    if (!h->ev_x) CK(cudaEventCreateWithFlags(&h->ev_x.raw, cudaEventDisableTiming));
    CK(cudaEventRecord(h->ev_x, h->stream));
    h->x_in_flight = true;
    return WFSA_OK;
}

// Allocates this rank's peer buffer, exchanges the IPC handles through one NCCL all-reduce (every rank fills its own
// slot of a zeroed table) and maps the peers.  Collective: called by every rank at the same point (set_param_map).
// Any failure leaves peer_ok = false on ALL ranks (the outcome is all-reduced), and NCCL stays in charge.
static int setup_peer_allreduce(wfsa_dev* h)
{
    h->peer_ok = false;
    if (!h->comm || h->nranks > 8 || getenv("WFSA_NO_PEER")) return WFSA_OK;
    const int words = (int)h->d_red.n;
    if (h->peer_local.p && h->peer_words == words) { h->peer_ok = true; return WFSA_OK; }
    if (h->peer_local.p) return WFSA_OK;                     // sized for another parameter map: keep NCCL (rare)
    // [packets of k_eval6: 2 parities x nranks senders x words x 2][words of k_peer_barrier: 2 x nranks]
    h->peer_ll_off = 0;
    h->peer_bar_off = h->peer_ll_off + (size_t)4 * h->nranks * words;       // then the words of k_peer_barrier: 2 x nranks
    const size_t total = h->peer_bar_off + (size_t)2 * h->nranks;
    unsigned long long ok = 1;
    cudaIpcMemHandle_t mine;
    std::memset(&mine, 0, sizeof(mine));
    if (h->peer_local.alloc(total) != cudaSuccess) ok = 0;
    if (ok && cudaMemset(h->peer_local.p, 0, total * 8) != cudaSuccess) ok = 0;
    if (ok && cudaIpcGetMemHandle(&mine, h->peer_local.p) != cudaSuccess) ok = 0;
    cudaGetLastError();
    // table: per rank 8 words of handle + 1 word "ok"
    const int per = (int)(sizeof(cudaIpcMemHandle_t) / 8) + 1;
    std::vector<unsigned long long> tab((size_t)h->nranks * per, 0ull);
    std::memcpy(&tab[(size_t)h->rank * per], &mine, sizeof(mine));
    tab[(size_t)h->rank * per + per - 1] = ok;
    DevBuf<unsigned long long> d_tab;
    CK(d_tab.upload(tab, h->stream));
    int rc = nccl_allreduce(h, d_tab.p, tab.size(), ncclUint64, ncclSum);
    if (rc != WFSA_OK) return rc;
    CK(cudaMemcpyAsync(tab.data(), d_tab.p, tab.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    unsigned long long all_ok = 1;
    for (int r = 0; r < h->nranks; ++r) all_ok &= tab[(size_t)r * per + per - 1];
    unsigned long long mapped = all_ok;
    if (all_ok)
        for (int r = 0; r < h->nranks; ++r) {
            if (r == h->rank) { h->peer_ptrs[r] = h->peer_local.p; continue; }
            cudaIpcMemHandle_t hd;
            std::memcpy(&hd, &tab[(size_t)r * per], sizeof(hd));
            void* ptr = nullptr;
            if (cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { mapped = 0; cudaGetLastError(); break; }
            h->peer_ptrs[r] = (unsigned long long*)ptr;
        }
    // every rank must take the same route
    unsigned long long* d_flag = reinterpret_cast<unsigned long long*>(h->d_red.p);
    unsigned long long bad = mapped ? 0 : 1;
    CK(cudaMemcpyAsync(d_flag, &bad, 8, cudaMemcpyHostToDevice, h->stream));
    rc = nccl_allreduce(h, d_flag, 1, ncclUint64, ncclSum);
    if (rc != WFSA_OK) return rc;
    CK(cudaMemcpyAsync(&bad, d_flag, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->peer_words = words;
    h->peer_bar_epoch = 0;
    h->peer_ok = bad == 0;
    return WFSA_OK;
}

static int eval_launch_body(wfsa_dev* h);

extern "C" int wfsa_dev_eval_launch(wfsa_dev* h)
{
    if (!h) return WFSA_ERR_INVALID;
    if (h->n < 0) return set_err(h, WFSA_ERR_STATE, "eval before set_param_map");
    CK(cudaSetDevice(h->device));
    cudaEvent_t s1 = nullptr;
    if (h->timing)                                 // one event pair around the whole evaluation (weights, kernels, fold, collective)
        if (const TimedSlot* s = h->sev.next(false)) { cudaEventRecord(s->begin, h->stream); s1 = s->end; }
    h->out_on_host = false;
    const int rc = eval_launch_body(h);
    if (s1) cudaEventRecord(s1, h->stream);
    if (rc == WFSA_OK) h->evaluated = true;
    return rc;
}

static int eval_launch_body(wfsa_dev* h)
{
    int rc = launch_pipeline(h, MODE_EVAL, h->kernel, h->d_order.p, h->n_active,
                             h->kernel >= 4 ? h->secondary : 0, h->d_order_w.p, h->n_active_w, true, true);
    if (rc != WFSA_OK) return rc;
    if (h->lean_finished) return WFSA_OK;          // k_fold_finish6 already wrote [loglik, bad, grad]
    rc = nccl_allreduce(h, h->d_red.p, h->d_red.n, ncclUint64, ncclSum);
    if (rc != WFSA_OK) return rc;
    CK(cudaMemsetAsync(h->d_out.p, 0, h->d_out.n * 8, h->stream));
    const int total = std::max(h->n_edges, 1);
    k_finish_eval<<<(total + 255) / 256, 256, 0, h->stream>>>(h->n_edges, h->n, h->d_red.p, h->d_edge_tp.p,
                                                             std::ldexp(1.0, -(int)h->fx_log2), std::ldexp(1.0, -(int)h->ll_log2), h->d_out.p);
    h->launches++;
    CK(cudaGetLastError());
    return WFSA_OK;
}

extern "C" int wfsa_dev_sync(wfsa_dev* h)
{
    if (!h) return WFSA_ERR_INVALID;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    return WFSA_OK;
}

// Waits for the per-string layout job of the current parameter map (if any) and uploads its arrays.
static int ensure_ks(wfsa_dev* h)
{
    if (!h->ks_sc) return WFSA_OK;
    CK(cudaSetDevice(h->device));
    if (h->ks_thread.joinable()) h->ks_thread.join();
    std::unique_ptr<SegmentedCorpus> sc = std::move(h->ks_sc);
    h->ks_job.reset();
    if (h->ks_failed) return set_err(h, WFSA_ERR_NOMEM, "segmented path: building the per-string layout failed");
    CK(h->d_kswords.upload(sc->swords, h->stream)); CK(h->d_ksgoff.upload(sc->sgoff, h->stream));
    CK(h->d_ksgref.upload(sc->sgref, h->stream)); CK(h->d_kssid.upload(sc->ksid, h->stream));
    CK(h->d_ksp.upload(sc->kp, h->stream));
    CK(h->d_kslogq.alloc(std::max<size_t>(sc->kp.size(), 1)));
    CK(cudaStreamSynchronize(h->stream));                        // the host vectors go away with sc
    h->ks_groups = (int64_t)sc->sgoff.size() - 1;               // KS counts super-groups
    h->seg_words += (int64_t)sc->swords.size();
    h->seg_host_ms += sc->host_ms;
    return WFSA_OK;
}

// the results of the evaluation are in h_out: error checks, then copies into the caller's buffers
static int finish_fetch(wfsa_dev* h, double* loglik, double* grad, const double* src = nullptr)
{
    if (src) {                                                 // results in mapped memory: one pass fills the caller's buffers and h_out
        h->h_out.p[0] = src[0]; h->h_out.p[1] = src[1]; h->h_out.p[h->n + 2] = src[h->n + 2];
        double* __restrict__ keep = h->h_out.p + 2;
        const double* __restrict__ g = src + 2;
        if (grad) for (int i = 0; i < h->n; ++i) { const double v = g[i]; keep[i] = v; grad[i] = v; }
        else std::memcpy(keep, g, (size_t)h->n * 8);
        grad = nullptr;
    }
    if (h->comm && (std::isnan(h->h_out.p[1]) || h->h_out.p[h->n + 2] != 0.0)) {
        // the ranks no longer agree on the epoch of the exchange: later evaluations of this handle fail as well
        h->comm_failed = true;
        return set_err(h, WFSA_ERR_NCCL, "all-reduce over peer memory: a rank did not deliver its share within the time limit");
    }
    if (loglik) *loglik = h->h_out.p[0];
    if (grad) std::memcpy(grad, h->h_out.p + 2, (size_t)h->n * 8);
    return WFSA_OK;
}

extern "C" int wfsa_dev_eval_fetch(wfsa_dev* h, double* loglik, double* logq, double* grad)
{
    if (!h) return WFSA_ERR_INVALID;
    if (h->n < 0) return set_err(h, WFSA_ERR_STATE, "fetch before set_param_map");
    if (!h->evaluated) return set_err(h, WFSA_ERR_STATE, "fetch before an evaluation was launched for this parameter map");
    if (!h->out_on_host) CK(cudaMemcpyAsync(h->h_out.p, h->d_out.p, ((size_t)h->n + 3) * 8, cudaMemcpyDeviceToHost, h->stream));
    if (logq && h->kernel == 6) { const int rc = ensure_ks(h); if (rc != WFSA_OK) return rc; }
    if (logq && h->kernel == 6 && h->ks_groups > 0) {
        if (!h->ks_done) {                       // per-string log q of the segmented path, from the lq of the last evaluation
            KSParams S{};
            S.logaw = h->d_seg_logaw.p; S.words = h->d_kswords.p; S.sgoff = h->d_ksgoff.p; S.gref = h->d_ksgref.p; S.lq = h->d_krlq.p;
            S.p = h->d_ksp.p; S.logq = h->d_kslogq.p; S.n_sgroups = h->ks_groups; S.counter = h->d_seg_counter.p + 1;
            S.n_arcs = h->larcs.n_arcs;
            CK(cudaMemsetAsync(h->d_seg_counter.p + 1, 0, 4, h->stream));
            if (h->e6_used && h->lean_now) {     // the single-launch evaluation keeps the arc weights on chip: log weights from x now
                k_arc_logw<<<(h->larcs.n_arcs + 255) / 256, 256, 0, h->stream>>>(h->larcs.n_arcs, h->d_arc_tp.p, h->d_x.p, h->d_seg_logaw.p);
                h->launches++;
            }
            if (h->awg) ks_strings<true><<<h->ks_grid, h->ks_block, 0, h->stream>>>(S); else ks_strings<false><<<h->ks_grid, h->ks_block, h->ks_smem, h->stream>>>(S);
            h->launches++;
            h->ks_done = true;
        }
        const long long nk = (long long)h->d_kssid.n;
        k_scatter_logq<<<(unsigned)((nk + 255) / 256), 256, 0, h->stream>>>(nk, h->d_kssid.p, h->d_kslogq.p, h->d_logq.p);
        h->launches++;
    }
    if (logq && h->n_strings) CK(cudaMemcpyAsync(logq, h->d_logq.p, (size_t)h->n_strings * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    return finish_fetch(h, loglik, grad);
}

// H2D x -> k_eval6 captured once per parameter map; every node's parameters are constant.  The kernel of this graph writes
// [loglik, bad, grad] and, when the last CTA is through, a completion word straight into mapped pinned host memory: the
// host polls that word instead of paying for a D2H copy node and the wake-up of cudaStreamSynchronize.
static bool eval6_graph(wfsa_dev* h)
{
    if (h->e6_exec) return true;
    if (h->e6_graph_tried || getenv("WFSA_NO_GRAPH")) return false;
    h->e6_graph_tried = true;
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) return false;
    const size_t words = (size_t)h->n + 3;
    if (h->hm_n != words) {
        h->hm_n = 0;
        if (h->hm_out.alloc(words, cudaHostAllocMapped) != cudaSuccess ||
            h->hm_flag.alloc(16, cudaHostAllocMapped) != cudaSuccess ||
            cudaHostGetDevicePointer(&h->hm_out_dev, h->hm_out.p, 0) != cudaSuccess ||
            cudaHostGetDevicePointer(&h->hm_flag_dev, h->hm_flag.p, 0) != cudaSuccess) { cudaGetLastError(); return false; }
        std::memset(h->hm_out.p, 0, words * 8);
        *h->hm_flag.p = 0u;
        h->hm_n = words;
    }
    if (cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); return false; }
    // x: CTA 0 of the kernel fetches it from the mapped staging buffer and publishes it to the other CTAs (k_eval6, P.x_host).
    // A copy node in front of the kernel cost 12.5 us per call (measured: the DMA set-up and the dependency between the two
    // nodes), the fetch inside the kernel ~3 us.  (WFSA_E2E_COPY_NODE=1 brings the copy node back.)
    const bool copy_node = !h->h_x_dev || getenv("WFSA_E2E_COPY_NODE");
    if (copy_node) cudaMemcpyAsync(h->d_x.p, h->h_x.p, ((size_t)h->n + 1) * 8, cudaMemcpyHostToDevice, h->stream);
    launch_eval6(h, h->stream, false, true, !copy_node);
    cudaGraph_t g = nullptr;
    if (cudaStreamEndCapture(h->stream, &g) != cudaSuccess || !g) { cudaGetLastError(); return false; }
    h->e6_graph.reset(g);
    cudaGraphExec_t ex = nullptr;
    if (cudaGraphInstantiate(&ex, g, 0) != cudaSuccess) { cudaGetLastError(); h->e6_graph.reset(); return false; }
    h->e6_exec.reset(ex);
    return true;
}

extern "C" int wfsa_dev_eval(wfsa_dev* h, const double* x, double* loglik, double* logq, double* grad)
{
    if (h && h->n >= 0 && !logq && h->kernel == 6 && h->e6_ok && !h->any_overflow && !h->timing && !h->comm_failed) {
        // the lean segmented path as one graph launch
        CK(cudaSetDevice(h->device));
        if (eval6_graph(h)) {
            static const bool e2e_dbg = getenv("WFSA_E2E_DEBUG") != nullptr;
            const auto tp0 = std::chrono::steady_clock::now();
            const int rc = stage_x(h, x);
            if (rc != WFSA_OK) return rc;
            const auto tp1 = std::chrono::steady_clock::now();
            const unsigned int before = *reinterpret_cast<volatile unsigned int*>(h->hm_flag.p);   // the kernel writes a new count when it is through
            ++h->hm_runs;
            CK(cudaGraphLaunch(h->e6_exec, h->stream));
            const auto tp2 = std::chrono::steady_clock::now();
            h->launches++; h->e6_used = true; h->evaluated = true; h->ks_done = false; h->lean_now = true; h->lean_finished = true;
            // wait for the completion word of this epoch; every now and then ask the stream whether it failed instead
            volatile unsigned int* flag = h->hm_flag.p;
            for (unsigned long long spin = 1; *flag == before; ++spin)
                if ((spin & 0xfffffull) == 0) {
                    const cudaError_t q = cudaStreamQuery(h->stream);
                    if (q != cudaErrorNotReady) { if (q != cudaSuccess) CK(q); if (*flag == before) { cudaGetLastError(); return set_err(h, WFSA_ERR_CUDA, "k_eval6 finished without its completion word"); } }
                }
            const auto tp3 = std::chrono::steady_clock::now();
            // (the same values are NOT in d_out: a later wfsa_dev_eval_fetch finds them in h_out)
            h->out_on_host = true;
            const int frc = finish_fetch(h, loglik, grad, h->hm_out.p);
            if (e2e_dbg) {
                const auto tp4 = std::chrono::steady_clock::now();
                auto ns = [](auto a, auto b) { return (double)std::chrono::duration_cast<std::chrono::nanoseconds>(b - a).count(); };
                h->e2e_ns[0] += ns(tp0, tp1); h->e2e_ns[1] += ns(tp1, tp2); h->e2e_ns[2] += ns(tp2, tp3); h->e2e_ns[3] += ns(tp3, tp4);
                if (++h->e2e_calls % 20 == 0) {
                    fprintf(stderr, "[wfsa_dev_eval] host us per call over the last 20: stage x %.2f, graph launch %.2f, wait for the completion word %.2f, copy out %.2f\n",
                            h->e2e_ns[0] / 2e4, h->e2e_ns[1] / 2e4, h->e2e_ns[2] / 2e4, h->e2e_ns[3] / 2e4);
                    h->e2e_ns[0] = h->e2e_ns[1] = h->e2e_ns[2] = h->e2e_ns[3] = 0;
                }
            }
            return frc;
        }
    }
    int rc = wfsa_dev_upload_x(h, x);
    if (rc != WFSA_OK) return rc;
    rc = wfsa_dev_eval_launch(h);
    if (rc != WFSA_OK) return rc;
    return wfsa_dev_eval_fetch(h, loglik, logq, grad);
}

// ---------------------------------------------------------------------------------------------
// uploads validated path blocks and fixes the fixed-point scale of H (collective when a communicator is attached)
static int upload_path_blocks(wfsa_dev* h, const std::vector<int64_t>& po, const std::vector<int64_t>& co, const std::vector<int64_t>& vo,
                              const std::vector<int32_t>& cols, const std::vector<double>& counts, const std::vector<double>& p,
                              const std::vector<int32_t>* slots, unsigned long long local_error)
{
    const int64_t nb = (int64_t)p.size();
    CK(h->d_hb_path_off.upload(po, h->stream)); CK(h->d_hb_col_off.upload(co, h->stream)); CK(h->d_hb_val_off.upload(vo, h->stream));
    CK(h->d_hb_cols.upload(cols, h->stream)); CK(h->d_hb_counts.upload(counts, h->stream)); CK(h->d_hb_p.upload(p, h->stream));
    if (slots) CK(h->d_hb_slot.upload(*slots, h->stream)); else h->d_hb_slot.release();
    CK(h->d_hb_r.alloc(std::max<int64_t>(po[nb], 1)));
    CK(h->d_Hfx.alloc(std::max<size_t>((size_t)h->n * h->n, 1)));
    CK(h->d_H.alloc(std::max<size_t>((size_t)h->n * h->n, 1)));
    CK(h->d_rmin.alloc(1));
    CK(cudaStreamSynchronize(h->stream));
    // fixed-point scale of H: a block adds p_b * Cov_b(c_j, c_k) to an entry, |Cov_b| <= cmax_b^2 (cmax_b = largest |count|
    // of the block), so every single contribution and every entry of the sum over all blocks of all ranks is bounded by
    // sum_b |p_b| cmax_b^2.  The block weights need not sum to 1: a type weighs all its instances, a string with several
    // regions counts once per region.  The range 2^63 / fx = 2^(bits+2) is at least 4 (cmax^2 + 1), cmax over all blocks,
    // as for blocks of one string each (p summing to at most 1), and at least twice that bound.
    constexpr long long kRangeCap = 1ll << 50;
    double bound = 0.0, cmax_all = 1.0;
    for (int64_t b = 0; b < nb; ++b) {
        double cmax = 0.0;
        for (int64_t i = vo[b]; i < vo[b + 1]; ++i) cmax = std::max(cmax, std::fabs(counts[i]));
        bound += std::fabs(p[b]) * cmax * cmax;
        cmax_all = std::max(cmax_all, cmax);
    }
    long long v[3] = {bound < (double)kRangeCap ? (long long)std::ceil(bound) + 1 : kRangeCap, (long long)local_error,
                      cmax_all * cmax_all < (double)kRangeCap ? (long long)std::ceil(cmax_all * cmax_all) + 1 : kRangeCap};
    if (h->comm) {         // every rank must see a failure of any rank BEFORE the all-reduce of H (a rank that returned early would leave the others waiting)
        long long* d = reinterpret_cast<long long*>(h->d_red.p);
        CK(cudaMemcpyAsync(d, v, 24, cudaMemcpyHostToDevice, h->stream));
        int rc = nccl_allreduce(h, d, 2, ncclInt64, ncclSum);
        if (rc == WFSA_OK) rc = nccl_allreduce(h, d + 2, 1, ncclInt64, ncclMax);
        if (rc != WFSA_OK) return rc;
        CK(cudaMemcpyAsync(v, d, 24, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    if (v[1]) { h->hb_blocks = -1; return set_err(h, WFSA_ERR_LIMIT, local_error ? h->err : "H_f blocks: another rank could not build its path blocks"); }
    int bits = 1;
    while (bits <= 50 && ((1ll << bits) <= v[2] || (1ll << (bits + 1)) <= v[0])) ++bits;
    if (bits > 50 || v[0] >= kRangeCap) {
        h->hb_blocks = -1;
        return set_err(h, WFSA_ERR_LIMIT, "H_f blocks: the sum over the blocks of p * (largest count)^2 reaches 2^50, beyond the fixed-point range of H");
    }
    h->hb_fx_log2 = 61 - bits;
    h->hb_blocks = nb; h->hb_paths = po[nb];
    return WFSA_OK;
}

extern "C" int wfsa_dev_set_path_blocks(wfsa_dev* h, const wfsa_path_blocks* b)
{
    if (!h || !b || b->n_blocks < 0) return set_err(h, WFSA_ERR_INVALID, "set_path_blocks: bad arguments");
    if (h->n < 0) return set_err(h, WFSA_ERR_STATE, "set_path_blocks before set_param_map");
    CK(cudaSetDevice(h->device));
    const int64_t nb = b->n_blocks;
    std::vector<int64_t> po(b->path_off, b->path_off + nb + 1), co(b->col_off, b->col_off + nb + 1), vo(b->val_off, b->val_off + nb + 1);
    for (int64_t i = 0; i < nb; ++i) {
        const int64_t L = po[i + 1] - po[i], D = co[i + 1] - co[i];
        if (L < 0 || D < 0 || vo[i + 1] - vo[i] != L * D) return set_err(h, WFSA_ERR_INVALID, "set_path_blocks: inconsistent block sizes");
    }
    std::vector<int32_t> cols(b->cols, b->cols + co[nb]);
    for (int32_t c : cols) if (c < 0 || c >= h->n) return set_err(h, WFSA_ERR_INVALID, "set_path_blocks: column out of range");
    std::vector<double> counts(b->counts, b->counts + vo[nb]), p(b->p, b->p + nb);
    h->hb_user = true; h->hb_from_types = false;
    return upload_path_blocks(h, po, co, vo, cols, counts, p, nullptr, 0);
}

// H_f without enumerating the paths of any STRING.  Counts add over the segments of a string and the segments are
// independent given the string, so Cov_s(c_j, c_k) = sum over the REGIONS of s of Cov_region(c_j, c_k) (bridges have
// no variance), and with the type weights W = sum of p_s over the instances
//     H_f = - sum_types W_type * Cov_type(c_j, c_k):
// the blocks of k5_hessian are the distinct region types of the compiled corpus.  Path-form types are their own path
// list; the paths of a DAG-form type are enumerated from its words (a region, not a string: bounded by max_paths).
// Strings that no type covers add one block per segment (OverflowStrings below), under the same bound.  Past the bound
// the blocks fail as a whole (B.fail): never a partial H.
// Replaces the per-string BFS of Learner::BuildPaths feeding HessianLearner::ComputeHf (src/HessianLearner.cpp:498-547).
struct TypeBlocks {
    std::vector<int64_t> po{0}, co{0}, vo{0};
    std::vector<int32_t> cols, slots;
    std::vector<double> counts, bp;
    std::string fail;
};

// Strings that no region type covers (more live nodes than pool slots: SegmentedCorpus::overflow) have blocks of their own:
// one per segment with a choice, its paths enumerated from the string's trimmed lattice (segment_paths), weight p_s and no
// type slot (-1).
struct OverflowStrings {
    const HostFsa* f;
    const uint8_t* alive;                                 // [n_arcs]
    const int32_t* tokens;
    const int64_t* offs;
    const double* p;
    const std::vector<int32_t>* ids;
};

static void make_type_blocks(const LatticeArcs& A, const std::vector<int32_t>& ttp, const std::vector<int32_t>& etp,
                             const std::vector<uint32_t>& rw, const std::vector<int64_t>& rgoff, const std::vector<int32_t>& rgrows,
                             const std::vector<double>& typeW, const OverflowStrings& ov, TypeBlocks& B)
{
    const int64_t n_rg = (int64_t)rgrows.size();
    const size_t max_paths = 1u << 20;
    std::vector<std::vector<int32_t>> paths;              // arcs of every path of the current type
    std::vector<int32_t> col_of, bcols;                  // parameter -> column of the current block (-1: none), its columns
    std::vector<double> dense;                            // paths x columns of the current block
    auto emit = [&](const std::vector<std::vector<int32_t>>& pl, int64_t slot, double W) {
        auto each_param = [&](int32_t a, auto&& fn) {
            const int tp = ttp[A.arc_tid[a]], ep = A.arc_eid[a] < 0 ? -1 : etp[A.arc_eid[a]];
            if (tp >= 0) fn(tp);
            if (ep >= 0) fn(ep);
        };
        bcols.clear();
        for (const auto& pa : pl)
            for (int32_t a : pa)
                each_param(a, [&](int j) {
                    if (j >= (int)col_of.size()) col_of.resize((size_t)j + 1, -1);
                    if (col_of[j] < 0) { col_of[j] = 0; bcols.push_back(j); }
                });
        std::sort(bcols.begin(), bcols.end());
        const size_t D = bcols.size();
        for (size_t k = 0; k < D; ++k) col_of[bcols[k]] = (int32_t)k;
        dense.assign(pl.size() * D, 0.0);
        for (size_t q = 0; q < pl.size(); ++q)
            for (int32_t a : pl[q]) each_param(a, [&](int j) { dense[q * D + col_of[j]] += 1.0; });
        std::vector<size_t> keep;                          // columns whose count differs between the paths (src/HessianLearner.cpp:409-443)
        for (size_t k = 0; k < D; ++k) {
            bool same = true;
            for (size_t q = 1; q < pl.size() && same; ++q) same = dense[q * D + k] == dense[k];
            if (!same) keep.push_back(k);
        }
        for (int j : bcols) col_of[j] = -1;
        for (size_t k : keep) B.cols.push_back(bcols[k]);
        for (size_t q = 0; q < pl.size(); ++q)
            for (size_t k : keep) B.counts.push_back(dense[q * D + k]);
        B.po.push_back(B.po.back() + (int64_t)pl.size());
        B.co.push_back((int64_t)B.cols.size());
        B.vo.push_back((int64_t)B.counts.size());
        B.bp.push_back(W);
        B.slots.push_back((int32_t)slot);
    };
    for (int64_t g = 0; g < n_rg && B.fail.empty(); ++g) {
        const int code = rgrows[g];
        const uint32_t* base = rw.data() + rgoff[g];
        for (int l = 0; l < 32 && B.fail.empty(); ++l) {
            const double W = typeW[(size_t)g * 32 + l];
            if (!(W > 0.0)) continue;
            paths.clear();
            if (code & 0x10000) {
                const int PP = (code >> 8) & 0xff, L = code & 0xff;
                for (int q = 0; q < PP; ++q) {
                    std::vector<int32_t> pa;
                    bool real = true;
                    for (int el = 0; el < L; ++el) {
                        const uint32_t a = base[(size_t)(el * PP + q) * 32 + l];
                        if ((int)a >= A.n_arcs) { real = false; break; }
                        pa.push_back((int32_t)a);
                    }
                    if (real) paths.push_back(std::move(pa));
                }
            } else {
                // DAG form: rebuild the nodes from the slot life times, then walk every path from the entry to the FIN node
                const int rows = (int)((rgoff[g + 1] - rgoff[g]) >> 5);
                std::vector<int> node_of(16, -1);
                std::vector<std::vector<std::pair<int, int32_t>>> out;      // node -> (dst node, arc)
                auto new_node = [&]() { out.emplace_back(); return (int)out.size() - 1; };
                const int entry_node = node_of[0] = new_node();          // (slot 0 may be taken by a later node)
                int exit_node = -1;
                for (int i = 0; i < rows; ++i) {
                    const uint32_t w = base[(size_t)i * 32 + l];
                    if ((i & (kCheckEvery - 1)) == kCheckEvery - 1) continue;               // CHECK word
                    if (w & kLatEdge) {
                        const int src = (w >> kLatSrcShift) & 15, dst = (w >> kLatDstShift) & 15;
                        if (w & kLatFirstIn) node_of[dst] = new_node();
                        out[node_of[src]].push_back({node_of[dst], (int32_t)(w & 0xffff)});
                    } else if (w & kLatFin) exit_node = node_of[w & 15];
                }
                if (exit_node < 0) { B.fail = "H_f blocks: a DAG-form region type has no FIN word"; break; }
                std::vector<std::pair<int, size_t>> stack{{entry_node, 0}};
                std::vector<int32_t> cur;
                while (!stack.empty()) {
                    auto& top = stack.back();
                    if (top.first == exit_node) {
                        paths.push_back(cur);
                        if (paths.size() > max_paths) { B.fail = "H_f blocks: a region type has more than 2^20 paths"; break; }
                        stack.pop_back(); if (!cur.empty()) cur.pop_back();
                        continue;
                    }
                    if (top.second >= out[top.first].size()) { stack.pop_back(); if (!cur.empty()) cur.pop_back(); continue; }
                    const auto ed = out[top.first][top.second++];
                    cur.push_back(ed.second);
                    stack.push_back({ed.first, 0});
                }
            }
            if (B.fail.empty() && paths.size() >= 2) emit(paths, g * 32 + l, W);
        }
    }
    LatticeScratch S;
    for (size_t i = 0; i < ov.ids->size() && B.fail.empty(); ++i) {
        const int32_t s = (*ov.ids)[i];
        if (!(ov.p[s] > 0.0)) continue;
        const int rc = segment_paths(*ov.f, A, ov.alive, ov.tokens + ov.offs[s], (int)(ov.offs[s + 1] - ov.offs[s]), max_paths, S,
                                     [&](const std::vector<std::vector<int32_t>>& seg) { emit(seg, -1, ov.p[s]); });
        if (rc < 0) B.fail = "H_f blocks: a segment of string " + std::to_string(s) + " (more live nodes than pool slots) has more than 2^20 paths";
    }
}

static int build_type_blocks(wfsa_dev* h)
{
    const LatticeArcs& A = h->larcs;
    std::vector<uint8_t> alive((size_t)A.n_arcs);          // as wfsa_dev_set_param_map compiled the strings
    for (int a = 0; a < A.n_arcs; ++a)
        alive[a] = h->h_ttp[A.arc_tid[a]] != -2 && (A.arc_eid[a] < 0 || h->h_etp[A.arc_eid[a]] != -2);
    const OverflowStrings ov{&h->fsa, alive.data(), h->h_tokens.data(), h->h_offs.data(), h->h_p.data(), &h->h_seg_overflow};
    TypeBlocks B;
    make_type_blocks(A, h->h_ttp, h->h_etp, h->hrw, h->hrgoff, h->hrgrows, h->hrW, ov, B);
    if (!B.fail.empty()) h->err = B.fail;
    CK(h->d_type_lrmin.alloc(h->hrgrows.size() * 32 + 1));
    CK(cudaMemsetAsync(h->d_type_lrmin.p, 0, h->d_type_lrmin.n * 8, h->stream));
    const int rc = upload_path_blocks(h, B.po, B.co, B.vo, B.cols, B.counts, B.bp, &B.slots, B.fail.empty() ? 0 : 1);
    if (rc == WFSA_OK) h->hb_from_types = true;
    return rc;
}

static int ensure_ks(wfsa_dev* h);

// rterm[s] = m_s - log q_s of the strings of one order list with fast tables (k3_minpath) or without (generic kernel:
// a (min, +) forward, an evaluation for log q, k_rmin_terms)
static void rmin_sweep_list(wfsa_dev* h, const int32_t* d_ord, int64_t n_ord)
{
    const HostFsa& F = h->fsa;
    const FastLayout& L = h->fast;
    cudaStream_t st = h->stream;
    if (n_ord <= 0) return;
    const CorpusD C{h->d_tokens.p, h->d_offs.p, h->d_p.p, d_ord, n_ord};
    if (L.ok) {
        K3MinParams P{};
        P.T = FastTablesD{h->d_cand_off.p, h->d_slot_state.p, h->d_frow.p, h->d_fent.p, h->d_brow.p, h->d_bent.p,
                          F.n_sym, F.n_states, L.n_arcs, L.n_slots, F.start, L.start_final_tid};
        P.W = EvalWeightsD{h->d_tw.p, h->d_sw.p, h->d_fw.p};
        P.mtw = h->d_mtw.p; P.msw = h->d_msw.p; P.mfw = h->d_mfw.p; P.C = C; P.rterm = h->d_rterm.p;
        const int nt = std::max(64, (L.max_cand + 31) / 32 * 32);
        const int grid = h->sm_count * std::max(1, std::min(4, 1024 / nt));
        k3_minpath<<<grid, nt, (size_t)(4 * nt + 64) * 8 + 32 * 4, st>>>(P);
        h->launches++;
        return;
    }
    GenericParams P{};
    P.G = GenericTablesD{h->d_emis_row.p, h->d_emis_tok_off.p, h->d_emis_tok.p, h->d_trans_row.p, h->d_trans_dst.p,
                         h->d_eps_order.p, F.n_states, F.n_trans(), F.start, F.end};
    P.C = C; P.scratch = h->d_gscratch.p; P.max_len = h->max_len;
    P.O.red = h->d_red.p; P.O.fx_scale = std::ldexp(1.0, (int)h->fx_log2); P.O.ll_scale = std::ldexp(1.0, (int)h->ll_log2);
    for (long long first = 0; first < n_ord; first += h->g_batch) {
        P.first = first; P.count = std::min<long long>(h->g_batch, n_ord - first);
        const int grid = (int)((P.count + 127) / 128);
        P.ltw = h->d_mtw.p; P.lew = h->d_mew.p; P.O.logq = h->d_mpath.p;             // m_s
        kg_fwdbwd<MODE_MINPATH><<<grid, 128, 0, st>>>(P);
        P.ltw = h->d_ltw.p; P.lew = h->d_lew.p; P.O.logq = h->d_mlq.p;               // log q (its posteriors go to the scratch d_red)
        kg_fwdbwd<MODE_EVAL><<<grid, 128, 0, st>>>(P);
        h->launches += 2;
    }
    k_rmin_terms<<<(unsigned)((n_ord + 255) / 256), 256, 0, st>>>(n_ord, d_ord, h->d_mpath.p, h->d_mlq.p, h->d_rterm.p);
    h->launches++;
}

// The smallest path posterior without enumerating paths: r_s = exp(m_s - log q_s), m_s the smallest log weight of a path
// of s, by a forward sweep in (min, +) over the lattice of the evaluation; rmin = min_s r_s (1 when no string has a choice).
// `all`: every active string (else, on the segmented path, its overflow strings only).  x is on the device; d_rsweep
// receives rmin.
static int rmin_sweep(wfsa_dev* h, bool all)
{
    const HostFsa& F = h->fsa;
    const FastLayout& L = h->fast;
    cudaStream_t st = h->stream;
    const size_t ns = (size_t)std::max<int64_t>(h->n_strings, 1);
    if (h->d_rterm.n < ns) {
        CK(h->d_rterm.alloc(ns)); CK(h->d_mlq.alloc(ns)); CK(h->d_rsweep.alloc(1));
        if (!L.ok) CK(h->d_mpath.alloc(ns));
        CK(h->d_mtw.alloc(std::max(F.n_trans(), 1))); CK(h->d_mew.alloc(std::max(F.n_emis(), 1)));
        CK(h->d_msw.alloc(std::max(L.ok ? L.n_slots : 0, 1))); CK(h->d_mfw.alloc(std::max(L.ok ? L.n_slots : 0, 1)));
    }
    CK(cudaMemsetAsync(h->d_rterm.p, 0, ns * 8, st));
    const int n_slots = L.ok ? L.n_slots : 0;
    const int total = F.n_trans() + F.n_emis() + n_slots;
    if (total > 0) {
        k_weights<<<(total + 255) / 256, 256, 0, st>>>(F.n_trans(), F.n_emis(), n_slots, h->d_trans_tp.p, h->d_emis_tp.p,
                                                      h->d_slot_emis.p, h->d_slot_final.p, h->d_x.p, 0, h->d_tw.p,
                                                      h->d_sw.p, h->d_fw.p, h->d_ltw.p, h->d_lew.p);
        k_minplus_weights<<<(total + 255) / 256, 256, 0, st>>>(F.n_trans(), F.n_emis(), n_slots, h->d_trans_tp.p, h->d_emis_tp.p,
                                                              h->d_slot_emis.p, h->d_slot_final.p, h->d_x.p, h->d_mtw.p,
                                                              h->d_mew.p, h->d_msw.p, h->d_mfw.p);
        h->launches += 2;
    }
    if (h->kernel == 6) {
        if (all) rmin_sweep_list(h, h->d_order.p, h->n_active + h->n_active_w);
        else rmin_sweep_list(h, h->d_order_w.p, h->n_active_w);
    } else if (h->kernel == 7 && h->k7_planes) {
        // K7's batches: the forward sweep of the evaluation (k7_fwd2, k7_finish_q) for log q, beside it the (min, +)
        // sweep (k7_minfwd2) in the two rows of the backward sweep, k7_finish_min where strings end; strings with unknown
        // symbols on the CTA-per-string kernel, as in the evaluation
        FastTablesD T{};
        T.cand_off = h->d_cand_off.p; T.slot_state = h->d_slot_state.p;
        T.frow = h->d_frow.p; T.fent = h->d_fent.p; T.brow = h->d_brow.p; T.bent = h->d_bent.p;
        T.n_sym = F.n_sym; T.n_states = F.n_states; T.n_arcs = L.n_arcs; T.n_slots = L.n_slots;
        T.start_state = F.start; T.start_final_tid = L.start_final_tid;
        const EvalWeightsD Wt{h->d_tw.p, h->d_sw.p, h->d_fw.p};
        EvalOutD O{};
        O.logq = h->d_mlq.p; O.red = h->d_red.p; O.ll_scale = std::ldexp(1.0, (int)h->ll_log2);   // (loglik goes to the scratch d_red)
        const int V = h->k7_V;
        const size_t smem = (size_t)kK7Chunk * V * 8;
        double* const lat = h->d_k7lat.p;
        double* const mu[2] = {h->d_k7bt.p, h->d_k7bt.p + h->k7_nb * (size_t)V};
        for (auto& B : h->k7) {
            K7FinParams Fn{};
            Fn.T = T; Fn.W = Wt; Fn.O = O; Fn.sid = B.d_sid.p; Fn.last_tok = B.d_last.p; Fn.p = h->d_p.p;
            Fn.scale = h->d_k7scale.p; Fn.EQ = h->d_k7EQ.p; Fn.F = h->d_k7F.p; Fn.V = V;
            K7Params P{};
            P.T = T; P.W = Wt; P.O = O; P.V = V; P.pe = h->d_k7pef.p; P.pr = h->d_k7prf.p;
            K7MinParams M{};
            M.T = T; M.mtw = h->d_mtw.p; M.msw = h->d_msw.p; M.pe = h->d_k7pef.p; M.pr = h->d_k7prf.p; M.V = V;
            K7MinFinParams Mf{};
            Mf.T = T; Mf.sid = B.d_sid.p; Mf.last_tok = B.d_last.p; Mf.mfw = h->d_mfw.p; Mf.logq = h->d_mlq.p; Mf.rterm = h->d_rterm.p; Mf.V = V;
            for (int t = 0; t < B.Tmax; ++t) {
                P.desc = M.desc = B.d_desc.p + B.desc_off[t]; P.perm = M.perm = B.d_perm.p + B.row_off[t];
                P.src = t ? lat + B.row_off[t - 1] * V : nullptr; P.dst = lat + B.row_off[t] * V;
                P.exp_src = t ? h->d_k7exp.p + B.row_off[t - 1] : nullptr; P.exp_dst = h->d_k7exp.p + B.row_off[t];
                P.rescale = (t & (kRescaleEvery - 1)) == kRescaleEvery - 1;
                M.src = t ? mu[(t - 1) & 1] : nullptr; M.dst = mu[t & 1];
                const unsigned nd = (unsigned)(B.desc_off[t + 1] - B.desc_off[t]);
                if (nd) {
                    if (V <= 320) { k7_fwd2<320, 4><<<nd, V, smem, st>>>(P); k7_minfwd2<320, 4><<<nd, V, smem, st>>>(M); }
                    else { k7_fwd2<512, 2><<<nd, V, smem, st>>>(P); k7_minfwd2<512, 2><<<nd, V, smem, st>>>(M); }
                    h->launches += 2;
                }
                if (B.n_t[t + 1] < B.n_t[t]) {
                    Fn.r0 = Mf.r0 = B.n_t[t + 1]; Fn.r1 = Mf.r1 = B.n_t[t];
                    Fn.lat = lat + B.row_off[t] * V; Fn.exp_t = h->d_k7exp.p + B.row_off[t]; Mf.mu = mu[t & 1];
                    k7_finish_q<<<(Fn.r1 - Fn.r0 + 7) / 8, 256, 0, st>>>(Fn);
                    k7_finish_min<<<(Mf.r1 - Mf.r0 + 7) / 8, 256, 0, st>>>(Mf);
                    h->launches += 2;
                }
            }
        }
        rmin_sweep_list(h, h->d_order_w.p, h->n_active_w);
    } else if (h->kernel == 7) {
        rmin_sweep_list(h, h->d_order.p, h->n_active + h->n_active_w);    // without pair planes: every string on k3_minpath
    } else {
        rmin_sweep_list(h, h->d_order.p, h->n_active);
        rmin_sweep_list(h, h->d_order_w.p, h->n_active_w);                  // (kernel 4: strings beyond its active sets)
    }
    if (h->n_strings) {
        k_min_exp<<<1, 1024, 0, st>>>((long long)h->n_strings, h->d_rterm.p, h->d_rsweep.p);
        h->launches++;
    } else {
        const double one = 1.0;
        CK(cudaMemcpyAsync(h->d_rsweep.p, &one, 8, cudaMemcpyHostToDevice, st));
    }
    CK(cudaGetLastError());
    return WFSA_OK;
}

// Backpointer slabs of k3_viterbi: a group (warp or CTA) holds max_len x pitch uint16; the grid shrinks when the slabs
// of all groups would take more than this (very long strings).  k3_nbest's slabs are k times as large, its budget K times.
constexpr size_t kViterbiSlabBudget = (size_t)256 << 20;

// k3_viterbi over one order list (fast tables): a warp per string when every symbol has at most 32 candidates, else a CTA
static int viterbi_fast_list(wfsa_dev* h, const int32_t* d_ord, int64_t n_ord)
{
    if (n_ord <= 0) return WFSA_OK;
    const HostFsa& F = h->fsa;
    const FastLayout& L = h->fast;
    K3VitParams P{};
    P.T = FastTablesD{h->d_cand_off.p, h->d_slot_state.p, h->d_frow.p, h->d_fent.p, h->d_brow.p, h->d_bent.p,
                      F.n_sym, F.n_states, L.n_arcs, L.n_slots, F.start, L.start_final_tid};
    P.vtw = h->d_vtw.p; P.vsw = h->d_vsw.p; P.vfw = h->d_vfw.p; P.slot_emis = h->d_slot_emis.p; P.slot_final = h->d_slot_final.p;
    P.C = CorpusD{h->d_tokens.p, h->d_offs.p, h->d_p.p, d_ord, n_ord};
    P.max_len = std::max(h->max_len, 1);
    P.logw = h->d_vlogw.p; P.trans_edge = h->d_vtrans.p; P.emis_edge = h->d_vemis.p;
    const bool warp = L.max_cand <= 32;
    const int nt = warp ? 256 : std::max(64, (L.max_cand + 31) / 32 * 32);
    const int per_cta = warp ? nt / 32 : 1;                                   // strings in flight per CTA
    P.pitch = warp ? 32 : nt;
    const size_t slab_bytes = (size_t)P.max_len * P.pitch * 2 * per_cta;     // per CTA
    long long grid = (long long)h->sm_count * (warp ? 8 : std::max(1, std::min(4, 1024 / nt)));
    grid = std::min<long long>(grid, (n_ord + per_cta - 1) / per_cta);
    grid = std::max<long long>(1, std::min<long long>(grid, (long long)(kViterbiSlabBudget / slab_bytes)));
    const size_t need = (size_t)grid * per_cta * P.max_len * P.pitch;
    if (h->d_vbp.n < need) CK(h->d_vbp.alloc(need));
    P.bp = h->d_vbp.p;
    const size_t smem = (size_t)2 * nt * 8 + 32 * 8 + 32 * 4;
    if (warp) k3_viterbi<true><<<(unsigned)grid, nt, smem, h->stream>>>(P);
    else k3_viterbi<false><<<(unsigned)grid, nt, smem, h->stream>>>(P);
    h->launches++;
    return WFSA_OK;
}

// k3_nbest<WARP, K> over one order list (fast tables), K the power of two >= k: a warp per string as k3_viterbi, else a
// CTA.  The lists take 2 * K * G doubles of shared memory per group; WFSA_ERR_LIMIT when a CTA's do not fit, or when the
// CTA would need more threads than k3_nbest<false, K> allows.
static int nbest_fast_list(wfsa_dev* h, const int32_t* d_ord, int64_t n_ord, int k)
{
    if (n_ord <= 0) return WFSA_OK;
    const HostFsa& F = h->fsa;
    const FastLayout& L = h->fast;
    K3NbestParams P{};
    P.T = FastTablesD{h->d_cand_off.p, h->d_slot_state.p, h->d_frow.p, h->d_fent.p, h->d_brow.p, h->d_bent.p,
                      F.n_sym, F.n_states, L.n_arcs, L.n_slots, F.start, L.start_final_tid};
    P.vtw = h->d_vtw.p; P.vsw = h->d_vsw.p; P.vfw = h->d_vfw.p; P.slot_emis = h->d_slot_emis.p; P.slot_final = h->d_slot_final.p;
    P.C = CorpusD{h->d_tokens.p, h->d_offs.p, h->d_p.p, d_ord, n_ord};
    P.max_len = std::max(h->max_len, 1);
    P.k = k;
    P.logw = h->d_vlogw.p; P.trans_edge = h->d_vtrans.p; P.emis_edge = h->d_vemis.p;
    const int K = k <= 2 ? 2 : k <= 4 ? 4 : k <= 8 ? 8 : 16;
    const bool warp = L.max_cand <= 32;
    const int nt = warp ? 256 : std::max(64, (L.max_cand + 31) / 32 * 32);
    const size_t smem = (size_t)2 * K * nt * 8 + 32 * 8 + 32 * 4 + 32 * kNbestMax * 4;
    int optin = 0;
    CK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
    if (smem > (size_t)optin || nt > nbest_cta_threads(K))
        return set_err(h, WFSA_ERR_LIMIT, "nbest: the lists of " + std::to_string(nt) + " candidates at k = " + std::to_string(k) +
                                              " need " + std::to_string(smem) + " bytes of shared memory per CTA (at most " +
                                              std::to_string(optin) + ") and " + std::to_string(nt) + " threads (at most " +
                                              std::to_string(nbest_cta_threads(K)) + "); use a smaller k");
    const int per_cta = warp ? nt / 32 : 1;                                   // strings in flight per CTA
    P.pitch = warp ? 32 : nt;
    const size_t slab_bytes = (size_t)P.max_len * P.pitch * k * 2 * per_cta; // per CTA
    long long grid = (long long)h->sm_count * (warp ? 8 : std::max(1, std::min(4, 1024 / nt)));
    grid = std::min<long long>(grid, (n_ord + per_cta - 1) / per_cta);
    grid = std::max<long long>(1, std::min<long long>(grid, (long long)(kViterbiSlabBudget * K / slab_bytes)));
    const size_t need = (size_t)grid * per_cta * P.max_len * P.pitch * k;
    if (h->d_vbp.n < need) CK(h->d_vbp.alloc(need));
    P.bp = h->d_vbp.p;
    auto launch = [&](auto kern) {
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<(unsigned)grid, nt, smem, h->stream>>>(P);
        return WFSA_OK;
    };
    int rc;
    switch (K) {
    case 2: rc = warp ? launch(k3_nbest<true, 2>) : launch(k3_nbest<false, 2>); break;
    case 4: rc = warp ? launch(k3_nbest<true, 4>) : launch(k3_nbest<false, 4>); break;
    case 8: rc = warp ? launch(k3_nbest<true, 8>) : launch(k3_nbest<false, 8>); break;
    default: rc = warp ? launch(k3_nbest<true, 16>) : launch(k3_nbest<false, 16>); break;
    }
    h->launches++;
    return rc;
}

// wfsa_dev_sample's arguments, for decode_paths
struct SampleSpec {
    uint64_t seed;
    double* logq;                            // [n_strings], on the host
};

// k3_sample over one order list (fast tables): k3_viterbi's groups and grid; its alpha slabs take four times the bytes of
// k3_viterbi's backpointer slabs, within four times their budget
static int sample_fast_list(wfsa_dev* h, const int32_t* d_ord, int64_t n_ord, int n, uint64_t seed)
{
    if (n_ord <= 0) return WFSA_OK;
    const HostFsa& F = h->fsa;
    const FastLayout& L = h->fast;
    K3SampleParams P{};
    P.T = FastTablesD{h->d_cand_off.p, h->d_slot_state.p, h->d_frow.p, h->d_fent.p, h->d_brow.p, h->d_bent.p,
                      F.n_sym, F.n_states, L.n_arcs, L.n_slots, F.start, L.start_final_tid};
    P.W = EvalWeightsD{h->d_stw.p, h->d_ssw.p, h->d_sfw.p};
    P.vtw = h->d_vtw.p; P.vew = h->d_vew.p; P.slot_emis = h->d_slot_emis.p; P.slot_final = h->d_slot_final.p;
    P.C = CorpusD{h->d_tokens.p, h->d_offs.p, h->d_p.p, d_ord, n_ord};
    P.max_len = std::max(h->max_len, 1);
    P.n = n; P.key0 = (uint32_t)seed; P.key1 = (uint32_t)(seed >> 32);
    P.logw = h->d_vlogw.p; P.logq = h->d_vlogw.p + (size_t)h->n_strings * n;
    P.trans_edge = h->d_vtrans.p; P.emis_edge = h->d_vemis.p;
    const bool warp = L.max_cand <= 32;
    const int nt = warp ? 256 : std::max(64, (L.max_cand + 31) / 32 * 32);
    const int per_cta = warp ? nt / 32 : 1;                                   // strings in flight per CTA
    P.pitch = warp ? 32 : nt;
    const size_t slab_bytes = (size_t)P.max_len * P.pitch * 8 * per_cta;     // per CTA
    long long grid = (long long)h->sm_count * (warp ? 8 : std::max(1, std::min(4, 1024 / nt)));
    grid = std::min<long long>(grid, (n_ord + per_cta - 1) / per_cta);
    grid = std::max<long long>(1, std::min<long long>(grid, (long long)(4 * kViterbiSlabBudget / slab_bytes)));
    const size_t need = (size_t)grid * per_cta * P.max_len * P.pitch;
    if (h->d_sslab.n < need) CK(h->d_sslab.alloc(need));
    P.slab = h->d_sslab.p;
    const size_t smem = (size_t)2 * nt * 8 + 32 * 8 + 32 * 4;
    if (warp) k3_sample<true><<<(unsigned)grid, nt, smem, h->stream>>>(P);
    else k3_sample<false><<<(unsigned)grid, nt, smem, h->stream>>>(P);
    h->launches++;
    return WFSA_OK;
}

// Over one order list without fast tables, step counts (d_voff == nullptr) or the steps: kg_fwdbwd<MODE_VITERBI> in g_batch
// batches (k = 1), else kg_nbest in batches of g_batch / k strings, whose lists take k times a string's scratch; with smp
// kg_sample in g_batch batches (k draws per string)
static void viterbi_generic_list(wfsa_dev* h, const int32_t* d_ord, int64_t n_ord, const int64_t* d_voff, int k,
                                 const SampleSpec* smp = nullptr)
{
    const HostFsa& F = h->fsa;
    GenericParams P{};
    P.G = GenericTablesD{h->d_emis_row.p, h->d_emis_tok_off.p, h->d_emis_tok.p, h->d_trans_row.p, h->d_trans_dst.p,
                         h->d_eps_order.p, F.n_states, F.n_trans(), F.start, F.end};
    P.C = CorpusD{h->d_tokens.p, h->d_offs.p, h->d_p.p, d_ord, n_ord};
    P.scratch = !smp && k > 1 && h->g_batch < k ? h->d_nscratch.p : h->d_gscratch.p; P.max_len = h->max_len;
    P.ltw = h->d_vtw.p; P.lew = h->d_vew.p; P.O.logq = h->d_vlogw.p;
    P.vit_cnt = h->d_vcnt.p; P.vit_off = d_voff; P.vit_trans = h->d_vtrans.p; P.vit_emis = h->d_vemis.p;
    const long long batch = smp ? h->g_batch : std::max<long long>(1, h->g_batch / k);
    for (long long first = 0; first < n_ord; first += batch) {
        P.first = first; P.count = std::min<long long>(batch, n_ord - first);
        if (smp) kg_sample<<<(unsigned)((P.count + 127) / 128), 128, 0, h->stream>>>(P, k, (uint32_t)smp->seed, (uint32_t)(smp->seed >> 32),
                                                                                    h->d_vlogw.p + (size_t)h->n_strings * k);
        else if (k == 1) kg_fwdbwd<MODE_VITERBI><<<(unsigned)((P.count + 127) / 128), 128, 0, h->stream>>>(P);
        else kg_nbest<<<(unsigned)((P.count + 127) / 128), 128, 0, h->stream>>>(P, k);
        h->launches++;
    }
}

// wfsa_dev_viterbi (k = 1: k3_viterbi, kg_fwdbwd<MODE_VITERBI>), wfsa_dev_nbest (k3_nbest, kg_nbest) and, with smp,
// wfsa_dev_sample (k draws: k3_sample, kg_sample); path i = s * k + r
static int decode_paths(wfsa_dev* h, const double* x, int k, double* logw, int64_t* path_off, const SampleSpec* smp = nullptr)
{
    CK(cudaSetDevice(h->device));
    h->v_done = false;
    const HostFsa& F = h->fsa;
    const FastLayout& L = h->fast;
    cudaStream_t st = h->stream;
    const int64_t ns = h->n_strings, np = ns * k;
    const int n_slots = L.ok ? L.n_slots : 0;
    if (h->d_vx.n < (size_t)h->n + 1) CK(h->d_vx.alloc((size_t)h->n + 1));
    if (!h->d_vtw.p) {
        CK(h->d_vtw.alloc(std::max(F.n_trans(), 1))); CK(h->d_vew.alloc(std::max(F.n_emis(), 1)));
        CK(h->d_vsw.alloc(std::max(n_slots, 1))); CK(h->d_vfw.alloc(std::max(n_slots, 1)));
    }
    const int64_t nw = np + (smp ? ns : 0);                                 // sampling: log q behind the draws' logw
    if (h->d_vlogw.n < (size_t)std::max<int64_t>(nw, 1)) CK(h->d_vlogw.alloc((size_t)std::max<int64_t>(nw, 1)));
    if (!L.ok && h->d_vcnt.n < (size_t)std::max<int64_t>(np, 1)) {
        CK(h->d_vcnt.alloc((size_t)std::max<int64_t>(np, 1))); CK(h->d_voff.alloc((size_t)np + 1));
    }
    if (smp && !h->d_stw.p) {
        CK(h->d_stw.alloc(std::max(F.n_trans(), 1)));
        CK(h->d_ssw.alloc(std::max(n_slots, 1))); CK(h->d_sfw.alloc(std::max(n_slots, 1)));
    }
    const int64_t padded = k * (h->n_tokens + ns);
    if (L.ok && h->d_vtrans.n < (size_t)padded) {                           // fast tables: len + 1 steps per path, padded
        if (h->d_vtrans.alloc((size_t)padded) != cudaSuccess || h->d_vemis.alloc((size_t)padded) != cudaSuccess) {
            h->d_vtrans.release(); h->d_vemis.release();
            cudaGetLastError();
            return set_err(h, WFSA_ERR_NOMEM, "cannot allocate the step buffer of " + std::to_string(k) + " x (" +
                                                  std::to_string(h->n_tokens) + " symbols + " + std::to_string(ns) +
                                                  " strings) = " + std::to_string(padded) + " steps (8 bytes each)");
        }
    }
    if (!L.ok && !smp && k > 1 && h->g_batch < k) {                         // kg_nbest needs room for one string's k lists
        const size_t per = (size_t)2 * (h->max_len + 1) * F.n_states * k;
        if (h->d_nscratch.n < per) CK(h->d_nscratch.alloc(per));
    }
    if (h->n > 0) CK(cudaMemcpyAsync(h->d_vx.p, x, (size_t)h->n * 8, cudaMemcpyHostToDevice, st));
    const long long total = (long long)F.n_trans() + F.n_emis() + n_slots + nw;
    if (total > 0) {
        k_maxplus_weights<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(F.n_trans(), F.n_emis(), n_slots, (long long)nw,
                                                                         h->d_trans_tp.p, h->d_emis_tp.p, h->d_slot_emis.p,
                                                                         h->d_slot_final.p, h->d_vx.p, h->d_vtw.p, h->d_vew.p,
                                                                         h->d_vsw.p, h->d_vfw.p, h->d_vlogw.p);
        h->launches++;
    }
    const long long nlin = (long long)F.n_trans() + F.n_emis() + n_slots;
    if (smp && nlin > 0) {              // linear weights as the evaluation builds them (its log weights are k_maxplus_weights')
        k_weights<<<(unsigned)((nlin + 255) / 256), 256, 0, st>>>(F.n_trans(), F.n_emis(), n_slots, h->d_trans_tp.p, h->d_emis_tp.p,
                                                                  h->d_slot_emis.p, h->d_slot_final.p, h->d_vx.p, 0, h->d_stw.p,
                                                                  h->d_ssw.p, h->d_sfw.p, h->d_vtw.p, h->d_vew.p);
        h->launches++;
    }
    // the strings that take part, as in the rmin sweep: the segmented and the batched kernel keep all of them in d_order
    const int32_t* lists[2] = {h->d_order.p, h->d_order_w.p};
    int64_t counts[2] = {h->n_active, h->n_active_w};
    if (h->kernel == 6 || h->kernel == 7) { counts[0] = h->n_active + h->n_active_w; counts[1] = 0; }
    std::vector<int32_t> cnt;
    if (L.ok) {
        for (int i = 0; i < 2; ++i) {
            const int rc = smp ? sample_fast_list(h, lists[i], counts[i], k, smp->seed)
                         : k == 1 ? viterbi_fast_list(h, lists[i], counts[i]) : nbest_fast_list(h, lists[i], counts[i], k);
            if (rc != WFSA_OK) return rc;
        }
    } else {
        // step counts first (they vary with empty and multi-token emissions), then their prefix sum, then the steps
        if (np) CK(cudaMemsetAsync(h->d_vcnt.p, 0, (size_t)np * 4, st));
        for (int i = 0; i < 2; ++i) if (counts[i] > 0) viterbi_generic_list(h, lists[i], counts[i], nullptr, k, smp);
        cnt.resize((size_t)np);
        if (np) CK(cudaMemcpyAsync(cnt.data(), h->d_vcnt.p, (size_t)np * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        CK(cudaGetLastError());
    }
    if (np) CK(cudaMemcpyAsync(logw, h->d_vlogw.p, (size_t)np * 8, cudaMemcpyDeviceToHost, st));
    if (smp && smp->logq && ns) CK(cudaMemcpyAsync(smp->logq, h->d_vlogw.p + np, (size_t)ns * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    path_off[0] = 0;
    for (int64_t i = 0; i < np; ++i) {
        const int64_t s = i / k;
        path_off[i + 1] = path_off[i] + (L.ok ? (logw[i] > -INFINITY ? h->h_offs[s + 1] - h->h_offs[s] + 1 : 0) : cnt[(size_t)i]);
    }
    h->h_vpath_off.assign(path_off, path_off + np + 1);
    if (!L.ok) {
        const int64_t steps = path_off[np];
        if (h->d_vtrans.n < (size_t)std::max<int64_t>(steps, 1)) {
            CK(h->d_vtrans.alloc((size_t)std::max<int64_t>(steps, 1))); CK(h->d_vemis.alloc((size_t)std::max<int64_t>(steps, 1)));
        }
        CK(cudaMemcpyAsync(h->d_voff.p, path_off, (size_t)(np + 1) * 8, cudaMemcpyHostToDevice, st));
        for (int i = 0; i < 2; ++i) if (counts[i] > 0) viterbi_generic_list(h, lists[i], counts[i], h->d_voff.p, k, smp);
        CK(cudaStreamSynchronize(st));
        CK(cudaGetLastError());
    }
    h->v_k = k;
    h->v_padded = L.ok;
    h->v_done = true;
    return WFSA_OK;
}

extern "C" int wfsa_dev_viterbi(wfsa_dev* h, const double* x, double* logw, int64_t* path_off)
{
    if (!h || !logw || !path_off) return set_err(h, WFSA_ERR_INVALID, "viterbi: bad arguments");
    if (h->n < 0) return set_err(h, WFSA_ERR_STATE, "viterbi before set_param_map");
    if (!x && h->n > 0) return set_err(h, WFSA_ERR_INVALID, "viterbi: bad arguments");
    return decode_paths(h, x, 1, logw, path_off);
}

extern "C" int wfsa_dev_nbest(wfsa_dev* h, const double* x, int32_t k, double* logw, int64_t* path_off)
{
    if (!h || !logw || !path_off || k < 1 || k > kNbestMax) return set_err(h, WFSA_ERR_INVALID, "nbest: bad arguments (k: 1..16)");
    if (h->n < 0) return set_err(h, WFSA_ERR_STATE, "nbest before set_param_map");
    if (!x && h->n > 0) return set_err(h, WFSA_ERR_INVALID, "nbest: bad arguments");
    return decode_paths(h, x, k, logw, path_off);
}

extern "C" int wfsa_dev_sample(wfsa_dev* h, const double* x, int32_t n, uint64_t seed, double* logw, double* logq, int64_t* path_off)
{
    if (!h || !logw || !path_off || n < 1 || n > kSampleMax) return set_err(h, WFSA_ERR_INVALID, "sample: bad arguments (n: 1..256)");
    if (h->n < 0) return set_err(h, WFSA_ERR_STATE, "sample before set_param_map");
    if (!x && h->n > 0) return set_err(h, WFSA_ERR_INVALID, "sample: bad arguments");
    const SampleSpec smp{seed, logq};
    return decode_paths(h, x, n, logw, path_off, &smp);
}

extern "C" int wfsa_dev_viterbi_paths(wfsa_dev* h, int32_t* trans_edge, int32_t* emis_edge)
{
    if (!h || !trans_edge || !emis_edge) return set_err(h, WFSA_ERR_INVALID, "viterbi_paths: bad arguments");
    if (!h->v_done) return set_err(h, WFSA_ERR_STATE, "viterbi_paths before viterbi, nbest or sample");
    CK(cudaSetDevice(h->device));
    const int64_t ns = h->n_strings, k = h->v_k, np = ns * k;
    const std::vector<int64_t>& po = h->h_vpath_off;
    if (!h->v_padded) {
        const size_t steps = (size_t)po[np];
        if (steps) {
            CK(cudaMemcpyAsync(trans_edge, h->d_vtrans.p, steps * 4, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaMemcpyAsync(emis_edge, h->d_vemis.p, steps * 4, cudaMemcpyDeviceToHost, h->stream));
        }
        CK(cudaStreamSynchronize(h->stream));
        return WFSA_OK;
    }
    // rank r of string s was written at k * (offs[s] + s) + r * (len_s + 1): copy the whole range, keep the paths found
    const size_t padded = (size_t)(k * (h->n_tokens + ns));
    std::vector<int32_t> tr(padded), em(padded);
    if (padded) {
        CK(cudaMemcpyAsync(tr.data(), h->d_vtrans.p, padded * 4, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(em.data(), h->d_vemis.p, padded * 4, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    for (int64_t i = 0; i < np; ++i) {
        const int64_t s = i / k, r = i % k, m = po[i + 1] - po[i];
        const int64_t src = k * (h->h_offs[s] + s) + r * (h->h_offs[s + 1] - h->h_offs[s] + 1);
        if (m) {
            std::memcpy(trans_edge + po[i], tr.data() + src, (size_t)m * 4);
            std::memcpy(emis_edge + po[i], em.data() + src, (size_t)m * 4);
        }
    }
    return WFSA_OK;
}

extern "C" int wfsa_dev_hessian(wfsa_dev* h, const double* x, double* Hf, double* rmin)
{
    if (!h || (!Hf && !rmin)) return set_err(h, WFSA_ERR_INVALID, "hessian: bad arguments");
    if (h->n < 0) return set_err(h, WFSA_ERR_STATE, "hessian before set_param_map");
    // rmin only, without path blocks: the (min, +) sweep over every active string, on every kernel (the segmented path
    // when its region types have too many paths for blocks)
    bool sweep_all = false;
    if (h->hb_blocks < 0) {
        if (h->kernel != 6) {
            if (Hf) return set_err(h, WFSA_ERR_STATE, "hessian before set_path_blocks");
            sweep_all = true;
        } else if (Hf || !h->hb_types_failed) {
            CK(cudaSetDevice(h->device));
            const int rc = build_type_blocks(h);          // the segmented path derives the blocks from its region types
            if (rc == WFSA_ERR_LIMIT) h->hb_types_failed = true;
            if (rc == WFSA_ERR_LIMIT && !Hf) sweep_all = true;
            else if (rc != WFSA_OK) return rc;
        } else sweep_all = true;
    }
    int rc = wfsa_dev_upload_x(h, x);
    if (rc != WFSA_OK) return rc;
    if (sweep_all) {
        rc = rmin_sweep(h, true);
        if (rc != WFSA_OK) return rc;
        double rm = 1.0;
        CK(cudaMemcpyAsync(&rm, h->d_rsweep.p, 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaGetLastError());
        if (h->comm) { rm = -rm; const int r2 = wfsa_dev_allreduce_f64(h, &rm, 1, 1); if (r2 != WFSA_OK) return r2; rm = -rm; }
        *rmin = rm;
        return WFSA_OK;
    }
    const size_t nn = Hf ? (size_t)h->n * h->n : 0;          // Hf == NULL: only rmin is wanted, nothing of H is touched
    if (Hf) CK(cudaMemsetAsync(h->d_Hfx.p, 0, std::max<size_t>(nn, 1) * 8, h->stream));
    const double inf = INFINITY;
    CK(cudaMemcpyAsync(h->d_rmin.p, &inf, 8, cudaMemcpyHostToDevice, h->stream));
    const double fx = std::ldexp(1.0, h->hb_fx_log2);
    if (h->hb_blocks > 0) {
        HessParams P{};
        P.n_blocks = h->hb_blocks; P.path_off = h->d_hb_path_off.p; P.col_off = h->d_hb_col_off.p; P.cols = h->d_hb_cols.p;
        P.val_off = h->d_hb_val_off.p; P.counts = h->d_hb_counts.p; P.p = h->d_hb_p.p; P.x = h->d_x.p; P.r_scratch = h->d_hb_r.p;
        P.H_fx = Hf ? h->d_Hfx.p : nullptr; P.rmin = h->d_rmin.p; P.n = h->n; P.fx_scale = fx;
        P.blk_slot = h->hb_from_types ? h->d_hb_slot.p : nullptr; P.slot_lrmin = h->hb_from_types ? h->d_type_lrmin.p : nullptr;
        const int warps_per_block = 8;
        const int64_t blocks = std::min<int64_t>((h->hb_blocks + warps_per_block - 1) / warps_per_block, (int64_t)h->sm_count * 8);
        k5_hessian<<<(int)std::max<int64_t>(blocks, 1), warps_per_block * 32, 0, h->stream>>>(P);
        h->launches++;
    }
    if (Hf) { rc = nccl_allreduce(h, h->d_Hfx.p, nn, ncclUint64, ncclSum); if (rc != WFSA_OK) return rc; }
    if (nn) {
        k_fx_to_double<<<(unsigned)((nn + 255) / 256), 256, 0, h->stream>>>(nn, h->d_Hfx.p, 1.0 / fx, h->d_H.p);
        h->launches++;
        CK(cudaMemcpyAsync(Hf, h->d_H.p, nn * 8, cudaMemcpyDeviceToHost, h->stream));
    }
    double rm = INFINITY;
    if (rmin && h->hb_from_types) {
        // The smallest path posterior of a STRING (the rmin column of the reference, src/HessianLearner.cpp:315) is the
        // product over its regions of their smallest path posteriors: ks_strings adds log rmin_type over the regions of
        // every string (zero table for the bridges), a reduction takes the minimum.
        rc = ensure_ks(h);
        if (rc != WFSA_OK) return rc;
        if (h->ks_groups > 0) {
            if (h->d_zero_logaw.n < (size_t)h->larcs.n_arcs + 16) { CK(h->d_zero_logaw.alloc((size_t)h->larcs.n_arcs + 16)); CK(cudaMemsetAsync(h->d_zero_logaw.p, 0, h->d_zero_logaw.n * 8, h->stream)); }
            KSParams S{};
            S.logaw = h->d_zero_logaw.p; S.words = h->d_kswords.p; S.sgoff = h->d_ksgoff.p; S.gref = h->d_ksgref.p; S.lq = h->d_type_lrmin.p;
            S.p = h->d_ksp.p; S.logq = h->d_kslogq.p; S.n_sgroups = h->ks_groups; S.counter = h->d_seg_counter.p + 1; S.n_arcs = h->larcs.n_arcs;
            CK(cudaMemsetAsync(h->d_seg_counter.p + 1, 0, 4, h->stream));
            CK(cudaMemsetAsync(h->d_kslogq.p, 0, h->d_kslogq.n * 8, h->stream));
            if (h->awg) ks_strings<true><<<h->ks_grid, h->ks_block, 0, h->stream>>>(S); else ks_strings<false><<<h->ks_grid, h->ks_block, h->ks_smem, h->stream>>>(S);
            k_min_exp<<<1, 1024, 0, h->stream>>>((long long)h->d_kslogq.n, h->d_kslogq.p, h->d_rmin.p);
            h->launches += 2;
            h->ks_done = false;                           // the per-string buffer no longer holds log q
        }
    }
    // the overflow strings of the segmented path are not in the per-string layout: the (min, +) sweep of the secondary kernel
    const bool overflow_sweep = rmin && h->hb_from_types && h->n_active_w > 0;
    if (overflow_sweep) { rc = rmin_sweep(h, false); if (rc != WFSA_OK) return rc; }
    CK(cudaMemcpyAsync(&rm, h->d_rmin.p, 8, cudaMemcpyDeviceToHost, h->stream));
    double rm_w = INFINITY;
    if (overflow_sweep) CK(cudaMemcpyAsync(&rm_w, h->d_rsweep.p, 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaGetLastError());
    rm = std::min(rm, rm_w);
    if (rmin) {
        if (h->comm) { rm = -rm; const int r2 = wfsa_dev_allreduce_f64(h, &rm, 1, 1); if (r2 != WFSA_OK) return r2; rm = -rm; }
        *rmin = rm;
    }
    return WFSA_OK;
}

// ---------------------------------------------------------------------------------------------
extern "C" int wfsa_dev_comm_unique_id(void* id_out)
{
    std::string err;
    if (!id_out) return WFSA_ERR_INVALID;
    if (!g_nccl.load(err)) { g_create_error = err; return WFSA_ERR_NCCL; }
    ncclUniqueId id;
    if (g_nccl.GetUniqueId(&id) != ncclSuccess) { g_create_error = "ncclGetUniqueId failed"; return WFSA_ERR_NCCL; }
    static_assert(sizeof(ncclUniqueId) == WFSA_UNIQUE_ID_BYTES, "unique id size");
    std::memcpy(id_out, &id, sizeof(id));
    return WFSA_OK;
}

extern "C" int wfsa_dev_comm_init(wfsa_dev* h, const void* id, int rank, int nranks)
{
    if (!h || !id || nranks < 1 || rank < 0 || rank >= nranks) return set_err(h, WFSA_ERR_INVALID, "comm_init: bad arguments");
    if (nranks == 1) return WFSA_OK;
    std::string err;
    if (!g_nccl.load(err)) return set_err(h, WFSA_ERR_NCCL, err);
    CK(cudaSetDevice(h->device));
    ncclUniqueId uid;
    std::memcpy(&uid, id, sizeof(uid));
    const int r = g_nccl.CommInitRank(&h->comm, nranks, uid, rank);
    if (r != ncclSuccess) { h->comm = nullptr; return set_err(h, WFSA_ERR_NCCL, "ncclCommInitRank failed"); }
    h->rank = rank; h->nranks = nranks;
    return WFSA_OK;
}

extern "C" int wfsa_dev_allreduce_f64(wfsa_dev* h, double* values, int n, int op)
{
    if (!h || n < 0 || (n && !values)) return set_err(h, WFSA_ERR_INVALID, "allreduce_f64: bad arguments");
    if (!h->comm || n == 0) return WFSA_OK;
    CK(cudaSetDevice(h->device));
    DevBuf<double> tmp;
    CK(tmp.alloc(n));
    CK(cudaMemcpyAsync(tmp.p, values, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
    const int rc = nccl_allreduce(h, tmp.p, n, 8 /* ncclFloat64 */, op == 1 ? ncclMax : ncclSum);
    if (rc != WFSA_OK) return rc;
    CK(cudaMemcpyAsync(values, tmp.p, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return WFSA_OK;
}

// In-kernel phase times of k_eval6 (globaltimer stamps of CTA 0): ns spent in [weights, region types, grid barrier, fold +
// exchange], summed over the evaluations since the last reset.
extern "C" int wfsa_dev_eval6_phases(wfsa_dev* h, double* out4, int reset)
{
    if (!h || !out4) return WFSA_ERR_INVALID;
    out4[0] = out4[1] = out4[2] = out4[3] = 0.0;
    if (!h->d_e6stamps.p) return WFSA_OK;
    CK(cudaSetDevice(h->device));
    unsigned long long v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    CK(cudaMemcpyAsync(v, h->d_e6stamps.p, 64, cudaMemcpyDeviceToHost, h->stream));
    if (reset) CK(cudaMemsetAsync(h->d_e6stamps.p, 0, 64, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (getenv("WFSA_E6_DEBUG"))
        fprintf(stderr, "[k_eval6 debug] longest group %.2f us (rows code 0x%x), latest end of the region phase %.2f us after the start of CTA 0, longest wait for staged words %.2f us\n",
                (double)(v[4] >> 32) * 1e-3, (unsigned)(v[4] & 0xffffffffu), (double)v[5] * 1e-3, (double)v[7] * 1e-3);
    if (getenv("WFSA_E6_DEBUG") && (atoi(getenv("WFSA_E6_DEBUG")) & 16) && h->seg_grid <= 1024) {
        // per-CTA timeline of the last launch: when each phase ended, relative to the earliest CTA start
        std::vector<unsigned long long> tl((size_t)h->seg_grid * 8);
        CK(cudaMemcpy(tl.data(), h->d_e6stamps.p + 8, tl.size() * 8, cudaMemcpyDeviceToHost));
        unsigned long long t0 = ~0ull;
        for (int b = 0; b < h->seg_grid; ++b) t0 = std::min(t0, tl[(size_t)b * 8]);
        const char* nm[5] = {"start", "weights done", "regions done", "barrier passed", "end"};
        for (int k = 0; k < 5; ++k) {
            double mn = 1e30, mx = 0, sum = 0; int amx = 0;
            for (int b = 0; b < h->seg_grid; ++b) { const double d = (double)(tl[(size_t)b * 8 + k] - t0) * 1e-3; if (d < mn) mn = d; if (d > mx) { mx = d; amx = b; } sum += d; }
            fprintf(stderr, "[k_eval6 timeline] %-14s min %7.2f  mean %7.2f  max %7.2f us (CTA %d)\n", nm[k], mn, sum / h->seg_grid, mx, amx);
        }
        if (atoi(getenv("WFSA_E6_DEBUG")) & 32) {             // every CTA: time from the grid barrier to its end (fold + exchange)
            std::string line = "[k_eval6 timeline] rank " + std::to_string(h->rank) + " fold+exchange us per CTA:";
            char buf[32];
            for (int b = 0; b < h->seg_grid; ++b) { snprintf(buf, sizeof buf, " %.1f", (double)(tl[(size_t)b * 8 + 4] - tl[(size_t)b * 8 + 3]) * 1e-3); line += buf; }
            fprintf(stderr, "%s\n", line.c_str());
        }
    }
    for (int i = 0; i < 4; ++i) out4[i] = (double)v[i];
    return WFSA_OK;
}

extern "C" int wfsa_dev_timer_begin(wfsa_dev* h)
{
    if (!h) return WFSA_ERR_INVALID;
    h->timing = true; h->kev.used = 0; h->sev.used = 0; h->timing_detail = true;
    CK(cudaEventRecord(h->ev_begin, h->stream));
    return WFSA_OK;
}

// Like timer_begin, but only the event pair around each whole evaluation is recorded: no events between the kernels
// of an evaluation, so they keep their dependent launches (timer_kernel_ms / split / phase then report nothing).
extern "C" int wfsa_dev_timer_begin_steps(wfsa_dev* h)
{
    const int rc = wfsa_dev_timer_begin(h);
    if (rc == WFSA_OK) h->timing_detail = false;
    return rc;
}

extern "C" int wfsa_dev_timer_end(wfsa_dev* h, float* ms)
{
    if (!h) return WFSA_ERR_INVALID;
    CK(cudaEventRecord(h->ev_end, h->stream));
    CK(cudaEventSynchronize(h->ev_end));
    h->timing = false;
    if (ms) CK(cudaEventElapsedTime(ms, h->ev_begin, h->ev_end));
    return WFSA_OK;
}

extern "C" int wfsa_dev_timer_kernel_ms(wfsa_dev* h, float* ms, int64_t* launches)
{
    if (!h) return WFSA_ERR_INVALID;
    float total = 0.f;
    for (size_t i = 0; i < h->kev.used; ++i) {
        const TimedSlot& s = h->kev.slots[i];
        float t = 0.f;
        CK(cudaEventSynchronize(s.end));
        CK(cudaEventElapsedTime(&t, s.begin, s.end));
        total += t;
    }
    if (ms) *ms = total;
    if (launches) *launches = (int64_t)h->kev.used;
    return WFSA_OK;
}

extern "C" int wfsa_dev_timer_step_ms(wfsa_dev* h, float* ms, int64_t* steps)
{
    if (!h) return WFSA_ERR_INVALID;
    float total = 0.f;
    for (size_t i = 0; i < h->sev.used; ++i) {
        const TimedSlot& s = h->sev.slots[i];
        float t = 0.f;
        CK(cudaEventSynchronize(s.end));
        CK(cudaEventElapsedTime(&t, s.begin, s.end));
        total += t;
    }
    if (ms) *ms = total;
    if (steps) *steps = (int64_t)h->sev.used;
    return WFSA_OK;
}

__global__ void k_read_sweep(const uint4* __restrict__ p, size_t n, unsigned int* sink)
{
    unsigned int s = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) { const uint4 v = p[i]; s ^= v.x ^ v.y ^ v.z ^ v.w; }
    if (s == 0x12345677u) *sink = s;      // never true for a memset pattern: keeps the loads alive
}

// Evicts the L2 between two timed evaluations: a memset of a buffer twice the size of the L2 on the evaluation
// stream (it runs between the per-evaluation event pairs of wfsa_dev_timer_step_ms, not inside them).
extern "C" int wfsa_dev_l2_flush(wfsa_dev* h)
{
    if (!h) return WFSA_ERR_INVALID;
    CK(cudaSetDevice(h->device));
    if (!h->d_flush.p) {
        int l2 = 0;
        CK(cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, h->device));
        CK(h->d_flush.alloc(2 * (size_t)std::max(l2, 64 << 20)));
        CK(h->d_flush_sink.alloc(1));
    }
    h->flush_byte ^= 1;
    CK(cudaMemsetAsync(h->d_flush.p, h->flush_byte, h->d_flush.n, h->stream));
    if (!getenv("WFSA_FLUSH_WRITE_ONLY")) {
        // the memset leaves the L2 full of DIRTY lines: the first misses of the next kernel would each wait for a write-back
        // (measured: DRAM round trips of ~5 us instead of ~1.5 us for the first 20 us of the evaluation).  A read sweep over
        // the same buffer replaces them with clean lines of unrelated data: the L2 is just as cold for the evaluation.
        k_read_sweep<<<h->sm_count * 4, 512, 0, h->stream>>>(reinterpret_cast<const uint4*>(h->d_flush.p), h->d_flush.n / 16, h->d_flush_sink.p);
        h->launches++;
    }
    return WFSA_OK;
}

// [0] from the start of an evaluation to the dominant kernel(s) (weights, resets), [1] the dominant kernel(s),
// [2] from there to the end of the evaluation (fold, collective, conversion); sums over the evaluations since timer_begin
extern "C" int wfsa_dev_timer_phase_ms(wfsa_dev* h, float* out3)
{
    if (!h || !out3) return WFSA_ERR_INVALID;
    out3[0] = out3[1] = out3[2] = 0.f;
    const size_t n = std::min(h->sev.used, h->kev.used);
    for (size_t i = 0; i < n; ++i) {
        const TimedSlot &s = h->sev.slots[i], &k = h->kev.slots[i];
        float t = 0.f;
        CK(cudaEventSynchronize(s.end));
        if (cudaEventElapsedTime(&t, s.begin, k.begin) == cudaSuccess) out3[0] += t;
        if (cudaEventElapsedTime(&t, k.begin, k.end) == cudaSuccess) out3[1] += t;
        if (cudaEventElapsedTime(&t, k.end, s.end) == cudaSuccess) out3[2] += t;
    }
    cudaGetLastError();
    return WFSA_OK;
}

// Lines the ranks of the communicator up on the evaluation stream (benchmark helper, see wfsa_dev.h).
extern "C" int wfsa_dev_rank_barrier(wfsa_dev* h)
{
    if (!h) return WFSA_ERR_INVALID;
    if (!h->comm || h->nranks <= 1) return WFSA_OK;
    CK(cudaSetDevice(h->device));
    if (h->peer_ok) {
        PeerBarrierParams B{};
        for (int r = 0; r < h->nranks; ++r) B.peers[r] = h->peer_ptrs[r];
        B.bar_off = h->peer_bar_off; B.nranks = h->nranks; B.rank = h->rank; B.epoch = ++h->peer_bar_epoch;
        k_peer_barrier<<<1, 32, 0, h->stream>>>(B);
        h->launches++;
        CK(cudaGetLastError());
        return WFSA_OK;
    }
    if (!h->d_bar.p) { CK(h->d_bar.alloc(1)); CK(cudaMemsetAsync(h->d_bar.p, 0, 8, h->stream)); }
    return nccl_allreduce(h, h->d_bar.p, 1, ncclUint64, ncclSum);
}

extern "C" int wfsa_dev_timer_split_ms(wfsa_dev* h, float* first_ms, float* second_ms)
{
    if (!h) return WFSA_ERR_INVALID;
    float a = 0.f, b = 0.f;
    if (h->kernel == 6)
        for (size_t i = 0; i < h->kev.used; ++i) {
            const TimedSlot& k = h->kev.slots[i];
            if (!k.mid) continue;
            float t = 0.f;
            CK(cudaEventSynchronize(k.end));
            if (cudaEventElapsedTime(&t, k.begin, k.mid) == cudaSuccess) a += t;
            if (cudaEventElapsedTime(&t, k.mid, k.end) == cudaSuccess) b += t;
        }
    cudaGetLastError();
    if (first_ms) *first_ms = a;
    if (second_ms) *second_ms = b;
    return WFSA_OK;
}

extern "C" int wfsa_lattice_compile(const wfsa_fsa_desc* fd, const int32_t* trimmed, const int32_t* tokens, int32_t len,
                                    int32_t n_slots, uint32_t* words, int64_t capacity, int64_t* n_words,
                                    int32_t* arc_tid, int32_t* arc_eid, int32_t arc_capacity, int32_t* n_arcs)
{
    g_create_error.clear();
    if (!fd || len < 0 || (len && !tokens) || !n_words || n_slots < 1 || n_slots > kLatMaxSlots) { g_create_error = "lattice_compile: bad arguments"; return WFSA_ERR_INVALID; }
    HostFsa f; GenericLayout g; LatticeArcs A;
    int status = WFSA_OK;
    std::string msg = copy_and_validate(fd, f, status);
    if (status == WFSA_OK) msg = build_generic_layout(f, g, status);
    if (status != WFSA_OK) { g_create_error = msg; return status; }
    build_lattice_arcs(f, g, A);
    if (A.n_arcs >= (1 << kLatArcBits)) { g_create_error = "lattice_compile: too many combined arcs"; return WFSA_ERR_LIMIT; }
    if (n_arcs) *n_arcs = A.n_arcs;
    if (arc_tid && arc_eid) {
        if (arc_capacity < A.n_arcs) { g_create_error = "lattice_compile: arc_capacity too small"; return WFSA_ERR_INVALID; }
        std::copy(A.arc_tid.begin(), A.arc_tid.end(), arc_tid);
        std::copy(A.arc_eid.begin(), A.arc_eid.end(), arc_eid);
    }
    std::vector<uint8_t> alive((size_t)A.n_arcs, 1);
    if (trimmed)
        for (int a = 0; a < A.n_arcs; ++a) {
            const int tp = f.trans_param[A.arc_tid[a]], ep = A.arc_eid[a] < 0 ? -1 : f.emis_param[A.arc_eid[a]];
            alive[a] = (tp < 0 || trimmed[tp] != -2) && (ep < 0 || trimmed[ep] != -2);
        }
    LatticeScratch S;
    std::vector<uint32_t> w;
    std::vector<int32_t> bridges;
    const int rc = compile_lattice(f, A, alive.data(), tokens, len, n_slots, S, w, bridges);
    if (rc != 1) { *n_words = rc; return WFSA_OK; }
    if ((int64_t)w.size() > capacity || !words) { g_create_error = "lattice_compile: capacity too small"; *n_words = (int64_t)w.size(); return WFSA_ERR_INVALID; }
    std::copy(w.begin(), w.end(), words);
    *n_words = (int64_t)w.size();
    return WFSA_OK;
}

struct wfsa_segmented {
    SegmentedCorpus sc;
    LatticeArcs arcs;
    std::vector<int64_t> stats;
    TypeBlocks blocks;                          // what wfsa_dev_hessian derives from the region types
};

extern "C" int wfsa_segmented_compile(const wfsa_fsa_desc* fd, const wfsa_corpus_desc* cd, const int32_t* trimmed,
                                      int32_t n_slots, double fx_scale, wfsa_segmented** out)
{
    g_create_error.clear();
    if (!fd || !cd || !out || (n_slots & 63) < 1 || (n_slots & 63) > kLatMaxSlots || cd->n_strings < 0) { g_create_error = "segmented_compile: bad arguments"; return WFSA_ERR_INVALID; }   // bit 6: DAG form only
    *out = nullptr;
    HostFsa f; GenericLayout g;
    int status = WFSA_OK;
    std::string msg = copy_and_validate(fd, f, status);
    if (status == WFSA_OK) msg = build_generic_layout(f, g, status);
    if (status != WFSA_OK) { g_create_error = msg; return status; }
    wfsa_segmented* s = new wfsa_segmented();
    build_lattice_arcs(f, g, s->arcs);
    const LatticeArcs& A = s->arcs;
    if (A.n_arcs >= 65520 || A.n_arcs >= (1 << kLatArcBits)) { delete s; g_create_error = "segmented_compile: too many combined arcs"; return WFSA_ERR_LIMIT; }
    std::vector<uint8_t> alive((size_t)A.n_arcs, 1);
    if (trimmed)
        for (int a = 0; a < A.n_arcs; ++a) {
            const int tp = f.trans_param[A.arc_tid[a]], ep = A.arc_eid[a] < 0 ? -1 : f.emis_param[A.arc_eid[a]];
            alive[a] = (tp < 0 || trimmed[tp] != -2) && (ep < 0 || trimmed[ep] != -2);
        }
    std::vector<int32_t> ids((size_t)cd->n_strings);
    std::iota(ids.begin(), ids.end(), 0);
    std::stable_sort(ids.begin(), ids.end(), [&](int32_t a, int32_t b) {
        return (cd->offsets[a + 1] - cd->offsets[a]) > (cd->offsets[b + 1] - cd->offsets[b]);
    });
    compile_corpus_segmented(f, A, alive.data(), cd->tokens, cd->offsets, cd->p, ids, n_slots, fx_scale, s->sc);
    int64_t blocks_omitted = 0;
    {   // H_f blocks in the numbering of `trimmed` (raw parameter ids when trimmed is NULL)
        std::vector<int32_t> ttp(f.n_trans()), etp(f.n_emis());
        for (int t = 0; t < f.n_trans(); ++t) ttp[t] = f.trans_param[t] < 0 ? -1 : (trimmed ? trimmed[f.trans_param[t]] : f.trans_param[t]);
        for (int e = 0; e < f.n_emis(); ++e) etp[e] = f.emis_param[e] < 0 ? -1 : (trimmed ? trimmed[f.emis_param[e]] : f.emis_param[e]);
        const OverflowStrings ov{&f, alive.data(), cd->tokens, cd->offsets, cd->p, &s->sc.overflow};
        make_type_blocks(A, ttp, etp, s->sc.rwords, s->sc.rgoff, s->sc.rgrows, s->sc.typeW, ov, s->blocks);
        // the evaluation does not need the blocks: a region type with too many paths leaves them out (zero blocks), not the shard
        if (!s->blocks.fail.empty()) { s->blocks = TypeBlocks(); blocks_omitted = 1; }
    }
    s->stats = {s->sc.n_types, s->sc.n_region_instances, s->sc.n_region_edges, s->sc.n_type_edges, s->sc.n_bridge, s->sc.n_strings,
                (int64_t)(s->sc.host_ms * 1000.0), blocks_omitted};
    *out = s;
    return WFSA_OK;
}

extern "C" int wfsa_segmented_get(const wfsa_segmented* s, int which, const void** data, int64_t* count)
{
    if (!s || !data || !count) return WFSA_ERR_INVALID;
    const SegmentedCorpus& c = s->sc;
#define SEG_ARR(i, v) case i: *data = (v).data(); *count = (int64_t)(v).size(); return WFSA_OK;
    switch (which) {
        SEG_ARR(0, c.rwords) SEG_ARR(1, c.rgoff) SEG_ARR(2, c.rgrows) SEG_ARR(3, c.typeW) SEG_ARR(4, c.swords) SEG_ARR(5, c.sgoff)
        SEG_ARR(6, c.sgref) SEG_ARR(7, c.ksid) SEG_ARR(8, c.kp) SEG_ARR(9, c.overflow) SEG_ARR(10, c.rejected) SEG_ARR(11, c.const_acc)
        SEG_ARR(12, s->stats) SEG_ARR(13, s->blocks.po) SEG_ARR(14, s->blocks.co) SEG_ARR(15, s->blocks.vo) SEG_ARR(16, s->blocks.cols)
        SEG_ARR(17, s->blocks.counts) SEG_ARR(18, s->blocks.bp) SEG_ARR(19, s->blocks.slots) SEG_ARR(20, c.pwords) SEG_ARR(21, c.pgoff)
        default: return WFSA_ERR_INVALID;
    }
#undef SEG_ARR
}

extern "C" void wfsa_segmented_free(wfsa_segmented* s) { delete s; }

extern "C" int wfsa_dev_get_info(wfsa_dev* h, wfsa_dev_info* info)
{
    if (!h || !info) return WFSA_ERR_INVALID;
    std::memset(info, 0, sizeof(*info));
    info->kernel = h->kernel; info->accum_mode = h->accum;
    info->n_trans = h->fsa.n_trans(); info->n_emis = h->fsa.n_emis();
    info->n_arcs = h->fast.ok ? h->fast.n_arcs : 0; info->n_slots = h->fast.ok ? h->fast.n_slots : 0;
    info->max_candidates = h->fast.ok ? h->fast.max_cand : 0;
    info->sm_count = h->sm_count;
    info->grid = h->kernel == 6 ? h->seg_grid : (h->kernel == 4 ? h->kt_grid : (h->kernel == 2 ? h->k3_grid : h->grid));
    info->block = h->kernel == 6 ? h->seg_block : (h->kernel == 4 ? h->kt_block : (h->kernel == 2 ? h->k3_block : (h->kernel == 3 ? 128 : h->block)));
    if (h->kernel == 7) { info->grid = 0; info->block = h->k7_V; }
    info->n_strings = h->n_strings; info->n_tokens = h->n_tokens;
    info->n_active_tokens = h->n_active_tokens;
    info->smem_bytes = (int64_t)(h->kernel == 6 ? h->seg_smem : (h->kernel == 4 ? h->kt_smem : (h->kernel == 2 ? h->k3_smem : h->smem_bytes)));
    if (h->kernel == 7) { info->smem_bytes = (int64_t)kK7Chunk * h->k7_V * 8; info->seg_host_ms = h->k7_host_ms; info->lattice_words = (int64_t)h->k7_rows * h->k7_V * 2; info->pool_slots = (int32_t)h->k7.size(); }
    if (h->kernel == 6) {
        { const int rc = ensure_ks(h); if (rc != WFSA_OK) return rc; }     // word counts and compile time include the per-string layout
        info->n_arcs = h->larcs.n_arcs;
        info->lattice_words = h->seg_words; info->lattice_edges = h->seg_bridges + h->seg_region_edges;
        info->lattice_bridge_edges = h->seg_bridges; info->n_overflow_strings = h->n_active_w; info->pool_slots = h->seg_slots;
        info->seg_types = h->seg_types; info->seg_region_instances = h->seg_instances; info->seg_region_edges = h->seg_region_edges;
        info->seg_type_edges = h->seg_type_edges; info->seg_host_ms = h->seg_host_ms;
        if (h->n >= 0) {                                           // the conditions of k_eval6's P1 (kernels_eval6.cuh)
            info->e6_big_groups = h->kr_big_groups; info->e6_big_dedicate = eval6_big_dedicate(h);
            info->e6_big_slots = h->e6_big_slots; info->e6_big_rows = h->e6_big_rows; info->e6_max_big_rows = (int32_t)h->seg_max_big_rows;
            int two = 0;
            if (h->kr_big_groups <= h->seg_grid && h->e6_big_slots >= 2)
                for (int64_t b = 0; b < h->kr_big_groups; ++b)
                    two += (h->hrgoff[b + 1] - h->hrgoff[b]) >> 5 <= h->e6_big_rows && !(h->hrgrows[b] & 0x10000);
            info->e6_two_warp_eligible = two;
        }
    }
    info->n_active_strings = h->n_active + h->n_active_w; info->table_bytes = (int64_t)h->table_bytes;
    info->kernels_launched = h->launches; info->fixed_point_scale_log2 = h->fx_log2;
    {
        const bool single = h->kernel == 6 && h->e6_ok && !h->any_overflow && h->n >= 0;
        info->eval_path = (single ? 1 : 0) | (single && h->comm ? 2 : 0) | (!single && h->comm ? 4 : 0) | (h->any_overflow ? 8 : 0);
    }
    return WFSA_OK;
}
