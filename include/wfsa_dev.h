/* include/wfsa_dev.h -- C ABI of the B200 evaluation backend for w-fsa.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no FFI layer: the
 * hot path sits behind C++ member functions of `Learner` that share protected vectors
 * (/root/reference/inc/Learner.h:24,54,56,65,83,89-102,143-168).  Each entry point below
 * names the reference member(s) it replaces.  Plain pointers and sizes only; no C++ or torch
 * types cross this line; nothing throws; every call returns a wfsa_status.
 *
 * Data contracts (same as the reference):
 *   - x holds natural-log weights of the TRIMMED parameters (src/Learner.cpp:350-436);
 *   - p is normalised over the WHOLE corpus, unrecognised strings included (src/main.cpp:154);
 *   - per-string outputs are in the caller's string order (corpus order of this shard).
 * Ownership: the caller owns every host buffer; descriptors are copied at create time;
 * the backend owns all device memory.  Calls are synchronous unless named *_launch and a
 * handle is not re-entrant.
 */
#ifndef WFSA_DEV_H
#define WFSA_DEV_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    WFSA_OK = 0,
    WFSA_ERR_INVALID = 1,      /* bad argument / inconsistent descriptor                     */
    WFSA_ERR_CUDA = 2,         /* CUDA runtime error (message via wfsa_dev_last_error)       */
    WFSA_ERR_NO_DEVICE = 3,    /* no usable sm_100 device: there is NO CPU fallback          */
    WFSA_ERR_EPS_CYCLE = 4,    /* empty-emission cycle: path sum diverges (reference loops)  */
    WFSA_ERR_STATE = 5,        /* call order violated (e.g. eval before set_param_map)       */
    WFSA_ERR_LIMIT = 6,        /* automaton exceeds a compiled limit                         */
    WFSA_ERR_NCCL = 7,         /* NCCL unavailable or failed                                 */
    WFSA_ERR_NOMEM = 8
} wfsa_status;

/* Lowered automaton: what replaces Fsa::State / NamedProb / NextState
 * (inc/Fsa.h:26-66).  States are dense ids; an emission is a sequence of 0..L tokens
 * (the reference's emission strings, possibly empty); the emission consumed on a step is the
 * one of the TARGET state (inc/Recognize.h:49-57).  Edge parameter ids follow
 * Fsa::AssignIndices (src/Fsa.cpp:207-238): -1 for the single emission / single transition
 * of a state, otherwise a raw parameter id in [0, n_raw_params). */
typedef struct {
    int32_t n_states;            /* including start and end                                  */
    int32_t start_state;
    int32_t end_state;
    int32_t n_symbols;           /* tokens are in [0, n_symbols); <0 in a corpus = unknown   */
    int32_t n_raw_params;
    const int32_t* emis_row;     /* [n_states+1] CSR of emission edges by state              */
    const int32_t* emis_tok_off; /* [n_emis+1]   token range of each emission edge           */
    const int32_t* emis_tok;     /* [emis_tok_off[n_emis]]                                   */
    const int32_t* emis_param;   /* [n_emis]     raw parameter id or -1                      */
    const int32_t* trans_row;    /* [n_states+1] CSR of transition edges by source state     */
    const int32_t* trans_dst;    /* [n_trans]                                                */
    const int32_t* trans_param;  /* [n_trans]    raw parameter id or -1                      */
} wfsa_fsa_desc;

/* Packed corpus shard: replaces Corpus = vector<pair<string,double>> (inc/Corpus.h:16). */
typedef struct {
    int64_t n_strings;
    const int64_t* offsets;      /* [n_strings+1] */
    const int32_t* tokens;       /* [offsets[n_strings]] */
    const double*  p;            /* [n_strings] normalised over the whole corpus */
} wfsa_corpus_desc;

typedef struct {
    int32_t device;              /* CUDA device ordinal                                       */
    int32_t force_kernel;        /* 0 auto, 1 warp-per-string, 2 CTA-per-string, 3 generic,
                                    4 thread-per-string (table walk),
                                    6 segmented compiled lattices (bridges folded into constants + region types),
                                    7 position-synchronous, pair-batched (dense automata: more than 32 states emit one symbol) */
    int32_t accum_mode;          /* 0 auto, 1 shared-memory accumulators, 2 global (L2) REDs  */
    int32_t reserved;
} wfsa_dev_options;

typedef struct wfsa_dev wfsa_dev;

/* Builds the device layout (combined arcs in CSR by (state, symbol), packed int32 tokens in
 * length buckets) and uploads it.  Replaces the data side of Learner::BuildFrom
 * (src/Learner.cpp:269-274) and Learner::Finalize's MKL handle creation (:483-485). */
int wfsa_dev_create(const wfsa_fsa_desc* fsa, const wfsa_corpus_desc* corpus,
                    const wfsa_dev_options* opt, wfsa_dev** out);

/* Structural pass: replaces Learner::BuildPaths' recognition loop
 * (src/Learner.cpp:276-348 driving inc/Recognize.h:62-96).  recognised[s] = 1 iff the string
 * has an accepting path; path_count[s] = number of accepting paths (a double; the DP counts,
 * it does not enumerate); param_used[i] = 1 iff raw parameter i lies on an accepting path of
 * some string of this shard (feeds Learner::Trim, :350-425).  Any pointer may be NULL.
 * The pass reuses the evaluation's string-order buffers: a parameter map set earlier is void
 * afterwards (evaluations return WFSA_ERR_STATE until wfsa_dev_set_param_map is called again). */
int wfsa_dev_structure(wfsa_dev* h, uint8_t* recognised, double* path_count, uint8_t* param_used);

/* trimmed[i] for every raw parameter: -2 unused (weight exp(-inf)=0), -1 pinned (weight 1),
 * otherwise index into x (src/Learner.cpp:427-436).  n = number of trimmed parameters.
 * recognised (or NULL = all) selects the strings that take part in evaluations; with several
 * ranks it must be called after the used-flags were combined across ranks. */
int wfsa_dev_set_param_map(wfsa_dev* h, const int32_t* trimmed, int32_t n, const uint8_t* recognised);

/* One evaluation = Learner::ComputeModeledProbs + ComputeObjective (src/Learner.cpp:515-553)
 * + {QuasiNewton,Hessian}Learner::ComputeGrad (src/QuasiNewtonLearner.cpp:93-125,
 * src/HessianLearner.cpp:565-597):
 *   loglik = sum_s p_s log q_s   (KL = plogp - loglik),   grad_i = -sum_s p_s E_s[count_i].
 * With a communicator attached both are the sums over ALL ranks.  logq (may be NULL) receives
 * log q_s of this shard's strings, -inf/NaN-free only for recognised strings (others: -inf).
 * logq is the reference's protected intermediate (inc/Learner.h:95), not needed for the objective or the
 * gradient: with NULL the segmented path skips its per-string pass altogether (it runs on demand, also from a
 * later wfsa_dev_eval_fetch with a logq buffer, for the evaluation launched last). */
int wfsa_dev_eval(wfsa_dev* h, const double* x, double* loglik, double* logq, double* grad);

/* Same evaluation with x already resident (last uploaded x); results stay on the device.
 * Used for kernel-only timing and by callers that pipeline their own copies. */
int wfsa_dev_upload_x(wfsa_dev* h, const double* x);
int wfsa_dev_eval_launch(wfsa_dev* h);           /* asynchronous on the handle's stream */
int wfsa_dev_eval_fetch(wfsa_dev* h, double* loglik, double* logq, double* grad);
int wfsa_dev_sync(wfsa_dev* h);

/* H_f block of HessianLearner::ComputeHf (src/HessianLearner.cpp:498-547):
 *   Hf[j*n+k] = sum_s p_s ( g_j g_k - sum_pi r_pi P_pij P_pik ),  full symmetric n x n, row major.
 * Paths of ambiguous strings are supplied as dense count blocks: for block b,
 * rows = paths, cols = the block's parameter list.  */
typedef struct {
    int64_t n_blocks;
    const int64_t* path_off;     /* [n_blocks+1] paths of block b: path_off[b]..path_off[b+1]   */
    const int64_t* col_off;      /* [n_blocks+1] parameter list of block b                       */
    const int32_t* cols;         /* [col_off[n_blocks]] trimmed parameter ids                    */
    const int64_t* val_off;      /* [n_blocks+1] start of block b's row-major (paths x cols) data */
    const double*  counts;       /* [val_off[n_blocks]]                                          */
    const double*  p;            /* [n_blocks] p_s of the block's string                         */
} wfsa_path_blocks;
int wfsa_dev_set_path_blocks(wfsa_dev* h, const wfsa_path_blocks* blocks);
/* rmin = the smallest path posterior over all strings of all ranks, min_s min_pi w(pi) / q_s (at most 1; 1 when no string
 * has a choice).  Where it comes from:
 *   - blocks set by wfsa_dev_set_path_blocks: from the blocks (Hf needs them on every kernel but the segmented one);
 *   - no blocks, Hf == NULL, any kernel: no enumeration -- a forward sweep in the (min, +) semiring over the lattice of the
 *     evaluation gives m_s = min_pi log w(pi), and r_s = exp(m_s - log q_s);
 *   - segmented kernel (6) without blocks: blocks and per-string minima from the compiled region types; the strings
 *     that no type covers (more live lattice nodes than pool slots) add one block per segment of their lattice to H and
 *     are taken into rmin by the sweep.  When a region type or such a segment has more than 2^20 paths an rmin-only call
 *     sweeps every string, a call with Hf returns WFSA_ERR_LIMIT (never a partial H).
 * H is summed in 64-bit fixed point whose range is sized from sum_b p_b * cmax_b^2 over the blocks of all ranks (cmax_b =
 * largest |count| of block b); WFSA_ERR_LIMIT when that sum reaches 2^50.
 * Without blocks a call with Hf != NULL returns WFSA_ERR_STATE on the other kernels.  Collective with a communicator.
 * The (min, +) sweep gives the weight of the least probable path; the most probable path itself, of every string, comes
 * from wfsa_dev_viterbi below. */
int wfsa_dev_hessian(wfsa_dev* h, const double* x, double* Hf /* n*n, or NULL: only rmin is computed */, double* rmin /* or NULL */);

/* Most probable accepting path of every string of this shard (Viterbi), at x (trimmed parameters, as wfsa_dev_eval):
 *   logw[s] = max over accepting paths pi of s of the summed log weights of pi's edges  (-inf: no accepting path under
 *             the parameter map and x, or the string does not take part in evaluations);
 *   path_off[s]..path_off[s+1]: the steps of that path (path_off: n_strings + 1 entries; 0 steps when logw[s] = -inf).
 * logw[s] is the left-to-right sum of the log weights of the steps (transition, then emission, ..., final transition), bit
 * for bit.  Ties are broken deterministically (same bits on every call).  The paths stay on the device until the next
 * wfsa_dev_viterbi, wfsa_dev_nbest, wfsa_dev_sample or wfsa_dev_destroy.  Local to the shard: no collective, also with a communicator attached.  The call
 * keeps its own copy of x: it changes nothing an evaluation returns, also between wfsa_dev_eval_launch and
 * wfsa_dev_eval_fetch.  WFSA_ERR_STATE before wfsa_dev_set_param_map. */
int wfsa_dev_viterbi(wfsa_dev* h, const double* x, double* logw, int64_t* path_off);
/* The k most probable accepting paths of every string of this shard (N-best), 1 <= k <= 16, at x; path i = s * k + r is the
 * r-th most probable path of string s (r = 0: the best):
 *   logw[i] = summed log weight of that path (-inf, and 0 steps, when s has at most r paths, or none under the parameter
 *             map and x, or does not take part in evaluations); non-increasing in r;
 *   path_off[i]..path_off[i+1]: its steps (path_off: n_strings * k + 1 entries).
 * The k paths of a string are pairwise distinct step sequences.  Summation order is wfsa_dev_viterbi's, so logw[i] is the
 * left-to-right sum of the log weights of the steps, bit for bit, and the values do not depend on the kernel.  Ties: a
 * node keeps the first strictly larger candidates, in the order (fent entry, source rank) with fast tables and (source
 * state in eps_order, transition, emission, source rank) otherwise; the end in the order (candidate slot, rank),
 * respectively (source state, transition, rank).  So rank 0 is the path and value of wfsa_dev_viterbi, bit for bit, and k = 1
 * is wfsa_dev_viterbi.  Same bits on every call.  Local to the shard and without effect on evaluations, as
 * wfsa_dev_viterbi.  WFSA_ERR_INVALID: k outside 1..16 or a null pointer; WFSA_ERR_STATE before wfsa_dev_set_param_map;
 * WFSA_ERR_LIMIT when the handle decodes a CTA per string (more than 32 candidates per symbol) and the lists of its
 * candidates at this k do not fit a CTA: 2 * K * G doubles of shared memory (K the power of two >= k, G the candidates
 * rounded up to 32) over the device's opt-in limit, or, at K = 16, G over 768 threads; a smaller k may fit. */
int wfsa_dev_nbest(wfsa_dev* h, const double* x, int32_t k, double* logw /* [n_strings*k] */, int64_t* path_off /* [n_strings*k + 1] */);
/* n independent draws from p(pi | s) = w(pi) / q_s for every string of this shard, 1 <= n <= 256, at x; path i = s * n + r is
 * draw r of string s:
 *   logw[i] = summed log weight of the draw's steps, the left-to-right sum (acc + log a) + log b of wfsa_dev_viterbi, bit
 *             for bit, so a draw that is also an N-best path has that path's wfsa_dev_nbest value (-inf, and 0 steps, for
 *             every draw of a string without a path under the parameter map and x, or that does not take part in
 *             evaluations);
 *   logq[s] = log q_s from the sampler's own forward sweep, as the evaluation's log q (logq may be NULL);
 *   path_off[i]..path_off[i+1]: the draw's steps (path_off: n_strings * n + 1 entries), through wfsa_dev_viterbi_paths.
 * Randomness: Philox4x32-10 (wfsa_philox4x32_10 of wfsa_host.h) under the key (seed & 0xffffffff, seed >> 32); choice d of
 * draw r of string s (s the shard's string index, d counted from 0 within the draw) uses the counter (d, r, s, 0) and
 * u = ((o0 << 32 | o1) >> 11) * 2^-53.  At a node the draw takes the first entry, in table order, whose running sum exceeds
 * u * total; when rounding leaves none, the last entry of positive weight.  Draw r of string s is therefore a function of
 * (automaton, parameter map, x, seed, s, r) only: the first m draws of a call with n > m are the draws of a call with
 * n = m, and every handle with fast tables (kernels 1, 2, 4, 6, 7, a warp or a CTA per string) returns the same bits.
 * Handles without fast tables choose in another order (forward from the start state instead of back from the end): their
 * draws differ but follow the same distribution.  Same bits on every call.  Local to the shard and without effect on
 * evaluations, as wfsa_dev_viterbi.  WFSA_ERR_INVALID: n outside 1..256 or a null pointer (other than logq);
 * WFSA_ERR_STATE before wfsa_dev_set_param_map; WFSA_ERR_NOMEM, with a message, when the padded step buffer of
 * n * (symbols + strings) steps cannot be allocated (checked before any launch). */
int wfsa_dev_sample(wfsa_dev* h, const double* x, int32_t n, uint64_t seed, double* logw /* [n_strings*n] */,
                    double* logq /* [n_strings] or NULL */, int64_t* path_off /* [n_strings*n + 1] */);
/* Steps of the last wfsa_dev_viterbi, wfsa_dev_nbest or wfsa_dev_sample, path_off[n_paths] of them, in path order:
 * trans_edge = index of the transition edge in the descriptor (trans_dst order); emis_edge = index of the emission edge
 * of its target state (emis_tok_off order), -1 for the final transition into the end state.  WFSA_ERR_STATE before any
 * wfsa_dev_viterbi, wfsa_dev_nbest or wfsa_dev_sample. */
int wfsa_dev_viterbi_paths(wfsa_dev* h, int32_t* trans_edge, int32_t* emis_edge);

/* Multi-GPU: one handle per process/GPU; results of eval/structure/hessian are all-reduced as exact integer
 * sums, so every rank holds the same bits (the evaluation through an all-reduce over NVLink peer memory fused
 * into its last kernel, with ncclAllReduce as the fall-back; structure and hessian through ncclAllReduce). */
#define WFSA_UNIQUE_ID_BYTES 128
int wfsa_dev_comm_unique_id(void* id_out /* WFSA_UNIQUE_ID_BYTES */);
int wfsa_dev_comm_init(wfsa_dev* h, const void* id, int rank, int nranks);

/* Sum (op 0) or max (op 1) of n host doubles over all ranks, in place; a no-op without a
 * communicator.  For the O(1) host scalars of Learner (common support, plogp, counts). */
int wfsa_dev_allreduce_f64(wfsa_dev* h, double* values, int n, int op);

/* Timing on the handle's own stream with CUDA events (torch events cannot see this stream). */
int wfsa_dev_timer_begin(wfsa_dev* h);
/* Like timer_begin, but without the events between the kernels of an evaluation (only wfsa_dev_timer_step_ms is
 * meaningful afterwards).  Events between kernels serialise the stream, so this is the timer to use for throughput:
 * the kernels of an evaluation keep their programmatic dependent launches. */
int wfsa_dev_timer_begin_steps(wfsa_dev* h);
int wfsa_dev_timer_end(wfsa_dev* h, float* ms);
/* ms spent in the dominant kernel (forward-backward) over the launches since timer_begin. */
int wfsa_dev_timer_kernel_ms(wfsa_dev* h, float* ms, int64_t* launches);
/* segmented kernel (6): the same time split into kr_regions (first) and whatever follows it inside the timed bracket
 * (second; overflow strings on the secondary kernel, else ~0); 0 otherwise */
int wfsa_dev_timer_split_ms(wfsa_dev* h, float* first_ms, float* second_ms);
/* Sum of the device times of the evaluations launched since timer_begin, each measured by its own event pair around
 * the WHOLE evaluation (weights, kernels, fold, collective); `steps` = how many.  Work queued between two evaluations
 * (wfsa_dev_l2_flush) is not included. */
int wfsa_dev_timer_step_ms(wfsa_dev* h, float* ms, int64_t* steps);
/* The same evaluations split into three phases (sums, ms): [0] start of the evaluation -> dominant kernel (weights,
 * resets), [1] the dominant kernel(s), [2] from there to the end (fold, collective, conversion). */
int wfsa_dev_timer_phase_ms(wfsa_dev* h, float* out3);
/* Segmented path, single-launch evaluation (k_eval6): nanoseconds CTA 0 spent in [arc weights, region types, grid barrier,
 * fold + exchange + conversion] (globaltimer stamps inside the kernel), summed over the evaluations since the last reset. */
int wfsa_dev_eval6_phases(wfsa_dev* h, double* out4, int reset);
/* Benchmark helper: a barrier over the ranks of the communicator, executed on the evaluation stream (through peer
 * memory when the peer all-reduce is in use, else a one-word ncclAllReduce).  Collective.  No-op without a communicator. */
int wfsa_dev_rank_barrier(wfsa_dev* h);
/* Benchmark helper: evicts the L2 cache (memset of a buffer twice its size on the evaluation stream). */
int wfsa_dev_l2_flush(wfsa_dev* h);

/* Introspection */
typedef struct {
    int32_t kernel;              /* 1 warp-per-string, 2 CTA-per-string, 3 generic, 4 thread-per-string
                                    (table walk),
                                    6 segmented compiled lattices (k_eval6 / kr_regions + ks_strings),
                                    7 position-synchronous pair-batched kernels (k7_fwd / k7_bwd)     */
    int32_t accum_mode;          /* 1 shared, 2 global                                          */
    int32_t n_trans, n_emis, n_arcs, n_slots;
    int32_t max_candidates;      /* max over symbols of states emitting it                      */
    int32_t sm_count, grid, block;
    int64_t n_strings, n_active_strings, n_tokens, n_active_tokens;
    int64_t smem_bytes, table_bytes;
    int64_t kernels_launched;    /* total kernels this handle has launched                      */
    double  fixed_point_scale_log2;
    /* segmented kernel (6): words of the region types and the per-string layout, lattice edges, edges whose posterior
       is exactly 1 (bridges, folded into constant accumulators), strings handed to the secondary kernel, pool size */
    int64_t lattice_words, lattice_edges, lattice_bridge_edges, n_overflow_strings;
    int32_t pool_slots;
    int32_t eval_path;           /* bit 0: objective+gradient in ONE launch (k_eval6); bit 1: ranks combined through NVLink peer
                                    memory inside that launch; bit 2: ranks combined by ncclAllReduce; bit 3: strings on the secondary kernel */
    /* segmented kernels (6): distinct region types, region instances over all strings, edges of all
       instances / of the distinct types (what one evaluation walks), host milliseconds of the compile */
    int64_t seg_types, seg_region_instances, seg_region_edges, seg_type_edges;
    double  seg_host_ms;
    /* schedule of the region phase of k_eval6 (segmented kernel 6, 0 otherwise), as the next launch would run it:
       big DAG groups (dealt out statically, big group b to warp b / grid of CTA b % grid); 1 if the CTAs that own a big group
       are dedicated to it (the environment as it is now); staging areas per CTA and word rows each (0 slots: every big group is
       streamed from HBM); rows of the longest big group; big groups the two-warp chain takes (at most one per CTA, when
       e6_big_groups <= grid, the group is staged and at least two staging areas exist) */
    int64_t e6_big_groups;
    int32_t e6_big_dedicate, e6_big_slots, e6_big_rows, e6_max_big_rows, e6_two_warp_eligible;
} wfsa_dev_info;
int wfsa_dev_get_info(wfsa_dev* h, wfsa_dev_info* info);

/* Host-only introspection (no device needed): compiles the lattice stream of ONE string in the word format
 * that the DAG form of region types uses (w-fsa_b200/csrc/lattice.hpp documents it), so that tests can
 * interpret the stream on the CPU.  trimmed may be NULL (no parameter removed).  *n_words = words written, 0 = no accepting path, -1 = needs more than n_slots
 * pool slots.  arc_tid / arc_eid (capacity arc_capacity, may be NULL) receive the combined-arc table:
 * arc -> (transition edge, emission edge or -1 for a final transition). */
int wfsa_lattice_compile(const wfsa_fsa_desc* fsa, const int32_t* trimmed, const int32_t* tokens, int32_t len,
                         int32_t n_slots, uint32_t* words, int64_t capacity, int64_t* n_words,
                         int32_t* arc_tid, int32_t* arc_eid, int32_t arc_capacity, int32_t* n_arcs);

/* Host-only introspection of the SEGMENTED compiled form (w-fsa_b200/csrc/lattice.hpp, kernels 6): compiles a
 * whole shard exactly as wfsa_dev_set_param_map does and exposes the arrays the device kernels read, so that
 * tests can interpret them on the CPU.  All strings of the corpus take part, longest first.  n_slots = pool slots
 * (1..16), plus 64 to keep every region in DAG form (no path lists).
 * which: 0 rwords(u32) 1 rgoff(i64) 2 rgrows(i32) 3 typeW(f64) 4 swords(u32) 5 sgoff(i64) 6 sgref(i32)
 *        7 ksid(i32) 8 kp(f64) 9 overflow(i32) 10 rejected(i32) 11 const_acc(i64)
 *        12 stats(i64): types, region instances, instance edges, type edges, bridges, strings, host microseconds,
 *           path blocks omitted (1: a region type, or a segment of an overflow string, has more than 2^20 paths, so
 *           arrays 13-19 describe zero blocks)
 *        13 path_off(i64) 14 col_off(i64) 15 val_off(i64) 16 cols(i32) 17 counts(f64) 18 p(f64) 19 type slot(i32): the path blocks
 *           wfsa_dev_hessian derives from the region types (layout of wfsa_path_blocks, p = weight of the type), then one
 *           block per segment with a choice of every overflow string (p = p_s, type slot -1).  The
 *           evaluation does not need them: a shard whose blocks cannot be built still compiles (wfsa_dev_hessian of such
 *           a shard returns WFSA_ERR_LIMIT).
 *        20 pwords(u32) 21 pgoff(i64): the reduction plan of the path-form groups (lattice.hpp, SegmentedCorpus::pwords) */
typedef struct wfsa_segmented wfsa_segmented;
int wfsa_segmented_compile(const wfsa_fsa_desc* fsa, const wfsa_corpus_desc* corpus, const int32_t* trimmed,
                           int32_t n_slots, double fx_scale, wfsa_segmented** out);
int wfsa_segmented_get(const wfsa_segmented* s, int which, const void** data, int64_t* count);
void wfsa_segmented_free(wfsa_segmented* s);

void wfsa_dev_destroy(wfsa_dev* h);
/* Bytes of device and pinned host memory held by all handles of this process, for leak tests: a handle that is
 * destroyed, or a parameter map that is replaced, must give back all it took.  (cudaMemGetInfo would see every
 * process on the device.) */
int64_t wfsa_dev_held_bytes(void);
const char* wfsa_dev_last_error(const wfsa_dev* h);   /* h may be NULL: last create() error */
const char* wfsa_dev_version(void);

#ifdef __cplusplus
}
#endif
#endif /* WFSA_DEV_H */
