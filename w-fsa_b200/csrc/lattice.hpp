// w-fsa_b200/csrc/lattice.hpp -- compiled per-string lattices: the word stream and the segmented form.
//
// The reference freezes the structure of every corpus string once, as the path matrices P and M
// (/root/reference/src/Learner.cpp:276-348), and every later evaluation is arithmetic on that
// frozen structure (src/Learner.cpp:515-553).  The device path does the same with a structure that
// does not grow with the number of paths: the *trimmed lattice* of the string -- nodes
// (position, state) that lie on an accepting path, edges = combined arcs (transition u->v taken,
// then v emits a substring that matches the input, inc/Recognize.h:49-57) plus the final
// transitions into the end state.  Which nodes/edges exist depends only on the automaton, the
// string and the trim map, never on the weights x, so it is compiled once per
// wfsa_dev_set_param_map and streamed by every evaluation.
//
// Stream = 32-bit words in a topological order of the edges (grouped by source node).  The DAG form of a region type
// (big_fwd / big_bwd in kernels_seg.cuh) is the stream of one region with region-local slots; compile_lattice writes
// the stream of a whole string, which the tests interpret on the CPU:
//
//   EDGE  bit31=1 | first_in<<29 | last_out<<28 | bridge<<27 | dst_slot<<23 | src_slot<<19 | arc
//         forward :  x = pool[src] * w[arc];  pool[dst] = first_in ? x : pool[dst] + x
//         backward:  post = x * pool[dst];    pool[src] = last_out ? w*pool[dst] : pool[src] + ...
//         A node owns a pool slot from its first incoming edge to its last outgoing edge; the
//         same interval is the life time of its alpha in the forward sweep and of its beta in
//         the backward sweep, so one slot assignment serves both.
//         bridge = every accepting path uses this edge (posterior exactly 1): its contribution
//         p_s to the gradient is folded into a constant accumulator at compile time.
//   CHECK every kCheckEvery-th word (same index in all 32 streams of a warp => no divergence):
//         low 16 bits = mask of live slots; the kernel renormalises the live values by a power
//         of two when their largest exponent leaves a band (exact) and records the exponent.
//   FIN   bit30=1 | slot of the end node   (last word of the stream; q = pool[slot])
//   PAD   0
#pragma once
#include <cstdint>
#include <functional>
#include <string>
#include <memory>
#include <vector>
#include "layout.hpp"

namespace wfsa {

constexpr uint32_t kLatEdge = 1u << 31, kLatFin = 1u << 30, kLatFirstIn = 1u << 29, kLatLastOut = 1u << 28,
                   kLatBridge = 1u << 27;
constexpr int kLatDstShift = 23, kLatSrcShift = 19, kLatArcBits = 16, kLatMaxSlots = 16;
constexpr int kCheckEvery = 16;           // words between CHECK words (power of two, multiple of the kernel's chunk)

// combined arcs of an automaton: (transition, emission of its target) pairs and final transitions
struct LatticeArcs {
    int n_arcs = 0;
    std::vector<int32_t> arc_tid, arc_eid;     // [n_arcs]; arc_eid = -1 for a final transition
    // compile index: row (state u, first token c) for c in [0, n_sym), c = n_sym: empty emissions
    int n_sym = 0, n_states = 0;
    std::vector<int32_t> row;                  // [n_states*(n_sym+1) + 1]
    std::vector<int32_t> ent_arc, ent_dst, ent_eid;
    std::vector<uint64_t> ent_pack;            // ent_arc | ent_dst << 32: one load per entry in the layered fast path
    std::vector<int32_t> final_arc;            // [n_states] arc id of u -> end, or -1
    std::vector<int32_t> eps_rank;             // [n_states] position in GenericLayout::eps_order
    bool has_eps = false, layered = false;     // layered: every emission is exactly one token long
};
void build_lattice_arcs(const HostFsa& f, const GenericLayout& g, LatticeArcs& out);

struct LatticeScratch {
    std::vector<int32_t> node_of;              // [(max_len+1)*n_states] -> node id or -1
    std::vector<int32_t> npos, nstate, nslot, nout, per_pos, topo, kept, topo_tmp;
    std::vector<uint8_t> coreach, done;
    std::vector<int32_t> esrc, edst, earc;
    std::vector<std::vector<int32_t>> bucket;  // node ids by position
};

// Compiles one string.  arc_alive[a] == 0 removes arc a (a trimmed-away parameter: weight 0).
// Returns 1 and appends the stream to `words` (without padding), 0 when the string has no accepting
// path, -1 when more than n_slots nodes are alive at once (the caller evaluates such strings with
// another kernel).  bridge_arcs receives the arcs of bridge edges (for the constant accumulators).
int compile_lattice(const HostFsa& f, const LatticeArcs& A, const uint8_t* arc_alive, const int32_t* tok, int len,
                    int n_slots, LatticeScratch& S, std::vector<uint32_t>& words, std::vector<int32_t>& bridge_arcs);


// ---------------------------------------------------------------------------------------------
// Segmented form (kernels KR + KS, kernels_seg.cuh).  A *cut node* of the trimmed lattice is a node
// every accepting path goes through (start, end, and every node no kept edge jumps over in the
// topological order).  Consecutive cut nodes delimit SEGMENTS; path weights factor over segments:
//     q(string) = prod_segments q_seg        posterior(edge) depends on its own segment only.
//   - a segment of ONE edge is a *bridge*: it contributes log w[arc] to log q and posterior exactly 1
//     (p_s goes to the constant accumulator of the arc at compile time);
//   - any other segment is a *region*: a small DAG between two cut nodes, evaluated by forward-
//     backward with region-local pool slots (entry node = slot 0, alpha(entry) = 1).
// This is what the reference's unique-path shortcut (logq = P.x, src/Learner.cpp:517-525) and its
// removal of columns "identical in every path" from H_f (src/HessianLearner.cpp:409-443) do, applied
// per segment instead of per string.  Regions that compile to the same words (same sub-lattice: same
// entry state, same consumed symbols) are merged into one TYPE with weight W = sum of the p_s of its
// instances; KR evaluates every type once per evaluation (log q_type and the posteriors scaled by W),
// KS adds up, per string, log w over its bridges and log q_type over its regions.
//
// Region words: EDGE words as above with region-local slots.  Regions of at most kSegSmallMax edges
// are stored as bare EDGE words (the exit node is the dst of the last edge); larger regions use the
// full stream format above (CHECK every kCheckEvery-th word, FIN last) so that they can be rescaled.
constexpr int kSegSmallMax = 0;           // edges of a "small" region (bare EDGE words).  0: every DAG-form region uses the stream format --
                                          // path form takes nearly all small regions, and one code path on the device beats a second,
                                          // rarely executed one (cold instruction fetches cost more than the padding rows)
constexpr int kSegMaxPaths = 8;           // path form: a region with at most this many paths ...
constexpr int kSegMaxPathLen = 16;        // ... all of one length, at most this many edges
constexpr int kKsSuper = 16;              // groups (warps) per super-group of the KS layout
constexpr int kKsChunkRows = 8;           // rows per interleaving chunk of the KS layout
constexpr int kSegSmallStep = 4;          // small regions are padded to 4, 8, 12 or 16 word rows
constexpr uint32_t kPlanLast = 1u << 31;  // reduction plan: last contributor of an entry (SegmentedCorpus::pwords)

struct SegString {                         // one string, compiled
    int status = 0;                        // 1 ok, 0 no accepting path, -1 needs another kernel
    std::vector<uint16_t> bridges;         // arcs of the bridge segments
    std::vector<uint32_t> rwords;          // region words, concatenated
    std::vector<int32_t> roff;             // [n_regions+1] into rwords
};
int compile_segments(const HostFsa& f, const LatticeArcs& A, const uint8_t* arc_alive, const int32_t* tok, int len,
                     int n_slots, LatticeScratch& S, SegString& out);

// The paths of every segment of one string, without a pool-slot limit: the trimmed lattice is cut at its cut nodes as
// compile_segments cuts it, and `emit` receives, for each segment with at least two paths, the arcs of all its paths (in
// DFS order).  Returns 1, 0 when the string has no accepting path, -1 when a segment has more than max_paths paths (the
// segments before it have been emitted).  For the H_f blocks of strings that no region type covers.
int segment_paths(const HostFsa& f, const LatticeArcs& A, const uint8_t* arc_alive, const int32_t* tok, int len,
                  size_t max_paths, LatticeScratch& S, const std::function<void(const std::vector<std::vector<int32_t>>&)>& emit);

struct SegmentedCorpus {
    // KR: region types in groups of 32 (one warp), word j of lane l of group g at rgoff[g] + j*32 + l;
    // type id = g*32 + l; rgrows[g] = word rows of the group (4/8/12/16 = small, otherwise a multiple of 16, at least 32)
    std::vector<uint32_t> rwords;
    std::vector<int64_t> rgoff;                // [n_rgroups+1]
    std::vector<int32_t> rgrows;               // [n_rgroups]
    std::vector<double> typeW;                 // [n_rgroups*32] sum of p_s over the instances (0 = padding lane)
    // reduction plan of the path-form groups (kr_paths): word r of lane l of group g at pgoff[g] + r*32 + l; a lane's
    // stream is a list of entries, one word per contributing cell:  arc | (lane' << 3 | p) << 16 | kPlanLast on the
    // entry's last word.  The kernel sums v[p] of lane' over an entry and issues one RED to `arc`.  Entries cover every
    // non-padding cell of the group once; a stream ends in 0 words.  DAG groups have no plan (pgoff[g+1] == pgoff[g]).
    std::vector<uint32_t> pwords;
    std::vector<int64_t> pgoff;                // [n_rgroups+1]
    int64_t n_types = 0, n_region_instances = 0, n_region_edges = 0, n_type_edges = 0, max_big_rows = 0;
    // KS: strings in groups of 32 (one warp), longest first; string position kpos = g*32 + l.  kKsSuper groups
    // form a super-group (one CTA); its words are chunk-interleaved:
    //   word (super-group sg, chunk c, group w in sg, row j in chunk, lane l)
    //        at sgoff[sg] + (((c*kKsSuper + w)*kKsChunkRows + j)*32 + l,   chunks(sg) from sgoff[sg+1]-sgoff[sg]
    //   rows [0, sgref[g])   of group g: region type ids (padding = dummy type n_rgroups*32, log q = 0)
    //   the rows after them  : two 16-bit bridge arcs per word (padding ids n_arcs .. n_arcs+15, log w = 0),
    //                          scheduled per half-warp against shared-memory bank conflicts (BridgeScheduler)
    std::vector<uint32_t> swords;
    std::vector<int64_t> sgoff;                // [n_supergroups+1]
    std::vector<int32_t> sgref;                // [n_supergroups*kKsSuper]
    std::vector<int32_t> ksid;                 // [n_supergroups*kKsSuper*32] string id or -1
    std::vector<double> kp;                    // [n_supergroups*kKsSuper*32] p_s (0 = padding lane)
    std::vector<int32_t> overflow, rejected;
    std::vector<long long> const_acc;          // [n_arcs] fixed-point constant gradient part (bridges)
    int64_t n_bridge = 0, n_strings = 0;
    double host_ms = 0;
};
void compile_corpus_segmented(const HostFsa& f, const LatticeArcs& A, const uint8_t* arc_alive, const int32_t* tokens,
                              const int64_t* offs, const double* p, const std::vector<int32_t>& ids, int n_slots,
                              double fx_scale, SegmentedCorpus& out);

// The same in two steps.  compile_corpus_regions fills everything an objective+gradient evaluation needs (region types,
// constants, overflow/rejected lists, statistics) and returns a job that builds the per-string layout (swords, sgoff,
// sgref, ksid, kp: only read when log q of every string is asked for) when run() is called -- later, on another thread,
// or never.  `p` must stay valid until then; `out` of run() may be another object than the one of the first step.
struct SegmentedStringsJob {
    struct State;
    State* st;
    SegmentedStringsJob();
    ~SegmentedStringsJob();
    SegmentedStringsJob(const SegmentedStringsJob&) = delete;
    SegmentedStringsJob& operator=(const SegmentedStringsJob&) = delete;
    void run(SegmentedCorpus& out);
};
std::shared_ptr<SegmentedStringsJob> compile_corpus_regions(const HostFsa& f, const LatticeArcs& A, const uint8_t* arc_alive,
                                                            const int32_t* tokens, const int64_t* offs, const double* p,
                                                            const std::vector<int32_t>& ids, int n_slots, double fx_scale,
                                                            SegmentedCorpus& out);

}  // namespace wfsa
