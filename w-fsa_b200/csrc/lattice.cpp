// w-fsa_b200/csrc/lattice.cpp -- see lattice.hpp.
#include "lattice.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <thread>

namespace wfsa {

void build_lattice_arcs(const HostFsa& f, const GenericLayout& g, LatticeArcs& A)
{
    A = LatticeArcs();
    const int S = f.n_states, NS = f.n_sym;
    A.n_sym = NS; A.n_states = S;
    A.final_arc.assign(S, -1);
    A.eps_rank.assign(S, 0);
    for (int i = 0; i < (int)g.eps_order.size(); ++i) A.eps_rank[g.eps_order[i]] = i;
    A.layered = true;
    for (int s = 0; s < S; ++s) {
        if (s == f.start || s == f.end) continue;
        for (int e = f.emis_row[s]; e < f.emis_row[s + 1]; ++e) {
            if (f.emis_len(e) == 0) A.has_eps = true;
            if (f.emis_len(e) != 1) A.layered = false;
        }
    }
    // arcs in (source, transition, emission) order; the compile index is a CSR over (source, first token)
    std::vector<int32_t> key;          // row of every non-final arc
    std::vector<int32_t> dst;
    for (int u = 0; u < S; ++u) {
        if (u == f.end) continue;
        for (int t = f.trans_row[u]; t < f.trans_row[u + 1]; ++t) {
            const int v = f.trans_dst[t];
            if (v == f.end) {
                A.final_arc[u] = (int32_t)A.arc_tid.size();
                A.arc_tid.push_back(t); A.arc_eid.push_back(-1);
                key.push_back(-1); dst.push_back(-1);
                continue;
            }
            for (int e = f.emis_row[v]; e < f.emis_row[v + 1]; ++e) {
                const int c = f.emis_len(e) == 0 ? NS : f.emis_tok[f.emis_tok_off[e]];
                A.arc_tid.push_back(t); A.arc_eid.push_back(e);
                key.push_back(u * (NS + 1) + c); dst.push_back(v);
            }
        }
    }
    A.n_arcs = (int)A.arc_tid.size();
    const size_t n_rows = (size_t)S * (NS + 1);
    A.row.assign(n_rows + 1, 0);
    for (int a = 0; a < A.n_arcs; ++a) if (key[a] >= 0) A.row[key[a] + 1]++;
    for (size_t r = 0; r < n_rows; ++r) A.row[r + 1] += A.row[r];
    const int n_ent = A.row[n_rows];
    A.ent_arc.resize(n_ent); A.ent_dst.resize(n_ent); A.ent_eid.resize(n_ent);
    std::vector<int32_t> fill(A.row.begin(), A.row.end() - 1);
    for (int a = 0; a < A.n_arcs; ++a) {
        if (key[a] < 0) continue;
        const int i = fill[key[a]]++;
        A.ent_arc[i] = a; A.ent_dst[i] = dst[a]; A.ent_eid[i] = A.arc_eid[a];
    }
    A.ent_pack.resize(n_ent);
    for (int i = 0; i < n_ent; ++i) A.ent_pack[i] = (uint64_t)(uint32_t)A.ent_arc[i] | (uint64_t)(uint32_t)A.ent_dst[i] << 32;
}

// Forward reachability + co-reachability of one string's lattice.  On return S.esrc/edst/earc hold every
// forward-reachable edge in a topological order (grouped by source node), S.coreach marks the nodes that
// reach the end node.  Returns the end node id, or -1 when the string has no accepting path.
static int build_and_trim(const HostFsa& f, const LatticeArcs& A, const uint8_t* alive, const int32_t* tok, int len,
                          LatticeScratch& S)
{
    const int NSt = f.n_states, NS = f.n_sym;
    const size_t need = (size_t)(len + 1) * NSt;
    if (S.node_of.size() < need) S.node_of.resize(need, -1);
    if ((int)S.bucket.size() < len + 1) S.bucket.resize(len + 1);
    S.npos.clear(); S.nstate.clear(); S.esrc.clear(); S.edst.clear(); S.earc.clear();
    int end_node = -1;
    auto get_node = [&](int pos, int st) -> int {
        int32_t& slot = S.node_of[(size_t)pos * NSt + st];
        if (slot < 0) {
            slot = (int32_t)S.npos.size();
            S.npos.push_back(pos); S.nstate.push_back(st);
            S.bucket[pos].push_back(slot);
        }
        return slot;
    };
    auto process = [&](int n) {
        const int pos = S.npos[n], u = S.nstate[n];
        if (pos < len) {
            const int c = tok[pos];
            if (c >= 0 && c < NS) {
                const size_t r = (size_t)u * (NS + 1) + c;
                for (int i = A.row[r]; i < A.row[r + 1]; ++i) {
                    const int a = A.ent_arc[i];
                    if (alive && !alive[a]) continue;
                    const int e = A.ent_eid[i];
                    const int e0 = f.emis_tok_off[e], el = f.emis_tok_off[e + 1] - e0;
                    if (el > 1) {
                        if (pos + el > len) continue;
                        bool m = true;
                        for (int k = 1; k < el; ++k) if (tok[pos + k] != f.emis_tok[e0 + k]) { m = false; break; }
                        if (!m) continue;
                    }
                    const int d = get_node(pos + el, A.ent_dst[i]);
                    S.esrc.push_back(n); S.edst.push_back(d); S.earc.push_back(a);
                }
            }
        }
        if (A.has_eps) {
            const size_t r = (size_t)u * (NS + 1) + NS;
            for (int i = A.row[r]; i < A.row[r + 1]; ++i) {
                const int a = A.ent_arc[i];
                if (alive && !alive[a]) continue;
                const int d = get_node(pos, A.ent_dst[i]);       // later in eps order than u
                S.esrc.push_back(n); S.edst.push_back(d); S.earc.push_back(a);
            }
        }
        if (pos == len && A.final_arc[u] >= 0 && (!alive || alive[A.final_arc[u]])) {
            if (end_node < 0) {
                end_node = (int)S.npos.size();
                S.npos.push_back(len + 1); S.nstate.push_back(f.end);
            }
            S.esrc.push_back(n); S.edst.push_back(end_node); S.earc.push_back(A.final_arc[u]);
        }
    };
    // ---- forward reachability, nodes processed in a topological order
    if (A.layered) {
        // Every emission is one token long: the nodes of position pos + 1 are created, in order, while those of pos are
        // processed, so a position is an index range of the node array (no buckets), and an entry is one packed load.
        // Same node and edge order as the general loop below.  The state -> node index is needed for one position at
        // a time only: it is the first n_states entries of node_of (1 KB for config 4, cache resident), cleared again
        // after every position.
        S.npos.push_back(0); S.nstate.push_back(f.start);
        int32_t* const next_of = S.node_of.data();
        int lo = 0, hi = 1;
        for (int pos = 0; pos <= len; ++pos) {
            const int c = pos < len ? tok[pos] : -1;
            for (int n = lo; n < hi; ++n) {
                const int u = S.nstate[n];
                if (c >= 0 && c < NS) {
                    const size_t r = (size_t)u * (NS + 1) + c;
                    for (int i = A.row[r]; i < A.row[r + 1]; ++i) {
                        const uint64_t pk = A.ent_pack[i];
                        const int a = (int)(uint32_t)pk, dstate = (int)(pk >> 32);
                        if (alive && !alive[a]) continue;
                        int32_t& slot = next_of[dstate];
                        if (slot < 0) {
                            slot = (int32_t)S.npos.size();
                            S.npos.push_back(pos + 1); S.nstate.push_back(dstate);
                        }
                        S.esrc.push_back(n); S.edst.push_back(slot); S.earc.push_back(a);
                    }
                }
                if (pos == len && A.final_arc[u] >= 0 && (!alive || alive[A.final_arc[u]])) {
                    if (end_node < 0) {
                        end_node = (int)S.npos.size();
                        S.npos.push_back(len + 1); S.nstate.push_back(f.end);
                    }
                    S.esrc.push_back(n); S.edst.push_back(end_node); S.earc.push_back(A.final_arc[u]);
                }
            }
            lo = hi;
            hi = (int)S.npos.size();
            for (int m = lo; m < hi; ++m) next_of[S.nstate[m]] = -1;
            if (lo == hi) break;                                  // nothing reaches the next position
        }
    } else {
    get_node(0, f.start);
    for (int pos = 0; pos <= len; ++pos) {
        std::vector<int32_t>& B = S.bucket[pos];
        if (!A.has_eps) {
            for (size_t bi = 0; bi < B.size(); ++bi) process(B[bi]);
        } else {
            S.done.assign(B.size(), 0);
            for (;;) {
                int best = -1;
                if (S.done.size() < B.size()) S.done.resize(B.size(), 0);
                for (size_t bi = 0; bi < B.size(); ++bi)
                    if (!S.done[bi] && (best < 0 || A.eps_rank[S.nstate[B[bi]]] < A.eps_rank[S.nstate[B[best]]])) best = (int)bi;
                if (best < 0) break;
                S.done[best] = 1;
                process(B[best]);
            }
        }
    }
    for (int pos = 0; pos <= len; ++pos) S.bucket[pos].clear();
    // reset the scratch index for the next string
    for (size_t n = 0; n < S.npos.size(); ++n) if (S.npos[n] <= len) S.node_of[(size_t)S.npos[n] * NSt + S.nstate[n]] = -1;
    }
    const int n_nodes = (int)S.npos.size(), n_e = (int)S.esrc.size();
    if (end_node < 0) return -1;
    // ---- co-reachability (edges are ordered by source in topological order => reverse sweep)
    S.coreach.assign(n_nodes, 0);
    S.coreach[end_node] = 1;
    for (int e = n_e - 1; e >= 0; --e) if (S.coreach[S.edst[e]]) S.coreach[S.esrc[e]] = 1;
    if (!S.coreach[0]) return -1;
    return end_node;
}

int compile_lattice(const HostFsa& f, const LatticeArcs& A, const uint8_t* alive, const int32_t* tok, int len,
                    int n_slots, LatticeScratch& S, std::vector<uint32_t>& words, std::vector<int32_t>& bridge_arcs)
{
    const int end_node = build_and_trim(f, A, alive, tok, len, S);
    if (end_node < 0) return 0;
    const int n_nodes = (int)S.npos.size(), n_e = (int)S.esrc.size();
    S.nout.assign(n_nodes, 0);
    S.per_pos.assign(len + 2, 0);
    for (int n = 0; n < n_nodes; ++n) if (S.coreach[n]) S.per_pos[S.npos[n]]++;
    for (int e = 0; e < n_e; ++e) if (S.coreach[S.edst[e]]) S.nout[S.esrc[e]]++;
    // ---- emit the stream
    const size_t base = words.size(), bridge_base = bridge_arcs.size();
    S.nslot.assign(n_nodes, -1);
    uint32_t free_mask = n_slots >= 32 ? 0xffffffffu : ((1u << n_slots) - 1u), live = 0;
    auto alloc = [&]() -> int {
        if (!free_mask) return -1;
        const int s = __builtin_ctz(free_mask);
        free_mask &= free_mask - 1; live |= 1u << s;
        return s;
    };
    auto release = [&](int s) { free_mask |= 1u << s; live &= ~(1u << s); };
    S.nslot[0] = alloc();
    int cur_src = -1;
    size_t last_edge = 0;
    auto check_word = [&]() { if (((words.size() - base) & (kCheckEvery - 1)) == kCheckEvery - 1) words.push_back(live & 0xffffu); };
    for (int e = 0; e < n_e; ++e) {
        const int d = S.edst[e];
        if (!S.coreach[d]) continue;
        const int s = S.esrc[e];
        if (s != cur_src) {
            if (cur_src >= 0) { words[last_edge] |= kLatLastOut; release(S.nslot[cur_src]); }
            cur_src = s;
        }
        check_word();
        uint32_t w = kLatEdge | (uint32_t)S.earc[e];
        if (S.nslot[d] < 0) {
            S.nslot[d] = alloc();
            if (S.nslot[d] < 0) { words.resize(base); bridge_arcs.resize(bridge_base); return -1; }
            w |= kLatFirstIn;
        }
        if (A.layered && S.per_pos[S.npos[s]] == 1 && S.nout[s] == 1) { w |= kLatBridge; bridge_arcs.push_back(S.earc[e]); }
        w |= (uint32_t)S.nslot[d] << kLatDstShift | (uint32_t)S.nslot[s] << kLatSrcShift;
        last_edge = words.size();
        words.push_back(w);
    }
    words[last_edge] |= kLatLastOut;
    release(S.nslot[cur_src]);
    check_word();
    words.push_back(kLatFin | (uint32_t)S.nslot[end_node]);
    return 1;
}

// ---------------------------------------------------------------------------------------------
// Segmented form
// ---------------------------------------------------------------------------------------------
int compile_segments(const HostFsa& f, const LatticeArcs& A, const uint8_t* alive, const int32_t* tok, int len,
                     int n_slots, LatticeScratch& S, SegString& out)
{
    out.bridges.clear(); out.rwords.clear(); out.roff.assign(1, 0);
    out.status = 0;
    const int end_node = build_and_trim(f, A, alive, tok, len, S);
    if (end_node < 0) return 0;
    const int n_nodes = (int)S.npos.size(), n_e = (int)S.esrc.size();
    // kept edges (both ends on an accepting path) and the topological index of their nodes
    S.kept.clear();
    S.topo.assign(n_nodes, -1);
    int nt = 0;
    for (int e = 0; e < n_e; ++e) {
        if (!S.coreach[S.edst[e]]) continue;
        S.kept.push_back(e);
        if (S.topo[S.esrc[e]] < 0) S.topo[S.esrc[e]] = nt++;
    }
    S.topo[end_node] = nt;
    S.nslot.assign(n_nodes, -1);
    S.nout.assign(n_nodes, -1);
    const int nk = (int)S.kept.size();
    const bool allow_paths = !(n_slots & 64);             // bit 6 of n_slots: DAG form only (tests, experiments)
    n_slots &= 63;
    // PATH FORM of a region: when it has at most kSegMaxPaths paths, all of one length L <= kSegMaxPathLen, the region
    // is stored as its explicit path list (what the reference's P matrix holds for a whole string,
    // src/Learner.cpp:295-314, here for one small segment): header word, then L*P arcs, edge l of path p at
    // [1 + l*P + p].  q = sum_p prod_l w, posterior of a path = its product / q: registers only on the device.
    std::vector<int32_t>& pstk = S.per_pos;                 // scratch: DFS stack of edge indices (kept[] positions)
    std::vector<int32_t>& first_out = S.nout;               // scratch: first kept edge of a node inside the segment
    auto try_paths = [&](int b, int e) -> bool {
        if (!allow_paths) return false;
        const int entry = S.esrc[S.kept[b]], exitn = S.edst[S.kept[e - 1]];
        for (int i = b; i < e; ++i) first_out[S.esrc[S.kept[i]]] = -1;
        for (int i = e - 1; i >= b; --i) first_out[S.esrc[S.kept[i]]] = i;      // edges of a node are contiguous
        int n_paths = 0, L = -1;
        std::vector<int32_t>& arcs = S.topo_tmp;            // path-major arcs of the paths found so far
        arcs.clear();
        pstk.clear();
        // iterative DFS: pstk holds the current path as kept[] positions
        int node = entry, next_edge = first_out[entry];
        for (;;) {
            if (node == exitn) {
                if (L < 0) L = (int)pstk.size();
                if ((int)pstk.size() != L || L > kSegMaxPathLen || ++n_paths > kSegMaxPaths) return false;
                for (int i : pstk) arcs.push_back(S.earc[S.kept[i]]);
                next_edge = -1;                             // backtrack
            }
            if (next_edge >= 0 && next_edge < e && S.esrc[S.kept[next_edge]] == node) {
                if ((int)pstk.size() >= kSegMaxPathLen) return false;
                pstk.push_back(next_edge);
                node = S.edst[S.kept[next_edge]];
                next_edge = node == exitn ? -1 : first_out[node];
                continue;
            }
            if (pstk.empty()) break;
            const int last = pstk.back();
            pstk.pop_back();
            node = S.esrc[S.kept[last]];
            next_edge = last + 1;
        }
        if (n_paths < 2) return false;
        out.rwords.push_back(kLatFin | (uint32_t)n_paths << 8 | (uint32_t)L);   // header: bit 31 clear, bit 30 set
        for (int l = 0; l < L; ++l)
            for (int q = 0; q < n_paths; ++q) out.rwords.push_back(kLatEdge | (uint32_t)arcs[(size_t)q * L + l]);
        out.roff.push_back((int32_t)out.rwords.size());
        return true;
    };
    // one segment = kept edges [b, e): all edges whose source lies between two consecutive cut nodes
    auto emit_segment = [&](int b, int e) -> bool {
        if (e - b == 1) { out.bridges.push_back((uint16_t)S.earc[S.kept[b]]); return true; }
        if (try_paths(b, e)) return true;
        const bool big = e - b > kSegSmallMax;
        const size_t base = out.rwords.size();
        uint32_t free_mask = n_slots >= 32 ? 0xffffffffu : ((1u << n_slots) - 1u), live = 0;
        auto alloc = [&]() -> int {
            if (!free_mask) return -1;
            const int sl = __builtin_ctz(free_mask);
            free_mask &= free_mask - 1; live |= 1u << sl;
            return sl;
        };
        auto check_word = [&]() {
            if (big && ((out.rwords.size() - base) & (kCheckEvery - 1)) == kCheckEvery - 1) out.rwords.push_back(live & 0xffffu);
        };
        int cur_src = -1, exit_slot = -1;
        size_t last_edge = 0;
        S.nslot[S.esrc[S.kept[b]]] = alloc();              // the entry node owns slot 0
        for (int i = b; i < e; ++i) {
            const int ed = S.kept[i], sN = S.esrc[ed], dN = S.edst[ed];
            if (sN != cur_src) {
                if (cur_src >= 0) {
                    out.rwords[last_edge] |= kLatLastOut;
                    const int sl = S.nslot[cur_src];
                    free_mask |= 1u << sl; live &= ~(1u << sl);
                }
                cur_src = sN;
            }
            check_word();
            uint32_t w = kLatEdge | (uint32_t)S.earc[ed];
            if (S.nslot[dN] < 0) {
                S.nslot[dN] = alloc();
                if (S.nslot[dN] < 0) return false;
                w |= kLatFirstIn;
            }
            exit_slot = S.nslot[dN];
            w |= (uint32_t)S.nslot[dN] << kLatDstShift | (uint32_t)S.nslot[sN] << kLatSrcShift;
            last_edge = out.rwords.size();
            out.rwords.push_back(w);
        }
        out.rwords[last_edge] |= kLatLastOut;
        { const int sl = S.nslot[cur_src]; free_mask |= 1u << sl; live &= ~(1u << sl); }
        if (big) { check_word(); out.rwords.push_back(kLatFin | (uint32_t)exit_slot); }
        // slots are region-local: forget them (the exit node is the entry of the next segment)
        for (int i = b; i < e; ++i) { S.nslot[S.esrc[S.kept[i]]] = -1; S.nslot[S.edst[S.kept[i]]] = -1; }
        out.roff.push_back((int32_t)out.rwords.size());
        return true;
    };
    int seg_begin = 0, maxdst = 0, cur = -1;
    for (int i = 0; i < nk; ++i) {
        const int ed = S.kept[i], sN = S.esrc[ed];
        if (sN != cur) {
            cur = sN;
            if (S.topo[sN] == maxdst && i > seg_begin) {       // sN is a cut node: close the segment before it
                if (!emit_segment(seg_begin, i)) { out.status = -1; return -1; }
                seg_begin = i;
            }
        }
        maxdst = std::max(maxdst, S.topo[S.edst[ed]]);
    }
    if (nk > seg_begin && !emit_segment(seg_begin, nk)) { out.status = -1; return -1; }
    out.status = 1;
    return 1;
}

int segment_paths(const HostFsa& f, const LatticeArcs& A, const uint8_t* alive, const int32_t* tok, int len,
                  size_t max_paths, LatticeScratch& S, const std::function<void(const std::vector<std::vector<int32_t>>&)>& emit)
{
    const int end_node = build_and_trim(f, A, alive, tok, len, S);
    if (end_node < 0) return 0;
    const int n_nodes = (int)S.npos.size(), n_e = (int)S.esrc.size();
    S.kept.clear();
    S.topo.assign(n_nodes, -1);
    int nt = 0;
    for (int e = 0; e < n_e; ++e) {
        if (!S.coreach[S.edst[e]]) continue;
        S.kept.push_back(e);
        if (S.topo[S.esrc[e]] < 0) S.topo[S.esrc[e]] = nt++;
    }
    S.topo[end_node] = nt;
    std::vector<int32_t>& first_out = S.nout;               // first kept edge of a node (the edges of a node are contiguous)
    first_out.assign(n_nodes, -1);
    for (int i = (int)S.kept.size() - 1; i >= 0; --i) first_out[S.esrc[S.kept[i]]] = i;
    std::vector<std::vector<int32_t>> paths;
    std::vector<int32_t>& stk = S.per_pos;                  // the current path as kept[] positions
    // kept edges [b, e) between two consecutive cut nodes: every path from the entry to the exit (the dst of the last edge)
    auto segment = [&](int b, int e) -> bool {
        if (e - b == 1) return true;                        // a bridge: one path
        const int exitn = S.edst[S.kept[e - 1]];
        paths.clear();
        stk.clear();
        int node = S.esrc[S.kept[b]], next_edge = b;
        for (;;) {
            if (node == exitn) {
                paths.emplace_back();
                for (int i : stk) paths.back().push_back(S.earc[S.kept[i]]);
                if (paths.size() > max_paths) return false;
                next_edge = -1;                             // backtrack
            }
            if (next_edge >= 0 && next_edge < e && S.esrc[S.kept[next_edge]] == node) {
                stk.push_back(next_edge);
                node = S.edst[S.kept[next_edge]];
                next_edge = node == exitn ? -1 : first_out[node];
                continue;
            }
            if (stk.empty()) break;
            const int last = stk.back();
            stk.pop_back();
            node = S.esrc[S.kept[last]];
            next_edge = last + 1;
        }
        if (paths.size() >= 2) emit(paths);
        return true;
    };
    const int nk = (int)S.kept.size();
    int seg_begin = 0, maxdst = 0, cur = -1;
    for (int i = 0; i < nk; ++i) {                          // the cut of compile_segments
        const int ed = S.kept[i], sN = S.esrc[ed];
        if (sN != cur) {
            cur = sN;
            if (S.topo[sN] == maxdst && i > seg_begin) {
                if (!segment(seg_begin, i)) return -1;
                seg_begin = i;
            }
        }
        maxdst = std::max(maxdst, S.topo[S.edst[ed]]);
    }
    if (nk > seg_begin && !segment(seg_begin, nk)) return -1;
    return 1;
}

namespace {
inline uint64_t fnv1a(const uint32_t* w, size_t n)
{
    uint64_t h = 1469598103934665603ull;
    for (size_t i = 0; i < n; ++i) { h ^= w[i]; h *= 1099511628211ull; }
    return h ^ (h >> 29);
}
}  // namespace

// Schedules the bridge arcs of the (up to) 16 strings of one half-warp into time slots.  In one slot every lane
// reads one 8-byte table entry; entries whose ids agree mod 16 live in the same pair of shared-memory banks, and
// a slot costs one wavefront per lane sharing a bank pair.  The schedule is a proper edge colouring of the
// bipartite multigraph lanes x classes with T = (longest string of the half-warp) colours, i.e. no padding
// beyond the length differences; a class that holds more than T arcs is split in two virtual classes that may
// both appear in one slot (a two-way conflict -- cheaper than a padded slot, which costs a wavefront AND
// memory traffic).  Lanes with nothing to read in a slot get one of 16 padding entries (ids n_arcs ..
// n_arcs+15, log w = 0), of a class nobody else reads in that slot when there is one.
struct BridgeScheduler {
    static constexpr int NK = 32;                    // virtual classes
    uint16_t pad0;
    int slack_pct = 8;
    std::vector<int16_t> laneCol, classCol;          // [16][T] / [NK][T]: colour -> class of the lane's edge / lane of the class's edge
    std::vector<std::vector<uint16_t>> bucket;       // [16*NK] arcs of (lane, virtual class)
    explicit BridgeScheduler(uint16_t pad) : pad0(pad), bucket(16 * NK)
    {
        if (const char* e = std::getenv("WFSA_KS_SLACK")) slack_pct = std::max(0, std::min(100, std::atoi(e)));   // tuning knob
    }
    int run(const uint16_t* const* arcs, const int* cnt, std::vector<uint16_t>& out)
    {
        int degL[16] = {0}, load[16] = {0};
        for (int l = 0; l < 16; ++l)
            for (int i = 0; i < cnt[l]; ++i) { degL[l]++; load[arcs[l][i] & 15]++; }
        int maxdeg = 0, maxload = 0;
        for (int i = 0; i < 16; ++i) { maxdeg = std::max(maxdeg, degL[i]); maxload = std::max(maxload, load[i]); }
        // slots: the longest string, plus up to slack_pct % padding when that removes conflicts
        int T = std::max(maxdeg, std::min(maxload, maxdeg + (maxdeg * slack_pct + 99) / 100));
        T = std::max(T, (maxload + 1) / 2);
        out.assign((size_t)T * 16, 0);
        if (T == 0) return 0;
        for (auto& b : bucket) b.clear();
        int filled[16] = {0};
        for (int l = 0; l < 16; ++l)
            for (int i = 0; i < cnt[l]; ++i) {
                const int k = arcs[l][i] & 15;
                bucket[l * NK + (filled[k]++ < T ? k : k + 16)].push_back(arcs[l][i]);
            }
        const int D = T;
        laneCol.assign((size_t)16 * D, -1); classCol.assign((size_t)NK * D, -1);
        int freeL[16] = {0}, freeK[NK] = {0};           // lowest colour that may be free (hint; verified below)
        std::vector<int> path;
        for (int l = 0; l < 16; ++l)
            for (int k = 0; k < NK; ++k)
                for (size_t m = 0; m < bucket[l * NK + k].size(); ++m) {
                    int a = freeL[l]; while (laneCol[(size_t)l * D + a] >= 0) ++a;
                    int b = freeK[k]; while (classCol[(size_t)k * D + b] >= 0) ++b;
                    freeL[l] = a; freeK[k] = b;
                    if (classCol[(size_t)k * D + a] >= 0) {
                        // colour a is taken at class k: flip the a/b alternating path that starts there
                        path.clear();
                        int ck = k;
                        for (;;) {
                            const int x = classCol[(size_t)ck * D + a];
                            if (x < 0) break;
                            path.push_back(x); path.push_back(ck); path.push_back(a);
                            const int nk = laneCol[(size_t)x * D + b];
                            if (nk < 0) break;
                            path.push_back(x); path.push_back(nk); path.push_back(b);
                            ck = nk;
                        }
                        for (size_t q = 0; q < path.size(); q += 3) { laneCol[(size_t)path[q] * D + path[q + 2]] = -1; classCol[(size_t)path[q + 1] * D + path[q + 2]] = -1; }
                        for (size_t q = 0; q < path.size(); q += 3) {
                            const int c2 = path[q + 2] == a ? b : a;
                            laneCol[(size_t)path[q] * D + c2] = (int16_t)path[q + 1]; classCol[(size_t)path[q + 1] * D + c2] = (int16_t)path[q];
                        }
                        for (size_t q = 0; q < path.size(); q += 3) {       // the hints of touched nodes may have moved down
                            freeL[path[q]] = std::min(freeL[path[q]], std::min(a, b)); freeK[path[q + 1]] = std::min(freeK[path[q + 1]], std::min(a, b));
                        }
                    }
                    laneCol[(size_t)l * D + a] = (int16_t)k; classCol[(size_t)k * D + a] = (int16_t)l;
                }
        size_t taken[16 * NK] = {0};
        for (int c = 0; c < D; ++c) {
            unsigned used = 0;
            for (int l = 0; l < 16; ++l) { const int k = laneCol[(size_t)l * D + c]; if (k >= 0) used |= 1u << (k & 15); }
            for (int l = 0; l < 16; ++l) {
                const int k = laneCol[(size_t)l * D + c];
                if (k >= 0) out[(size_t)c * 16 + l] = bucket[l * NK + k][taken[l * NK + k]++];
                else {
                    const unsigned fr = ~used & 0xffffu;                         // bank pairs no lane reads in this slot
                    const int fk = fr ? __builtin_ctz(fr) : l;
                    used |= 1u << fk;
                    out[(size_t)c * 16 + l] = (uint16_t)(pad0 + ((fk - pad0) & 15));   // the padding entry of class fk
                }
            }
        }
        return D;
    }
};

namespace {
// what one compile thread produced for its strings (strings i = t, t+T, ... on thread t)
struct SegLocal {
    std::vector<uint16_t> bridges; std::vector<int64_t> boff;      // bridges of string j at [boff[j], boff[j+1])
    std::vector<uint32_t> rwords;                                   // region words
    std::vector<int64_t> rbeg; std::vector<int32_t> rlen;           // per region
    std::vector<uint64_t> rhash;
    std::vector<int64_t> sreg;                                      // regions of string j at [sreg[j], sreg[j+1])
    std::vector<int8_t> status;
    std::vector<long long> cacc;
    int64_t region_edges = 0;                                       // EDGE words over all regions of the thread's accepted strings
};
}  // namespace

// Everything the per-string layout (phase 4) needs from the region phases; kept alive by the job object so that the
// layout can be built later, on another thread, or not at all.
struct SegmentedStringsJob::State {
    std::vector<SegLocal> loc;
    int T = 1, n_arcs = 0;
    std::vector<int64_t> ok;
    std::vector<std::vector<int32_t>> reg_type;
    std::vector<int32_t> type_slot;
    int64_t n_rg = 0;
    std::vector<int32_t> ids;
    const double* p = nullptr;
};
// Reduction plan of every path-form group (layout: SegmentedCorpus::pwords).  Types are sorted by their arcs, so the 32
// types of a group share most of them: summing the contributions of a group per distinct arc before the RED leaves
// 0.6 of the REDs at 100 k config-4 strings (the sums are integers: the same bits in any order).  An entry lists the
// cells (lane, p) of one arc in (level, path, lane) order, an arc on several levels of a path once per level; an entry
// longer than the group's ideal stream (cells / 32 rows) is cut, so that no lane walks much more than its share.  Entries
// are dealt out largest first (ties: lower arc), each to the lane with the shortest stream (ties: lower lane).  Groups
// are planned on T threads in contiguous ranges: the result does not depend on T.
static void build_path_plans(SegmentedCorpus& out, int n_arcs, int T)
{
    const int64_t n_rg = (int64_t)out.rgrows.size();
    std::vector<int64_t> rows_of((size_t)n_rg, 0);
    std::vector<std::vector<uint32_t>> part(T);
    auto plan = [&](int t) {
        const int64_t g0 = n_rg * t / T, g1 = n_rg * (t + 1) / T;
        std::vector<uint64_t> cells;                                      // arc << 32 | cell index (level, path, lane) << 8 | code
        std::vector<std::pair<int, int>> ent;                             // [begin, end) in cells
        std::vector<uint32_t> lanes[32];
        for (int64_t g = g0; g < g1; ++g) {
            const int32_t code = out.rgrows[g];
            if (!(code & 0x10000)) continue;
            const int PP = (code >> 8) & 0xff, L = code & 0xff;
            const uint32_t* w = out.rwords.data() + out.rgoff[g];
            cells.clear();
            for (int k = 0; k < PP * L; ++k)
                for (int ln = 0; ln < 32; ++ln)
                    if (w[(size_t)k * 32 + ln] != (uint32_t)n_arcs)
                        cells.push_back((uint64_t)w[(size_t)k * 32 + ln] << 32 | (uint64_t)(k * 32 + ln) << 8 | (uint64_t)(ln << 3 | k % PP));
            if (cells.empty()) continue;
            std::sort(cells.begin(), cells.end());
            const int cap = (int)((cells.size() + 31) / 32);
            ent.clear();
            for (size_t b = 0; b < cells.size();) {
                size_t e = b;
                while (e < cells.size() && (cells[e] >> 32) == (cells[b] >> 32)) ++e;
                for (size_t c = b; c < e; c += (size_t)cap) ent.emplace_back((int)c, (int)std::min(e, c + (size_t)cap));
                b = e;
            }
            std::stable_sort(ent.begin(), ent.end(), [](const std::pair<int, int>& x, const std::pair<int, int>& y) {
                return x.second - x.first > y.second - y.first;
            });
            for (auto& v : lanes) v.clear();
            for (const auto& [b, e] : ent) {
                int best = 0;
                for (int ln = 1; ln < 32; ++ln) if (lanes[ln].size() < lanes[best].size()) best = ln;
                for (int c = b; c < e; ++c)
                    lanes[best].push_back((uint32_t)(cells[c] >> 32) | (uint32_t)(cells[c] & 0xff) << 16 | (c + 1 == e ? kPlanLast : 0u));
            }
            size_t rows = 0;
            for (const auto& v : lanes) rows = std::max(rows, v.size());
            rows_of[g] = (int64_t)rows;
            std::vector<uint32_t>& dst = part[t];
            for (size_t r = 0; r < rows; ++r)
                for (int ln = 0; ln < 32; ++ln) dst.push_back(r < lanes[ln].size() ? lanes[ln][r] : 0u);
        }
    };
    {
        std::vector<std::thread> th;
        for (int t = 1; t < T; ++t) th.emplace_back(plan, t);
        plan(0);
        for (auto& x : th) x.join();
    }
    out.pgoff.assign((size_t)n_rg + 1, 0);
    for (int64_t g = 0; g < n_rg; ++g) out.pgoff[g + 1] = out.pgoff[g] + rows_of[g] * 32;
    out.pwords.clear();
    out.pwords.reserve((size_t)out.pgoff[n_rg] + 32);
    for (int t = 0; t < T; ++t) { out.pwords.insert(out.pwords.end(), part[t].begin(), part[t].end()); std::vector<uint32_t>().swap(part[t]); }
    out.pwords.resize((size_t)out.pgoff[n_rg] + 32, 0u);
}

SegmentedStringsJob::SegmentedStringsJob() : st(new State) {}
SegmentedStringsJob::~SegmentedStringsJob() { delete st; }

void compile_corpus_segmented(const HostFsa& f, const LatticeArcs& A, const uint8_t* alive, const int32_t* tokens,
                              const int64_t* offs, const double* p, const std::vector<int32_t>& ids, int n_slots,
                              double fx_scale, SegmentedCorpus& out)
{
    std::shared_ptr<SegmentedStringsJob> job = compile_corpus_regions(f, A, alive, tokens, offs, p, ids, n_slots, fx_scale, out);
    job->run(out);
}

std::shared_ptr<SegmentedStringsJob> compile_corpus_regions(const HostFsa& f, const LatticeArcs& A, const uint8_t* alive,
                                                            const int32_t* tokens, const int64_t* offs, const double* p,
                                                            const std::vector<int32_t>& ids, int n_slots, double fx_scale,
                                                            SegmentedCorpus& out)
{
    const auto t_begin = std::chrono::steady_clock::now();
    const bool report = getenv("WFSA_COMPILE_TIMES") != nullptr;        // phase times of this function to stderr
    auto t_last = t_begin;
    auto lap = [&](const char* what) {
        const auto now = std::chrono::steady_clock::now();
        if (report) fprintf(stderr, "[segmented compile] %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
        t_last = now;
    };
    out = SegmentedCorpus();
    const size_t n = ids.size();
    out.const_acc.assign(A.n_arcs, 0);
    unsigned hw = std::thread::hardware_concurrency();
    const int T = (int)std::max<size_t>(1, std::min<size_t>({(size_t)(hw ? hw : 4), (size_t)64, n / 256 + 1}));
    // ---- 1. per-string compilation, strings i = t, t+T, ... on thread t
    using Local = SegLocal;
    std::vector<Local> loc(T);
    auto work = [&](int t) {
        Local& L = loc[t];
        LatticeScratch S; SegString seg;
        L.cacc.assign(A.n_arcs, 0);
        L.boff.push_back(0); L.sreg.push_back(0);
        for (size_t i = t; i < n; i += T) {
            const int32_t sid = ids[i];
            const int len = (int)(offs[sid + 1] - offs[sid]);
            const int rc = compile_segments(f, A, alive, tokens + offs[sid], len, n_slots, S, seg);
            L.status.push_back((int8_t)rc);
            if (rc == 1) {
                const long long c = llrint(p[sid] * fx_scale);
                for (uint16_t a : seg.bridges) L.cacc[a] += c;
                L.bridges.insert(L.bridges.end(), seg.bridges.begin(), seg.bridges.end());
                for (size_t r = 0; r + 1 < seg.roff.size(); ++r) {
                    const int b = seg.roff[r], e = seg.roff[r + 1];
                    L.rbeg.push_back((int64_t)L.rwords.size()); L.rlen.push_back(e - b);
                    L.rhash.push_back(fnv1a(seg.rwords.data() + b, (size_t)(e - b)));
                    for (int k = b; k < e; ++k) L.region_edges += (seg.rwords[k] >> 31);
                    L.rwords.insert(L.rwords.end(), seg.rwords.begin() + b, seg.rwords.begin() + e);
                }
            }
            L.boff.push_back((int64_t)L.bridges.size());
            L.sreg.push_back((int64_t)L.rbeg.size());
        }
    };
    {
        std::vector<std::thread> th;
        for (int t = 1; t < T; ++t) th.emplace_back(work, t);
        work(0);
        for (auto& x : th) x.join();
    }
    for (int t = 0; t < T; ++t)
        for (int a = 0; a < A.n_arcs; ++a) out.const_acc[a] += loc[t].cacc[a];
    lap("per-string compilation");
    // ---- 2. merge identical regions into types, strings visited in `ids` order (deterministic weights)
    // Partitioned by hash: partition k (one thread) merges the regions whose hash falls into it, walking ALL accepted
    // strings in `ids` order, so every type still sums the p_s of its instances in that order and keeps the first
    // instance as its representative: the result does not depend on the number of threads.
    struct Type { int t; int64_t beg; int32_t len; double W; };
    std::vector<std::vector<int32_t>> reg_type(T);                        // type of every region, per compile thread
    for (int t = 0; t < T; ++t) reg_type[t].resize(loc[t].rbeg.size());
    std::vector<int64_t> ok;                                              // indices into ids
    for (size_t i = 0; i < n; ++i) {
        const Local& L = loc[i % T];
        const size_t j = i / T;
        const int st = L.status[j];
        if (st < 0) { out.overflow.push_back(ids[i]); continue; }
        if (st == 0) { out.rejected.push_back(ids[i]); continue; }
        ok.push_back((int64_t)i);
        out.n_bridge += L.boff[j + 1] - L.boff[j];
        out.n_region_instances += L.sreg[j + 1] - L.sreg[j];
    }
    const int K = std::max(1, std::min(T, 32));
    auto part_of = [K](uint64_t h) { return (int)((h >> 40) % (uint64_t)K); };
    std::vector<std::vector<Type>> ptypes(K);
    auto merge_part = [&](int k) {
        std::vector<Type>& types = ptypes[k];
        std::vector<int32_t> bucket_head((size_t)1 << 18, -1);            // open hashing on the low hash bits
        std::vector<int32_t> next_in_bucket;
        std::vector<uint64_t> thash;
        for (const int64_t i : ok) {
            const Local& L = loc[i % T];
            const size_t j = (size_t)(i / T);
            const double ps = p[ids[i]];
            for (int64_t r = L.sreg[j]; r < L.sreg[j + 1]; ++r) {
                const uint64_t h = L.rhash[r];
                if (part_of(h) != k) continue;
                const uint32_t* w = L.rwords.data() + L.rbeg[r];
                const int32_t len = L.rlen[r];
                int32_t& head = bucket_head[h & (bucket_head.size() - 1)];
                int32_t ty = head;
                for (; ty >= 0; ty = next_in_bucket[ty]) {
                    const Type& Y = types[ty];
                    if (thash[ty] == h && Y.len == len && !std::memcmp(loc[Y.t].rwords.data() + Y.beg, w, (size_t)len * 4)) break;
                }
                if (ty < 0) {
                    ty = (int32_t)types.size();
                    types.push_back(Type{(int)(i % T), L.rbeg[r], len, 0.0});
                    thash.push_back(h); next_in_bucket.push_back(head); head = ty;
                }
                types[ty].W += ps;
                reg_type[i % T][r] = ty;                                  // index inside the partition; made global below
            }
        }
    };
    {
        std::vector<std::thread> th;
        for (int k = 1; k < K; ++k) th.emplace_back(merge_part, k);
        merge_part(0);
        for (auto& x : th) x.join();
    }
    std::vector<int32_t> pbase(K + 1, 0);
    for (int k = 0; k < K; ++k) pbase[k + 1] = pbase[k] + (int32_t)ptypes[k].size();
    std::vector<Type> types;
    types.reserve((size_t)pbase[K]);
    for (int k = 0; k < K; ++k) { types.insert(types.end(), ptypes[k].begin(), ptypes[k].end()); std::vector<Type>().swap(ptypes[k]); }
    {
        auto globalise = [&](int t) {                                     // regions of rejected strings hold a meaningless 0: harmless
            const Local& L = loc[t];
            for (size_t r = 0; r < reg_type[t].size(); ++r) reg_type[t][r] += pbase[part_of(L.rhash[r])];
        };
        std::vector<std::thread> th;
        for (int t = 1; t < T; ++t) th.emplace_back(globalise, t);
        globalise(0);
        for (auto& x : th) x.join();
    }
    for (int t = 0; t < T; ++t) out.n_region_edges += loc[t].region_edges;
    out.n_strings = (int64_t)ok.size();
    out.n_types = (int64_t)types.size();
    lap("type merging");
    // ---- 3. KR layout: types by class, sorted by content.  Class key (descending = roughly by cost):
    //   DAG form, big   : 3<<24 | rows          rows = padded stream length (multiple of 16), groups may mix rows
    //   DAG form, small : 2<<24 | rows          rows = 4, 8, 12, 16 bare edge words
    //   path form       : 1<<24 | P'<<8 | L     P' = paths padded to 2, 3, 4, 6 or 8; word (l, p) at row l*P' + p
    auto pad_paths = [](int P) { return P <= 4 ? std::max(P, 2) : (P <= 6 ? 6 : 8); };
    auto class_of = [&](const Type& Y) -> int {
        const uint32_t* w = loc[Y.t].rwords.data() + Y.beg;
        if (!(w[0] >> 31)) return (1 << 24) | pad_paths((int)((w[0] >> 8) & 0xff)) << 8 | (int)(w[0] & 0xff);     // path form header
        int edges = 0;
        bool fin = false;
        for (int32_t k = 0; k < Y.len; ++k) { edges += (w[k] >> 31); fin = fin || (!(w[k] >> 31) && (w[k] & kLatFin)); }
        if (!fin) return (2 << 24) | (edges + kSegSmallStep - 1) / kSegSmallStep * kSegSmallStep;
        return (3 << 24) | (Y.len + kCheckEvery - 1) / kCheckEvery * kCheckEvery;
    };
    auto rows_of_class = [](int c) { return (c >> 24) == 1 ? ((c >> 8) & 0xff) * (c & 0xff) : (c & 0xffffff); };
    std::vector<int32_t> order(types.size()), tcls(types.size());
    {
        auto classify = [&](int t) {
            const size_t i0 = types.size() * (size_t)t / T, i1 = types.size() * (size_t)(t + 1) / T;
            for (size_t i = i0; i < i1; ++i) { order[i] = (int32_t)i; tcls[i] = class_of(types[i]); }
        };
        std::vector<std::thread> th;
        for (int t = 1; t < T; ++t) th.emplace_back(classify, t);
        classify(0);
        for (auto& x : th) x.join();
    }
    auto type_less = [&](int32_t a, int32_t b) {
        if (tcls[a] != tcls[b]) return tcls[a] > tcls[b];
        const Type &X = types[a], &Y = types[b];
        const uint32_t* wa = loc[X.t].rwords.data() + X.beg; const uint32_t* wb = loc[Y.t].rwords.data() + Y.beg;
        const int32_t m = std::min(X.len, Y.len);
        for (int32_t k = 0; k < m; ++k) if (wa[k] != wb[k]) return (wa[k] & 0xffffu) != (wb[k] & 0xffffu) ? (wa[k] & 0xffffu) < (wb[k] & 0xffffu) : wa[k] < wb[k];
        return X.len < Y.len;
    };
    {
        // types are pairwise different, so the order is total: chunks sorted on the compile threads and merged pairwise
        // give the same permutation as one std::sort
        const int parts = order.size() >= 4096 ? std::min(T, 16) : 1;
        std::vector<size_t> cut(parts + 1);
        for (int k = 0; k <= parts; ++k) cut[k] = order.size() * (size_t)k / parts;
        {
            std::vector<std::thread> th;
            for (int k = 1; k < parts; ++k) th.emplace_back([&, k] { std::sort(order.begin() + cut[k], order.begin() + cut[k + 1], type_less); });
            std::sort(order.begin() + cut[0], order.begin() + cut[1], type_less);
            for (auto& x : th) x.join();
        }
        for (int width = 1; width < parts; width *= 2) {
            std::vector<std::thread> th;
            for (int k = 0; k + width < parts; k += 2 * width) {
                const size_t lo = cut[k], mid = cut[k + width], hi = cut[std::min(k + 2 * width, parts)];
                th.emplace_back([&, lo, mid, hi] { std::inplace_merge(order.begin() + lo, order.begin() + mid, order.begin() + hi, type_less); });
            }
            for (auto& x : th) x.join();
        }
    }
    std::vector<int32_t> type_slot(types.size(), -1);                     // type -> g*32 + lane
    out.rgoff.assign(1, 0);
    {
        size_t i = 0;
        while (i < order.size()) {
            const int cls = tcls[order[i]];
            const bool bigdag = (cls >> 24) == 3;
            size_t j = i;
            // a group holds up to 32 types of one class (big DAGs: any big class, rows of its first = longest)
            while (j < order.size() && j - i < 32 && (bigdag ? (tcls[order[j]] >> 24) == 3 : tcls[order[j]] == cls)) ++j;
            const int64_t g = (int64_t)out.rgrows.size();
            const int rows = rows_of_class(cls);
            out.rgrows.push_back((cls >> 24) == 1 ? (0x10000 | (cls & 0xffff)) : rows);
            out.rgoff.push_back(out.rgoff.back() + (int64_t)rows * 32);
            for (size_t k = i; k < j; ++k) type_slot[order[k]] = (int32_t)(g * 32 + (int64_t)(k - i));
            if (bigdag) out.max_big_rows = std::max<int64_t>(out.max_big_rows, rows);
            i = j;
        }
    }
    const int64_t n_rg = (int64_t)out.rgrows.size();
    out.rwords.assign((size_t)out.rgoff[n_rg] + 32, 0u);
    out.typeW.assign((size_t)n_rg * 32, 0.0);
    {
        // filled on the compile threads: thread t takes a contiguous range of groups (padding cells) and of the sorted
        // type order (words of the types: different lanes of a group never share a word)
        std::vector<int64_t> edges_of(T, 0);
        auto fill_regions = [&](int t) {
            const int64_t g0 = n_rg * t / T, g1 = n_rg * (t + 1) / T;
            for (int64_t g = g0; g < g1; ++g)
                if (out.rgrows[g] & 0x10000) {                            // path form: every unused cell reads the zero-weight arc
                    uint32_t* dst = out.rwords.data() + out.rgoff[g];
                    const int64_t cells = out.rgoff[g + 1] - out.rgoff[g];
                    for (int64_t k = 0; k < cells; ++k) dst[k] = (uint32_t)A.n_arcs;
                }
        };
        auto fill_types = [&](int t) {
            const size_t i0 = order.size() * (size_t)t / T, i1 = order.size() * (size_t)(t + 1) / T;
            int64_t ne = 0;
            for (size_t i = i0; i < i1; ++i) {
                const size_t ty = (size_t)order[i];
                const Type& Y = types[ty];
                const int32_t slot = type_slot[ty];
                const int64_t g = slot >> 5; const int l = slot & 31;
                const uint32_t* w = loc[Y.t].rwords.data() + Y.beg;
                uint32_t* dst = out.rwords.data() + out.rgoff[g] + l;
                if (!(w[0] >> 31)) {
                    const int P = (int)((w[0] >> 8) & 0xff), L = (int)(w[0] & 0xff), PP = pad_paths(P);
                    for (int el = 0; el < L; ++el)
                        for (int q = 0; q < P; ++q) dst[(size_t)(el * PP + q) * 32] = w[1 + el * P + q] & 0xffffu;
                    ne += (int64_t)P * L;
                } else {
                    for (int32_t k = 0; k < Y.len; ++k) { dst[(size_t)k * 32] = w[k]; ne += (w[k] >> 31); }
                }
                out.typeW[slot] = Y.W;
            }
            edges_of[t] = ne;
        };
        {
            std::vector<std::thread> th;
            for (int t = 1; t < T; ++t) th.emplace_back(fill_regions, t);
            fill_regions(0);
            for (auto& x : th) x.join();
        }
        {
            std::vector<std::thread> th;
            for (int t = 1; t < T; ++t) th.emplace_back(fill_types, t);
            fill_types(0);
            for (auto& x : th) x.join();
        }
        for (int t = 0; t < T; ++t) out.n_type_edges += edges_of[t];
    }
    lap("region layout");
    build_path_plans(out, A.n_arcs, T);
    lap("reduction plans");
    out.host_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    auto job = std::make_shared<SegmentedStringsJob>();
    SegmentedStringsJob::State& S = *job->st;
    S.loc = std::move(loc); S.T = T; S.n_arcs = A.n_arcs; S.ok = std::move(ok); S.reg_type = std::move(reg_type);
    S.type_slot = std::move(type_slot); S.n_rg = n_rg; S.ids = ids; S.p = p;
    return job;
}

// ---- 4. KS layout: strings by bridge count, longest first; the bridges of the 16 strings of a half-warp are
//         scheduled so that the 16 table reads of one shared-memory phase fall into 16 different bank pairs
void SegmentedStringsJob::run(SegmentedCorpus& out)
{
    const auto t_begin = std::chrono::steady_clock::now();
    const bool report = getenv("WFSA_COMPILE_TIMES") != nullptr;
    auto t_last = t_begin;
    auto lap = [&](const char* what) {
        const auto now = std::chrono::steady_clock::now();
        if (report) fprintf(stderr, "[segmented compile] %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
        t_last = now;
    };
    using Local = SegLocal;
    std::vector<Local>& loc = st->loc;
    const int T = st->T;
    std::vector<int64_t>& ok = st->ok;
    const std::vector<std::vector<int32_t>>& reg_type = st->reg_type;
    const std::vector<int32_t>& type_slot = st->type_slot;
    const int64_t n_rg = st->n_rg;
    const std::vector<int32_t>& ids = st->ids;
    const double* p = st->p;
    const struct { int n_arcs; } A = {st->n_arcs};
    const int32_t dummy_type = (int32_t)(n_rg * 32);
    auto nbr = [&](int64_t i) { const Local& L = loc[i % T]; return (int)(L.boff[i / T + 1] - L.boff[i / T]); };
    auto nref = [&](int64_t i) { const Local& L = loc[i % T]; return (int)(L.sreg[i / T + 1] - L.sreg[i / T]); };
    std::stable_sort(ok.begin(), ok.end(), [&](int64_t a, int64_t b) {
        const int wa = nbr(a), wb = nbr(b);
        return wa != wb ? wa > wb : nref(a) > nref(b);
    });
    const int64_t n_sg = ((int64_t)ok.size() + 31) / 32;
    std::vector<std::vector<uint16_t>> gsched((size_t)n_sg);              // per group: [slots][32] arc ids
    std::vector<int32_t> gslots((size_t)n_sg, 0);
    auto schedule = [&](int t) {
        BridgeScheduler sch((uint16_t)A.n_arcs);
        const uint16_t* ptr[16]; int cnt[16];
        std::vector<uint16_t> half[2];
        for (int64_t g = t; g < n_sg; g += T) {
            int slots[2] = {0, 0};
            for (int hh = 0; hh < 2; ++hh) {
                for (int l = 0; l < 16; ++l) {
                    const int64_t k = g * 32 + hh * 16 + l;
                    if (k < (int64_t)ok.size()) {
                        const int64_t i = ok[k];
                        const Local& L = loc[i % T];
                        ptr[l] = L.bridges.data() + L.boff[i / T]; cnt[l] = (int)(L.boff[i / T + 1] - L.boff[i / T]);
                    } else { ptr[l] = nullptr; cnt[l] = 0; }
                }
                slots[hh] = sch.run(ptr, cnt, half[hh]);
            }
            const int S2 = (std::max(slots[0], slots[1]) + 1) / 2 * 2;       // two slots per word
            gslots[g] = S2;
            std::vector<uint16_t>& G = gsched[g];
            G.resize((size_t)S2 * 32);
            for (int s2 = 0; s2 < S2; ++s2)
                for (int hh = 0; hh < 2; ++hh)
                    for (int l = 0; l < 16; ++l)
                        G[(size_t)s2 * 32 + hh * 16 + l] = s2 < slots[hh] ? half[hh][(size_t)s2 * 16 + l] : (uint16_t)(A.n_arcs + l);
        }
    };
    {
        std::vector<std::thread> th;
        for (int t = 1; t < T; ++t) th.emplace_back(schedule, t);
        schedule(0);
        for (auto& x : th) x.join();
    }
    lap("bridge scheduling");
    // super-groups of kKsSuper groups (the warps of one CTA), chunk-interleaved:
    //   word (sg, chunk c, group-in-super w, row j, lane l) at sgoff[sg] + (((c*kKsSuper + w)*kKsChunkRows + j)*32 + l
    // so that the warps of a CTA, walking their groups chunk by chunk, read one contiguous region together
    // (profiles/microbench_stream.cu: 5.6 TB/s against 4.3 TB/s for one private block per warp)
    const int64_t n_ssg = (n_sg + kKsSuper - 1) / kKsSuper;
    const int64_t n_sgp = n_ssg * kKsSuper;                                  // groups incl. the padding of the last super-group
    out.sgref.assign((size_t)n_sgp, 0);
    out.ksid.assign((size_t)n_sgp * 32, -1);
    out.kp.assign((size_t)n_sgp * 32, 0.0);
    out.sgoff.assign((size_t)n_ssg + 1, 0);
    for (int64_t g = 0; g < n_sg; ++g) {
        int mr = 0;
        for (int64_t k = g * 32; k < std::min<int64_t>((int64_t)ok.size(), g * 32 + 32); ++k) mr = std::max(mr, nref(ok[k]));
        out.sgref[g] = mr;
    }
    for (int64_t sg = 0; sg < n_ssg; ++sg) {
        int chunks = 1;
        for (int64_t g = sg * kKsSuper; g < std::min(n_sg, (sg + 1) * kKsSuper); ++g)
            chunks = std::max(chunks, (out.sgref[g] + gslots[g] / 2 + kKsChunkRows - 1) / kKsChunkRows);
        out.sgoff[sg + 1] = out.sgoff[sg] + (int64_t)chunks * kKsSuper * kKsChunkRows * 32;
    }
    out.swords.assign((size_t)out.sgoff[n_ssg] + 32, 0u);
    auto fill = [&](int t) {
        for (int64_t sg = t; sg < n_ssg; sg += T) {
            uint32_t* sbase = out.swords.data() + out.sgoff[sg];
            const int chunks = (int)((out.sgoff[sg + 1] - out.sgoff[sg]) / (kKsSuper * kKsChunkRows * 32));
            for (int w = 0; w < kKsSuper; ++w) {
                const int64_t g = sg * kKsSuper + w;
                const int mr = g < n_sg ? out.sgref[g] : 0;
                const int slots = g < n_sg ? gslots[g] : 0;
                auto at = [&](int row, int l) -> uint32_t& {
                    return sbase[(((size_t)(row / kKsChunkRows) * kKsSuper + w) * kKsChunkRows + row % kKsChunkRows) * 32 + l];
                };
                for (int l = 0; l < 32; ++l) {
                    const int64_t k = g * 32 + l;
                    for (int r = 0; r < mr; ++r) at(r, l) = (uint32_t)dummy_type;
                    if (g < n_sg && k < (int64_t)ok.size()) {
                        const int64_t i = ok[k];
                        const Local& L = loc[i % T];
                        const size_t j = i / T;
                        out.ksid[k] = ids[i]; out.kp[k] = p[ids[i]];
                        int r = 0;
                        for (int64_t q = L.sreg[j]; q < L.sreg[j + 1]; ++q, ++r) at(r, l) = (uint32_t)type_slot[reg_type[i % T][q]];
                    }
                    const uint32_t padw = (uint32_t)(A.n_arcs + (l & 15)) * 0x10001u;     // both halves: the lane's own padding entry
                    for (int row = mr; row < chunks * kKsChunkRows; ++row) {
                        const int s2 = (row - mr) * 2;
                        at(row, l) = s2 < slots ? (uint32_t)gsched[g][(size_t)s2 * 32 + l] | ((uint32_t)gsched[g][(size_t)(s2 + 1) * 32 + l] << 16) : padw;
                    }
                }
                if (g < n_sg) std::vector<uint16_t>().swap(gsched[g]);
            }
        }
    };
    {
        std::vector<std::thread> th;
        for (int t = 1; t < T; ++t) th.emplace_back(fill, t);
        fill(0);
        for (auto& x : th) x.join();
    }
    lap("per-string layout fill");
    out.host_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
}

}  // namespace wfsa
