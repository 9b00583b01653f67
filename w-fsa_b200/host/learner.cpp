// w-fsa_b200/host/learner.cpp -- see learner.hpp.
#include "learner.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <deque>
#include <map>
#include <numeric>
#include <sstream>

namespace wfsa {

double LogFactorial(size_t d)               // src/Utils.cpp:244-261
{
    static std::vector<double> memory(2, 0.0);
    if (memory.size() > d) return memory[d];
    double result = memory.back();
    for (size_t i = memory.size(); i <= d; ++i) { result += std::log((double)i); memory.push_back(result); }
    return result;
}
double LogSimplexVolume(size_t d) { return d > 0 ? 0.5 * std::log((double)d) - LogFactorial(d - 1) : 0.0; }   // src/Utils.cpp:221-227
double mxlogx(double x) { return x > 0 ? x * (-std::log(x)) : (x == 0 ? 0.0 : INFINITY); }                    // src/Utils.cpp:234-242

Learner::Learner() {}
Learner::~Learner() { if (dev) wfsa_dev_destroy(dev); }

void Learner::check(int rc, const char* what) const
{
    if (rc == WFSA_OK) return;
    std::ostringstream o;
    o << what << " failed (" << rc << "): " << wfsa_dev_last_error(dev);
    throw LearnerError(o.str());
}

void Learner::AllReduceHost(double* v, int n)
{
    if (opts.nranks > 1) check(wfsa_dev_allreduce_f64(dev, v, n, 0), "wfsa_dev_allreduce_f64");
}

// ---------------------------------------------------------------------------------------------
void Learner::BuildConstraints(const Fsa& fsa)       // src/Learner.cpp:221-265
{
    model_volume = 0;
    const size_t n_raw = fsa.GetNumberOfParameters();
    _x.assign(n_raw, 0.0);
    Ccol_raw.assign(n_raw, 0);
    int k = 0;
    size_t next = 0;
    auto collect = [&](size_t size, auto&& edge_at) {
        if (size <= 1) return;
        for (size_t i = 0; i < size; ++i) {
            const auto e = edge_at(i);
            if ((size_t)e.first != next) {
                std::ostringstream o; o << "Indexing error: " << e.first << " != " << next;
                throw LearnerError(o.str());
            }
            Ccol_raw[next] = k;
            _x[next] = e.second;
            ++next;
        }
        ++k;
        model_volume += LogSimplexVolume(size);
    };
    for (const auto& s : fsa.States()) {
        collect(s.emissions.size(), [&](size_t i) { return std::make_pair(s.emissions[i].index, s.emissions[i].logprob); });
        collect(s.transitions.size(), [&](size_t i) { return std::make_pair(s.transitions[i].index, s.transitions[i].logprob); });
    }
}

void Learner::BuildFrom(const Fsa& fsa, const Corpus& corpus, bool)
{
    BuildConstraints(fsa);
    BuildPaths(fsa, corpus);
    Trim();
    check(wfsa_dev_set_param_map(dev, trimmed_weights.data(), GetNumberOfParameters(), recognised.data()),
          "wfsa_dev_set_param_map");
}

// Recognition: the reference enumerates every accepting path of every word
// (src/Learner.cpp:276-348); here one structural forward-backward pass on the device returns
// recognised flags, path counts and the used-parameter flags that Trim needs.
void Learner::BuildPaths(const Fsa& fsa, const Corpus& corpus)
{
    fsa_ptr = &fsa;
    lower_fsa(fsa, lowered);
    size_t first = 0, count = corpus.size();
    if (opts.nranks > 1) {
        const auto cut = balanced_ranges(corpus, opts.nranks);
        first = cut[opts.rank]; count = cut[opts.rank + 1] - cut[opts.rank];
    }
    lower_corpus(corpus, lowered, first, count, shard);
    shard_words.clear();
    for (size_t i = first; i < first + count; ++i) shard_words.push_back(corpus[i].first);

    wfsa_dev_options o{};
    o.device = opts.device; o.force_kernel = opts.force_kernel; o.accum_mode = opts.accum_mode; o.reserved = opts.accum_variant;
    const wfsa_fsa_desc fd = lowered.desc();
    const wfsa_corpus_desc cd = shard.desc();
    if (dev) { wfsa_dev_destroy(dev); dev = nullptr; }
    const int rc = wfsa_dev_create(&fd, &cd, &o, &dev);
    if (rc != WFSA_OK) {
        std::ostringstream m; m << "wfsa_dev_create failed (" << rc << "): " << wfsa_dev_last_error(nullptr);
        throw LearnerError(m.str());
    }
    if (opts.nranks > 1) check(wfsa_dev_comm_init(dev, opts.unique_id, opts.rank, opts.nranks), "wfsa_dev_comm_init");

    recognised.assign(count, 0);
    path_counts.assign(count, 0.0);
    std::vector<uint8_t> used(lowered.n_raw, 0);
    check(wfsa_dev_structure(dev, recognised.data(), path_counts.data(), used.data()), "wfsa_dev_structure");

    trimmed_weights.assign(lowered.n_raw, -2);          // per default every index is unused
    for (int i = 0; i < lowered.n_raw; ++i) if (used[i]) trimmed_weights[i] = 0;

    p.clear();
    common_support = 0.0; aux_hessian = 0.0; auxiliary_parameters = 0; n_paths = 0.0;
    double all_unique = 1.0;
    for (size_t s = 0; s < count; ++s) {
        if (recognised[s]) {
            common_support += shard.p[s];
            p.push_back(shard.p[s]);
            n_paths += path_counts[s];
            if (path_counts[s] != 1.0) all_unique = 0.0;
        } else {
            ++auxiliary_parameters;
            aux_hessian -= std::log(shard.p[s]);
        }
    }
    double v[6] = {common_support, aux_hessian, (double)auxiliary_parameters, n_paths, (double)p.size(), all_unique};
    AllReduceHost(v, 6);
    common_support = v[0]; aux_hessian = v[1]; auxiliary_parameters = (size_t)std::llround(v[2]); n_paths = v[3];
    n_strings = (int)std::llround(v[4]);
    unique_paths = (v[5] == (double)opts.nranks) || n_strings == 0;
    have_blocks = false;
}

void Learner::Trim()                                   // src/Learner.cpp:350-425
{
    const int n_raw = (int)trimmed_weights.size();
    int c = -1, nnz_in_c = -1;
    for (int i = 0; i < n_raw; ++i) {
        const int this_c = Ccol_raw[i];
        if (this_c != c) {
            c = this_c;
            if (nnz_in_c >= 0) trimmed_weights[nnz_in_c] = -1;   // lone survivor of a constraint is pinned
            nnz_in_c = -1;
        }
        if (trimmed_weights[i] >= 0) nnz_in_c = (nnz_in_c == -1) ? i : -2;
    }
    if (nnz_in_c >= 0) trimmed_weights[nnz_in_c] = -1;
    Ccol.clear();
    int good_indices = 0, good_constraints = -1;
    c = -1;
    for (int i = 0; i < n_raw; ++i) {
        if (trimmed_weights[i] == 0) {
            trimmed_weights[i] = good_indices++;
            if (trimmed_weights[i] < i) _x[trimmed_weights[i]] = _x[i];
            if (c < Ccol_raw[i]) { ++good_constraints; c = Ccol_raw[i]; }
            Ccol.push_back(good_constraints);
        }
    }
    _x.resize(good_indices);
}

double Learner::GetWeight(int i) const                 // src/Learner.cpp:427-436
{
    switch (trimmed_weights[i]) {
    case -2: return -INFINITY;
    case -1: return 0.0;
    default: return _x[trimmed_weights[i]];
    }
}

void Learner::RewriteWeights(Fsa& fsa) const
{
    for (auto& s : fsa.States()) {
        for (auto& e : s.emissions) e.logprob = e.index >= 0 ? GetWeight(e.index) : 0.0;
        for (auto& t : s.transitions) t.logprob = t.index >= 0 ? GetWeight(t.index) : 0.0;
    }
}

void Learner::Renormalize()
{
    const int n = GetNumberOfParameters(), k = GetNumberOfConstraints();
    std::vector<double> g(k, 0.0);
    for (int i = 0; i < n; ++i) g[Ccol[i]] += std::exp(_x[i]);
    for (int j = 0; j < k; ++j) g[j] = std::log(g[j]);
    for (int i = 0; i < n; ++i) _x[i] -= g[Ccol[i]];
}

void Learner::LambdaUpdate(double* lstep, double* l, double eta, bool exponential) const
{
    const int k = GetNumberOfConstraints();
    if (!exponential) {
        for (int j = 0; j < k; ++j) l[j] -= eta * lstep[j];
    } else {
        for (int j = 0; j < k; ++j) l[j] *= std::exp(-eta * (lstep[j] / l[j]));
    }
}

void Learner::Finalize()
{
    double s = 0.0;
    for (double v : p) s += v * std::log(v);
    AllReduceHost(&s, 1);
    plogp = s;
    grad_cache.assign(GetNumberOfParameters(), 0.0);
    FinalizeCallback();
}

void Learner::Init(int flags, const double* initialx)
{
    if (initialx) std::copy(initialx, initialx + GetNumberOfParameters(), _x.begin());
    InitCallback(flags);
}

void Learner::EvalAt(const double* x)
{
    check(wfsa_dev_eval(dev, x, &loglik, nullptr, grad_cache.data()), "wfsa_dev_eval");
    logq_cache.clear();
}

void Learner::ComputeModeledProbs() { EvalAt(_x.data()); }

void Learner::ComputeObjective() { kl = plogp - loglik; }

const std::vector<double>& Learner::LogQ()
{
    if (logq_cache.empty()) {
        std::vector<double> all(recognised.size());
        check(wfsa_dev_eval_fetch(dev, nullptr, all.data(), nullptr), "wfsa_dev_eval_fetch");
        for (size_t s = 0; s < recognised.size(); ++s) if (recognised[s]) logq_cache.push_back(all[s]);
    }
    return logq_cache;
}

void Learner::Decode(Decoding& d, int k) { DecodePaths(d, k, false, 0); }

void Learner::Sample(Decoding& d, int n, uint64_t seed) { DecodePaths(d, n, true, seed); }

void Learner::DecodePaths(Decoding& d, int k, bool sample, uint64_t seed)
{
    const size_t ns = shard_words.size(), np = ns * (size_t)k;
    d.k = k;
    d.logw.assign(std::max<size_t>(np, 1), 0.0); d.logq.assign(std::max<size_t>(ns, 1), 0.0); d.path_off.assign(np + 1, 0);
    if (sample) check(wfsa_dev_sample(dev, _x.data(), k, seed, d.logw.data(), d.logq.data(), d.path_off.data()), "wfsa_dev_sample");
    else {
        double ll = 0.0;
        std::vector<double> g(std::max(GetNumberOfParameters(), 1));
        check(wfsa_dev_eval(dev, _x.data(), &ll, d.logq.data(), g.data()), "wfsa_dev_eval");
        if (k == 1) check(wfsa_dev_viterbi(dev, _x.data(), d.logw.data(), d.path_off.data()), "wfsa_dev_viterbi");
        else check(wfsa_dev_nbest(dev, _x.data(), k, d.logw.data(), d.path_off.data()), "wfsa_dev_nbest");
    }
    d.trans_edge.assign(std::max<int64_t>(d.path_off[np], 1), 0); d.emis_edge.assign(d.trans_edge.size(), 0);
    check(wfsa_dev_viterbi_paths(dev, d.trans_edge.data(), d.emis_edge.data()), "wfsa_dev_viterbi_paths");
    d.logw.resize(np); d.logq.resize(ns); d.trans_edge.resize(d.path_off[np]); d.emis_edge.resize(d.path_off[np]);
}

// ---------------------------------------------------------------------------------------------
// Route A of SURVEY.md section 7: enumerate the paths of AMBIGUOUS strings only (structure,
// once), ship dense count blocks; the numeric contraction runs on the device.
// Which parameters a step counts follows src/Learner.cpp:285-293; the per-string index set
// drops (column,count) pairs that are identical on every path (src/HessianLearner.cpp:409-443).
void Learner::BuildPathBlocks()
{
    if (have_blocks) return;
    const Fsa& fsa = *fsa_ptr;
    const auto& S = fsa.States();
    const int end = fsa.EndIndex();
    std::vector<int64_t> path_off{0}, col_off{0}, val_off{0};
    std::vector<int32_t> cols;
    std::vector<double> counts, bp;
    struct Item { size_t pos; int state; std::map<int, double> hist; };
    const double limit = 4e6;
    double total = 0;
    for (size_t s = 0; s < shard_words.size(); ++s) if (recognised[s] && path_counts[s] > 1.0) total += path_counts[s];
    {   // with several ranks every rank must fail together: wfsa_dev_set_path_blocks below is collective
        double too_many = total > limit ? 1.0 : 0.0;
        if (opts.nranks > 1) check(wfsa_dev_allreduce_f64(dev, &too_many, 1, 1), "wfsa_dev_allreduce_f64");
        if (too_many > 0.0) throw LearnerError("too many paths to enumerate for the H_f blocks");
    }
    for (size_t s = 0; s < shard_words.size(); ++s) {
        if (!recognised[s] || !(path_counts[s] > 1.0)) continue;
        const std::string& w = shard_words[s];
        std::vector<std::map<int, double>> paths;
        std::deque<Item> queue;
        queue.push_back({0, fsa.StartIndex(), {}});
        while (!queue.empty()) {
            Item it = std::move(queue.front());
            queue.pop_front();
            for (const auto& tr : S[it.state].transitions) {
                auto add = [&](std::map<int, double>& h, int raw) {
                    if (raw >= 0 && trimmed_weights[raw] >= 0) h[trimmed_weights[raw]] += 1.0;
                };
                if (tr.next == end) {
                    if (it.pos == w.size()) { auto h = it.hist; add(h, tr.index); paths.push_back(std::move(h)); }
                    continue;
                }
                for (const auto& em : S[tr.next].emissions) {
                    if (w.compare(it.pos, em.str.size(), em.str) != 0 || it.pos + em.str.size() > w.size()) continue;
                    Item nx{it.pos + em.str.size(), tr.next, it.hist};
                    add(nx.hist, tr.index);
                    add(nx.hist, em.index);
                    queue.push_back(std::move(nx));
                }
            }
        }
        if ((double)paths.size() != path_counts[s]) {
            std::ostringstream o;
            o << "path enumeration found " << paths.size() << " paths where the device counted " << path_counts[s];
            throw LearnerError(o.str());
        }
        std::map<int, int> colset;
        for (const auto& h : paths) for (const auto& kv : h) colset[kv.first] = 0;
        std::vector<int> keep;
        for (const auto& kv : colset) {
            const int j = kv.first;
            bool same = true;
            auto first = paths[0].find(j);
            const double c0 = first == paths[0].end() ? 0.0 : first->second;
            for (const auto& h : paths) {
                auto f = h.find(j);
                if ((f == h.end() ? 0.0 : f->second) != c0) { same = false; break; }
            }
            if (!same) keep.push_back(j);
        }
        // NB: the path posterior needs ALL columns, the Hessian only the varying ones; the
        // constant columns shift every path score of the string equally, so they cancel in r.
        for (int j : keep) cols.push_back(j);
        for (const auto& h : paths)
            for (int j : keep) { auto f = h.find(j); counts.push_back(f == h.end() ? 0.0 : f->second); }
        path_off.push_back(path_off.back() + (int64_t)paths.size());
        col_off.push_back((int64_t)cols.size());
        val_off.push_back((int64_t)counts.size());
        bp.push_back(shard.p[s]);
    }
    wfsa_path_blocks b{};
    b.n_blocks = (int64_t)bp.size();
    b.path_off = path_off.data(); b.col_off = col_off.data(); b.val_off = val_off.data();
    b.cols = cols.data(); b.counts = counts.data(); b.p = bp.data();
    check(wfsa_dev_set_path_blocks(dev, &b), "wfsa_dev_set_path_blocks");
    have_blocks = true;
}

void Learner::ComputeHfDense(std::vector<double>& Hf, double* rmin)
{
    const int n = GetNumberOfParameters();
    Hf.assign((size_t)n * n, 0.0);
    if (HasUniquePaths()) { if (rmin) *rmin = 0.0; return; }
    double rm = 0.0;
    // The segmented backend derives the blocks of the contraction from its compiled region types (no path enumeration per
    // string); backends without a compiled form answer WFSA_ERR_STATE until they are given the blocks of the host
    // enumeration (route A: fixtures and small corpora only).
    int rc = wfsa_dev_hessian(dev, _x.data(), Hf.data(), &rm);
    if (rc == WFSA_ERR_STATE && !have_blocks) {
        BuildPathBlocks();
        rc = wfsa_dev_hessian(dev, _x.data(), Hf.data(), &rm);
    }
    check(rc, "wfsa_dev_hessian");
    if (rmin) *rmin = std::isfinite(rm) ? rm : 1.0;
}

// ---------------------------------------------------------------------------------------------
// QuasiNewtonLearner
// ---------------------------------------------------------------------------------------------
void QuasiNewtonLearner::FinalizeCallback()
{
    const int n = GetNumberOfParameters(), k = GetNumberOfConstraints();
    grad.assign(n, 0.0); expx.assign(n, 0.0); rhs.assign(n, 0.0);
    lambda.assign(k, 1.0); g.assign(k, 0.0);
}

void QuasiNewtonLearner::InitCallback(int flags)
{
    const int n = GetNumberOfParameters(), k = GetNumberOfConstraints();
    if (flags & 1) _x.assign(n, 0.0);
    if (flags & 2) Renormalize();
    if (flags & 4) {
        ComputeExpX();
        ComputeGrad();
        lambda.assign(k, 0.0);
        for (int i = 0; i < n; ++i) lambda[Ccol[i]] -= grad[i];     // l <- -C^t.gradf
    }
    exponential_lambda = (flags & 32) != 0;
}

void QuasiNewtonLearner::ComputeExpX() { for (size_t i = 0; i < expx.size(); ++i) expx[i] = std::exp(_x[i]); }

void QuasiNewtonLearner::ComputeG()
{
    const int n = GetNumberOfParameters(), k = GetNumberOfConstraints();
    g.assign(k, -1.0);
    for (int i = 0; i < n; ++i) g[Ccol[i]] += expx[i];
    g_min = *std::min_element(g.begin(), g.end());
    g_max = *std::max_element(g.begin(), g.end());
}

void QuasiNewtonLearner::ComputeGrad()
{
    ComputeModeledProbs();
    grad = Gradient();
}

void QuasiNewtonLearner::ComputeLambdaNext(std::vector<double>& result)
{
    const int n = GetNumberOfParameters(), k = GetNumberOfConstraints();
    result.assign(k, 0.0);
    for (int j = 0; j < k; ++j) result[j] = lambda[j] * g[j];
    for (int i = 0; i < n; ++i) result[Ccol[i]] -= grad[i];
    for (int j = 0; j < k; ++j) { g[j] += 1.0; result[j] /= g[j]; }
}

void QuasiNewtonLearner::OptimizationStep(double eta, bool)     // src/QuasiNewtonLearner.cpp:162-201
{
    const int n = GetNumberOfParameters(), k = GetNumberOfConstraints();
    ComputeExpX();
    ComputeG();
    ComputeGrad();
    ComputeObjective();
    rmin = ComputeRmin();                                  // relative_path_probs of this evaluation, src/QuasiNewtonLearner.cpp:80-84
    aux.assign(n, 0.0);
    for (int i = 0; i < n; ++i) { aux[i] = expx[i] * lambda[Ccol[i]]; rhs[i] = grad[i] + aux[i]; }
    grad_error = 0.0;
    for (int i = 0; i < n; ++i) grad_error = std::max(grad_error, std::fabs(rhs[i]));
    lambda_min = *std::min_element(lambda.begin(), lambda.end());
    std::vector<double> laux(k);
    ComputeLambdaNext(laux);
    for (int i = 0; i < n; ++i) {
        rhs[i] = (grad[i] + expx[i] * laux[Ccol[i]]) / aux[i];
        _x[i] -= eta * rhs[i];
    }
    for (int j = 0; j < k; ++j) laux[j] = lambda[j] - laux[j];
    LambdaUpdate(laux.data(), lambda.data(), eta, exponential_lambda);
}

std::string QuasiNewtonLearner::GetOptimizationHeader() const
{
    return "       KL   graderr     g_min     g_max lambdamin      rmin";
}

std::vector<double> QuasiNewtonLearner::GetOptimizationInfo()
{
    // rmin = smallest path posterior (src/QuasiNewtonLearner.cpp:80-84); its argmin is a path index of the reference's
    // enumeration order, which a DP backend does not have: reported as 0
    return {GetKLDistance(), grad_error, g_min, g_max, lambda_min, rmin, 0.0};
}

bool QuasiNewtonLearner::HaltCondition(double tol)
{
    return grad_error <= tol && std::fabs(g_min) <= tol && std::fabs(g_max) <= tol;
}

// smallest path posterior over all strings at the current x (the rmin column of both optimisers): the H_f entry point of the
// backend without its matrix, which needs no path enumeration on any kernel
double Learner::ComputeRmin()
{
    if (HasUniquePaths()) return 0.0;
    double rm = 0.0;
    check(wfsa_dev_hessian(dev, _x.data(), nullptr, &rm), "wfsa_dev_hessian");
    return std::isfinite(rm) ? rm : 1.0;
}

// ---------------------------------------------------------------------------------------------
// HessianLearner
// ---------------------------------------------------------------------------------------------
void HessianLearner::FinalizeCallback()
{
    rhs.assign(GetNumberOfAugmentedParameters(), 0.0);
    _x.resize(GetNumberOfAugmentedParameters(), 1.0);
    expx.assign(GetNumberOfParameters(), 0.0);
}

void HessianLearner::InitCallback(int flags)           // src/HessianLearner.cpp:132-191
{
    const int n = GetNumberOfParameters(), k = GetNumberOfConstraints();
    exponential_lambda = (flags & 32) != 0;
    if (flags & 1) { _x.assign(n, 0.0); _x.resize(n + k, 1.0); }
    if (flags & 2) Renormalize();
    if (flags & 4) InitSlackVariables();
    include_Hf = (flags & 8) != 0;
    degenerate = false;
    factored = false;
}

void HessianLearner::ComputeExpX() { for (size_t i = 0; i < expx.size(); ++i) expx[i] = std::exp(_x[i]); }

void HessianLearner::ComputeGrad()
{
    ComputeModeledProbs();
    std::copy(Gradient().begin(), Gradient().end(), rhs.begin());
}

void HessianLearner::ComputeG()
{
    const int n = GetNumberOfParameters(), k = GetNumberOfConstraints();
    for (int j = 0; j < k; ++j) rhs[n + j] = 0.0;
    for (int i = 0; i < n; ++i) rhs[n + Ccol[i]] += expx[i];
    for (int j = 0; j < k; ++j) rhs[n + j] -= 1.0;
}

void HessianLearner::InitSlackVariables()
{
    const int n = GetNumberOfParameters(), k = GetNumberOfConstraints();
    ComputeExpX();
    ComputeGrad();
    for (int j = 0; j < k; ++j) _x[n + j] = 0.0;
    for (int i = 0; i < n; ++i) _x[n + Ccol[i]] -= rhs[i];
}

void HessianLearner::ComputeRhs()
{
    const int n = GetNumberOfParameters();
    ComputeExpX();
    ComputeGrad();
    ComputeG();
    for (int i = 0; i < n; ++i) rhs[i] += expx[i] * _x[n + Ccol[i]];
}

void HessianLearner::ComputeHg()                        // src/HessianLearner.cpp:622-639
{
    const int n = GetNumberOfParameters(), N = GetNumberOfAugmentedParameters();
    const double* lambda = _x.data() + n;
    for (int i = 0; i < n; ++i) {
        H[(size_t)i * N + i] += expx[i] * lambda[Ccol[i]];
        H[(size_t)i * N + n + Ccol[i]] += expx[i];
        H[(size_t)(n + Ccol[i]) * N + i] += expx[i];
    }
}

// Newton system of the optimiser WITHOUT H_f:  [D B; B^T 0] [dx; dl] = [r_x; r_l]  with D = diag(e^x_i lambda_c(i)) and one entry
// e^x_i per row of B (every parameter sits in exactly one constraint, src/HessianLearner.cpp:622-639).  The Schur complement
// B^T D^-1 B on the multipliers is DIAGONAL, S_jj = sum_{i in j} e^x_i / lambda_j: solve and inertia in O(n) instead of a dense
// (n+k)^3 factorisation (the reference hands the same sparse matrix to MKL DSS, :100-113); inertia by Haynsworth,
// In(K) = In(D) + In(-S).  Returns false on a zero or non-finite pivot (the caller falls back to the dense factorisation).
bool SolveDiagonalKKT(int n, int k, const double* expx, const double* lambda, const int* Ccol, const double* rhs,
                      std::vector<double>& sol, int& pos, int& neg)
{
    std::vector<double> S(k, 0.0), t(k, 0.0);
    pos = neg = 0;
    for (int i = 0; i < n; ++i) {
        const double d = expx[i] * lambda[Ccol[i]];
        if (d == 0.0 || !std::isfinite(d)) return false;
        (d > 0 ? pos : neg)++;
        S[Ccol[i]] += expx[i] * expx[i] / d;
        t[Ccol[i]] += expx[i] * rhs[i] / d;
    }
    for (int j = 0; j < k; ++j) { if (S[j] == 0.0 || !std::isfinite(S[j])) return false; (S[j] < 0 ? pos : neg)++; }
    sol.assign((size_t)n + k, 0.0);
    for (int j = 0; j < k; ++j) sol[n + j] = (t[j] - rhs[n + j]) / S[j];
    for (int i = 0; i < n; ++i) sol[i] = (rhs[i] - expx[i] * sol[n + Ccol[i]]) / (expx[i] * lambda[Ccol[i]]);
    return true;
}

void HessianLearner::OptimizationStep(double eta, bool)  // src/HessianLearner.cpp:63-130
{
    const int n = GetNumberOfParameters(), N = GetNumberOfAugmentedParameters();
    ComputeRhs();
    ComputeObjective();
    rmin = 0.0;
    diag_solved = false;
    if (!include_Hf) {
        int pos = 0, neg = 0;
        if (SolveDiagonalKKT(n, N - n, expx.data(), _x.data() + n, Ccol.data(), rhs.data(), aux, pos, neg)) {
            diag_solved = true; diag_pos = pos; diag_neg = neg;
            lambda_min = *std::min_element(_x.begin() + n, _x.end());
            factored = true;
        }
    }
    if (diag_solved) {
        if (std::find_if(aux.begin(), aux.end(), [](double v) { return !std::isfinite(v); }) != aux.end()) diag_solved = false;
    }
    if (diag_solved) {
        for (int i = 0; i < n; ++i) _x[i] -= eta * aux[i];
        LambdaUpdate(aux.data() + n, _x.data() + n, eta, exponential_lambda);
        return;
    }
    H.assign((size_t)N * N, 0.0);
    if (include_Hf) {
        ComputeHfDense(Hf, &rmin);
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n; ++j) H[(size_t)i * N + j] += Hf[(size_t)i * n + j];
    }
    ComputeHg();
    lambda_min = *std::min_element(_x.begin() + n, _x.end());
    solver.Factor(N, H);
    factored = true;
    aux.assign(N, 0.0);
    solver.Solve(rhs.data(), aux.data());
    if (std::find_if(aux.begin(), aux.end(), [](double v) { return !std::isfinite(v); }) != aux.end()) {
        degenerate = true;
        fprintf(stderr, "Solution of Newton step is degenerate at %f%% of the parameters and %f%% of the constraints!\n",
                100.0 * std::count_if(aux.begin(), aux.begin() + n, [](double v) { return !std::isfinite(v); }) / n,
                100.0 * std::count_if(aux.begin() + n, aux.end(), [](double v) { return !std::isfinite(v); }) / GetNumberOfConstraints());
    } else {
        for (int i = 0; i < n; ++i) _x[i] -= eta * aux[i];
        LambdaUpdate(aux.data() + n, _x.data() + n, eta, exponential_lambda);
    }
}

std::string HessianLearner::GetOptimizationHeader() const
{
    return "       KL   graderr     g_min     g_max         +         - lambdamin      rmin";
}

std::vector<double> HessianLearner::GetOptimizationInfo()
{
    const int n = GetNumberOfParameters();
    std::vector<double> result(9, 0.0);
    result[0] = GetKLDistance();
    double ge = 0.0;
    for (int i = 0; i < n; ++i) ge = std::max(ge, std::fabs(rhs[i]));
    result[1] = ge;
    result[2] = *std::min_element(rhs.begin() + n, rhs.end());
    result[3] = *std::max_element(rhs.begin() + n, rhs.end());
    error = std::max(std::max(result[1], std::fabs(result[2])), std::fabs(result[3]));
    if (!degenerate && factored) {
        int pos, neg, zero;
        if (diag_solved) { pos = diag_pos; neg = diag_neg; }
        else solver.Inertia(pos, neg, zero);
        result[4] = pos; result[5] = neg;
    }
    result[6] = lambda_min;
    if (!HasUniquePaths()) result[7] = rmin;   // argmin (result[8]) is a path index of the enumeration: not reproduced
    return result;
}

bool HessianLearner::HaltCondition(double tol)
{
    if (degenerate) throw LearnerError("Unable to continue!");
    return error <= tol;
}

double HessianLearner::ComputeLogDetHessian()           // src/HessianLearner.cpp:219-260
{
    const int n = GetNumberOfParameters();
    ComputeExpX();
    ComputeGrad();
    std::vector<double> Hy;
    ComputeHfDense(Hy, nullptr);
    for (int j = 0; j < n; ++j) Hy[(size_t)j * n + j] -= rhs[j];
    for (int j = 0; j < n; ++j)
        for (int k = 0; k < n; ++k) Hy[(size_t)j * n + k] /= expx[j] * expx[k];
    if (HasUniquePaths()) {                            // diagonal: src/Utils.cpp:300-311
        double result = 0;
        for (int i = 0; i < n; ++i) {
            if (Hy[(size_t)i * n + i] > 0) result += std::log(Hy[(size_t)i * n + i]);
            else return INFINITY;
        }
        return result;
    }
    SymIndefinite s;
    s.Factor(n, Hy);
    double logabs; int sign;
    s.LogDet(logabs, sign);
    return sign > 0 ? logabs : INFINITY;
}

std::vector<double> HessianLearner::GetOptimizationResult(bool)
{
    ComputeModeledProbs();
    ComputeObjective();
    const double logdet = ComputeLogDetHessian();
    return {GetKLDistance(), mxlogx(GetCommonSupport()), LogModelVolume(), LogAuxiliaryVolume(), logdet,
            LogDetAuxiliaryHessian(), (double)(GetNumberOfParameters() - GetNumberOfConstraints()),
            (double)std::max<int>(0, GetNumberOfAuxParameters() - 1)};
}

}  // namespace wfsa
