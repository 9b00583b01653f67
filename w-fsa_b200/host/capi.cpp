// w-fsa_b200/host/capi.cpp -- C ABI over the host side (include/wfsa_host.h).
#include "../../include/wfsa_host.h"

#include <cmath>
#include <cstring>
#include <memory>
#include <sstream>

#include "../csrc/philox.hpp"
#include "fsa.hpp"
#include "learner.hpp"

using namespace wfsa;

static thread_local std::string g_err, g_json;

static void jstr(std::ostringstream& o, const std::string& s)
{
    o << '"';
    for (unsigned char c : s) {
        if (c == '"' || c == '\\') o << '\\' << c;
        else if (c < 0x20) { char b[8]; snprintf(b, sizeof(b), "\\u%04x", c); o << b; }
        else o << c;
    }
    o << '"';
}
static void jnum(std::ostringstream& o, double v)
{
    if (std::isnan(v)) o << "\"nan\"";
    else if (std::isinf(v)) o << (v > 0 ? "\"inf\"" : "\"-inf\"");
    else { char b[40]; snprintf(b, sizeof(b), "%.17g", v); o << b; }
}

static void describe_fsa(std::ostringstream& o, const Fsa& fsa, const std::vector<int32_t>* trimmed)
{
    o << "\"states\":" << fsa.GetNumberOfStates() << ",\"transitions\":" << fsa.GetNumberOfTransitions()
      << ",\"emissions\":" << fsa.GetNumberOfEmissions() << ",\"raw_parameters\":" << fsa.GetNumberOfParameters()
      << ",\"raw_constraints\":" << fsa.GetNumberOfConstraints() << ",\"free_parameters\":" << fsa.GetNumberOfFreeParameters()
      << ",\"start\":" << fsa.StartIndex() << ",\"end\":" << fsa.EndIndex() << ",\"state_names\":[";
    for (size_t i = 0; i < fsa.States().size(); ++i) { if (i) o << ','; jstr(o, fsa.States()[i].name); }
    o << "],\"edges\":[";
    bool first = true;
    auto tr = [&](int raw) { return raw < 0 ? -1 : (trimmed ? (*trimmed)[raw] : raw); };
    for (const auto& s : fsa.States()) {
        for (const auto& e : s.emissions) {
            if (!first) o << ',';
            first = false;
            o << "{\"state\":"; jstr(o, s.name); o << ",\"kind\":\"E\",\"label\":"; jstr(o, e.str);
            o << ",\"raw\":" << e.index << ",\"trimmed\":" << tr(e.index) << ",\"file_logprob\":"; jnum(o, e.logprob); o << '}';
        }
        for (const auto& t : s.transitions) {
            if (!first) o << ',';
            first = false;
            o << "{\"state\":"; jstr(o, s.name); o << ",\"kind\":\"T\",\"label\":"; jstr(o, fsa.States()[t.next].name);
            o << ",\"raw\":" << t.index << ",\"trimmed\":" << tr(t.index) << ",\"file_logprob\":"; jnum(o, t.logprob); o << '}';
        }
    }
    o << ']';
}

extern "C" void wfsa_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    wfsa::philox4x32_10(ctr, key, out);
}

extern "C" int wfsa_host_kkt_solve(int32_t n, int32_t k, const double* expx, const double* lambda, const int32_t* ccol, const double* rhs,
                                   double* sol_schur, double* sol_dense, int32_t* inertia4)
{
    const int N = n + k;
    std::vector<double> H((size_t)N * N, 0.0), sol;
    for (int i = 0; i < n; ++i) {                      // HessianLearner::ComputeHg
        H[(size_t)i * N + i] += expx[i] * lambda[ccol[i]];
        H[(size_t)i * N + n + ccol[i]] += expx[i];
        H[(size_t)(n + ccol[i]) * N + i] += expx[i];
    }
    SymIndefinite solver;
    solver.Factor(N, H);
    solver.Solve(rhs, sol_dense);
    int pos = 0, neg = 0, zero = 0;
    solver.Inertia(pos, neg, zero);
    inertia4[2] = pos; inertia4[3] = neg;
    int sp = 0, sn = 0;
    if (!SolveDiagonalKKT(n, k, expx, lambda, ccol, rhs, sol, sp, sn)) { inertia4[0] = inertia4[1] = -1; return 1; }
    std::copy(sol.begin(), sol.end(), sol_schur);
    inertia4[0] = sp; inertia4[1] = sn;
    return 0;
}

extern "C" const char* wfsa_host_last_error(void) { return g_err.c_str(); }

extern "C" int wfsa_host_parse(const char* fsa_text, size_t fsa_len, const char* corpus_text, size_t corpus_len, const char** json_out)
{
    g_err.clear();
    try {
        Fsa fsa; Corpus corpus;
        corpus.ReadText(std::string(corpus_text, corpus_len));
        const double sum = corpus.Sum();
        fsa.ReadText(std::string(fsa_text, fsa_len));
        std::ostringstream o;
        o << "{\"corpus_size\":" << corpus.size() << ",\"corpus_sum\":"; jnum(o, sum); o << ',';
        describe_fsa(o, fsa, nullptr);
        o << ",\"corpus\":[";
        for (size_t i = 0; i < corpus.size(); ++i) {
            if (i) o << ',';
            o << "{\"word\":"; jstr(o, corpus[i].first); o << ",\"weight\":"; jnum(o, corpus[i].second); o << '}';
        }
        o << "]}";
        g_json = o.str();
        if (json_out) *json_out = g_json.c_str();
        return WFSA_OK;
    } catch (const MyError& e) { g_err = e.what(); return WFSA_HOST_ERR_PARSE; }
    catch (const std::exception& e) { g_err = e.what(); return WFSA_ERR_INVALID; }
}

struct wfsa_session {
    Fsa fsa;
    Corpus corpus;
    double corpus_sum = 0;
    std::unique_ptr<Learner> learner;
    bool hessian = false, degenerate = false;
    std::string err, json, dump, degenerate_msg;
};

template <class F> static int guarded(wfsa_session* s, F&& f)
{
    if (!s) return WFSA_ERR_INVALID;
    try { f(); return WFSA_OK; }
    catch (const LearnerError& e) { s->err = e.what(); return WFSA_HOST_ERR_LEARNER; }
    catch (const MyError& e) { s->err = e.what(); return WFSA_HOST_ERR_PARSE; }
    catch (const std::exception& e) { s->err = e.what(); return WFSA_ERR_INVALID; }
}

extern "C" int wfsa_session_create(const char* fsa_text, size_t fsa_len, const char* corpus_text, size_t corpus_len,
                                   const char* optimizer, const wfsa_session_options* opt, wfsa_session** out)
{
    g_err.clear();
    if (!out) return WFSA_ERR_INVALID;
    *out = nullptr;
    std::unique_ptr<wfsa_session> s(new wfsa_session());
    try {
        s->corpus.ReadText(std::string(corpus_text, corpus_len));     // src/main.cpp:141-155
        s->corpus_sum = s->corpus.Sum();
        s->corpus.Renormalize();
        s->fsa.ReadText(std::string(fsa_text, fsa_len));              // src/main.cpp:159-163
        s->hessian = optimizer && std::strcmp(optimizer, "Hessian") == 0;
        if (!s->hessian && optimizer && std::strcmp(optimizer, "QuasiNewton") != 0) { g_err = "optimizer must be Hessian or QuasiNewton"; return WFSA_ERR_INVALID; }
        if (s->hessian) s->learner.reset(new HessianLearner()); else s->learner.reset(new QuasiNewtonLearner());
        BackendOptions bo;
        if (opt) {
            bo.device = opt->device; bo.force_kernel = opt->force_kernel; bo.accum_mode = opt->accum_mode;
            bo.accum_variant = opt->accum_variant; bo.rank = opt->rank; bo.nranks = opt->nranks > 0 ? opt->nranks : 1;
            bo.unique_id = opt->unique_id;
        }
        s->learner->SetBackend(bo);
        s->learner->BuildFrom(s->fsa, s->corpus, true);                // src/main.cpp:206
        if (s->learner->GetNumberOfParameters() == 0) { s->degenerate = true; s->degenerate_msg = "Empty automaton!"; }
        else if (s->learner->GetNumberOfStrings() == 0) { s->degenerate = true; s->degenerate_msg = "Automaton cannot generate any of the strings!"; }
        else s->learner->Finalize();                                   // src/main.cpp:229
    } catch (const LearnerError& e) { g_err = e.what(); return WFSA_HOST_ERR_LEARNER; }
    catch (const MyError& e) { g_err = e.what(); return WFSA_HOST_ERR_PARSE; }
    catch (const std::exception& e) { g_err = e.what(); return WFSA_ERR_INVALID; }
    *out = s.release();
    return WFSA_OK;
}

extern "C" void wfsa_session_destroy(wfsa_session* s) { delete s; }
extern "C" const char* wfsa_session_error(const wfsa_session* s) { return s ? s->err.c_str() : g_err.c_str(); }
extern "C" int wfsa_session_n(const wfsa_session* s) { return s ? s->learner->GetNumberOfParameters() : -1; }
extern "C" int wfsa_session_k(const wfsa_session* s) { return s ? s->learner->GetNumberOfConstraints() : -1; }
extern "C" wfsa_dev* wfsa_session_backend(wfsa_session* s) { return s ? s->learner->Backend() : nullptr; }
extern "C" int wfsa_session_n_recognised_local(const wfsa_session* s)
{
    if (!s) return -1;
    int c = 0;
    for (uint8_t r : s->learner->Recognised()) c += r;
    return c;
}

extern "C" const char* wfsa_session_describe(wfsa_session* s)
{
    if (!s) return "";
    std::ostringstream o;
    const Learner& L = *s->learner;
    o << "{\"corpus_size\":" << s->corpus.size() << ",\"corpus_sum\":"; jnum(o, s->corpus_sum); o << ',';
    describe_fsa(o, s->fsa, &L.TrimmedMap());
    o << ",\"strings\":" << L.GetNumberOfStrings() << ",\"paths\":"; jnum(o, L.GetNumberOfPaths());
    o << ",\"common_support\":"; jnum(o, L.GetCommonSupport());
    o << ",\"unique_paths\":" << (L.HasUniquePaths() ? "true" : "false") << ",\"n\":" << L.GetNumberOfParameters()
      << ",\"k\":" << L.GetNumberOfConstraints() << ",\"degenerate\":" << (s->degenerate ? "true" : "false")
      << ",\"degenerate_message\":"; jstr(o, s->degenerate_msg);
    o << ",\"x\":[";
    for (int i = 0; i < L.GetNumberOfParameters(); ++i) { if (i) o << ','; jnum(o, L.GetWeights()[i]); }
    o << "],\"shard\":[";
    const auto& rec = L.Recognised(); const auto& pc = L.PathCounts();
    for (size_t i = 0; i < rec.size(); ++i) { if (i) o << ','; o << "[" << (int)rec[i] << ","; jnum(o, pc[i]); o << "]"; }
    o << "]";
    wfsa_dev_info info;
    if (L.Backend() && wfsa_dev_get_info(L.Backend(), &info) == WFSA_OK)
        o << ",\"kernel\":" << info.kernel << ",\"accum_mode\":" << info.accum_mode << ",\"n_arcs\":" << info.n_arcs
          << ",\"max_candidates\":" << info.max_candidates << ",\"grid\":" << info.grid << ",\"block\":" << info.block
          << ",\"smem_bytes\":" << info.smem_bytes << ",\"table_bytes\":" << info.table_bytes
          << ",\"n_active_tokens\":" << info.n_active_tokens << ",\"n_tokens\":" << info.n_tokens
          << ",\"fx_log2\":" << info.fixed_point_scale_log2;
    o << "}";
    s->json = o.str();
    return s->json.c_str();
}

static int need_ready(wfsa_session* s)
{
    if (!s) return WFSA_ERR_INVALID;
    if (s->degenerate) { s->err = s->degenerate_msg; return WFSA_HOST_ERR_DEGENERATE; }
    return WFSA_OK;
}

extern "C" int wfsa_session_init(wfsa_session* s, int flags, const double* x)
{
    if (int rc = need_ready(s)) return rc;
    return guarded(s, [&] { s->learner->Init(flags, x); });
}

extern "C" int wfsa_session_eval(wfsa_session* s, const double* x, double* kl, double* loglik, double* grad, double* logq)
{
    if (int rc = need_ready(s)) return rc;
    return guarded(s, [&] {
        Learner& L = *s->learner;
        if (x) L.SetX(x);
        L.ComputeModeledProbs();
        L.ComputeObjective();
        if (kl) *kl = L.GetKLDistance();
        if (loglik) *loglik = L.LogLikelihood();
        if (grad) std::copy(L.Gradient().begin(), L.Gradient().end(), grad);
        if (logq) { const auto& lq = L.LogQ(); std::copy(lq.begin(), lq.end(), logq); }
    });
}

extern "C" int wfsa_session_hessian(wfsa_session* s, const double* x, double* Hf)
{
    if (int rc = need_ready(s)) return rc;
    return guarded(s, [&] {
        Learner& L = *s->learner;
        if (x) L.SetX(x);
        std::vector<double> H;
        L.ComputeHfDense(H, nullptr);
        std::copy(H.begin(), H.end(), Hf);
    });
}

extern "C" int wfsa_session_step(wfsa_session* s, double eta, double* info, int* n_info)
{
    if (int rc = need_ready(s)) return rc;
    return guarded(s, [&] {
        s->learner->OptimizationStep(eta, false);
        const auto v = s->learner->GetOptimizationInfo();
        if (info) std::copy(v.begin(), v.end(), info);
        if (n_info) *n_info = (int)v.size();
    });
}

extern "C" int wfsa_session_halt(wfsa_session* s, double tol, int* halted)
{
    if (int rc = need_ready(s)) return rc;
    return guarded(s, [&] { const bool h = s->learner->HaltCondition(tol); if (halted) *halted = h ? 1 : 0; });
}

extern "C" int wfsa_session_get_x(wfsa_session* s, double* x, int count)
{
    if (!s || !x) return WFSA_ERR_INVALID;
    const int avail = s->learner->GetNumberOfParameters() + (s->hessian && !s->degenerate ? s->learner->GetNumberOfConstraints() : 0);
    if (count > avail) return WFSA_ERR_INVALID;
    std::copy(s->learner->GetWeights(), s->learner->GetWeights() + count, x);
    return WFSA_OK;
}

extern "C" int wfsa_session_renormalize(wfsa_session* s)
{
    if (int rc = need_ready(s)) return rc;
    return guarded(s, [&] { s->learner->Renormalize(); });
}

extern "C" int wfsa_session_result(wfsa_session* s, double* out8)
{
    if (int rc = need_ready(s)) return rc;
    return guarded(s, [&] {
        const auto v = s->learner->GetOptimizationResult(false);
        if (v.size() != 8) throw LearnerError("this optimizer has no evaluation result");
        std::copy(v.begin(), v.end(), out8);
    });
}

extern "C" const char* wfsa_session_dump(wfsa_session* s, int full_precision)
{
    if (!s) return "";
    Fsa tmp = s->fsa;
    s->learner->RewriteWeights(tmp);
    s->dump = tmp.DumpString(full_precision != 0);
    return s->dump.c_str();
}
