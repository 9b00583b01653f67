// w-fsa_b200/host/learner.hpp -- host-side optimiser loops over the device evaluation backend.
//
// Mirrors the reference's operator interface for this path -- same class and method names,
// argument meaning and error behaviour (/root/reference/inc/Learner.h:24-102,
// inc/QuasiNewtonLearner.h, inc/HessianLearner.h) -- but holds no path matrices P / M:
// every objective / gradient / H_f evaluation goes through the C ABI of include/wfsa_dev.h.
// Everything here is O(n + k) host arithmetic per epoch (plus a dense (n+k)^3 solve for the
// Hessian optimiser, where the reference calls MKL DSS).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/wfsa_dev.h"
#include "fsa.hpp"
#include "ldlt.hpp"
#include "lower.hpp"

namespace wfsa {

struct BackendOptions {
    int device = 0;
    int force_kernel = 0;
    int accum_mode = 0;
    int accum_variant = 0;
    int rank = 0, nranks = 1;
    const void* unique_id = nullptr;     // WFSA_UNIQUE_ID_BYTES, required when nranks > 1
};

bool SolveDiagonalKKT(int n, int k, const double* expx, const double* lambda, const int* Ccol, const double* rhs,
                      std::vector<double>& sol, int& pos, int& neg);
double LogFactorial(size_t d);
double LogSimplexVolume(size_t d);
double mxlogx(double x);

class Learner {
public:
    Learner();
    virtual ~Learner();
    void SetBackend(const BackendOptions& o) { opts = o; }

    // src/Learner.cpp:269-274: constraints, recognition (device structural pass), Trim
    void BuildFrom(const Fsa& fsa, const Corpus& corpus, bool bfs = true);
    void Renormalize();                                    // src/Learner.cpp:23-43
    void RewriteWeights(Fsa& fsa) const;                   // src/Learner.cpp:45-58
    const double* GetWeights() const { return _x.data(); }

    virtual std::vector<double> GetOptimizationInfo() { return {}; }
    virtual std::string GetOptimizationHeader() const { return ""; }
    virtual std::vector<double> GetOptimizationResult(bool = false) { return {}; }
    virtual bool HaltCondition(double) { return false; }

    double GetCommonSupport() const { return common_support; }
    void ComputeModeledProbs();                            // src/Learner.cpp:515-547 -> device
    void ComputeObjective();                               // src/Learner.cpp:549-553

    int GetNumberOfStrings() const { return n_strings; }   // recognised strings (all ranks)
    double GetNumberOfPaths() const { return n_paths; }    // counted by the DP, not enumerated
    int GetNumberOfParameters() const { return (int)Ccol.size(); }
    int GetNumberOfConstraints() const { return Ccol.empty() ? 0 : Ccol.back() + 1; }
    bool HasUniquePaths() const { return unique_paths; }
    double GetKLDistance() const { return kl; }
    double gKLDistance() const { return kl + mxlogx(common_support); }

    virtual void OptimizationStep(double eta = 1.0, bool verbose = false) = 0;
    virtual void Init(int flags, const double* initialx = nullptr);
    double LogModelVolume() const { return model_volume; }
    double LogAuxiliaryVolume() const { return LogSimplexVolume(auxiliary_parameters); }
    double LogDetAuxiliaryHessian() const { return aux_hessian; }
    int GetNumberOfAuxParameters() const { return (int)auxiliary_parameters; }
    void Finalize();                                       // src/Learner.cpp:466-488

    // extras the tests and the CLI use
    const std::vector<int32_t>& TrimmedMap() const { return trimmed_weights; }
    const std::vector<double>& LogQ();                     // log q of this shard's recognised strings
    const std::vector<double>& Gradient() const { return grad_cache; }
    const std::vector<uint8_t>& Recognised() const { return recognised; }
    const std::vector<double>& PathCounts() const { return path_counts; }
    double LogLikelihood() const { return loglik; }
    void SetX(const double* x) { for (int i = 0; i < GetNumberOfParameters(); ++i) _x[i] = x[i]; }
    wfsa_dev* Backend() const { return dev; }
    const LoweredFsa& Lowered() const { return lowered; }
    // dense H_f (n x n, row major) at the current x; builds the path blocks on first use
    void ComputeHfDense(std::vector<double>& Hf, double* rmin = nullptr);
    double ComputeRmin();
    // the k most probable paths of every string of this shard at the current x (k = 1: wfsa_dev_viterbi, else
    // wfsa_dev_nbest; path s * k + r is rank r of string s), with log q_s at the same x; local to the shard (the evaluation
    // inside is collective with several ranks)
    struct Decoding { int k = 1; std::vector<double> logw, logq; std::vector<int64_t> path_off; std::vector<int32_t> trans_edge, emis_edge; };
    void Decode(Decoding& d, int k = 1);
    // n independent draws from the path posterior of every string of this shard at the current x (wfsa_dev_sample; path
    // s * n + r is draw r of string s), with log q_s from the sampler; local to the shard, no evaluation
    void Sample(Decoding& d, int n, uint64_t seed);

protected:
    virtual void FinalizeCallback() {}
    void DecodePaths(Decoding& d, int k, bool sample, uint64_t seed);
    virtual void InitCallback(int) {}
    void LambdaUpdate(double* lstep, double* l, double eta, bool exponential) const;   // src/Learner.cpp:438-462
    void EvalAt(const double* x);            // device evaluation: loglik, grad
    void BuildPathBlocks();                  // host enumeration of ambiguous strings -> device blocks
    void check(int rc, const char* what) const;

    std::vector<double> _x;
    std::vector<double> p;                   // recognised strings of this shard, corpus order
    std::vector<double> grad_cache, logq_cache;
    std::vector<int32_t> Ccol;               // constraint of every trimmed parameter
    double common_support = 0, plogp = 0, kl = 0, aux_hessian = 0, model_volume = 0, loglik = 0;
    size_t auxiliary_parameters = 0;
    double n_paths = 0;
    int n_strings = 0;
    bool unique_paths = true;
    bool have_blocks = false;

private:
    void BuildConstraints(const Fsa& fsa);
    void BuildPaths(const Fsa& fsa, const Corpus& corpus);
    void Trim();
    double GetWeight(int i) const;
    void AllReduceHost(double* v, int n);

    BackendOptions opts;
    wfsa_dev* dev = nullptr;
    LoweredFsa lowered;
    LoweredCorpus shard;
    const Fsa* fsa_ptr = nullptr;
    std::vector<std::string> shard_words;
    std::vector<int32_t> trimmed_weights, Ccol_raw;
    std::vector<uint8_t> recognised;
    std::vector<double> path_counts;
};

// src/QuasiNewtonLearner.cpp
class QuasiNewtonLearner : public Learner {
public:
    void OptimizationStep(double eta = 1.0, bool verbose = false) override;
    std::vector<double> GetOptimizationInfo() override;
    std::string GetOptimizationHeader() const override;
    bool HaltCondition(double tol) override;
protected:
    void FinalizeCallback() override;
    void InitCallback(int flags) override;
    void ComputeExpX();
    void ComputeG();
    void ComputeGrad();
    void ComputeLambdaNext(std::vector<double>& result);
private:
    std::vector<double> grad, expx, lambda, g, rhs, aux;
    double grad_error = 0, lambda_min = 0, g_min = 0, g_max = 0, rmin = 0;
    bool exponential_lambda = false;
};

// src/HessianLearner.cpp
class HessianLearner : public Learner {
public:
    void OptimizationStep(double eta = 1.0, bool verbose = false) override;
    std::vector<double> GetOptimizationInfo() override;
    std::vector<double> GetOptimizationResult(bool verbose = false) override;
    std::string GetOptimizationHeader() const override;
    bool HaltCondition(double tol) override;
    int GetNumberOfAugmentedParameters() const { return GetNumberOfParameters() + GetNumberOfConstraints(); }
    double ComputeLogDetHessian();
    const std::vector<double>& LastH() const { return H; }
protected:
    void FinalizeCallback() override;
    void InitCallback(int flags) override;
private:
    void ComputeExpX();
    void ComputeGrad();     // rhs[:n] <- grad f
    void ComputeG();        // rhs[n:] <- C^T exp(x) - 1
    void ComputeRhs();
    void ComputeHg();
    void InitSlackVariables();
    std::vector<double> rhs, H, expx, Hf, aux;
    SymIndefinite solver;
    double error = 0, lambda_min = 0, rmin = 0;
    bool include_Hf = false, degenerate = false, exponential_lambda = false, factored = false;
    bool diag_solved = false; int diag_pos = 0, diag_neg = 0;     // Newton step taken through the diagonal Schur complement (no H_f)
};

}  // namespace wfsa
