/* include/wfsa_host.h -- C ABI over the host side (file formats, model compiler, optimiser
 * loops) so that tests and bench.py can drive the C++ host code through ctypes.  The product
 * for a w-fsa maintainer is include/wfsa_dev.h; this header only exposes what the reference's
 * `wfsa` executable does (/root/reference/src/main.cpp:121-347) one call at a time. */
#ifndef WFSA_HOST_H
#define WFSA_HOST_H
#include <stddef.h>
#include <stdint.h>
#include "wfsa_dev.h"
#ifdef __cplusplus
extern "C" {
#endif

#define WFSA_HOST_ERR_PARSE 100       /* FsaError / CorpusError (message available)            */
#define WFSA_HOST_ERR_LEARNER 101     /* LearnerError                                          */
#define WFSA_HOST_ERR_DEGENERATE 102  /* "Empty automaton!" / no recognised string (main.cpp:217-228) */

/* Parse both files and describe them as JSON (no device needed): counts of src/main.cpp:152-176,
 * every edge with its raw parameter id, the corpus.  *json_out is owned by the library until the
 * next call on this thread. */
int wfsa_host_parse(const char* fsa_text, size_t fsa_len, const char* corpus_text, size_t corpus_len,
                    const char** json_out);
const char* wfsa_host_last_error(void);

/* Host-only (no device): the Newton system of HessianLearner without H_f, [D B; B^T 0] [dx; dl] = rhs with
 * D = diag(expx_i * lambda[ccol_i]) and B[i, ccol_i] = expx_i (src/HessianLearner.cpp:622-639), solved twice -- through its
 * diagonal Schur complement (what the optimiser does, O(n)) and through the dense Bunch-Kaufman factorisation that stands
 * where the reference calls MKL DSS (:100-113).  sol_schur / sol_dense: [n + k]; inertia4 = {+, - of the Schur path, +, - of
 * the dense path}.  Returns 0, or 1 when the Schur path meets a zero pivot (sol_schur untouched). */
int wfsa_host_kkt_solve(int32_t n, int32_t k, const double* expx, const double* lambda, const int32_t* ccol, const double* rhs,
                        double* sol_schur, double* sol_dense, int32_t* inertia4);

/* Host-only: the Philox4x32-10 block function (10 rounds, Random123's constants) that wfsa_dev_sample draws with, from the
 * same source as the kernels: out = philox(ctr, key). */
void wfsa_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

typedef struct wfsa_session wfsa_session;
typedef struct {
    int32_t device, force_kernel, accum_mode, accum_variant;
    int32_t rank, nranks;
    const void* unique_id;            /* WFSA_UNIQUE_ID_BYTES when nranks > 1 */
} wfsa_session_options;

/* optimizer: "QuasiNewton" or "Hessian".  Parses, lowers, runs BuildFrom (device structural
 * pass + Trim) and, unless degenerate, Finalize. */
int wfsa_session_create(const char* fsa_text, size_t fsa_len, const char* corpus_text, size_t corpus_len,
                        const char* optimizer, const wfsa_session_options* opt, wfsa_session** out);
void wfsa_session_destroy(wfsa_session* s);
const char* wfsa_session_error(const wfsa_session* s);
/* JSON: counts, strings/paths/common support, n, k, Ccol, every edge with raw + trimmed index and
 * file log-weight, every corpus string of this shard with recognised flag and path count. */
const char* wfsa_session_describe(wfsa_session* s);
int wfsa_session_n(const wfsa_session* s);
int wfsa_session_k(const wfsa_session* s);
int wfsa_session_n_recognised_local(const wfsa_session* s);
int wfsa_session_init(wfsa_session* s, int flags, const double* x_or_null);
/* objective + gradient at x (n doubles); any output may be NULL; logq: recognised strings of this shard */
int wfsa_session_eval(wfsa_session* s, const double* x, double* kl, double* loglik, double* grad, double* logq);
int wfsa_session_hessian(wfsa_session* s, const double* x, double* Hf /* n*n */);
/* one OptimizationStep + GetOptimizationInfo; info needs room for 9 doubles */
int wfsa_session_step(wfsa_session* s, double eta, double* info, int* n_info);
int wfsa_session_halt(wfsa_session* s, double tol, int* halted);
int wfsa_session_get_x(wfsa_session* s, double* x, int count);
int wfsa_session_renormalize(wfsa_session* s);
int wfsa_session_result(wfsa_session* s, double* out8);          /* -eval line, Hessian only */
const char* wfsa_session_dump(wfsa_session* s, int full_precision);   /* RewriteWeights + Dump */
wfsa_dev* wfsa_session_backend(wfsa_session* s);

#ifdef __cplusplus
}
#endif
#endif
