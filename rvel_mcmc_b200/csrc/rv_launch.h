// rv_launch.h -- host-callable launchers of the sm_100a kernels (internal to librvgpu.so).
#pragma once
#include <cuda_runtime.h>
namespace rv {
struct LoglikArgs;
cudaError_t launch_loglik(const LoglikArgs& a, int P, int D, int mapping, int dense, int num_sms, cudaStream_t stream);
cudaError_t launch_finalize(const double* part_chi2, const int* part_status, long long W, double npoints,
                            double* logp, int* status, unsigned long long* item_counter, cudaStream_t stream);
cudaError_t launch_curve_finalize(unsigned long long* item_counter, cudaStream_t stream);
struct Model;
cudaError_t launch_initial_conditions(const Model* md, const double* theta, long long W, double* out, int* status,
                                      cudaStream_t stream);
cudaError_t launch_fp64_peak(double* d_out, int blocks, int iters, cudaStream_t stream);
constexpr int RV_COST_BINS = 1024;
cudaError_t launch_cost_order(const Model* md, const double* theta, long long W, int* bin, int* hist, int* cursor, int* order,
                              cudaStream_t stream);
// variational path (rv_var_kernels.cu)
struct VarArgs;
int var_threads_needed(int P, int nv);
int var_model_fits(int P, int D, int nv);   // launch_var has a configuration for this model (one launch or chunks of pairs)
size_t var_hist_doubles_needed(int P, int D, int nv, int num_sms);
cudaError_t launch_var(const VarArgs& a, int P, int D, int nv, int num_sms, cudaStream_t stream);
cudaError_t launch_var_finalize(const double* part, const int* pstat, long long W, int nv, double* logp, double* grad,
                                double* hess, int* status, unsigned long long* item_counter, cudaStream_t stream);
// optional WHFast variant (rv_whfast_kernels.cu)
struct WhArgs;
cudaError_t launch_whfast(const WhArgs& a, int P, int D, int num_sms, cudaStream_t stream);
// samplers (rv_samplers.cu)
cudaError_t launch_mh_propose(const double* theta, const double* scales, double step_size, int nvars, long long W,
                              unsigned long long seed, unsigned long long first_id, unsigned step, double* prop,
                              cudaStream_t s);
cudaError_t launch_mh_accept(double* theta, double* logp, const double* prop, const double* prop_logp,
                             const int* prop_status, int nvars, long long W, unsigned long long seed,
                             unsigned long long first_id, unsigned step, unsigned long long* n_accept,
                             unsigned char* accepted, double* chain_row, double* chain_logp_row, long long chain_w,
                             cudaStream_t s);
cudaError_t launch_stretch_propose(const double* S, const double* C, int nvars, long long nS, long long nC, double a,
                                   unsigned long long seed, unsigned long long id0_S, unsigned step, unsigned half,
                                   double* q, double* zz, cudaStream_t s);
cudaError_t launch_stretch_accept(double* S, double* lnp, const double* q, const double* q_lnp, const int* q_status,
                                  const double* zz, int nvars, long long nS, unsigned long long seed,
                                  unsigned long long id0_S, unsigned step, unsigned half, unsigned long long* n_accept,
                                  unsigned char* accepted, cudaStream_t s);
cudaError_t launch_smala_propose(const double* theta, const double* grad, const double* hess, const int* cur_status, int n,
                                 long long W, double eps, double alpha, unsigned long long seed, unsigned long long first_id,
                                 unsigned step, double* prop, double* q_fwd, int* geo_status, double* scratch, cudaStream_t s);
cudaError_t launch_smala_accept(double* theta, double* logp, double* grad, double* hess, const double* prop,
                                const double* p_logp, const double* p_grad, const double* p_hess, const int* p_status,
                                const int* geo_status, const double* q_fwd, int n, long long W, double eps, double alpha,
                                unsigned long long seed, unsigned long long first_id, unsigned step,
                                unsigned long long* n_accept, unsigned char* accepted, int* flag, double* chain_row,
                                double* chain_logp_row, long long chain_w, double* scratch, int mala, cudaStream_t s);
// multi-GPU stretch: the full ensemble copies of every GPU of a group (own + peer-mapped pointers)
constexpr int RV_MAX_GROUP = 16;
struct PeerCopies { double* theta[RV_MAX_GROUP]; double* lnp[RV_MAX_GROUP]; int n; };
cudaError_t launch_stretch_accept_peer(const PeerCopies& pc, int self, long long row0, const double* q, const double* q_lnp,
                                       const int* q_status, const double* zz, int nvars, long long nS, unsigned long long seed,
                                       unsigned long long id0_S, unsigned step, unsigned half, unsigned long long* n_accept,
                                       cudaStream_t s);
cudaError_t launch_mask_logp(double* logp, const int* status, long long W, cudaStream_t s);
// maximum-likelihood fit (rv_map.cu)
cudaError_t launch_map_init(long long W, double mu0, int* code, int* n_iter, double* mu, int* run, int* eval, cudaStream_t s);
cudaError_t launch_map_gather(const int* list, long long m, const double* theta, int n, double* out, cudaStream_t s);
cudaError_t launch_map_scatter(const int* list, long long m, int n, const double* g_logp, const double* g_grad,
                               const double* g_hess, const int* g_status, double* logp, double* grad, double* hess,
                               int* status, int* code, const int* n_iter, cudaStream_t s);
cudaError_t launch_map_step(const int* run, long long m, int n, const double* theta, const double* grad, const double* hess,
                            const double* mu, const int* n_iter, int* code, int max_iter, double tol, int n_trial,
                            double* rows, double* scratch, cudaStream_t s);
cudaError_t launch_map_select(const int* run, long long m, int n, int n_trial, const double* rows, const double* tlogp,
                              const int* tstatus, double* theta, double* mu, int* n_iter, int* code, int* run_next,
                              int* eval, int* counts, cudaStream_t s);
}  // namespace rv
