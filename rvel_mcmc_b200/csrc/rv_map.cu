// rv_map.cu -- kernels of the batched maximum-likelihood fit (rv_map_fit, rv_abi.cu): gather / scatter around the
// variational evaluation, the Newton step, the line-search selection with compaction of the running walkers.  One thread
// per walker: the per-walker linear algebra (rv_map.cuh) is microseconds against the milliseconds of a variational
// evaluation.  Walkers are addressed through index lists, so a walker's results never depend on its list position.
#include <cuda_runtime.h>
#include "rv_launch.h"
#include "rv_map.cuh"

namespace rv {

__global__ void map_init_kernel(long long W, double mu0, int* __restrict__ code, int* __restrict__ n_iter,
                                double* __restrict__ mu, int* __restrict__ run, int* __restrict__ eval) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    code[w] = MAP_RUNNING; n_iter[w] = 0; mu[w] = mu0;
    run[w] = (int)w; eval[w] = (int)w;
}

__global__ void map_gather_kernel(const int* __restrict__ list, long long m, const double* __restrict__ theta, int n,
                                  double* __restrict__ out) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= m) return;
    const long long w = list[s];
    for (int i = 0; i < n; i++) out[s * n + i] = theta[w * n + i];
}

// A failed evaluation stops the walker: at the start (n_iter = 0) with MAP_NOSTART, after a step with MAP_STALLED.
__global__ void map_scatter_kernel(const int* __restrict__ list, long long m, int n, const double* __restrict__ g_logp,
                                   const double* __restrict__ g_grad, const double* __restrict__ g_hess,
                                   const int* __restrict__ g_status, double* __restrict__ logp, double* __restrict__ grad,
                                   double* __restrict__ hess, int* __restrict__ status, int* __restrict__ code,
                                   const int* __restrict__ n_iter) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= m) return;
    const long long w = list[s];
    const size_t nn = (size_t)n * n;
    logp[w] = g_logp[s];
    status[w] = g_status[s];
    for (int i = 0; i < n; i++) grad[w * n + i] = g_grad[s * n + i];
    for (size_t i = 0; i < nn; i++) hess[w * nn + i] = g_hess[s * nn + i];
    if (g_status[s] != ST_OK) code[w] = n_iter[w] == 0 ? MAP_NOSTART : MAP_STALLED;
}

__global__ void map_step_kernel(const int* __restrict__ run, long long m, int n, const double* __restrict__ theta,
                                const double* __restrict__ grad, const double* __restrict__ hess,
                                const double* __restrict__ mu, const int* __restrict__ n_iter, int* __restrict__ code,
                                int max_iter, double tol, int n_trial, double* __restrict__ rows,
                                double* __restrict__ scratch) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= m) return;
    const long long w = run[s];
    double* r = rows + (size_t)s * (n_trial + 1) * n;
    if (code[w] != MAP_RUNNING) {       // stopped by its evaluation: rows of theta keep the trial launch well defined
        for (int j = 0; j <= n_trial; j++)
            for (int i = 0; i < n; i++) r[j * n + i] = theta[w * n + i];
        return;
    }
    const int c = map_step_one(n, theta + w * n, grad + w * n, hess + (size_t)w * n * n, mu[w], n_iter[w], max_iter, tol,
                               n_trial, r, nullptr, scratch + (size_t)s * 2 * n * n);
    if (c != MAP_RUNNING) code[w] = c;
}

// Selection, then compaction: walkers still running go to run_next, those whose theta moved also to eval (one
// warp-aggregated atomic per list and warp).  counts[0] / counts[1] must be zero on entry.
__global__ void map_select_kernel(const int* __restrict__ run, long long m, int n, int n_trial,
                                  const double* __restrict__ rows, const double* __restrict__ tlogp,
                                  const int* __restrict__ tstatus, double* __restrict__ theta, double* __restrict__ mu,
                                  int* __restrict__ n_iter, int* __restrict__ code, int* __restrict__ run_next,
                                  int* __restrict__ eval, int* __restrict__ counts) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= m) return;
    const int w = run[s];
    bool keep = false, moved = false;
    if (code[w] == MAP_RUNNING) {
        const size_t r0 = (size_t)s * (n_trial + 1);
        double mw = mu[w];
        int it = n_iter[w], c = MAP_RUNNING;
        moved = map_select_one(n, n_trial, rows + r0 * n, tlogp + r0, tstatus + r0, theta + (size_t)w * n, mw, it, c) != 0;
        mu[w] = mw; n_iter[w] = it; code[w] = c;
        keep = c == MAP_RUNNING;
    }
    const unsigned act = __activemask();
    const int lane = threadIdx.x & 31, leader = __ffs(act) - 1;
    const unsigned below = (1u << lane) - 1u;
    const unsigned bk = __ballot_sync(act, keep), bm = __ballot_sync(act, moved);
    int base_k = 0, base_m = 0;
    if (lane == leader) {
        if (bk) base_k = atomicAdd(&counts[0], __popc(bk));
        if (bm) base_m = atomicAdd(&counts[1], __popc(bm));
    }
    base_k = __shfl_sync(act, base_k, leader);
    base_m = __shfl_sync(act, base_m, leader);
    if (keep) run_next[base_k + __popc(bk & below)] = w;
    if (moved) eval[base_m + __popc(bm & below)] = w;
}

static inline unsigned nblk(long long n, int nt) { return (unsigned)((n + nt - 1) / nt > 0 ? (n + nt - 1) / nt : 1); }

cudaError_t launch_map_init(long long W, double mu0, int* code, int* n_iter, double* mu, int* run, int* eval, cudaStream_t s) {
    map_init_kernel<<<nblk(W, 256), 256, 0, s>>>(W, mu0, code, n_iter, mu, run, eval);
    return cudaGetLastError();
}

cudaError_t launch_map_gather(const int* list, long long m, const double* theta, int n, double* out, cudaStream_t s) {
    map_gather_kernel<<<nblk(m, 128), 128, 0, s>>>(list, m, theta, n, out);
    return cudaGetLastError();
}

cudaError_t launch_map_scatter(const int* list, long long m, int n, const double* g_logp, const double* g_grad,
                               const double* g_hess, const int* g_status, double* logp, double* grad, double* hess,
                               int* status, int* code, const int* n_iter, cudaStream_t s) {
    map_scatter_kernel<<<nblk(m, 128), 128, 0, s>>>(list, m, n, g_logp, g_grad, g_hess, g_status, logp, grad, hess, status,
                                                    code, n_iter);
    return cudaGetLastError();
}

cudaError_t launch_map_step(const int* run, long long m, int n, const double* theta, const double* grad, const double* hess,
                            const double* mu, const int* n_iter, int* code, int max_iter, double tol, int n_trial,
                            double* rows, double* scratch, cudaStream_t s) {
    map_step_kernel<<<nblk(m, 64), 64, 0, s>>>(run, m, n, theta, grad, hess, mu, n_iter, code, max_iter, tol, n_trial, rows,
                                               scratch);
    return cudaGetLastError();
}

cudaError_t launch_map_select(const int* run, long long m, int n, int n_trial, const double* rows, const double* tlogp,
                              const int* tstatus, double* theta, double* mu, int* n_iter, int* code, int* run_next,
                              int* eval, int* counts, cudaStream_t s) {
    map_select_kernel<<<nblk(m, 128), 128, 0, s>>>(run, m, n, n_trial, rows, tlogp, tstatus, theta, mu, n_iter, code,
                                                   run_next, eval, counts);
    return cudaGetLastError();
}

}  // namespace rv
