// rv_map.cuh -- per-walker arithmetic of the batched maximum-likelihood fit (rv_map_fit): one damped saddle-free Newton
// step and the line-search decision.  Host + device (RV_HD), so the test-only host mirror compiles this exact source.
//
//   A = -(H + H^T)/2 = Q diag(lam) Q^T                       (jacobi_eig)
//   lam~_i = max(|lam_i|, 1e-12 lam_max) + mu lam_max         lam_max = max_i |lam_i|, mu = the walker's damping
//   d = Q diag(1/lam~) Q^T g                                  ascent direction
//   delta = g^T d at mu = 0                                   Newton decrement; delta/2 <= tol stops the walker
//   trial rows: theta, theta + 2^-j d (j = 0 .. n_trial-1)    evaluated by the plain likelihood in one launch
#pragma once
#include "rv_smala.cuh"

namespace rv {

// fit codes (include/rvgpu.h RV_FIT_*); MAP_RUNNING marks a walker that is still iterating
enum : int { MAP_RUNNING = -1, MAP_CONVERGED = 0, MAP_MAXITER = 1, MAP_STALLED = 2, MAP_SADDLE = 3, MAP_NOSTART = 4 };
constexpr int MAP_MAX_TRIAL = 16;
constexpr double MAP_EIG_FLOOR = 1e-12;   // |lam| floor, relative to lam_max: a flat direction gets a finite, long step
constexpr double MAP_MU_MIN = 1e-6;       // first damping after a rejected step; an accepted step divides by 10, below -> 0
constexpr double MAP_MU_MAX = 1.0;        // a rejection that takes the damping above this stops the walker (STALLED)

// The Newton step at theta (status OK).  A: 2 n^2 doubles of scratch.  Writes rows[(n_trial + 1) * n] and returns
// MAP_RUNNING, or returns the code the walker stops with (every row is then theta): MAP_CONVERGED / MAP_SADDLE when
// delta/2 <= tol (min lam > 1e-12 lam_max or not; also MAP_SADDLE when the Hessian has no usable eigenvalue), MAP_MAXITER when
// n_iter >= max_iter.  *dec = delta (0 when no decomposition was possible).
RV_HD int map_step_one(int n, const double* __restrict__ th, const double* __restrict__ g, const double* __restrict__ H,
                       double mu, int n_iter, int max_iter, double tol, int n_trial, double* __restrict__ rows,
                       double* dec_out, double* __restrict__ A) {
    double* Q = A + n * n;
    double lam[SMAX], y[SMAX];
    for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) A[i * n + j] = -0.5 * (H[i * n + j] + H[j * n + i]);
    const bool ok = jacobi_eig(n, A, Q, lam);
    double lmax = 0.0, lmin = lam[0];
    for (int i = 0; i < n; i++) { lmax = fmax(lmax, fabs(lam[i])); lmin = fmin(lmin, lam[i]); }
    const double lfloor = MAP_EIG_FLOOR * lmax;
    int code = MAP_RUNNING;
    double dec = 0.0;
    if (!ok || !(lmax > 0.0) || !isfinite(lmax)) {
        code = MAP_SADDLE;
    } else {
        for (int k = 0; k < n; k++) {
            double s = 0.0;
            for (int i = 0; i < n; i++) s += Q[i * n + k] * g[i];
            y[k] = s;
            dec += s * s / fmax(fabs(lam[k]), lfloor);
        }
        // positive definite beyond the floor: an exactly flat direction comes out of an eigensolver as +-1e-17 lam_max
        if (!(0.5 * dec > tol)) code = lmin > lfloor ? MAP_CONVERGED : MAP_SADDLE;
        else if (n_iter >= max_iter) code = MAP_MAXITER;
    }
    if (dec_out) *dec_out = dec;
    for (int i = 0; i < n; i++) rows[i] = th[i];
    if (code != MAP_RUNNING) {
        for (int j = 1; j <= n_trial; j++)
            for (int i = 0; i < n; i++) rows[j * n + i] = th[i];
        return code;
    }
    for (int k = 0; k < n; k++) y[k] /= fmax(fabs(lam[k]), lfloor) + mu * lmax;
    for (int i = 0; i < n; i++) {
        double d = 0.0;
        for (int k = 0; k < n; k++) d += Q[i * n + k] * y[k];
        for (int j = 0; j < n_trial; j++) rows[(j + 1) * n + i] = th[i] + ldexp(d, -j);
    }
    return MAP_RUNNING;
}

// The line-search decision for one walker from the plain logps of its rows (row 0 = theta, same launch).  The best row
// with status OK wins, the lowest j on ties; it is taken when its logp exceeds row 0's.  Returns 1 when theta moved
// (then mu /= 10, 0 below MAP_MU_MIN, and n_iter += 1), else 0 (mu = max(10 mu, MAP_MU_MIN); above MAP_MU_MAX
// *code = MAP_STALLED).
RV_HD int map_select_one(int n, int n_trial, const double* __restrict__ rows, const double* __restrict__ tlogp,
                         const int* __restrict__ tstatus, double* __restrict__ th, double& mu, int& n_iter, int& code) {
    int best = 0;
    for (int j = 1; j <= n_trial; j++)
        if (tstatus[j] == ST_OK && (best == 0 || tlogp[j] > tlogp[best])) best = j;
    if (best > 0 && tlogp[best] > tlogp[0]) {
        for (int i = 0; i < n; i++) th[i] = rows[best * n + i];
        mu = mu / 10.0;
        if (mu < MAP_MU_MIN) mu = 0.0;
        n_iter += 1;
        return 1;
    }
    mu = fmax(10.0 * mu, MAP_MU_MIN);
    if (mu > MAP_MU_MAX) code = MAP_STALLED;
    return 0;
}

}  // namespace rv
