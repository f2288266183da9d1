// rv_smala.cuh -- per-chain SMALA arithmetic (mcmc.py:126-187): SoftAbs metric, proposal, transition density.
//
//   softabs (mcmc.py:135-139)      lam, Q = eig(-H);  lam~ = lam / tanh(alpha lam);  G = Q diag(lam~) Q^T
//   generate_proposal (:144-153)   Ginv = inv(G); L = cholesky(Ginv); mu = theta + eps^2 Ginv g / 2; theta* = mu + eps L z
//   transitionProbability (:158-162)  log N(to; mu(from), eps^2 Ginv(from))
//   step (:167-187)                accept iff exp(logp* - logp + q(theta|theta*) - q(theta*|theta)) > u
// Nvars x Nvars (<= 35) linear algebra, one chain per thread: cyclic Jacobi, explicit G and G^-1, Cholesky.
#pragma once
#include "rv_rng.cuh"

namespace rv {

constexpr int SMAX = MAXP_VAR * NELEM;   // 35: SMALA needs the variational kernels

// Cyclic Jacobi eigen-decomposition of the symmetric n x n matrix A (row-major, destroyed): A -> diag(lam), Q columns.
RV_HD bool jacobi_eig(int n, double* A, double* Q, double* lam) {
    for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) Q[i * n + j] = (i == j) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 60; sweep++) {
        double off = 0.0, diag = 0.0;
        for (int i = 0; i < n; i++) {
            diag += A[i * n + i] * A[i * n + i];
            for (int j = i + 1; j < n; j++) off += A[i * n + j] * A[i * n + j];
        }
        if (!(off > 0.0) || off <= 1e-40 * diag) break;
        for (int p = 0; p < n - 1; p++)
            for (int q = p + 1; q < n; q++) {
                const double apq = A[p * n + q];
                if (apq == 0.0) continue;
                const double app = A[p * n + p], aqq = A[q * n + q];
                if (fabs(apq) < 1e-300) continue;
                const double theta = (aqq - app) / (2.0 * apq);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < n; k++) {
                    const double akp = A[k * n + p], akq = A[k * n + q];
                    A[k * n + p] = c * akp - s * akq;
                    A[k * n + q] = s * akp + c * akq;
                }
                for (int k = 0; k < n; k++) {
                    const double apk = A[p * n + k], aqk = A[q * n + k];
                    A[p * n + k] = c * apk - s * aqk;
                    A[q * n + k] = s * apk + c * aqk;
                }
                for (int k = 0; k < n; k++) {
                    const double qkp = Q[k * n + p], qkq = Q[k * n + q];
                    Q[k * n + p] = c * qkp - s * qkq;
                    Q[k * n + q] = s * qkp + c * qkq;
                }
            }
    }
    bool ok = true;
    for (int i = 0; i < n; i++) { lam[i] = A[i * n + i]; ok = ok && isfinite(lam[i]); }
    return ok;
}

// SoftAbs geometry at one point.  Out: G (metric), Gi (its inverse), logdetG.  Returns false when the metric is
// not finite / not positive definite (numpy would raise LinAlgError, mcmc.py:179-183).
RV_HD bool smala_geometry(int n, const double* __restrict__ H, double alpha, double* G, double* Gi,
                                      double& logdetG, double* A, double* Q) {
    double lam[SMAX];
    for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) A[i * n + j] = -0.5 * (H[i * n + j] + H[j * n + i]);
    if (!jacobi_eig(n, A, Q, lam)) return false;
    logdetG = 0.0;
    for (int i = 0; i < n; i++) {
        lam[i] = lam[i] * 1. / tanh(alpha * lam[i]);
        if (!(lam[i] > 0.0) || !isfinite(lam[i])) return false;
        logdetG += log(lam[i]);
    }
    for (int i = 0; i < n; i++)
        for (int j = 0; j <= i; j++) {
            double g = 0.0, gi = 0.0;
            for (int k = 0; k < n; k++) {
                const double qq = Q[i * n + k] * Q[j * n + k];
                g += qq * lam[k];
                gi += qq / lam[k];
            }
            G[i * n + j] = G[j * n + i] = g;
            Gi[i * n + j] = Gi[j * n + i] = gi;
        }
    return true;
}

// log N(x; mu, eps^2 G^-1) = -1/2 [k ln 2pi + 2k ln eps - ln|G| + (x-mu)^T G (x-mu) / eps^2]
RV_HD double mvn_logpdf(int n, const double* x, const double* mu, const double* G, double logdetG, double eps) {
    double quad = 0.0;
    for (int i = 0; i < n; i++) {
        double r = 0.0;
        for (int j = 0; j < n; j++) r += G[i * n + j] * (x[j] - mu[j]);
        quad += (x[i] - mu[i]) * r;
    }
    return -0.5 * ((double)n * log(2.0 * M_PI) + 2.0 * (double)n * log(eps) - logdetG + quad / (eps * eps));
}

RV_HD void smala_mean(int n, const double* theta, const double* Gi, const double* g, double eps, double* mu) {
    for (int i = 0; i < n; i++) {
        double r = 0.0;
        for (int j = 0; j < n; j++) r += Gi[i * n + j] * g[j];
        mu[i] = theta[i] + eps * eps * r / 2.;
    }
}


// One chain's proposal.  scratch: 5 n^2 doubles.  Returns ST_OK or ST_NOT_SPD (then prop = theta, q_fwd = 0).
RV_HD int smala_propose_one(int n, const double* __restrict__ th, const double* __restrict__ g, const double* __restrict__ H,
                            int cur_status, double eps, double alpha, uint64_t seed, uint64_t id, uint32_t step,
                            double* __restrict__ prop, double& q_fwd, double* __restrict__ A) {
    double *Q = A + n * n, *G = Q + n * n, *Gi = G + n * n, *L = Gi + n * n;
    double logdetG;
    bool ok = cur_status == ST_OK && smala_geometry(n, H, alpha, G, Gi, logdetG, A, Q);
    if (ok) {   // lower Cholesky factor of Ginv
        for (int i = 0; i < n && ok; i++)
            for (int j = 0; j <= i; j++) {
                double s = Gi[i * n + j];
                for (int k = 0; k < j; k++) s -= L[i * n + k] * L[j * n + k];
                if (i == j) {
                    if (!(s > 0.0)) { ok = false; break; }
                    L[i * n + i] = sqrt(s);
                } else {
                    L[i * n + j] = s / L[j * n + j];
                }
            }
    }
    if (!ok) {
        for (int i = 0; i < n; i++) prop[i] = th[i];
        q_fwd = 0.0;
        return ST_NOT_SPD;
    }
    double mu[SMAX], z[SMAX + 1], x[SMAX];
    smala_mean(n, th, Gi, g, eps, mu);
    for (int j = 0; 2 * j < n; j++) normal_pair(seed, id, step, (uint32_t)j, z[2 * j], z[2 * j + 1]);
    for (int i = 0; i < n; i++) {
        double r = 0.0;
        for (int j = 0; j <= i; j++) r += L[i * n + j] * z[j];
        x[i] = mu[i] + eps * r;
        prop[i] = x[i];
    }
    q_fwd = mvn_logpdf(n, x, mu, G, logdetG, eps);
    return ST_OK;
}

// One chain's accept test.  Returns 1 accept, 0 reject; *flag = ST_NOT_SPD when a metric could not be built.
// For an ALSMALA "MALA" step (Alsmala.step_mala, mcmc.py:201-234) pass the CURRENT state's stale gradient and Hessian as
// p_grad / p_hess: the reference copies them onto the proposal (mcmc.py:205-206), so both transition densities use them.
RV_HD int smala_accept_one(int n, const double* __restrict__ th, double logp, const double* __restrict__ prop, double p_logp,
                           const double* __restrict__ p_grad, const double* __restrict__ p_hess, int p_status,
                           int geo_status, double q_fwd, double eps, double alpha, uint64_t seed, uint64_t id,
                           uint32_t step, int* flag, double* __restrict__ A) {
    // a chain whose START state already carries a status (hard prior, Encounter) keeps that status: it can never move
    if (geo_status != ST_OK) { if (flag && *flag == ST_OK) *flag = ST_NOT_SPD; return 0; }
    if (p_status != ST_OK) return 0;
    double *Q = A + n * n, *G = Q + n * n, *Gi = G + n * n;
    double logdetG;
    if (!smala_geometry(n, p_hess, alpha, G, Gi, logdetG, A, Q)) { if (flag) *flag = ST_NOT_SPD; return 0; }
    double mu[SMAX];
    smala_mean(n, prop, Gi, p_grad, eps, mu);
    const double q_back = mvn_logpdf(n, th, mu, G, logdetG, eps);
    const U4 r = philox4x32_10(seed, id, step, RNG_ACCEPT);
    return exp(p_logp - logp + q_back - q_fwd) > u53(r.x, r.y) ? 1 : 0;
}

}  // namespace rv
