// rv_var.cuh -- value + gradient + Hessian of the RV log-likelihood (SMALA), one CTA per walker leg.
//
// Replaces, on the GPU, what the reference does per State.get_logp_d_dd (state.py:290-294) through rebound:
//   state.py:229-248  setup_sim_vars   real set + Nvars first-order + Nvars(Nvars+1)/2 second-order variational sets
//   state.py:253-285  get_chi2_d_dd    forward sweep, fresh simulation, monotone backward sweep; chi2, d, dd sums
// Mapping: one thread per (set, planet).  The star of every set is implicit (barycentric frame:
// r* = -sum mu_p r_p and its first/second variations).  All sets share one IAS15 step sequence, as in rebound:
// the predictor-corrector monitor runs over every coordinate, the step-size controller over the real
// particles only (rebound >= Dec 2020; the 2017 all-particle norm changes derivatives by 1e-10 relative).
// The CTA algorithm is written against an executor (each / sync / block max / fetch) so that the same source
// runs as a CUDA block (rv_var_kernels.cu) and, in the CPU test-suite, as a sequential emulation of the block.
#pragma once
#include "rv_core.cuh"
#include "rv_jet.cuh"

namespace rv {

struct VarArgs {
    const Model* model;
    const double* theta;   // [W][nvars]
    long long W;
    const double *ot, *orv, *oerr;   // forward leg [0,nf), backward leg [nf,nf+nb) in obs.tb (ascending) order
    int nf, nb;
    double npoints;        // the `fac` of state.py:258
    int check_prior;       // per call: 1 = test priorHard first (status ST_PRIOR, no integration), 0 = integrate regardless
                           // (State.get_logp_d_dd itself has no prior test, state.py:290-294; the samplers do, mcmc.py:171)
    double* part;          // [2W][nsets]: chi2, d[a], dd[a][b] (a >= b, row-major in a) of one leg
    int* part_status;      // [2W]: item w = backward leg of walker w, item W+w = forward leg
    unsigned long long* item_counter;
    unsigned long long* work_counters;   // [0] force evaluations, [1] step attempts (may be null)
    double* hist;          // warp-group layout (rv_var2.cuh): global scratch for the rejected-step history, per resident group
    size_t hist_doubles;
};

RV_HD int var_nsets(int nv) { return 1 + nv + nv * (nv + 1) / 2; }
RV_HD int round32(int x) { return (x + 31) & ~31; }

// Thread / shared-memory layout of one CTA; identical on host and device.
struct VarLayout {
    int P, D, nv, n2, nsets;       // n2 / nsets: the second-order sets / all sets THIS launch carries (see k2_lo)
    int k2_lo, nsets_total;        // first second-order pair of this launch; sets of the model (the row length of VarArgs::part)
    int base1;     // first thread of the (real + first-order) group; second-order slots start at thread 0
    int need;      // threads that carry a (set, planet)
    int NT;        // threads launched
    int npos;      // doubles per position buffer
    int o_pos, o_vx, o_dm, o_red, o_e, o_hist, total;   // offsets in doubles
};
// A second-order set depends on the real set and on its two first-order parents only, so a model whose sets do not fit one
// CTA is integrated in several launches: each carries the real set, all first-order sets and the second-order pairs
// [k2_lo, k2_lo + k2_n) (k2_n < 0: all of them).  The launches share the step sequence (the step-size controller reads the
// real particles only); their predictor-corrector iteration counts may differ, i.e. the real trajectory agrees to rounding.
RV_HD VarLayout var_layout(int P, int D, int nv, int NT, int k2_lo = 0, int k2_n = -1) {
    VarLayout L;
    const int n2_all = nv * (nv + 1) / 2;
    L.P = P; L.D = D; L.nv = nv; L.n2 = (k2_n < 0) ? n2_all : k2_n; L.nsets = 1 + nv + L.n2;
    L.k2_lo = k2_lo; L.nsets_total = 1 + nv + n2_all;
    L.base1 = round32(L.n2 * P);
    L.need = L.base1 + (nv + 1) * P;
    L.NT = NT;
    L.npos = L.nsets * P * D;
    int o = 0;
    L.o_pos = o; o += 2 * L.npos;
    L.o_vx = o; o += L.nsets * P;
    L.o_dm = o; o += (nv > 0 ? nv : 1) * P;
    L.o_red = o; o += 2 * 2 * 32 + 2;      // ping-pong block-max scratch + the item broadcast slot
    L.o_e = o; o += 7 * D * NT;
    L.o_hist = o; o += 14 * D * NT;
    L.total = o;
    return L;
}

// second-order pairs one launch of NT threads can carry beside the real + first-order group (0: the model does not fit)
RV_HD int var_chunk_pairs(int P, int nv, int NT) {
    int n = (NT - (nv + 1) * P) / P;
    while (n > 0 && round32(n * P) + (nv + 1) * P > NT) n--;
    return n > 0 ? n : 0;
}

template <int P, int D>
struct VarThread {
    int tid, set, planet, order;   // order: 0 real, 1 first, 2 second, -1 idle; set: index among the sets of this launch
    int gset;                      // index among the sets of the model (= set unless the launch carries a chunk of the pairs)
    int sa, sb;                    // parent sets (first-order sets of parameters pa, pb)
    int pa, pb;                    // parameter indices (pa >= pb)
    int ou, oa, ob;                // element offsets of the own / parent sets in a position buffer (set * P * D)
    int ma, mb;                    // offsets of the parents' mass-derivative rows (pa * P, pb * P)
    double x0[D], v0[D], a0[D], ha0[D], csx[D], csv[D], x0c[D];
    double q[7][D];                // b coefficients between step attempts, g coefficients inside the predictor-corrector loop
    double xn[D], at[D], dg6[D];   // last predictor position, last force, last change of g6 (= b6)
    double acc;                    // planet-0 thread of a set: running chi2 / d[a] / dd[a][b]
};

template <int P>
struct VarUniform {
    double mu[P], gm[P], gm0, min2, epsilon;
};

struct VarClock { double t, dt, dt_last_done; };

// 1/r from r^2
RV_HD double rinv1(double r2) {
#if defined(__CUDA_ARCH__)
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(r2));
    const double t = r2 * y;
    const double e = fma(-t, y, 1.0);
    const double p = fma(0.375, e, 0.5) * e;
    return fma(y, p, y);
#else
    return 1.0 / sqrt(r2);
#endif
}

// positions of the P planets of one set from an exchange buffer (16-byte loads when D == 2)
template <int P, int D>
RV_D void load_set(const double* __restrict__ Xs, double (&out)[P][D]) {
#if defined(__CUDA_ARCH__)
    if constexpr (D == 2) {
#pragma unroll
        for (int j = 0; j < P; j++) {
            const double2 v = *reinterpret_cast<const double2*>(Xs + 2 * j);
            out[j][0] = v.x; out[j][1] = v.y;
        }
        return;
    }
#endif
#pragma unroll
    for (int j = 0; j < P; j++)
#pragma unroll
        for (int d = 0; d < D; d++) out[j][d] = Xs[j * D + d];
}

// Acceleration (order 0), first variation (order 1) or second variation (order 2) of the thread's planet,
// from the positions X[(set*P + p)*D + d] of every planet of every set.
//   a_i = -sum_j m_j f(d),  f(d) = d/r^3,  d = r_i - r_j
//   Df[u]    = u/r^3 - 3 d (d.u)/r^5
//   D2f[u,w] = -3 [u (d.w) + w (d.u) + d (u.w)]/r^5 + 15 d (d.u)(d.w)/r^7
//   order 1: -sum_j { m_j Df[U] + dm_j f(d) }
//   order 2: -sum_j { m_j (Df[U] + D2f[A,B]) + dm_j^a Df[B] + dm_j^b Df[A] }     (d2 m = 0)
template <int P, int D>
RV_D void var_force(const VarThread<P, D>& th, const double* __restrict__ X, const double* __restrict__ dm,
                    const VarUniform<P>& u, double (&an)[D]) {
    const int p = th.planet;
    const double* X0 = X;
    if (th.order == 0) {
        double S[D], dp[D];
#pragma unroll
        for (int d = 0; d < D; d++) {
            S[d] = 0.0;
#pragma unroll
            for (int j = 0; j < P; j++) S[d] = fma(u.mu[j], X0[j * D + d], S[d]);
        }
        double r2 = 0.0;
#pragma unroll
        for (int d = 0; d < D; d++) { dp[d] = X0[p * D + d] + S[d]; r2 = fma(dp[d], dp[d], r2); }
        double y = rinv1(r2);
        double k = -u.gm0 * (y * y * y);
#pragma unroll
        for (int d = 0; d < D; d++) an[d] = k * dp[d];
#pragma unroll
        for (int j = 0; j < P; j++) {
            if (j == p) continue;
            r2 = 0.0;
#pragma unroll
            for (int d = 0; d < D; d++) { dp[d] = X0[p * D + d] - X0[j * D + d]; r2 = fma(dp[d], dp[d], r2); }
            y = rinv1(r2);
            k = -u.gm[j] * (y * y * y);
#pragma unroll
            for (int d = 0; d < D; d++) an[d] = fma(k, dp[d], an[d]);
        }
    } else if (th.order == 1) {
        const double* XU = X + th.ou;
        const double* dma = dm + th.ma;
        double S[D], SU[D];
#pragma unroll
        for (int d = 0; d < D; d++) {
            S[d] = 0.0; SU[d] = 0.0;
#pragma unroll
            for (int j = 0; j < P; j++) {
                S[d] = fma(u.mu[j], X0[j * D + d], S[d]);
                SU[d] = fma(u.mu[j], XU[j * D + d], fma(dma[j], X0[j * D + d], SU[d]));
            }
        }
#pragma unroll
        for (int d = 0; d < D; d++) an[d] = 0.0;
#pragma unroll
        for (int j = -1; j < P; j++) {
            if (j == p) continue;
            double dd[D], U[D], r2 = 0.0, du = 0.0;
#pragma unroll
            for (int d = 0; d < D; d++) {
                if (j < 0) { dd[d] = X0[p * D + d] + S[d]; U[d] = XU[p * D + d] + SU[d]; }
                else { dd[d] = X0[p * D + d] - X0[j * D + d]; U[d] = XU[p * D + d] - XU[j * D + d]; }
                r2 = fma(dd[d], dd[d], r2);
                du = fma(dd[d], U[d], du);
            }
            const double mj = (j < 0) ? u.gm0 : u.gm[j];
            const double dmj = (j < 0) ? 0.0 : dma[j];
            const double y = rinv1(r2), y2 = y * y, r3i = y * y2, r5i = r3i * y2;
            const double kU = mj * r3i;
            const double kd = fma(mj * (-3.0 * r5i), du, dmj * r3i);
#pragma unroll
            for (int d = 0; d < D; d++) an[d] -= fma(kU, U[d], kd * dd[d]);
        }
    } else {
        double x0[P][D], xa[P][D], xb[P][D], xu[P][D];
        load_set<P, D>(X, x0);
        load_set<P, D>(X + th.oa, xa);
        load_set<P, D>(X + th.ob, xb);
        load_set<P, D>(X + th.ou, xu);
        const double* dma = dm + th.ma;
        const double* dmb = dm + th.mb;
        double S[D], SA[D], SB[D], SU[D];
#pragma unroll
        for (int d = 0; d < D; d++) {
            S[d] = 0.0; SA[d] = 0.0; SB[d] = 0.0; SU[d] = 0.0;
#pragma unroll
            for (int j = 0; j < P; j++) {
                S[d] = fma(u.mu[j], x0[j][d], S[d]);
                SA[d] = fma(u.mu[j], xa[j][d], fma(dma[j], x0[j][d], SA[d]));
                SB[d] = fma(u.mu[j], xb[j][d], fma(dmb[j], x0[j][d], SB[d]));
                SU[d] = fma(u.mu[j], xu[j][d], fma(dma[j], xb[j][d], fma(dmb[j], xa[j][d], SU[d])));
            }
        }
#pragma unroll
        for (int d = 0; d < D; d++) an[d] = 0.0;
#pragma unroll
        for (int j = -1; j < P; j++) {
            if (j == p) continue;
            double dd[D], A[D], B[D], U[D];
            double r2 = 0.0, da = 0.0, db = 0.0, ab = 0.0, du = 0.0;
#pragma unroll
            for (int d = 0; d < D; d++) {
                // own planet's values: p is a runtime index into register arrays of length P -> select
                double x0p = x0[0][d], xap = xa[0][d], xbp = xb[0][d], xup = xu[0][d];
#pragma unroll
                for (int k = 1; k < P; k++) {
                    x0p = (p == k) ? x0[k][d] : x0p; xap = (p == k) ? xa[k][d] : xap;
                    xbp = (p == k) ? xb[k][d] : xbp; xup = (p == k) ? xu[k][d] : xup;
                }
                if (j < 0) {
                    dd[d] = x0p + S[d]; A[d] = xap + SA[d]; B[d] = xbp + SB[d]; U[d] = xup + SU[d];
                } else {
                    dd[d] = x0p - x0[j][d]; A[d] = xap - xa[j][d]; B[d] = xbp - xb[j][d]; U[d] = xup - xu[j][d];
                }
                r2 = fma(dd[d], dd[d], r2);
                da = fma(dd[d], A[d], da);
                db = fma(dd[d], B[d], db);
                ab = fma(A[d], B[d], ab);
                du = fma(dd[d], U[d], du);
            }
            const double mj = (j < 0) ? u.gm0 : u.gm[j];
            const double dmaj = (j < 0) ? 0.0 : dma[j];
            const double dmbj = (j < 0) ? 0.0 : dmb[j];
            const double y = rinv1(r2), y2 = y * y, r3i = y * y2, r5i = r3i * y2, r7i = r5i * y2;
            const double c5 = -3.0 * r5i;
            // coefficients of U, A, B, d
            const double kU = mj * r3i;
            const double kA = fma(mj * c5, db, dmbj * r3i);
            const double kB = fma(mj * c5, da, dmaj * r3i);
            double kd = mj * fma(c5, du + ab, 15.0 * r7i * (da * db));
            kd = fma(c5, fma(dmaj, db, dmbj * da), kd);
#pragma unroll
            for (int d = 0; d < D; d++) an[d] -= fma(kU, U[d], fma(kA, A[d], fma(kB, B[d], kd * dd[d])));
        }
    }
}

// predict_next_step (rebound) for one coordinate: new e,b from the stored (_e,_b) scaled by q = dt_new/dt_old.
template <int D>
RV_D void var_predict(double q, const double (&_e)[7], const double (&_b)[7], double (&e)[7], double (&b)[7][D], int c) {
    if (q > 20.0) {
#pragma unroll
        for (int k = 0; k < 7; k++) { e[k] = 0.0; b[k][c] = 0.0; }
        return;
    }
    const double q1 = q, q2 = q1 * q1, q3 = q1 * q2, q4 = q2 * q2, q5 = q2 * q3, q6 = q3 * q3, q7 = q3 * q4;
    double be[7];
#pragma unroll
    for (int k = 0; k < 7; k++) be[k] = _b[k] - _e[k];
    e[0] = q1 * (_b[6] * 7.0 + _b[5] * 6.0 + _b[4] * 5.0 + _b[3] * 4.0 + _b[2] * 3.0 + _b[1] * 2.0 + _b[0]);
    e[1] = q2 * (_b[6] * 21.0 + _b[5] * 15.0 + _b[4] * 10.0 + _b[3] * 6.0 + _b[2] * 3.0 + _b[1]);
    e[2] = q3 * (_b[6] * 35.0 + _b[5] * 20.0 + _b[4] * 10.0 + _b[3] * 4.0 + _b[2]);
    e[3] = q4 * (_b[6] * 35.0 + _b[5] * 15.0 + _b[4] * 5.0 + _b[3]);
    e[4] = q5 * (_b[6] * 21.0 + _b[5] * 6.0 + _b[4]);
    e[5] = q6 * (_b[6] * 7.0 + _b[5]);
    e[6] = q7 * _b[6];
#pragma unroll
    for (int k = 0; k < 7; k++) b[k][c] = e[k] + be[k];
}

// One Gauss-Radau substep, first half: predicted position at h_n from the g coefficients (PG = PRED * C^T),
// published to the exchange buffer.  n is a RUNTIME index: the substep loop is not unrolled, so the force code
// exists once in the instruction stream (the unrolled form thrashed the instruction cache: 2.6 stall cycles per
// issued instruction on no_instruction, profiles/r01g_ncu_var_kernel.txt).
template <int P, int D>
RV_D void var_substep_predict(VarThread<P, D>& th, int n, double dt, double* __restrict__ Xw) {
    const double dth = dt * rvtabm::H[n];
    const double c0 = rvtabm::PG[n][0], c1 = rvtabm::PG[n][1], c2 = rvtabm::PG[n][2], c3 = rvtabm::PG[n][3],
                 c4 = rvtabm::PG[n][4], c5 = rvtabm::PG[n][5], c6 = rvtabm::PG[n][6];
#pragma unroll
    for (int c = 0; c < D; c++) {
        double p0 = fma(c0, th.q[0][c], th.ha0[c]);
        p0 = fma(c1, th.q[1][c], p0);
        p0 = fma(c2, th.q[2][c], p0);
        double p1 = c3 * th.q[3][c];
        p1 = fma(c4, th.q[4][c], p1);
        p1 = fma(c5, th.q[5][c], p1);
        p1 = fma(c6, th.q[6][c], p1);
        const double inner = fma(dth, p0 + p1, th.v0[c]);
        th.xn[c] = fma(dth, inner, th.x0c[c]);
        Xw[th.ou + th.planet * D + c] = th.xn[c];
    }
}

// Second half: g_{n-1} from the force at the predicted positions (static n: the g chain indexes registers).
template <int n, int P, int D>
RV_D void var_substep_corrector(VarThread<P, D>& th, const double (&an)[D]) {
#pragma unroll
    for (int c = 0; c < D; c++) {
        const double gk = an[c] - th.a0[c];
        double s0 = gk * rvtab::GA[n], s1 = 0.0;
#pragma unroll
        for (int i = 0; i < n - 1; i++) {
            if (i & 1) s1 = fma(-th.q[i][c], rvtab::GB[n][i], s1);
            else s0 = fma(-th.q[i][c], rvtab::GB[n][i], s0);
        }
        const double gn = s0 + s1;
        if (n == 7) { th.dg6[c] = gn - th.q[6][c]; th.at[c] = an[c]; }
        th.q[n - 1][c] = gn;
    }
}

template <int P, int D>
RV_D void var_substep_update(VarThread<P, D>& th, int n, const double* __restrict__ Xr, const double* __restrict__ dm,
                             const VarUniform<P>& u) {
    double an[D];
    var_force(th, Xr, dm, u, an);
    switch (n) {
        case 1: var_substep_corrector<1>(th, an); break;
        case 2: var_substep_corrector<2>(th, an); break;
        case 3: var_substep_corrector<3>(th, an); break;
        case 4: var_substep_corrector<4>(th, an); break;
        case 5: var_substep_corrector<5>(th, an); break;
        case 6: var_substep_corrector<6>(th, an); break;
        default: var_substep_corrector<7>(th, an); break;
    }
}

// reb_run_heartbeat on the real set held in an exchange buffer
template <int P, int D>
RV_D bool var_encounter(const double* __restrict__ X0, const VarUniform<P>& u) {
    if (u.min2 == 0.0) return false;
    bool hit = false;
    double S[D];
#pragma unroll
    for (int d = 0; d < D; d++) {
        S[d] = 0.0;
#pragma unroll
        for (int j = 0; j < P; j++) S[d] = fma(u.mu[j], X0[j * D + d], S[d]);
    }
#pragma unroll
    for (int i = 0; i < P; i++) {
        double r2 = 0.0;
#pragma unroll
        for (int d = 0; d < D; d++) { const double ds = X0[i * D + d] + S[d]; r2 = fma(ds, ds, r2); }
        hit = hit || (r2 < u.min2);
#pragma unroll
        for (int j = i + 1; j < P; j++) {
            double q2 = 0.0;
#pragma unroll
            for (int d = 0; d < D; d++) { const double dp = X0[i * D + d] - X0[j * D + d]; q2 = fma(dp, dp, q2); }
            hit = hit || (q2 < u.min2);
        }
    }
    return hit;
}

// (set, planet) of a thread
template <int P, int D>
RV_D void var_assign(VarThread<P, D>& th, int tid, const VarLayout& L) {
    th.tid = tid;
    th.order = -1; th.set = 0; th.gset = 0; th.planet = 0; th.sa = th.sb = 0; th.pa = th.pb = 0;
    if (tid < L.n2 * P) {
        const int kl = tid / P;
        const int k = L.k2_lo + kl;
        th.planet = tid - kl * P;
        th.set = 1 + L.nv + kl;
        th.gset = 1 + L.nv + k;
        th.order = 2;
        int a = 0;
        while ((a + 1) * (a + 2) / 2 <= k) a++;
        th.pa = a; th.pb = k - a * (a + 1) / 2;
        th.sa = 1 + th.pa; th.sb = 1 + th.pb;
    } else if (tid >= L.base1 && tid < L.need) {
        const int q = tid - L.base1;
        th.set = q / P;
        th.gset = th.set;
        th.planet = q - th.set * P;
        th.order = th.set == 0 ? 0 : 1;
        th.pa = th.pb = th.set == 0 ? 0 : th.set - 1;
        th.sa = th.sb = th.set;
    }
    th.ou = th.set * P * D; th.oa = th.sa * P * D; th.ob = th.sb * P * D;
    th.ma = th.pa * P; th.mb = th.pb * P;
}

// Initial conditions of the thread's (set, planet): the jet of the barycentric state with respect to the
// set's parameters (state.py:229-248: add_variation + vary + move_to_com).
template <int P, int D>
RV_D void var_initial(VarThread<P, D>& th, const Model* __restrict__ md, const double (&el)[P][NELEM]) {
    const double m0 = md->m_star;
    Jet mt = J(m0), cx[3], cv[3];
#pragma unroll
    for (int d = 0; d < 3; d++) { cx[d] = J(0.0); cv[d] = J(0.0); }
    JState own;
    own.m = J(0.0);
    for (int d = 0; d < 3; d++) { own.x[d] = J(0.0); own.v[d] = J(0.0); }
    for (int i = 0; i < P; i++) {
        Jet ej[NELEM];
#pragma unroll
        for (int k = 0; k < NELEM; k++) ej[k] = J(el[i][k]);
        if (th.order >= 1 && md->free_planet[th.pa] == i) ej[md->free_elem[th.pa]].d1 = 1.0;
        if (th.order == 2 && md->free_planet[th.pb] == i) ej[md->free_elem[th.pb]].d2 = 1.0;
        const JState s = pal_to_cart_jet(ej, m0);
        mt = mt + s.m;
#pragma unroll
        for (int d = 0; d < 3; d++) { cx[d] = cx[d] + s.m * s.x[d]; cv[d] = cv[d] + s.m * s.v[d]; }
        if (i == th.planet) own = s;
    }
    const Jet im = jinv(mt);
#pragma unroll
    for (int d = 0; d < D; d++) {
        const Jet x = own.x[d] - cx[d] * im, v = own.v[d] - cv[d] * im;
        th.x0[d] = th.order == 0 ? x.v : (th.order == 1 ? x.d1 : x.d12);
        th.v0[d] = th.order == 0 ? v.v : (th.order == 1 ? v.d1 : v.d12);
    }
}

// Star x-velocity of a set (value, first or second variation) from the planets' x-velocities vx[set*P + p]
template <int P>
RV_D double var_star_vx(const double* __restrict__ vx, const double* __restrict__ dm, const VarUniform<P>& u,
                        int order, int set, int sa, int sb, int pa, int pb) {
    double s = 0.0;
    if (order == 0) {
#pragma unroll
        for (int j = 0; j < P; j++) s = fma(u.mu[j], vx[j], s);
    } else if (order == 1) {
#pragma unroll
        for (int j = 0; j < P; j++) s = fma(u.mu[j], vx[set * P + j], fma(dm[pa * P + j], vx[j], s));
    } else {
#pragma unroll
        for (int j = 0; j < P; j++)
            s = fma(u.mu[j], vx[set * P + j], fma(dm[pa * P + j], vx[sb * P + j], fma(dm[pb * P + j], vx[sa * P + j], s)));
    }
    return -s;
}

// ---------------------------------------------------------------------------------------------
// Step logic that does not depend on the thread layout: var_run_items below and var2_run_items (rv_var2.cuh) share it.

// setup_sim, uniform part: the walker's elements; true when they violate the hard prior
template <int P>
RV_D bool var_item_setup(const Model* __restrict__ md, const double* __restrict__ theta, long long wi, int nv, double (&el)[P][NELEM]) {
    bool bad = false;
#pragma unroll
    for (int i = 0; i < P; i++) {
#pragma unroll
        for (int k = 0; k < NELEM; k++) {
            const int s = md->src[i * NELEM + k];
            el[i][k] = (s >= 0) ? theta[wi * nv + s] : md->fixed[i * NELEM + k];
        }
        bad = bad || prior_hard(el[i]);
    }
    return bad;
}

// squared exit distance of the encounter test: (hill_factor x the largest Hill radius)^2
template <int P>
RV_D double var_exit_min2(const double (&el)[P][NELEM], double m0, double hill_factor) {
    double hill = 0.0;
#pragma unroll
    for (int i = 0; i < P; i++) {
        const double rh = el[i][EL_A] * pow(el[i][EL_M] / (3.0 * m0), 1.0 / 3.0);
        if (rh > hill) hill = rh;
    }
    const double emd = hill_factor * hill;
    return emd * emd;
}

// g from b, in place (g_j needs b_k for k > j only), coordinate c
template <int N>
RV_D void var_g_from_b(double (&q)[7][N], int c) {
#pragma unroll
    for (int j = 0; j < 7; j++) {
        double s = q[j][c];
#pragma unroll
        for (int k = 6; k > j; k--) s = fma(q[k][c], rvtab::DD[k][j], s);
        q[j][c] = s;
    }
}

// b from g, in place (b_k needs g_j for j > k only), coordinate c
template <int N>
RV_D void var_b_from_g(double (&q)[7][N], int c) {
#pragma unroll
    for (int k = 0; k < 7; k++) {
        double s = q[k][c];
#pragma unroll
        for (int j = 6; j > k; j--) s = fma(q[j][c], rvtab::CC[j][k], s);
        q[k][c] = s;
    }
}

// rebound's step-size controller after an attempt of length dt, from the real particles' maxima of |b6| and |a|.  Sets the
// next step in w.dt and returns true when the step is accepted; the caller then advances w.t and w.dt_last_done by dt after
// committing the coordinates (updating the clock here, before the commit, costs var2_kernel spill stores).
RV_HD bool var_step_control(double maxb6, double maxak, double epsilon, VarClock& w, double dt) {
    const double err = maxb6 / maxak;
    double dt_new;
    if (is_normal(err)) dt_new = inv_root7(err / epsilon) * dt;
    else dt_new = dt * 4.0;
    if (fabs(dt_new) < 0.25 * fabs(dt)) {
        w.dt = dt_new;
        return false;
    }
    if (fabs(dt_new) > 4.0 * fabs(dt)) dt_new = dt * 4.0;
    w.dt = dt_new;
    return true;
}

// The per-coordinate step commit.  e(k, c): the coordinate's predicted e[k]; hist(k, c): the history of the last accepted
// step, its e[k] at k < 7 and its b[k - 7] at k >= 7.  Rejected step: e and b re-predicted from the history, with
// qr = new dt / that step's dt.
template <int N, class E, class H>
RV_D void var_reject_coord(double (&q)[7][N], int c, double qr, E&& e, H&& hist) {
    double _e[7], _b[7], en[7];
#pragma unroll
    for (int k = 0; k < 7; k++) { _e[k] = hist(k, c); _b[k] = hist(7 + k, c); }
    var_predict<N>(qr, _e, _b, en, q, c);
#pragma unroll
    for (int k = 0; k < 7; k++) e(k, c) = en[k];
}

// Accepted step of length dt (dt2 = dt^2): x0 and v0 advance with compensated summation (carries csx, csv), e and b become
// the history, and the next step's e and b are predicted with qr = new dt / dt.
template <int N, class E, class H>
RV_D void var_accept_coord(double (&q)[7][N], int c, double& x0, double& csx, double& v0, double& csv, const double& a0,
                           double dt, double dt2, double qr, E&& e, H&& hist) {
    {
        const double x = x0;
        double cs = csx;
        double s = q[6][c] * (1. / 72.);
        s = fma(q[5][c], 1. / 56., s); s = fma(q[4][c], 1. / 42., s); s = fma(q[3][c], 1. / 30., s);
        s = fma(q[2][c], 1. / 20., s); s = fma(q[1][c], 1. / 12., s); s = fma(q[0][c], 1. / 6., s);
        s = fma(a0, 0.5, s);
        cs += fma(s, dt2, v0 * dt);
        const double xnew = x + cs;
        cs += x - xnew;
        x0 = xnew; csx = cs;
    }
    {
        const double v = v0;
        double cs = csv;
        double s = q[6][c] * (1. / 8.);
        s = fma(q[5][c], 1. / 7., s); s = fma(q[4][c], 1. / 6., s); s = fma(q[3][c], 1. / 5., s);
        s = fma(q[2][c], 1. / 4., s); s = fma(q[1][c], 1. / 3., s); s = fma(q[0][c], 1. / 2., s);
        s += a0;
        cs = fma(s, dt, cs);
        const double vnew = v + cs;
        cs += v - vnew;
        v0 = vnew; csv = cs;
    }
    double _e[7], _b[7], en[7];
#pragma unroll
    for (int k = 0; k < 7; k++) {
        _e[k] = e(k, c);
        _b[k] = q[k][c];
        hist(k, c) = _e[k];
        hist(7 + k, c) = _b[k];
    }
    var_predict<N>(qr, _e, _b, en, q, c);
#pragma unroll
    for (int k = 0; k < 7; k++) e(k, c) = en[k];
}

// chi2 / d[a] / dd[a][b] term of one set at an epoch (state.py:264-271): res = star vx - observed RV, den = err^2 npoints.
// order 0 real, 1 first-order set `set` of parameter pa, 2 second-order set `set` with first-order parents sa / sb (pa, pb).
template <int P>
RV_D double var_epoch_term(const double* __restrict__ vxs, const double* __restrict__ dm, const VarUniform<P>& u, int order,
                           int set, int sa, int sb, int pa, int pb, double res, double den) {
    if (order == 0) return res * res / den;
    if (order == 1) {
        const double da = var_star_vx<P>(vxs, dm, u, 1, set, 0, 0, pa, 0);
        return 2. * da * res / den;
    }
    const double da = var_star_vx<P>(vxs, dm, u, 1, sa, 0, 0, pa, 0);
    const double db = var_star_vx<P>(vxs, dm, u, 1, sb, 0, 0, pb, 0);
    const double dab = var_star_vx<P>(vxs, dm, u, 2, set, sa, sb, pa, pb);
    return 2. * dab * res / den + 2. * da * db / den;
}

// The reference's epoch loop (state.py:262-284) over the leg of `item`: forward in order, backward reversed.
//   attempt()      one IAS15 step attempt of the whole CTA / group: bit 0 accepted, bit 1 encounter after the step
//   encounter()    the encounter test on the current positions
//   on_epoch(ie)   epoch ie reached: accumulate chi2 / d / dd; false when the star velocity is not finite
// Returns the leg's status.
template <class Exec, class Attempt, class Encounter, class OnEpoch>
RV_D int var_leg_epochs(Exec& ex, const VarArgs& a, const Model* __restrict__ md, long long item, VarClock& w,
                        Attempt&& attempt, Encounter&& encounter, OnEpoch&& on_epoch) {
    const bool backward = item < a.W;
    const int n = backward ? a.nb : a.nf;
    const int base = backward ? a.nf : 0;
    LegCursor c;
    c.status = RUN; c.ie = 0; c.n = n; c.attempts = 0; c.tmax = 0.0; c.last_full_dt = 0.0; c.chi2 = 0.0;
    int final_status = -1;
    for (int ii = 0; ii < n && final_status < 0; ii++) {
        const int ie = backward ? (base + n - 1 - ii) : (base + ii);
        c.tmax = a.ot[ie];
        c.last_full_dt = w.dt;
        w.dt_last_done = 0.0;
        c.status = RUN;
        if (encounter()) c.status = ST_ENCOUNTER;
        while (check_exit(w, c) < 0) {
            int r;
            bool dead = false;
            for (;;) {
                r = attempt();
                c.attempts++;
                if (c.attempts > md->max_attempts || !isfinite(w.dt) || w.dt == 0.0) { dead = true; break; }
                if (r & 1) break;
            }
            if (dead) { c.status = ST_NONFINITE; break; }
            if (r & 2) c.status = ST_ENCOUNTER;
        }
        w.dt = c.last_full_dt;
        if (c.status != ST_OK) { final_status = c.status; break; }
        if (!on_epoch(ie)) final_status = ST_NONFINITE;
        ex.sync();
    }
    return final_status < 0 ? ST_OK : final_status;
}

// ---------------------------------------------------------------------------------------------
// The CTA algorithm.  Exec provides:
//   each(f)                  run f(VarThread&) for every thread of the CTA
//   sync()                   CTA barrier
//   stage_max(th, a, b)      contribute to a two-value block maximum (inside each)
//   read_max(a, b)           the block maxima (after sync); resets the staging area
//   fetch(ctr)               next work item, uniform over the CTA
//   add_work(ptr, nf, na)    accumulate the work counters (once per CTA)
template <int P, int D, class Exec>
RV_D void var_run_items(Exec& ex, const VarArgs& a, const VarLayout& L, double* __restrict__ sm) {
    const Model* __restrict__ md = a.model;
    const int nv = md->nvars;
    const int NT = L.NT;
    double* const pos = sm + L.o_pos;
    double* const vxs = sm + L.o_vx;
    double* const dm = sm + L.o_dm;
    double* const esm = sm + L.o_e;
    double* const hist = sm + L.o_hist;
    const double m0 = md->m_star;
    const long long n_items = 2 * a.W;
    VarUniform<P> u;
    u.gm0 = m0;
    u.epsilon = md->epsilon;

    ex.each([&](VarThread<P, D>& th) {
        if (th.tid < nv * P) {
            const int q = th.tid / P, j = th.tid - q * P;
            dm[th.tid] = (md->free_planet[q] == j && md->free_elem[q] == EL_M) ? 1.0 / m0 : 0.0;
        }
    });

    for (;;) {
        const long long item = ex.fetch(a.item_counter);
        if (item >= n_items) break;
        const long long wi = item < a.W ? item : item - a.W;
        double el[P][NELEM];
        const bool bad = var_item_setup<P>(md, a.theta, wi, nv, el);
        int final_status = ST_PRIOR;
        unsigned long long n_force = 0, n_attempt = 0;
        if (!(bad && a.check_prior)) {
#pragma unroll
            for (int i = 0; i < P; i++) { u.gm[i] = el[i][EL_M]; u.mu[i] = el[i][EL_M] / m0; }
            u.min2 = var_exit_min2<P>(el, m0, md->hill_factor);
            int cur = 0;
            ex.each([&](VarThread<P, D>& th) {
                if (th.order < 0) return;
                var_initial(th, md, el);
                th.acc = 0.0;
#pragma unroll
                for (int c = 0; c < D; c++) {
                    th.csx[c] = 0.0; th.csv[c] = 0.0; th.a0[c] = 0.0; th.ha0[c] = 0.0;
                    th.xn[c] = th.x0[c]; th.at[c] = 0.0; th.dg6[c] = 0.0; th.x0c[c] = th.x0[c];
#pragma unroll
                    for (int k = 0; k < 7; k++) {
                        th.q[k][c] = 0.0;
                        esm[(k * D + c) * NT + th.tid] = 0.0;
                        hist[(k * D + c) * NT + th.tid] = 0.0;
                        hist[((7 + k) * D + c) * NT + th.tid] = 0.0;
                    }
                    pos[cur * L.npos + (th.set * P + th.planet) * D + c] = th.x0[c];
                }
            });
            ex.sync();

            VarClock w;
            w.t = 0.0; w.dt = md->dt0; w.dt_last_done = 0.0;

            // ---- one IAS15 step attempt of the whole CTA; bit0 accepted, bit1 encounter after the step ----
            auto attempt = [&]() -> int {
                n_attempt++;
                const double* X0 = pos + cur * L.npos;
                ex.each([&](VarThread<P, D>& th) {
                    if (th.order < 0) return;
                    var_force(th, X0, dm, u, th.a0);
#pragma unroll
                    for (int cc = 0; cc < D; cc++) {
                        th.ha0[cc] = 0.5 * th.a0[cc];
                        th.x0c[cc] = th.x0[cc] - th.csx[cc];
                        var_g_from_b<D>(th.q, cc);
                    }
                });
                int buf = cur ^ 1;
                Ratio pc_err{1e300, 1.0}, pc_last{2.0, 1.0};
                int it = 0;
                const double dt = w.dt;
                while (true) {
                    if (ratio_lt(pc_err, 1e-16) || (it > 2 && ratio_le(pc_last, pc_err)) || it >= 12) break;
                    pc_last = pc_err;
                    it++;
#pragma unroll 1
                    for (int n = 1; n <= 7; n++) {
                        double* Xw = pos + buf * L.npos;
                        ex.each([&](VarThread<P, D>& th) { if (th.order >= 0) var_substep_predict(th, n, dt, Xw); });
                        ex.sync();
                        ex.each([&](VarThread<P, D>& th) { if (th.order >= 0) var_substep_update(th, n, Xw, dm, u); });
                        buf ^= 1;
                    }
                    // convergence monitor over every coordinate: max |change of b6| / max |a|
                    ex.each([&](VarThread<P, D>& th) {
                        double mg = 0.0, ma = 0.0;
                        if (th.order >= 0) {
#pragma unroll
                            for (int cc = 0; cc < D; cc++) {
                                const double ak = fabs(th.at[cc]), dg = fabs(th.dg6[cc]);
                                norm_max(ak, ma);
                                norm_max(dg, mg);
                            }
                        }
                        ex.stage_max(th, mg, ma);
                    });
                    ex.sync();
                    double maxdg, maxat;
                    ex.read_max(maxdg, maxat);
                    pc_err.num = maxdg; pc_err.den = maxat;
                    n_force += 7;
                }
                n_force += 1;
                // b from g; then step-size control over the real particles
                ex.each([&](VarThread<P, D>& th) {
                    double mb = 0.0, ma = 0.0;
                    if (th.order >= 0) {
#pragma unroll
                        for (int cc = 0; cc < D; cc++) var_b_from_g<D>(th.q, cc);
                    }
                    if (th.order == 0) {
                        double v2 = 0.0, x2 = 0.0;
#pragma unroll
                        for (int cc = 0; cc < D; cc++) { v2 = fma(th.v0[cc], th.v0[cc], v2); x2 = fma(th.xn[cc], th.xn[cc], x2); }
                        const bool keep = !(fabs(v2 * dt * dt) < 1e-16 * x2);
#pragma unroll
                        for (int cc = 0; cc < D; cc++) {
                            const double ak = fabs(th.at[cc]), b6 = fabs(th.q[6][cc]);
                            if (keep) norm_max(ak, ma);
                            if (keep) norm_max(b6, mb);
                        }
                    }
                    ex.stage_max(th, mb, ma);
                });
                ex.sync();
                double maxb6, maxak;
                ex.read_max(maxb6, maxak);
                const bool accepted = var_step_control(maxb6, maxak, u.epsilon, w, dt);
                if (!accepted) {
                    if (w.dt_last_done != 0.0) {
                        const double q = w.dt / w.dt_last_done;
                        ex.each([&](VarThread<P, D>& th) {
                            if (th.order < 0) return;
                            auto e = [&](int k, int c) -> double& { return esm[(k * D + c) * NT + th.tid]; };
                            auto h = [&](int k, int c) -> double& { return hist[(k * D + c) * NT + th.tid]; };
#pragma unroll
                            for (int cc = 0; cc < D; cc++) var_reject_coord<D>(th.q, cc, q, e, h);
                        });
                    }
                } else {
                    const double dt2 = dt * dt, q = w.dt / dt;
                    ex.each([&](VarThread<P, D>& th) {
                        if (th.order < 0) return;
                        auto e = [&](int k, int c) -> double& { return esm[(k * D + c) * NT + th.tid]; };
                        auto h = [&](int k, int c) -> double& { return hist[(k * D + c) * NT + th.tid]; };
#pragma unroll
                        for (int cc = 0; cc < D; cc++)
                            var_accept_coord<D>(th.q, cc, th.x0[cc], th.csx[cc], th.v0[cc], th.csv[cc], th.a0[cc], dt, dt2, q, e, h);
                    });
                    w.t += dt;
                    w.dt_last_done = dt;
                }
                // publish x0 for the encounter test and the next attempt's a0
                double* Xp = pos + cur * L.npos;
                ex.each([&](VarThread<P, D>& th) {
                    if (th.order < 0) return;
#pragma unroll
                    for (int cc = 0; cc < D; cc++) Xp[(th.set * P + th.planet) * D + cc] = th.x0[cc];
                });
                ex.sync();
                return (accepted ? 1 : 0) | (var_encounter<P, D>(Xp, u) ? 2 : 0);
            };

            final_status = var_leg_epochs(ex, a, md, item, w, attempt,
                [&]() { return var_encounter<P, D>(pos + cur * L.npos, u); },
                [&](int ie) {
                    // star vx of every set, chi2 / d / dd sums (state.py:264-271)
                    ex.each([&](VarThread<P, D>& th) { if (th.order >= 0) vxs[th.set * P + th.planet] = th.v0[0]; });
                    ex.sync();
                    const double svx = var_star_vx<P>(vxs, dm, u, 0, 0, 0, 0, 0, 0);
                    if (!isfinite(svx)) return false;
                    const double res = svx - a.orv[ie], er = a.oerr[ie];
                    const double den = er * er * a.npoints;
                    ex.each([&](VarThread<P, D>& th) {
                        if (th.order >= 0 && th.planet == 0)
                            th.acc += var_epoch_term<P>(vxs, dm, u, th.order, th.set, th.sa, th.sb, th.pa, th.pb, res, den);
                    });
                    return true;
                });
        }
        // ---- results of this leg -----------------------------------------------------------------
        const int fs = final_status;
        ex.each([&](VarThread<P, D>& th) {
            if (th.tid == 0 && (L.k2_lo == 0 || fs != ST_OK)) a.part_status[item] = fs;     // a failure in any launch fails the leg
            // value and gradient come from the launch that carries the first pairs
            if (fs == ST_OK && th.order >= 0 && th.planet == 0 && (th.order == 2 || L.k2_lo == 0))
                a.part[item * L.nsets_total + th.gset] = th.acc;
        });
        ex.add_work(a.work_counters, n_force, n_attempt);
    }
}

}  // namespace rv
