// rv_core.cuh -- per-walker RV log-likelihood engine (fp64 IAS15 Gauss-Radau, adaptive step).
//
// Replaces, on the GPU, what the reference does per likelihood evaluation through rebound:
//   state.py:36-47   setup_sim      (Pal elements -> cartesian, move_to_com, exit_min_distance)
//   state.py:61-73   get_rv         (sim.integrate(t) to every epoch, star vx)
//   state.py:89-110  get_chi2/get_logp
// Mapping: one lane per planet (PL=1, G=P lanes per walker, positions exchanged with warp shuffles) or
// one thread per walker (PL=P).  The star is implicit: in the barycentric frame total momentum is
// conserved, so r_star = -sum(m_p r_p)/m_star and v_star likewise; only the planets are integrated.
// Coplanar systems (no ix/iy) drop the identically-zero z coordinate (D=2).
//
// The step sequence follows rebound's reb_integrate/exact_finish_time/IAS15 logic decision by decision
// (same accept/reject rule, same predictor-corrector stopping rule, same encounter sampling after every
// accepted step), so Encounter outcomes match the reference; only the rounding of individual operations
// differs (FMA contraction, closed-form divided differences, rsqrt by Newton).
#pragma once
#include <math.h>
#include <float.h>
#include <stdint.h>
#include "rv_tables.cuh"

#if defined(__CUDACC__)
#define RV_HD __host__ __device__ __forceinline__
#define RV_D __device__ __forceinline__
#else
#define RV_HD inline __attribute__((always_inline))
#define RV_D inline __attribute__((always_inline))
#endif

namespace rv {

constexpr int MAXP = 5;            // planets per system supported by the compiled plain-likelihood kernels
constexpr int MAXP_VAR = 5;        // ... by the variational (gradient + Hessian) kernels
constexpr int NELEM = 7;           // m, a, h, k, l, ix, iy
constexpr int MAXV = MAXP * NELEM; // free parameters

enum : int { ST_OK = 0, ST_PRIOR = 1, ST_ENCOUNTER = 3, ST_NONFINITE = 8, ST_NOT_SPD = 9 };
enum : int { RUN = -1, RUN_LAST = -3 };
enum : int { EL_M = 0, EL_A, EL_H, EL_K, EL_L, EL_IX, EL_IY };

// Model description resident in HBM (one per rv_model handle).
struct Model {
    int P;                  // planets
    int nvars;              // free parameters
    int D;                  // 2 = coplanar specialisation, 3 = general
    int src[MAXP * NELEM];  // element (p,e) <- theta[src] if src >= 0, else fixed[]
    double fixed[MAXP * NELEM];
    int free_planet[MAXV], free_elem[MAXV];
    double hill_factor;     // exit_min_distance = hill_factor * max Hill radius (state.py:42-46)
    double dt0;             // rebound default 1e-3
    double epsilon;         // rebound default 1e-9
    double m_star;          // 1.0 (state.py:38)
    int max_attempts;       // safety bound on IAS15 step attempts per leg
    int check_prior;        // variational entry point: test priorHard first (1, default) or integrate regardless (0)
    int integrator;         // 0 = IAS15 (rebound's default, what the reference runs); 1 = WHFast with fixed step dt0
    int dense_output;       // plain path, 0 (default): every integrate() hop ends exactly on its epoch (rebound's
                            // exact_finish_time = 1: at least one truncated step per epoch); 1 = one continuous
                            // integration per leg with natural steps, the star's velocity at each epoch read from
                            // the step's own acceleration polynomial (implies monotone_backward)
    int monotone_backward;  // plain path: 0 (default) visit obs.tb in stored (ascending) order as state.py:91 does --
                            // first hop to the most negative epoch, then forward; 1 = sweep 0 -> most negative once
                            // (the order state.py:273 uses), half the backward steps, logp equal to ~1e-11
};

RV_HD bool is_normal(double x) {
    const double a = fabs(x);
    return a >= DBL_MIN && a <= DBL_MAX;
}

// m = max(m, a) over the NORMAL values only (rebound's isnormal() guards in the IAS15 norms); a = |x| (or NaN), m >= 0.
// Device: exponent-field test and ordering on the integer pipe (for non-negative doubles the IEEE order is the integer order)
// -- the FP64 pipe, which bounds the kernels, is spared three DSETP per value.
RV_HD void norm_max(double a, double& m) {
#if defined(__CUDA_ARCH__)
    const unsigned e = ((unsigned)__double2hiint(a) & 0x7ff00000u) - 0x00100000u;   // exponent field 1..0x7fe <=> e < 0x7fe00000
    if (e < 0x7fe00000u && __double_as_longlong(a) > __double_as_longlong(m)) m = a;
#else
    if (is_normal(a) && a > m) m = a;
#endif
}

// 1/r^3 from r^2.
RV_HD double rinv3(double r2) {
#if defined(__CUDA_ARCH__)
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(r2));
    // one cubic (Halley-type) correction: y <- y (1 + e/2 + 3e^2/8), e = 1 - r2 y^2 ; seed error ~2^-22 -> < 2^-60
    const double t = r2 * y;
    const double e = fma(-t, y, 1.0);
    const double p = fma(0.375, e, 0.5) * e;
    y = fma(y, p, y);
    return y * y * y;
#else
    const double r = sqrt(r2);
    return 1.0 / (r2 * r);
#endif
}

// s / r^3 from r^2 (s = a mass factor, folded into the Newton step).  rsqrt seed y0 (relative error ~2^-22), then
//   1/r^3 = y0^3 (1 - e)^(-3/2),  e = 1 - r2 y0^2,  (1 - e)^(-3/2) = 1 + e (3/2 + 15/8 e) + O(e^3) ~ 2^-62:
// five dependent operations after the seed (mul, fma, fma, mul, fma), the mass product runs beside them.
RV_HD double rinv3_scaled(double r2, double s) {
#if defined(__CUDA_ARCH__)
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(r2));
    const double y2 = y * y;
    const double e = fma(-r2, y2, 1.0);
    const double k0 = (y2 * y) * s;
    const double c = fma(1.875, e, 1.5) * e;
    return fma(k0, c, k0);
#else
    const double r = sqrt(r2);
    return s / (r2 * r);
#endif
}

// u^(-1/7) for the IAS15 step-size controller (rebound: pow(epsilon/err, 1./7.)).  Device: single-precision seed and
// two division-free Newton steps on y^-7 = u (y <- y (8 - u y^7)/7), ~15 FP64 instructions instead of pow()'s ~150.
RV_HD double inv_root7(double u) {
#if defined(__CUDA_ARCH__)
    if (!(u > 1e-30 && u < 1e30)) return pow(u, -1.0 / 7.0);
    // seed: relative error <= ~6e-7 (float log2 of |log2 u| <= 100); Newton on y^-7 = u squares it with a factor 4:
    // 1.4e-12 after one step, < 1e-23 after two
    double y = (double)exp2f(-log2f((float)u) * (1.0f / 7.0f));
#pragma unroll
    for (int k = 0; k < 2; k++) {
        const double y2 = y * y, y4 = y2 * y2;
        const double y7 = y4 * y2 * y;
        y = y * fma(-u, y7, 8.0) * (1.0 / 7.0);
    }
    return y;
#else
    return pow(u, -1.0 / 7.0);
#endif
}

// The predictor-corrector monitor of IAS15 compares ratios maxdg/maxat; carried as (numerator, denominator) pairs and
// compared by cross-multiplication, which removes an IEEE division (a ~45-instruction subroutine, 9% of the stall
// samples in profiles/r01e) from every iteration.  All quantities are >= 0.
struct Ratio {
    double num, den;
};
RV_HD bool ratio_lt(const Ratio& a, double c) { return a.num < c * a.den; }                       // a < c
RV_HD bool ratio_le(const Ratio& a, const Ratio& b) { return a.num * b.den <= b.num * a.den; }      // a <= b

// Kepler's equation in Pal's form: p - k sin(l+p) + h cos(l+p) = 0 (rebound: reb_tools_solve_kepler_pal).
RV_HD void kepler_pal(double h, double k, double l, double& slp, double& clp, double& p) {
    const double e2 = h * h + k * k;
    if (e2 < 0.09) {
        p = 0.0;
    } else {
        const double e = sqrt(e2), w = atan2(h, k);
        double M = fmod(l - w, 2.0 * M_PI);
        if (M > M_PI) M -= 2.0 * M_PI;
        if (M < -M_PI) M += 2.0 * M_PI;
        p = 0.85 * e * (sin(M) >= 0.0 ? 1.0 : -1.0);
    }
    for (int it = 0; it < 60; it++) {
        sincos(l + p, &slp, &clp);
        const double f = p - k * slp + h * clp, f1 = 1.0 - k * clp - h * slp;
        const double dp = -f / f1;
        p += dp;
        if (!(fabs(dp) >= 1e-16 * (1.0 + fabs(p)))) break;
    }
    sincos(l + p, &slp, &clp);
}

// Pal elements -> cartesian relative to a primary of mass Mp at rest at the origin (G = 1).
// out: x[3], v[3]
RV_HD void pal_to_cart(const double* el, double Mp, double* x, double* v) {
    const double m = el[EL_M], a = el[EL_A], h = el[EL_H], k = el[EL_K], l = el[EL_L], ix = el[EL_IX], iy = el[EL_IY];
    double slp, clp, p;
    kepler_pal(h, k, l, slp, clp, p);
    const double q = k * clp + h * slp;
    const double lp = 1.0 - sqrt(1.0 - h * h - k * k);
    const double xi = a * (clp + p / (2.0 - lp) * h - k);
    const double eta = a * (slp - p / (2.0 - lp) * k - h);
    const double iz = sqrt(fabs(4.0 - ix * ix - iy * iy));
    const double W = eta * ix - xi * iy;
    x[0] = xi + 0.5 * iy * W;
    x[1] = eta - 0.5 * ix * W;
    x[2] = 0.5 * iz * W;
    const double an = sqrt((m + Mp) / a);
    const double dxi = an / (1.0 - q) * (-slp + q / (2.0 - lp) * h);
    const double deta = an / (1.0 - q) * (+clp - q / (2.0 - lp) * k);
    const double dW = deta * ix - dxi * iy;
    v[0] = dxi + 0.5 * iy * dW;
    v[1] = deta - 0.5 * ix * dW;
    v[2] = 0.5 * iz * dW;
}

// priorHard for one planet (state.py:299-315)
RV_HD bool prior_hard(const double* el) {
    if (el[EL_A] <= 0.02) return true;
    if (el[EL_M] <= 5e-6) return true;
    if (el[EL_H] * el[EL_H] + el[EL_K] * el[EL_K] >= 1.0) return true;
    if (el[EL_IX] * el[EL_IX] + el[EL_IY] * el[EL_IY] >= 4.0) return true;
    return false;
}

// ---------------------------------------------------------------------------------------------
// Lane group: the G lanes that share one walker.  Every exchange exists in two flavours:
//   U = true  : full-mask shuffle, only legal where all 32 lanes of the warp execute it together
//               (the step-attempt body, which the warp runs in lock-step);
//   U = false : group-mask shuffle for the divergent bookkeeping between attempts.
template <int G>
struct Group {
    static constexpr int lanes = G;
    unsigned mask;
    int base, rank;
    RV_HD void init(int lane) {
        base = (lane / G) * G;
        rank = lane - base;
        mask = (G >= 32) ? 0xffffffffu : (((1u << G) - 1u) << base);
    }
    // value held by the lane with rank r
    template <bool U>
    RV_D double from(double v, int r) const {
#if defined(__CUDA_ARCH__)
        if (G > 1) return __shfl_sync(U ? 0xffffffffu : mask, v, base + r);
#endif
        (void)r;
        return v;
    }
    // value held by the lane `o` ranks ahead (cyclic) -- for G == 2 this is the xor-1 partner
    template <bool U>
    RV_D double ahead(double v, int o) const {
#if defined(__CUDA_ARCH__)
        if (G == 2) return __shfl_xor_sync(U ? 0xffffffffu : mask, v, 1);
        if (G > 2) {
            int r = rank + o;
            if (r >= G) r -= G;
            return __shfl_sync(U ? 0xffffffffu : mask, v, base + r);
        }
#endif
        (void)o;
        return v;
    }
    template <bool U>
    RV_D double gmax(double v) const {
        double m = v;
#if defined(__CUDA_ARCH__)
        if (G == 2) {
            m = fmax(m, __shfl_xor_sync(U ? 0xffffffffu : mask, v, 1));
        } else if (G > 2) {
#pragma unroll
            for (int r = 0; r < G; r++) m = fmax(m, __shfl_sync(U ? 0xffffffffu : mask, v, base + r));
        }
#endif
        return m;
    }
    template <bool U>
    RV_D bool any(bool f) const {
#if defined(__CUDA_ARCH__)
        if (G > 1) {
            const unsigned bal = __ballot_sync(U ? 0xffffffffu : mask, f);
            return (bal & mask) != 0u;
        }
#endif
        return f;
    }
    // canonical (rank-ordered) sum: identical bits on every lane of the group
    template <bool U>
    RV_D double sum(double v) const {
#if defined(__CUDA_ARCH__)
        if (G > 1) {
            double s = __shfl_sync(U ? 0xffffffffu : mask, v, base);
#pragma unroll
            for (int r = 1; r < G; r++) s += __shfl_sync(U ? 0xffffffffu : mask, v, base + r);
            return s;
        }
#endif
        return v;
    }
};

// all 32 lanes of the warp vote (device); identity on the host mirror
RV_D bool warp_any(bool f) {
#if defined(__CUDA_ARCH__)
    return __any_sync(0xffffffffu, f) != 0;
#else
    return f;
#endif
}
RV_D double sel(bool c, double a, double b) { return c ? a : b; }
// re-converge the warp (lets the compiler emit plain SHFL for the full-mask exchanges that follow)
RV_D void warp_converge() {
#if defined(__CUDA_ARCH__)
    __syncwarp();
#endif
}

// Per-lane store of the state touched once per step attempt or less (layout: Walker::SLOT_*), strided so that
// consecutive lanes touch consecutive doubles (shared memory on the device).
struct Hist {
    double* p;
    int stride;
    RV_HD double& at(int i) const { return p[(size_t)i * stride]; }
};

// ---------------------------------------------------------------------------------------------
// One walker (or one planet of a walker when PL == 1): state, gravity, encounter test, set-up.  The IAS15 step
// itself is WalkerG::attempt (rv_core_g.cuh).
// VAR: compile-time switches -- bit1 (2): IAS15 tables read from the constant bank (else folded into immediates; measured
// identical on B200, profiles/r01c_variants.txt); bit2 (4): dense-output instantiation (model option dense_output).
template <int VAR> RV_D double tH(int n) { if constexpr ((VAR & 2) != 0) return rvtabm::H[n]; else return rvtab::H[n]; }
template <int VAR> RV_D double tGA(int n) { if constexpr ((VAR & 2) != 0) return rvtabm::GA[n]; else return rvtab::GA[n]; }
template <int VAR> RV_D double tPRED(int n, int k) { if constexpr ((VAR & 2) != 0) return rvtabm::PRED[n][k]; else return rvtab::PRED[n][k]; }
template <int VAR> RV_D double tGB(int n, int k) { if constexpr ((VAR & 2) != 0) return rvtabm::GB[n][k]; else return rvtab::GB[n][k]; }
template <int VAR> RV_D double tCC(int n, int k) { if constexpr ((VAR & 2) != 0) return rvtabm::CC[n][k]; else return rvtab::CC[n][k]; }
template <int VAR> RV_D double tDD(int n, int k) { if constexpr ((VAR & 2) != 0) return rvtabm::DD[n][k]; else return rvtab::DD[n][k]; }
template <int P, int D, int PL, int VAR = 0>
struct Walker {
    static constexpr int G = P / PL;    // lanes per walker
    static constexpr int NC = PL * D;   // coordinates held by this lane
    static_assert(PL == 1 || PL == P, "PL must be 1 or P");

    // Per-lane shared-memory slots (Hist), in units of NC doubles:
    //   [0, 21)  two banks of 7 that alternate as rebound's e and er (EBANK: which one holds e), then br[7]
    //   21, 22, 23  x0, csx, csv: read once per accepted step (and by the encounter test), never in the loop
    //   then four scalars, t, dt_last_done and the current hop's tmax, last_full_dt (LegCursor): read between attempts
    // x0c = x0 - csx, v0 and a0/2 are the forms of the state the predictor-corrector loop reads; they stay in registers.
    static constexpr int SLOT_BR = 7 * NC, SLOT_X0 = 21 * NC, SLOT_CSX = 22 * NC, SLOT_CSV = 23 * NC;
    static constexpr int SLOT_T = 24 * NC, SLOT_DT_LAST_DONE = 24 * NC + 1, SLOT_TMAX = 24 * NC + 2, SLOT_LAST_FULL_DT = 24 * NC + 3;
    static constexpr int STATE_DOUBLES = 24 * NC + 4;
    static constexpr int EBANK = 14 * NC;      // the bank of e when ebank == 0 (else of er)

    Group<G> grp;
    Hist hist;
    // IAS15 state
    double x0c[NC], v0[NC], ha0[NC];   // ha0 = a0 / 2 = accel(x0) / 2
    double b[7][NC];      // b between step attempts; the g coefficients inside the predictor-corrector loop
    double dt;
    int ebank;            // slot of er (0 or EBANK); e is at EBANK - ebank.  An accepted step swaps the two roles
    bool a0_stale;        // set up without its first force (accel needs the full warp; evaluated by the next attempt)
    // masses: own planets and (PL==1) the other planets in relative rank order
    double gm[PL];        // G*m of own planets
    double mu[PL];        // m/m_star of own planets
    double gmo[P > 1 ? P - 1 : 1], muo[P > 1 ? P - 1 : 1];
    double mu1;           // PL == 1: 1 + mu of the own planet
    double gm0;           // G*m_star
    double min2;          // exit_min_distance^2
    double inv_eps;       // 1 / epsilon (the step-size controller multiplies: one IEEE division less per attempt)
    bool star_in_norm;    // sum(mu) >= 1: the star can dominate the max-norms (never for planets)
    // diagnostic work counters per item, 32 bits (fewer registers): at most 85 forces per attempt and max_attempts attempts
    // per leg, exact for max_attempts up to 2^25 (default 2^20); larger user settings can wrap them, never the results
    unsigned n_force, n_attempt;

    RV_HD double& x0(int c) const { return hist.at(SLOT_X0 + c); }
    RV_HD double& csx(int c) const { return hist.at(SLOT_CSX + c); }
    RV_HD double& csv(int c) const { return hist.at(SLOT_CSV + c); }
    RV_HD double& t() const { return hist.at(SLOT_T); }
    RV_HD double& dt_last_done() const { return hist.at(SLOT_DT_LAST_DONE); }
    RV_HD double& tmax() const { return hist.at(SLOT_TMAX); }
    RV_HD double& last_full_dt() const { return hist.at(SLOT_LAST_FULL_DT); }

    // PL == 1: positions of the other planets of the walker, in relative rank order (unused for PL == P)
    using Others = double[P > 1 ? P - 1 : 1][D];
    template <bool U>
    RV_D void others(const double (&x)[NC], Others& xo) const {
        if constexpr (PL == 1) {
#pragma unroll
            for (int o = 0; o < P - 1; o++)
#pragma unroll
                for (int d = 0; d < D; d++) xo[o][d] = grp.template ahead<U>(x[d], o + 1);
        }
    }

    // ---- gravity on own coordinates from positions x (own lane's coordinates) -------------------
    // Runs only inside the warp-uniform attempt body (full-mask shuffles).
    RV_D void accel(const double (&x)[NC], double (&a)[NC]) {
        Others xo;
        others<true>(x, xo);
        accel(x, xo, a);
    }
    RV_D void accel(const double (&x)[NC], const Others& xo, double (&a)[NC]) const {
        if constexpr (PL == 1) {
            // planet - star separation ds = x + sum_j mu_j x_j = (1 + mu_own) x + sum_others mu_o x_o  (mu1 = 1 + mu_own)
            double ds[D], r2 = 0.0;
#pragma unroll
            for (int d = 0; d < D; d++) ds[d] = mu1 * x[d];
#pragma unroll
            for (int o = 0; o < P - 1; o++) {
#pragma unroll
                for (int d = 0; d < D; d++) ds[d] = fma(muo[o], xo[o][d], ds[d]);
            }
#pragma unroll
            for (int d = 0; d < D; d++) r2 = fma(ds[d], ds[d], r2);
            const double ks = rinv3_scaled(r2, -gm0);
#pragma unroll
            for (int d = 0; d < D; d++) a[d] = ks * ds[d];
#pragma unroll
            for (int o = 0; o < P - 1; o++) {
                double dp[D], q2 = 0.0;
#pragma unroll
                for (int d = 0; d < D; d++) { dp[d] = x[d] - xo[o][d]; q2 = fma(dp[d], dp[d], q2); }
                const double kp = rinv3_scaled(q2, -gmo[o]);
#pragma unroll
                for (int d = 0; d < D; d++) a[d] = fma(kp, dp[d], a[d]);
            }
        } else {
            double S[D];
#pragma unroll
            for (int d = 0; d < D; d++) {
                S[d] = 0.0;
#pragma unroll
                for (int j = 0; j < P; j++) S[d] = fma(mu[j], x[j * D + d], S[d]);
            }
#pragma unroll
            for (int i = 0; i < P; i++) {
                double ds[D], r2 = 0.0;
#pragma unroll
                for (int d = 0; d < D; d++) { ds[d] = x[i * D + d] + S[d]; r2 = fma(ds[d], ds[d], r2); }
                const double ks = rinv3_scaled(r2, -gm0);
#pragma unroll
                for (int d = 0; d < D; d++) a[i * D + d] = ks * ds[d];
            }
#pragma unroll
            for (int i = 0; i < P; i++)
#pragma unroll
                for (int j = i + 1; j < P; j++) {
                    double dp[D], q2 = 0.0;
#pragma unroll
                    for (int d = 0; d < D; d++) { dp[d] = x[i * D + d] - x[j * D + d]; q2 = fma(dp[d], dp[d], q2); }
                    const double r3 = rinv3(q2);
                    const double ki = -gm[j] * r3, kj = gm[i] * r3;
#pragma unroll
                    for (int d = 0; d < D; d++) {
                        a[i * D + d] = fma(ki, dp[d], a[i * D + d]);
                        a[j * D + d] = fma(kj, dp[d], a[j * D + d]);
                    }
                }
        }
    }

    // star coordinate d of a planet-linear quantity q (q_star = -sum_p mu_p q_p), canonical order
    template <bool U>
    RV_D double star_of(const double (&q)[NC], int d) const {
        if constexpr (PL == 1) {
            return -grp.template sum<U>(mu[0] * q[d]);
        } else {
            double s = 0.0;
#pragma unroll
            for (int j = 0; j < P; j++) s += mu[j] * q[j * D + d];
            return -s;
        }
    }

    // reb_run_heartbeat: any pair (star included) closer than exit_min_distance?  At positions x (others: see `others`).
    template <bool U>
    RV_D bool encounter(const double (&x)[NC], const Others& xo) const {
        bool hit = false;
        if constexpr (PL == 1) {
            double S[D];
#pragma unroll
            for (int d = 0; d < D; d++) S[d] = mu[0] * x[d];
#pragma unroll
            for (int o = 0; o < P - 1; o++) {
#pragma unroll
                for (int d = 0; d < D; d++) S[d] = fma(muo[o], xo[o][d], S[d]);
            }
            double r2 = 0.0;
#pragma unroll
            for (int d = 0; d < D; d++) { const double ds = x[d] + S[d]; r2 = fma(ds, ds, r2); }
            hit = r2 < min2;
#pragma unroll
            for (int o = 0; o < P - 1; o++) {
                double q2 = 0.0;
#pragma unroll
                for (int d = 0; d < D; d++) { const double dp = x[d] - xo[o][d]; q2 = fma(dp, dp, q2); }
                hit = hit || (q2 < min2);
            }
            hit = grp.template any<U>(hit);
        } else {
            double S[D];
#pragma unroll
            for (int d = 0; d < D; d++) {
                S[d] = 0.0;
#pragma unroll
                for (int j = 0; j < P; j++) S[d] = fma(mu[j], x[j * D + d], S[d]);
            }
#pragma unroll
            for (int i = 0; i < P; i++) {
                double r2 = 0.0;
#pragma unroll
                for (int d = 0; d < D; d++) { const double ds = x[i * D + d] + S[d]; r2 = fma(ds, ds, r2); }
                hit = hit || (r2 < min2);
#pragma unroll
                for (int j = i + 1; j < P; j++) {
                    double q2 = 0.0;
#pragma unroll
                    for (int d = 0; d < D; d++) { const double dp = x[i * D + d] - x[j * D + d]; q2 = fma(dp, dp, q2); }
                    hit = hit || (q2 < min2);
                }
            }
        }
        return hit && (min2 != 0.0);
    }
    // ... at the current position x0 (between attempts: group-mask exchanges)
    RV_D bool encounter() const {
        double x[NC];
        Others xo;
#pragma unroll
        for (int c = 0; c < NC; c++) x[c] = x0(c);
        others<false>(x, xo);
        return encounter<false>(x, xo);
    }

    // barycentric x-velocity of the star = the RV observable (state.py:72)
    RV_D double star_vx() const { return star_of<false>(v0, 0); }

    // ---- item setup: theta -> elements -> barycentric cartesian (setup_sim) ---------------------
    // returns status (ST_OK or ST_PRIOR).  check_prior=false mirrors get_rv (no prior test, state.py:61).
    RV_D int setup(const Model* __restrict__ md, const double* __restrict__ theta, bool check_prior) {
        double el[PL][NELEM];
        double xr[PL][3], vr[PL][3];
        bool bad = false;
        const double m0 = md->m_star;
#pragma unroll
        for (int pl = 0; pl < PL; pl++) {
            const int pidx = (PL == 1) ? grp.rank : pl;
#pragma unroll
            for (int k = 0; k < NELEM; k++) {
                const int s = md->src[pidx * NELEM + k];
                el[pl][k] = (s >= 0) ? theta[s] : md->fixed[pidx * NELEM + k];
            }
            bad = bad || prior_hard(el[pl]);
        }
        bad = grp.template any<false>(bad);
        if (check_prior && bad) return ST_PRIOR;
        double hill = 0.0, msum = 0.0;
#pragma unroll
        for (int pl = 0; pl < PL; pl++) {
            pal_to_cart(el[pl], m0, xr[pl], vr[pl]);
            gm[pl] = el[pl][EL_M];
            mu[pl] = el[pl][EL_M] / m0;
            if (PL == 1) mu1 = 1.0 + mu[pl];
            msum += el[pl][EL_M];
            const double rh = el[pl][EL_A] * pow(el[pl][EL_M] / (3.0 * m0), 1.0 / 3.0);
            if (rh > hill) hill = rh;
        }
        if constexpr (PL == 1) {
#pragma unroll
            for (int o = 0; o < P - 1; o++) {
                int r = grp.rank + 1 + o;
                if (r >= P) r -= P;
                gmo[o] = grp.template from<false>(gm[0], r);
                muo[o] = grp.template from<false>(mu[0], r);
            }
        }
        hill = grp.template gmax<false>(hill);
        msum = grp.template sum<false>(msum);
        const double mtot = m0 + msum;
        star_in_norm = (msum / m0 >= 1.0);
        gm0 = m0;
        const double emd = md->hill_factor * hill;
        min2 = emd * emd;
        inv_eps = 1.0 / md->epsilon;
        // move_to_com: the star sits at the origin before the shift
        double com_x[3], com_v[3];
#pragma unroll
        for (int d = 0; d < 3; d++) {
            double sx = 0.0, sv = 0.0;
#pragma unroll
            for (int pl = 0; pl < PL; pl++) { sx += el[pl][EL_M] * xr[pl][d]; sv += el[pl][EL_M] * vr[pl][d]; }
            com_x[d] = grp.template sum<false>(sx) / mtot;
            com_v[d] = grp.template sum<false>(sv) / mtot;
        }
#pragma unroll
        for (int pl = 0; pl < PL; pl++)
#pragma unroll
            for (int d = 0; d < D; d++) {
                x0(pl * D + d) = xr[pl][d] - com_x[d];
                x0c[pl * D + d] = xr[pl][d] - com_x[d];      // x0 - csx with csx = 0
                v0[pl * D + d] = vr[pl][d] - com_v[d];
            }
#pragma unroll
        for (int c = 0; c < NC; c++) {
            csx(c) = 0.0; csv(c) = 0.0; ha0[c] = 0.0;
#pragma unroll
            for (int k = 0; k < 7; k++) {
                b[k][c] = 0.0;
                hist.at(k * NC + c) = 0.0; hist.at((7 + k) * NC + c) = 0.0; hist.at((14 + k) * NC + c) = 0.0;
            }
        }
        ebank = 0;
        a0_stale = true;
        t() = 0.0; dt = md->dt0; dt_last_done() = 0.0;
        return ST_OK;
    }
};

// ---------------------------------------------------------------------------------------------
// Leg driver: the reference's `for t in times: sim.integrate(t)` loop flattened into a state machine
// whose only expensive state is "one IAS15 step attempt", so that the lane groups of a warp stay
// converged on the attempt body while each follows its own epoch / leg / item schedule.
struct LegCursor {
    int status;            // RUN / RUN_LAST / >=0 exit
    int ie;                // next epoch index
    int n;                 // epochs in this leg
    int attempts;          // attempts made in this leg
    double tmax, last_full_dt;
    double chi2;
};

// reb_check_exit with exact_finish_time = 1
template <class W>
RV_D int check_exit(W& w, LegCursor& c) {
    if (c.status >= 0) return c.status;
    const double sgn = copysign(1.0, w.dt);
    if ((w.t + w.dt) * sgn >= c.tmax * sgn) {
        if (w.t == c.tmax) {
            c.status = ST_OK;
        } else if (c.status == RUN_LAST) {
            double tscale = 1e-12 * fabs(c.tmax);
            if (tscale < 1e-200) tscale = 1e-12;
            if (fabs(w.t - c.tmax) < tscale) c.status = ST_OK;
            else w.dt = c.tmax - w.t;
        } else {
            c.status = RUN_LAST;
            if (w.dt_last_done != 0.0) c.last_full_dt = w.dt_last_done;
            w.dt = c.tmax - w.t;
        }
    } else if (c.status == RUN_LAST) {
        c.status = RUN;
    }
    return c.status;
}

}  // namespace rv
