// rv_core_g.cuh -- IAS15 step with the predictor-corrector loop written on the g coefficients only.
//
// rebound keeps both g and b current inside the loop (b += dg * c after every substep) because its predictor reads b.
// Here the predictor reads g through PG = PRED * C^T, so the loop carries only g (7 values per coordinate): b is
// formed once per step (b = C^T g) for the error estimate, the position / velocity update and the next-step
// prediction.  Per coordinate and substep that removes the (n-1)+1 b-update FMAs and 7 live registers; the e
// coefficients (touched once per step) live in shared memory next to the rejected-step history.  The step
// sequence, accept / reject rule and stopping rule are unchanged; results differ from the b-carrying form by
// rounding only.
#pragma once
#include "rv_core.cuh"

namespace rv {

template <int VAR> RV_D double tPG(int n, int k) { if constexpr ((VAR & 2) != 0) return rvtabm::PG[n][k]; else return rvtab::PG[n][k]; }

template <int P, int D, int PL, int VAR = 0>
struct WalkerG : Walker<P, D, PL, VAR> {
    using B = Walker<P, D, PL, VAR>;
    static constexpr int NC = B::NC;
    static constexpr int DENSE0 = B::STATE_DOUBLES;        // after Walker's slots: 9 per own planet, v0x, a0x, b0x..b6x of the last step
    static constexpr bool kDense = (VAR & 4) != 0;         // dense-output instantiation (model option dense_output)
    // off-chain sums of a substep: one accumulator (fewest FP64 instructions: +1 % in the default mode, which is bound by
    // FP64-pipe throughput) or two (shorter chains: +4 % in the dense-output mode); measured, profiles/r02p_loglik_variants.txt
    static constexpr bool kSplitAcc = kDense;
    static constexpr int LANE_DOUBLES = DENSE0 + (kDense ? 9 * PL : 0);   // shared-memory doubles per lane
    using B::mu;
    using B::x0c; using B::v0; using B::ha0; using B::ebank; using B::a0_stale;
    using B::b;                       // holds b between attempts and g inside the predictor-corrector loop
    using B::dt; using B::grp; using B::hist; using B::inv_eps;
    using B::star_in_norm; using B::n_force; using B::n_attempt;

    // One Gauss-Radau substep, software-pipelined: the only predictor term on the dependency chain is the one of the g
    // coefficient the PREVIOUS substep has just updated (index kl); every other term was summed into pp while that substep's
    // force evaluation was in flight.  Likewise the corrector's divided-difference sum over the older g (and a0) is formed
    // before the force is known, so that g_{n-1} = fma(a_n, GA[n], sc) is one operation after it.  Same arithmetic as the
    // straightforward form up to the order of summation.
    //   pp[c]  in : ha0 + sum_{k != kl} PG[n][k] g_k         out: the same for the next substep (n % 7 + 1), without k = n - 1
    template <int n>
    RV_D void substep_g(bool commit, const double (&x0c)[NC], double (&xp)[NC], double (&at)[NC], double (&dg6)[NC],
                        double (&pp)[NC]) {
        constexpr int kl = (n == 1) ? 6 : n - 2;
        constexpr int m = (n % 7) + 1;
        const double dth = dt * tH<VAR>(n);
        double xn[NC], an[NC], sc[NC], ppn[NC];
#pragma unroll
        for (int c = 0; c < NC; c++) {
            const double p = fma(tPG<VAR>(n, kl), b[kl][c], pp[c]);
            const double inner = fma(dth, p, v0[c]);
            xn[c] = fma(dth, inner, x0c[c]);
        }
        // off the dependency chain of the force evaluation below
#pragma unroll
        for (int c = 0; c < NC; c++) {
          if constexpr (!kSplitAcc) {
            double s0 = ha0[c] * (-2.0 * tGA<VAR>(n));
#pragma unroll
            for (int i = 0; i < n - 1; i++) s0 = fma(-b[i][c], tGB<VAR>(n, i), s0);
            sc[c] = s0;
            double q0 = ha0[c];
#pragma unroll
            for (int k = 0; k < 7; k++) {
                if (k == n - 1) continue;
                q0 = fma(tPG<VAR>(m, k), b[k][c], q0);
            }
            ppn[c] = q0;
          } else {
            double s0 = ha0[c] * (-2.0 * tGA<VAR>(n)), s1 = 0.0;
#pragma unroll
            for (int i = 0; i < n - 1; i++) {
                if (i & 1) s1 = fma(-b[i][c], tGB<VAR>(n, i), s1);
                else s0 = fma(-b[i][c], tGB<VAR>(n, i), s0);
            }
            sc[c] = s0 + s1;
            double q0 = ha0[c], q1 = 0.0;
#pragma unroll
            for (int k = 0; k < 7; k++) {
                if (k == n - 1) continue;
                if (k & 1) q1 = fma(tPG<VAR>(m, k), b[k][c], q1);
                else q0 = fma(tPG<VAR>(m, k), b[k][c], q0);
            }
            ppn[c] = q0 + q1;
          }
        }
        this->accel(xn, an);
#pragma unroll
        for (int c = 0; c < NC; c++) {
            const double gn = fma(an[c], tGA<VAR>(n), sc[c]);
            if (n == 7) {
                dg6[c] = sel(commit, gn - b[6][c], dg6[c]);
                at[c] = sel(commit, an[c], at[c]);
                xp[c] = sel(commit, xn[c], xp[c]);
            }
            b[n - 1][c] = sel(commit, gn, b[n - 1][c]);
            pp[c] = ppn[c];
        }
    }

    // Star x-velocity at fraction h in (0, 1] of the step just accepted (size dt_done), from that step's acceleration
    // polynomial a(h) = a0 + b0 h + ... + b6 h^7:  v(h) = v0 + dt h (a0 + h (b0/2 + h (b1/3 + ... + h b6/8))).
    RV_D double dense_star_vx(double h, double dt_done) const {
        double s = 0.0;
#pragma unroll
        for (int pl = 0; pl < PL; pl++) {
            double p = hist.at(DENSE0 + 9 * pl + 8) * (1. / 8.);
            p = fma(p, h, hist.at(DENSE0 + 9 * pl + 7) * (1. / 7.));
            p = fma(p, h, hist.at(DENSE0 + 9 * pl + 6) * (1. / 6.));
            p = fma(p, h, hist.at(DENSE0 + 9 * pl + 5) * (1. / 5.));
            p = fma(p, h, hist.at(DENSE0 + 9 * pl + 4) * (1. / 4.));
            p = fma(p, h, hist.at(DENSE0 + 9 * pl + 3) * (1. / 3.));
            p = fma(p, h, hist.at(DENSE0 + 9 * pl + 2) * 0.5);
            p = fma(p, h, hist.at(DENSE0 + 9 * pl + 1));
            const double vx = fma(dt_done * h, p, hist.at(DENSE0 + 9 * pl + 0));
            s += mu[pl] * vx;
        }
        return -grp.template sum<false>(s);
    }

    // b of the next attempt, and its e into the slots from eo on
    RV_D void predict_g(double q, const double (&_e)[7], const double (&_b)[7], int c, int eo) {
        // rebound: ratio > 20 -> e = b = 0.  Branch-free and select-free: q -> 0 zeroes every e, keep = 0 drops (b - e_old)
        // (for finite coefficients; a walker with non-finite coefficients is already on its way to ST_NONFINITE)
        const bool far = q > 20.0;
        const double keep = far ? 0.0 : 1.0;
        const double q1 = far ? 0.0 : q, q2 = q1 * q1, q3 = q1 * q2, q4 = q2 * q2, q5 = q2 * q3, q6 = q3 * q3, q7 = q3 * q4;
        double e[7];
        e[0] = q1 * (_b[6] * 7.0 + _b[5] * 6.0 + _b[4] * 5.0 + _b[3] * 4.0 + _b[2] * 3.0 + _b[1] * 2.0 + _b[0]);
        e[1] = q2 * (_b[6] * 21.0 + _b[5] * 15.0 + _b[4] * 10.0 + _b[3] * 6.0 + _b[2] * 3.0 + _b[1]);
        e[2] = q3 * (_b[6] * 35.0 + _b[5] * 20.0 + _b[4] * 10.0 + _b[3] * 4.0 + _b[2]);
        e[3] = q4 * (_b[6] * 35.0 + _b[5] * 15.0 + _b[4] * 5.0 + _b[3]);
        e[4] = q5 * (_b[6] * 21.0 + _b[5] * 6.0 + _b[4]);
        e[5] = q6 * (_b[6] * 7.0 + _b[5]);
        e[6] = q7 * _b[6];
#pragma unroll
        for (int k = 0; k < 7; k++) {
            b[k][c] = fma(keep, _b[k] - _e[k], e[k]);
            hist.at(eo + k * NC + c) = e[k];
        }
    }

    // One IAS15 step attempt, executed by all 32 lanes of the warp together (full-mask exchanges); `active`: this lane's
    // group is integrating.  Returns bit 0: the step was accepted; bit 1: it was accepted and ends in an Encounter.
    //
    // The first force of an attempt, accel(x0), is evaluated at the end of the attempt before it: on the position the
    // step would reach if accepted, beside the step-size controller's latency chain (group maxima, division, seventh
    // root), and committed with the step.  A rejected step leaves x0 and so a0 as they were.  The encounter test after an
    // accepted step reads the same positions and shares their exchange.
    RV_D int attempt(bool active) {
        warp_converge();
        if (active) { n_attempt++; }
        if (warp_any(a0_stale)) {          // the first attempt of an item (set up between attempts, see Walker::a0_stale)
            double x[NC], a[NC];
#pragma unroll
            for (int c = 0; c < NC; c++) x[c] = this->x0(c);
            this->accel(x, a);              // bit-identical to the a0 of the lanes that are not stale
#pragma unroll
            for (int c = 0; c < NC; c++) ha0[c] = 0.5 * a[c];
            a0_stale = false;
        }
#pragma unroll
        for (int c = 0; c < NC; c++) {
            // g from b, in place (g_j needs b_k for k > j only)
#pragma unroll
            for (int j = 0; j < 7; j++) {
                double s = b[j][c];
#pragma unroll
                for (int k = 6; k > j; k--) s = fma(b[k][c], tDD<VAR>(k, j), s);
                b[j][c] = s;
            }
        }
        double xp[NC], at[NC], dg6[NC], pp[NC];
#pragma unroll
        for (int c = 0; c < NC; c++) {
            // every active lane commits xp, at, dg6 in its first iteration; inactive lanes' values are never used
            xp[c] = 0.0; at[c] = 0.0; dg6[c] = 0.0;
            // predictor partial sum of substep 1: every term but g6's (see substep_g)
            double q0 = tPG<VAR>(1, 0) * b[0][c];
#pragma unroll
            for (int k = 1; k < 6; k++) q0 = fma(tPG<VAR>(1, k), b[k][c], q0);
            pp[c] = q0 + ha0[c];
        }
        Ratio pc_err{1e300, 1.0}, pc_last{2.0, 1.0};
        int it = 0;
        bool iterating = active;
        while (true) {
            // rebound's stopping rule, evaluated without short-circuit branches (three predicates, one vote)
            const bool stop = ratio_lt(pc_err, 1e-16) | ((it > 2) & ratio_le(pc_last, pc_err)) | (it >= 12);
            iterating = iterating & !stop;
            if (!warp_any(iterating)) break;
            if (iterating) { pc_last = pc_err; it++; }
            substep_g<1>(iterating, x0c, xp, at, dg6, pp);
            substep_g<2>(iterating, x0c, xp, at, dg6, pp);
            substep_g<3>(iterating, x0c, xp, at, dg6, pp);
            substep_g<4>(iterating, x0c, xp, at, dg6, pp);
            substep_g<5>(iterating, x0c, xp, at, dg6, pp);
            substep_g<6>(iterating, x0c, xp, at, dg6, pp);
            substep_g<7>(iterating, x0c, xp, at, dg6, pp);
            double maxdg = 0.0, maxat = 0.0;
#pragma unroll
            for (int c = 0; c < NC; c++) {
                const double ak = fabs(at[c]), dg = fabs(dg6[c]);
                norm_max(ak, maxat);
                norm_max(dg, maxdg);
            }
            if (warp_any(star_in_norm)) {
#pragma unroll
                for (int d = 0; d < D; d++) {
                    const double sa = fabs(this->template star_of<true>(at, d)), sg = fabs(this->template star_of<true>(dg6, d));
                    if (star_in_norm) { norm_max(sa, maxat); norm_max(sg, maxdg); }
                }
            }
            maxdg = grp.template gmax<true>(maxdg);
            maxat = grp.template gmax<true>(maxat);
            if (iterating) { pc_err.num = maxdg; pc_err.den = maxat; }
        }
        if (active) n_force += 7 * it + 1;
        // b from g, in place (b_k needs g_j for j > k only)
#pragma unroll
        for (int c = 0; c < NC; c++) {
#pragma unroll
            for (int k = 0; k < 7; k++) {
                double s = b[k][c];
#pragma unroll
                for (int j = 6; j > k; j--) s = fma(b[j][c], tCC<VAR>(j, k), s);
                b[k][c] = s;
            }
        }
        // step-size control
        double maxak = 0.0, maxb6 = 0.0;
#pragma unroll
        for (int pl = 0; pl < PL; pl++) {
            double v2 = 0.0, x2 = 0.0;
#pragma unroll
            for (int d = 0; d < D; d++) { v2 = fma(v0[pl * D + d], v0[pl * D + d], v2); x2 = fma(xp[pl * D + d], xp[pl * D + d], x2); }
            const bool keep = !(fabs(v2 * dt * dt) < 1e-16 * x2);
#pragma unroll
            for (int d = 0; d < D; d++) {
                const double ak = fabs(at[pl * D + d]), b6 = fabs(b[6][pl * D + d]);
                if (keep) { norm_max(ak, maxak); norm_max(b6, maxb6); }
            }
        }
        if (warp_any(star_in_norm)) {
            double v2 = 0.0, x2 = 0.0, sa[D], sb[D];
#pragma unroll
            for (int d = 0; d < D; d++) {
                const double sv = this->template star_of<true>(v0, d), sx = this->template star_of<true>(xp, d);
                v2 = fma(sv, sv, v2); x2 = fma(sx, sx, x2);
                sa[d] = fabs(this->template star_of<true>(at, d)); sb[d] = fabs(this->template star_of<true>(b[6], d));
            }
            const bool keep = star_in_norm && !(fabs(v2 * dt * dt) < 1e-16 * x2);
#pragma unroll
            for (int d = 0; d < D; d++) {
                if (keep) { norm_max(sa[d], maxak); norm_max(sb[d], maxb6); }
            }
        }
        maxak = grp.template gmax<true>(maxak);
        maxb6 = grp.template gmax<true>(maxb6);
        // The position this step reaches if it is accepted (compensated summation), x0c = x0 - csx there, and the force
        // and the encounter test at it: they depend on b only, so they run beside the controller's chain below.
        const double dt_done = dt;
        const double dt2 = dt_done * dt_done;
        double xn[NC], csxn[NC], an[NC];
#pragma unroll
        for (int c = 0; c < NC; c++) {
            double s = b[6][c] * (1. / 72.);
            s = fma(b[5][c], 1. / 56., s); s = fma(b[4][c], 1. / 42., s); s = fma(b[3][c], 1. / 30., s);
            s = fma(b[2][c], 1. / 20., s); s = fma(b[1][c], 1. / 12., s); s = fma(b[0][c], 1. / 6., s);
            const double sx = ha0[c] + s;
            const double a = this->x0(c);
            double cs = this->csx(c) + fma(sx, dt2, v0[c] * dt_done);
            xn[c] = a + cs;
            csxn[c] = cs + (a - xn[c]);
        }
        typename B::Others xo;
        this->template others<true>(xn, xo);
        this->accel(xn, xo, an);
        const bool hit = this->template encounter<true>(xn, xo);
        int result = 0;
        if (active) {
            const double err = maxb6 / maxak;
            // ratio = dt_new / dt_done as the controller produces it (rebound divides the product again; same to 1 ulp)
            double ratio = 4.0;
            if (is_normal(err)) ratio = inv_root7(err * inv_eps);
            double dt_new = ratio * dt_done;
            if (fabs(dt_new) < 0.25 * fabs(dt_done)) {
                dt = dt_new;
                if (this->dt_last_done() != 0.0) {
                    const double q = dt / this->dt_last_done();
#pragma unroll
                    for (int c = 0; c < NC; c++) {
                        double _e[7], _b[7];
#pragma unroll
                        for (int k = 0; k < 7; k++) { _e[k] = hist.at(ebank + k * NC + c); _b[k] = hist.at(B::SLOT_BR + k * NC + c); }
                        predict_g(q, _e, _b, c, B::EBANK - ebank);
                    }
                } else {
                    // no history yet: rebound retries with the b it holds (the corrected ones)
                }
            } else {
                if (fabs(dt_new) > 4.0 * fabs(dt_done)) { dt_new = dt_done * 4.0; ratio = 4.0; }   // same sign: dt_new/dt_done > 1/safety
                dt = dt_new;
                if constexpr (kDense) {
#pragma unroll
                    for (int pl = 0; pl < PL; pl++) {
                        hist.at(DENSE0 + 9 * pl + 0) = v0[pl * D];
                        hist.at(DENSE0 + 9 * pl + 1) = ha0[pl * D] + ha0[pl * D];
#pragma unroll
                        for (int k = 0; k < 7; k++) hist.at(DENSE0 + 9 * pl + 2 + k) = b[k][pl * D];
                    }
                }
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    double u = b[6][c] * (1. / 8.);
                    u = fma(b[5][c], 1. / 7., u); u = fma(b[4][c], 1. / 6., u); u = fma(b[3][c], 1. / 5., u);
                    u = fma(b[2][c], 1. / 4., u); u = fma(b[1][c], 1. / 3., u); u = fma(b[0][c], 1. / 2., u);
                    const double sv = u + (ha0[c] + ha0[c]);
                    this->x0(c) = xn[c];
                    this->csx(c) = csxn[c];
                    x0c[c] = xn[c] - csxn[c];
                    ha0[c] = 0.5 * an[c];
                    const double a = v0[c];
                    double cs = fma(sv, dt_done, this->csv(c));
                    v0[c] = a + cs;
                    this->csv(c) = cs + (a - v0[c]);
                }
                this->t() += dt_done;
                this->dt_last_done() = dt_done;
                // this step's e becomes er (a swap of the two banks' roles); br is stored from the b just accepted
                ebank = B::EBANK - ebank;
                const double q = ratio;
#pragma unroll
                for (int c = 0; c < NC; c++) {
                    double _e[7], _b[7];
#pragma unroll
                    for (int k = 0; k < 7; k++) {
                        _e[k] = hist.at(ebank + k * NC + c); _b[k] = b[k][c];
                        hist.at(B::SLOT_BR + k * NC + c) = _b[k];
                    }
                    predict_g(q, _e, _b, c, B::EBANK - ebank);
                }
                result = hit ? 3 : 1;
            }
        }
        return result;
    }

};

}  // namespace rv
