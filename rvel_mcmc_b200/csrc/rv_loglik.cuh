// rv_loglik.cuh -- work-item state machine around rv::Walker.
//
// A work item is one leg of one walker's likelihood evaluation: the reference builds a fresh
// simulation per leg (state.py:90-91: get_rv(obs.tf) then get_rv(obs.tb)), so the two legs are
// independent integrations.  Lane groups pull items from a global counter; each iteration of the warp
// loop runs exactly one IAS15 step attempt for every group that is mid-integration, and the cheap
// bookkeeping (epoch reached -> record RV / chi2, next epoch, next item) happens in between.
#pragma once
#include "rv_core.cuh"

namespace rv {

struct LoglikArgs {
    const Model* model;
    const double* theta;      // [W][nvars] row-major
    long long W;
    // optional scheduling order: the i-th item of a leg is walker order[i] (most expensive first, walkers of similar cost
    // adjacent: the lane groups of a warp then stay in step, see cost_order in rv_kernels.cu); null = identity.  Results are
    // stored by walker, so the order never shows in the output.
    const int* order;
    // observation epochs: forward leg [0,nf), backward leg [nf,nf+nb) (order of obs.tf / obs.tb)
    const double* ot;
    const double* orv;
    const double* oerr;
    int nf, nb;
    int stage_obs;            // set by the launcher: copy the observation arrays into shared memory
    // RV-curve mode (state.py:61-73 get_rv on arbitrary times): one item per walker, no prior test
    const double* times;
    int nt;
    double* rv_out;           // [W][nt]
    // per-item results
    double* part_chi2;        // [2W]: item w = backward leg of walker w, item W+w = forward leg
    int* part_status;         // [2W] (curve mode: [W])
    unsigned long long* item_counter;
    unsigned long long* work_counters;  // [0] force evaluations, [1] step attempts (may be null)
};

enum : int { PH_NEED_ITEM = 0, PH_ENTRY, PH_CHECK, PH_STEP, PH_DONE };

// the integration clock as check_exit reads it (it changes dt only)
struct Clock { double t, dt, dt_last_done; };

// Fetch / WarpAll are policy objects: device = atomicAdd + shuffle / __all_sync, host mirror = trivial.
template <class WK, class Fetch, class WarpAll>
RV_D void run_items(WK& w, const LoglikArgs& a, const double* st, const double* srv,
                    const double* serr, Fetch& fetch, WarpAll& warp_all, bool lane_active) {
    const bool curve = (a.times != nullptr);
    const long long n_items = curve ? a.W : 2 * a.W;
    const int max_attempts = a.model->max_attempts;
    const int nvars = a.model->nvars;
    const bool leader = (w.grp.rank == 0);
    const bool dense_mode = WK::kDense && !curve;       // the launcher picks the dense instantiation from the model option
    const bool mono = a.model->monotone_backward != 0 || dense_mode;
    double sgn = 1.0;       // dense output: direction of the leg's single integration
    bool rev = false;       // this item visits its epochs in reversed storage order
    int phase = lane_active ? PH_NEED_ITEM : PH_DONE;
    long long item = -1, wi = 0, slot = 0;   // slot: where this item's partial results go (leg * W + walker)
    const double* lt = nullptr;              // the leg's epochs; its velocities and errors are srv / serr from index lo
    int lo = 0;
    LegCursor c;
    c.status = RUN; c.ie = 0; c.n = 0; c.attempts = 0; c.tmax = 0.0; c.last_full_dt = 0.0; c.chi2 = 0.0;

    auto finish = [&](int status) {
        if (leader) {
            a.part_status[slot] = status;
            if (!curve) a.part_chi2[slot] = c.chi2;
#if defined(__CUDA_ARCH__)
            if (a.work_counters) {
                atomicAdd(&a.work_counters[0], w.n_force);
                atomicAdd(&a.work_counters[1], w.n_attempt);
            }
#else
            if (a.work_counters) { a.work_counters[0] += w.n_force; a.work_counters[1] += w.n_attempt; }
#endif
        }
        phase = PH_NEED_ITEM;
    };

    for (;;) {
        while (phase != PH_STEP && phase != PH_DONE) {
            if (phase == PH_NEED_ITEM) {
                item = fetch(w.grp);
                if (item >= n_items) { phase = PH_DONE; break; }
                if (curve) {
                    wi = item; slot = item; lt = a.times; lo = 0; c.n = a.nt; rev = false;
                } else if (item < a.W) {       // backward legs first: they are the longer ones
                    wi = a.order ? (long long)a.order[item] : item; slot = wi;
                    lt = st + a.nf; lo = a.nf; c.n = a.nb; rev = mono;
                } else {
                    wi = a.order ? (long long)a.order[item - a.W] : item - a.W; slot = a.W + wi;
                    lt = st; lo = 0; c.n = a.nf; rev = false;
                }
                w.n_force = 0; w.n_attempt = 0;
                c.ie = 0; c.chi2 = 0.0; c.attempts = 0;
                const int s = w.setup(a.model, a.theta + wi * nvars, !curve);
                if (s != ST_OK) { finish(s); continue; }
                phase = PH_ENTRY;
                if (dense_mode) {
                    // one integration per leg: natural steps away from t = 0, RVs read inside the steps
                    sgn = (item < a.W) ? -1.0 : 1.0;
                    w.dt = sgn * fabs(w.dt);
                    if (w.encounter()) { finish(ST_ENCOUNTER); continue; }
                    int st0 = ST_OK;
                    while (c.ie < c.n) {            // epochs at the start time itself (obs.tf[0] = 0, obs.tb[-1] = 0)
                        const int io = rev ? c.n - 1 - c.ie : c.ie;
                        const double d = (lt[io] - w.t()) * sgn;
                        if (d > 0.0) break;
                        if (d < 0.0) { st0 = ST_NONFINITE; break; }       // an epoch behind the start: not a monotone leg
                        const double vx = w.star_vx();
                        const double r = vx - srv[lo + io], er = serr[lo + io];
                        c.chi2 += (r * r) / (er * er);
                        c.ie++;
                    }
                    if (st0 != ST_OK || c.ie == c.n) { finish(st0); continue; }
                    phase = PH_STEP;
                    break;
                }
            }
            if (phase == PH_ENTRY) {            // sim.integrate(t) entry (rebound: reb_integrate)
                if (c.ie == c.n) { finish(ST_OK); continue; }
                w.tmax() = lt[rev ? c.n - 1 - c.ie : c.ie];
                w.last_full_dt() = w.dt;
                w.dt_last_done() = 0.0;
                c.status = RUN;
                if (w.encounter()) c.status = ST_ENCOUNTER;
                phase = PH_CHECK;
            }
            if (phase == PH_CHECK) {
                // the clock and the hop's tmax / last_full_dt live in shared memory (Walker::SLOT_T ...)
                Clock k{w.t(), w.dt, w.dt_last_done()};
                c.tmax = w.tmax(); c.last_full_dt = w.last_full_dt();
                const int s = check_exit(k, c);
                w.dt = k.dt;
                w.last_full_dt() = c.last_full_dt;
                if (s < 0) { phase = PH_STEP; break; }
                w.dt = c.last_full_dt;
                if (s != ST_OK) { finish(s); continue; }
                const double vx = w.star_vx();
                if (!isfinite(vx)) { finish(ST_NONFINITE); continue; }
                if (curve) {
                    if (leader) a.rv_out[wi * a.nt + c.ie] = vx;
                } else {
                    const int io = rev ? c.n - 1 - c.ie : c.ie;
                    const double r = vx - srv[lo + io], er = serr[lo + io];
                    c.chi2 += (r * r) / (er * er);
                }
                c.ie++;
                phase = PH_ENTRY;
            }
        }
        if (warp_all(phase == PH_DONE)) break;
        // one step attempt, executed by the whole warp in lock-step (see Walker::attempt)
        const bool stepping = (phase == PH_STEP);
        const int r = w.attempt(stepping);
        if (stepping) {
            c.attempts++;
            if (c.attempts > max_attempts || !isfinite(w.dt) || w.dt == 0.0) {
                finish(ST_NONFINITE);
            } else if ((r & 1) && dense_mode) {
                // epochs inside the step just accepted: (t - dt_done, t]
                const double dt_done = w.dt_last_done();
                int st1 = (r & 2) ? ST_ENCOUNTER : ST_OK;
                while (st1 == ST_OK && c.ie < c.n) {
                    const int io = rev ? c.n - 1 - c.ie : c.ie;
                    if ((lt[io] - w.t()) * sgn > 0.0) break;
                    const double h = 1.0 + (lt[io] - w.t()) / dt_done;
                    double vx = 0.0;
                    if constexpr (WK::kDense) vx = w.dense_star_vx(h, dt_done);
                    if (!isfinite(vx)) { st1 = ST_NONFINITE; break; }
                    const double rr = vx - srv[lo + io], er = serr[lo + io];
                    c.chi2 += (rr * rr) / (er * er);
                    c.ie++;
                }
                if (st1 != ST_OK || c.ie == c.n) finish(st1);
            } else if (r & 1) {
                if (r & 2) c.status = ST_ENCOUNTER;
                phase = PH_CHECK;
            }
        }
    }
}

}  // namespace rv
