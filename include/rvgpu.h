/*
 * rvgpu.h -- C ABI of librvgpu.so: the B200 (sm_100a) replacement for the reference's per-evaluation
 * FFI into librebound.
 *
 * What it replaces.  rvel-mcmc reaches native code through ctypes, one call per observation epoch:
 *   clibrebound.reb_integrate(byref(sim), c_double(tmax))      (rebound/simulation.py, reached from
 *                                                               state.py:71, state.py:263, state.py:275)
 * preceded by per-evaluation set-up calls (state.py:37-46: Simulation(), add(), move_to_com()) and
 * followed by reads of sim.particles[0].vx (state.py:72).  A return value of 3 (REB_EXIT_ENCOUNTER)
 * becomes the Python exception rebound.Encounter (mcmc.py:119,176).  This library moves the whole
 * evaluation (set-up, every integrate() hop, the chi^2 sum of state.py:89-98) behind ONE call for a
 * whole batch of parameter vectors, and reports Encounter / hard-prior / non-finite outcomes as a
 * per-walker status instead of an exception.
 *
 * Conventions: every entry point returns 0 on success or a negative error code (rv_last_error() gives
 * the message); no exception crosses the ABI; all arrays are C-contiguous float64 / int32 owned by the
 * caller; the library keeps no host pointer after a call returns.  Element slots of a planet are
 * ordered m, a, h, k, l, ix, iy (RV_EL_*).
 */
#ifndef RVGPU_H
#define RVGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Threading: an rv_ctx owns grow-only scratch buffers and a work-queue counter that every entry point (the host-buffer
 * calls and the *_dev(stream) calls alike) reuses, so a context carries ONE call chain at a time: use it from one host
 * thread, and give all *_dev calls on one context the same stream (or synchronise between streams).  Concurrent work
 * = one context per host thread / rank / GPU; contexts are cheap.                                                 */
typedef struct rv_ctx rv_ctx;     /* one GPU + stream + scratch; one per host thread / rank       */
typedef struct rv_obs rv_obs;     /* observation set resident in HBM (observations.py:6-16)        */
typedef struct rv_model rv_model; /* parameter schema resident in HBM (state.py:8-31)              */

/* per-walker status */
#define RV_OK          0   /* evaluated                                                            */
#define RV_PRIOR       1   /* State.priorHard() true (state.py:299-315): logp = -inf, no integration */
#define RV_ENCOUNTER   3   /* rebound.Encounter (REB_EXIT_ENCOUNTER): logp = -inf                  */
#define RV_NONFINITE   8   /* non-finite state or step-count bound hit                             */
#define RV_NOT_SPD     9   /* SMALA metric not positive definite (mcmc.py:179-183 quits)           */

/* per-walker fit code of rv_map_fit */
#define RV_FIT_CONVERGED 0 /* Newton decrement / 2 <= tol and -H positive definite (min eigenvalue > 1e-12 max |eigenvalue|) */
#define RV_FIT_MAXITER   1 /* max_iter accepted steps, not converged                                  */
#define RV_FIT_STALLED   2 /* the line search found no ascent up to damping 1, or an evaluation after a step failed (status says why) */
#define RV_FIT_SADDLE    3 /* decrement / 2 <= tol but -H not positive definite: a saddle or a direction the data do not constrain */
#define RV_FIT_NOSTART   4 /* the start does not evaluate (status: RV_PRIOR, RV_ENCOUNTER, RV_NONFINITE); theta unchanged */

/* element slots */
#define RV_EL_M 0
#define RV_EL_A 1
#define RV_EL_H 2
#define RV_EL_K 3
#define RV_EL_L 4
#define RV_EL_IX 5
#define RV_EL_IY 6
#define RV_NELEM 7
#define RV_MAX_PLANETS 5      /* plain likelihood, samplers without derivatives (MH, stretch), WHFast */
#define RV_MAX_PLANETS_VAR 5  /* value + gradient + Hessian (rv_loglik_d_dd*, SMALA, ALSMALA): error -30 above */

/* ---- context ---------------------------------------------------------------------------------- */
int rv_ctx_create(int device, rv_ctx** out);
int rv_ctx_destroy(rv_ctx* ctx);
const char* rv_last_error(const rv_ctx* ctx);   /* ctx may be NULL: last creation error           */
int rv_device_info(const rv_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, int* clock_khz);
/* context options: "chain_walkers" (0 = all): the fused samplers (rv_mh_run, rv_stretch_run, rv_smala_run, rv_alsmala_run)
 * record only chains / walkers [0, n) in their chain rows -- chain[rows][min(n, W)][nvars], chain_logp[rows][min(n, W)] --
 * so that very large ensembles can be sampled without moving every position to the host; "count_work" (0/1).        */
int rv_ctx_set_option(rv_ctx* ctx, const char* key, double value);


/* ---- observations: replaces the Observation container (observations.py:6-16, 52-69) ----------- */
/* tf/rvf/errf: forward leg in obs.tf order; tb/rvb/errb: backward leg in obs.tb order (ascending, as
 * the reference integrates it, state.py:91); npoints: the Npoints normaliser of state.py:98.      */
int rv_obs_create(rv_ctx* ctx, const double* tf, const double* rvf, const double* errf, int nf,
                  const double* tb, const double* rvb, const double* errb, int nb, double npoints,
                  rv_obs** out);
int rv_obs_destroy(rv_obs* obs);

/* ---- model: replaces State's schema (state.py:8-31) + setup_sim constants (state.py:36-47) ---- */
/* fixed[n_planets][7]: element values used where a slot is not free (absent keys = 0);
 * free_planet/free_elem[nvars]: slot of each entry of a parameter vector, in State.get_params() order;
 * hill_factor: State.hillRadiusFactor; dims: 0 auto, 2 coplanar, 3 general.                       */
int rv_model_create(rv_ctx* ctx, int n_planets, const double* fixed, int nvars, const int32_t* free_planet,
                    const int32_t* free_elem, double hill_factor, int dims, rv_model** out);
int rv_model_destroy(rv_model* model);
/* options: "integrator" (0 = IAS15, rebound's default and what the reference runs; 1 = WHFast, fixed step "dt0", each leg
 *   swept monotonically -- no reference call site, parity unpinned; rv_loglik_d_dd / rv_smala_run refuse it),
 * "dt0" (1e-3), "epsilon" (1e-9), "max_attempts", "hill_factor", "mapping" (0 lane-per-planet, 1 thread-per-walker),
 * "check_prior" (1; 0 = rv_loglik_d_dd / rv_loglik_d_dd_dev integrate even outside the hard prior, as state.py:290
 *   does; the samplers ignore it and always test the prior; prefer rv_loglik_d_dd_opt's per-call argument),
 * "monotone_backward" (0 = rv_loglik visits obs.tb in its stored order as state.py:91 does; 1 = one sweep from 0 to the
 *   most negative epoch, the order state.py:273 uses: about half the backward steps, logp equal to ~1e-11),
 * "dense_output" (0 = every hop ends exactly on its epoch, rebound's exact_finish_time = 1; 1 = rv_loglik integrates each
 *   leg once with natural IAS15 steps and reads the RV at every epoch from the step's acceleration polynomial: the
 *   number of steps no longer grows with the number of epochs; implies monotone_backward; logp equal to ~1e-10),
 * "cost_order" (1 = batches of >= 4096 walkers are integrated most-expensive-first, walkers of similar cost side by side
 *   (key: max over planets of the pericentre distance^-3/2); scheduling only -- results are bit-identical to 0)      */
int rv_model_set_option(rv_model* model, const char* key, double value);

/* ---- State.get_logp (state.py:103-110) for W parameter vectors; HOST buffers -------------------- */
/* theta[W][nvars] -> logp[W], status[W].  Copies in, runs, copies out, synchronises.              */
int rv_loglik(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, const double* theta, int64_t W,
              double* logp, int32_t* status);

/* Same with DEVICE buffers, asynchronous on `stream` (a cudaStream_t; NULL = the legacy default stream,
 * rv_ctx_stream() = the context's own).  The context's scratch is reused: one call in flight per context. */
int rv_loglik_dev(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, const double* d_theta, int64_t W,
                  double* d_logp, int32_t* d_status, void* stream);

/* ---- State.get_rv (state.py:61-73): star vx at times[nt] (visited in the given order) ---------- */
/* rv[W][nt]; status[W]; no prior test (as the reference).  HOST buffers.                          */
int rv_rv_curve(rv_ctx* ctx, const rv_model* model, const double* theta, int64_t W, const double* times,
                int nt, double* rv, int32_t* status);

/* ---- State.setup_sim (state.py:36-47) made visible: the barycentric particles every integration starts from ---- */
/* particles[W][n_planets+1][7] = m, x, y, z, vx, vy, vz (star first), after rebound's Pal -> cartesian conversion
 * and move_to_com; status[W] = RV_PRIOR where priorHard() holds (the particles are still written).        */
int rv_initial_conditions(rv_ctx* ctx, const rv_model* model, const double* theta, int64_t W, double* particles,
                          int32_t* status);

/* ---- State.get_logp_d_dd (state.py:290-294; setup_sim_vars state.py:229-248, get_chi2_d_dd state.py:253-285) ---- */
/* theta[W][nvars] -> logp[W], grad[W][nvars], hess[W][nvars][nvars] (symmetric), status[W].  The hard prior is tested
 * first (status RV_PRIOR), as the reference's callers do (mcmc.py:171).  On a non-zero status logp = -inf and the
 * walker's grad / hess rows are zero.  Returns -30 when the model has more than RV_MAX_PLANETS_VAR planets.  Models whose
 * variational sets do not fit one thread block (three planets with more than 15 free parameters, four and five planets)
 * run their second-order sets in several launches; the results are those of one launch to rounding.             */
int rv_loglik_d_dd(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, const double* theta, int64_t W,
                   double* logp, double* grad, double* hess, int32_t* status);
/* Same with the prior test chosen PER CALL (check_prior = 0: integrate even outside the hard prior, which is what
 * State.get_logp_d_dd itself does, state.py:290-294) -- no model option is touched, so models shared between callers
 * keep their behaviour.  The samplers (rv_smala_run, rv_alsmala_run) always test the prior (mcmc.py:171).          */
int rv_loglik_d_dd_opt(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, const double* theta, int64_t W,
                       int check_prior, double* logp, double* grad, double* hess, int32_t* status);
/* Same with DEVICE buffers, asynchronous on `stream`. */
int rv_loglik_d_dd_dev(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, const double* d_theta, int64_t W,
                       double* d_logp, double* d_grad, double* d_hess, int32_t* d_status, void* stream);

/* ---- maximum-likelihood fit from W starts (no reference counterpart; DESIGN.md 3.6) ------------------------------- */
/* theta[W][nvars]: starts in, optima out.  Per walker, damped saddle-free Newton: the eigen-decomposition of -H gives
 * d = Q diag(1/lam~) Q^T g with lam~ = max(|lam|, 1e-12 lam_max) + mu lam_max; the walker stops when the Newton decrement
 * g^T d (mu = 0) halved is <= tol.  Otherwise n_trial rows theta + 2^-j d (j < n_trial) and theta itself are evaluated by
 * the plain likelihood in one launch; the best row with status RV_OK is taken if its logp exceeds theta's (damping
 * mu /= 10, 0 below 1e-6), else mu = max(10 mu, 1e-6) and the walker retries from the same point (RV_FIT_STALLED once
 * mu > 1).  damping0 is every walker's starting mu.  Derivatives come from the variational path with the hard prior
 * tested (as rv_smala_run).  Out: logp[W], status[W], grad[W][nvars] and hess[W][nvars][nvars] (optional, NULL to skip)
 * at the returned theta -- -inv(hess) is the Laplace covariance -- fit_code[W] (RV_FIT_*) and n_iter[W] (accepted
 * steps).  A walker's results depend on its start only, not on W or its position.  n_trial 1..16, max_iter >= 0
 * (0: the evaluation at the start), tol >= 0, damping0 >= 0; -30 / -31 as rv_loglik_d_dd.                          */
int rv_map_fit(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* theta, int64_t W, int max_iter, int n_trial,
               double tol, double damping0, double* logp, double* grad, double* hess, int32_t* status, int32_t* fit_code,
               int32_t* n_iter);

/* ---- Mh.step (mcmc.py:107-121) for W independent chains, nsteps steps, device-resident ---------- */
/* theta[W][nvars], logp[W]: start state in, final state out (have_logp = 0: logp is computed first, as
 * Mh.step's state.get_logp).  Proposal = theta + step_size*scales*z (mcmc.py:89-93); a proposal that fails
 * priorHard or raises Encounter is rejected (mcmc.py:112,119).  RNG: Philox-4x32-10 keyed by
 * (seed, first_chain_id + w, first_step + s) -- independent of sharding.  Optional outputs (NULL to skip):
 * chain[nsteps/thin][W][nvars] and chain_logp[nsteps/thin][W] (state after every thin-th step),
 * n_accept[W], accepted[nsteps][W].                                                                     */
int rv_mh_run(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* theta, double* logp, int have_logp,
              const double* scales, double step_size, uint64_t seed, uint64_t first_chain_id, uint32_t first_step,
              int nsteps, int thin, int64_t W, double* chain, double* chain_logp, uint64_t* n_accept,
              uint8_t* accepted);

/* ---- Ensemble.step (mcmc.py:57-65): emcee-2.2.1 affine stretch move, W walkers (even), nsteps steps ---- */
/* Each step = two half-steps (first half against the second, then the reverse).  lnp[W] as logp above.
 * walker ids for the RNG are the ensemble indices 0..W-1.  Same optional outputs as rv_mh_run.          */
int rv_stretch_run(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* theta, double* lnp, int have_lnp,
                   double a, uint64_t seed, uint32_t first_step, int nsteps, int thin, int64_t W, double* chain,
                   double* chain_lnp, uint64_t* n_accept, uint8_t* accepted);

/* One half-step on DEVICE buffers for walker shards (multi-GPU): updates d_S[nS] (global ids id0_S..) in place
 * against the complementary half d_C[nC]; the caller all-gathers the updated half afterwards.             */
int rv_stretch_half_dev(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* d_S, int64_t nS,
                        uint64_t id0_S, const double* d_C, int64_t nC, double* d_lnp_S, double a, uint64_t seed,
                        uint32_t step, uint32_t half, uint64_t* d_n_accept, uint8_t* d_accepted, void* stream);

/* The same ensemble over several GPUs of ONE process (one rv_ctx / rv_model / rv_obs per GPU, same schema and data on each):
 * every GPU keeps a full copy of the ensemble and owns one slice of each half; a slice's accept kernel stores its accepted
 * walkers into every copy through peer-mapped pointers (NVLink P2P), events order the half-steps across devices -- there
 * is no separate exchange step and no host synchronisation inside the loop.  W/2 must be a multiple of n_gpus; all pairs of
 * GPUs need peer access (-40 otherwise).  Results are bit-identical to rv_stretch_run for every n_gpus (random numbers are
 * keyed by the ensemble index).  Reference semantics: Ensemble.step, mcmc.py:57-65.                                   */
int rv_stretch_run_multi(int n_gpus, rv_ctx* const* ctxs, const rv_model* const* models, const rv_obs* const* obss,
                         double* theta, double* lnp, int have_lnp, double a, uint64_t seed, uint32_t first_step, int nsteps,
                         int thin, int64_t W, double* chain, double* chain_lnp, uint64_t* n_accept);


/* nsteps MH steps on DEVICE buffers (chains sharded over GPUs need no exchange). */
int rv_mh_steps_dev(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* d_theta, double* d_logp,
                    const double* d_scales, double step_size, uint64_t seed, uint64_t first_chain_id,
                    uint32_t first_step, int nsteps, int64_t W, uint64_t* d_n_accept, void* stream);

/* ---- Smala.step (mcmc.py:167-187) for W independent chains, nsteps steps, device-resident ---------------------- */
/* theta[W][nvars]: start state in, final state out; logp[W] out.  Per step and chain: SoftAbs metric of the Hessian
 * (mcmc.py:135-139, alpha), proposal theta* = mu + eps*chol(Ginv) z (mcmc.py:144-153), one value+gradient+Hessian
 * evaluation at theta*, accept iff exp(logp* - logp + q(theta|theta*) - q(theta*|theta)) > u.  A proposal outside the hard
 * prior or raising Encounter is rejected (mcmc.py:171,176).  Where the reference quits on LinAlgError (mcmc.py:179-183)
 * the step is rejected and status[w] is set to RV_NOT_SPD (status[w] is otherwise the status of the start state).
 * RNG and optional outputs as rv_mh_run.                                                                              */
int rv_smala_run(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* theta, double* logp, double eps,
                 double alpha, uint64_t seed, uint64_t first_chain_id, uint32_t first_step, int nsteps, int thin, int64_t W,
                 double* chain, double* chain_logp, uint64_t* n_accept, uint8_t* accepted, int32_t* status);

/* ---- Alsmala (mcmc.py:191-234) driven by run_alsmala's schedule (driver.py:171-200) ---------------------------------- */
/* Iteration i (= first_step + k) is a full SMALA step with probability exp(-bern_a * i / niter_total) (driver.py:181), else
 * Alsmala.step_mala: proposal and both transition densities from the STALE gradient / Hessian of the last full step
 * (mcmc.py:195-212), one plain likelihood evaluation.  The schedule draw is one per iteration, shared by all chains.
 * full_step[nsteps] (optional) records which iterations were full steps.  Other arguments as rv_smala_run.           */
int rv_alsmala_run(rv_ctx* ctx, const rv_model* model, const rv_obs* obs, double* theta, double* logp, double eps,
                   double alpha, double bern_a, int64_t niter_total, uint64_t seed, uint64_t first_chain_id,
                   uint32_t first_step, int nsteps, int thin, int64_t W, double* chain, double* chain_logp,
                   uint64_t* n_accept, uint8_t* accepted, int32_t* status, uint8_t* full_step);

/* ---- device buffers for callers without a GPU array library (single-process multi-GPU: multigpu.DeviceGroup) ---- */
/* Plain device allocations on the context's GPU and synchronous copies; rv_dev_copy_peer copies between two contexts'
 * GPUs (cudaMemcpyPeer: NVLink peer-to-peer where the driver allows it, staged through the host otherwise).       */
int rv_dev_alloc(rv_ctx* ctx, int64_t nbytes, void** out);
int rv_dev_free(rv_ctx* ctx, void* p);
int rv_dev_upload(rv_ctx* ctx, void* dst_dev, const void* src_host, int64_t nbytes);
int rv_dev_download(rv_ctx* ctx, void* dst_host, const void* src_dev, int64_t nbytes);
int rv_dev_copy_peer(rv_ctx* dst_ctx, void* dst_dev, rv_ctx* src_ctx, const void* src_dev, int64_t nbytes);

/* ---- work accounting: force evaluations and IAS15 step attempts since the last reset ----------- */
int rv_work_counters(rv_ctx* ctx, uint64_t out[2], int reset);
int rv_count_work(rv_ctx* ctx, int enable);     /* off by default (atomics per item when on)       */

/* ---- FP64 FMA-pipe peak of this GPU (TFLOP/s), the roofline denominator ------------------------ */
int rv_fp64_peak(rv_ctx* ctx, double* tflops);

int rv_sync(rv_ctx* ctx);
void* rv_ctx_stream(rv_ctx* ctx);   /* the context's cudaStream_t */

#ifdef __cplusplus
}
#endif
#endif /* RVGPU_H */
