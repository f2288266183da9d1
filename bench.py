#!/usr/bin/env python3
"""bench.py -- headline benchmark of the hot path (BASELINE.json: RV log-lik evals/sec & ESS/sec, HD155358 2-planet).

One "step" = one pass of the hot path over one batch of synthetic walkers: the log-likelihood
(State.get_logp, state.py:103) of `--walkers` parameter vectors per GPU drawn as the reference's ensemble
start ball (mcmc.py:49-51) around the published HD155358 solution, on the real HD155358.vels epochs
(122 epochs, Npoints=100, hillRadiusFactor=2).  Weak scaling: every rank owns its own walker shard, no
data-path collective in the headline loop.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--walkers 65536] [--impl reference]
                  [--no-ess] [--no-var] [--no-sharded] [--ess-rows 2000] [--quick] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `value` = evaluations/s with inputs resident in HBM (CUDA events on the
launching stream, max over ranks); `e2e` = the same through the host-buffer C-ABI call rv_loglik (pinned
host memory, H2D + D2H inside the timed region).  Beside the headline the line carries
  * `ess`             ESS/s of the stretch / MH / SMALA device samplers from a committed EQUILIBRATED ensemble
                      (tests/golden/hd155358_equilibrated_ensemble.npy), >= 2000 recorded rows, reference AC time
                      (driver.py:366-377) and Sokal's integrated time; at N > 1 every rank runs its own chains /
                      ensemble replica and the aggregate is sum(ESS) / max(seconds);
  * `var`             value + gradient + Hessian evaluations/s (State.get_logp_d_dd) and that kernel's roofline;
  * `stretch_sharded` (N > 1) the affine ensemble sharded over the ranks with the per-half-step NCCL all-gather:
                      weak (56 832 walkers per GPU) and strong (65 536 walkers in total) evals/s, CUDA-event split
                      kernel / all-gather, host share, bit-identity against the single-GPU ensemble.
`--impl reference` times the reference's CPU path: the oracle port of rebound's algorithm (oracle/, OpenMP over
all host cores) on a bounded sample.
`--dump-outputs DIR` writes what the timed path returned for its last timed step (rank 0's walkers) as DIR/logp.npy and
DIR/status.npy (float64; logp is -inf where status != 0).  The walkers of every step come from fixed seeds, so two builds
run with the same arguments can be compared output for output.  Above DUMP_SAMPLE walkers a fixed seeded sample of them is
written, with their indices in DIR/walker_index.npy.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "rv_loglik_evals_per_sec_hd155358_2planet"
UNIT = "evals/s"
HD_SOL = [6.57730330e-01, -9.72263877e-02, -7.82798396e-02, 8.84031737e-04, 4.42804990e+00,
          1.04404207e+00, -2.05622789e-02, -1.08797961e-01, 8.30379710e-04, 1.49919861e+00]
HD_SCALES = {"m": 5.5e-6, "a": 0.001, "h": 0.02, "k": 0.02, "l": np.pi / 4}
FP10 = [0, 0, 0, 0, 0, 1, 1, 1, 1, 1]
FE10 = [1, 2, 3, 0, 4, 1, 2, 3, 0, 4]
EQUILIBRATED = os.path.join(ROOT, "tests", "golden", "hd155358_equilibrated_ensemble.npy")
ROOFLINE_INPUTS = os.path.join(ROOT, "profiles", "roofline_inputs.json")     # ncu-derived figures, one file, committed
DUMP_SAMPLE = 1 << 21         # --dump-outputs: at most this many walkers, 48 MB with their indices


def walker_ball(W, seed):
    rng = np.random.RandomState(seed)
    sc = np.array([HD_SCALES[k] for k in ("a", "h", "k", "m", "l")] * 2)
    return np.asarray(HD_SOL)[None, :] + 1e-3 * sc[None, :] * rng.normal(size=(W, 10))


def load_obs():
    from rvel_mcmc_b200 import observations
    return observations.Observation_FromFile(os.path.join(ROOT, "tests", "golden", "HD155358.vels"), Npoints=100)


def flops_per_eval(S, T):
    """SURVEY 8(d): W_eval = S*[3N*36 + N(N-1)*18] + T*3N*150 with N = 3 bodies."""
    return S * (9 * 36 + 6 * 18) + T * 9 * 150


def var_flops_per_eval(S, T, nv=10, N=3):
    """SURVEY 8(d), variational evaluation: per force evaluation 3*(30 + nv*45 + nv(nv+1)/2*140) gravity flops plus 36 per
    coordinate of the (1 + nv + nv(nv+1)/2) sets of N bodies; per step attempt 150 per coordinate."""
    n2 = nv * (nv + 1) // 2
    coords = 3 * N * (1 + nv + n2)
    return S * (3 * (30 + nv * 45 + n2 * 140) + coords * 36) + T * coords * 150


_STDOUT_FD = None


def quiet_stdout():
    """stdout carries exactly ONE JSON line (the driver parses it): from here on everything any library writes to file
    descriptor 1 (the NCCL version banner, NCCL_DEBUG output, warnings printed from native code) goes to stderr instead."""
    global _STDOUT_FD
    if _STDOUT_FD is None:
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def emit_line(line):
    data = (json.dumps(line) + "\n").encode()
    if _STDOUT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_STDOUT_FD, data)


def dump_outputs(out_dir, logp, status):
    """--dump-outputs: one step's per-walker results as float64 .npy files; a fixed seeded sample above DUMP_SAMPLE walkers."""
    arrays = {"logp": np.asarray(logp, dtype=np.float64), "status": np.asarray(status, dtype=np.float64)}
    n = len(arrays["logp"])
    if n > DUMP_SAMPLE:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))
        arrays = {k: v[idx] for k, v in arrays.items()}
        arrays["walker_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


def roofline_inputs():
    """Figures that only a profiler can give (DRAM traffic per launch, FP64-pipe utilisation): read from ONE committed
    file that names the ncu summary each comes from -- never typed into this script."""
    try:
        with open(ROOFLINE_INPUTS) as f:
            return json.load(f)
    except Exception:
        return {}


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.samples = []
        self.reasons = set()
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def oracle_batch(obs, theta, nthreads):
    import rvtest as T
    o = T.Obs()
    o.tf, o.tb, o.rvf, o.rvb, o.errorf, o.errorb, o.Npoints = obs.tf, obs.tb, obs.rvf, obs.rvb, obs.errorf, obs.errorb, obs.Npoints
    t0 = time.perf_counter()
    logp, st, cnt = T.orc_logp_batch(np.zeros((2, 7)), FP10, FE10, 2.0, o, theta, nthreads=nthreads, lib=T.oracle_fast())
    return time.perf_counter() - t0, logp, st, cnt


# ---------------------------------------------------------------------------------------------------------------
# ESS/s (BASELINE metric, second half): the three device samplers from an equilibrated start

def run_ess(ctx, model, oh, rank, world, dist, dev, rows, torch, budgets=(150.0, 80.0, 130.0)):
    from rvel_mcmc_b200.samplers import ess
    from rvel_mcmc_b200 import driver
    if not os.path.exists(EQUILIBRATED):
        return {"unavailable": "tests/golden/hd155358_equilibrated_ensemble.npy is missing (tools/make_equilibrated_ensemble.py)"}
    eq = np.load(EQUILIBRATED)
    post_std = eq.std(axis=0)
    slots = ctx.device_info()["sm_count"] * 3 * 64          # resident (walker, leg) lane groups of loglik_kernel
    out = {"start": "committed equilibrated stretch ensemble (%d walkers; tools/make_equilibrated_ensemble.py); nothing inside the "
                    "clocks is burn-in" % len(eq),
           "definition": "ESS = recorded rows x walkers / max_i tau_i; tau_int = Sokal's windowed integrated autocorrelation "
                         "time of the walker-averaged autocovariance (256 walkers), ac_time_ref = driver.py:366-377 (first lag with "
                         "autocorrelation < 0.5; mean over 16 walkers, as driver.py:355-370 does for ensembles); seconds = "
                         "wall time of the whole library call (chain download included)",
           "aggregate": "sum over ranks of ESS / max over ranks of seconds; every rank runs its own chains (MH, SMALA: "
                        "global chain ids) or its own ensemble replica (stretch: rank-specific seed)"}

    REC = 512          # walkers whose positions are recorded (context option chain_walkers): the autocorrelation estimate
                       # needs a sample of the chains, not a host copy of every position

    def summarise(name, chain, walkers, seconds, evals, extra):
        _, tau = ess(chain)
        n_eff = chain.shape[0] * walkers / max(tau, 1.0)
        ac_ref = max(float(np.mean([driver.ac_time(chain[:, w, i]) for w in range(min(16, chain.shape[1]))]))
                     for i in range(chain.shape[2]))
        vals = [float(n_eff), float(seconds), float(evals)]
        if world > 1:
            t = torch.tensor(vals, dtype=torch.float64, device=dev)
            s = t.clone(); dist.all_reduce(s, op=dist.ReduceOp.SUM)
            m = t.clone(); dist.all_reduce(m, op=dist.ReduceOp.MAX)
            n_eff_tot, sec, ev = float(s[0]), float(m[1]), float(s[2])
        else:
            n_eff_tot, sec, ev = vals
        d = {"walkers_per_gpu": int(walkers), "recorded_walkers": int(chain.shape[1]), "recorded_rows": int(chain.shape[0]),
             "seconds": sec, "evals_per_s": ev / sec, "tau_int_max_rows": tau, "ac_time_ref_max_rows": ac_ref,
             "ess_per_s": n_eff_tot / sec, "ess_per_s_ref_definition": n_eff_tot * max(tau, 1.0) / max(ac_ref, 1.0) / sec}
        d.update(extra)
        out[name] = d

    def sized(name, budget_s, pilot, nsteps_pilot):
        """Recorded rows for one sampler: `rows` unless the time budget says fewer (pilot = seconds of a short run)."""
        per_step = pilot / nsteps_pilot
        n = int(min(rows, max(50, budget_s / max(per_step, 1e-6))))
        out.setdefault("time_budget", {})[name] = {"budget_s": budget_s, "pilot_ms_per_step": 1e3 * per_step, "rows": n,
                                                   "rows_limited_by_time_budget": bool(n < rows)}
        return n

    # The ensemble is sized to keep the machine full THROUGH the long tail of the posterior's expensive walkers: four waves
    # of (walker, leg) items per half-step.  It is built from four copies of the committed equilibrated ensemble,
    # decorrelated by an UNTIMED burn-in of `mix` stretch steps (every walker is still a draw from the stationary
    # distribution; the copies separate at their first accepted move).
    copies, mix = 4, 60
    W = min(copies * len(eq), copies * slots) & ~1
    start = np.concatenate([eq] * copies)[:W]
    start = np.ascontiguousarray(start.reshape(copies, -1, 10).transpose(1, 0, 2).reshape(-1, 10))   # interleave the copies
    t0 = time.perf_counter()
    r = model.stretch_run(oh, start, mix, seed=7 + 1000 * rank, record_chain=False)
    pilot = time.perf_counter() - t0
    start, lnp0 = r["theta"], r["lnp"]
    out["ensemble"] = {"walkers_per_gpu": int(W), "copies_of_committed_ensemble": copies, "untimed_burn_in_steps": mix,
                       "burn_in_seconds": pilot, "burn_in_accept_rate": float(r["n_accept"].mean() / mix)}
    # affine stretch
    n = sized("stretch", budgets[0], pilot, mix)
    t0 = time.perf_counter()
    r = model.stretch_run(oh, start, n, seed=11 + 1000 * rank, first_step=mix, lnp=lnp0, thin=1, chain_walkers=REC)
    summarise("stretch", r["chain"], W, time.perf_counter() - t0, W * n,
              {"accept_rate": float(r["n_accept"].mean() / n), "a": 2.0})
    del r
    # Metropolis-Hastings: proposal scale 0.25 x the posterior standard deviations; chains start from the same walkers
    Wm = W // 2
    t0 = time.perf_counter()
    model.mh_run(oh, start[:Wm], post_std, 0.25, 10, seed=1, record_chain=False)
    n = sized("mh", budgets[1], time.perf_counter() - t0, 10)
    t0 = time.perf_counter()
    r = model.mh_run(oh, start[:Wm], post_std, 0.25, n, seed=12, first_chain_id=rank * Wm, logp=lnp0[:Wm], thin=1, chain_walkers=REC)
    summarise("mh", r["chain"], Wm, time.perf_counter() - t0, Wm * n,
              {"accept_rate": float(r["n_accept"].mean() / n), "step_size": 0.25, "scales": "posterior std"})
    del r
    # SMALA with the reference's step size and SoftAbs constant ((Ex)HD155358.ipynb:640): two waves of warp groups
    # (4 walker legs per SM resident in var2_kernel)
    Ws = ctx.device_info()["sm_count"] * 4
    t0 = time.perf_counter()
    model.smala_run(oh, start[:Ws], 0.025, 1.4, 5, seed=1, record_chain=False)
    n = sized("smala", budgets[2], time.perf_counter() - t0, 6)
    t0 = time.perf_counter()
    r = model.smala_run(oh, start[:Ws], 0.025, 1.4, n, seed=13, first_chain_id=rank * Ws, thin=1, chain_walkers=REC)
    summarise("smala", r["chain"], Ws, time.perf_counter() - t0, Ws * (n + 1),
              {"accept_rate": float(r["n_accept"].mean() / n), "eps": 0.025, "alpha": 1.4,
               "not_spd_flags": int((r["status"] == 9).sum())})
    ctx.set_option("chain_walkers", 0)
    return out


# ---------------------------------------------------------------------------------------------------------------
# value + gradient + Hessian (State.get_logp_d_dd): var_kernel throughput and roofline

def run_var(ctx, model, oh, dev, peak, torch):
    W = ctx.device_info()["sm_count"] * 2 * 8              # eight waves of warp groups (4 walker legs per SM resident)
    th = torch.from_numpy(walker_ball(W, 4242)).to(dev)
    lp = torch.empty(W, dtype=torch.float64, device=dev); st = torch.empty(W, dtype=torch.int32, device=dev)
    g = torch.empty((W, 10), dtype=torch.float64, device=dev); h = torch.empty((W, 10, 10), dtype=torch.float64, device=dev)
    s = torch.cuda.current_stream().cuda_stream

    def call():
        model.loglik_d_dd_dev(oh, th.data_ptr(), W, lp.data_ptr(), g.data_ptr(), h.data_ptr(), st.data_ptr(), s)
    call(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); call(); e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    ctx.count_work(True); ctx.work_counters(reset=True)
    call(); torch.cuda.synchronize()
    S, T_ = ctx.work_counters(reset=True)
    ctx.count_work(False)
    S, T_ = S / W, T_ / W
    fl = var_flops_per_eval(S, T_)
    achieved = fl * W / (ms * 1e-3) / 1e12
    prof = roofline_inputs().get("var_kernel", {})
    return {"value": W / (ms * 1e-3), "unit": "value+gradient+Hessian evals/s per GPU", "walkers": W, "ms": ms,
            "ok_fraction": float((st == 0).float().mean().item()),
            "roofline": {"bound": "fp64_fma_pipe", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "note": "SURVEY 8(d) algorithmic flops of the variational evaluation (S=%.0f force evaluations, T=%.0f "
                                 "step attempts per eval, real-only step-size norm) / CUDA-event time" % (S, T_),
                         "from_profile": prof},
            "reference": "0.58 tries/s (rebound + Python 2, one 2017 core; (Ex)HD155358.ipynb:628-640) -- context only"}


# ---------------------------------------------------------------------------------------------------------------
# N > 1: the affine ensemble sharded over the ranks, all-gather of the updated half after every half-step

def run_stretch_sharded(ctx, model, oh, rank, world, dist, dev, torch, nsteps):
    from rvel_mcmc_b200.samplers import ShardedStretch
    stream = torch.cuda.current_stream(dev).cuda_stream
    out = {"exchange": "torch.distributed all_gather_into_tensor (NCCL) of the updated half-ensemble's positions after every "
                       "half-step; random numbers keyed by ensemble index, nothing else crosses ranks"}
    slots = ctx.device_info()["sm_count"] * 3 * 64

    def one(W, label):
        theta0 = walker_ball(W, 5)
        theta = torch.from_numpy(theta0).to(dev)
        h, n_loc = W // 2, (W // 2) // world
        lnp = torch.empty(2 * n_loc, dtype=torch.float64, device=dev)
        stl = torch.empty(2 * n_loc, dtype=torch.int32, device=dev)
        for half in (0, 1):
            lo = half * h + rank * n_loc
            model.loglik_dev(oh, theta[lo:lo + n_loc].data_ptr(), n_loc, lnp[half * n_loc:].data_ptr(), stl[half * n_loc:].data_ptr(), stream)
        lnp[stl != 0] = float("-inf")
        send = torch.empty((n_loc, 10), dtype=torch.float64, device=dev)

        def half_step(k, half, ev=None):
            lo = half * h + rank * n_loc
            S = theta[lo:lo + n_loc]
            C = theta[h:] if half == 0 else theta[:h]
            if ev: ev[0].record()
            model.stretch_half_dev(oh, S.data_ptr(), n_loc, lo, C.data_ptr(), h, lnp[half * n_loc:].data_ptr(), 2.0, 5, k, half,
                                   stream=stream)
            if ev: ev[1].record()
            send.copy_(S)
            dist.all_gather_into_tensor(theta[half * h:(half + 1) * h], send)
            if ev: ev[2].record()
        half_step(0, 0); half_step(0, 1)                       # warm-up (NCCL channels, scratch growth)
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(2 * nsteps)]
        t0 = time.perf_counter()
        for k in range(nsteps):
            for half in (0, 1):
                half_step(1 + k, half, evs[2 * k + half])
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        kern = float(np.mean([e[0].elapsed_time(e[1]) for e in evs]))
        gath = float(np.mean([e[1].elapsed_time(e[2]) for e in evs]))
        t = torch.tensor([wall, kern, gath], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall, kern, gath = [float(x) for x in t]
        per_half = 1e3 * wall / (2 * nsteps)
        d = {"walkers_total": W, "walkers_per_gpu": W // world, "ensemble_steps": nsteps,
             "evals_per_s": W * nsteps / wall, "ms_per_half_step": per_half, "kernel_ms_per_half_step": kern,
             "allgather_ms_per_half_step": gath, "host_and_idle_ms_per_half_step": max(0.0, per_half - kern - gath),
             "allgather_bytes_per_half_step": h * 10 * 8,
             "items_per_gpu_per_half_step": 2 * n_loc, "resident_item_slots_per_gpu": slots}
        d["limiter"] = ("kernel: one half-step cannot be shorter than the serial IAS15 integration of its longest leg (~5 ms for "
                        "HD155358's 1244-step backward leg); %d items for %d resident slots per GPU"
                        % (2 * n_loc, slots)) if kern > 4 * gath else "exchange"
        out[label] = d
        return theta, lnp, theta0

    W_weak = 2 * slots * world                                  # two full waves of items per half-step and GPU
    one(W_weak, "weak")
    W_strong = 65536
    theta, lnp, theta0 = one(W_strong, "strong")
    # bit-identity: rank 0 repeats the strong-scaled ensemble on its own GPU (same seed, same steps: 1 warm-up + nsteps)
    if rank == 0:
        r = model.stretch_run(oh, theta0, nsteps + 1, seed=5, record_chain=False)
        out["bit_identical_to_single_gpu"] = bool(np.array_equal(r["theta"], theta.cpu().numpy()))
        t0 = time.perf_counter()
        model.stretch_run(oh, theta0, nsteps, seed=5, record_chain=False)
        one_gpu = W_strong * (nsteps + 1) / (time.perf_counter() - t0)
        out["strong"]["single_gpu_evals_per_s"] = one_gpu
        out["strong"]["speedup_vs_single_gpu"] = out["strong"]["evals_per_s"] / one_gpu
    dist.barrier()
    return out


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; rebound itself is not installable here)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    obs = load_obs()
    cores = os.cpu_count() or 1
    sample = 4096                      # ~2 s of work per step on 16 cores
    theta = walker_ball(sample, 1234)
    for _ in range(min(args.warmup, 1)):
        oracle_batch(obs, theta[: cores * 4], cores)
    times = []
    cnt = None
    for k in range(args.steps):
        dt, logp, status, cnt = oracle_batch(obs, walker_ball(sample, 1234 + k), cores)
        times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, logp, status)
    tot = float(np.sum(times))
    value = sample * args.steps / tot
    line = {"metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic walkers on HD155358.vels epochs",
            "config": {"workload": "HD155358 2-planet log-likelihood, %d-walker sample per step (bounded CPU sample)" % sample,
                       "walkers_per_step": sample, "epochs": 122},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d walkers x %d steps, oracle/rv_oracle.c (gcc -O3 -march=native, OpenMP, %d threads)" % (sample, args.steps, cores)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit_line(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--walkers", type=int, default=65536, help="walkers per GPU per step")
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--mapping", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=0, help="walkers in the timed CPU sample (0: about 15 s of work)")
    ap.add_argument("--no-ess", action="store_true", help="skip the ESS/s block (three sampler runs, ~2 min)")
    ap.add_argument("--ess", action="store_true", help="(default on; kept for compatibility)")
    ap.add_argument("--ess-rows", type=int, default=2000, help="recorded rows (= sampler steps) per ESS run (fewer if the "
                                                               "per-sampler time budget says so; the line reports it)")
    ap.add_argument("--ess-budget", default=None, help="seconds for the stretch, MH and SMALA ESS runs (default 150,80,130 on "
                                                       "one GPU; 90,50,80 at N > 1, where the driver's per-N limit is tighter)")
    ap.add_argument("--no-var", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="N > 1: skip the sharded stretch block")
    ap.add_argument("--sharded-steps", type=int, default=6)
    ap.add_argument("--quick", action="store_true", help="smoke-sized side blocks (200 ESS rows, no CPU baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write logp.npy and status.npy of the last timed step (rank 0's walkers) to DIR")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    quiet_stdout()
    if args.impl == "reference":
        run_reference(args)
        return
    if args.quick:
        args.ess_rows = min(args.ess_rows, 100)
        args.ess_budget = "5,3,5"
        args.no_cpu_baseline = True

    import torch
    import torch.distributed as dist
    from rvel_mcmc_b200 import _abi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if args.ess_budget is None:
        args.ess_budget = "150,80,130" if world == 1 else "90,50,80"
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    ctx = _abi.Context(local)
    obs = load_obs()
    oh = obs._handle(ctx)
    model = _abi.ModelHandle(ctx, np.zeros((2, 7)), FP10, FE10, 2.0)
    if args.mapping:
        model.set_option("mapping", args.mapping)
    W = args.walkers
    nsets = max(args.steps + args.warmup, 3)       # the CPU baseline below draws on sets 0, 1 and 2
    # a fresh batch of walkers for every step (global walker ids are disjoint across ranks)
    host_theta = [torch.from_numpy(walker_ball(W, 1000 * (rank + 1) + s)).pin_memory() for s in range(nsets)]
    d_theta = [t.to(dev, non_blocking=True) for t in host_theta]
    d_logp = torch.empty(W, dtype=torch.float64, device=dev)
    d_status = torch.empty(W, dtype=torch.int32, device=dev)
    h_logp = torch.empty(W, dtype=torch.float64).pin_memory()
    h_status = torch.empty(W, dtype=torch.int32).pin_memory()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
    tstream = torch.cuda.Stream(device=dev)      # the launching stream: kernels and timing events both go here
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    torch.cuda.synchronize()

    def step_dev(i):
        model.loglik_dev(oh, d_theta[i].data_ptr(), W, d_logp.data_ptr(), d_status.data_ptr(), stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing ---------------------------------------------------------------
    for i in range(args.warmup):
        step_dev(i)
    sampler = ClockSampler(local)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    sampler.start()
    for k in range(args.steps):
        flush.zero_()                        # L2 flush between timed iterations
        ev[k][0].record()
        step_dev(args.warmup + k)
        ev[k][1].record()
    barrier()
    ms = np.array([a.elapsed_time(b) for a, b in ev])
    total_ms = float(ms.sum())
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    st_np = d_status.cpu().numpy()
    ok_frac = float((st_np == 0).mean())
    last_logp = d_logp.cpu().numpy()               # the blocks below reuse d_logp / d_status

    # ---- end-to-end through the host-buffer C ABI (rv_loglik): pinned host memory in, results out ----
    lib = ctx.lib
    import ctypes as C

    def step_e2e(i):
        rc = lib.rv_loglik(ctx.h, model.h, oh.h, C.c_void_p(host_theta[i].data_ptr()), W,
                           C.c_void_p(h_logp.data_ptr()), C.c_void_p(h_status.data_ptr()))
        ctx.check(rc, "rv_loglik")
    step_e2e(0)
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        step_e2e(args.warmup + k)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())

    # keep the GPU under the same load until the clock sampler (nvidia-smi, ~0.3 s per query) has a few samples
    t_load = time.perf_counter()
    while len(sampler.samples) < 4 and time.perf_counter() - t_load < 5.0:
        step_dev(0)
        torch.cuda.synchronize()
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- side blocks that every rank takes part in --------------------------------------------------------------
    del flush
    torch.cuda.empty_cache()
    sharded = None
    if world > 1 and not args.no_sharded:
        sharded = run_stretch_sharded(ctx, model, oh, rank, world, dist, dev, torch, args.sharded_steps)
    ess_block = None
    if not args.no_ess:
        ess_block = run_ess(ctx, model, oh, rank, world, dist if world > 1 else None, dev, args.ess_rows, torch,
                            tuple(float(x) for x in args.ess_budget.split(",")))
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- roofline: algorithmic flops (SURVEY 8(d)) / kernel time vs the measured FP64 FMA peak -----------
    ctx.count_work(True)
    ctx.work_counters(reset=True)
    step_dev(0)
    torch.cuda.synchronize()
    S_gpu, T_gpu = ctx.work_counters(reset=True)
    ctx.count_work(False)
    S_eval, T_eval = S_gpu / W, T_gpu / W
    flops_eval = flops_per_eval(S_eval, T_eval)
    kernel_ms = float(ms.mean())             # loglik kernel + finalize (finalize is ~us)
    achieved = flops_eval * W / (kernel_ms * 1e-3) / 1e12
    peak = ctx.fp64_peak_tflops()
    prof = roofline_inputs()
    lk = prof.get("loglik_kernel", {})
    roofline = {"bound": "fp64_fma_pipe", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": lk.get("dram_bytes_per_launch"),
                "algorithmic_bytes_per_launch": W * 92,
                "from_profile": {"file": "profiles/roofline_inputs.json", "loglik_kernel": lk, "fp64_peak_record": prof.get("fp64_peak")},
                "executed_note": "frac uses SURVEY 8(d)'s ALGORITHMIC flop count (rebound's formulation); the kernel executes fewer "
                                 "FP64 instructions per decision (implicit star, coplanar, g-only corrector loop, no divisions), so frac can "
                                 "exceed the pipe's real occupancy: the ncu figure sm__pipe_fp64_cycles_active is from_profile.loglik_kernel",
                "note": "achieved = SURVEY 8(d) algorithmic flops (S=%.0f force evals, T=%.0f step attempts per eval, "
                        "432*S+1350*T) / CUDA-event kernel time; peak = dependent-free fma.rn.f64 microbenchmark run now on this GPU "
                        "(rv_fp64_peak; MEASURED_PEAKS.json has no FP64 entry)" % (S_eval, T_eval)}

    # ---- the same evaluations under the two non-default epoch-handling options (never the headline value) ----
    ref_logp = d_logp.clone()
    options = {}
    for key, note in (("monotone_backward", "backward leg visited 0 -> most negative epoch once (state.py:273 order) instead of "
                                            "state.py:91's stored order"),
                      ("dense_output", "one continuous IAS15 integration per leg with natural steps, RVs read from the step's "
                                       "acceleration polynomial instead of a truncated step per epoch")):
        model.set_option(key, 1)
        step_dev(0); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); step_dev(0); e1.record(); torch.cuda.synchronize()
        okm = (d_status == 0)
        options[key] = {"value": W / (e0.elapsed_time(e1) * 1e-3), "unit": UNIT + " per GPU", "ms_per_step": e0.elapsed_time(e1),
                        "max_abs_logp_diff_vs_default": float((d_logp[okm] - ref_logp[okm]).abs().max().item()),
                        "note": "model option %s=1: %s; NOT the headline value (the default keeps the reference's step "
                                "sequence)" % (key, note)}
        model.set_option(key, 0)
    step_dev(0); torch.cuda.synchronize()

    var_block = None
    if not args.no_var:
        var_block = run_var(ctx, model, oh, dev, peak, torch)

    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:        # a reported baseline: rank 0 at N = 1 only
        cores = os.cpu_count() or 1
        t_probe, _, _, _ = oracle_batch(obs, host_theta[1][:cores * 8].numpy(), cores)      # size the sample: ~15 s of CPU work
        sample = args.cpu_sample or int(min(W, max(cores * 32, 15.0 / max(t_probe, 1e-3) * cores * 8)))
        dt, lo, so, cnt = oracle_batch(obs, host_theta[0][:sample].numpy(), cores)
        # parity spot check on the same vectors
        step_dev(0)
        torch.cuda.synchronize()
        lg = d_logp[:sample].cpu().numpy(); sg = d_status[:sample].cpu().numpy()
        okm = (so == 0) & (sg == 0)
        n1 = 256
        dt1, _, _, _ = oracle_batch(obs, host_theta[2][:n1].numpy(), 1)                 # the same port on ONE core
        cpu_baseline = {"value": sample / dt, "unit": UNIT, "cores": cores, "kind": "port",
                        "single_core_value": n1 / dt1,
                        "historical_reference": "16.6 evals/s: rebound + emcee under Python 2 on an unknown 2017 CPU, one core, "
                                                "Encounter storms included ((Ex)HD155358.ipynb:181-456; BASELINE.md section 1) -- context only",
                        "sample": "%d walkers of step 0, oracle/rv_oracle.c (gcc -O3 -march=native) OpenMP %d threads, %.1f s" % (sample, cores, dt),
                        "oracle_S_per_eval": cnt[0] / sample, "oracle_T_per_eval": cnt[1] / sample,
                        "parity_max_abs_logp_diff": float(np.abs(lg[okm] - lo[okm]).max()) if okm.any() else None,
                        "parity_status_equal": bool(np.array_equal(so, sg))}

    n_total = W * world * args.steps
    line = {"metric": METRIC, "value": n_total / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic walkers (ensemble start ball) on HD155358.vels epochs",
            "config": {"workload": "HD155358.vels 2-planet log-likelihood (configs[1] shape), %d walkers per GPU per step" % W,
                       "walkers_per_gpu": W, "epochs": 122, "nvars": 10, "integrator": "ias15", "l2": "flushed between steps",
                       "mapping": "lane-per-planet" if args.mapping == 0 else "thread-per-walker", "ok_fraction": ok_frac},
            "e2e": {"value": n_total / e2e_s, "unit": UNIT, "h2d_bytes_per_step": W * 10 * 8, "d2h_bytes_per_step": W * 12},
            # per step: cost_bin / cost_scan / cost_scatter (item order, W >= 4096), loglik_kernel, finalize_kernel
            "gpu_launches": (5 if W >= 4096 else 2) * args.steps, "clocks": sampler.summary(), "roofline": roofline}
    line["non_default_options"] = options
    if cpu_baseline:
        line["cpu_baseline"] = cpu_baseline
    if ess_block is not None:
        line["ess"] = ess_block
    if var_block is not None:
        line["var"] = var_block
    if sharded is not None:
        line["stretch_sharded"] = sharded
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_logp, st_np)
    emit_line(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True                 # the benchmark leaves the tree as it found it (it may be read-only)
    main()
