#!/usr/bin/env python3
"""Throughput of the batched maximum-likelihood fit (rv_map_fit) on HD155358 (hill factor 2, default fit settings) from
balls HD_SOL + HD_SCALE_VEC * N(0,1) of 1, 64, 1 024, 4 096 and 16 384 starts: wall time and fits/s (host clock around the
synchronous call, after a warm-up fit), iterations per start, and -- in a second, profiled run of the same fit -- the
split of the wall time into the variational evaluations (var kernels + their finalize), the trial launches (plain
likelihood kernel, finalize, cost ordering), the fit's own kernels (map_*: gather / scatter / step / select +
compaction) and the rest (host loop, launch gaps, copies).  One JSON line per start count.
Usage: python tools/time_map.py [--out profiles/r04a_map_fit.jsonl] [--sizes 1,64,1024,4096,16384]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import rvtest as T  # noqa: E402
from rvel_mcmc_b200 import _abi  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return [s.strip() for s in q.split(",")]
    except Exception as e:          # the measurement itself does not depend on it
        return ["unknown: %s" % e]


def kernel_split(run):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run()
        torch.cuda.synchronize()
    split = dict(variational=0.0, trial=0.0, map_kernels=0.0, other_kernels=0.0)
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
        name = ev.name
        if "var" in name:
            split["variational"] += us
        elif "map_" in name:
            split["map_kernels"] += us
        elif "loglik" in name or "finalize" in name or "cost_" in name:
            split["trial"] += us
        else:
            split["other_kernels"] += us
    return {k: v * 1e-6 for k, v in split.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04a_map_fit.jsonl"))
    ap.add_argument("--sizes", default="1,64,1024,4096,16384")
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "time_map.py measures on a GPU"
    ctx = _abi.Context(0)
    obs = T.load_vels("HD155358.vels")
    oh = _abi.ObsHandle(ctx, obs.tf, obs.rvf, obs.errorf, obs.tb, obs.rvb, obs.errorb, obs.Npoints)
    m = _abi.ModelHandle(ctx, np.zeros((2, 7)), T.FP10, T.FE10, 2.0)
    info = gpu_info()
    rng = np.random.default_rng(0)
    m.map_fit(oh, np.array(T.HD_SOL)[None, :] + np.array(T.HD_SCALE_VEC)[None, :] * rng.normal(size=(64, 10)))   # warm-up
    lines = []
    for W in [int(s) for s in a.sizes.split(",")]:
        X = np.array(T.HD_SOL)[None, :] + np.array(T.HD_SCALE_VEC)[None, :] * np.random.default_rng(W).normal(size=(W, 10))
        t0 = time.perf_counter()
        r = m.map_fit(oh, X)
        wall = time.perf_counter() - t0
        split = kernel_split(lambda: m.map_fit(oh, X))
        it = r["n_iter"]
        codes = {str(c): int((r["fit_code"] == c).sum()) for c in np.unique(r["fit_code"])}
        rec = dict(tool="tools/time_map.py", gpu=info, problem="HD155358 hill 2, ball HD_SOL + HD_SCALE_VEC*N(0,1)",
                   settings=dict(max_iter=50, n_trial=8, tol=1e-10, damping=0.0), starts=W, wall_s=round(wall, 4),
                   fits_per_s=round(W / wall, 2), n_iter_mean=round(float(it.mean()), 2),
                   n_iter_p50=int(np.percentile(it, 50)), n_iter_p90=int(np.percentile(it, 90)), n_iter_max=int(it.max()),
                   fit_codes=codes, split_s={k: round(v, 4) for k, v in split.items()},
                   variational_share_of_kernel_time=round(split["variational"] / max(sum(split.values()), 1e-12), 4),
                   variational_share_of_wall=round(split["variational"] / wall, 4))
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
