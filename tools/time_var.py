#!/usr/bin/env python3
"""Throughput of the variational kernel (value + gradient + Hessian) on the HD155358 ball.
Usage: python tools/time_var.py [walkers ...]"""
import json
import os
import sys
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import rvtest as T
from rvel_mcmc_b200 import _abi

ctx = _abi.Context(0)
obs = T.load_vels("HD155358.vels")
oh = _abi.ObsHandle(ctx, obs.tf, obs.rvf, obs.errorf, obs.tb, obs.rvb, obs.errorb, obs.Npoints)
m = _abi.ModelHandle(ctx, np.zeros((2, 7)), T.FP10, T.FE10, 2.0)
sizes = [int(x) for x in sys.argv[1:]] or [222, 1776, 3552]
s = torch.cuda.current_stream().cuda_stream
for W in sizes:
    theta = torch.from_numpy(T.gaussian_ball(T.HD_SOL, T.HD_SCALE_VEC, W, 1)).cuda()
    lp = torch.empty(W, dtype=torch.float64, device="cuda"); st = torch.empty(W, dtype=torch.int32, device="cuda")
    g = torch.empty((W, 10), dtype=torch.float64, device="cuda"); h = torch.empty((W, 10, 10), dtype=torch.float64, device="cuda")
    m.loglik_d_dd_dev(oh, theta.data_ptr(), min(W, 64), lp.data_ptr(), g.data_ptr(), h.data_ptr(), st.data_ptr(), s)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); m.loglik_d_dd_dev(oh, theta.data_ptr(), W, lp.data_ptr(), g.data_ptr(), h.data_ptr(), st.data_ptr(), s); e1.record()
        torch.cuda.synchronize(); best = min(best, e0.elapsed_time(e1))
    ok = float((st.cpu().numpy() == 0).mean())
    print(json.dumps({"walkers": W, "ms": best, "var_evals_per_s": W / best * 1e3, "ok": ok}), flush=True)
