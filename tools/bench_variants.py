#!/usr/bin/env python3
"""Times tuning variants of the plain log-likelihood kernel (model option "mapping" >= 10, see rv_kernels.cu)
on the bench workload (HD155358 ball, 65536 walkers).  Usage: python tools/bench_variants.py 0 1 10 11 ...
0: default (4 CTAs x 128 threads), 1: thread per walker, 10: IAS15 tables from the constant bank, 11: 3 CTAs x 128 threads,
12: 4 x 128 with the constant-bank tables, 13: 2 CTAs x 256 threads."""
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
W = int(os.environ.get("WALKERS", "65536"))
theta = torch.from_numpy(T.gaussian_ball(T.HD_SOL, T.HD_SCALE_VEC, W, 1001)).cuda()
logp = torch.empty(W, dtype=torch.float64, device="cuda"); st = torch.empty(W, dtype=torch.int32, device="cuda")
s = torch.cuda.current_stream().cuda_stream
m.set_option("cost_order", int(os.environ.get("COST_ORDER", "1")))     # cost-ordered item schedule (default on)
ref = None
for mp in [int(x) for x in sys.argv[1:]] or [0]:
    m.set_option("mapping", mp)
    try:
        m.loglik_dev(oh, theta.data_ptr(), W, logp.data_ptr(), st.data_ptr(), s); torch.cuda.synchronize()
    except Exception as e:
        print("mapping %d: %s" % (mp, e)); continue
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); m.loglik_dev(oh, theta.data_ptr(), W, logp.data_ptr(), st.data_ptr(), s); e1.record()
        torch.cuda.synchronize(); best = min(best, e0.elapsed_time(e1))
    lp = logp.cpu().numpy()
    if ref is None: ref = lp.copy()
    print("mapping %2d: %.2f ms  %.3f Mevals/s  max|dlogp vs first|=%.2e" % (mp, best, W / best / 1e3, np.abs(lp - ref).max()), flush=True)

# non-default epoch handling: monotone backward sweep, dense output
for key in ("monotone_backward", "dense_output"):
    m.set_option("mapping", 0); m.set_option(key, 1)
    m.loglik_dev(oh, theta.data_ptr(), W, logp.data_ptr(), st.data_ptr(), s); torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); m.loglik_dev(oh, theta.data_ptr(), W, logp.data_ptr(), st.data_ptr(), s); e1.record()
        torch.cuda.synchronize(); best = min(best, e0.elapsed_time(e1))
    lp = logp.cpu().numpy()
    print("%s=1: %.2f ms  %.3f Mevals/s  max|dlogp vs default|=%.2e" % (key, best, W / best / 1e3, np.abs(lp - ref).max() if ref is not None else -1))
    m.set_option(key, 0)

# optional WHFast variant, dt = P_inner/20 (BASELINE configs[4])
m.set_option("mapping", 0)
for dt_div in (20, 50):
    m.set_option("dt0", 2 * np.pi * 0.65773033 ** 1.5 / dt_div); m.set_option("integrator", 1)
    m.loglik_dev(oh, theta.data_ptr(), W, logp.data_ptr(), st.data_ptr(), s); torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); m.loglik_dev(oh, theta.data_ptr(), W, logp.data_ptr(), st.data_ptr(), s); e1.record()
        torch.cuda.synchronize(); best = min(best, e0.elapsed_time(e1))
    lp = logp.cpu().numpy()
    print("WHFast dt=P_inner/%d: %.2f ms  %.3f Mevals/s  max|dlogp vs IAS15|=%.2e" % (dt_div, best, W / best / 1e3, np.abs(lp - ref).max() if ref is not None else -1))
m.set_option("integrator", 0); m.set_option("dt0", 1e-3)
