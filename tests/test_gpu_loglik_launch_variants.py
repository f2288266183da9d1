"""The plain log-likelihood kernel's launch shapes compute the same bits: the headline instantiation (two planets, coplanar)
at its default shape and at the tuning shapes kept beside it (model option mapping >= 10, rv_kernels.cu) run one source,
so logp and status must be identical -- not merely close -- on the benchmark's start ball and on posterior walkers, with
and without the cost-ordered item schedule."""
import os

import numpy as np
import pytest

import rvtest as T

pytestmark = pytest.mark.gpu

# 11: 3 CTAs x 128 threads, 13: 2 CTAs x 256 threads (the default is 4 x 128)
VARIANTS = [11, 13]


@pytest.fixture(scope="module")
def setup():
    from rvel_mcmc_b200 import _abi
    ctx = _abi.Context(0)
    obs = T.load_vels("HD155358.vels")
    oh = _abi.ObsHandle(ctx, obs.tf, obs.rvf, obs.errorf, obs.tb, obs.rvb, obs.errorb, obs.Npoints)
    m = _abi.ModelHandle(ctx, np.zeros((2, 7)), T.FP10, T.FE10, 2.0)
    ball = T.gaussian_ball(T.HD_SOL, T.HD_SCALE_VEC, 65536, 1001)        # the bench workload's shape
    # a few walkers that end early: prior violations, a non-finite parameter and the reference's Encounter vectors
    ball[17, 3] = 1e-6; ball[18, 0] = 0.01; ball[19, 1] = np.nan
    ball[20:23] = np.array([k[0] for k in T.KAT5])
    ens = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hd155358_equilibrated_ensemble.npy"))
    yield m, oh, {"ball": ball, "posterior": ens}
    ctx.close()


@pytest.mark.parametrize("cost_order", [0, 1])
@pytest.mark.parametrize("walkers", ["ball", "posterior"])
def test_launch_variants_are_bit_identical(setup, walkers, cost_order):
    m, oh, sets = setup
    theta = sets[walkers]
    m.set_option("cost_order", cost_order)
    m.set_option("mapping", 0)
    l0, s0 = m.loglik(oh, theta)
    assert (s0 == 0).sum() > 0.9 * len(theta)
    if walkers == "ball":
        assert (s0 == 1).sum() >= 2 and (s0 == 3).sum() >= 3
    try:
        for mp in VARIANTS:
            m.set_option("mapping", mp)
            l1, s1 = m.loglik(oh, theta)
            assert np.array_equal(s0, s1), mp
            assert np.array_equal(l0, l1), (mp, np.nanmax(np.abs(l0 - l1)))
    finally:
        m.set_option("mapping", 0)
        m.set_option("cost_order", 1)


def test_start_ball_results_are_pinned(setup):
    # The plain kernel's results on the benchmark's start ball (65 536 walkers, seed 1, default options), pinned bit for bit:
    # sha256 of logp (float64) and status (int32) as computed on B200 by the kernel that still evaluated the first force at
    # the start of every step attempt.  Carrying it across attempts, the e / er bank swap and the state moved to shared
    # memory must not change one bit.  A change that is meant to alter the arithmetic updates this value.
    import hashlib
    m, oh, _ = setup
    theta = T.gaussian_ball(T.HD_SOL, T.HD_SCALE_VEC, 65536, 1)
    m.set_option("mapping", 0)
    m.set_option("cost_order", 1)
    lp, st = m.loglik(oh, theta)
    h = hashlib.sha256(np.asarray(lp, np.float64).tobytes() + np.asarray(st, np.int32).tobytes()).hexdigest()
    assert h == "0b3fd0f7218b60936f90385e62250dbe99aec79c12ade18ced4a53b796d0b2a3"
