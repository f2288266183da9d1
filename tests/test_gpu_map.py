"""GPU tests of the batched maximum-likelihood fit (rv_map_fit): the HD155358 fit from the published solution and the
16-start ball against the golden run of the numpy restatement (oracle/map_oracle.py, tools/make_map_golden.py), batch
invariance, statuses and argument checks, synthetic one- and three-planet problems, State / driver / DeviceGroup."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import parity_horizon as PH
import rvtest as T

pytestmark = pytest.mark.gpu
Z2 = np.zeros((2, 7))
GOLD = json.load(open(os.path.join(T.GOLDEN, "hd155358_map_multistart.json")))


@pytest.fixture(scope="module")
def ctx():
    from rvel_mcmc_b200 import _abi
    c = _abi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def hd(ctx):
    from rvel_mcmc_b200 import _abi
    obs = T.load_vels("HD155358.vels")
    oh = _abi.ObsHandle(ctx, obs.tf, obs.rvf, obs.errorf, obs.tb, obs.rvb, obs.errorb, obs.Npoints)
    return oh, _abi.ModelHandle(ctx, Z2, T.FP10, T.FE10, 2.0)


def _half_decrement(g, H):
    lam, Q = np.linalg.eigh(-0.5 * (H + H.T))
    y = Q.T @ g
    return 0.5 * float(np.sum(y * y / np.maximum(np.abs(lam), 1e-12 * np.abs(lam).max())))


def _sigma(H):
    return np.sqrt(np.diag(np.linalg.inv(-H)))


def test_fit_from_published_solution(hd):
    from rvel_mcmc_b200 import _abi
    oh, m = hd
    g = GOLD["single"]
    r = m.map_fit(oh, np.array(T.HD_SOL)[None, :])
    assert r["fit_code"][0] == _abi.RV_FIT_CONVERGED and r["status"][0] == 0
    assert abs(r["logp"][0] - g["logp"]) <= 1e-10, (r["logp"][0], g["logp"])
    assert np.abs((r["theta"][0] - np.array(g["theta"])) / _sigma(r["hess"][0])).max() <= 1e-6
    assert _half_decrement(r["grad"][0], r["hess"][0]) <= 1e-10
    assert abs(r["n_iter"][0] - g["n_iter"]) <= 1
    assert r["logp"][0] > T.KAT2_LOGP + 0.5


@pytest.fixture(scope="module")
def ball(hd):
    oh, m = hd
    return m.map_fit(oh, np.array(GOLD["starts"]))


def test_multistart_ball_matches_golden(ball):
    from rvel_mcmc_b200 import _abi
    bad = []
    for w, g in enumerate(GOLD["multistart"]):
        same = ball["fit_code"][w] == g["fit_code"] and ball["status"][w] == g["status"]
        if same and g["fit_code"] == _abi.RV_FIT_CONVERGED:
            same = abs(ball["logp"][w] - g["logp"]) <= 1e-9
        if not same:
            bad.append((w, int(ball["fit_code"][w]), int(ball["status"][w]), float(ball["logp"][w]), int(ball["n_iter"][w]),
                        g["fit_code"], g["status"], g["logp"], g["n_iter"]))
    assert not bad, bad


def test_find_map_gpu_reports_both_maxima():
    from rvel_mcmc_b200 import _abi, driver, observations, state
    obs = observations.Observation_FromFile(os.path.join(T.GOLDEN, "HD155358.vels"), Npoints=100)
    st = state.State(T.planets_from_vec(T.HD_SOL)); st.hillRadiusFactor = 2.
    out = driver.find_map_gpu(st, obs, 16, T.HD_SCALES, width=1.0, seed=GOLD["seed"])
    res = out["results"]
    assert np.array_equal(np.sort(res["start"], axis=0), np.sort(np.array(GOLD["starts"]), axis=0))
    assert np.all(np.diff(res["logp"][np.isfinite(res["logp"])]) <= 0)
    gl = np.array([g["logp"] for g in GOLD["multistart"] if g["fit_code"] == _abi.RV_FIT_CONVERGED])
    levels = sorted(set(np.round(gl, 7)), reverse=True)
    assert len(out["maxima"]) == len(levels) == 2
    for mx, lv in zip(out["maxima"], levels):
        assert abs(mx["logp"] - lv) < 1e-7
        assert mx["count"] == int(np.sum(np.round(gl, 7) == lv))
        assert mx["state"].hillRadiusFactor == 2. and mx["state"].fit_code == _abi.RV_FIT_CONVERGED
        assert np.array_equal(mx["state"].get_params(), mx["theta"]) and np.allclose(mx["sigma"] ** 2, np.diag(mx["cov"]))


def test_batch_invariance(hd):
    oh, m = hd
    rng = np.random.default_rng(11)
    big = np.array(T.HD_SOL)[None, :] + np.array(T.HD_SCALE_VEC)[None, :] * rng.normal(size=(4096, 10))
    sl = slice(1500, 1564)
    a = m.map_fit(oh, big[sl])
    b = m.map_fit(oh, big)
    for k in a:
        assert np.array_equal(a[k], b[k][sl], equal_nan=True), k
    assert (b["fit_code"] == 0).mean() > 0.5


def test_statuses_and_max_iter(hd):
    from rvel_mcmc_b200 import _abi
    oh, m = hd
    prior = np.array(T.HD_SOL); prior[0] = 0.01               # a <= 0.02
    enc = np.array(T.KAT5[0][0])
    X = np.vstack([prior, enc, T.HD_SOL])
    r = m.map_fit(oh, X)
    assert list(r["status"][:2]) == [_abi.RV_PRIOR, _abi.RV_ENCOUNTER]
    assert list(r["fit_code"][:2]) == [_abi.RV_FIT_NOSTART] * 2 and list(r["n_iter"][:2]) == [0, 0]
    assert np.array_equal(r["theta"][:2], X[:2]) and np.isneginf(r["logp"][:2]).all()
    # max_iter = 0: the evaluation at the start
    r0 = m.map_fit(oh, X[2:], max_iter=0)
    lo, go, ho, so = m.loglik_d_dd(oh, X[2:])
    assert r0["fit_code"][0] == _abi.RV_FIT_MAXITER and r0["n_iter"][0] == 0 and np.array_equal(r0["theta"], X[2:])
    assert np.array_equal(r0["logp"], lo) and np.array_equal(r0["grad"], go) and np.array_equal(r0["hess"], ho)
    # W = 0
    e = m.map_fit(oh, np.zeros((0, 10)))
    assert all(len(v) == 0 for v in e.values())


def test_argument_checks(ctx, hd):
    from rvel_mcmc_b200 import _abi
    oh, m = hd
    X = np.array(T.HD_SOL)[None, :]
    for kw in (dict(n_trial=0), dict(n_trial=17), dict(max_iter=-1), dict(tol=-1.0), dict(damping=np.nan)):
        with pytest.raises(_abi.RvGpuError, match="rv_map_fit"):
            m.map_fit(oh, X, **kw)
    lib = ctx.lib
    buf = np.zeros(64)
    ib = np.zeros(8, dtype=np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert lib.rv_map_fit(ctx.h, m.h, oh.h, p(buf), -1, 5, 8, 1e-10, 0.0, p(buf), None, None, p(ib), p(ib), p(ib)) < 0
    assert b"rv_map_fit" in lib.rv_last_error(ctx.h)
    for k in range(5):
        args = [p(buf), p(buf), p(ib), p(ib), p(ib)]
        args[k] = None
        rc = lib.rv_map_fit(ctx.h, m.h, oh.h, args[0], 1, 5, 8, 1e-10, 0.0, args[1], None, None, args[2], args[3], args[4])
        assert rc == -1 and b"NULL" in lib.rv_last_error(ctx.h)
    wh = _abi.ModelHandle(ctx, Z2, T.FP10, T.FE10, 2.0)
    wh.set_option("integrator", 1)
    with pytest.raises(_abi.RvGpuError, match="-31"):
        wh.map_fit(oh, X)


def test_synthetic_one_planet():
    from rvel_mcmc_b200 import _abi, driver, observations, state
    truth = state.State([{"m": 1.2e-3, "a": 1.1, "h": 0.05, "k": -0.03, "l": 0.7}])
    np.random.seed(31)
    obs = observations.FakeObservation(truth, Npoints=60, error=4e-5, tmax=12.0)
    lp_truth = truth.deepcopy().get_logp(obs)
    scal = {"m": 1e-4, "a": 0.01, "h": 0.02, "k": 0.02, "l": 0.05}
    out = driver.find_map_gpu(truth, obs, 8, scal, width=1.0, seed=3)
    best = out["maxima"][0]
    assert best["logp"] >= lp_truth
    assert np.all(np.abs(truth.get_params() - best["theta"]) <= 3 * best["sigma"]), (truth.get_params() - best["theta"]) / best["sigma"]
    assert best["state"].fit_code == _abi.RV_FIT_CONVERGED


def test_c4_three_planets_converge(ctx):
    from rvel_mcmc_b200 import _abi
    obs, fixed, fp, fe, hill, center, sc = PH.problem("c4")
    oh, m = PH._handles(ctx, obs, fixed, fp, fe, hill)
    X = np.vstack([center, T.gaussian_ball(center, sc, 3, 5, width=1e-3)])
    lp_truth = m.loglik_d_dd(oh, center[None, :])[0][0]
    r = m.map_fit(oh, X)
    assert (r["fit_code"] == _abi.RV_FIT_CONVERGED).all(), r["fit_code"]
    assert (r["logp"] >= lp_truth).all()


def test_state_find_map_matches_batch_and_device_group(hd):
    from rvel_mcmc_b200 import _abi, multigpu, observations, state
    obs = observations.Observation_FromFile(os.path.join(T.GOLDEN, "HD155358.vels"), Npoints=100)
    st = state.State(T.planets_from_vec(T.HD_SOL)); st.hillRadiusFactor = 2.
    fit = st.find_map(obs)
    oh, m = hd
    r = m.map_fit(oh, np.array(T.HD_SOL)[None, :])
    assert np.array_equal(fit.get_params(), r["theta"][0]) and fit.logp == r["logp"][0]
    assert np.array_equal(fit.logp_d, r["grad"][0]) and np.array_equal(fit.logp_dd, r["hess"][0])
    assert fit.hillRadiusFactor == 2. and fit.fit_code == _abi.RV_FIT_CONVERGED and fit.n_iter == r["n_iter"][0]
    assert np.allclose(fit.laplace_cov, np.linalg.inv(-r["hess"][0]), rtol=1e-12, atol=0)
    assert fit.get_logp_d_dd(obs)[0] == r["logp"][0]                  # cached
    bad = state.State(T.planets_from_vec(T.KAT5[0][0])); bad.hillRadiusFactor = 2.
    with pytest.raises(_abi.Encounter):
        bad.find_map(obs)
    out = state.State(T.planets_from_vec(T.HD_SOL)); out.planets[0]["a"] = 0.01
    with pytest.raises(_abi.RvGpuError):
        out.find_map(obs)
    try:
        group = multigpu.DeviceGroup()
    except _abi.RvGpuError:
        pytest.skip("no device group")
    try:
        if len(group) < 2:
            pytest.skip("needs two GPUs")
        X = np.array(GOLD["starts"])
        a = group.map_fit(st, obs, X)
        b = m.map_fit(oh, X)
        for k in b:
            assert np.array_equal(a[k], b[k], equal_nan=True), k
    finally:
        group.close()
