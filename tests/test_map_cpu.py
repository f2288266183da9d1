"""The maximum-likelihood fit on the CPU: the device's per-walker arithmetic (rv_map.cuh, compiled for the host) against
numpy.linalg.eigh, and the device algorithm run on the host (mirror variational + mirror plain likelihood + mirror step /
select, in the loop order of rv_abi.cu's map_fit_impl) against the numpy restatement oracle/map_oracle.py."""
import ctypes as C
import json
import os
import sys

import numpy as np
import pytest

import rvtest as T
from test_samplers_cpu import _small_problem

sys.path.insert(0, os.path.join(T.ROOT, "oracle"))
import map_oracle as M  # noqa: E402

Z2 = np.zeros((2, 7))
_map_lib = None


def map_mirror():
    """mirror_map.cpp (the fit's step / select from rv_map.cuh) compiled for the host into a temporary directory, which is
    removed once the library is loaded: the tree is never written."""
    global _map_lib
    if _map_lib is None:
        import shutil
        import subprocess
        import tempfile
        tmp = tempfile.mkdtemp(prefix="rvmirror_map_")
        try:
            out = os.path.join(tmp, "librvmirror_map.so")
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            r = subprocess.run([cxx, "-O2", "-std=c++17", "-x", "c++", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas",
                                "-o", out, os.path.join(T.ROOT, "tests", "hostmirror", "mirror_map.cpp"), "-lm"],
                               capture_output=True, text=True, timeout=300)
            assert r.returncode == 0, r.stderr[-4000:]
            _map_lib = C.CDLL(out)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    return _map_lib


def mirror_step(th, g, H, mu=0.0, n_iter=0, max_iter=50, tol=1e-10, n_trial=8):
    n = len(th)
    rows = np.zeros((n_trial + 1, n))
    dec = C.c_double()
    c = map_mirror().mirror_map_step(n, T.vp(np.ascontiguousarray(th, dtype=np.float64)),
                                   T.vp(np.ascontiguousarray(g, dtype=np.float64)),
                                   T.vp(np.ascontiguousarray(H, dtype=np.float64)), C.c_double(mu), int(n_iter),
                                   int(max_iter), C.c_double(tol), int(n_trial), T.vp(rows), C.byref(dec))
    return c, rows, dec.value


def mirror_select(rows, tlogp, tstatus, th, mu, n_iter, code=M.RUNNING):
    n_trial, n = rows.shape[0] - 1, rows.shape[1]
    th = np.ascontiguousarray(th, dtype=np.float64).copy()
    m, it, c = C.c_double(mu), C.c_int(n_iter), C.c_int(code)
    moved = map_mirror().mirror_map_select(n, n_trial, T.vp(rows), T.vp(np.ascontiguousarray(tlogp, dtype=np.float64)),
                                         T.vp(np.ascontiguousarray(tstatus, dtype=np.int32)), T.vp(th), C.byref(m),
                                         C.byref(it), C.byref(c))
    return bool(moved), th, m.value, it.value, c.value


def _matrix(rng, n, cond, kind):
    """-H for the step tests.  'scaled': a well-conditioned core under a diagonal scaling, the structure of an RV
    Hessian (parameters in different units; HD155358's condition number is ~1e7).  'rotated': eigenvalues spread
    geometrically under a random rotation.  'flat': one parameter the data do not constrain (a zero row and column)."""
    Q, _ = np.linalg.qr(rng.normal(size=(n, n)))
    if kind == "scaled":
        D = np.geomspace(1.0, 1.0 / np.sqrt(cond), n)[rng.permutation(n)]
        A = D[:, None] * ((Q * np.linspace(1.0, 3.0, n)) @ Q.T) * D[None, :]
    else:
        lam = np.geomspace(1.0, 1.0 / cond, n) * rng.uniform(1, 10)
        A = (Q * lam) @ Q.T
    if kind == "indefinite":
        lam = np.geomspace(1.0, 1.0 / cond, n) * np.where(np.arange(n) % 3 == 1, -1.0, 1.0)
        A = (Q * lam) @ Q.T
    A = 0.5 * (A + A.T)
    if kind == "flat":
        k = rng.integers(n)
        A[k, :] = 0.0; A[:, k] = 0.0
    return A


# Rotated matrices stop at cond 1e5: a random rotation mixes scales, so the small eigenvalues of the rounded matrix are
# only determined to ~cond * 1e-16 relative and two correct solvers (Jacobi, LAPACK) differ by that much -- 1e-9 at 1e7.
# Scaled matrices keep their small eigenvalues well determined and are checked up to cond 1e8, against numpy applied to the
# equilibrated matrix S A S (S = diag(A)^-1/2): LAPACK's eigh on A itself is accurate to eps * |A| only, i.e. to ~1e-9
# relative in the smallest eigenvalue at cond 1e7, while Jacobi resolves it.
CASES = [(n, cond, kind) for n in (2, 5, 10, 15, 35) for cond, kind in
         [(1e2, "rotated"), (1e5, "rotated"), (1e3, "indefinite"), (1e5, "indefinite"), (1e4, "flat"),
          (1e3, "scaled"), (1e7, "scaled"), (1e8, "scaled")]]


@pytest.mark.parametrize("n,cond,kind", CASES)
def test_step_matches_numpy_eigh(n, cond, kind):
    rng = np.random.default_rng([n, int(np.log10(cond)), CASES.index((n, cond, kind))])
    for rep in range(4):
        A = _matrix(rng, n, cond, kind)
        th, g = rng.normal(size=n), rng.normal(size=n)
        mu = (0.0, 1e-6, 1e-3, 1.0)[rep]
        c, rows, dec = mirror_step(th, g, -A, mu=mu)
        co, ro, deco = M.step(th, g, -A, mu, 0, 50, 1e-10, 8)
        assert c == co == M.RUNNING
        if kind == "scaled":                 # positive definite, eigenvalues far above the floor: d = (A + mu lam_max)^-1 g
            S = 1.0 / np.sqrt(np.diag(A))
            As, lmax = S[:, None] * A * S[None, :], np.linalg.eigvalsh(A).max()
            ro = th[None, :] + (2.0 ** -np.arange(-1, 8))[:, None] * (S * np.linalg.solve(As + mu * lmax * np.diag(S * S),
                                                                                            S * g))[None, :]
            ro[0] = th
            deco = g @ (S * np.linalg.solve(As, S * g))
        assert np.array_equal(rows[0], th)
        d, do = rows[1] - th, ro[1] - th
        assert np.abs(d - do).max() <= 1e-10 * np.abs(do).max(), (rep, np.abs(d - do).max() / np.abs(do).max())
        assert abs(dec - deco) <= 1e-10 * abs(deco)
        assert np.abs(rows[1:] - ro[1:]).max() <= 1e-10 * np.abs(do).max()
        # the definiteness test at a stop (tol above the decrement)
        c2, rows2, _ = mirror_step(th, g, -A, tol=1e300)
        c2o, _, _ = M.step(th, g, -A, 0.0, 0, 50, 1e300, 8)
        assert c2 == c2o == (M.CONVERGED if kind in ("rotated", "scaled") else M.SADDLE)
        assert (rows2 == th[None, :]).all()


def test_step_stop_rules():
    th, g = np.array([1.0, 2.0]), np.array([1e-6, -2e-6])
    H = -np.diag([4.0, 1.0])
    c, rows, dec = mirror_step(th, g, H, tol=1e-10)           # decrement 4.25e-12 / 2 <= tol
    assert c == M.CONVERGED and abs(dec - (1e-12 / 4 + 4e-12)) < 1e-24
    c, _, _ = mirror_step(th, g, -H, tol=1e-10)               # same decrement at a minimum
    assert c == M.SADDLE
    c, _, _ = mirror_step(th, 1e3 * g, H, n_iter=5, max_iter=5)
    assert c == M.MAXITER
    c, _, _ = mirror_step(th, 1e3 * g, H, n_iter=0, max_iter=0)
    assert c == M.MAXITER
    c, _, _ = mirror_step(th, g, np.zeros((2, 2)))             # no usable eigenvalue
    assert c == M.SADDLE


def test_select_rules():
    th = np.array([0.5, 0.1])
    rows = th[None, :] + np.arange(9)[:, None] * np.array([1e-3, 0.0])[None, :]
    st = np.zeros(9, dtype=np.int32)
    lp = np.array([-2.0, -1.5, -1.2, -1.2, -3.0, -2.5, -2.1, -2.0, -9.0])
    moved, th2, mu, it, code = mirror_select(rows, lp, st, th, 1e-6, 3)
    assert moved and np.array_equal(th2, rows[2]) and mu == 0.0 and it == 4 and code == M.RUNNING   # lowest j on ties
    moved, th2, mu, it, code = mirror_select(rows, lp, st, th, 1e-3, 3)
    assert moved and mu == 1e-4
    st2 = st.copy(); st2[1:4] = 3                             # the best rows did not evaluate
    moved, th2, mu, it, code = mirror_select(rows, lp, st2, th, 0.0, 3)
    assert not moved and np.array_equal(th2, th) and mu == 1e-6 and it == 3 and code == M.RUNNING
    moved, th2, mu, it, code = mirror_select(rows, lp, st2, th, 0.1, 3)
    assert not moved and mu == 1.0 and code == M.RUNNING
    moved, th2, mu, it, code = mirror_select(rows, lp, st2, th, 1.0, 3)
    assert not moved and mu == 10.0 and code == M.STALLED
    for args in ((rows, lp, st, th, 1e-6, 3), (rows, lp, st2, th, 0.1, 3), (rows, lp, st2, th, 1.0, 3)):
        a, b = mirror_select(*args), M.select(args[0], args[1], args[2], args[4], args[5])
        assert a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2] == b[2] and a[3] == b[3] and a[4] == b[4]


def device_fit_on_host(evaluate, plain, theta0, max_iter=50, n_trial=8, tol=1e-10, damping=0.0):
    """map_fit_impl's loop with the mirror's step / select and the mirror's evaluations (every walker's rows evaluated,
    rows of theta for a stopped walker, as the device does)."""
    theta = np.array(theta0, dtype=np.float64, ndmin=2)
    W, n = theta.shape
    logp = np.zeros(W); grad = np.zeros((W, n)); hess = np.zeros((W, n, n)); status = np.zeros(W, dtype=np.int32)
    code = np.full(W, M.RUNNING); iters = np.zeros(W, dtype=np.int32); mu = np.full(W, float(damping))
    run, ev = list(range(W)), list(range(W))
    while run:
        if ev:
            lo, go, ho, so = evaluate(theta[ev])
            for s, w in enumerate(ev):
                logp[w], grad[w], hess[w], status[w] = lo[s], go[s], ho[s], so[s]
                if so[s] != 0:
                    code[w] = M.NOSTART if iters[w] == 0 else M.STALLED
        rows = []
        for w in run:
            if code[w] != M.RUNNING:
                rows.append(np.tile(theta[w], (n_trial + 1, 1)))
                continue
            c, r, _ = mirror_step(theta[w], grad[w], hess[w], mu[w], iters[w], max_iter, tol, n_trial)
            if c != M.RUNNING:
                code[w] = c
            rows.append(r)
        tl, ts = plain(np.vstack(rows))
        tl, ts = tl.reshape(len(run), n_trial + 1), ts.reshape(len(run), n_trial + 1)
        nxt, ev = [], []
        for s, w in enumerate(run):
            if code[w] != M.RUNNING:
                continue
            moved, theta[w], mu[w], iters[w], code[w] = mirror_select(rows[s], tl[s], ts[s], theta[w], mu[w], iters[w])
            if code[w] == M.RUNNING:
                nxt.append(w)
            if moved:
                ev.append(w)
        run = nxt
    return dict(theta=theta, logp=logp, grad=grad, hess=hess, status=status, fit_code=code, n_iter=iters)


def _fns(obs, E, fp, fe, hill):
    def o_eval(X):
        return T.orc_logp_d_dd_batch(E, fp, fe, hill, obs, X)[:4]

    def o_plain(X):
        return T.orc_logp_batch(E, fp, fe, hill, obs, X)[:2]

    def m_eval(X):
        return T.mirror_loglik_d_dd(E, fp, fe, hill, obs, X)[:4]

    def m_plain(X):
        return T.mirror_loglik(E, fp, fe, hill, obs, X)[:2]
    return o_eval, o_plain, m_eval, m_plain


def _agree(r, o):
    assert np.array_equal(r["fit_code"], o["fit_code"]), (r["fit_code"], o["fit_code"])
    assert np.array_equal(r["status"], o["status"])
    assert np.abs(r["n_iter"] - o["n_iter"]).max() <= 1
    ok = o["status"] == 0
    assert np.abs(r["logp"][ok] - o["logp"][ok]).max() <= 1e-10
    for w in np.flatnonzero(o["fit_code"] == M.CONVERGED):
        sig = np.sqrt(np.diag(np.linalg.inv(-o["hess"][w])))
        assert np.abs((r["theta"][w] - o["theta"][w]) / sig).max() <= 1e-6, w


def test_device_algorithm_on_host_matches_oracle_small_problem():
    obs, E, fp, fe, center = _small_problem()
    o_eval, o_plain, m_eval, m_plain = _fns(obs, E, fp, fe, 1.0)
    rng = np.random.default_rng(3)
    X = center[None, :] + np.array([0.01, 0.05, 0.05])[None, :] * rng.normal(size=(5, 3))
    X = np.vstack([X, [[0.01, 0.02, 0.01]]])                  # a = 0.01: outside the hard prior
    o = M.map_fit(o_eval, o_plain, X)
    r = device_fit_on_host(m_eval, m_plain, X)
    _agree(r, o)
    assert o["fit_code"][-1] == M.NOSTART and o["status"][-1] == 1 and o["n_iter"][-1] == 0
    assert np.array_equal(r["theta"][-1], X[-1])
    assert (o["fit_code"][:-1] == M.CONVERGED).all()
    assert (r["logp"][:-1] >= o_eval(center[None, :])[0][0] - 1e-12).all()


def test_device_algorithm_on_host_matches_oracle_from_hd_sol():
    obs = T.load_vels("HD155358.vels")
    o_eval, o_plain, m_eval, m_plain = _fns(obs, Z2, T.FP10, T.FE10, 2.0)
    X = np.array(T.HD_SOL)[None, :]
    o = M.map_fit(o_eval, o_plain, X)
    r = device_fit_on_host(m_eval, m_plain, X)
    _agree(r, o)
    assert o["fit_code"][0] == M.CONVERGED
    g = json.load(open(os.path.join(T.GOLDEN, "hd155358_map_multistart.json")))["single"]
    assert abs(o["logp"][0] - g["logp"]) <= 1e-12 and o["fit_code"][0] == g["fit_code"] and o["n_iter"][0] == g["n_iter"]
    assert o["logp"][0] > T.KAT2_LOGP + 0.5                   # the published point is not the maximum


def test_product_does_not_reference_the_fit_oracle():
    pkg = os.path.join(T.ROOT, "rvel_mcmc_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                assert "map_oracle" not in open(os.path.join(dirpath, f), errors="ignore").read(), f
