"""Shared helpers for the tests: ctypes wrappers of the CPU oracle (oracle/) and of the test-only host
mirror, golden fixtures, parameter helpers.  The oracle is the checker only."""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
ELEMS = ("m", "a", "h", "k", "l", "ix", "iy")

_oracle = None
_mirror = None


def oracle():
    global _oracle
    if _oracle is None:
        _oracle = C.CDLL(os.path.join(ROOT, "oracle", "_build", "librvoracle.so"))
    return _oracle


_oracle_fast = None


def oracle_fast():
    """The oracle sources compiled -O3 -march=native ON THIS MACHINE (timing only; bench.py's CPU legs).  Built afresh in a
    temporary directory that is removed once the library is loaded, so the tree is never written (it may be read-only)
    and a build made elsewhere or from other sources is never loaded; falls back to the checker build if the compiler is
    missing."""
    global _oracle_fast
    if _oracle_fast is None:
        import shutil
        import subprocess
        import tempfile
        tmp = tempfile.mkdtemp(prefix="rvoracle_fast_")
        try:
            path = os.path.join(tmp, "librvoracle_fast.so")
            subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "fast", "FAST_OUT=" + path],
                           capture_output=True, timeout=300)
            _oracle_fast = C.CDLL(path) if os.path.exists(path) else oracle()
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    return _oracle_fast


def mirror():
    global _mirror
    if _mirror is None:
        _mirror = C.CDLL(os.path.join(ROOT, "tests", "hostmirror", "_build", "librvmirror.so"))
    return _mirror


def vp(a):
    return None if a is None else np.ascontiguousarray(a).ctypes.data_as(C.c_void_p)


def elems_from_planets(planets):
    out = np.zeros((len(planets), 7))
    for i, p in enumerate(planets):
        for k, v in p.items():
            out[i, ELEMS.index(k)] = v
    return out


def planets_from_vec(v):
    """Reference parameter order a,h,k,m,l per planet (SURVEY F6)."""
    v = np.asarray(v, dtype=float).reshape(-1, 5)
    return [dict(a=r[0], h=r[1], k=r[2], m=r[3], l=r[4]) for r in v]


class Obs(object):
    pass


def load_vels(name, npoints=100):
    """observations.py:52-69 restated for the oracle side."""
    d = np.genfromtxt(os.path.join(GOLDEN, name))
    t = d[:, 0] * 0.01720
    rv = d[:, 1] * 3.355e-5
    er = d[:, 2] * 3.355e-5
    tb, tf = np.array_split(t, 2)
    shift = tb[-1]
    o = Obs()
    o.tf, o.tb = tf - shift, tb - shift
    o.rvb, o.rvf = np.array_split(rv, 2)
    o.errorb, o.errorf = np.array_split(er, 2)
    o.Npoints = npoints
    return o


def orc_logp(E, hill, obs, counters=False):
    E = np.ascontiguousarray(E, dtype=np.float64)
    out = C.c_double()
    cnt = (C.c_long * 3)()
    legs = (C.c_int * 2)()
    st = oracle().orc_get_logp(E.shape[0], vp(E), C.c_double(hill), vp(obs.tf), vp(obs.rvf), vp(obs.errorf), len(obs.tf),
                               vp(obs.tb), vp(obs.rvb), vp(obs.errorb), len(obs.tb), C.c_double(obs.Npoints),
                               C.byref(out), cnt, legs)
    if counters:
        return st, out.value, list(cnt), list(legs)
    return st, out.value


def orc_rv(E, hill, times):
    E = np.ascontiguousarray(E, dtype=np.float64)
    times = np.ascontiguousarray(times, dtype=np.float64)
    rv = np.zeros(len(times))
    st = oracle().orc_get_rv(E.shape[0], vp(E), C.c_double(hill), vp(times), len(times), vp(rv), None)
    return st, rv


def orc_logp_batch(fixed, fp, fe, hill, obs, theta, nthreads=8, lib=None):
    fixed = np.ascontiguousarray(fixed, dtype=np.float64)
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    fp = np.ascontiguousarray(fp, dtype=np.int32)
    fe = np.ascontiguousarray(fe, dtype=np.int32)
    W = theta.shape[0]
    logp = np.zeros(W)
    status = np.zeros(W, dtype=np.int32)
    cnt = (C.c_long * 3)()
    (lib or oracle()).orc_logp_batch(fixed.shape[0], vp(fixed), len(fp), vp(fp), vp(fe), C.c_double(hill),
                            vp(obs.tf), vp(obs.rvf), vp(obs.errorf), len(obs.tf),
                            vp(obs.tb), vp(obs.rvb), vp(obs.errorb), len(obs.tb), C.c_double(obs.Npoints),
                            vp(theta), C.c_long(W), vp(logp), vp(status), cnt, nthreads)
    return logp, status, list(cnt)


def mirror_loglik(fixed, fp, fe, hill, obs, theta, dims=0, times=None):
    fixed = np.ascontiguousarray(fixed, dtype=np.float64)
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    fp = np.ascontiguousarray(fp, dtype=np.int32)
    fe = np.ascontiguousarray(fe, dtype=np.int32)
    W = theta.shape[0]
    logp = np.zeros(W)
    status = np.zeros(W, dtype=np.int32)
    cnt = (C.c_ulonglong * 2)()
    rv = None
    nt = 0
    if times is not None:
        times = np.ascontiguousarray(times, dtype=np.float64)
        nt = len(times)
        rv = np.zeros((W, nt))
    rc = mirror().mirror_loglik(fixed.shape[0], vp(fixed), len(fp), vp(fp), vp(fe), C.c_double(hill), dims,
                                vp(obs.tf), vp(obs.rvf), vp(obs.errorf), len(obs.tf),
                                vp(obs.tb), vp(obs.rvb), vp(obs.errorb), len(obs.tb), C.c_double(obs.Npoints),
                                vp(theta), C.c_longlong(W), vp(logp), vp(status), vp(times), nt, vp(rv), cnt)
    assert rc == 0, rc
    if times is not None:
        return rv, status
    return logp, status, list(cnt)


# reference order a,h,k,m,l for a 2-planet system -> (planet, ABI slot)
FP10 = [0, 0, 0, 0, 0, 1, 1, 1, 1, 1]
FE10 = [1, 2, 3, 0, 4, 1, 2, 3, 0, 4]

# SURVEY App. B golden values ------------------------------------------------------------------
HD_SOL = [6.57730330e-01, -9.72263877e-02, -7.82798396e-02, 8.84031737e-04, 4.42804990e+00,
          1.04404207e+00, -2.05622789e-02, -1.08797961e-01, 8.30379710e-04, 1.49919861e+00]
KAT2_LOGP = -2.41616612321          # (Ex)HD155358.ipynb:149
KAT6_VEC = [0.655966504, -0.0913957298, -0.0778916533, 0.000877209959, 4.75859384,
            1.04807688, -0.0267169122, -0.106648719, 0.000852818253, 1.4898423]
KAT6_LOGP = -6.7971014711           # (Ex)HD155358.ipynb:717-721 (weak: 9-digit params)
KAT5 = [   # (vector, leg that raises Encounter)  HD155358.ipynb:123-144,158-179,193-214
    ([0.678164812, -0.143058422, -0.306362671, 0.00126310873, 4.47837618,
      0.952247435, 0.0250317187, 0.0728550379, 0.00100432639, 1.91949611], "backward"),
    ([0.675027661, -0.161500043, -0.282542633, 0.0013430272, 4.62275061,
      0.962435601, 0.00346167619, 0.0294076924, 0.000942574591, 1.86928008], "forward"),
    ([0.671347869, -0.224912885, -0.266654234, 0.00148856083, 4.4032721,
      0.957707432, -0.0220906811, -0.0401350668, 0.00104525084, 1.07695102], "forward"),
]
KAT3_PLANETS = [{"m": 0.92e-3, "a": 0.2275, "h": -0.06, "k": 0.015, "l": -1.0},
                {"m": 1.95e-3, "a": 0.3665, "h": 0.02, "k": 0.0, "l": 2.1}]       # mcmc_benchmark_smala.py:32
KAT4_PLANETS = [{"m": 0.92e-3, "a": 0.2285, "h": 0.05, "k": 0.015, "l": -1.8},
                {"m": 1.95e-3, "a": 0.4778, "h": 0.01, "k": 0.0, "l": 2.15}]      # mcmc_benchmark_smala.py:33


def load_rvcurve(name):
    g = np.loadtxt(os.path.join(GOLDEN, name))
    return g[:1000], g[1000:]


def gaussian_ball(center, scales, W, seed, width=1e-3):
    """Ensemble.__init__'s start distribution (mcmc.py:49-51): theta + 1e-3*scales*N(0,1)."""
    rng = np.random.RandomState(seed)
    return np.asarray(center)[None, :] + width * np.asarray(scales)[None, :] * rng.normal(size=(W, len(center)))


HD_SCALES = {"m": 5.5e-6, "a": 0.001, "h": 0.02, "k": 0.02, "l": np.pi / 4}   # (Ex)HD155358.ipynb:456
HD_SCALE_VEC = [HD_SCALES[k] for k in ("a", "h", "k", "m", "l")] * 2


def orc_logp_d_dd_batch(fixed, fp, fe, hill, obs, theta, var_in_norm=0, nthreads=8):
    """Oracle State.get_logp_d_dd for a batch: (logp[W], grad[W][nv], hess[W][nv][nv], status[W], counters)."""
    fixed = np.ascontiguousarray(fixed, dtype=np.float64)
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    fp = np.ascontiguousarray(fp, dtype=np.int32)
    fe = np.ascontiguousarray(fe, dtype=np.int32)
    W, nv = theta.shape[0], len(fp)
    logp = np.zeros(W)
    grad = np.zeros((W, nv))
    hess = np.zeros((W, nv, nv))
    status = np.zeros(W, dtype=np.int32)
    cnt = (C.c_long * 3)()
    oracle().orc_logp_d_dd_batch(fixed.shape[0], vp(fixed), nv, vp(fp), vp(fe), C.c_double(hill),
                                 vp(obs.tf), vp(obs.rvf), vp(obs.errorf), len(obs.tf),
                                 vp(obs.tb), vp(obs.rvb), vp(obs.errorb), len(obs.tb), C.c_double(obs.Npoints),
                                 int(var_in_norm), vp(theta), C.c_long(W), vp(logp), vp(grad), vp(hess), vp(status), cnt,
                                 nthreads)
    return logp, grad, hess, status, list(cnt)


def mirror_loglik_d_dd(fixed, fp, fe, hill, obs, theta, dims=0):
    fixed = np.ascontiguousarray(fixed, dtype=np.float64)
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    fp = np.ascontiguousarray(fp, dtype=np.int32)
    fe = np.ascontiguousarray(fe, dtype=np.int32)
    W, nv = theta.shape[0], len(fp)
    logp = np.zeros(W)
    grad = np.zeros((W, nv))
    hess = np.zeros((W, nv, nv))
    status = np.zeros(W, dtype=np.int32)
    cnt = (C.c_ulonglong * 2)()
    rc = mirror().mirror_loglik_d_dd(fixed.shape[0], vp(fixed), nv, vp(fp), vp(fe), C.c_double(hill), dims,
                                     vp(obs.tf), vp(obs.rvf), vp(obs.errorf), len(obs.tf),
                                     vp(obs.tb), vp(obs.rvb), vp(obs.errorb), len(obs.tb), C.c_double(obs.Npoints),
                                     vp(theta), C.c_longlong(W), vp(logp), vp(grad), vp(hess), vp(status), cnt)
    assert rc == 0, rc
    return logp, grad, hess, status, list(cnt)


def orc_whfast_rv(E, hill, dt0, times):
    E = np.ascontiguousarray(E, dtype=np.float64)
    times = np.ascontiguousarray(times, dtype=np.float64)
    rv = np.zeros(len(times))
    cnt = (C.c_long * 3)()
    st = oracle().orc_whfast_get_rv(E.shape[0], vp(E), C.c_double(hill), C.c_double(dt0), vp(times), len(times), vp(rv), cnt)
    return st, rv, int(cnt[1])


def orc_whfast_logp_batch(fixed, fp, fe, hill, dt0, obs, theta, nthreads=8):
    fixed = np.ascontiguousarray(fixed, dtype=np.float64)
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    fp = np.ascontiguousarray(fp, dtype=np.int32)
    fe = np.ascontiguousarray(fe, dtype=np.int32)
    W = theta.shape[0]
    logp = np.zeros(W)
    status = np.zeros(W, dtype=np.int32)
    cnt = (C.c_long * 3)()
    oracle().orc_whfast_logp_batch(fixed.shape[0], vp(fixed), len(fp), vp(fp), vp(fe), C.c_double(hill), C.c_double(dt0),
                                   vp(obs.tf), vp(obs.rvf), vp(obs.errorf), len(obs.tf),
                                   vp(obs.tb), vp(obs.rvb), vp(obs.errorb), len(obs.tb), C.c_double(obs.Npoints),
                                   vp(theta), C.c_long(W), vp(logp), vp(status), cnt, nthreads)
    return logp, status, list(cnt)


def mirror_whfast(fixed, fp, fe, hill, dt0, obs, theta, dims=0, times=None):
    fixed = np.ascontiguousarray(fixed, dtype=np.float64)
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    fp = np.ascontiguousarray(fp, dtype=np.int32)
    fe = np.ascontiguousarray(fe, dtype=np.int32)
    W = theta.shape[0]
    logp = np.zeros(W)
    status = np.zeros(W, dtype=np.int32)
    cnt = (C.c_ulonglong * 2)()
    rv = None
    nt = 0
    if times is not None:
        times = np.ascontiguousarray(times, dtype=np.float64)
        nt = len(times)
        rv = np.zeros((W, nt))
    if obs is None:
        obs = Obs()
        obs.tf = obs.tb = obs.rvf = obs.rvb = obs.errorf = obs.errorb = np.zeros(0)
        obs.Npoints = 1
    rc = mirror().mirror_whfast(fixed.shape[0], vp(fixed), len(fp), vp(fp), vp(fe), C.c_double(hill), dims, C.c_double(dt0),
                                vp(obs.tf), vp(obs.rvf), vp(obs.errorf), len(obs.tf),
                                vp(obs.tb), vp(obs.rvb), vp(obs.errorb), len(obs.tb), C.c_double(obs.Npoints),
                                vp(theta), C.c_longlong(W), vp(logp), vp(status), vp(times), nt, vp(rv), cnt)
    assert rc == 0, rc
    if times is not None:
        return rv, status, list(cnt)
    return logp, status, list(cnt)


# ---- BASELINE configs[3] ("C4"): synthetic 3-planet near-resonant system -------------------------------
# the 2:1 pair of mcmc_benchmark_smala.py:32 plus a third planet near the next 2:1; scales / step of mcmc_benchmark_mh.py:52-53
C4_PLANETS = [{"m": 0.92e-3, "a": 0.2275, "h": -0.06, "k": 0.015, "l": -1.0},
              {"m": 1.95e-3, "a": 0.3665, "h": 0.02, "k": 0.0, "l": 2.1},
              {"m": 1.0e-3, "a": 0.59, "h": 0.0, "k": 0.03, "l": 0.7}]
C4_SCALES = {"m": 1e-3, "a": 0.3, "h": 0.5, "k": 0.5, "l": np.pi / 2}
FP15 = [p for p in range(3) for _ in range(5)]
FE15 = [1, 2, 3, 0, 4] * 3                      # a, h, k, m, l per planet (reference parameter order)


def c4_problem(nper=40, tmax=30.0, seed=17, err=1.5e-4):
    """(obs, fixed[3][7], center[15], scale_vec[15]): RVs of the true system from the oracle plus Gaussian noise."""
    rng = np.random.RandomState(seed)
    obs = Obs()
    obs.tf = np.append([0.0], np.sort(rng.uniform(0, tmax / 2, nper)))
    obs.tb = np.sort(rng.uniform(-tmax / 2, 0, nper))
    E = elems_from_planets(C4_PLANETS)
    st, rvf = orc_rv(E, 0.0, obs.tf)
    st2, rvb = orc_rv(E, 0.0, obs.tb)
    assert st == 0 and st2 == 0
    obs.errorf = np.full(nper + 1, err); obs.errorb = np.full(nper, err)
    obs.rvf = rvf + err * rng.normal(size=nper + 1); obs.rvb = rvb + err * rng.normal(size=nper)
    obs.Npoints = 2 * nper
    center = np.array([[p[k] for k in ("a", "h", "k", "m", "l")] for p in C4_PLANETS]).reshape(-1)
    scale_vec = np.array([C4_SCALES[k] for k in ("a", "h", "k", "m", "l")] * 3)
    return obs, np.zeros((3, 7)), center, scale_vec


# ---- beyond the BASELINE configs: the reference's schema is open in the number of planets (state.py:8-31) ----------------
FIVE_PLANETS = [{"m": 0.92e-3, "a": 0.2275, "h": -0.06, "k": 0.015, "l": -1.0},
                {"m": 1.95e-3, "a": 0.3665, "h": 0.02, "k": 0.0, "l": 2.1},
                {"m": 1.1e-3, "a": 0.59, "h": 0.01, "k": 0.03, "l": 0.4},
                {"m": 0.6e-3, "a": 0.95, "h": -0.02, "k": 0.01, "l": 2.9},
                {"m": 0.3e-3, "a": 1.55, "h": 0.03, "k": -0.02, "l": -2.2}]


def many_planet_problem(npl, nper=30, tmax=24.0, seed=23, err=1.5e-4):
    """(obs, fixed[npl][7], fp, fe, center[5 npl], scale_vec[5 npl]) for the first npl of FIVE_PLANETS, all (a, h, k, m, l) free."""
    rng = np.random.RandomState(seed)
    planets = FIVE_PLANETS[:npl]
    obs = Obs()
    obs.tf = np.append([0.0], np.sort(rng.uniform(0, tmax / 2, nper)))
    obs.tb = np.sort(rng.uniform(-tmax / 2, 0, nper))
    E = elems_from_planets(planets)
    st, rvf = orc_rv(E, 0.0, obs.tf)
    st2, rvb = orc_rv(E, 0.0, obs.tb)
    assert st == 0 and st2 == 0
    obs.errorf = np.full(nper + 1, err); obs.errorb = np.full(nper, err)
    obs.rvf = rvf + err * rng.normal(size=nper + 1); obs.rvb = rvb + err * rng.normal(size=nper)
    obs.Npoints = 2 * nper
    fp = [p for p in range(npl) for _ in range(5)]
    fe = [1, 2, 3, 0, 4] * npl
    center = np.array([[p[k] for k in ("a", "h", "k", "m", "l")] for p in planets]).reshape(-1)
    scale_vec = np.array([C4_SCALES[k] for k in ("a", "h", "k", "m", "l")] * npl)
    return obs, np.zeros((npl, 7)), fp, fe, center, scale_vec
