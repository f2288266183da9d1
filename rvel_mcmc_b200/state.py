"""State -- Python-3 mirror of the reference's state.py, backed by the CUDA engine.

Public names, argument meaning and error behaviour follow state.py:7-315.  What changed underneath:
``get_rv`` / ``get_logp`` call librvgpu (one call per evaluation instead of one ctypes call per epoch),
``rebound.Encounter`` becomes ``rvel_mcmc_b200.Encounter``.  Python-2 behaviours that shaped published
results are reproduced on purpose: the parameter-vector order is CPython-2.7's dict order
(``a, ix, h, k, m, l, iy`` filtered to the keys present; SURVEY App. B.8), and ``ignore_vars`` keeps its
``x not in ignore_vars`` semantics (a substring test when a str is passed; state.py:26).
"""
import copy

import numpy as np

from . import _abi
from ._abi import Encounter

# CPython-2.7 iteration order of a dict with these string keys (state.py:129-138 relies on it)
PY2_KEY_ORDER = ("a", "ix", "h", "k", "m", "l", "iy")
_ELEM_SLOT = {k: i for i, k in enumerate(_abi.ELEMS)}


def _py2_order(planet):
    known = [k for k in PY2_KEY_ORDER if k in planet]
    other = [k for k in planet.keys() if k not in PY2_KEY_ORDER]
    return known + other


class _Particle(object):
    __slots__ = ("m", "x", "y", "z", "vx", "vy", "vz")

    def __init__(self, row):
        self.m, self.x, self.y, self.z, self.vx, self.vy, self.vz = [float(v) for v in row]


class _SimSnapshot(object):
    """Initial particles of a simulation (see State.setup_sim)."""

    def __init__(self, rows, exit_min_distance):
        self.particles = [_Particle(r) for r in rows]
        self.exit_min_distance = exit_min_distance
        self.N = len(self.particles)
        self.t = 0.0


class State(object):
    verbose_prior = False    # the reference prints on every prior rejection (state.py:302-313)
    # Not in the reference (which always runs rebound's default IAS15): "whfast" selects the optional fixed-step
    # variant with step `dt` (what `sim.integrator = "whfast"; sim.dt = dt` would be in setup_sim).
    integrator = "ias15"
    dt = 0.001
    # Not in the reference either: True evaluates get_logp with one continuous integration per leg and RVs read inside
    # the natural IAS15 steps (model option dense_output) -- same likelihood to ~1e-12, up to several times fewer steps.
    dense_output = False

    def __init__(self, planets, ignore_vars=[], ignore_params=None):
        for planet in planets:            # re-key in place so iteration order matches the reference's
            items = [(k, planet[k]) for k in _py2_order(planet)]
            planet.clear()
            planet.update(items)
        self.planets = planets
        self.logp = None
        self.logp_d = None
        self.logp_dd = None
        self.planets_vars = []
        self.Nvars = 0
        self.hillRadiusMax = 0.0
        self.hillRadiusFactor = 1.
        self.planet1x = []
        self.planet1y = []
        self.planet2x = []
        self.planet2y = []
        self.ignore_vars = ignore_vars
        self.ignore_params = ignore_params
        for p, planet in enumerate(planets):
            planet_vars = [x for x in planet.keys() if (x not in ignore_vars)]
            if ignore_params is not None:
                for o in range(len(ignore_params[p])):
                    planet_vars.remove(ignore_params[p][o])
            self.planets_vars.append(planet_vars)
            self.Nvars += len(planet_vars)
        for planet in planets:
            for k in planet.keys():
                if k not in _ELEM_SLOT:
                    raise AttributeError("unknown orbital element '%s' (expected a subset of m,a,h,k,l,ix,iy)" % k)

    # ------------------------------------------------------------------ engine plumbing
    def _free_slots(self):
        """(planet index, element slot) of every entry of get_params(), in order."""
        fp, fe = [], []
        for i, planet in enumerate(self.planets):
            for k in planet.keys():
                if self._is_free(i, k):
                    fp.append(i)
                    fe.append(_ELEM_SLOT[k])
        return fp, fe

    def _is_free(self, i, k):
        if self.ignore_params is not None:
            return (k not in self.ignore_vars) and (k not in self.ignore_params[i])
        return k not in self.ignore_vars

    def _fixed_matrix(self):
        fixed = np.zeros((len(self.planets), len(_abi.ELEMS)))
        for i, planet in enumerate(self.planets):
            for k, v in planet.items():
                fixed[i, _ELEM_SLOT[k]] = v
        return fixed

    def _model(self, ctx=None, hill_factor=None, all_free=False):
        """rv_model for this schema.  Fixed values are part of the cache key (they live in HBM)."""
        ctx = ctx or _abi.default_context()
        hf = self.hillRadiusFactor if hill_factor is None else hill_factor
        fixed = self._fixed_matrix()
        fp, fe = self._free_slots()
        fixed_key = fixed.copy()
        for p, e in zip(fp, fe):
            fixed_key[p, e] = 0.0
        whfast = {"ias15": 0, "whfast": 1}[self.integrator]
        key = (tuple(fp), tuple(fe), fixed_key.tobytes(), float(hf), whfast, float(self.dt), bool(self.dense_output))
        def make():
            m = _abi.ModelHandle(ctx, fixed, fp, fe, hf)
            if whfast or self.dt != 0.001:
                m.set_option("dt0", self.dt)
            if whfast:
                m.set_option("integrator", 1)
            if self.dense_output:
                m.set_option("dense_output", 1)
            return m
        # LRU cache on the context: eviction only drops the cache's reference; a handle still held by a caller (a
        # DeviceGroup, another thread) stays valid and is freed by its own finalizer
        return ctx.cached(ctx._models, key, make, limit=64)

    # ------------------------------------------------------------------ reference API
    def setup_sim(self):
        """The reference returns a rebound.Simulation ready to integrate (state.py:36-47).  The CUDA engine builds and
        integrates the simulation on the device, so what is returned here is a read-only snapshot of that initial
        simulation: `.particles` (objects with m, x, y, z, vx, vy, vz; star first, barycentric frame, i.e. after
        move_to_com) and `.exit_min_distance`, computed by the same device code the integrating kernels start from."""
        parts, _ = self._model().initial_conditions(self.get_params()[None, :])
        hill = max(p["a"] * (p["m"] / 3.) ** (1. / 3.) for p in self.planets)
        self.hillRadiusMax = hill
        return _SimSnapshot(parts[0], self.hillRadiusFactor * hill)

    def _rv_no_encounter_check(self, times):
        model = self._model(hill_factor=0.0)
        rv, status = model.rv_curve(self.get_params()[None, :], times)
        if status[0] != _abi.RV_OK:
            raise _abi.RvGpuError("integration failed with status %d" % status[0])
        return rv[0]

    def get_rv(self, times):
        """RV of the star at `times`, visited in the given order (state.py:61-73)."""
        model = self._model()
        rv, status = model.rv_curve(self.get_params()[None, :], np.asarray(times, dtype=np.float64))
        if status[0] == _abi.RV_ENCOUNTER:
            raise Encounter("Two particles had a close encounter (d<exit_min_distance).")
        if status[0] != _abi.RV_OK:
            raise _abi.RvGpuError("integration failed with status %d" % status[0])
        return rv[0]

    def get_rv_plotting(self, obs, Npoints=1000):
        times = np.linspace(obs.tb[0], obs.tf[len(obs.tf) - 1], Npoints)
        a = None
        try:
            a = self.get_rv(times)
        except Encounter:
            print("You are trying to plot a set parameters which give a collision.")
        return times, a

    def get_chi2(self, obs):
        """state.py:89-98: two fresh integrations (obs.tf, then obs.tb in its stored order), summed on the host."""
        rvf = self.get_rv(obs.tf)
        rvb = self.get_rv(obs.tb)
        chi2f = 0.
        chi2b = 0.
        for i in range(len(obs.tf)):
            chi2f += ((rvf[i] - obs.rvf[i]) ** 2.) / (obs.errorf[i] ** 2.)
        for i in range(len(obs.tb)):
            chi2b += ((rvb[i] - obs.rvb[i]) ** 2.) / (obs.errorb[i] ** 2.)
        return (chi2b + chi2f) / (obs.Npoints)

    def get_logp(self, obs):
        """state.py:103-110 -- one fused kernel evaluation (prior, both legs, chi2)."""
        if self.priorHard():
            return -np.inf
        softlnpri = 0.0
        if self.logp is None:
            ctx = _abi.default_context()
            logp, status = self._model(ctx).loglik(obs._handle(ctx), self.get_params()[None, :])
            if status[0] == _abi.RV_ENCOUNTER:
                raise Encounter("Two particles had a close encounter (d<exit_min_distance).")
            if status[0] != _abi.RV_OK:
                raise _abi.RvGpuError("likelihood evaluation failed with status %d" % status[0])
            self.logp = float(logp[0])
        return self.logp + softlnpri

    @staticmethod
    def lnprior(theta):
        m, a, h, k, l = theta
        if (1e-7 < m < 0.1) and (1e-2 < a < 500.0) and ((h ** 2 + k ** 2) < 1.0) and (-2 * np.pi < l < 2 * np.pi):
            return 0.0
        return -np.inf

    def shift_params(self, vec):
        self.logp = None
        if len(vec) != self.Nvars:
            raise AttributeError("vector has wrong length")
        varindex = 0
        for i, planet in enumerate(self.planets):
            for k in planet.keys():
                if self._is_free(i, k):
                    self.planets[i][k] += vec[varindex]
                    varindex += 1

    def get_params(self):
        params = np.zeros(self.Nvars)
        parindex = 0
        for i, planet in enumerate(self.planets):
            for k in planet.keys():
                if self._is_free(i, k):
                    params[parindex] = self.planets[i][k]
                    parindex += 1
        return params

    def set_params(self, vec):
        self.logp = None
        if len(vec) != self.Nvars:
            raise AttributeError("vector has wrong length")
        varindex = 0
        for i, planet in enumerate(self.planets):
            for k in planet.keys():
                if self._is_free(i, k):
                    self.planets[i][k] = vec[varindex]
                    varindex += 1

    def get_keys(self):
        keys = [""] * self.Nvars
        parindex = 0
        for i, planet in enumerate(self.planets):
            for k in planet.keys():
                if self._is_free(i, k):
                    keys[parindex] = "$%s_%d$" % (k, i)
                    parindex += 1
        return keys

    def get_rawkeys(self):
        keys = [""] * self.Nvars
        parindex = 0
        for i, planet in enumerate(self.planets):
            for k in planet.keys():
                if self._is_free(i, k):
                    keys[parindex] = k
                    parindex += 1
        return keys

    def deepcopy(self):
        # NB like the reference (state.py:212-213) the copy is a fresh State: hillRadiusFactor is back to 1.
        c = State(copy.deepcopy(self.planets), copy.deepcopy(self.ignore_vars),
                  ignore_params=copy.deepcopy(self.ignore_params))
        if self.integrator != "ias15":
            c.integrator, c.dt = self.integrator, self.dt
        if self.dense_output:
            c.dense_output = True
        return c

    def var_pindex_vname(self, vindex):
        vi = 0
        for pindex, p in enumerate(self.planets_vars):
            for v in p:
                if vindex == vi:
                    return pindex + 1, v
                vi += 1

    def get_chi2_d_dd(self, obs):
        """state.py:253-285 -- chi2, its gradient and Hessian from one fused variational kernel evaluation
        (real system + Nvars first-order + Nvars(Nvars+1)/2 second-order sets; forward leg, then a fresh
        monotone backward leg).  Like the reference, no prior test here (callers do it, mcmc.py:171)."""
        ctx = _abi.default_context()
        model = self._model(ctx)
        logp, grad, hess, status = model.loglik_d_dd(obs._handle(ctx), self.get_params()[None, :], check_prior=False)
        if status[0] == _abi.RV_ENCOUNTER:
            raise Encounter("Two particles had a close encounter (d<exit_min_distance).")
        if status[0] != _abi.RV_OK:
            raise _abi.RvGpuError("variational evaluation failed with status %d" % status[0])
        return -float(logp[0]), -grad[0], -hess[0]

    def get_logp_d_dd(self, obs):
        if self.logp is None or self.logp_d is None:
            chi, chi_d, chi_dd = self.get_chi2_d_dd(obs)
            self.logp, self.logp_d, self.logp_dd = -chi, -chi_d, -chi_dd
        return self.logp, self.logp_d, self.logp_dd

    def find_map(self, obs, **kw):
        """Maximum-likelihood fit started at this state (ModelHandle.map_fit; keyword arguments max_iter, n_trial, tol,
        damping).  Not in the reference.  Returns a new State at the optimum with logp / logp_d / logp_dd cached, `fit_code`
        (RV_FIT_*) and `laplace_cov` (-inv(logp_dd) when the fit converged, else None).  Like get_logp, the evaluation keeps
        this state's hillRadiusFactor.  Raises Encounter / RvGpuError when the start itself does not evaluate."""
        ctx = _abi.default_context()
        r = self._model(ctx).map_fit(obs._handle(ctx), self.get_params()[None, :], **kw)
        if r["fit_code"][0] == _abi.RV_FIT_NOSTART:
            if r["status"][0] == _abi.RV_ENCOUNTER:
                raise Encounter("Two particles had a close encounter (d<exit_min_distance).")
            raise _abi.RvGpuError("the fit's start does not evaluate (status %d)" % r["status"][0])
        return self._fitted(r, 0)

    def _fitted(self, r, w):
        """New State at walker w of a map_fit result, with this state's hillRadiusFactor (the fit is an evaluation like
        get_logp, not a sampler, so deepcopy's reset to 1 does not apply)."""
        st = self.deepcopy()
        st.hillRadiusFactor = self.hillRadiusFactor
        st.set_params(r["theta"][w])
        st.logp, st.logp_d, st.logp_dd = float(r["logp"][w]), r["grad"][w].copy(), r["hess"][w].copy()
        st.fit_code = int(r["fit_code"][w])
        st.n_iter = int(r["n_iter"][w])
        st.laplace_cov = np.linalg.inv(-st.logp_dd) if st.fit_code == _abi.RV_FIT_CONVERGED else None
        return st

    def priorHard(self):
        """state.py:299-315."""
        for i, planet in enumerate(self.planets):
            if self.planets[i]["a"] <= 0.02:
                if self.verbose_prior:
                    print("Invalid state was proposed (a)")
                return True
            if self.planets[i]["m"] <= 5e-6:
                if self.verbose_prior:
                    print("Invalid state was proposed (m)")
                return True
            if "h" in planet or "k" in planet:
                if self.planets[i]["h"] ** 2 + self.planets[i]["k"] ** 2 >= 1.0:
                    if self.verbose_prior:
                        print("Invalid state was proposed (h & k)")
                    return True
            if "ix" in planet or "iy" in planet:
                if self.planets[i]["ix"] ** 2 + self.planets[i]["iy"] ** 2 >= 4.0:
                    if self.verbose_prior:
                        print("Invalid state was proposed (ix & iy)")
                    return True
        return False
