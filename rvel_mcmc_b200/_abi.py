"""ctypes binding of librvgpu.so (include/rvgpu.h).

This is the analogue of rebound's own ctypes layer (``clibrebound.reb_integrate(byref(sim), c_double(tmax))``
reached from state.py:71): one thin call per *batch* of parameter vectors instead of one per epoch.
"""
import collections
import ctypes as C
import hashlib
import os
import threading
import weakref

import numpy as np

RV_OK, RV_PRIOR, RV_ENCOUNTER, RV_NONFINITE, RV_NOT_SPD = 0, 1, 3, 8, 9
RV_FIT_CONVERGED, RV_FIT_MAXITER, RV_FIT_STALLED, RV_FIT_SADDLE, RV_FIT_NOSTART = 0, 1, 2, 3, 4   # rv_map_fit fit codes
ELEMS = ("m", "a", "h", "k", "l", "ix", "iy")       # ABI slot order (RV_EL_*)
MAX_PLANETS = 5          # RV_MAX_PLANETS (plain likelihood, MH, stretch, WHFast)
MAX_PLANETS_VAR = 5      # RV_MAX_PLANETS_VAR (gradient + Hessian, SMALA)


class RvGpuError(RuntimeError):
    """The CUDA library is missing or a call into it failed (there is no CPU fallback)."""


class Encounter(Exception):
    """Two bodies came closer than exit_min_distance (mirrors rebound.Encounter; mcmc.py:119,176)."""


def lib_path():
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "librvgpu.so")


_lib = None
_lib_lock = threading.RLock()       # re-entrant: default_context() -> Context() -> load()
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)

_SIGNATURES = {
    "rv_ctx_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "rv_ctx_destroy": (C.c_int, [C.c_void_p]),
    "rv_last_error": (C.c_char_p, [C.c_void_p]),
    "rv_ctx_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_double]),
    "rv_device_info": (C.c_int, [C.c_void_p, _ip, _ip, _ip, _ip]),
    "rv_obs_create": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_int, C.c_double, C.POINTER(C.c_void_p)]),
    "rv_obs_destroy": (C.c_int, [C.c_void_p]),
    "rv_model_create": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_double,
                                  C.c_int, C.POINTER(C.c_void_p)]),
    "rv_model_destroy": (C.c_int, [C.c_void_p]),
    "rv_model_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_double]),
    "rv_loglik": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "rv_loglik_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                C.c_void_p]),
    "rv_loglik_d_dd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "rv_loglik_d_dd_opt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p]),
    "rv_loglik_d_dd_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p]),
    "rv_map_fit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_double,
                             C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rv_initial_conditions": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "rv_rv_curve": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p,
                              C.c_void_p]),
    "rv_mh_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_double,
                            C.c_uint64, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p,
                            C.c_void_p, C.c_void_p]),
    "rv_smala_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                               C.c_uint64, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p]),
    "rv_alsmala_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                 C.c_double, C.c_int64, C.c_uint64, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int64,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "rv_stretch_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_double,
                                 C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int64, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "rv_stretch_half_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_uint64, C.c_void_p,
                                      C.c_int64, C.c_void_p, C.c_double, C.c_uint64, C.c_uint32, C.c_uint32,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "rv_stretch_run_multi": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                       C.c_double, C.c_uint64, C.c_uint32, C.c_int, C.c_int, C.c_int64, C.c_void_p,
                                       C.c_void_p, C.c_void_p]),
    "rv_mh_steps_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double,
                                  C.c_uint64, C.c_uint64, C.c_uint32, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]),
    "rv_dev_alloc": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]),
    "rv_dev_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "rv_dev_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "rv_dev_download": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "rv_dev_copy_peer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "rv_work_counters": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.c_int]),
    "rv_count_work": (C.c_int, [C.c_void_p, C.c_int]),
    "rv_fp64_peak": (C.c_int, [C.c_void_p, _dp]),
    "rv_sync": (C.c_int, [C.c_void_p]),
    "rv_ctx_stream": (C.c_void_p, [C.c_void_p]),
}


def exported_symbols():
    """Every entry point include/rvgpu.h declares (used by the CPU-side load test)."""
    return sorted(_SIGNATURES)


def load():
    """Load librvgpu.so; raises RvGpuError if it has not been built (no fallback)."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        path = lib_path()
        if not os.path.exists(path):
            raise RvGpuError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                             "(rvel_mcmc_b200 has no CPU fallback)" % path)
        lib = C.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            try:
                fn = getattr(lib, name)
            except AttributeError:
                continue          # optional entry points are checked where they are used
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class Context(object):
    """One GPU (rv_ctx).  Calls are synchronous; one Context per host thread / rank."""

    def __init__(self, device=0):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.rv_ctx_create(int(device), C.byref(h))
        if rc != 0:
            raise RvGpuError("rv_ctx_create failed (%d): %s" % (rc, self.lib.rv_last_error(None).decode()))
        self.h = h
        self.device = int(device)
        # Handle bookkeeping: every rv_obs / rv_model created on this context is tracked weakly and destroyed with it;
        # the caches below only hold references (eviction drops a reference, it never frees a handle somebody else
        # still uses -- the handle's own finalizer does that once it is unreferenced).
        self._handles = weakref.WeakSet()
        self._models = collections.OrderedDict()        # State schema key -> ModelHandle (LRU, see State._model)
        self._obs = collections.OrderedDict()           # observation content digest -> ObsHandle (LRU, see obs_handle)
        self._lock = threading.RLock()

    def check(self, rc, what):
        if rc != 0:
            raise RvGpuError("%s failed (%d): %s" % (what, rc, self.lib.rv_last_error(self.h).decode()))

    def device_info(self):
        v = [C.c_int32() for _ in range(4)]
        self.check(self.lib.rv_device_info(self.h, *[C.byref(x) for x in v]), "rv_device_info")
        return dict(sm_count=v[0].value, cc=(v[1].value, v[2].value), clock_khz=v[3].value)

    def fp64_peak_tflops(self):
        out = C.c_double()
        self.check(self.lib.rv_fp64_peak(self.h, C.byref(out)), "rv_fp64_peak")
        return out.value

    def count_work(self, enable=True):
        self.check(self.lib.rv_count_work(self.h, 1 if enable else 0), "rv_count_work")

    def work_counters(self, reset=False):
        out = (C.c_uint64 * 2)()
        self.check(self.lib.rv_work_counters(self.h, out, 1 if reset else 0), "rv_work_counters")
        return int(out[0]), int(out[1])

    def sync(self):
        self.check(self.lib.rv_sync(self.h), "rv_sync")

    def set_option(self, key, value):
        self.check(self.lib.rv_ctx_set_option(self.h, key.encode(), float(value)), "rv_ctx_set_option")

    def chain_rows_width(self, W, chain_walkers):
        """Sets the context's chain_walkers option for the next sampler call; returns the recorded width."""
        cw = int(chain_walkers) if chain_walkers else 0
        self.set_option("chain_walkers", cw)
        return min(cw, W) if cw > 0 else W

    # ---- plain device buffers (addresses as ints) ----
    def dev_alloc(self, nbytes):
        p = C.c_void_p()
        self.check(self.lib.rv_dev_alloc(self.h, int(nbytes), C.byref(p)), "rv_dev_alloc")
        return p.value or 0

    def dev_free(self, addr):
        self.check(self.lib.rv_dev_free(self.h, C.c_void_p(addr)), "rv_dev_free")

    def dev_upload(self, addr, array):
        a = np.ascontiguousarray(array)
        self.check(self.lib.rv_dev_upload(self.h, C.c_void_p(addr), _ptr(a), a.nbytes), "rv_dev_upload")

    def dev_download(self, array, addr):
        assert array.flags["C_CONTIGUOUS"]
        self.check(self.lib.rv_dev_download(self.h, _ptr(array), C.c_void_p(addr), array.nbytes), "rv_dev_download")

    def dev_copy_to(self, dst_ctx, dst_addr, src_addr, nbytes):
        self.check(self.lib.rv_dev_copy_peer(dst_ctx.h, C.c_void_p(dst_addr), self.h, C.c_void_p(src_addr), int(nbytes)),
                   "rv_dev_copy_peer")

    def cached(self, cache, key, make, limit=64):
        """LRU lookup in one of this context's handle caches (thread-safe)."""
        with self._lock:
            h = cache.get(key)
            if h is not None and getattr(h, "h", None):
                cache.move_to_end(key)
                return h
            h = make()
            cache[key] = h
            while len(cache) > limit:
                cache.popitem(last=False)              # drop OUR reference only
            return h

    def obs_handle(self, obs):
        """rv_obs for an Observation-like object, keyed on the CONTENT of its arrays: editing or replacing
        obs.rvf / errorf / tf ... (same length or not) re-uploads; the reference reads obs on every call."""
        arrays = [_f64(getattr(obs, k)) for k in ("tf", "rvf", "errorf", "tb", "rvb", "errorb")]
        dg = hashlib.blake2b(digest_size=16)
        for a in arrays:
            dg.update(np.int64(a.size).tobytes()); dg.update(a.tobytes())
        dg.update(np.float64(obs.Npoints).tobytes())
        return self.cached(self._obs, dg.digest(), lambda: ObsHandle(self, *arrays, obs.Npoints), limit=16)

    def close(self):
        if getattr(self, "h", None):
            with self._lock:
                for hd in list(self._handles):
                    hd.close()
                self._models.clear(); self._obs.clear()
            self.lib.rv_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _Handle(object):
    """Device object owned by a Context: destroyed explicitly, by its finalizer, or with the context."""
    _destroy = None

    def _register(self, ctx, h):
        self.ctx, self.h = ctx, h
        ctx._handles.add(self)

    def close(self):
        h, self.h = getattr(self, "h", None), None
        if h and getattr(self.ctx, "h", None):          # a closed context has already released its device memory
            getattr(self.ctx.lib, self._destroy)(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ObsHandle(_Handle):
    """Observation arrays resident in HBM (rv_obs)."""
    _destroy = "rv_obs_destroy"

    def __init__(self, ctx, tf, rvf, errf, tb, rvb, errb, npoints):
        self.ctx = ctx
        tf, rvf, errf, tb, rvb, errb = [_f64(x) for x in (tf, rvf, errf, tb, rvb, errb)]
        if not (len(tf) == len(rvf) == len(errf) and len(tb) == len(rvb) == len(errb)):
            raise ValueError("observation arrays of one leg must have equal lengths")
        self.nf, self.nb, self.npoints = len(tf), len(tb), float(npoints)
        h = C.c_void_p()
        ctx.check(ctx.lib.rv_obs_create(ctx.h, _ptr(tf), _ptr(rvf), _ptr(errf), len(tf), _ptr(tb), _ptr(rvb),
                                        _ptr(errb), len(tb), float(npoints), C.byref(h)), "rv_obs_create")
        self._register(ctx, h)


class ModelHandle(_Handle):
    """Parameter schema resident in HBM (rv_model)."""
    _destroy = "rv_model_destroy"

    def __init__(self, ctx, fixed, free_planet, free_elem, hill_factor, dims=0):
        self.ctx = ctx
        fixed = _f64(fixed).reshape(-1, len(ELEMS))
        self.n_planets = fixed.shape[0]
        fp = np.ascontiguousarray(free_planet, dtype=np.int32)
        fe = np.ascontiguousarray(free_elem, dtype=np.int32)
        self.nvars = len(fp)
        h = C.c_void_p()
        ctx.check(ctx.lib.rv_model_create(ctx.h, self.n_planets, _ptr(fixed), self.nvars, _ptr(fp), _ptr(fe),
                                          float(hill_factor), int(dims), C.byref(h)), "rv_model_create")
        self._register(ctx, h)

    def _theta(self, theta):
        theta = np.asarray(theta, dtype=np.float64)
        if self.nvars == 0:       # every element pinned: only the walker count matters
            return np.zeros((theta.shape[0] if theta.ndim >= 1 else 1, 0))
        return np.ascontiguousarray(theta.reshape(-1, self.nvars))

    def set_option(self, key, value):
        self.ctx.check(self.ctx.lib.rv_model_set_option(self.h, key.encode(), float(value)), "rv_model_set_option")

    def loglik(self, obs, theta):
        """theta[W][nvars] (host) -> (logp[W], status[W]); State.get_logp for a batch."""
        theta = self._theta(theta)
        W = theta.shape[0]
        logp = np.empty(W, dtype=np.float64)
        status = np.empty(W, dtype=np.int32)
        self.ctx.check(self.ctx.lib.rv_loglik(self.ctx.h, self.h, obs.h, _ptr(theta), W, _ptr(logp), _ptr(status)),
                       "rv_loglik")
        return logp, status

    def loglik_dev(self, obs, d_theta, W, d_logp, d_status, stream=None):
        """Device-pointer variant (ints from torch .data_ptr()), asynchronous on `stream` (a raw cudaStream_t
        value, e.g. torch.cuda.current_stream().cuda_stream; None = the context's own stream)."""
        if stream is None:
            stream = self.ctx.lib.rv_ctx_stream(self.ctx.h)
        self.ctx.check(self.ctx.lib.rv_loglik_dev(self.ctx.h, self.h, obs.h, C.c_void_p(d_theta), int(W),
                                                  C.c_void_p(d_logp), C.c_void_p(d_status),
                                                  C.c_void_p(stream) if stream else None), "rv_loglik_dev")

    def loglik_d_dd(self, obs, theta, check_prior=True):
        """theta[W][nvars] (host) -> (logp[W], grad[W][nvars], hess[W][nvars][nvars], status[W]);
        State.get_logp_d_dd for a batch (state.py:290-294)."""
        theta = self._theta(theta)
        W = theta.shape[0]
        logp = np.empty(W, dtype=np.float64)
        grad = np.zeros((W, self.nvars), dtype=np.float64)
        hess = np.zeros((W, self.nvars, self.nvars), dtype=np.float64)
        status = np.empty(W, dtype=np.int32)
        # the prior test is a per-call argument: the (possibly shared, cached) device model is never modified
        self.ctx.check(self.ctx.lib.rv_loglik_d_dd_opt(self.ctx.h, self.h, obs.h, _ptr(theta), W, 1 if check_prior else 0,
                                                       _ptr(logp), _ptr(grad), _ptr(hess), _ptr(status)), "rv_loglik_d_dd_opt")
        return logp, grad, hess, status

    def loglik_d_dd_dev(self, obs, d_theta, W, d_logp, d_grad, d_hess, d_status, stream=None):
        if stream is None:
            stream = self.ctx.lib.rv_ctx_stream(self.ctx.h)
        self.ctx.check(self.ctx.lib.rv_loglik_d_dd_dev(self.ctx.h, self.h, obs.h, C.c_void_p(d_theta), int(W),
                                                       C.c_void_p(d_logp), C.c_void_p(d_grad), C.c_void_p(d_hess),
                                                       C.c_void_p(d_status), C.c_void_p(stream) if stream else None),
                       "rv_loglik_d_dd_dev")

    def map_fit(self, obs, theta, max_iter=50, n_trial=8, tol=1e-10, damping=0.0):
        """Maximum-likelihood fit from every row of theta[W][nvars] (rv_map_fit: damped saddle-free Newton, batched line
        search).  Returns dict(theta, logp, grad, hess, status, fit_code, n_iter), per walker; -inv(hess) at a converged
        walker (fit_code RV_FIT_CONVERGED) is its Laplace covariance."""
        theta = self._theta(theta).copy()
        W = theta.shape[0]
        logp = np.zeros(W)
        grad = np.zeros((W, self.nvars))
        hess = np.zeros((W, self.nvars, self.nvars))
        status = np.zeros(W, dtype=np.int32)
        code = np.zeros(W, dtype=np.int32)
        n_iter = np.zeros(W, dtype=np.int32)
        self.ctx.check(self.ctx.lib.rv_map_fit(self.ctx.h, self.h, obs.h, _ptr(theta), W, int(max_iter), int(n_trial),
                                               float(tol), float(damping), _ptr(logp), _ptr(grad), _ptr(hess), _ptr(status),
                                               _ptr(code), _ptr(n_iter)), "rv_map_fit")
        return dict(theta=theta, logp=logp, grad=grad, hess=hess, status=status, fit_code=code, n_iter=n_iter)

    def initial_conditions(self, theta):
        """theta[W][nvars] -> (particles[W][P+1][7] = m,x,y,z,vx,vy,vz in the barycentric frame, status[W]);
        what State.setup_sim builds (state.py:36-47)."""
        theta = self._theta(theta)
        W = theta.shape[0]
        out = np.zeros((W, self.n_planets + 1, 7), dtype=np.float64)
        status = np.empty(W, dtype=np.int32)
        self.ctx.check(self.ctx.lib.rv_initial_conditions(self.ctx.h, self.h, _ptr(theta), W, _ptr(out), _ptr(status)),
                       "rv_initial_conditions")
        return out, status

    def rv_curve(self, theta, times):
        """theta[W][nvars], times[nt] -> (rv[W][nt], status[W]); State.get_rv for a batch."""
        theta = self._theta(theta)
        times = _f64(times)
        W, nt = theta.shape[0], len(times)
        rv = np.zeros((W, nt), dtype=np.float64)
        status = np.empty(W, dtype=np.int32)
        self.ctx.check(self.ctx.lib.rv_rv_curve(self.ctx.h, self.h, _ptr(theta), W, _ptr(times), nt, _ptr(rv),
                                                _ptr(status)), "rv_rv_curve")
        return rv, status

    # ---- fused device samplers -------------------------------------------------------------------
    def mh_run(self, obs, theta, scales, step_size, nsteps, seed=0, first_chain_id=0, first_step=0, thin=1,
               logp=None, record_chain=True, record_accepts=False, chain_walkers=None):
        """W independent Metropolis-Hastings chains (Mh.step, mcmc.py:107-121) run on the device.
        Returns dict(theta, logp, chain[nsteps//thin][W][nvars], chain_logp, n_accept[W], accepted[nsteps][W])."""
        theta = self._theta(theta).copy()
        W = theta.shape[0]
        have = logp is not None
        lp = _f64(logp).copy() if have else np.zeros(W)
        scales = _f64(scales)
        rows = nsteps // thin
        cw = self.ctx.chain_rows_width(W, chain_walkers)        # chain rows hold chains [0, chain_walkers) only
        chain = np.zeros((rows, cw, self.nvars)) if record_chain else None
        chain_lp = np.zeros((rows, cw)) if record_chain else None
        nacc = np.zeros(W, dtype=np.uint64)
        acc = np.zeros((nsteps, W), dtype=np.uint8) if record_accepts else None
        self.ctx.check(self.ctx.lib.rv_mh_run(self.ctx.h, self.h, obs.h, _ptr(theta), _ptr(lp), 1 if have else 0,
                                              _ptr(scales), float(step_size), int(seed), int(first_chain_id),
                                              int(first_step), int(nsteps), int(thin), W, _ptr(chain), _ptr(chain_lp),
                                              _ptr(nacc), _ptr(acc)), "rv_mh_run")
        return dict(theta=theta, logp=lp, chain=chain, chain_logp=chain_lp, n_accept=nacc, accepted=acc)

    def smala_run(self, obs, theta, eps, alpha, nsteps, seed=0, first_chain_id=0, first_step=0, thin=1,
                  record_chain=True, record_accepts=False, chain_walkers=None):
        """W independent SMALA chains (Smala.step, mcmc.py:167-187) run on the device.
        Returns dict(theta, logp, chain, chain_logp, n_accept[W], accepted[nsteps][W], status[W])."""
        theta = self._theta(theta).copy()
        W = theta.shape[0]
        lp = np.zeros(W)
        rows = nsteps // thin
        cw = self.ctx.chain_rows_width(W, chain_walkers)
        chain = np.zeros((rows, cw, self.nvars)) if record_chain else None
        chain_lp = np.zeros((rows, cw)) if record_chain else None
        nacc = np.zeros(W, dtype=np.uint64)
        acc = np.zeros((nsteps, W), dtype=np.uint8) if record_accepts else None
        status = np.zeros(W, dtype=np.int32)
        self.ctx.check(self.ctx.lib.rv_smala_run(self.ctx.h, self.h, obs.h, _ptr(theta), _ptr(lp), float(eps), float(alpha),
                                                 int(seed), int(first_chain_id), int(first_step), int(nsteps), int(thin), W,
                                                 _ptr(chain), _ptr(chain_lp), _ptr(nacc), _ptr(acc), _ptr(status)),
                       "rv_smala_run")
        return dict(theta=theta, logp=lp, chain=chain, chain_logp=chain_lp, n_accept=nacc, accepted=acc, status=status)

    def alsmala_run(self, obs, theta, eps, alpha, bern_a, nsteps, niter_total=0, seed=0, first_chain_id=0, first_step=0,
                    thin=1, record_chain=True, record_accepts=False):
        """W independent ALSMALA chains (Alsmala + run_alsmala's schedule, mcmc.py:191-234, driver.py:171-200) on the device.
        Returns smala_run's dict plus full_step[nsteps] (1 where the iteration was a full SMALA step)."""
        theta = self._theta(theta).copy()
        W = theta.shape[0]
        lp = np.zeros(W)
        rows = nsteps // thin
        cw = self.ctx.chain_rows_width(W, None)
        chain = np.zeros((rows, cw, self.nvars)) if record_chain else None
        chain_lp = np.zeros((rows, cw)) if record_chain else None
        nacc = np.zeros(W, dtype=np.uint64)
        acc = np.zeros((nsteps, W), dtype=np.uint8) if record_accepts else None
        status = np.zeros(W, dtype=np.int32)
        full = np.zeros(max(nsteps, 1), dtype=np.uint8)
        self.ctx.check(self.ctx.lib.rv_alsmala_run(self.ctx.h, self.h, obs.h, _ptr(theta), _ptr(lp), float(eps), float(alpha),
                                                   float(bern_a), int(niter_total), int(seed), int(first_chain_id),
                                                   int(first_step), int(nsteps), int(thin), W, _ptr(chain), _ptr(chain_lp),
                                                   _ptr(nacc), _ptr(acc), _ptr(status), _ptr(full)), "rv_alsmala_run")
        return dict(theta=theta, logp=lp, chain=chain, chain_logp=chain_lp, n_accept=nacc, accepted=acc, status=status,
                    full_step=full[:nsteps])

    def stretch_run(self, obs, theta, nsteps, a=2.0, seed=0, first_step=0, thin=1, lnp=None, record_chain=True,
                    record_accepts=False, chain_walkers=None):
        """Affine stretch ensemble (Ensemble.step, mcmc.py:57-65; emcee 2.2.1 move) run on the device."""
        theta = self._theta(theta).copy()
        W = theta.shape[0]
        have = lnp is not None
        lp = _f64(lnp).copy() if have else np.zeros(W)
        rows = nsteps // thin
        cw = self.ctx.chain_rows_width(W, chain_walkers)
        chain = np.zeros((rows, cw, self.nvars)) if record_chain else None
        chain_lp = np.zeros((rows, cw)) if record_chain else None
        nacc = np.zeros(W, dtype=np.uint64)
        acc = np.zeros((nsteps, W), dtype=np.uint8) if record_accepts else None
        self.ctx.check(self.ctx.lib.rv_stretch_run(self.ctx.h, self.h, obs.h, _ptr(theta), _ptr(lp), 1 if have else 0,
                                                   float(a), int(seed), int(first_step), int(nsteps), int(thin), W,
                                                   _ptr(chain), _ptr(chain_lp), _ptr(nacc), _ptr(acc)), "rv_stretch_run")
        return dict(theta=theta, lnp=lp, chain=chain, chain_lnp=chain_lp, n_accept=nacc, accepted=acc)

    def stretch_half_dev(self, obs, d_S, nS, id0_S, d_C, nC, d_lnp_S, a, seed, step, half, d_n_accept=0, d_accepted=0,
                         stream=None):
        if stream is None:
            stream = self.ctx.lib.rv_ctx_stream(self.ctx.h)
        self.ctx.check(self.ctx.lib.rv_stretch_half_dev(self.ctx.h, self.h, obs.h, C.c_void_p(d_S), int(nS), int(id0_S),
                                                        C.c_void_p(d_C), int(nC), C.c_void_p(d_lnp_S), float(a), int(seed),
                                                        int(step), int(half), C.c_void_p(d_n_accept) if d_n_accept else None,
                                                        C.c_void_p(d_accepted) if d_accepted else None,
                                                        C.c_void_p(stream) if stream else None), "rv_stretch_half_dev")

    def mh_steps_dev(self, obs, d_theta, d_logp, d_scales, step_size, seed, first_chain_id, first_step, nsteps, W,
                     d_n_accept=0, stream=None):
        if stream is None:
            stream = self.ctx.lib.rv_ctx_stream(self.ctx.h)
        self.ctx.check(self.ctx.lib.rv_mh_steps_dev(self.ctx.h, self.h, obs.h, C.c_void_p(d_theta), C.c_void_p(d_logp),
                                                    C.c_void_p(d_scales), float(step_size), int(seed), int(first_chain_id),
                                                    int(first_step), int(nsteps), int(W),
                                                    C.c_void_p(d_n_accept) if d_n_accept else None,
                                                    C.c_void_p(stream) if stream else None), "rv_mh_steps_dev")

def stretch_run_multi(models, obss, theta, nsteps, a=2.0, seed=0, first_step=0, thin=1, lnp=None, record_chain=True):
    """Affine stretch ensemble over several GPUs of this process (rv_stretch_run_multi): models[g] / obss[g] are the
    handles of GPU g (same schema and data on each).  Returns the dict of ModelHandle.stretch_run (without `accepted`);
    bit-identical to the single-GPU run."""
    G = len(models)
    ctx0 = models[0].ctx
    theta = models[0]._theta(theta).copy()
    W = theta.shape[0]
    have = lnp is not None
    lp = _f64(lnp).copy() if have else np.zeros(W)
    rows = nsteps // thin
    chain = np.zeros((rows, W, models[0].nvars)) if record_chain else None
    chain_lp = np.zeros((rows, W)) if record_chain else None
    nacc = np.zeros(W, dtype=np.uint64)
    arr = lambda hs: (C.c_void_p * G)(*[h.h for h in hs])
    ctx0.check(ctx0.lib.rv_stretch_run_multi(G, arr([m.ctx for m in models]), arr(models), arr(obss), _ptr(theta), _ptr(lp),
                                             1 if have else 0, float(a), int(seed), int(first_step), int(nsteps), int(thin), W,
                                             _ptr(chain), _ptr(chain_lp), _ptr(nacc)), "rv_stretch_run_multi")
    return dict(theta=theta, lnp=lp, chain=chain, chain_lnp=chain_lp, n_accept=nacc)


_default_ctx = None


def default_context():
    """Process-wide context on cuda:LOCAL_RANK (or 0)."""
    global _default_ctx
    with _lib_lock:
        if _default_ctx is None or not getattr(_default_ctx, "h", None):
            _default_ctx = Context(int(os.environ.get("LOCAL_RANK", "0")))
        return _default_ctx


def set_default_context(ctx):
    global _default_ctx
    _default_ctx = ctx
