"""Several GPUs from ONE Python process (the reference is a single process; `script.sh` only backgrounds 8 unrelated
jobs).  A DeviceGroup owns one rv_ctx per visible GPU and shards a batch of parameter vectors / independent chains over
them by contiguous blocks, one host thread per GPU (ctypes releases the GIL during the library call).  Nothing crosses
GPUs: MH / SMALA chains and likelihood batches are independent, and the random streams are keyed by the GLOBAL chain id,
so the results are bit-identical to a single-GPU run.  The affine stretch ensemble needs one exchange per half-step:
DeviceGroup.stretch_run is one call into rv_stretch_run_multi: a full copy of the ensemble on every GPU, accepted walkers
stored into all copies by the accept kernel itself over peer-mapped memory (NVLink P2P), half-steps ordered by events;
under torchrun (one process per GPU), samplers.stretch_run_sharded does the exchange with an NCCL all-gather."""
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from . import _abi
from .samplers import chain_shard


class DeviceGroup(object):
    def __init__(self, devices=None):
        if devices is None:
            import ctypes as C
            lib = _abi.load()
            devices = []
            d = 0
            while True:          # probe devices until rv_ctx_create refuses
                h = C.c_void_p()
                if lib.rv_ctx_create(d, C.byref(h)) != 0:
                    break
                lib.rv_ctx_destroy(h)
                devices.append(d)
                d += 1
            if not devices:
                raise _abi.RvGpuError("no usable GPU: %s" % lib.rv_last_error(None).decode())
        self.devices = list(devices)
        self.ctxs = [_abi.Context(d) for d in self.devices]
        self.pool = ThreadPoolExecutor(len(self.ctxs))

    def __len__(self):
        return len(self.ctxs)

    def close(self):
        self.pool.shutdown()
        for c in self.ctxs:
            c.close()

    def _handles(self, state, obs):
        return [(state._model(c), _obs_handle(obs, c)) for c in self.ctxs]

    def _map(self, W, fn):
        """fn(rank, lo, hi) on every GPU's block of [0, W); returns the list of results in rank order."""
        shards = [chain_shard(W, r, len(self.ctxs)) for r in range(len(self.ctxs))]
        futs = [self.pool.submit(fn, r, lo, hi) for r, (lo, hi) in enumerate(shards) if hi > lo]
        return [f.result() for f in futs]

    # ---- State.get_logp / get_logp_d_dd for a batch -------------------------------------------------------------
    def loglik(self, state, obs, theta):
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        hs = self._handles(state, obs)
        parts = self._map(len(theta), lambda r, lo, hi: hs[r][0].loglik(hs[r][1], theta[lo:hi]))
        return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])

    def loglik_d_dd(self, state, obs, theta):
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        hs = self._handles(state, obs)
        parts = self._map(len(theta), lambda r, lo, hi: hs[r][0].loglik_d_dd(hs[r][1], theta[lo:hi]))
        return tuple(np.concatenate([p[k] for p in parts]) for k in range(4))

    def map_fit(self, state, obs, theta, **kw):
        """ModelHandle.map_fit with the starts sharded over the GPUs (every walker's fit is independent)."""
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        hs = self._handles(state, obs)
        parts = self._map(len(theta), lambda r, lo, hi: hs[r][0].map_fit(hs[r][1], theta[lo:hi], **kw))
        return {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}

    # ---- independent chains -------------------------------------------------------------------------------------
    @staticmethod
    def _merge(parts):
        out = {}
        for k in parts[0]:
            vals = [p[k] for p in parts]
            if vals[0] is None:
                out[k] = None
            elif k in ("chain", "chain_logp", "accepted"):
                out[k] = np.concatenate(vals, axis=1)          # [steps][W][...]
            else:
                out[k] = np.concatenate(vals, axis=0)
        return out

    def mh_run(self, state, obs, theta, scales, step_size, nsteps, seed=0, logp=None, first_chain_id=0, **kw):
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        hs = self._handles(state, obs)
        if logp is not None:
            logp = np.ascontiguousarray(logp, dtype=np.float64)
            if logp.shape != (len(theta),):
                raise ValueError("logp must hold one value per chain")
        # per-chain arguments are sliced with the chains; the RNG streams are keyed by the GLOBAL chain id
        return self._merge(self._map(len(theta), lambda r, lo, hi: hs[r][0].mh_run(
            hs[r][1], theta[lo:hi], scales, step_size, nsteps, seed=seed, first_chain_id=first_chain_id + lo,
            logp=None if logp is None else logp[lo:hi], **kw)))

    def smala_run(self, state, obs, theta, eps, alpha, nsteps, seed=0, first_chain_id=0, **kw):
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        hs = self._handles(state, obs)
        return self._merge(self._map(len(theta), lambda r, lo, hi: hs[r][0].smala_run(
            hs[r][1], theta[lo:hi], eps, alpha, nsteps, seed=seed, first_chain_id=first_chain_id + lo, **kw)))


def _stretch_run(group, state, obs, theta0, nsteps, a=2.0, seed=0, first_step=0, thin=1, lnp=None, record_chain=False):
    """One library call (rv_stretch_run_multi): every GPU keeps a full copy of the ensemble, a slice's accept kernel stores
    its accepted walkers into all copies over peer memory, events order the half-steps -- no host synchronisation and no
    separate exchange inside the loop."""
    hs = group._handles(state, obs)
    return _abi.stretch_run_multi([m for m, _ in hs], [o for _, o in hs], theta0, nsteps, a=a, seed=seed, first_step=first_step,
                                  thin=thin, lnp=lnp, record_chain=record_chain)


DeviceGroup.stretch_run = _stretch_run


def _obs_handle(obs, ctx):
    """One rv_obs per context, from that context's content-keyed cache (closed with the context)."""
    return ctx.obs_handle(obs)
