"""driver -- Python-3 mirror of the reference's driver.py loops and diagnostics (no plotting).

run_mh / run_emcee / run_smala / run_alsmala keep the reference's loop shape, chain layout and
McmcBundle fields (driver.py:20-200); the autocorrelation-time, efficacy and KS helpers keep its
definitions (driver.py:37-44, 343-425).  Plot functions are out of scope (matplotlib is not a
dependency of the hot path).
"""
import hashlib
from datetime import datetime, timezone

import numpy as np

from . import mcmc, observations

def _utcnow():
    """Naive UTC timestamp, what the reference's datetime.utcnow() returned (driver.py:64)."""
    return datetime.now(timezone.utc).replace(tzinfo=None)



class McmcBundle(object):
    def __init__(self, mcmc, chain, chainlogp, clocktimes, obs, Niter, initial_state, trimmedchain=None,
                 trimmedchainlogp=None, actimes=None, is_emcee=False, Nwalkers=32):
        self.mcmc = mcmc
        self.mcmc_is_emcee = is_emcee
        self.mcmc_Nwalkers = Nwalkers
        self.mcmc_chain = chain
        self.mcmc_chainlogp = chainlogp
        self.mcmc_clocktimes = clocktimes
        self.mcmc_obs = obs
        self.mcmc_Niter = Niter
        self.mcmc_initial_state = initial_state
        self.mcmc_trimmedchain = trimmedchain
        self.mcmc_trimmedchainlogp = trimmedchainlogp
        self.mcmc_actimes = actimes


def auto_correlation(x):
    x = np.asarray(x)
    y = x - x.mean()
    result = np.correlate(y, y, mode='full')
    result = result[len(result) // 2:]
    result /= result[0]
    return result


def _run_id(true_state, label):
    h = hashlib.md5()
    h.update(str(true_state.planets).encode())
    h.update(str(label).encode())
    return h


def _single_chain(sampler, label, Niter, true_state, obs, printing_every, stepper=None):
    chain = np.zeros((Niter + 1, sampler.state.Nvars))
    chainlogp = np.zeros(Niter + 1)
    tries = 0
    clocktimes = [_utcnow()]
    chainlogp[0] = true_state.get_logp(obs)
    chain[0] = true_state.get_params()
    for i in range(Niter):
        if (stepper(i) if stepper else sampler.step()):
            tries += 1
        chainlogp[i + 1] = sampler.state.get_logp(obs)
        chain[i + 1] = sampler.state.get_params()
        if i % printing_every == 1:
            print("Progress: {p:.5}%, {n} accepted steps have been made, time: {t}".format(
                p=100. * (float(i) / Niter), t=_utcnow(), n=tries))
            clocktimes.append(_utcnow())
    clocktimes.append(_utcnow())
    print("Acceptance rate: %.3f%%" % ((tries / float(Niter)) * 100))
    h = _run_id(true_state, label)
    return McmcBundle(sampler, chain, chainlogp, clocktimes, obs, Niter, true_state), h


def run_mh(label, Niter, true_state, obs, scal, step, printing_every=400):
    mh = mcmc.Mh(true_state, obs)
    mh.set_scales(scal)
    mh.step_size = step
    return _single_chain(mh, label, Niter, true_state, obs, printing_every)


def run_emcee(label, Niter, true_state, obs, Nwalkers, scal, printing_every=400):
    ens = mcmc.Ensemble(true_state, obs, scales=scal, nwalkers=Nwalkers)
    nsteps = int(Niter / Nwalkers)
    listchain = np.zeros((Nwalkers, ens.state.Nvars, nsteps))
    listchainlogp = np.zeros((Nwalkers, nsteps))
    clocktimes = [_utcnow()]
    for i in range(nsteps):
        ens.step()
        listchainlogp[:, i] = ens.lnprob
        listchain[:, :, i] = ens.states
        if i % printing_every == 1:
            print("Progress: {p:.5}%, time: {t}".format(p=100. * (float(i) / nsteps), t=_utcnow()))
            clocktimes.append(_utcnow())
    clocktimes.append(_utcnow())
    print("Error(s): {e}".format(e=ens.totalErrorCount))
    h = _run_id(true_state, label)
    # walker-major concatenation, as driver.py:108-112
    chain = np.concatenate([listchain[i] for i in range(Nwalkers)], axis=1)
    chainlogp = np.concatenate([listchainlogp[i] for i in range(Nwalkers)])
    bundle = McmcBundle(ens, np.transpose(chain), chainlogp, clocktimes, obs, Niter, true_state, is_emcee=True,
                        Nwalkers=Nwalkers)
    return bundle, h


def run_smala(label, Niter, true_state, obs, eps, alpha, printing_every=40):
    smala = mcmc.Smala(true_state, obs, eps, alpha)
    return _single_chain(smala, label, Niter, true_state, obs, printing_every)


def run_alsmala(label, Niter, true_state, obs, eps, alpha, bern_a, bern_b, printing_every=40):
    alsmala = mcmc.Alsmala(true_state, obs, eps, alpha)

    def stepper(i):
        if np.exp(-bern_a * i / Niter) > np.random.uniform():
            return alsmala.step()
        return alsmala.step_mala()
    return _single_chain(alsmala, label, Niter, true_state, obs, printing_every, stepper)


# ---------------------------------------------------------------------------------------------------------------
# Fused device drivers: the same bundles as run_mh / run_emcee / run_smala / run_alsmala, but the whole propose --
# evaluate -- accept loop of `nchains` chains (or one ensemble) runs on the GPU in ONE library call
# (rv_mh_run / rv_stretch_run / rv_smala_run / rv_alsmala_run) instead of one Python iteration per step.  Chains are laid
# out walker-major like run_emcee's (driver.py:108-112), so ac_times / efficacy / calc_kstatistic apply unchanged.
# Random numbers are the library's counter-based streams (seed), not numpy's global state.

def _bundle_from_device(sampler_name, r, lp_key, true_state, obs, Niter, nchains, label, t0):
    chain, chain_lp = r["chain"], r[lp_key]                      # [steps][W][nvars], [steps][W]
    flat = np.concatenate([chain[:, w, :] for w in range(nchains)], axis=0)
    flat_lp = np.concatenate([chain_lp[:, w] for w in range(nchains)])
    bundle = McmcBundle(sampler_name, flat, flat_lp, [t0, _utcnow()], obs, Niter, true_state, is_emcee=True,
                        Nwalkers=nchains)
    bundle.device_result = r
    return bundle, _run_id(true_state, label)


def _scale_vector(state, scal):
    return np.array([scal[k] for k in state.get_rawkeys()], dtype=np.float64)


def _sampler_state(true_state, fast=False):
    """The state a sampler object would hold: Mcmc.__init__ deep-copies the initial state (mcmc.py:13), and the reference's
    deepcopy builds a fresh State, so hillRadiusFactor is back to 1 for everything the sampler evaluates (state.py:212-213).
    fast=True selects the dense-output likelihood (State.dense_output: same logp to ~1e-12, ~1.65x the throughput on
    HD155358) instead of the reference's one-truncated-step-per-epoch sequence."""
    st = true_state.deepcopy()
    if fast:
        st.dense_output = True
    return st


def run_mh_gpu(label, Niter, true_state, obs, scal, step, nchains=1, seed=0, fast=False):
    """`nchains` independent MH chains of Niter steps each (Mh.step semantics, mcmc.py:107-121), all started at true_state."""
    from . import _abi
    ctx = _abi.default_context()
    t0 = _utcnow()
    r = _sampler_state(true_state, fast)._model(ctx).mh_run(obs._handle(ctx), np.tile(true_state.get_params(), (nchains, 1)),
                                                      _scale_vector(true_state, scal), step, Niter, seed=seed)
    print("Acceptance rate: %.3f%%" % (100. * r["n_accept"].mean() / max(Niter, 1)))
    return _bundle_from_device("mh", r, "chain_logp", true_state, obs, Niter * nchains, nchains, label, t0)


def run_emcee_gpu(label, Niter, true_state, obs, Nwalkers, scal, seed=0, fast=False):
    """One affine-stretch ensemble of Nwalkers (Ensemble + run_emcee, mcmc.py:40-75, driver.py:86-120): Niter/Nwalkers
    ensemble steps from the reference's start ball theta + 1e-3*scales*N(0,1) (mcmc.py:49-51, numpy RNG as there)."""
    from . import _abi
    ctx = _abi.default_context()
    t0 = _utcnow()
    sc = _scale_vector(true_state, scal)
    start = np.array([true_state.get_params() + 1e-3 * sc * np.random.normal(size=true_state.Nvars) for _ in range(Nwalkers)])
    nsteps = int(Niter / Nwalkers)
    r = _sampler_state(true_state, fast)._model(ctx).stretch_run(obs._handle(ctx), start, nsteps, seed=seed)
    return _bundle_from_device("emcee", r, "chain_lnp", true_state, obs, Niter, Nwalkers, label, t0)


def run_smala_gpu(label, Niter, true_state, obs, eps, alpha, nchains=1, seed=0):
    """`nchains` independent SMALA chains (Smala.step, mcmc.py:167-187)."""
    from . import _abi
    ctx = _abi.default_context()
    t0 = _utcnow()
    r = _sampler_state(true_state)._model(ctx).smala_run(obs._handle(ctx), np.tile(true_state.get_params(), (nchains, 1)),
                                                         eps, alpha, Niter, seed=seed)
    print("Acceptance rate: %.3f%%" % (100. * r["n_accept"].mean() / max(Niter, 1)))
    return _bundle_from_device("smala", r, "chain_logp", true_state, obs, Niter * nchains, nchains, label, t0)


def run_alsmala_gpu(label, Niter, true_state, obs, eps, alpha, bern_a, bern_b=None, nchains=1, seed=0):
    """`nchains` ALSMALA chains under run_alsmala's schedule exp(-bern_a*i/Niter) (driver.py:171-200; bern_b is unused there)."""
    from . import _abi
    ctx = _abi.default_context()
    t0 = _utcnow()
    r = _sampler_state(true_state)._model(ctx).alsmala_run(obs._handle(ctx), np.tile(true_state.get_params(), (nchains, 1)),
                                                           eps, alpha, bern_a, Niter, niter_total=Niter, seed=seed)
    print("Acceptance rate: %.3f%%" % (100. * r["n_accept"].mean() / max(Niter, 1)))
    return _bundle_from_device("alsmala", r, "chain_logp", true_state, obs, Niter * nchains, nchains, label, t0)


def find_map_gpu(true_state, obs, nstarts, scal, width=1.0, seed=0, **kw):
    """Multi-start maximum-likelihood fit (ModelHandle.map_fit; keyword arguments max_iter, n_trial, tol, damping) from the
    ball true_state + width*scales*N(0,1), drawn from np.random.default_rng(seed).  Not in the reference.

    Returns dict(results, maxima).  results: the per-start arrays of map_fit plus `start`, sorted by logp (highest first).
    maxima: the distinct converged maxima, highest first; converged starts are grouped greedily in that order -- a start
    joins the first group whose best point it lies within 0.1 Laplace sigma of in every coordinate (that best point's
    covariance) -- and each maximum is dict(state, theta, logp, count, cov, sigma)."""
    from . import _abi
    ctx = _abi.default_context()
    sc = _scale_vector(true_state, scal)
    rng = np.random.default_rng(seed)
    start = true_state.get_params()[None, :] + width * sc[None, :] * rng.normal(size=(nstarts, true_state.Nvars))
    r = true_state._model(ctx).map_fit(obs._handle(ctx), start, **kw)
    r["start"] = start
    order = np.argsort(-r["logp"], kind="stable")
    results = {k: v[order] for k, v in r.items()}
    maxima = []
    for w in range(nstarts):
        if results["fit_code"][w] != _abi.RV_FIT_CONVERGED:
            continue
        th = results["theta"][w]
        for g in maxima:
            if np.all(np.abs(th - g["theta"]) <= 0.1 * g["sigma"]):
                g["count"] += 1
                break
        else:
            st = true_state._fitted(results, w)
            cov = st.laplace_cov
            maxima.append(dict(state=st, theta=th, logp=st.logp, count=1, cov=cov, sigma=np.sqrt(np.diag(cov))))
    return dict(results=results, maxima=maxima)


def create_obs(state, npoint, err, errVar, t):
    return observations.FakeObservation(state, Npoints=npoint, error=err, errorVar=errVar, tmax=t)


def read_obs(filen):
    return observations.Observation_FromFile(filename=filen, Npoints=100)


def save_obs(obs, true_state, label):
    """.vels writer (driver.py:215-222; the reference writes the rv column twice -- fixed here: col3 = err)."""
    col1 = obs.t / 1.720e-2
    col2 = obs.rv / 3.355e-5
    col3 = obs.err / 3.355e-5
    h = _run_id(true_state, label)
    name = 'obs_{ha}.vels'.format(ha=h.hexdigest())
    np.savetxt(name, np.c_[col1, col2, col3])
    return name


def ac_time(series):
    """First lag at which the normalised autocorrelation drops below 0.5 (driver.py:366-377)."""
    r = auto_correlation(series)
    below = np.nonzero(r < 0.5)[0]
    return int(below[0]) if len(below) else len(r)


def ac_times(bundle):
    """Per-parameter AC times as plot_ACTimes computes them (driver.py:343-382): an ensemble bundle uses mcmc_chain and
    averages the per-walker AC times (walker-major blocks of Niter/Nwalkers rows); a single chain uses the trimmed chain
    (mcmc_trimmedchain) when one is set, else the whole chain.  Stored on bundle.mcmc_actimes and returned."""
    if bundle.mcmc_is_emcee:
        chain = bundle.mcmc_chain
        nw = bundle.mcmc_Nwalkers
        per = chain.shape[0] // nw
        out = np.array([np.mean([ac_time(chain[w * per:(w + 1) * per, j]) for w in range(nw)])
                        for j in range(chain.shape[1])])
    else:
        chain = bundle.mcmc_trimmedchain if bundle.mcmc_trimmedchain is not None else bundle.mcmc_chain
        out = np.array([float(ac_time(chain[:, j])) for j in range(chain.shape[1])])
    bundle.mcmc_actimes = out
    return out


def plot_ACTimes(bundle, size=None, name='Name_left_empty', save=False):
    """The reference's entry point for AC times (driver.py:343-382) without the figure: prints and stores them."""
    act = ac_times(bundle)
    for t in act:
        print("AC time {t}".format(t=t))
    return act


def efficacy(Niter, AC, clockTimes):
    """Niter / (wall seconds * max AC time), wall clock from the SECOND stamp to the last (driver.py:412-414)."""
    dt = (clockTimes[len(clockTimes) - 1] - clockTimes[1]).total_seconds()
    return (Niter / (dt * np.amax(AC)))


def calc_kstatistic(chain1, chain2, verbose=False):
    """Two-sample KS test per parameter (driver.py:423-425 prints scipy's result; here the D statistics are returned)."""
    from scipy import stats
    out = []
    for i in range(len(np.transpose(chain1))):
        r = stats.ks_2samp(np.transpose(chain1)[i], np.transpose(chain2)[i])
        if verbose:
            print(r)
        out.append(r[0])
    return out


# ---- persistence (driver.py:46-54, 429-448): same file names and formats as the reference ------------------------

def save_data(dat, name, h):
    """np.save of one array under '<name>_<md5>.npy' (driver.py:432-433)."""
    np.save('{n}_{h}'.format(n=name, h=h.hexdigest()), dat)


def load_data(name, h):
    """Inverse of save_data (driver.py:429-430)."""
    return np.load('{n}_{h}.npy'.format(n=name, h=h.hexdigest()))


def save_bundle(bundle, h):
    """chain, chainlogp and clocktimes of a bundle, the three arrays the notebooks store per run."""
    save_data(bundle.mcmc_chain, "chain", h)
    save_data(bundle.mcmc_chainlogp, "chainlogp", h)
    save_data(np.array([t.isoformat() for t in bundle.mcmc_clocktimes]), "clocktimes", h)


def writing_to_log(obj, name, logging):
    """Append every element of `obj` (np.ndenumerate order), space separated, as one line of 'log<name>'
    (driver.py:46-54, mcmc_benchmark_mh.py:21-28; the reference's version raises NameError on a typo)."""
    if not logging:
        return
    with open("log{r}".format(r=name), "a") as a:
        for _, value in np.ndenumerate(obj):
            a.write("{v} ".format(v=value))
        a.write("\n")


def _save_aux(h, true_state, line):
    with open('aux_{h}'.format(h=h.hexdigest()), "w") as text_file:
        text_file.write('initial = ' + str(true_state.planets))
        text_file.write(line)


def save_aux_smala(h, true_state, label, Niter, eps, alpha):
    _save_aux(h, true_state, "\nlabel, Niter, Eps, Alpha = '{l}', {n}, {e}, {a}".format(l=label, n=Niter, e=eps, a=alpha))


def save_aux_emcee(h, true_state, label, Niter, Nwalkers, scal):
    _save_aux(h, true_state, "\nlabel, Niter, Nwalkers, Scale = '{l}', {n}, {s}, {t}".format(l=label, n=Niter, s=Nwalkers, t=scal))


def save_aux_mh(h, true_state, label, Niter, scal, step):
    _save_aux(h, true_state, "\nlabel, Niter, Scale, Stepsize = '{l}', {n}, {s}, {t}".format(l=label, n=Niter, s=scal, t=step))
