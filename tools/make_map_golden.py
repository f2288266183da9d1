"""Writes tests/golden/hd155358_map_multistart.json: the maximum-likelihood fit of HD155358 (hill factor 2) computed by the
numpy restatement of the device fit (oracle/map_oracle.py) on the CPU oracle -- the single fit from the published solution
HD_SOL and 16 starts HD_SOL + HD_SCALE_VEC * N(0,1) from np.random.default_rng(5) (driver.find_map_gpu's ball, width 1).
Fit settings are the defaults of ModelHandle.map_fit.  A few CPU minutes."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import map_oracle as M  # noqa: E402
import rvtest as T  # noqa: E402

Z2 = np.zeros((2, 7))
SETTINGS = dict(max_iter=50, n_trial=8, tol=1e-10, damping=0.0)
SEED, NSTARTS = 5, 16


def oracle_fns(obs, hill=2.0):
    def evaluate(X):
        lo, go, ho, so, _ = T.orc_logp_d_dd_batch(Z2, T.FP10, T.FE10, hill, obs, X)
        return lo, go, ho, so

    def plain(X):
        lo, so, _ = T.orc_logp_batch(Z2, T.FP10, T.FE10, hill, obs, X)
        return lo, so
    return evaluate, plain


def starts():
    rng = np.random.default_rng(SEED)
    return np.array(T.HD_SOL)[None, :] + np.array(T.HD_SCALE_VEC)[None, :] * rng.normal(size=(NSTARTS, 10))


def _rows(r):
    return [dict(theta=r["theta"][w].tolist(), logp=float(r["logp"][w]), fit_code=int(r["fit_code"][w]),
                 n_iter=int(r["n_iter"][w]), status=int(r["status"][w])) for w in range(len(r["logp"]))]


def main():
    obs = T.load_vels("HD155358.vels")
    evaluate, plain = oracle_fns(obs)
    single = M.map_fit(evaluate, plain, np.array(T.HD_SOL)[None, :], **SETTINGS)
    X = starts()
    multi = M.map_fit(evaluate, plain, X, **SETTINGS)
    out = dict(source="tools/make_map_golden.py (oracle/map_oracle.py on the CPU oracle)", data="HD155358.vels",
               hill_factor=2.0, settings=SETTINGS, seed=SEED, width=1.0, center="HD_SOL", scales="HD_SCALE_VEC",
               single=_rows(single)[0], starts=X.tolist(), multistart=_rows(multi))
    path = os.path.join(ROOT, "tests", "golden", "hd155358_map_multistart.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("single: code %d n_iter %d logp %.11f" % (single["fit_code"][0], single["n_iter"][0], single["logp"][0]))
    for w in range(NSTARTS):
        print(w, multi["fit_code"][w], multi["n_iter"][w], "%.11f" % multi["logp"][w])


if __name__ == "__main__":
    main()
