"""numpy restatement of the batched maximum-likelihood fit (rv_map_fit; DESIGN.md 3.6), the checker of the device fit.

`evaluate(X) -> (logp[m], grad[m][n], hess[m][n][n], status[m])` is State.get_logp_d_dd with the hard prior tested, and
`plain(X) -> (logp[m], status[m])` State.get_logp, both for a batch of rows (the CPU oracle through tests/rvtest.py).
Walkers are independent; they are batched here only so that the oracle's threads are used.  Test infrastructure only.
"""
import numpy as np

CONVERGED, MAXITER, STALLED, SADDLE, NOSTART = 0, 1, 2, 3, 4
RUNNING = -1
EIG_FLOOR, MU_MIN, MU_MAX = 1e-12, 1e-6, 1.0


def step(th, g, H, mu, n_iter, max_iter, tol, n_trial):
    """(code, rows[n_trial + 1][n], decrement): RUNNING with the trial rows, or the code the walker stops with."""
    lam, Q = np.linalg.eigh(-0.5 * (H + H.T))
    lmax = np.abs(lam).max()
    rows = np.tile(th, (n_trial + 1, 1))
    if not (lmax > 0) or not np.isfinite(lmax):
        return SADDLE, rows, 0.0
    lt0 = np.maximum(np.abs(lam), EIG_FLOOR * lmax)
    y = Q.T @ g
    dec = float(np.sum(y * y / lt0))
    if not (0.5 * dec > tol):
        return (CONVERGED if lam.min() > EIG_FLOOR * lmax else SADDLE), rows, dec
    if n_iter >= max_iter:
        return MAXITER, rows, dec
    d = Q @ (y / (lt0 + mu * lmax))
    rows[1:] = th[None, :] + (2.0 ** -np.arange(n_trial))[:, None] * d[None, :]
    return RUNNING, rows, dec


def select(rows, tlogp, tstatus, mu, n_iter):
    """(moved, theta, mu, n_iter, code) after the line search over one walker's rows."""
    ok = np.flatnonzero(tstatus[1:] == 0) + 1
    if len(ok):
        best = ok[np.argmax(tlogp[ok])]          # argmax takes the first maximum: the lowest j on ties
        if tlogp[best] > tlogp[0]:
            mu = mu / 10.0
            return True, rows[best].copy(), (0.0 if mu < MU_MIN else mu), n_iter + 1, RUNNING
    mu = max(10.0 * mu, MU_MIN)
    return False, rows[0].copy(), mu, n_iter, (STALLED if mu > MU_MAX else RUNNING)


def map_fit(evaluate, plain, theta0, max_iter=50, n_trial=8, tol=1e-10, damping=0.0, trace=None):
    """The device loop: evaluate the walkers that moved, step every running walker, one plain evaluation of all trial
    rows, select.  Returns dict(theta, logp, grad, hess, status, fit_code, n_iter).  trace (a list) receives, per
    iteration, {walker: (rows, trial logps, trial statuses)}."""
    theta = np.array(theta0, dtype=np.float64, ndmin=2)
    W, n = theta.shape
    logp = np.zeros(W); grad = np.zeros((W, n)); hess = np.zeros((W, n, n)); status = np.zeros(W, dtype=np.int32)
    code = np.full(W, RUNNING); iters = np.zeros(W, dtype=np.int32); mu = np.full(W, float(damping))
    run = list(range(W)); ev = list(range(W))
    while run:
        if ev:
            lo, go, ho, so = evaluate(theta[ev])
            for s, w in enumerate(ev):
                logp[w], grad[w], hess[w], status[w] = lo[s], go[s], ho[s], so[s]
                if so[s] != 0:
                    code[w] = NOSTART if iters[w] == 0 else STALLED
        rows = {}
        for w in run:
            if code[w] != RUNNING:
                continue
            c, r, _ = step(theta[w], grad[w], hess[w], mu[w], iters[w], max_iter, tol, n_trial)
            if c != RUNNING:
                code[w] = c
            else:
                rows[w] = r
        nxt, ev = [], []
        if rows:
            ws = list(rows)
            tl, ts = plain(np.vstack([rows[w] for w in ws]))
            tl = tl.reshape(len(ws), n_trial + 1); ts = ts.reshape(len(ws), n_trial + 1)
            if trace is not None:
                trace.append({w: (rows[w], tl[i], ts[i]) for i, w in enumerate(ws)})
            for i, w in enumerate(ws):
                moved, theta[w], mu[w], iters[w], code[w] = select(rows[w], tl[i], ts[i], mu[w], iters[w])
                if code[w] == RUNNING:
                    nxt.append(w)
                if moved:
                    ev.append(w)
        run = nxt
    return dict(theta=theta, logp=logp, grad=grad, hess=hess, status=status, fit_code=code.astype(np.int32), n_iter=iters)
