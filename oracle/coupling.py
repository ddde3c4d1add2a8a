"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference coupling path.

Functional restatement (numpy / torch-CPU / scipy) of what
``torchcfm.optimal_transport.OTPlanSampler`` does around the POT solver, so that
the parity tests and bench.py's CPU baseline can run where the reference
package is not installed.  Every function cites the reference lines it
follows.  tests/test_oracle.py checks this file against the committed fixtures in
tests/golden/, which the unmodified reference package (on top of oracle/ot) wrote.

PARITY STATUS: exact-OT pinned (scipy LSA, reference tests, golden fixtures
generated from the reference glue).  Sinkhorn plan values: parity unpinned at the
POT boundary (see oracle/ot/__init__.py).
"""
import math
import warnings

import numpy as np
import torch

from . import ot as _ot


def flatten2d(x):
    """optimal_transport.py:80-83 -- (bs, *dim) -> (bs, prod(dim))."""
    return x.reshape(x.shape[0], -1) if x.dim() > 2 else x


def cost_matrix(x0, x1, normalize_cost=False):
    """optimal_transport.py:84-86 -- squared Euclidean cost, fp32, via cdist."""
    M = torch.cdist(flatten2d(x0), flatten2d(x1)) ** 2
    if normalize_cost:
        M = M / M.max()
    return M


def solve_plan(M, method="exact", reg=0.05, sinkhorn_method="sinkhorn", warn=True,
               **solver_kw):
    """optimal_transport.py:79,87-96 -- marginals, solver call and the guards.

    ``sinkhorn_method`` selects POT's kernel-space ('sinkhorn', what the
    reference calls) or log-domain ('sinkhorn_log', what north_star targets)
    algorithm.  Returns the float64 (n0, n1) plan.
    """
    Mn = M.detach().cpu().numpy() if torch.is_tensor(M) else np.asarray(M)
    a, b = _ot.unif(Mn.shape[0]), _ot.unif(Mn.shape[1])
    if method == "exact":
        p = _ot.emd(a, b, Mn)
    elif method == "sinkhorn":
        p = _ot.sinkhorn(a, b, Mn, reg=reg, method=sinkhorn_method, **solver_kw)
    else:
        raise ValueError(f"Unknown method: {method}")
    if abs(p.sum()) < 1e-8:
        if warn:
            warnings.warn("Numerical errors in OT plan, reverting to uniform plan.")
        p = np.ones_like(p) / p.size
    return p


def draw_pairs(pi, batch_size, replace=True):
    """optimal_transport.py:116-121 -- multinomial draw over the flattened plan
    using the global legacy NumPy RNG, then divmod into (row, col)."""
    p = pi.flatten()
    p = p / p.sum()
    k = np.random.choice(pi.shape[0] * pi.shape[1], p=p, size=batch_size, replace=replace)
    return np.divmod(k, pi.shape[1])


def sample_plan(x0, x1, method="exact", reg=0.05, normalize_cost=False, replace=True,
                sinkhorn_method="sinkhorn", **solver_kw):
    """optimal_transport.py:123-145 -- full coupling: cost, plan, draw, gather."""
    M = cost_matrix(x0, x1, normalize_cost)
    pi = solve_plan(M, method, reg, sinkhorn_method, **solver_kw)
    i, j = draw_pairs(pi, x0.shape[0], replace)
    return x0[i], x1[j], i, j


def trajectory_chain(X, method="exact", reg=0.05, normalize_cost=False, sinkhorn_method="sinkhorn",
                     **solver_kw):
    """optimal_transport.py:221-251 -- chain of per-sample conditional draws across the populations
    X[:, 0], X[:, 1], ...: all plans first (:233-236), then for every transition one
    ``np.random.choice(n, p=pi[i] / pi[i].sum())`` per sample, in order (:239-248).  Returns the
    index chain [(bs,) int arrays] and the stacked (bs, times, *dim) NumPy array (:249-251)."""
    times = X.shape[1]
    pis = [solve_plan(cost_matrix(X[:, t], X[:, t + 1], normalize_cost), method, reg, sinkhorn_method,
                      **solver_kw) for t in range(times - 1)]
    chain = [np.arange(X.shape[0])]
    for pi in pis:
        chain.append(np.array([np.random.choice(pi.shape[1], p=pi[i] / pi[i].sum()) for i in chain[-1]]))
    Xn = X.detach().cpu().numpy() if torch.is_tensor(X) else np.asarray(X)
    return chain, np.stack([Xn[:, t][chain[t]] for t in range(times)], axis=1)


def assignment(M):
    """optimal_transport.py:179 -- sigma from scipy's exact LSA on float64 costs."""
    from scipy.optimize import linear_sum_assignment
    Mn = M.detach().cpu().numpy() if torch.is_tensor(M) else np.asarray(M)
    return linear_sum_assignment(Mn.astype(np.float64))[1]


def wasserstein(x0, x1, method=None, reg=0.05, power=2):
    """optimal_transport.py:254-303."""
    assert power in (1, 2)
    M = torch.cdist(flatten2d(x0), flatten2d(x1))
    if power == 2:
        M = M ** 2
    Mn = M.detach().cpu().numpy()
    a, b = _ot.unif(Mn.shape[0]), _ot.unif(Mn.shape[1])
    if method == "exact" or method is None:
        ret = _ot.emd2(a, b, Mn, numItermax=int(1e7))
    elif method == "sinkhorn":
        ret = _ot.sinkhorn2(a, b, Mn, reg=reg, numItermax=int(1e7))
    else:
        raise ValueError(f"Unknown method: {method}")
    return math.sqrt(ret) if power == 2 else ret


# ----- flow-matcher formulas (conditional_flow_matching.py) --------------------

def _pad(t, x):
    """conditional_flow_matching.py:17-38."""
    if isinstance(t, (float, int)):
        return t
    return t.reshape(-1, *([1] * (x.dim() - 1)))


def matcher_xt_ut(kind, x0, x1, t, eps, sigma):
    """Closed forms of (xt, ut) for the five matchers.

    i_cfm / exact_ot_cfm: conditional_flow_matching.py:62-83,104-129,131-154
    t_cfm:                :329-394        sb_cfm: :429-478       vp_cfm: :569-618
    """
    tp = _pad(t, x0)
    if kind in ("i_cfm", "exact_ot_cfm"):
        mu = tp * x1 + (1 - tp) * x0
        xt = mu + _pad(sigma, x0) * eps
        ut = x1 - x0
    elif kind == "t_cfm":
        mu = tp * x1
        st = 1 - (1 - sigma) * tp
        xt = mu + st * eps
        ut = (x1 - (1 - sigma) * xt) / (1 - (1 - sigma) * tp)
    elif kind == "sb_cfm":
        mu = tp * x1 + (1 - tp) * x0
        st = _pad(sigma * torch.sqrt(t * (1 - t)), x0)
        xt = mu + st * eps
        ut = (1 - 2 * tp) / (2 * tp * (1 - tp) + 1e-8) * (xt - mu) + x1 - x0
    elif kind == "vp_cfm":
        c, s = torch.cos(math.pi / 2 * tp), torch.sin(math.pi / 2 * tp)
        mu = c * x0 + s * x1
        xt = mu + _pad(sigma, x0) * eps
        ut = math.pi / 2 * (c * x1 - s * x0)
    else:
        raise ValueError(kind)
    return xt, ut
