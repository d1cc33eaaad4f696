"""Independent dense multivariate-normal likelihood on a network.

TEST INFRASTRUCTURE (see oracle/__init__.py).  This is the cross-check the
reference's own tests use in their comments (`vcv(net)` + `MvNormal`,
test/test_evomodels.jl:265-316, test/test_calibration.jl:119-124,167-175): the
joint covariance of all node states is built by the network recursion

    Cov(X_i, X_j) = sum_k gamma_k Cov(X_pa_k, X_j)                (j before i)
    Var(X_i)      = sum_k gamma_k^2 t_k R_k + sum_kl gamma_k gamma_l Cov(X_pa_k, X_pa_l)

and the tip block is factorised densely.  It shares no code with the belief
propagation path.
"""
from __future__ import annotations

import math

import numpy as np

LOG2PI = math.log(2 * math.pi)


def network_covariance(net, rate_of_edge, p, rootvar=None):
    """(n*p x n*p) covariance of all node states, node-major / trait-minor, in
    preorder.  rate_of_edge(edge) -> p x p variance rate."""
    pre = net.vec_node
    n = len(pre)
    idx = {id(v): i for i, v in enumerate(pre)}
    C = np.zeros((n * p, n * p))
    if rootvar is not None:
        C[:p, :p] = rootvar
    for i in range(1, n):
        v = pre[i]
        pes = v.parent_edges()
        sl = slice(i * p, (i + 1) * p)
        for j in range(i):
            sj = slice(j * p, (j + 1) * p)
            blk = np.zeros((p, p))
            for e in pes:
                k = idx[id(e.parent)]
                blk += e.gamma * C[k * p:(k + 1) * p, sj]
            C[sl, sj] = blk
            C[sj, sl] = blk.T
        var = np.zeros((p, p))
        for e in pes:
            var += e.gamma ** 2 * e.length * rate_of_edge(e)
            k = idx[id(e.parent)]
            for e2 in pes:
                l = idx[id(e2.parent)]
                var += e.gamma * e2.gamma * C[k * p:(k + 1) * p, l * p:(l + 1) * p]
        C[sl, sl] = var
    return C


def loglik_bm(net, tbl, taxa, rate_of_edge, mu, rootvar=None, improper=False):
    """Log-likelihood of tip data `tbl` (ntaxa x p, NaN = missing).
    rootvar=None/0 => fixed root at mu; improper=True => flat prior on the root
    mean (restricted likelihood, what an infinite root variance gives)."""
    tbl = np.asarray(tbl, dtype=float)
    p = tbl.shape[1]
    mu = np.atleast_1d(np.asarray(mu, dtype=float))
    C = network_covariance(net, rate_of_edge, p, None if improper else rootvar)
    idx = {v.name: i for i, v in enumerate(net.vec_node)}
    sel, y, tr = [], [], []
    for r, name in enumerate(taxa):
        for t in range(p):
            if not math.isnan(tbl[r, t]):
                sel.append(idx[name] * p + t)
                y.append(tbl[r, t])
                tr.append(t)
    sel = np.array(sel)
    y = np.array(y)
    S = C[np.ix_(sel, sel)]
    L = np.linalg.cholesky(S)
    ld = 2 * float(np.sum(np.log(np.diag(L))))
    n = y.size
    if not improper:
        r = np.linalg.solve(L, y - mu[tr])
        return -(n * LOG2PI + ld + float(r @ r)) / 2
    X = np.zeros((n, p))
    X[np.arange(n), tr] = 1.0
    LX = np.linalg.solve(L, X)
    Ly = np.linalg.solve(L, y)
    A = LX.T @ LX
    beta = np.linalg.solve(A, LX.T @ Ly)
    r = Ly - LX @ beta
    _, ldA = np.linalg.slogdet(A)
    return -((n - p) * LOG2PI + ld + ldA + float(r @ r)) / 2


def ou_moments(net, sigma2, alpha, theta, mu, v=0.0):
    """Moments of all node states under the univariate Ornstein-Uhlenbeck model, nodes in preorder:
    (m, w, C) with X = m + w (X_root - mu) + noise of covariance C, where C has the root variance v in
    C[0, 0] (0 for a fixed root and for v = inf: an improper root enters through w only).  Per parent edge k
    of node i, with expm1 so that the moments stay exact as alpha -> 0:

        q_k = exp(-alpha t_k),  omega_k = (1 - q_k) theta,  var_k = sigma2 / (2 alpha) (1 - q_k^2)
        m_i = sum_k gamma_k (q_k m_pa(k) + omega_k),     w_i = sum_k gamma_k q_k w_pa(k)
        C_ij = sum_k gamma_k q_k C_pa(k),j  (j before i)
        C_ii = sum_k gamma_k^2 var_k + sum_kl gamma_k gamma_l q_k q_l C_pa(k),pa(l)."""
    pre = net.vec_node
    n = len(pre)
    idx = {id(x): i for i, x in enumerate(pre)}
    m, w, C = np.zeros(n), np.zeros(n), np.zeros((n, n))
    m[0], w[0] = mu, 1.0
    C[0, 0] = v if math.isfinite(v) else 0.0
    rate = sigma2 / (2 * alpha)
    for i in range(1, n):
        ks, cq, om, var = [], [], 0.0, 0.0
        for e in pre[i].parent_edges():
            q = math.exp(-alpha * e.length)
            k = idx[id(e.parent)]
            ks.append(k)
            cq.append(e.gamma * q)
            om += e.gamma * (-math.expm1(-alpha * e.length) * theta)
            var += e.gamma ** 2 * (rate * -math.expm1(-2 * alpha * e.length))
        cq = np.array(cq)
        m[i] = cq @ m[ks] + om
        w[i] = cq @ w[ks]
        C[i, :i] = cq @ C[ks, :i]
        C[:i, i] = C[i, :i]
        C[i, i] = var + cq @ C[np.ix_(ks, ks)] @ cq
    return m, w, C


def loglik_ou(net, tbl, taxa, sigma2, alpha, theta, mu, v=0.0):
    """Log-likelihood of the tip values `tbl` (one per taxon, NaN = missing) under the univariate OU model:
    v = 0 fixed root at mu, 0 < v < inf proper prior N(mu, v), v = inf flat prior on the root (the likelihood
    integrated over the root value: with S the covariance of the observed tips, c = m - w mu and r the GLS
    residual of y - c on w, -((n-1) log 2pi + log|S| + log(w'S^-1 w) + r'S^-1 r)/2)."""
    y = np.asarray(tbl, dtype=float).ravel()
    m, w, C = ou_moments(net, sigma2, alpha, theta, mu, v)
    idx = {x.name: i for i, x in enumerate(net.vec_node)}
    obs = np.array([idx[name] for name, yi in zip(taxa, y) if not math.isnan(yi)])
    y = y[~np.isnan(y)]
    L = np.linalg.cholesky(C[np.ix_(obs, obs)])
    ld = 2 * float(np.sum(np.log(np.diag(L))))
    n = y.size
    if math.isfinite(v):
        r = np.linalg.solve(L, y - m[obs])
        return -(n * LOG2PI + ld + float(r @ r)) / 2
    Lw = np.linalg.solve(L, w[obs])
    Lr = np.linalg.solve(L, y - (m[obs] - w[obs] * mu))
    ww = float(Lw @ Lw)
    r = Lr - Lw * (float(Lw @ Lr) / ww)
    return -((n - 1) * LOG2PI + ld + math.log(ww) + float(r @ r)) / 2
