"""Forward simulation down the network on the device (pgbp_simulate) against a numpy restatement of its contract.

The restatement below follows include/pgbp_b200.h (section "forward simulation") line by line: Philox4x32-10 with
Box-Muller, nodes in preorder, K1's factor for Brownian motion (coefficient 1 and t R_c for one parent, gamma_k and
gamma_k^2 t_k R_{c_k} for hybrids, sqrt(t0) chol_lower(R_c) when the parent edges share a colour) and the univariate
OU factor.  Independently of it, sample moments are checked against oracle/densemvn.py's network covariance, the
log-likelihood of simulated data against the dense likelihood and its expectation, and posterior node moments
against the simulated true values (coverage)."""
import json
import math
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import pgbp_b200  # noqa: E402
from harness import BACKENDS, Case, get_lib, synth_oracle_objects  # noqa: E402
from oracle import densemvn  # noqa: E402
from oracle import models as M  # noqa: E402
from oracle.network import readnewick  # noqa: E402
from workloads import synth  # noqa: E402

GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_goldens.json")))
MULLER = json.load(open(os.path.join(ROOT, "tests", "golden", "muller_2022.json")))
LAZ_TAXA = ["Mbuti", "Onge", "Karitiana", "MA1", "Loschbour", "European", "Stuttgart"]
MASK32 = np.uint64(0xFFFFFFFF)


def status(msg, pivot):
    return int(np.int32(np.uint32(((msg + 1) << 8) | (pivot & 0xFF))))


IMPROPER, BAD_RATE, BAD_HYBRID = status(0x7ffff7, 1), status(0x7ffffd, 1), status(0x7ffffc, 1)


# ------------------------------------------------------------------ restatement of the generator
def philox(c, k):
    """Philox4x32-10 of counter words c[0..3] and key words k[0..1] (numpy uint64 arrays holding 32-bit values)."""
    c0, c1, c2, c3 = (np.asarray(x, dtype=np.uint64) for x in c)
    k0, k1 = (np.asarray(x, dtype=np.uint64) for x in k)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & MASK32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & MASK32
        k0 = (k0 + np.uint64(0x9E3779B9)) & MASK32
        k1 = (k1 + np.uint64(0xBB67AE85)) & MASK32
    return c0, c1, c2, c3


def normals(seed, v, r, p):
    """z[len(r), p] of node v for replicates r (array), trait pair k from counter (v, k, r lo, r hi)."""
    s = np.uint64(int(seed) % 2 ** 64)
    r = np.asarray(r, dtype=np.uint64)
    z = np.empty((r.size, 2 * ((p + 1) // 2)))
    for k in range((p + 1) // 2):
        x0, x1, x2, x3 = philox((np.full_like(r, v), np.full_like(r, k), r & MASK32, r >> np.uint64(32)),
                                (s & MASK32, s >> np.uint64(32)))
        u1 = (((x0 >> np.uint64(5)) << np.uint64(26)) + (x1 >> np.uint64(6)) + np.uint64(1)).astype(float) * 2.0 ** -53
        u2 = (((x2 >> np.uint64(5)) << np.uint64(26)) + (x3 >> np.uint64(6))).astype(float) * 2.0 ** -53
        rho = np.sqrt(-2.0 * np.log(u1))
        z[:, 2 * k] = rho * np.cos(6.283185307179586 * u2)
        z[:, 2 * k + 1] = rho * np.sin(6.283185307179586 * u2)
    return z[:, :p]


def restate(fam, p, model, params, seed, first, B, ncolors=1):
    """(tipdata[B, ntips, p], nodes[B, nnodes, p], status[B]) of the header's contract."""
    n, mp = fam["nnodes"], fam["mem_parent"]
    off, gam, ln, col = fam["mem_off"], fam["mem_gamma"], fam["mem_length"], fam["mem_color"]
    params = np.atleast_2d(params)
    X = np.full((B, n, p), np.nan)
    st = np.zeros(B, dtype=np.int64)
    for e in range(B):
        rec = params[min(e, params.shape[0] - 1)]
        r = first + e
        if model == "ou":
            s2, al, th, mu, v = rec
            if not (s2 > 0 and al > 0):
                st[e] = BAD_RATE; continue
            if v == math.inf:
                st[e] = IMPROPER; continue
            for u in range(n):
                z = normals(seed, u, [r], 1)[0, 0]
                ks = range(off[u] + 1, off[u + 1])
                if u == 0:
                    X[e, 0, 0] = mu + (math.sqrt(v) * z if v > 0 else 0.0)
                    continue
                m = var = 0.0
                for k in ks:
                    g = 1.0 if len(ks) == 1 else gam[k]
                    m += g * (math.exp(-al * ln[k]) * X[e, mp[k], 0] - math.expm1(-al * ln[k]) * th)
                    var += g * g * s2 / (2 * al) * -math.expm1(-2 * al * ln[k])
                X[e, u, 0] = m + math.sqrt(var) * z
            continue
        pp = p * p
        R = [rec[c * pp:(c + 1) * pp].reshape(p, p).T for c in range(ncolors)]
        mu = rec[ncolors * pp:ncolors * pp + p]
        V = rec[ncolors * pp + p:].reshape(p, p).T
        try:
            Lc = [np.linalg.cholesky(Rc) for Rc in R]
        except np.linalg.LinAlgError:
            st[e] = BAD_RATE; continue
        if np.all(V == 0):
            LV = None
        elif np.any(np.diag(V) == math.inf):
            st[e] = IMPROPER; continue
        else:
            LV = np.linalg.cholesky(V)
        for u in range(n):
            ks = list(range(off[u] + 1, off[u + 1]))
            z = normals(seed, u, [r], p)[0]
            if u == 0:
                X[e, 0] = mu if LV is None else mu + LV @ z
                continue
            if len(ks) == 1:
                mean, t0 = X[e, mp[ks[0]]], ln[ks[0]]
            else:
                mean = sum(gam[k] * X[e, mp[k]] for k in ks)
                t0 = sum(gam[k] ** 2 * ln[k] for k in ks)
            if len({col[k] for k in ks}) == 1:
                X[e, u] = mean if t0 == 0 else mean + math.sqrt(t0) * (Lc[col[ks[0]]] @ z)
            else:
                S = sum(gam[k] ** 2 * ln[k] * R[col[k]] for k in ks)
                X[e, u] = mean + np.linalg.cholesky(S) @ z
    tips = np.full((B, fam["ntips"], p), np.nan)
    for u in range(n):
        if fam["node_datarow"][u] >= 0:
            tips[:, fam["node_datarow"][u]] = X[:, u]
    if fam.get("tip_missing") is not None:
        tm = np.asarray(fam["tip_missing"], dtype=bool).reshape(fam["ntips"], p)
        tips[:, tm] = np.nan
    return tips, X, st


def test_philox_known_answers():
    f = lambda c, k: ["%08x" % int(x) for x in philox(c, k)]  # noqa: E731
    assert f([0, 0, 0, 0], [0, 0]) == ["6627e8d5", "e169c58d", "bc57ac4c", "9b00dbd8"]
    assert f([0xffffffff] * 4, [0xffffffff] * 2) == ["408f276d", "41c83b0e", "a20bc7c6", "6d5451fd"]
    assert f([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        ["d16cfe09", "94fdcceb", "5001e420", "24126ea1"]
    # Box-Muller of the first vector: u1 = ((x0 >> 5) 2^26 + (x1 >> 6) + 1) 2^-53, u2 likewise without the + 1
    x0, x1, x2, x3 = 0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8
    u1 = (((x0 >> 5) << 26) + (x1 >> 6) + 1) * 2.0 ** -53
    u2 = (((x2 >> 5) << 26) + (x3 >> 6)) * 2.0 ** -53
    z = normals(0, 0, [0], 2)[0]
    rho = math.sqrt(-2 * math.log(u1))
    assert z[0] == rho * math.cos(6.283185307179586 * u2) and z[1] == rho * math.sin(6.283185307179586 * u2)


# ------------------------------------------------------------------ networks
def synth_case(ntips, nretic, seed, p, ncolors=1, root_fixed=True):
    """(network tables, edge colours, plan dict) of a level-1 network of workloads/synth.py and its clique tree; with
    ncolors > 1 every edge gets a random colour, so that hybrids' parent edges may differ in colour"""
    tab = synth.level1_network(ntips, nretic, seed)
    rng = np.random.default_rng(seed)
    col = {e: int(rng.integers(ncolors)) for par in tab["parents"] for (_, _, _, e) in par} if ncolors > 1 else None
    d = synth.cliquetree_plan(tab, p, root_fixed, col)
    return tab, col, d


def plan_of(d, lib):
    return pgbp_b200.ClusterGraphPlan(d["nclusters"], d["belief_dim"], d["sepset_clusters"], d["upind"], d["trees"],
                                      d["ntraits"], d["families"], lib)


def oracle_case(netstr, taxa, p, lib, method, **kw):
    model = M.MvFullBrownianMotion(np.eye(p), np.zeros(p)) if p > 1 else M.UnivariateBrownianMotion(1.0, 0.0)
    net = readnewick(netstr)
    return Case(net, method, np.zeros((len(taxa), p)), taxa, model, lib, **kw)


def rate(p, rng):
    A = rng.normal(size=(p, p))
    return A @ A.T / p + 0.2 * np.eye(p)


def bm_record(kind, p, ncolors, rng, root="fixed"):
    if kind == "univariate":
        Rs = [np.array([[rng.uniform(0.5, 2.0)]]) for _ in range(ncolors)]
    elif kind == "diag":
        Rs = [np.diag(rng.uniform(0.5, 2.0, size=p)) for _ in range(ncolors)]
    else:
        Rs = [rate(p, rng) for _ in range(ncolors)]
    mu = rng.normal(size=p)
    V = None if root == "fixed" else rate(p, rng)
    return pgbp_b200.bm_params(Rs, mu, V)


def close(a, b, tol=1e-12):
    a, b = np.asarray(a), np.asarray(b)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    ok = ~np.isnan(b)
    err = np.abs(a[ok] - b[ok]) / (1 + np.abs(b[ok]))
    assert err.size == 0 or err.max() <= tol, err.max()


def run(lib_plan, fam, p, params, seed, first, B, model="bm", ncolors=1, **kw):
    bt = pgbp_b200.BatchedClusterGraphBelief(lib_plan, B, **kw)
    tips, nodes = bt.simulate(params, seed, first, model=model, ncolors=ncolors, nodes=True)
    return tips, nodes, bt.status()


# ------------------------------------------------------------------ exact restatement
SYNTH = [(8, 0, 1), (10, 1, 2), (12, 2, 3), (14, 3, 4), (16, 4, 5)]
KINDS = [("univariate", 1), ("diag", 2), ("full", 3), ("full", 8), ("full", 16), ("diag", 16)]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("kind,p", KINDS, ids=lambda x: str(x))
@pytest.mark.parametrize("ntips,nretic,seed", SYNTH, ids=lambda x: str(x))
def test_restatement_synth_bm(backend, ntips, nretic, seed, kind, p):
    lib = get_lib(backend)
    _, _, d = synth_case(ntips, nretic, seed, p)
    fam = d["families"]
    rng = np.random.default_rng(seed * 100 + p)
    B = 5
    # nparamsets = B with a proper root, then 1 with a fixed root; replicates from an offset, seeds above 2^63
    params = np.stack([bm_record(kind, p, 1, rng, root="random") for _ in range(B)])
    pl = plan_of(d, lib)
    for prm, first, seed_ in ((params, 3, 0x1234_5678_9ABC), (params[:1] * 0 + bm_record(kind, p, 1, rng), 0, 2 ** 63 + 5)):
        tips, nodes, st = run(pl, fam, p, prm, seed_, first, B)
        rt, rn, rs = restate(fam, p, "bm", prm, seed_, first, B)
        assert (st == 0).all() and (rs == 0).all()
        close(tips, rt)
        close(nodes, rn)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("p", [1, 3])
def test_restatement_two_colours(backend, p):
    """two rate colours on a network whose hybrids' parent edges differ in colour (the per-thread Cholesky path)"""
    lib = get_lib(backend)
    for ntips, nretic, seed in ((12, 3, 7), (20, 4, 11)):
        tab, col, d = synth_case(ntips, nretic, seed, p, ncolors=2)
        fam = d["families"]
        mixed = [v for v in range(fam["nnodes"]) if len({fam["mem_color"][k] for k in range(fam["mem_off"][v] + 1, fam["mem_off"][v + 1])}) > 1]
        rng = np.random.default_rng(seed)
        B = 4
        params = np.stack([bm_record("full", p, 2, rng, root="random") for _ in range(B)])
        tips, nodes, st = run(plan_of(d, lib), fam, p, params, 99, 10, B, ncolors=2)
        rt, rn, _ = restate(fam, p, "bm", params, 99, 10, B, ncolors=2)
        assert (st == 0).all()
        close(tips, rt)
        close(nodes, rn)
        assert mixed, "the case must have a hybrid whose parent edges differ in colour"


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("name", ["lazaridis", "muller"])
def test_restatement_named_networks(backend, name):
    lib = get_lib(backend)
    if name == "lazaridis":
        case = oracle_case(GOLD["lazaridis"], LAZ_TAXA, 3, lib, "cliquetree", order_hint=GOLD["lazaridis_cluster_labels"])
        p = 3
    else:
        taxa = readnewick(MULLER["newick"]).tiplabels()
        case = oracle_case(MULLER["newick"], taxa, 1, lib, "bethe")
        p = 1
    fam = case.plan.families
    assert fam["mem_parent"][0] == -1
    rng = np.random.default_rng(5)
    B = 6
    params = np.stack([bm_record("full", p, 1, rng, root="random") for _ in range(B)])
    tips, nodes, st = run(case.plan, fam, p, params, 2024, 0, B)
    rt, rn, _ = restate(fam, p, "bm", params, 2024, 0, B)
    assert (st == 0).all()
    close(tips, rt)
    close(nodes, rn)


def ou_records(n, rng, root="fixed"):
    alpha = np.geomspace(1e-4, 50.0, n)
    mu = rng.normal(size=n)
    theta = mu + rng.choice([-1.0, 1.0], size=n) * rng.uniform(3.0, 6.0, size=n)
    v = np.zeros(n) if root == "fixed" else rng.uniform(0.2, 2.0, size=n)
    return np.stack([rng.uniform(0.5, 2.0, size=n), alpha, theta, mu, v], axis=1)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("root", ["fixed", "random"])
def test_restatement_ou(backend, root):
    lib = get_lib(backend)
    _, _, d = synth_case(14, 3, 21, 1)
    fam = d["families"]
    rng = np.random.default_rng(3)
    B = 9
    recs = ou_records(B, rng, root)
    pl = plan_of(d, lib)
    tips, nodes, st = run(pl, fam, 1, recs, 77, 1000, B, model="ou")
    rt, rn, _ = restate(fam, 1, "ou", recs, 77, 1000, B)
    assert (st == 0).all()
    close(tips, rt)
    close(nodes, rn)
    tips1, nodes1, _ = run(pl, fam, 1, recs[4], 77, 1000, B, model="ou")  # one record for all
    rt1, rn1, _ = restate(fam, 1, "ou", recs[4], 77, 1000, B)
    close(nodes1, rn1)


# ------------------------------------------------------------------ invariance
@pytest.mark.parametrize("backend", BACKENDS)
def test_invariance(backend):
    lib = get_lib(backend)
    p = 3
    _, _, d = synth_case(12, 3, 4, p)
    pl = plan_of(d, lib)
    rng = np.random.default_rng(0)
    prm = bm_record("full", p, 1, rng, root="random")
    big = pgbp_b200.BatchedClusterGraphBelief(pl, 300).simulate(prm, 42, nodes=True)
    for r in (0, 1, 31, 32, 33, 127, 128, 299):
        one = pgbp_b200.BatchedClusterGraphBelief(pl, 1).simulate(prm, 42, first_replicate=r, nodes=True)
        assert np.array_equal(one[0][0], big[0][r]) and np.array_equal(one[1][0], big[1][r])
    b5 = pgbp_b200.BatchedClusterGraphBelief(pl, 5)
    ten = pgbp_b200.BatchedClusterGraphBelief(pl, 10).simulate(prm, 42, first_replicate=0)
    assert np.array_equal(np.concatenate([b5.simulate(prm, 42, 0), b5.simulate(prm, 42, 5)]), ten)
    assert np.array_equal(ten, big[0][:10])
    # repeated calls: the same bits; another seed or replicate: other values
    assert np.array_equal(b5.simulate(prm, 42, 0), ten[:5])
    other = b5.simulate(prm, 43, 0)
    assert not np.any(other == ten[:5])
    assert not np.any(b5.simulate(prm, 42, 1) == ten[:5])
    # a shared-precision batch (groups of 5) equals an ordinary one
    sh = pgbp_b200.BatchedClusterGraphBelief(pl, 10, shared_precision_group=5).simulate(prm, 42)
    assert np.array_equal(sh, ten)


@pytest.mark.parametrize("backend", BACKENDS)
def test_device_entry_matches_host(backend):
    lib = get_lib(backend)
    p = 2
    _, _, d = synth_case(10, 2, 8, p)
    pl = plan_of(d, lib)
    fam = d["families"]
    rng = np.random.default_rng(1)
    B = 7
    prm = np.stack([bm_record("full", p, 1, rng, root="random") for _ in range(B)])
    bt = pgbp_b200.BatchedClusterGraphBelief(pl, B)
    tips, nodes = bt.simulate(prm, 5, 11, nodes=True)
    if backend == "emul":  # the emulation build's "device" is host memory
        dp = np.ascontiguousarray(prm)
        dt = np.empty_like(tips); dn = np.empty_like(nodes)
        bt.simulate_device(dp.ctypes.data, B, 5, dt.ctypes.data, dn.ctypes.data, first_replicate=11)
        dt2 = np.empty_like(tips)
        bt.simulate_device(dp.ctypes.data, B, 5, dt2.ctypes.data, None, first_replicate=11)
        dn2 = np.empty_like(nodes)
        bt.simulate_device(dp.ctypes.data, B, 5, None, dn2.ctypes.data, first_replicate=11)
        out = (dt, dn, dt2, dn2)
    else:
        import torch
        dp = torch.tensor(prm, device="cuda")
        torch.cuda.synchronize()  # the batch has its own stream
        dt = torch.empty(tips.shape, dtype=torch.float64, device="cuda")
        dn = torch.empty(nodes.shape, dtype=torch.float64, device="cuda")
        dt2, dn2 = torch.empty_like(dt), torch.empty_like(dn)
        bt.simulate_device(dp.data_ptr(), B, 5, dt.data_ptr(), dn.data_ptr(), first_replicate=11)
        bt.simulate_device(dp.data_ptr(), B, 5, dt2.data_ptr(), None, first_replicate=11)
        bt.simulate_device(dp.data_ptr(), B, 5, None, dn2.data_ptr(), first_replicate=11)
        bt.synchronize()
        out = tuple(x.cpu().numpy() for x in (dt, dn, dt2, dn2))
    assert np.array_equal(out[0], tips) and np.array_equal(out[1], nodes)
    assert np.array_equal(out[2], tips) and np.array_equal(out[3], nodes)


# ------------------------------------------------------------------ distribution
def moments_check(X, mean, cov, nsig=5.0):
    """sample mean / covariance of X[N, k] within nsig standard errors of (mean, cov)"""
    N = X.shape[0]
    sd = np.sqrt(np.diag(cov))
    assert np.all(np.abs(X.mean(0) - mean) <= nsig * sd / math.sqrt(N) + 1e-12)
    D = X - mean
    S = D.T @ D / N
    se = np.sqrt((np.outer(np.diag(cov), np.diag(cov)) + cov ** 2) / N)  # Var of x_i x_j under normality
    assert np.all(np.abs(S - cov) <= nsig * se + 1e-12), np.max(np.abs(S - cov) / (se + 1e-300))


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("model", ["bm", "ou"])
def test_distribution(backend, model):
    lib = get_lib(backend)
    p = 2 if model == "bm" else 1
    tab, _, d = synth_case(12, 3, 31, p)
    net, _, _, _ = synth_oracle_objects(tab, d)
    pl = plan_of(d, lib)
    B = 20000
    rng = np.random.default_rng(9)
    n = d["families"]["nnodes"]
    if model == "bm":
        R = rate(p, rng) * 3
        mu = rng.normal(size=p)
        V = rate(p, rng)
        X = pgbp_b200.BatchedClusterGraphBelief(pl, B).simulate(pgbp_b200.bm_params([R], mu, V), 123, nodes=True)[1]
        cov = densemvn.network_covariance(net, lambda e: R, p, rootvar=V)
        moments_check(X.reshape(B, n * p), np.tile(mu, n), cov)
    else:
        rec = np.array([1.5, 0.7, 4.0, -1.0, 0.5])
        X = pgbp_b200.BatchedClusterGraphBelief(pl, B).simulate(rec, 123, model="ou", nodes=True)[1]
        m, w, C = densemvn.ou_moments(net, *rec)
        cov = C + np.outer(w, w) * 0.0  # C already holds v in C[0, 0] and propagates it
        moments_check(X[:, :, 0], m, cov)


# ------------------------------------------------------------------ feeds K1
def loglik_of(bt, d):
    root = d["root_cluster"] + 1
    assert bt.propagate_1traversal_postorder(0).all()
    return bt.integratebelief(root, want_mu=False)[1]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("model", ["bm", "ou"])
def test_feeds_assignfactors(backend, model):
    lib = get_lib(backend)
    p = 3 if model == "bm" else 1
    tab, _, d = synth_case(12, 3, 41, p)
    net, _, _, taxa = synth_oracle_objects(tab, d)
    pl = plan_of(d, lib)
    B = 4000
    rng = np.random.default_rng(2)
    bt = pgbp_b200.BatchedClusterGraphBelief(pl, B)
    if model == "bm":
        R = rate(p, rng)
        mu = rng.normal(size=p)
        prm = pgbp_b200.bm_params([R], mu)
        tips = bt.simulate(prm, 7)
        bt.assignfactors(prm, tips)
        dense = lambda e: densemvn.loglik_bm(net, tips[e], taxa, lambda ed: R, mu)  # noqa: E731
        Sigma = densemvn.network_covariance(net, lambda ed: R, p)
    else:
        rec = np.array([1.2, 0.9, 2.0, -1.0, 0.0])
        tips = bt.simulate(rec, 7, model="ou")
        bt.assignfactors_ou(rec, tips)
        dense = lambda e: densemvn.loglik_ou(net, tips[e, :, 0], taxa, *rec)  # noqa: E731
        Sigma = densemvn.ou_moments(net, *rec)[2]
    ll = loglik_of(bt, d)
    assert (bt.status() == 0).all()
    for e in range(0, B, 397):
        assert abs(ll[e] - dense(e)) <= 1e-10 * (1 + abs(ll[e]))
    idx = {x.name: i for i, x in enumerate(net.vec_node)}
    sel = np.array([idx[t] * p + k for t in taxa for k in range(p)])
    nobs = sel.size
    expect = -nobs / 2 * densemvn.LOG2PI - 0.5 * np.linalg.slogdet(Sigma[np.ix_(sel, sel)])[1] - nobs / 2
    # -2 loglik = const + chi^2_n: sd of loglik = sqrt(n / 2)
    assert abs(ll.mean() - expect) <= 5 * math.sqrt(nobs / 2) / math.sqrt(B)


@pytest.mark.parametrize("backend", BACKENDS)
def test_feeds_missing_data_plan(backend):
    lib = get_lib(backend)
    p = 2
    tab, _, d = synth_case(10, 2, 51, p)
    net, cg, sched, taxa = synth_oracle_objects(tab, d)
    rng = np.random.default_rng(4)
    miss = rng.random((len(taxa), p)) < 0.3
    miss[0] = False
    tbl = np.where(miss, np.nan, 0.0)
    R = rate(p, rng)
    case = Case(net, "cliquetree", tbl, taxa, M.MvFullBrownianMotion(R, np.zeros(p)), lib, schedule=lambda c: sched, cg=cg)
    assert case.plan.families.get("tip_missing") is not None
    B = 3000
    bt = pgbp_b200.BatchedClusterGraphBelief(case.plan, B)
    prm = pgbp_b200.bm_params([R], np.zeros(p))
    tips, nodes = bt.simulate(prm, 8, nodes=True)
    assert np.array_equal(np.isnan(tips), np.broadcast_to(miss, tips.shape))
    fam = case.plan.families
    rt, rn, _ = restate(fam, p, "bm", prm, 8, 0, 3)
    close(tips[:3], rt)
    close(nodes[:3], rn)
    bt.assignfactors(prm, tips)
    assert (bt.status() == 0).all()
    ll = loglik_of_case(bt, case, sched)
    for e in (0, 1, 1500, B - 1):
        assert abs(ll[e] - densemvn.loglik_bm(net, tips[e], taxa, lambda ed: R, np.zeros(p))) <= 1e-10 * (1 + abs(ll[e]))
    idx = {x.name: i for i, x in enumerate(net.vec_node)}
    sel = np.array([idx[t] * p + k for i, t in enumerate(taxa) for k in range(p) if not miss[i, k]])
    Sigma = densemvn.network_covariance(net, lambda ed: R, p)
    expect = -sel.size / 2 * densemvn.LOG2PI - 0.5 * np.linalg.slogdet(Sigma[np.ix_(sel, sel)])[1] - sel.size / 2
    assert abs(ll.mean() - expect) <= 5 * math.sqrt(sel.size / 2) / math.sqrt(B)


def loglik_of_case(bt, case, sched):
    assert bt.propagate_1traversal_postorder(sched[0]).all()
    return bt.integratebelief(sched[0][2][0], want_mu=False)[1]


# ------------------------------------------------------------------ posterior coverage
@pytest.mark.parametrize("backend", BACKENDS)
def test_posterior_coverage(backend):
    lib = get_lib(backend)
    p = 2
    tab, _, d = synth_case(12, 3, 61, p)
    pl = plan_of(d, lib)
    B = 4000
    rng = np.random.default_rng(6)
    R = rate(p, rng)
    prm = pgbp_b200.bm_params([R], rng.normal(size=p))
    bt = pgbp_b200.BatchedClusterGraphBelief(pl, B)
    tips, nodes = bt.simulate(prm, 17, nodes=True)
    bt.assignfactors(prm, tips)
    succ, _ = bt.calibrate(None, 1)
    assert succ.all()
    mu, cov, ins = bt.node_moments()
    checked = 0
    for v in range(d["families"]["nnodes"]):
        for t in range(p):
            if not ins[v, t]:
                continue
            zs = (nodes[:, v, t] - mu[:, v, t]) / np.sqrt(cov[:, v, t, t])
            assert abs(zs.mean()) <= 5 / math.sqrt(B)
            assert abs(zs.var() - 1) <= 5 * math.sqrt(2 / B)
            checked += 1
    assert checked >= 10


# ------------------------------------------------------------------ invalid input
@pytest.mark.parametrize("backend", BACKENDS)
def test_invalid_input(backend):
    lib = get_lib(backend)
    p = 2
    _, _, d = synth_case(8, 1, 71, p)
    fam = d["families"]
    pl = plan_of(d, lib)
    B = 4
    bt = pgbp_b200.BatchedClusterGraphBelief(pl, B)
    prm = pgbp_b200.bm_params([np.eye(p)], np.zeros(p))
    mp = np.array(fam["mem_parent"], dtype=np.int32)
    out = np.empty((B, fam["ntips"], p))

    def call(model=0, ncolors=1, mem_parent=mp, params=prm, nparamsets=1, first=0, tip=out, nodes=None, b=bt):
        pa = np.ascontiguousarray(np.atleast_2d(params))
        mpp = np.ascontiguousarray(mem_parent, dtype=np.int32)
        return lib.pgbp_simulate(b.handle, model, ncolors, mpp.ctypes.data_as(pgbp_b200.api._i32p),
                                 pgbp_b200.api._fptr(pa), nparamsets, 1, first, pgbp_b200.api._fptr(tip),
                                 pgbp_b200.api._fptr(nodes))

    def err(rc, code, text):
        assert rc == code
        buf = __import__("ctypes").create_string_buffer(512)
        lib.pgbp_last_error(buf, 512)
        assert text in buf.value.decode(), buf.value

    assert call() == 0
    err(call(model=2), -1, "unknown model")
    err(call(model=1), -1, "Ornstein-Uhlenbeck")
    err(call(ncolors=0), -1, "ncolors")
    err(call(params=np.stack([prm] * 3), nparamsets=3), -1, "nparamsets must be 1 or B")
    err(call(first=-1), -1, "first_replicate < 0")
    err(call(tip=None), -1, "both outputs are null")
    bad = mp.copy(); bad[fam["mem_off"][3] + 1] = fam["nnodes"]
    err(call(mem_parent=bad), -1, "out of range")
    bad = mp.copy(); bad[fam["mem_off"][3] + 1] = 5
    err(call(mem_parent=bad), -1, "not before it")
    bad = mp.copy(); bad[fam["mem_off"][3]] = 0
    err(call(mem_parent=bad), -1, "own entry")
    # a non-root node without parents: a family table whose node 1 has no parent member
    f2 = dict(fam)
    o1 = fam["mem_off"][1]
    drop = o1 + 1
    for key in ("mem_pos", "mem_length", "mem_gamma", "mem_color", "mem_parent"):
        f2[key] = [x for i, x in enumerate(fam[key]) if i != drop]
    f2["mem_off"] = [x - (1 if i > 1 else 0) for i, x in enumerate(fam["mem_off"])]
    pl2 = pgbp_b200.ClusterGraphPlan(d["nclusters"], d["belief_dim"], d["sepset_clusters"], d["upind"], d["trees"], p, f2, lib)
    b2 = pgbp_b200.BatchedClusterGraphBelief(pl2, B)
    err(call(b=b2, mem_parent=np.array(f2["mem_parent"])), -1, "has no parent")
    with pytest.raises(ValueError, match="mem_parent"):
        f3 = {k: v for k, v in fam.items() if k != "mem_parent"}
        pl3 = pgbp_b200.ClusterGraphPlan(d["nclusters"], d["belief_dim"], d["sepset_clusters"], d["upind"], d["trees"], p, f3, lib)
        pgbp_b200.BatchedClusterGraphBelief(pl3, B).simulate(prm, 1)
    # shared-precision batch with several records
    sh = pgbp_b200.BatchedClusterGraphBelief(pl, B, shared_precision_group=2)
    err(call(b=sh, params=np.stack([prm] * B), nparamsets=B), -1, "shared-precision")
    # no family table
    pl4 = pgbp_b200.ClusterGraphPlan(d["nclusters"], d["belief_dim"], d["sepset_clusters"], d["upind"], d["trees"], p, None, lib)
    err(call(b=pgbp_b200.BatchedClusterGraphBelief(pl4, B)), -4, "no node-family table")


@pytest.mark.parametrize("backend", BACKENDS)
def test_element_status(backend):
    lib = get_lib(backend)
    p = 2
    _, _, d = synth_case(8, 1, 81, p)
    pl = plan_of(d, lib)
    ok = pgbp_b200.bm_params([np.eye(p)], np.zeros(p))
    improper = pgbp_b200.bm_params([np.eye(p)], np.zeros(p), [math.inf, 1.0])
    notpd = pgbp_b200.bm_params([np.array([[1.0, 2.0], [2.0, 1.0]])], np.zeros(p))
    bt = pgbp_b200.BatchedClusterGraphBelief(pl, 3)
    tips, nodes = bt.simulate(np.stack([ok, improper, notpd]), 3, nodes=True)
    st = bt.status()
    assert st[0] == 0 and st[1] == IMPROPER and st[2] == status(0x7ffffd, 2)
    assert np.isfinite(nodes[0]).all() and np.isnan(nodes[1:]).all() and np.isnan(tips[1:]).all()
    _, _, d1 = synth_case(8, 1, 81, 1)
    b1 = pgbp_b200.BatchedClusterGraphBelief(plan_of(d1, lib), 4)
    recs = np.array([[1.0, 1.0, 0.0, 0.0, 0.0], [0.0, 1.0, 0.0, 0.0, 0.0], [1.0, math.nan, 0.0, 0.0, 0.0],
                     [1.0, 1.0, 0.0, 0.0, math.inf]])
    t1 = b1.simulate(recs, 3, model="ou")
    assert list(b1.status()) == [0, BAD_RATE, BAD_RATE, IMPROPER]
    assert np.isfinite(t1[0]).all() and np.isnan(t1[1:]).all()


# ------------------------------------------------------------------ GPU, full size
def c_network(ntips, nretic, seed, p, ncolors):
    tab = synth.level1_network(ntips, nretic, seed)
    col = synth.edge_colors(tab, ncolors) if ncolors > 1 else None
    return synth.cliquetree_plan(tab, p, True, col)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c5", "c4"])
def test_fullsize_matches_emulation(name):
    """C5's network (p = 16) on a shared-precision batch of several scratch chunks, and the C4 network with four
    colours and one record per element: elements on both sides of every chunk boundary and the last element equal
    the emulation build run at first_replicate = r with B = 1.  The C5 batch is then assigned and calibrated."""
    import gc

    import torch
    try:
        fullsize(name)
    finally:  # the card is shared: hand the caching allocator's blocks back before the next test
        gc.collect()
        torch.cuda.empty_cache()


def fullsize(name):
    import torch
    cuda, emul = get_lib("cuda"), get_lib("emul")
    if name == "c5":
        d, p, nc, B, shared = c_network(100000, 10000, 0xB200 + 5, 16, 1), 16, 1, 600, 600
    else:
        d, p, nc, B, shared = c_network(10000, 1000, 0xB200 + 4, 8, 4), 8, 4, 4096, 0
    fam = d["families"]
    ninternal = sum(1 for r in fam["node_datarow"] if r < 0)
    chunk = max(32, (4 << 30) // (ninternal * p * 8) // 32 * 32)
    rng = np.random.default_rng(12)
    nrec = 1 if shared else B
    params = np.stack([bm_record("full", p, nc, rng, root="random") for _ in range(nrec)])
    pl = plan_of(d, cuda)
    bt = pgbp_b200.BatchedClusterGraphBelief(pl, B, factors=False, residuals=False, shared_precision_group=shared)
    dp = torch.tensor(params, device="cuda")
    torch.cuda.synchronize()  # the batch has its own stream
    dt = torch.empty((B, fam["ntips"], p), dtype=torch.float64, device="cuda")
    # every node's value only on C4 (5.8 GB); at C5's size that output would take 16.9 GB
    dn = torch.empty((B, fam["nnodes"], p), dtype=torch.float64, device="cuda") if name == "c4" else None
    bt.simulate_device(dp.data_ptr(), nrec, 99, dt.data_ptr(), dn.data_ptr() if dn is not None else None,
                       first_replicate=7, ncolors=nc)
    bt.synchronize()
    assert (bt.status() == 0).all()
    check = sorted({0, B - 1} | {x for c in range(chunk, B, chunk) for x in (c - 1, c)})
    if name == "c5":
        assert B > 2 * chunk  # at least three chunks
    pe = plan_of(d, emul)
    for r in check:
        one = pgbp_b200.BatchedClusterGraphBelief(pe, 1)
        tips, nodes = one.simulate(params[min(r, nrec - 1)], 99, first_replicate=7 + r, ncolors=nc, nodes=True)
        close(dt[r].cpu().numpy(), tips[0])  # libm and CUDA's log / sin / cos may differ in the last bit
        if dn is not None:
            close(dn[r].cpu().numpy(), nodes[0])
    if name == "c5":
        bt.assignfactors_device(dp.data_ptr(), 1, dt.data_ptr(), B, ncolors=nc)
        bt.calibrate_async(None, 1, update_residualnorm=False)
        norm = torch.empty(B, dtype=torch.float64, device="cuda")
        bt.integrate_device(d["root_cluster"] + 1, norm.data_ptr())
        bt.synchronize()
        assert (bt.status() == 0).all()
        assert torch.isfinite(norm).all()
