"""Posterior moments of node sets (pgbp_marginal_moments / BatchedClusterGraphBelief.node_moments): ancestral state
reconstruction from calibrated beliefs.

Every entry must equal the same entry of integratebelief_cov (pgbp_integrate_cov) bit for bit -- one arithmetic for
both calls -- on ordinary and shared-precision batches and on loopy graphs; node moments must reproduce the reference's
posterior goldens (test/test_calibration.jl:47-105, test/test_exactBM.jl:20-52)."""
import ctypes as C
import json
import math
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import pgbp_b200  # noqa: E402
from harness import BACKENDS, Case, get_lib, relerr  # noqa: E402
from oracle import bp as OBP  # noqa: E402
from oracle import models as M  # noqa: E402

TOL = 1e-10
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_goldens.json")))
NAN = math.nan
TAXA = ["A", "B1", "B2", "C"]
LAZ_TAXA = ["Mbuti", "Onge", "Karitiana", "MA1", "Loschbour", "European", "Stuttgart"]


def family_queries(bt):
    """(belief_j, positions) of every node family (child + parents in scope) in its home cluster."""
    fam, p = bt.plan.families, bt.plan.ntraits
    tpos = fam.get("mem_tpos")
    out = []
    for v in range(fam["nnodes"]):
        pos = []
        for a in range(fam["mem_off"][v], fam["mem_off"][v + 1]):
            if tpos is not None:
                pos.extend(int(x) for x in tpos[a * p:(a + 1) * p] if x >= 0)
            elif fam["mem_pos"][a] >= 0:
                pos.extend(fam["mem_pos"][a] + t for t in range(p))
        if pos:
            out.append((fam["node_cluster"][v] + 1, pos))
    return out


def assert_bit_identical(bt, queries):
    """marginal_moments == the matching entries of integratebelief_cov / integratebelief, bit for bit."""
    res = bt.marginal_moments(queries)
    full = {}
    for (j, pos), (mu, cov) in zip(queries, res):
        if j not in full:
            full[j] = bt.integratebelief_cov(j)
            assert np.array_equal(full[j][0], bt.integratebelief(j)[0])
        fm, fc, _ = full[j]
        pos = list(pos)
        assert mu.shape == (bt.B, len(pos)) and cov.shape == (bt.B, len(pos), len(pos))
        assert np.array_equal(mu, fm[:, pos]), (j, pos)
        assert np.array_equal(cov, fc[:, pos][:, :, pos]), (j, pos)
    return res


def mixed_queries(bt, rng):
    qs = [(j, pos) for _, _, j, pos in bt.node_queries()] + family_queries(bt)
    ncl = bt.nclusters
    for j in range(1, ncl + 1):
        m = bt.dimension(j)
        if m == 0:
            continue
        qs.append((j, list(range(m))))                      # whole cluster
        qs.append((j, [int(rng.integers(m))]))              # single position
        if m > 2:
            qs.append((j, list(rng.permutation(m)[:m - 1])))  # unsorted subset
    for j in range(ncl + 1, ncl + bt.nsepsets + 1):      # sepsets
        s = bt.dimension(j)
        if s:
            qs.append((j, list(range(s))[::-1]))
    return qs


def lazaridis_case(lib, p, method, rng, B):
    A = rng.normal(size=(p, p))
    R = A @ A.T / p + 0.1 * np.eye(p)
    data = rng.normal(size=(B, 7, p))
    model = M.MvFullBrownianMotion(R, np.zeros(p), np.diag([np.inf] * p))
    kw = dict(order_hint=GOLD["lazaridis_cluster_labels"]) if method == "cliquetree" else {}
    case = Case(GOLD["lazaridis"], method, data[0], LAZ_TAXA, model, lib, **kw)
    return case, R, data


@pytest.mark.parametrize("backend", BACKENDS)
def test_bit_identical_to_integrate_cov(backend):
    # lazaridis clique tree, MvFull BM p = 3, improper root, 5 data sets, fully calibrated
    lib = get_lib(backend)
    rng = np.random.default_rng(31)
    p, B = 3, 5
    case, R, data = lazaridis_case(lib, p, "cliquetree", rng, B)
    bt = pgbp_b200.BatchedClusterGraphBelief(case.plan, B)
    bt.assignfactors(pgbp_b200.bm_params([R], np.zeros(p), np.diag([np.inf] * p)), data)
    assert bt.calibrate(case.sched)[0].all()
    qs = mixed_queries(bt, rng)
    n0 = bt.launch_count(reset=True)
    assert_bit_identical(bt, qs)
    # against the oracle's calibrated beliefs
    cgbs = [case.oracle_cgb(tbl=data[e]) for e in range(B)]
    for c in cgbs:
        OBP.calibrate(c, case.sched)
    for (j, pos), (mu, cov) in zip(qs, bt.marginal_moments(qs)):
        for e in range(B):
            ob = cgbs[e].belief[j - 1]
            assert relerr(mu[e], np.linalg.solve(ob.J, ob.h)[pos]) <= TOL
            assert relerr(cov[e], np.linalg.inv(ob.J)[np.ix_(pos, pos)]) <= TOL
    # node moments are the node queries' results placed per node
    mu, cov, ins = bt.node_moments()
    for (v, tr, j, pos), (m, c) in zip(bt.node_queries(), bt.marginal_moments([(j, pos) for _, _, j, pos in bt.node_queries()])):
        assert ins[v, tr].all() and np.array_equal(mu[:, v, tr], m) and np.array_equal(cov[:, v][:, tr][:, :, tr], c)
    assert np.isnan(mu[:, ~ins]).all()
    assert n0 >= 0


@pytest.mark.parametrize("backend", BACKENDS)
def test_bit_identical_shared_precision_and_bethe(backend):
    lib = get_lib(backend)
    rng = np.random.default_rng(32)
    p, ntheta, nd = 3, 2, 4
    B = ntheta * nd
    case, _, data = lazaridis_case(lib, p, "cliquetree", rng, nd)
    Rs = []
    for _ in range(ntheta):
        A = rng.normal(size=(p, p))
        Rs.append(A @ A.T / p + 0.1 * np.eye(p))
    params = np.stack([pgbp_b200.bm_params([R], np.zeros(p), np.diag([np.inf] * p)) for R in Rs])
    # shared-precision batch: groups of data sets under one theta
    res = {}
    for name, group in (("own", 0), ("shared", nd)):
        bt = pgbp_b200.BatchedClusterGraphBelief(case.plan, B, shared_precision_group=group)
        bt.assignfactors(params, data, pairing="product")
        assert bt.calibrate(case.sched)[0].all()
        qs = mixed_queries(bt, np.random.default_rng(7))
        res[name] = assert_bit_identical(bt, qs)
    for (m1, c1), (m2, c2) in zip(res["own"], res["shared"]):
        assert np.array_equal(m1, m2) and np.array_equal(c1, c2)
    # loopy Bethe graph after regularizebeliefs_bycluster + calibrate
    case, R, data = lazaridis_case(lib, p, "bethe", rng, nd)
    bt = pgbp_b200.BatchedClusterGraphBelief(case.plan, nd)
    bt.assignfactors(pgbp_b200.bm_params([R], np.zeros(p), np.diag([np.inf] * p)), data)
    bt.regularizebeliefs_bycluster()
    bt.calibrate(case.sched, 3)
    assert (bt.status() == 0).all()
    assert_bit_identical(bt, mixed_queries(bt, rng))


def exactbm_case(lib):
    netstr = "((A:1.5,B:1.5):1,(C:1,(D:0.5, E:0.5):0.5):1.5);"
    taxa = ["A", "B", "C", "D", "E"]
    y = np.array([1.0, 0.9, 1.0, -1.0, -0.9])
    v0 = 1e10
    case = Case(netstr, "cliquetree", y[:, None], taxa, M.UnivariateBrownianMotion(1.0, 0.0, v0), lib, schedule="spanningtree")
    return case, taxa, y, v0


@pytest.mark.parametrize("backend", BACKENDS)
def test_phylogeneticem_node_moments_goldens(backend):
    # test/test_exactBM.jl:3-52: 5-taxon tree, PhylogeneticEM's conditional expectations, variances and parent-child
    # covariances (7 digits, atol 1e-6), in preorder; and the dense conditional Gaussian on the tree covariance (2e-6)
    lib = get_lib(backend)
    case, taxa, y, v0 = exactbm_case(lib)
    B = 2
    bt = pgbp_b200.BatchedClusterGraphBelief(case.plan, B)
    bt.assignfactors(pgbp_b200.bm_params([1.0], [0.0], [v0]), np.stack([y[:, None]] * B))
    assert bt.calibrate(case.sched)[0].all()
    order = [5, 7, 8, 4, 3, 2, 6, 1, 0]
    condexp = np.array([1, 0.9, 1, -1, -0.9, 0.4436893, 0.7330097, 0.009708738, -0.6300971])[order]
    condvar = np.array([0, 0, 0, 0, 0, 0.9174757, 0.5970874, 0.3786408, 0.2087379])[order]
    condcov = np.array([0, 0, 0, 0, 0, np.nan, 0.3932039, 0.2038835, 0.1262136])[order]
    nodes = case.net.vec_node
    n = len(nodes)
    leaf = np.array([nd.leaf for nd in nodes])
    mu, cov, ins = bt.node_moments()
    assert mu.shape == (B, n, 1) and cov.shape == (B, n, 1, 1)
    assert (ins[:, 0] == ~leaf).all() and np.isnan(mu[:, leaf]).all() and np.isnan(cov[:, leaf]).all()
    internal = np.flatnonzero(~leaf)
    assert len(internal) == 4
    for e in range(B):
        assert np.max(np.abs(mu[e, internal, 0] - condexp[internal])) <= 1e-6
        assert np.max(np.abs(cov[e, internal, 0, 0] - condvar[internal])) <= 1e-6
    # parent-child covariances from family queries (child first, then its parent)
    fq = family_queries(bt)
    fam = case.plan.families
    kids = [v for v in range(n) if any(fam["mem_pos"][a] >= 0 for a in range(fam["mem_off"][v], fam["mem_off"][v + 1]))]
    res = bt.marginal_moments(fq)
    nchecked = 0
    for v, (m, c) in zip(kids, res):
        if c.shape[1] == 2 and not np.isnan(condcov[v]):
            assert np.max(np.abs(c[:, 0, 1] - condcov[v])) <= 1e-6
            nchecked += 1
    assert nchecked == 3
    # dense conditional Gaussian of all 9 nodes (preorder) given the 5 tips
    idx = case.net.preorder_index()
    V = np.zeros((n, n))
    V[0, 0] = v0
    for i in range(1, n):
        (ed,) = nodes[i].parent_edges()
        q = idx[id(ed.parent)] - 1
        V[i, :i] = V[q, :i]
        V[:i, i] = V[i, :i]
        V[i, i] = V[q, q] + ed.length
    tip = np.flatnonzero(leaf)
    ytip = np.array([y[taxa.index(nodes[i].name)] for i in tip])
    K = np.linalg.solve(V[np.ix_(tip, tip)], V[np.ix_(tip, internal)]).T
    cmean = K @ ytip
    ccov = V[np.ix_(internal, internal)] - K @ V[np.ix_(tip, internal)]
    assert np.max(np.abs(mu[:, internal, 0] - cmean)) <= 2e-6
    assert np.max(np.abs(cov[:, internal, 0, 0] - np.diag(ccov))) <= 2e-6


@pytest.mark.parametrize("backend", BACKENDS)
def test_root_posterior_goldens_cliquetree_and_bethe(backend):
    lib = get_lib(backend)
    # test/test_calibration.jl:36-78: clique tree, posterior root mean and variance.  The variance golden is at the
    # unrounded REML rate 0.4714735834478194 (test_parity's exact-REML golden; the test there rounds it to 0.471474,
    # which moves the variance by 9e-7 relative); the mean does not depend on the rate (improper root)
    s2 = 0.4714735834478194
    tbl_y = np.array([[1.0], [.9], [1], [-1]])
    case = Case(GOLD["netstr_named"], "cliquetree", tbl_y, TAXA, M.UnivariateBrownianMotion(s2, 0, math.inf), lib,
                schedule="spanningtree")
    bt = pgbp_b200.BatchedClusterGraphBelief(case.plan, 2)
    bt.assignfactors(pgbp_b200.bm_params([s2], [0.0], [math.inf]), tbl_y[None])
    pgbp_b200.calibrate(bt, case.sched)
    mu, cov, ins = bt.node_moments()
    assert ins[0, 0]
    assert np.all(np.abs(mu[:, 0, 0] / -0.26000871507162693 - 1) <= TOL)
    assert np.all(np.abs(cov[:, 0, 0, 0] / 0.33501871740664146 - 1) <= TOL)
    # test/test_calibration.jl:79-105: Bethe graph, regularised on schedule, auto-stop at (iteration 5, tree 1).  The root
    # I4 is fixed (out of scope, NaN); the golden is the exact posterior mean of its child I3 (read there from cluster I3),
    # which loopy BP at its 1e-5 residual tolerance approximates to rtol 1e-5; here it comes from I3's home cluster I3I4
    tbl_y = np.array([[-1.81358], [0.468158], [0.658486], [0.643821]])
    case = Case(GOLD["netstr_unnamed"], "bethe", tbl_y, ["A", "B", "C", "D"], M.UnivariateBrownianMotion(0.0861249, 0), lib)
    bt = pgbp_b200.BatchedClusterGraphBelief(case.plan, 2)
    bt.assignfactors(pgbp_b200.bm_params([0.0861249], [0.0]), tbl_y[None])
    bt.regularizebeliefs_onschedule()
    succ, iscal, it = pgbp_b200.calibrate(bt, case.sched, 20, auto=True, info=True)
    assert succ.all() and iscal.all() and tuple(it[0]) == (5, 1)
    mu, cov, ins = bt.node_moments()
    names = [nd.name for nd in case.net.vec_node]
    i3, i4 = names.index("I3"), names.index("I4")
    assert i4 == 0 and not ins[i4].any() and np.isnan(mu[:, i4]).all() and np.isnan(cov[:, i4]).all()
    assert ins[i3, 0] and np.all(np.abs(mu[:, i3, 0] / 0.21511454631828986 - 1) <= 1e-5)


@pytest.mark.parametrize("backend", BACKENDS)
def test_missing_data_partial_scopes(backend):
    # Tips are always out of scope (observed values are evidence, missing ones are marginalised out of the tip's edge
    # factor, src/beliefs.jl:833-857), so a partially observed tip is NaN in every trait.  An internal node with no data
    # below it for a trait loses that trait from its scope (test/test_calibration.jl:107-129): its posterior is the
    # partial-scope query through mem_tpos -- finite moments for the traits in scope, NaN for the others.
    lib = get_lib(backend)
    tbl = np.array([[1, NAN], [1, NAN], [1.5, NAN], [1, 1.0]])
    taxa = ["A", "B", "C", "D"]
    model = M.MvDiagBrownianMotion([1, 2], [0, 0], [1, 1])
    case = Case("(((A:1.0, B:1.0)E:1.0, C:2.0)F:1.0, D:3.0)G;", "cliquetree", tbl, taxa, model, lib, schedule="spanningtree")
    assert case.plan.families.get("mem_tpos") is not None
    B = 3
    data = np.repeat(tbl[None], B, axis=0)
    data[1:] += np.random.default_rng(3).normal(size=(B - 1,) + tbl.shape)
    bt = pgbp_b200.BatchedClusterGraphBelief(case.plan, B)
    bt.assignfactors(pgbp_b200.bm_params([np.array([1.0, 2.0])], [0, 0], [1.0, 1.0]), data)
    assert bt.calibrate(case.sched)[0].all()
    mu, cov, ins = bt.node_moments()
    names = [nd.name for nd in case.net.vec_node]
    expect = {"G": [True, True], "F": [True, False], "E": [True, False], "A": [False, False], "B": [False, False],
              "C": [False, False], "D": [False, False]}
    for nm, sc in expect.items():
        v = names.index(nm)
        assert ins[v].tolist() == sc, nm
        t = np.array(sc)
        assert np.isfinite(mu[:, v, t]).all() and np.isnan(mu[:, v, ~t]).all()
        assert np.isfinite(cov[:, v][:, t][:, :, t]).all() and np.isnan(cov[:, v, ~t]).all() and np.isnan(cov[:, v, :, ~t]).all()
    qs = bt.node_queries()
    assert_bit_identical(bt, [(j, pos) for _, _, j, pos in qs] + family_queries(bt))
    cgbs = [case.oracle_cgb(tbl=data[e]) for e in range(B)]
    for c in cgbs:
        OBP.calibrate(c, case.sched)
    for v, tr, j, pos in qs:
        for e in range(B):
            ob = cgbs[e].belief[j - 1]
            assert relerr(mu[e, v, tr], np.linalg.solve(ob.J, ob.h)[pos]) <= TOL
            assert relerr(cov[e, v][np.ix_(tr, tr)], np.linalg.inv(ob.J)[np.ix_(pos, pos)]) <= TOL


def uploaded_lazaridis(lib, B, seed=41):
    rng = np.random.default_rng(seed)
    case, R, data = lazaridis_case(lib, 3, "cliquetree", rng, B)
    bt = pgbp_b200.BatchedClusterGraphBelief(case.plan, B)
    bt.assignfactors(pgbp_b200.bm_params([R], np.zeros(3), np.diag([np.inf] * 3)), data)
    assert bt.calibrate(case.sched)[0].all()
    return case, bt


@pytest.mark.parametrize("backend", BACKENDS)
def test_failures_and_invalid_input(backend):
    lib = get_lib(backend)
    B = 4
    case, bt = uploaded_lazaridis(lib, B)
    j = 2
    m = bt.dimension(j)
    qs = [(j, list(range(m))), (j, [m - 1, 0]), (1, [0])]
    ref = bt.marginal_moments(qs)
    # indefinite J for element 1 of belief j: status 0x7ffffe, NaN outputs of that belief; other elements unaffected
    J, h, g = bt.get_belief(j)
    J[1] = -np.eye(m)
    bt.set_belief(j, J, h, g)
    bt.clear_status()
    res = bt.marginal_moments(qs)
    st = bt.status()
    assert (st[1] >> 8) - 1 == 0x7ffffe and (st[1] & 0xff) == 1 and (np.delete(st, 1) == 0).all()
    keep = [0, 2, 3]
    for (m1, c1), (m2, c2) in zip(ref[:2], res[:2]):
        assert np.isnan(m2[1]).all() and np.isnan(c2[1]).all()
        assert np.array_equal(m1[keep], m2[keep]) and np.array_equal(c1[keep], c2[keep])
    assert np.array_equal(ref[2][0], res[2][0]) and np.array_equal(ref[2][1], res[2][1])
    # all-zero belief: +Inf (integratebelief's mean)
    bt.set_belief(j, np.zeros((B, m, m)), np.zeros((B, m)), np.zeros(B))
    for mu, cov in bt.marginal_moments(qs[:2]):
        assert np.isposinf(mu).all() and np.isposinf(cov).all()
    assert np.isposinf(bt.integratebelief(j)[0]).all()
    # invalid input
    nb = bt.nbeliefs()
    for bad in ([], [(0, [0])], [(nb + 1, [0])], [(j, [m])], [(j, [-1])], [(j, [0, 1, 0])], [(1, [0]), (j, [1, 1])]):
        with pytest.raises(pgbp_b200.PgbpError):
            bt.marginal_moments(bad)
    one = np.zeros(4, dtype=np.int32)
    ip = one.ctypes.data_as(C.POINTER(C.c_int32))
    out = np.zeros(64)
    fp = out.ctypes.data_as(C.POINTER(C.c_double))
    for args in ((None, ip, ip, fp, fp), (ip, None, ip, fp, fp), (ip, ip, None, fp, fp), (ip, ip, ip, None, fp)):
        with pytest.raises(pgbp_b200.PgbpError):
            lib.check(lib.pgbp_marginal_moments(bt.handle, 1, *args))
    with pytest.raises(pgbp_b200.PgbpError):
        lib.check(lib.pgbp_marginal_moments(None, 1, ip, ip, ip, fp, fp))
    with pytest.raises(pgbp_b200.PgbpError):
        lib.check(lib.pgbp_marginal_moments_device(bt.handle, 1, ip, ip, ip, None, None))
    # node moments need the family table
    plan = pgbp_b200.ClusterGraphPlan(case.plan.nclusters, case.plan.belief_dim, case.plan.sepset_clusters,
                                      case.plan.upind, case.plan.trees, 3, None, lib)
    with pytest.raises(ValueError):
        pgbp_b200.BatchedClusterGraphBelief(plan, 2).node_moments()


@pytest.mark.parametrize("backend", BACKENDS)
def test_device_variant_equals_host_variant(backend):
    lib = get_lib(backend)
    B = 37
    case, bt = uploaded_lazaridis(lib, B)
    qs = mixed_queries(bt, np.random.default_rng(9))
    host = bt.marginal_moments(qs)
    _, ld, _ = bt.device_view()
    nmu = sum(len(p) for _, p in qs)
    ncov = sum(len(p) * (len(p) + 1) // 2 for _, p in qs)
    if backend == "cuda":
        import torch
        d_mu = torch.full((nmu, ld), -1.0, dtype=torch.float64, device="cuda")
        d_cov = torch.full((ncov, ld), -1.0, dtype=torch.float64, device="cuda")
        bt.marginal_moments_device(qs, d_mu.data_ptr(), d_cov.data_ptr())
        bt.synchronize()
        dm, dc = d_mu.cpu().numpy(), d_cov.cpu().numpy()
    else:  # the emulation build's device memory is host memory
        dm, dc = np.full((nmu, ld), -1.0), np.full((ncov, ld), -1.0)
        bt.marginal_moments_device(qs, dm.ctypes.data, dc.ctypes.data)
    r0 = c0 = 0
    for (j, pos), (mu, cov) in zip(qs, host):
        k = len(pos)
        assert np.array_equal(dm[r0:r0 + k, :B].T, mu)
        for c in range(k):
            for r in range(c + 1):
                assert np.array_equal(dc[c0 + c * (c + 1) // 2 + r, :B], cov[:, r, c])
        r0 += k
        c0 += k * (k + 1) // 2
    assert r0 == nmu and c0 == ncov
    # node_moments_device: the rows of the node queries, in node order
    nq = bt.node_queries()
    kmu = sum(len(q[1]) for q in nq)
    if backend == "cuda":
        import torch
        d_mu = torch.zeros((kmu, ld), dtype=torch.float64, device="cuda")
        bt.node_moments_device(d_mu.data_ptr())
        bt.synchronize()
        dm = d_mu.cpu().numpy()
    else:
        dm = np.zeros((kmu, ld))
        bt.node_moments_device(dm.ctypes.data)
    mu, _, _ = bt.node_moments()
    r0 = 0
    for v, tr, _, _ in nq:
        assert np.array_equal(dm[r0:r0 + len(tr), :B].T, mu[:, v, tr])
        r0 += len(tr)


@pytest.mark.gpu
def test_c4_node_moments_full_size():
    # the 10,000-tip network of BASELINE configs[3] (p = 8, fixed root), a handful of theta, fully calibrated:
    # every node's moments equal integrate_cov of its home cluster, on a seeded sample of nodes
    import bench
    lib = get_lib("cuda")
    w = bench.C4()
    B = 8
    params, tips = w.inputs(B, 0)
    d = w.d
    plan = pgbp_b200.ClusterGraphPlan(d["nclusters"], d["belief_dim"], d["sepset_clusters"], d["upind"], d["trees"],
                                      d["ntraits"], d["families"], lib)
    bt = pgbp_b200.BatchedClusterGraphBelief(plan, B, factors=False, residuals=True)
    bt.assignfactors(params, tips, ncolors=w.ncolors)
    assert bt.calibrate(None, 1)[0].all()
    mu, cov, ins = bt.node_moments()
    assert (bt.status() == 0).all()
    nq = bt.node_queries()
    assert len(nq) > 9000 and ins.sum() == sum(len(q[1]) for q in nq)
    assert np.isfinite(mu[:, ins]).all() and np.isnan(mu[:, ~ins]).all()
    rng = np.random.default_rng(2024)
    for i in rng.choice(len(nq), size=96, replace=False):
        v, tr, j, pos = nq[i]
        fm, fc, _ = bt.integratebelief_cov(j)
        assert np.array_equal(mu[:, v, tr], fm[:, pos])
        assert np.array_equal(cov[:, v][:, tr][:, :, tr], fc[:, pos][:, :, pos])


def test_julia_binding_binds_marginal_moments():
    # the prototype check of test_julia_binding.py covers the signatures of every ccall; here: both are bound
    src = open(os.path.join(ROOT, "julia", "PGBPB200.jl")).read()
    for name in ("pgbp_marginal_moments", "pgbp_marginal_moments_device"):
        assert "ccall((:%s, LIB)" % name in src, name
    assert "function marginal_moments!(b::BatchedClusterGraphBelief" in src
    assert "function marginal_moments_device!(b::BatchedClusterGraphBelief" in src
