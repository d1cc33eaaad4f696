"""The univariate Ornstein-Uhlenbeck model (pgbp_assign_factors_ou) against a dense OU likelihood.

The oracle restates the reference's OU factor, so it shares its formulas with the device.  oracle/densemvn.py's
ou_moments / loglik_ou share nothing with either: they build the mean, root weight and covariance of every node
state by the network recursion (with expm1, exact as alpha -> 0).  These tests check against them the
log-likelihood of synthetic level-1 networks over a wide range of alpha, with theta far from mu (so that a wrong
sign or a dropped omega shows), with fixed, proper and improper roots, on theta grids, with missing tips (the scoped
K1 path), the posterior node moments, and the fixed point of loopy BP; beliefs, residuals and factored energies
against the oracle; shared-precision batches against own-J batches bit for bit; and the Brownian-motion limit."""
import math
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import pgbp_b200  # noqa: E402
from harness import BACKENDS, Case, get_lib, relerr, synth_oracle_objects  # noqa: E402
from oracle import bp as OBP  # noqa: E402
from oracle import densemvn  # noqa: E402
from oracle import models as M  # noqa: E402
from test_loopy_multivariate import check_vs_oracle, network, regularize, max_residual  # noqa: E402
from test_missing_data import clades, missing_mask  # noqa: E402
from test_parity import GOLD, TAXA, TBL, check_all_beliefs  # noqa: E402
from workloads import synth  # noqa: E402

TOL = 1e-10
DENSE_TOL = 1e-9
# entries that are zero in exact arithmetic (g of a cluster whose only family is a marginalised missing tip) are
# roundoff of either sign on both sides (see check_all_beliefs).  The terms that cancel there reach j omega^2 / 2 ~ 1e3
# (alpha = 50, theta 6 away from mu), so that roundoff is ~1e-13; measured against FLOOR it must stay below 1e-11
FLOOR = 0.1
BAD_RECORD = int(np.int32(((0x7ffffd + 1) << 8) | 1))  # PGBP_STATUS(0x7ffffd, 1): invalid OU parameters
ROOTS = ("fixed", "random", "improper")


# ------------------------------------------------------------------ parameters, data
def records(n, root, seed):
    """n OU records (sigma2, alpha, theta, mu, v): alpha log-spaced over [1e-4, 50] (q = exp(-alpha t) from ~1 down
    to ~1e-60 on these networks), theta 3 to 6 away from mu on either side, v by root type.  Under an improper root
    alpha stays <= 2: the data's information on the root value decays like exp(-2 alpha depth), and at alpha = 50
    the root cluster's precision (~1e-130) is not positive definite in double precision."""
    rng = np.random.default_rng(seed)
    alpha = np.geomspace(1e-4, 2.0 if root == "improper" else 50.0, n)
    rng.shuffle(alpha)
    mu = rng.normal(size=n)
    theta = mu + rng.choice([-1.0, 1.0], size=n) * rng.uniform(3.0, 6.0, size=n)
    v = {"fixed": np.zeros(n), "random": rng.uniform(0.2, 2.0, size=n), "improper": np.full(n, math.inf)}[root]
    return np.stack([rng.uniform(0.5, 2.0, size=n), alpha, theta, mu, v], axis=1)


def simulate(net, taxa, rec, nd, seed):
    """nd data sets (nd, ntips, 1) simulated exactly down the network (nodes in preorder):
    X_i = sum_k gamma_k (q_k X_pa(k) + omega_k) + sqrt(sum_k gamma_k^2 var_k) eps.  An improper root starts at mu."""
    s2, al, th, mu, v = rec
    rng = np.random.default_rng(seed)
    pre = net.vec_node
    idx = {id(x): i for i, x in enumerate(pre)}
    X = np.zeros((nd, len(pre)))
    X[:, 0] = mu + (math.sqrt(v) * rng.normal(size=nd) if 0 < v < math.inf else 0.0)
    for i in range(1, len(pre)):
        var = 0.0
        for e in pre[i].parent_edges():
            q = math.exp(-al * e.length)
            X[:, i] += e.gamma * (q * X[:, idx[id(e.parent)]] - math.expm1(-al * e.length) * th)
            var += e.gamma ** 2 * s2 / (2 * al) * -math.expm1(-2 * al * e.length)
        X[:, i] += math.sqrt(var) * rng.normal(size=nd)
    name = {x.name: i for i, x in enumerate(pre)}
    return X[:, [name[t] for t in taxa]][:, :, None]


def ou_model(rec):
    s2, al, th, mu, v = rec
    return M.UnivariateOrnsteinUhlenbeck(s2, al, th, mu, None if v == 0 else v)


class OU:
    """A level-1 network of workloads/synth.py with its clique tree, np OU records of one root type and nd data sets
    (simulated from record 0), tips of `pattern` (test_missing_data
    patterns) missing in every data set.  The plan comes from the oracle front-end: with missing tips it has
    trait-level scopes and the scoped K1 path assigns its factors."""

    def __init__(self, lib, ntips, nretic, seed, root, np_=3, nd=3, pattern=None):
        tab = self.tab = synth.level1_network(ntips, nretic, seed)
        plan = synth.cliquetree_plan(tab, 1)
        self.net, cg, sched, self.taxa = synth_oracle_objects(tab, plan)
        self.recs = records(np_, root, seed)
        self.mask = np.zeros(len(self.taxa), dtype=bool)
        if pattern:
            self.mask = missing_mask(tab, plan["tip_nodes"], 1, pattern, seed)[:, 0]
        self.data = simulate(self.net, self.taxa, self.recs[0], nd, seed + 7)
        self.data[:, self.mask] = np.nan
        self.case = Case(self.net, "cliquetree", self.data[0], self.taxa, ou_model(self.recs[0]), lib,
                         schedule=lambda c: sched, cg=cg)
        self.sched = sched
        self.root = sched[0][2][0]

    def dense(self, ip, idd):
        return densemvn.loglik_ou(self.net, self.data[idd, :, 0], self.taxa, *self.recs[ip])

    def oracle(self, ip, idd):
        return self.case.oracle_cgb(tbl=self.data[idd], model=ou_model(self.recs[ip]))

    def batch(self, B, **kw):
        return pgbp_b200.BatchedClusterGraphBelief(self.case.plan, B, **kw)


def loglik_everywhere(s, bt):
    """log-likelihood at the root cluster after one postorder pass, then at every belief after calibration"""
    assert bt.propagate_1traversal_postorder(s.sched[0]).all()
    out = [bt.integratebelief(s.root, want_mu=False)[1]]
    succ, _ = bt.calibrate(s.sched)
    assert succ.all()
    for j in range(1, len(s.case.b) + 1):
        if bt.dimension(j) > 0:
            out.append(bt.integratebelief(j, want_mu=False)[1])
    return out


# ------------------------------------------------------------------ log-likelihood against the dense OU likelihood
# (id, ntips, nretic, seed, root, missing tips).  Five records per case, each with its own data set (zip pairing,
# np = nd = B).  The clade pattern removes internal nodes from every scope (p = 1: a node keeps its only trait
# only if some tip below it is observed).
CASES = [
    ("t8-h0-fixed", 8, 0, 1, "fixed", None),
    ("t16-h2-random", 16, 2, 2, "random", None),
    ("t30-h3-improper", 30, 3, 3, "improper", None),
    ("t60-h4-fixed", 60, 4, 4, "fixed", None),
    ("t45-h4-random", 45, 4, 5, "random", None),
    ("sisters-t10-h2-fixed", 10, 2, 11, "fixed", "sisters"),
    ("sisters-t20-h3-improper", 20, 3, 12, "improper", "sisters"),
    ("clade-t14-h3-random", 14, 3, 13, "random", "clade"),
    ("clade-t24-h4-fixed", 24, 4, 14, "fixed", "clade"),
    ("clade-t18-h2-improper", 18, 2, 15, "improper", "clade"),
    ("tipall-t9-h2-random", 9, 2, 16, "random", "tipall"),
    ("tipall-t12-h3-fixed", 12, 3, 17, "fixed", "tipall"),
    ("tipall-t16-h4-improper", 16, 4, 18, "improper", "tipall"),
    ("scatter-t20-h3-fixed", 20, 3, 19, "fixed", "scatter"),
    ("scatter-t40-h4-random", 40, 4, 20, "random", "scatter"),
    ("all-t30-h4-improper", 30, 4, 21, "improper", "sisters+clade+tipall+scatter"),
]
NREC = 5
MISSING_CASES = [c for c in CASES if c[5]]


def case_setup(lib, cs):
    _, ntips, nretic, seed, root, pattern = cs
    s = OU(lib, ntips, nretic, seed, root, NREC, 1, pattern)
    # one data set per record, each simulated from its own record
    s.data = np.concatenate([simulate(s.net, s.taxa, s.recs[k], 1, seed + 100 + k) for k in range(NREC)])
    s.data[:, s.mask] = np.nan
    return s


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("cs", CASES, ids=lambda c: c[0])
def test_loglik_matches_dense_ou(backend, cs):
    s = case_setup(get_lib(backend), cs)
    dense = np.array([s.dense(e, e) for e in range(NREC)])
    bt = s.batch(NREC)
    bt.assignfactors_ou(s.recs, s.data)
    assert (bt.status() == 0).all()
    for k, ll in enumerate(loglik_everywhere(s, bt)):
        assert np.max(np.abs(ll / dense - 1)) <= DENSE_TOL, (k, ll, dense)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("cs", [c for c in CASES if c[1] <= 30], ids=lambda c: c[0])
def test_beliefs_match_oracle(backend, cs):
    # every belief after assignment and after calibration against the oracle's assignfactors! / calibrate!
    s = case_setup(get_lib(backend), cs)
    bt = s.batch(NREC)
    bt.assignfactors_ou(s.recs, s.data)
    assert (bt.status() == 0).all()
    cgbs = [s.oracle(e, e) for e in range(NREC)]
    check_all_beliefs(s.case, bt, cgbs, floor=FLOOR)
    assert bt.calibrate(s.sched)[0].all()
    for c in cgbs:
        OBP.calibrate(c, s.sched)
    check_all_beliefs(s.case, bt, cgbs, floor=FLOOR)


@pytest.mark.parametrize("cs", MISSING_CASES, ids=lambda c: c[0])
def test_missing_tip_plans_are_scoped(cs):
    # the missing-data cases above run the scoped K1 path; clade patterns take internal nodes out of every scope
    s = case_setup(get_lib("emul"), cs)
    fam = s.case.plan.families
    assert fam.get("mem_tpos") is not None and fam.get("tip_missing") is not None
    assert np.asarray(fam["tip_missing"]).reshape(-1).astype(bool).tolist() == s.mask.tolist()
    # an internal node keeps its trait exactly when some tip below it is observed (mem_tpos of its own member)
    _, below = clades(s.tab)
    row = {int(t[1:]): i for i, t in enumerate(s.taxa)}
    tpos = np.asarray(fam["mem_tpos"]).reshape(-1)
    off = np.asarray(fam["mem_off"])
    internal = [v for v in range(1, s.tab["nnodes"]) if not s.tab["leaf"][v]]
    gone = [v for v in internal if all(s.mask[row[t]] for t in below[v])]
    assert [v for v in internal if tpos[off[v]] < 0] == gone
    if "clade" in cs[5]:
        assert len(gone) >= 2


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("pattern", [[10.0, 10.0, math.nan, 0.0], [10.0, math.nan, math.nan, 0.0]], ids=["B2", "B1B2"])
def test_named_network_missing_tips(backend, pattern):
    # trait x of the 4-tip network with tip B2 missing (-438.6709189569596, the oracle and the dense likelihood
    # agree), and with B1 and B2 missing: nodes i6 and H5 then have no trait in scope, their clusters dimension 0
    lib = get_lib(backend)
    rec = (2.0, 3.0, -2.0, 0.0, 0.4)
    tbl = np.array(pattern)[:, None]
    case = Case(GOLD["netstr_named"], "cliquetree", tbl, TAXA, ou_model(rec), lib, schedule="spanningtree")
    assert case.plan.families.get("mem_tpos") is not None
    data = np.stack([tbl, tbl + 0.5, tbl - 2.0])
    bt = pgbp_b200.BatchedClusterGraphBelief(case.plan, 3)
    bt.assignfactors_ou([rec], data)
    assert (bt.status() == 0).all()
    cgbs = [case.oracle_cgb(tbl=data[e]) for e in range(3)]
    check_all_beliefs(case, bt, cgbs, floor=FLOOR)
    spt = case.sched[0]
    assert bt.propagate_1traversal_postorder(spt).all()
    ll = bt.integratebelief(spt[2][0])[1]
    dense = [densemvn.loglik_ou(case.net, data[e, :, 0], TAXA, *rec) for e in range(3)]
    assert np.max(np.abs(ll / dense - 1)) <= DENSE_TOL, (ll, dense)
    if math.isnan(pattern[1]):
        assert any(case.plan.belief_dim[j] == 0 for j in range(case.nclusters))
    else:
        assert abs(ll[0] / -438.6709189569596 - 1) <= TOL
    assert bt.calibrate(case.sched)[0].all()
    for c in cgbs:
        OBP.calibrate(c, case.sched)
    check_all_beliefs(case, bt, cgbs, floor=FLOOR)


# ------------------------------------------------------------------ theta grids
GRID_NP, GRID_ND = 250, 4  # B = 1000: not a multiple of 32 or 128


def grid_setup(lib, pattern=None, root="random"):
    s = OU(lib, 20, 3, 31, root, GRID_NP, GRID_ND, pattern)
    s.dense_grid = np.array([[s.dense(ip, idd) for idd in range(GRID_ND)] for ip in range(GRID_NP)])
    return s


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("pattern", [None, "clade+scatter"], ids=["full", "missing"])
def test_theta_grid_product_matches_dense(backend, pattern):
    # 250 records x 4 data sets, element e = (record e // 4, data set e % 4)
    s = grid_setup(get_lib(backend), pattern)
    B = GRID_NP * GRID_ND
    bt = s.batch(B)
    bt.assignfactors_ou(s.recs, s.data, pairing="product")
    assert (bt.status() == 0).all()
    assert bt.propagate_1traversal_postorder(s.sched[0]).all()
    ll = bt.integratebelief(s.root, want_mu=False)[1]
    dense = s.dense_grid.reshape(-1)
    assert np.max(np.abs(ll / dense - 1)) <= DENSE_TOL


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("pattern", [None, "sisters"], ids=["full", "missing"])
def test_theta_grid_zip_matches_dense(backend, pattern):
    # zip pairing with np = B = 1000 records and one data set
    s = grid_setup(get_lib(backend), pattern, root="fixed")
    recs = records(1000, "fixed", 32)
    bt = s.batch(1000)
    bt.assignfactors_ou(recs, s.data[:1])
    assert (bt.status() == 0).all()
    assert bt.propagate_1traversal_postorder(s.sched[0]).all()
    ll = bt.integratebelief(s.root, want_mu=False)[1]
    dense = np.array([densemvn.loglik_ou(s.net, s.data[0, :, 0], s.taxa, *r) for r in recs])
    assert np.max(np.abs(ll / dense - 1)) <= DENSE_TOL


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("pattern", [None, "clade+scatter"], ids=["full", "missing"])
def test_invalid_record_in_grid(backend, pattern):
    # records with sigma2 <= 0, alpha <= 0 and alpha = NaN inside a product grid: their elements fail with
    # PGBP_STATUS(0x7ffffd, 1), every other element is bit-identical to the same grid without them
    s = grid_setup(get_lib(backend), pattern)
    B = GRID_NP * GRID_ND
    bad = s.recs.copy()
    bad[0, 0] = 0.0
    bad[137, 1] = -1.0
    bad[GRID_NP - 1, 1] = math.nan
    out = {}
    for name, recs in (("good", s.recs), ("bad", bad)):
        bt = s.batch(B)
        bt.assignfactors_ou(recs, s.data, pairing="product")
        st = bt.status()
        assigned = [bt.get_belief(j) for j in range(1, len(s.case.b) + 1)]
        bt.calibrate(s.sched)
        out[name] = dict(st=st, assigned=assigned, calibrated=[bt.get_belief(j) for j in range(1, len(s.case.b) + 1)],
                         ll=bt.integratebelief(s.root, want_mu=False)[1])
    rec_of = np.arange(B) // GRID_ND
    failed = np.isin(rec_of, [0, 137, GRID_NP - 1])
    assert (out["good"]["st"] == 0).all()
    assert (out["bad"]["st"][failed] == BAD_RECORD).all() and (out["bad"]["st"][~failed] == 0).all()
    assert np.array_equal(out["good"]["ll"][~failed], out["bad"]["ll"][~failed])
    for key in ("assigned", "calibrated"):
        for x, y in zip(out["good"][key], out["bad"][key]):
            for u, v in zip(x, y):
                assert np.array_equal(u[~failed], v[~failed]), key


# ------------------------------------------------------------------ posterior node moments
@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("root,pattern", [("fixed", None), ("random", None), ("fixed", "clade+tipall"),
                                          ("random", "sisters+scatter")])
def test_node_moments_match_dense_conditional(backend, root, pattern):
    # posterior mean m_v + C_v,o S^-1 (y - m_o) and variance C_vv - C_v,o S^-1 C_o,v of every node in scope
    s = OU(get_lib(backend), 24, 3, 41, root, 3, 3, pattern)
    s.data = np.concatenate([simulate(s.net, s.taxa, s.recs[k], 1, 50 + k) for k in range(3)])
    s.data[:, s.mask] = np.nan
    bt = s.batch(3)
    bt.assignfactors_ou(s.recs, s.data)
    assert bt.calibrate(s.sched)[0].all()
    mu, cov, ins = bt.node_moments()
    nodes = np.flatnonzero(ins[:, 0])
    assert len(nodes) >= 10 and not ins[0, 0] == (root == "fixed")
    idx = {x.name: i for i, x in enumerate(s.net.vec_node)}
    obs = np.array([idx[t] for t, m in zip(s.taxa, s.mask) if not m])
    for e in range(3):
        m, _, C = densemvn.ou_moments(s.net, *s.recs[e])
        y = s.data[e, ~s.mask, 0]
        K = np.linalg.solve(C[np.ix_(obs, obs)], C[np.ix_(obs, nodes)]).T
        assert relerr(mu[e, nodes, 0], m[nodes] + K @ (y - m[obs])) <= DENSE_TOL, e
        assert relerr(cov[e, nodes, 0, 0], np.diag(C[np.ix_(nodes, nodes)] - K @ C[np.ix_(obs, nodes)])) <= DENSE_TOL, e
        assert np.isnan(mu[e, ~ins[:, 0], 0]).all()


# ------------------------------------------------------------------ loopy cluster graphs
class LoopyOU:
    """A Newick network of the reference goldens with a loopy cluster graph and B data sets of one OU record."""

    def __init__(self, lib, name, method, root, B=3, seed=0):
        net, taxa, _ = network(name)
        self.rec = records(1, root, 60 + seed)[0]
        self.rec[1] = 0.8  # alpha: q well inside (0, 1) on these unit-scale networks
        self.case = Case(net, method, np.zeros((len(taxa), 1)), taxa, ou_model(self.rec), lib)
        self.net, self.taxa, self.p, self.B = self.case.net, taxa, 1, B
        self.data = simulate(self.net, taxa, self.rec, B, 70 + seed)
        self.sched = self.case.sched

    def batch(self, B=None, **kw):
        return pgbp_b200.BatchedClusterGraphBelief(self.case.plan, B or self.B, **kw)

    def oracle(self, e):
        return self.case.oracle_cgb(tbl=self.data[e])

    def dense_means(self, e):
        """E[X | y] of every node: m + C[:, o] S^-1 (y - m_o) (fixed and proper root); for an improper root,
        X = c + w r + D with r flat, and r is replaced by its GLS estimate (the limit v -> inf)."""
        m, w, C = densemvn.ou_moments(self.net, *self.rec)
        idx = {x.name: i for i, x in enumerate(self.net.vec_node)}
        o = np.array([idx[t] for t in self.taxa])
        y = self.data[e, :, 0]
        if math.isinf(self.rec[4]):
            c = m - w * self.rec[3]
            Siw = np.linalg.solve(C[np.ix_(o, o)], w[o])
            r = float(Siw @ (y - c[o])) / float(Siw @ w[o])
            m = c + w * r
        return m + C[:, o] @ np.linalg.solve(C[np.ix_(o, o)], y - m[o])


LOOPY_CASES = [
    ("bethe-lipson-fixed-onschedule", "lipson", "bethe", "fixed", "onschedule"),
    ("ltrip-lipson-random-bycluster", "lipson", "ltrip", "random", "bycluster"),
    ("bethe-mateescu-improper-bynodesubtree", "mateescu", "bethe", "improper", "bynodesubtree"),
    ("ltrip-mateescu-random-onschedule", "mateescu", "ltrip", "random", "onschedule"),
]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("cs", LOOPY_CASES, ids=lambda c: c[0])
def test_loopy_ou_matches_oracle_and_dense_fixed_point(backend, cs):
    # OU factors have h != 0 before any evidence.  Beliefs, residuals, KL divergences and the factored energy (from
    # the eager OU factor snapshot) against the oracle after regularisation and 3 iterations; then, at the fixed
    # point, every cluster mean against the dense posterior mean
    _, name, method, root, reg = cs
    s = LoopyOU(get_lib(backend), name, method, root)
    bt = s.batch()
    bt.assignfactors_ou([s.rec], s.data)
    assert (bt.status() == 0).all()
    cgbs = [s.oracle(e) for e in range(s.B)]
    check_all_beliefs(s.case, bt, cgbs, floor=FLOOR)
    regularize(s, reg, bt, cgbs)
    assert s.case.plan.nsepsets >= s.case.nclusters  # the cluster graph has cycles
    for it in range(1, 4):
        succ, iscal = bt.calibrate(s.sched, 1, update_residualkldiv=True)
        ref = [OBP.calibrate(c, s.sched, 1, update_residualkldiv=True) for c in cgbs]
        assert list(succ) == [r[0] for r in ref] and list(iscal) == [r[1] for r in ref], it
        assert succ.all() and (bt.status() == 0).all()
        check_vs_oracle(s, bt, cgbs, it)
    for _ in range(40):
        assert bt.calibrate(s.sched, 10)[0].all()
        if max_residual(s, bt) <= 1e-12:
            break
    assert max_residual(s, bt) <= 1e-12
    dense = [s.dense_means(e) for e in range(s.B)]
    for j in range(1, s.case.nclusters + 1):
        b = s.case.b[j - 1]
        pos = [nl - 1 for ni, nl in enumerate(b.nodelabel) if b.inscope[0, ni]]
        mu, _ = bt.integratebelief(j)
        for e in range(s.B):
            assert relerr(mu[e], dense[e][pos]) <= DENSE_TOL, (j, e)


# ------------------------------------------------------------------ shared-precision batches
@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("pattern", [None, "clade+tipall"], ids=["full", "missing"])
@pytest.mark.parametrize("group,nrec", [(4, 3), (37, 2)])
def test_shared_precision_bit_identical(backend, pattern, group, nrec):
    # product pairing, groups of `group` elements per record: J once per group in the group batch, h and g per
    # element; equal to own-J batches bit for bit after assignment and after calibration
    nd = 2 * group
    s = OU(get_lib(backend), 18, 3, 81, "random", nrec, nd, pattern)
    B = nrec * nd
    out = {}
    for name, gs in (("own", 0), ("shared", group)):
        bt = s.batch(B, shared_precision_group=gs)
        bt.assignfactors_ou(s.recs, s.data, pairing="product")
        assigned = [bt.get_belief(j) for j in range(1, len(s.case.b) + 1)]
        succ, iscal = bt.calibrate(s.sched, 2, update_residualkldiv=True)
        out[name] = dict(succ=succ, iscal=iscal, st=bt.status(), ll=bt.integratebelief(s.root, want_mu=False)[1],
                         fe=bt.factored_energy(),
                         arrays=assigned + [bt.get_belief(j) for j in range(1, len(s.case.b) + 1)])
    a, b_ = out["own"], out["shared"]
    assert a["succ"].all() and (a["st"] == 0).all()
    for key in ("succ", "iscal", "st", "ll", "fe"):
        assert np.array_equal(a[key], b_[key]), key
    for x, y in zip(a["arrays"], b_["arrays"]):
        for u, v in zip(x, y):
            assert np.array_equal(u, v)
    dense = np.array([s.dense(e // nd, e % nd) for e in (0, B - 1)])
    assert np.max(np.abs(a["ll"][[0, B - 1]] / dense - 1)) <= DENSE_TOL


# ------------------------------------------------------------------ the Brownian-motion limit
ULP = 2.2e-16


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("net", ["named", "synth"])
@pytest.mark.parametrize("root", ROOTS)
def test_brownian_motion_limit(backend, net, root):
    # theta = mu, alpha -> 0.  The device forms 1 - q^2 as the reference does, which loses digits when alpha t is
    # small: against the expm1 dense likelihood its relative error stays below ULP / (alpha t_min) (the bound stated
    # on pgbp_assign_factors_ou), so within DENSE_TOL for alpha t_min >= 1e-6.  The dense OU likelihood itself tends
    # to densemvn.loglik_bm at the same sigma2 (within ~alpha times the total edge length); on the named network
    # (t_min = 0.1) alpha = 1e-9 brings the device within 1e-8 of it as well
    lib = get_lib(backend)
    s2, mu = 1.3, 0.4
    v = {"fixed": 0.0, "random": 0.7, "improper": math.inf}[root]
    if net == "named":
        tbl = TBL[:, [1]]
        case = Case(GOLD["netstr_named"], "cliquetree", tbl, TAXA, ou_model((s2, 1.0, mu, mu, v)), lib,
                    schedule="spanningtree")
        N, taxa, data, sched = case.net, TAXA, np.stack([tbl, tbl + 0.25, 2 * tbl]), case.sched
    else:
        s = OU(lib, 12, 2, 91, root, 1, 3)
        N, taxa, data, sched, case = s.net, s.taxa, s.data, s.sched, s.case
    tmin = min(e.length for e in N.edges)
    bm = np.array([densemvn.loglik_bm(N, data[e], taxa, lambda ed: np.array([[s2]]), [mu],
                                      rootvar=np.array([[v]]) if root == "random" else None,
                                      improper=root == "improper") for e in range(3)])
    for alpha in (1e-2 / tmin, 1e-4 / tmin, 1e-6 / tmin, 1e-8 / tmin, 1e-9, 1e-12):
        at = alpha * tmin
        rec = (s2, alpha, mu, mu, v)
        bt = pgbp_b200.BatchedClusterGraphBelief(case.plan, 3)
        bt.assignfactors_ou([rec], data)
        assert (bt.status() == 0).all()
        assert bt.propagate_1traversal_postorder(sched[0]).all()
        ll = bt.integratebelief(sched[0][2][0], want_mu=False)[1]
        dense = np.array([densemvn.loglik_ou(N, data[e, :, 0], taxa, *rec) for e in range(3)])
        err = np.max(np.abs(ll / dense - 1))
        assert err <= max(ULP / at, 1e-14), (alpha, err)
        if at >= 1e-6:
            assert err <= DENSE_TOL
        if alpha <= 1e-9:
            assert np.max(np.abs(dense / bm - 1)) <= 1e-8, alpha
        if net == "named" and alpha == 1e-9:
            assert np.max(np.abs(ll / bm - 1)) <= 1e-8, (ll, bm)
