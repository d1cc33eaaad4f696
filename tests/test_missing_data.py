"""Missing data (trait-level scopes) on synthetic level-1 networks with short edges.

A node keeps a trait in its scope only if some tip below it observes that trait, so missing cells change the
beliefs' dimensions and route factor assignment through the scoped K1 path.  The log-likelihood is checked against
the dense multivariate-normal likelihood of the observed cells (oracle/densemvn.py: no belief propagation at all),
beliefs against the oracle, posterior moments against the dense conditional Gaussian; and since partial scopes give
message shapes that are not multiples of p, the plans below must reach given message-kernel branches, on which every
kernel variant and the shared-precision batch must agree bit for bit."""
import math
import os
import sys
from collections import Counter

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
from test_parity import check_all_beliefs  # noqa: E402
from workloads import synth  # noqa: E402

DENSE_TOL = 1e-9  # the dense solve is the looser side (as in test_synth)
TOL = 1e-10
SCOPED_MAXN = 48  # PGBP_SCOPED_MAXN: variables of one node family in the scoped K1 path


# ------------------------------------------------------------------ networks, missingness patterns, models
def clades(tab):
    """children of every node, and the set of tips below it (nodes are in preorder)."""
    n = tab["nnodes"]
    kids = [[] for _ in range(n)]
    for v in range(n):
        for (q, _, _, _) in tab["parents"][v]:
            kids[q].append(v)
    below = [set() for _ in range(n)]
    for v in reversed(range(n)):
        below[v] = {v} if tab["leaf"][v] else set().union(*(below[c] for c in kids[v]))
    return kids, below


def missing_mask(tab, tips, p, pattern, seed):
    """(ntips, p) bool, True = missing.  Patterns (combine with '+'):
    sisters  the last trait at both tips of the first cherry (two tips that are the only children of their parent)
    clade    the first trait at every tip of the smallest clade of >= 4 tips (not the whole network)
    onetip   trait min(1, p-1) observed at the last tip only
    tipall   every trait at the first tip
    scatter  single cells with probability 1/4, each trait kept at >= 2 tips"""
    kids, below = clades(tab)
    row = {v: i for i, v in enumerate(tips)}
    mask = np.zeros((len(tips), p), dtype=bool)
    for pat in pattern.split("+"):
        if pat == "sisters":
            v = next(v for v in range(tab["nnodes"]) if len(kids[v]) == 2 and all(tab["leaf"][c] for c in kids[v]))
            for c in kids[v]:
                mask[row[c], p - 1] = True
        elif pat == "clade":
            v = min((v for v in range(1, tab["nnodes"]) if 4 <= len(below[v]) <= len(tips) - 2), key=lambda v: len(below[v]))
            for c in below[v]:
                mask[row[c], 0] = True
        elif pat == "onetip":
            mask[:-1, min(1, p - 1)] = True
        elif pat == "tipall":
            mask[0, :] = True
        elif pat == "scatter":
            rng = np.random.default_rng(seed)
            sc = rng.random(mask.shape) < 0.25
            for t in range(p):
                keep = np.flatnonzero(~sc[:, t])
                if keep.size < 2:
                    sc[rng.choice(len(tips), 2, replace=False), t] = False
            mask |= sc
        else:
            raise ValueError(pattern)
    assert (~mask).sum(axis=0).min() >= 1, "every trait observed somewhere"
    return mask


class Setup:
    """A synthetic network with missing cells: oracle objects, product plan (through the oracle front-end, which
    gives the plan its scoped families), model, B simulated data sets with NaN at the missing cells, and the
    parameter vector.  hetero: every hybrid's minor parent edge has rate colour 1 (its major edge colour 0), so
    hybrid families take the p x p inverse of their summed variances."""

    def __init__(self, lib, ntips, nretic, seed, p, pattern, rk="full", root="fixed", hetero=False, B=3):
        self.p = p
        tab = self.tab = synth.level1_network(ntips, nretic, seed)
        plan = synth.cliquetree_plan(tab, p)
        self.net, cg, sched, self.taxa = synth_oracle_objects(tab, plan)
        rng = np.random.default_rng(1000 * seed + p)
        self.col = {}
        for v in range(tab["nnodes"]):
            for k, (_, _, _, e) in enumerate(tab["parents"][v]):
                self.col[e] = 1 if hetero and k == 0 and len(tab["parents"][v]) == 2 else 0
        self.Rs = []
        for _ in range(2 if hetero else 1):
            if rk == "diag":
                self.Rs.append(np.diag(rng.uniform(0.5, 2.0, size=p)))
            else:
                A = rng.normal(size=(p, p))
                self.Rs.append(A @ A.T / p + 0.1 * np.eye(p))
        self.mu = rng.normal(size=p)
        A = rng.normal(size=(p, p))
        self.V = {"fixed": None, "random": A @ A.T / p + 0.5 * np.eye(p), "improper": np.diag(np.full(p, math.inf))}[root]
        self.root = root
        self.model = M.HeterogeneousBrownianMotion(self.Rs, {e: c + 1 for e, c in self.col.items()}, self.mu, self.V)
        tips = plan["tip_nodes"]
        self.mask = missing_mask(tab, tips, p, pattern, seed)
        sim = synth.simulate_tips(plan, lambda v, k: self.Rs[self.col[tab["parents"][v][k][3]]], B, seed + 7, self.mu)
        sim[:, self.mask] = np.nan
        self.data = sim
        self.case = Case(self.net, "cliquetree", sim[0], self.taxa, self.model, lib, schedule=lambda c: sched, cg=cg,
                         edge_color=lambda e: self.col[e])
        assert self.case.plan.families.get("mem_tpos") is not None
        self.params = pgbp_b200.bm_params(self.Rs, self.mu, self.V)
        self.ncolors = len(self.Rs)

    def dense(self, e):
        return densemvn.loglik_bm(self.net, self.data[e], self.taxa, lambda ed: self.Rs[self.col[ed.number]], self.mu,
                                  rootvar=self.V if self.root == "random" else None, improper=self.root == "improper")

    def batch(self, B=None, **kw):
        return pgbp_b200.BatchedClusterGraphBelief(self.case.plan, B or len(self.data), **kw)

    def message_shapes(self):
        """(I, S) of every message of both traversals: integrated and kept (sepset) dimensions."""
        dims = self.case.plan.belief_dim
        out = Counter()
        for direction in (0, 1):
            lv = self.case.plan.levels(0, direction)
            for f, s in zip(lv["frm"], lv["sepset"]):
                out[(dims[f] - dims[s], dims[s])] += 1
        return out


def medium_kernel(I, S):
    """Kernel that the automatic mode (set_coop_mode(-1)) launches for a message of shape (I, S), restated from
    launch_medium (csrc/pgbp_message_medium.cu) with its shared-memory budgets; None for the small-shape class."""
    M_ = I + S
    if I == 0 or M_ <= 12:
        return None
    tri = I * (I + 1) // 2 + I * S + I
    fits = I <= 32 and 8 * 32 * tri + 4 * (M_ * (M_ + 3) // 2 + S * (S + 3) // 2 + 2) <= 200 * 1024
    mw = 8 * 32 * (tri + 2) + 4 * 32 * (2 + 8) + 2 * (M_ * (M_ + 1) // 2 + M_ + S * (S + 1) // 2 + S + 4)
    if 12 <= I <= 16 and mw <= 225 * 1024:
        return "smem_mw"
    if fits:
        return f"smem<{I}>" if I <= 16 else ("smem_rt<24>" if I <= 24 else "smem_rt<32>")
    if I <= 32 and 8 * 16 * tri <= 225 * 1024:
        mwp = 8 * 24 * (tri + 2) + 4 * 24 * (2 + 8) + 2 * (M_ * (M_ + 1) // 2 + M_ + S * (S + 1) // 2 + S + 4) + 16
        if I == 32 and mwp <= 225 * 1024:
            return "smem_mwp<32>"
        return "coop<48,16>" if M_ <= 48 else "message<64>"
    return "coop" if M_ <= 48 else "message"


# ------------------------------------------------------------------ log-likelihood against the dense Gaussian
# (id, ntips, nretic, seed, p, R, root, hetero, pattern).  Every case has a parent with a trait out of scope above a
# child that lost that trait (a cherry or clade missing it, or a lone tip below a subdivision or hybrid node missing
# everything): the family factor's rows for that parent trait are zero in exact arithmetic, roundoff in floating point.
DENSE_CASES = [
    ("sisters-p2-diag", 10, 2, 1, 2, "diag", "fixed", False, "sisters"),
    ("sisters-p2-full", 10, 2, 1, 2, "full", "fixed", False, "sisters"),
    ("sisters-p1-random", 10, 2, 1, 1, "diag", "random", False, "sisters"),
    ("clade-p3-full-random", 14, 3, 2, 3, "full", "random", False, "clade"),
    ("clade-p3-diag-improper", 14, 3, 2, 3, "diag", "improper", False, "clade"),
    ("clade-p1-improper", 14, 3, 2, 1, "diag", "improper", False, "clade"),
    ("onetip-p2-full-hetero", 9, 2, 3, 2, "full", "fixed", True, "onetip"),
    ("onetip-p5-diag-random", 9, 2, 3, 5, "diag", "random", False, "onetip"),
    ("tipall-p3-full", 8, 2, 4, 3, "full", "fixed", False, "tipall"),
    ("tipall-p5-full-improper", 8, 2, 4, 5, "full", "improper", True, "tipall"),
    ("scatter-p3-full-hetero", 12, 3, 5, 3, "full", "random", True, "scatter"),
    ("scatter-p8-diag", 10, 2, 6, 8, "diag", "fixed", False, "scatter"),
    ("all-p5-full-hetero", 16, 4, 7, 5, "full", "fixed", True, "sisters+clade+tipall+scatter"),
    ("all-p8-full-improper", 16, 4, 8, 8, "full", "improper", False, "sisters+clade+tipall+scatter"),
    ("clade-p8-full-hetero", 12, 3, 9, 8, "full", "random", True, "clade+sisters"),
    ("sisters-p16-diag", 8, 2, 10, 16, "diag", "fixed", False, "sisters+tipall"),
    ("all-p16-full-hetero", 12, 3, 11, 16, "full", "fixed", True, "sisters+clade+scatter"),
    ("onetip-p16-full-improper", 8, 2, 12, 16, "full", "improper", True, "onetip+sisters"),
]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("cs", DENSE_CASES, ids=lambda c: c[0])
def test_loglik_matches_dense_mvn(backend, cs):
    # one postorder pass: the root cluster integrates to the dense likelihood of the observed cells; after a full
    # calibration every belief (clusters and sepsets) does
    _, ntips, nretic, seed, p, rk, root, hetero, pattern = cs
    s = Setup(get_lib(backend), ntips, nretic, seed, p, pattern, rk, root, hetero)
    B = len(s.data)
    dense = np.array([s.dense(e) for e in range(B)])
    spt = s.case.sched[0]
    bt = s.batch()
    bt.assignfactors(s.params, s.data, ncolors=s.ncolors)
    assert (bt.status() == 0).all()
    assert bt.propagate_1traversal_postorder(spt).all()
    ll = bt.integratebelief(spt[2][0])[1]
    assert relerr(ll, dense) <= DENSE_TOL, (ll, dense)
    succ, _ = bt.calibrate(s.case.sched)
    assert succ.all() and (bt.status() == 0).all()
    for j in range(1, len(s.case.b) + 1):
        if bt.dimension(j) > 0:
            assert relerr(bt.integratebelief(j, want_mu=False)[1], dense) <= DENSE_TOL, j


@pytest.mark.parametrize("backend", BACKENDS)
def test_scoped_family_at_the_variable_limit(backend):
    # a hybrid family at p = 16 (3 members x 16 traits) has PGBP_SCOPED_MAXN variables, the largest the scoped K1
    # path accepts; its parent edges differ in colour, and the hybrid's clade misses a trait
    s = Setup(get_lib(backend), 8, 2, 10, 16, "sisters+clade", "full", "random", hetero=True)
    fam = s.case.plan.families
    nmem = np.diff(fam["mem_off"])
    assert nmem.max() * s.p == SCOPED_MAXN
    bt = s.batch()
    bt.assignfactors(s.params, s.data, ncolors=s.ncolors)
    assert (bt.status() == 0).all()
    succ, _ = bt.calibrate(s.case.sched)
    assert succ.all()
    dense = np.array([s.dense(e) for e in range(len(s.data))])
    for j in range(1, s.case.nclusters + 1):
        if bt.dimension(j) > 0:
            assert relerr(bt.integratebelief(j, want_mu=False)[1], dense) <= DENSE_TOL, j


# ------------------------------------------------------------------ beliefs against the oracle (small networks)
ORACLE_CASES = [
    ("sisters-p2-diag", 10, 2, 1, 2, "diag", "fixed", False, "sisters"),
    ("clade-p3-full-random", 9, 2, 13, 3, "full", "random", False, "clade"),
    ("onetip-p2-full-improper-hetero", 7, 2, 14, 2, "full", "improper", True, "onetip+tipall"),
    ("scatter-p3-diag-hetero", 8, 2, 15, 3, "diag", "fixed", True, "sisters+scatter"),
]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("cs", ORACLE_CASES, ids=lambda c: c[0])
def test_beliefs_match_oracle(backend, cs):
    # every belief after assignfactors and after calibration against the oracle; floor: a tip's missing trait
    # marginalised out of its edge factor leaves the parent's in-scope rows for that trait as roundoff of a zero
    _, ntips, nretic, seed, p, rk, root, hetero, pattern = cs
    s = Setup(get_lib(backend), ntips, nretic, seed, p, pattern, rk, root, hetero)
    B = len(s.data)
    bt = s.batch()
    bt.assignfactors(s.params, s.data, ncolors=s.ncolors)
    assert (bt.status() == 0).all()
    cgbs = [s.case.oracle_cgb(tbl=s.data[e]) for e in range(B)]
    check_all_beliefs(s.case, bt, cgbs, floor=1e-3)
    succ, _ = bt.calibrate(s.case.sched)
    assert succ.all()
    for cgb in cgbs:
        OBP.calibrate(cgb, s.case.sched)
    check_all_beliefs(s.case, bt, cgbs, floor=1e-3)
    root = s.case.sched[0][2][0]
    ll = bt.integratebelief(root)[1]
    for e in range(B):
        assert abs(ll[e] / OBP.integratebelief_cgb(cgbs[e], root)[1] - 1) <= TOL
        assert abs(ll[e] / s.dense(e) - 1) <= DENSE_TOL


# ------------------------------------------------------------------ message shapes that only partial scopes give
# p = 8 / 16 plans whose (I, S) histograms reach the medium-shape kernels that whole-node scopes never launch at
# these p (pinned here so that the coverage cannot vanish when the network generator changes)
SHAPE_CASES = {
    8: (dict(ntips=10, nretic=3, seed=6, pattern="scatter"),
        ["smem<11>", "smem_mw"]),
    16: (dict(ntips=10, nretic=3, seed=7, pattern="sisters+clade+tipall+scatter"),
         ["smem_rt<24>", "coop<48,16>", "smem_mwp<32>"]),
}


def shape_setup(lib, p, B, hetero=True):
    kw, _ = SHAPE_CASES[p]
    return Setup(lib, kw["ntips"], kw["nretic"], kw["seed"], p, kw["pattern"], "full", "fixed", hetero, B=B)


@pytest.mark.parametrize("p", [8, 16])
def test_partial_scopes_reach_the_medium_kernels(p):
    s = shape_setup(get_lib("emul"), p, 1)
    shapes = s.message_shapes()
    kernels = {medium_kernel(I, S) for (I, S) in shapes}
    for k in SHAPE_CASES[p][1]:
        assert k in kernels, (k, sorted(shapes))
    if p == 8:
        assert any(I == 11 and S >= 2 for I, S in shapes)
        assert any(12 <= I <= 16 and (I % p or S % p) for I, S in shapes)
    else:
        assert any(17 <= I <= 23 for I, S in shapes)
        assert any(I < 32 and medium_kernel(I, S) == "coop<48,16>" for I, S in shapes)
        assert any(I == 32 and S != 16 for I, S in shapes)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("p", [8, 16])
def test_partial_scope_shapes_every_kernel_variant_bit_identical(backend, p):
    # the automatic kernel choice, the single- and multi-warp shared-memory kernels and the 4 / 8-lane cooperative
    # kernels against the one-thread-per-element generic kernel, bit for bit; B = 37 leaves ragged tiles
    lib = get_lib(backend)
    B = 37
    s = shape_setup(lib, p, B)
    out = {}
    for mode in (0, -1, 1, 2, 4, 8):
        bt = s.batch()
        bt.set_coop_mode(mode)
        bt.assignfactors(s.params, s.data, ncolors=s.ncolors)
        succ, iscal = bt.calibrate(s.case.sched)
        out[mode] = dict(succ=succ, iscal=iscal, st=bt.status(), ll=bt.integratebelief(s.case.sched[0][2][0])[1],
                         beliefs=[bt.get_belief(j) for j in range(1, len(s.case.b) + 1)],
                         res=[bt.get_residual(s.case.nclusters + 1 + j, s.case.plan.sepset_clusters[j][k] + 1)
                              for j in range(s.case.plan.nsepsets) for k in (0, 1)])
    ref = out[0]
    assert ref["succ"].all() and (ref["st"] == 0).all()
    dense = np.array([s.dense(e) for e in (0, B - 1)])
    assert relerr(ref["ll"][[0, B - 1]], dense) <= DENSE_TOL
    for mode in (-1, 1, 2, 4, 8):
        o = out[mode]
        for key in ("succ", "iscal", "st", "ll"):
            assert np.array_equal(ref[key], o[key]), (mode, key)
        for x, y in zip(ref["beliefs"] + ref["res"], o["beliefs"] + o["res"]):
            for u, v in zip(x, y):
                assert np.array_equal(u, v), mode


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("p,nth,nd", [(8, 1, 37), (16, 1, 37), (8, 2, 128), (16, 2, 128)])
def test_partial_scope_shapes_shared_precision_bit_identical(backend, p, nth, nd):
    # shared-precision batches (J once per group of nd elements) on the same plans: equal to own-J batches bit for
    # bit.  One group of 37 has ragged tiles; groups of 128 run the bulk-copy element pass
    lib = get_lib(backend)
    B = nth * nd
    s = shape_setup(lib, p, nd)
    rng = np.random.default_rng(p + nth)
    params = np.stack([s.params] + [pgbp_b200.bm_params([R * rng.uniform(0.5, 2) for R in s.Rs], s.mu)
                                    for _ in range(nth - 1)])
    out = {}
    for name, group in (("own", 0), ("shared", nd)):
        bt = s.batch(B, shared_precision_group=group)
        bt.assignfactors(params, s.data, ncolors=s.ncolors, pairing="product")
        assigned = [bt.get_belief(j) for j in range(1, len(s.case.b) + 1)]
        succ, iscal = bt.calibrate(s.case.sched, 2, update_residualkldiv=True)
        out[name] = dict(succ=succ, iscal=iscal, st=bt.status(), ll=bt.integratebelief(s.case.sched[0][2][0])[1],
                         fe=bt.factored_energy(), arrays=assigned + [bt.get_belief(j) for j in range(1, len(s.case.b) + 1)]
                         + [bt.get_residual(s.case.nclusters + 1 + j, s.case.plan.sepset_clusters[j][k] + 1)
                            for j in range(s.case.plan.nsepsets) for k in (0, 1)])
    a, b_ = out["own"], out["shared"]
    assert a["succ"].all() and (a["st"] == 0).all()
    for key in ("succ", "iscal", "st", "ll", "fe"):
        assert np.array_equal(a[key], b_[key]), key
    for x, y in zip(a["arrays"], b_["arrays"]):
        for u, v in zip(x, y):
            assert np.array_equal(u, v)
    assert abs(a["ll"][nd - 1] / s.dense(nd - 1) - 1) <= DENSE_TOL  # parameter set 0, last data set


# ------------------------------------------------------------------ posterior moments of partially observed nodes
@pytest.mark.parametrize("backend", BACKENDS)
def test_node_moments_partial_scopes_match_dense_conditional(backend):
    # a clade misses trait 0: its internal nodes keep traits 1, 2 only.  Their posterior mean and covariance given
    # the observed cells, against the dense conditional Gaussian of the network covariance (fixed root)
    s = Setup(get_lib(backend), 14, 3, 2, 3, "clade", "full", "fixed", B=2)
    p, n = s.p, s.tab["nnodes"]
    bt = s.batch()
    bt.assignfactors(s.params, s.data, ncolors=s.ncolors)
    assert bt.calibrate(s.case.sched)[0].all()
    mu, cov, ins = bt.node_moments()
    partial = [v for v in range(n) if 0 < ins[v].sum() < p]
    assert len(partial) >= 3 and all(not s.tab["leaf"][v] for v in partial)
    C = densemvn.network_covariance(s.net, lambda ed: s.Rs[s.col[ed.number]], p)
    idx = {nd.name: i for i, nd in enumerate(s.net.vec_node)}
    nchecked = 0
    for e in range(len(s.data)):
        obs, y = [], []
        for r, name in enumerate(s.taxa):
            for t in range(p):
                if not s.mask[r, t]:
                    obs.append(idx[name] * p + t)
                    y.append(s.data[e, r, t])
        obs, y = np.array(obs), np.array(y)
        mobs = s.mu[obs % p]
        for v in partial:
            T = np.flatnonzero(ins[v])
            q = v * p + T
            K = np.linalg.solve(C[np.ix_(obs, obs)], C[np.ix_(obs, q)]).T
            cmean = s.mu[T] + K @ (y - mobs)
            ccov = C[np.ix_(q, q)] - K @ C[np.ix_(obs, q)]
            assert np.isnan(mu[e, v, ~ins[v]]).all()
            assert relerr(mu[e, v, T], cmean) <= DENSE_TOL
            assert relerr(cov[e, v][np.ix_(T, T)], ccov) <= DENSE_TOL
            nchecked += 1
    assert nchecked == len(partial) * len(s.data)
