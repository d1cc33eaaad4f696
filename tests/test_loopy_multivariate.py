"""Loopy belief propagation with several traits (p >= 2) on Bethe, LTRIP and join-graph cluster graphs.

Anchors: the oracle (oracle/bp.py) for beliefs, residuals, flags, KL divergences and factored energies after
regularisation and after each of the first iterations; and, sharing no code with belief propagation, the dense
Gaussian posterior of the network (oracle/densemvn.py) for the belief means at the fixed point, which loopy Gaussian
BP gets exactly (Weiss & Freeman 2001; its variances are not exact and are not checked).  On the device, the kernel
variants that loopy schedules reach at these shapes (shared-memory message kernels, the walk kernel, the tile walk,
the shared-precision group pass, CUDA-graph replay, element pipelining) must agree with each other bit for bit; the
plans below are pinned to reach them."""
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
from oracle.network import readnewick  # noqa: E402
from test_missing_data import medium_kernel, missing_mask  # noqa: E402
from test_parity import GOLD, check_all_beliefs  # noqa: E402
from workloads import synth  # noqa: E402

TOL = 1e-10
KL_TOL = 1e-8
KL_ABS = 1e-6      # below this a KL divergence is the cancellation of O(1) log-determinants: compared absolutely
DENSE_TOL = 1e-9
# entries that are zero in exact arithmetic (h of beliefs that no data has reached yet, under a flat root prior) are
# roundoff of either sign on both sides: differences are measured against max(|reference|, FLOOR), as in
# test_missing_data
FLOOR = 1e-3
ATOL_RESID = 1e-5  # iscalibrated_residnorm's tolerance (src/beliefs.jl:994-1003)
TW_MAXM = 4        # PGBP_TW_MAXM: largest sender dimension of the tile walk
WALK_MAXP = 4      # PGBP_WALK_MAXP
T0_MAX = 12        # PGBP_T0_MAX


# ------------------------------------------------------------------ networks, models, data
def network(name):
    """(Network, taxa, synthetic table or None).  name: a Newick network of the reference goldens, or
    'synth:<ntips>:<nretic>:<seed>' for a level-1 network of workloads/synth.py (nodes n<preorder index>)."""
    if name.startswith("synth:"):
        ntips, nretic, seed = (int(x) for x in name.split(":")[1:])
        tab = synth.level1_network(ntips, nretic, seed)
        net, _, _, taxa = synth_oracle_objects(tab, synth.cliquetree_plan(tab, 1))
        return net, taxa, tab
    taxa = {"lipson": GOLD["lipson_taxa"], "mateescu": ["g", "d"], "netstr_level3": ["A", "B"],
            "netstr_unnamed": ["A", "B", "C", "D"]}[name]
    return readnewick(GOLD[name]), taxa, None


def newick_mask(taxa, p, pattern):
    """(ntips, p) bool, True = missing.  onetip: trait min(1, p-1) observed at the last tip only (every node that
    is not an ancestor of that tip loses the trait); tipall: every trait of the first tip."""
    mask = np.zeros((len(taxa), p), dtype=bool)
    for pat in pattern.split("+"):
        if pat == "onetip":
            mask[:-1, min(1, p - 1)] = True
        elif pat == "tipall":
            mask[0, :] = True
        else:
            raise ValueError(pattern)
    return mask


class Loopy:
    """A network, a loopy cluster graph of it with every spanning tree of the schedule, a Brownian-motion model and
    B data sets simulated from it (from the dense network covariance, so any network works).
    rk: "full" (MvFull), "diag" (MvDiag) or "hetero" (HeterogeneousBrownianMotion: minor hybrid edges colour 1).
    root: "fixed" (at mu), "random" (prior N(mu, V)) or "improper" (flat prior).
    missing: a pattern of test_missing_data.missing_mask (newick_mask for Newick networks): cells set to NaN in
    every data set, so that nodes above them lose traits from their scope."""

    def __init__(self, lib, name, method, p, rk="full", root="fixed", B=3, seed=0, missing=None, **cgkw):
        self.p, self.root, self.rk = p, root, rk
        net, taxa, tab = network(name)
        rng = np.random.default_rng(1000 + 17 * p + seed)
        ncol = 2 if rk == "hetero" else 1
        self.Rs = []
        for _ in range(ncol):
            if rk == "diag":
                self.Rs.append(np.diag(rng.uniform(0.5, 2.0, size=p)))
            else:
                A = rng.normal(size=(p, p))
                self.Rs.append(A @ A.T / p + 0.2 * np.eye(p))
        self.mu = rng.normal(size=p)
        A = rng.normal(size=(p, p))
        self.V = {"fixed": None, "random": A @ A.T / p + 0.5 * np.eye(p),
                  "improper": np.diag(np.full(p, math.inf))}[root]
        if rk == "diag" and root == "random":
            self.V = np.diag(np.diag(self.V))
        mask = np.zeros((len(taxa), p), dtype=bool)
        if missing:
            mask = missing_mask(tab, [int(t[1:]) for t in taxa], p, missing, seed) if tab else newick_mask(taxa, p, missing)
        self.mask = mask
        tbl0 = np.where(mask, np.nan, 0.0)
        # colours by edge number: minor hybrid edges 1, every other edge 0
        self.col = {}
        for e in net.edges:
            self.col[e.number] = 1 if (rk == "hetero" and e.hybrid and e.gamma < 0.5) else 0
        if rk == "diag":
            vv = None if self.V is None else np.diag(self.V)
            model = M.MvDiagBrownianMotion(np.diag(self.Rs[0]), self.mu, vv)
        elif rk == "full":
            model = M.MvFullBrownianMotion(self.Rs[0], self.mu, self.V)
        else:
            model = M.HeterogeneousBrownianMotion(self.Rs, {e: c + 1 for e, c in self.col.items()}, self.mu, self.V)
        self.model = model
        self.case = Case(net, method, tbl0, taxa, model, lib, edge_color=lambda e: self.col[e], **cgkw)
        self.net, self.taxa = self.case.net, taxa
        self.params = pgbp_b200.bm_params(self.Rs, self.mu, self.V)
        self.ncolors = ncol
        # simulated tips: y = mu + chol(C_tips) z  (C: network covariance, with the root prior when it is proper)
        self.C0 = densemvn.network_covariance(self.net, self.rate, p)
        C = densemvn.network_covariance(self.net, self.rate, p, self.V if root == "random" else None)
        idx = {nd.name: i for i, nd in enumerate(self.net.vec_node)}
        self.tip_pos = np.array([idx[t] * p + k for t in taxa for k in range(p)])
        L = np.linalg.cholesky(C[np.ix_(self.tip_pos, self.tip_pos)])
        z = np.random.default_rng(7 + seed).normal(size=(B, len(self.tip_pos)))
        data = (np.tile(self.mu, len(taxa)) + z @ L.T).reshape(B, len(taxa), p)
        data[:, mask] = np.nan
        self.data = data
        self.B = B

    def rate(self, edge):
        return self.Rs[self.col[edge.number]]

    @property
    def sched(self):
        return self.case.sched

    def batch(self, B=None, **kw):
        return pgbp_b200.BatchedClusterGraphBelief(self.case.plan, B or self.B, **kw)

    def oracle(self, e):
        return self.case.oracle_cgb(tbl=self.data[e])

    def message_shapes(self):
        """Counter of (I, S) over the messages of every tree and direction: integrated and kept dimensions."""
        dims = self.case.plan.belief_dim
        out = Counter()
        for t in range(len(self.case.plan.trees)):
            for direction in (0, 1):
                lv = self.case.plan.levels(t, direction)
                for f, s in zip(lv["frm"], lv["sepset"]):
                    out[(dims[f] - dims[s], dims[s])] += 1
        return out

    def dense_means(self, e):
        """Posterior mean of every node state given the observed tip cells of data set e (node-major, trait-minor).
        fixed root: X = mu + D with D ~ N(0, C0) (C0: covariance with a fixed root), so
            E[X | y] = mu + C0[:, o] C0[o, o]^-1 (y - mu_o).
        random root: the same with the covariance C that includes the prior V of the root.
        improper root: X = 1 r + D, r flat.  Given r, E[X | y, r] = r + C0[:, o] C0[o, o]^-1 (y - r_o) is linear in
        r, and the posterior mean of r under a flat prior is the GLS estimate
            r^ = (A' S^-1 A)^-1 A' S^-1 y,   S = C0[o, o],  A = the trait indicator of the observed cells,
        so E[X | y] = r^ + C0[:, o] S^-1 (y - A r^) (the universal-kriging predictor; the limit V -> inf of the
        random-root mean)."""
        p = self.p
        obs_mask = ~self.mask.reshape(-1)
        o = self.tip_pos[obs_mask]
        y = self.data[e].reshape(-1)[obs_mask]
        tr = o % p
        n = len(self.net.vec_node)
        C = self.C0 if self.root != "random" else densemvn.network_covariance(self.net, self.rate, p, self.V)
        S = C[np.ix_(o, o)]
        if self.root == "improper":
            A = np.zeros((o.size, p))
            A[np.arange(o.size), tr] = 1.0
            SiA = np.linalg.solve(S, A)
            m = np.linalg.solve(A.T @ SiA, SiA.T @ y)
        else:
            m = self.mu
        return np.tile(m, n) + C[:, o] @ np.linalg.solve(S, y - m[tr])

    def belief_positions(self, j):
        """Positions in dense_means of the variables of cluster j (1-based), in the belief's order."""
        b = self.case.b[j - 1]
        return [(nl - 1) * self.p + t for ni, nl in enumerate(b.nodelabel) for t in range(self.p) if b.inscope[t, ni]]


def regularize(s, reg, bt, cgbs):
    if reg == "bycluster":
        bt.regularizebeliefs_bycluster()
        for c in cgbs:
            OBP.regularizebeliefs_bycluster(c, s.case.cg)
    elif reg == "onschedule":
        bt.regularizebeliefs_onschedule()
        for c in cgbs:
            OBP.regularizebeliefs_onschedule(c, s.case.cg)
    else:
        prog = OBP.bynodesubtree_program(cgbs[0] if cgbs else s.oracle(0), s.case.cg)
        bt.regularizebeliefs_bynodesubtree(prog)
        for c in cgbs:
            OBP.regularizebeliefs_bynodesubtree(c, s.case.cg)


def directed_messages(s):
    """(sepset belief index, receiving cluster index, sending cluster index) of both messages of every sepset,
    1-based belief indices."""
    plan = s.case.plan
    out = []
    for j in range(plan.nsepsets):
        a, b = plan.sepset_clusters[j]
        out += [(s.case.nclusters + 1 + j, a + 1, b + 1), (s.case.nclusters + 1 + j, b + 1, a + 1)]
    return out


def snapshot(s, bt):
    """Everything a calibration leaves in a batch: beliefs, residuals (dJ, dh, flag, KL), status, energies."""
    return dict(st=bt.status(), fe=bt.factored_energy(),
                beliefs=[bt.get_belief(j) for j in range(1, len(s.case.b) + 1)],
                res=[bt.get_residual(sj, to) for (sj, to, _) in directed_messages(s)])


def assert_same(a, b, keys=(), elems=None, what=""):
    """Bit-for-bit equality of two snapshots (and of the extra per-element arrays `keys`); elems: element mask of
    the belief / residual / energy comparison (elements with a failed message hold undefined beliefs)."""
    sel = slice(None) if elems is None else elems
    assert np.array_equal(a["st"], b["st"]), what
    for k in keys:
        assert np.array_equal(a[k], b[k]), (what, k)
    assert np.array_equal(a["fe"][sel], b["fe"][sel], equal_nan=True), what
    for x, y in zip(a["beliefs"] + a["res"], b["beliefs"] + b["res"]):
        for u, v in zip(x, y):
            assert np.array_equal(u[sel], v[sel], equal_nan=True), what


# ------------------------------------------------------------------ 1. beliefs, residuals, KL and energies vs the oracle
# (id, network, method, cluster-graph options, p, model, root, regulariser, missing cells).  Loopy graphs only:
# the level-1 synthetic networks have triangles for cycles, which the cluster graphs absorb into one cluster.
ORACLE_CASES = [
    ("bethe-lipson-p2-full-fixed-onschedule", "lipson", "bethe", {}, 2, "full", "fixed", "onschedule", None),
    ("bethe-lipson-p3-diag-random-bynodesubtree", "lipson", "bethe", {}, 3, "diag", "random", "bynodesubtree", None),
    ("ltrip-lipson-p5-full-improper-bycluster", "lipson", "ltrip", {}, 5, "full", "improper", "bycluster", None),
    ("bethe-lipson-p8-hetero-fixed-bynodesubtree", "lipson", "bethe", {}, 8, "hetero", "fixed", "bynodesubtree", None),
    ("jgs-lipson-p8-full-random-onschedule", "lipson", "jgs", {"maxclustersize": 3}, 8, "full", "random",
     "onschedule", None),
    ("ltrip-level3-p3-full-improper-bynodesubtree", "netstr_level3", "ltrip", {}, 3, "full", "improper",
     "bynodesubtree", None),
    ("jgs-mateescu-p16-diag-fixed-bycluster", "mateescu", "jgs", {"maxclustersize": 3}, 16, "diag", "fixed",
     "bycluster", None),
    ("bethe-lipson-p3-hetero-improper-bynodesubtree-missing", "lipson", "bethe", {}, 3, "hetero", "improper",
     "bynodesubtree", "onetip+tipall"),
    ("bethe-mateescu-p2-hetero-improper-bynodesubtree", "mateescu", "bethe", {}, 2, "hetero", "improper",
     "bynodesubtree", None),
    ("bethe-level3-p5-hetero-random-onschedule", "netstr_level3", "bethe", {}, 5, "hetero", "random", "onschedule",
     None),
]


def oracle_setup(lib, cs, B=3):
    _, name, method, cgkw, p, rk, root, reg, missing = cs
    return Loopy(lib, name, method, p, rk, root, B=B, seed=p, missing=missing, **cgkw), reg


def check_vs_oracle(s, bt, cgbs, what):
    """Beliefs, residuals (dJ, dh, flag), KL divergences and factored energies against the oracle.  A residual is
    the difference of the new and the old sepset belief, so its error is measured against the scale of the sepset
    belief it updated (max of |residual|, |sepset belief| and FLOOR)."""
    check_all_beliefs(s.case, bt, cgbs, tol=TOL, floor=FLOOR)
    labs = s.case.cg.labels
    for sj, to, frm in directed_messages(s):
        dJ, dh, fl, kl = bt.get_residual(sj, to)
        Js, hs, _ = bt.get_belief(sj)
        for e, c in enumerate(cgbs):
            ref = c.messageresidual[(labs[to - 1], labs[frm - 1])]
            scJ = max(np.max(np.abs(ref.dJ), initial=0.0), np.max(np.abs(c.belief[sj - 1].J), initial=0.0), FLOOR)
            sch = max(np.max(np.abs(ref.dh), initial=0.0), np.max(np.abs(c.belief[sj - 1].h), initial=0.0), FLOOR)
            assert np.max(np.abs(dJ[e] - ref.dJ), initial=0.0) <= TOL * scJ, (what, sj, to, e)
            assert np.max(np.abs(dh[e] - ref.dh), initial=0.0) <= TOL * sch, (what, sj, to, e)
            assert fl[e] == ref.iscalibrated_resid, (what, sj, to, e)
            r = ref.kldiv
            if r in (-1.0, 0.0) or abs(r) < KL_ABS:
                assert abs(kl[e] - r) <= TOL, (what, sj, to, e, kl[e], r)
            else:
                assert abs(kl[e] / r - 1) <= KL_TOL, (what, sj, to, e, kl[e], r)
    fe = bt.factored_energy()
    for e, c in enumerate(cgbs):
        ref = np.array(OBP.factored_energy(c))
        assert np.all(np.abs(fe[e] - ref) <= TOL * np.maximum(np.abs(ref), 1.0)), (what, e, fe[e], ref)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("cs", ORACLE_CASES, ids=lambda c: c[0])
def test_loopy_iterations_match_oracle(backend, cs):
    # after regularisation and after each of 3 iterations (every spanning tree once per iteration; later trees send
    # over sepsets that regularisation and earlier trees made non-zero), with KL divergences
    s, reg = oracle_setup(get_lib(backend), cs)
    bt = s.batch()
    bt.assignfactors(s.params, s.data, ncolors=s.ncolors)
    assert (bt.status() == 0).all()
    cgbs = [s.oracle(e) for e in range(s.B)]
    check_all_beliefs(s.case, bt, cgbs, tol=TOL, floor=FLOOR)
    regularize(s, reg, bt, cgbs)
    check_all_beliefs(s.case, bt, cgbs, tol=TOL, floor=FLOOR)
    assert s.case.plan.nsepsets >= s.case.nclusters  # the cluster graph has cycles
    for it in range(1, 4):
        succ, iscal = bt.calibrate(s.sched, 1, update_residualkldiv=True)
        ref = [OBP.calibrate(c, s.sched, 1, update_residualkldiv=True) for c in cgbs]
        assert list(succ) == [r[0] for r in ref] and list(iscal) == [r[1] for r in ref], it
        assert succ.all() and (bt.status() == 0).all()
        check_vs_oracle(s, bt, cgbs, it)


# ------------------------------------------------------------------ 2. fixed-point means vs the dense Gaussian
# (id, network, method, options, p, model, root, regulariser, missing cells)
FIXEDPOINT_CASES = [
    ("bethe-lipson-p3-full-fixed-onschedule", "lipson", "bethe", {}, 3, "full", "fixed", "onschedule", None),
    ("ltrip-lipson-p5-diag-random-bycluster", "lipson", "ltrip", {}, 5, "diag", "random", "bycluster", None),
    ("bethe-level3-p2-full-improper-bynodesubtree", "netstr_level3", "bethe", {}, 2, "full", "improper",
     "bynodesubtree", None),
    ("jgs-lipson-p3-hetero-improper-onschedule-missing", "lipson", "jgs", {"maxclustersize": 3}, 3, "hetero",
     "improper", "onschedule", "onetip+tipall"),
    ("jgs-mateescu-p8-hetero-random-onschedule", "mateescu", "jgs", {"maxclustersize": 3}, 8, "hetero", "random",
     "onschedule", None),
]


def max_residual(s, bt):
    w = 0.0
    for sj, to, _ in directed_messages(s):
        dJ, dh, _, _ = bt.get_residual(sj, to)
        w = max(w, np.max(np.abs(dJ), initial=0.0), np.max(np.abs(dh), initial=0.0))
    return w


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("cs", FIXEDPOINT_CASES, ids=lambda c: c[0])
def test_fixed_point_means_match_dense_posterior(backend, cs):
    # loopy Gaussian BP at its fixed point: every cluster mean J^-1 h equals the exact posterior mean, at every
    # (node, trait) in the cluster's scope; the variances are not exact and are not checked
    s, reg = oracle_setup(get_lib(backend), cs)
    bt = s.batch()
    bt.assignfactors(s.params, s.data, ncolors=s.ncolors)
    regularize(s, reg, bt, [])
    for _ in range(40):
        succ, _ = bt.calibrate(s.sched, 10)
        assert succ.all()
        if max_residual(s, bt) <= 1e-12:
            break
    assert max_residual(s, bt) <= 1e-12
    dense = [s.dense_means(e) for e in range(s.B)]
    nchecked = 0
    for j in range(1, s.case.nclusters + 1):
        if bt.dimension(j) == 0:
            continue
        pos = s.belief_positions(j)
        mu, _ = bt.integratebelief(j)
        for e in range(s.B):
            assert relerr(mu[e], dense[e][pos]) <= DENSE_TOL, (j, e)
        nchecked += 1
    assert nchecked >= s.case.nclusters // 2


# (id, network, method, options, p, model, root, regulariser, missing cells); the data sets of these cases keep the
# 1 % margin that test_autostop_point_matches_oracle asserts
AUTOSTOP_CASES = [
    ("bethe-mateescu-p2-full-fixed-onschedule", "mateescu", "bethe", {}, 2, "full", "fixed", "onschedule", None),
    ("ltrip-level3-p3-hetero-random-bycluster", "netstr_level3", "ltrip", {}, 3, "hetero", "random", "bycluster",
     None),
    ("bethe-unnamed-p2-diag-improper-bynodesubtree", "netstr_unnamed", "bethe", {}, 2, "diag", "improper",
     "bynodesubtree", None),
]


def residnorm(c):
    """max over directed messages of iscalibrated_residnorm's norms: calibrated iff <= ATOL_RESID."""
    w = 0.0
    for m in c.messageresidual.values():
        for x in (m.dh, m.dJ):
            if x.size:
                w = max(w, float(np.max(np.abs(x / math.sqrt(x.size)))))
    return w


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("cs", AUTOSTOP_CASES, ids=lambda c: c[0])
def test_autostop_point_matches_oracle(backend, cs):
    # calibrate(..., auto=True, info=True): the (iteration, tree) at which each element stops, bit for bit against
    # the oracle; the residual norm at every check up to the stop is more than 1 % away from the tolerance, so
    # roundoff cannot move the stop
    s, reg = oracle_setup(get_lib(backend), cs, B=4)
    niter = 60
    bt = s.batch()
    bt.assignfactors(s.params, s.data, ncolors=s.ncolors)
    cgbs = [s.oracle(e) for e in range(s.B)]
    regularize(s, reg, bt, cgbs)
    succ, iscal, info = bt.calibrate(s.sched, niter, auto=True, info=True)
    assert succ.all() and iscal.all()
    for e, c in enumerate(cgbs):
        m = s.oracle(e)  # a second copy, checked after every tree
        regularize(s, reg, _NoBatch(), [m])
        stop = None
        for it in range(1, niter + 1):
            for t, spt in enumerate(s.sched, start=1):
                assert OBP.calibrate_tree(m, spt)[0]
                w = residnorm(m)
                assert abs(w / ATOL_RESID - 1) > 0.01, (e, it, t, w)
                if w <= ATOL_RESID:
                    stop = (it, t)
                    break
            if stop:
                break
        assert all(OBP.calibrate(c, s.sched, niter, auto=True))
        assert OBP.calibrate.last_info == stop
        assert tuple(info[e]) == stop, (e, tuple(info[e]), stop)
    check_all_beliefs(s.case, bt, cgbs, tol=TOL)


class _NoBatch:
    """Stands in for a batch where only the oracle side of regularize() is wanted."""

    def regularizebeliefs_bycluster(self):
        pass

    def regularizebeliefs_onschedule(self):
        pass

    def regularizebeliefs_bynodesubtree(self, prog):
        pass


# ------------------------------------------------------------------ 3. kernel variants on regularised Bethe plans, bit for bit
# lipson Bethe graph: at p = 8 the family -> node messages are (I, S) = (8, 8) and (16, 8) (shared-memory kernels
# smem<8> and the multi-warp smem_mw); at p = 4 every message is inside the walk kernel's family
VARIANT_P = (4, 8)


def variant_setup(lib, p, B):
    return Loopy(lib, "lipson", "bethe", p, "full", "fixed", B=B, seed=p)


def break_elements(s, bt):
    """element 5: an indefinite largest cluster (its first message fails); element 7: another largest cluster all
    zero (messages out of it leave the receiver unchanged, until it has received some)."""
    big = [j for j in range(1, s.case.nclusters + 1) if bt.dimension(j) == max(s.case.plan.belief_dim)]
    assert len(big) >= 2
    J, h, g = bt.get_belief(big[0])
    J[5] = -np.eye(J.shape[1])
    bt.set_belief(big[0], J, h, g)
    J, h, g = bt.get_belief(big[-1])
    J[7] = 0.0
    h[7] = 0.0
    bt.set_belief(big[-1], J, h, g)


def run_setting(s, setting, kl, niter=3):
    """regularise, break elements 5 and 7, then niter calibrate calls of one iteration each (the second call of a
    captured CUDA graph replays it)"""
    bt = s.batch()
    for name, val in setting:
        {"coop": bt.set_coop_mode, "walk": bt.set_walk_mode, "pipeline": bt.set_pipeline,
         "graph": bt.set_graph_mode}[name](val)
    bt.assignfactors(s.params, s.data, ncolors=s.ncolors)
    bt.regularizebeliefs_onschedule()
    break_elements(s, bt)
    bt.launch_count(reset=True)
    for _ in range(niter):
        succ, iscal = bt.calibrate(s.sched, 1, update_residualkldiv=kl)
    nl = bt.launch_count()
    rec = snapshot(s, bt)
    rec.update(succ=succ, iscal=iscal, nl=nl)
    return rec


SETTINGS = [(("coop", m),) for m in (-1, 1, 2, 4, 8)] + [(("walk", m),) for m in (0, 1)] + \
    [(("pipeline", m),) for m in (1, 4)] + [(("graph", m),) for m in (0, 1)]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("p", VARIANT_P)
def test_loopy_kernel_variants_bit_identical(backend, p):
    # every message-kernel choice, walk mode, element pipelining and CUDA-graph replay against the generic
    # one-thread-per-element kernel, over 3 iterations with KL divergences; B = 37 leaves ragged tiles
    B = 37
    s = variant_setup(get_lib(backend), p, B)
    ref = run_setting(s, (("coop", 0),), kl=True)
    # element 7 fails too, later: once messages have reached its zeroed cluster, a message that integrates out one of
    # its still precision-free variables meets a zero pivot
    ok = ref["st"] == 0
    assert list(np.flatnonzero(~ok)) == [5, 7] and np.array_equal(ref["succ"], ok)
    for setting in SETTINGS:
        o = run_setting(s, setting, kl=True)
        assert_same(ref, o, keys=("succ", "iscal"), elems=ok, what=setting)
    if p <= WALK_MAXP:
        # the walk kernel does not compute KL divergences (those calls run per step): compare it with KL off
        w0 = run_setting(s, (("walk", 0),), kl=False)
        w1 = run_setting(s, (("walk", 1),), kl=False)
        assert_same(w0, w1, keys=("succ", "iscal"), elems=ok, what="walk")
        ntrees = len(s.sched)
        # 3 calls: one walk launch per tree and one iscal reduction per call; per-step launches need many more
        assert w1["nl"] <= 3 * (ntrees + 1) and w0["nl"] >= 20 * w1["nl"], (w0["nl"], w1["nl"])


# ------------------------------------------------------------------ 4. shared-precision batches on loopy graphs
@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("p,nth,nd", [(3, 1, 37), (8, 1, 37), (3, 2, 128), (8, 2, 128)])
def test_loopy_shared_precision_bit_identical(backend, p, nth, nd):
    # J once per group of nd elements sharing a parameter vector (the group pass divides by regularised, non-zero
    # sepset J): equal to own-J batches bit for bit after regularisation and after 3 iterations with KL.  Groups of
    # 128 run the bulk-copy element pass
    lib = get_lib(backend)
    s = variant_setup(lib, p, nd)
    rng = np.random.default_rng(p + nth)
    params = np.stack([s.params] + [pgbp_b200.bm_params([R * rng.uniform(0.5, 2) for R in s.Rs], s.mu)
                                    for _ in range(nth - 1)])
    out = {}
    for name, group in (("own", 0), ("shared", nd)):
        bt = s.batch(nth * nd, shared_precision_group=group)
        bt.assignfactors(params, s.data, ncolors=s.ncolors, pairing="product")
        bt.regularizebeliefs_onschedule()
        rec = dict(reg=[bt.get_belief(j) for j in range(1, len(s.case.b) + 1)])
        succ, iscal = bt.calibrate(s.sched, 3, update_residualkldiv=True)
        rec.update(snapshot(s, bt), succ=succ, iscal=iscal)
        out[name] = rec
    a, b_ = out["own"], out["shared"]
    assert a["succ"].all() and (a["st"] == 0).all()
    assert_same(a, b_, keys=("succ", "iscal"), what="shared")
    for x, y in zip(a["reg"], b_["reg"]):
        for u, v in zip(x, y):
            assert np.array_equal(u, v)


# ------------------------------------------------------------------ 5. tile walk at a multivariate shape
TILE_NET = "synth:128:0:1"  # a tree: its Bethe graph is a tree whose messages are (2, 2), (0, 2) at p = 2


def tile_setup(lib, B):
    return Loopy(lib, TILE_NET, "bethe", 2, "full", "fixed", B=B, seed=2)


@pytest.mark.parametrize("backend", BACKENDS)
def test_tilewalk_multivariate_bit_identical_and_oracle(backend):
    # one launch per run of narrow steps (block barrier between steps) == one launch per step and shape, bit for
    # bit, for 4, 8 and 16 message lanes and with wide steps split off, incl. auto-stop and a failing element
    B = 45
    s = tile_setup(get_lib(backend), B)
    assert (2, 2) in s.message_shapes()
    assert all(s.case.plan.levels(0, d)["nsteps"] >= 24 for d in (0, 1))
    jbig = next(j for j in range(1, s.case.nclusters + 1) if s.case.b[j - 1].dimension() == 4)
    out = {}
    for mode in [(0, 0)] + [(m, lanes) for m in (1, 2) for lanes in (4, 8, 16)]:
        bt = s.batch()
        bt.set_tilewalk_mode(min(mode[0], 1))
        if mode[0]:
            bt.set_tilewalk_params(lanes=mode[1], wide=1 if mode[0] == 2 else 0)
        bt.assignfactors(s.params, s.data, ncolors=s.ncolors)
        bt.regularizebeliefs_bycluster()
        J, h, g = bt.get_belief(jbig)
        J[5] = -np.eye(4)
        bt.set_belief(jbig, J, h, g)
        bt.launch_count(reset=True)
        succ, iscal, info = bt.calibrate(s.sched, 20, auto=True, info=True)
        nl = bt.launch_count()
        rec = snapshot(s, bt)
        rec.update(succ=succ, iscal=iscal, info=info, nl=nl)
        out[mode] = rec
    ok = np.arange(B) != 5
    ref = out[(0, 0)]
    assert ref["st"][5] != 0 and ref["succ"][ok].all() and ref["iscal"][ok].all()
    for mode, o in out.items():
        assert_same(ref, o, keys=("succ", "iscal", "info"), elems=ok, what=mode)
        if mode[0] == 1:
            assert o["nl"] < out[(2, mode[1])]["nl"] < ref["nl"], mode
    for e in (0, B - 1):
        c = s.oracle(e)
        OBP.regularizebeliefs_bycluster(c, s.case.cg)
        assert all(OBP.calibrate(c, s.sched, 20, auto=True))
        assert tuple(out[(1, 8)]["info"][e]) == OBP.calibrate.last_info
        check_all_beliefs(s.case, _Elem(out[(1, 8)]["beliefs"], e), [c], tol=TOL)


class _Elem:
    """get_belief of one element of a snapshot, as check_all_beliefs reads a batch."""

    def __init__(self, beliefs, e):
        self.beliefs, self.e = beliefs, e

    def get_belief(self, j):
        J, h, g = self.beliefs[j - 1]
        return J[self.e:self.e + 1], h[self.e:self.e + 1], g[self.e:self.e + 1]


# ------------------------------------------------------------------ 6. coverage pin (dispatch rules restated)
def kl_class(I, S):
    """kldiv_thread<MAXM> that launch_kldiv (csrc/pgbp_message.cu) picks: copy groups (nothing integrated) mix
    sepset dimensions and take the largest class; other groups are uniform in S."""
    if I == 0:
        return 64
    return 4 if S <= 4 else 12 if S <= 12 else 32 if S <= 32 else 64


def walk_shape_id(P, i, s):
    """csrc/pgbp_shapes.h: whole nodes (a, b) integrated / kept, a, b <= 3, a > 0 => (a + b) P <= PGBP_T0_MAX."""
    if P < 1 or P > WALK_MAXP or i % P or s % P:
        return -1
    a, b = i // P, s // P
    if a > 3 or b > 3 or (a > 0 and (a + b) * P > T0_MAX):
        return -1
    return 4 * a + b


def reached(s):
    """KL classes and kernels the plan of s launches."""
    shapes = s.message_shapes()
    kl = {kl_class(I, S) for (I, S) in shapes}
    kernels = {medium_kernel(I, S) for (I, S) in shapes} - {None}
    if all(walk_shape_id(s.p, I, S) >= 0 for (I, S) in shapes):
        kernels.add("walk")
    if max(I + S for (I, S) in shapes) <= TW_MAXM:
        kernels |= {f"tilewalk({I},{S})" for (I, S) in shapes}
    return kl, kernels


COVERAGE = dict(kl={4, 12, 32, 64}, kernels={"smem<8>", "smem<10>", "smem_mw", "walk", "tilewalk(2,2)"})


def test_loopy_plans_reach_the_kernels():
    lib = get_lib("emul")
    kl, kernels = set(), set()
    for cs in ORACLE_CASES:  # the KL divergences of test_loopy_iterations_match_oracle
        a, _ = reached(oracle_setup(lib, cs, B=1)[0])
        kl |= a
    for p in VARIANT_P:
        kernels |= reached(variant_setup(lib, p, 1))[1]
    kernels |= reached(tile_setup(lib, 1))[1]
    kernels |= reached(oracle_setup(lib, ORACLE_CASES[2], B=1)[0])[1]  # LTRIP p = 5: (10, 5) messages
    print("KL classes", sorted(kl), "kernels", sorted(kernels))
    assert COVERAGE["kl"] <= kl, sorted(kl)
    assert COVERAGE["kernels"] <= kernels, sorted(kernels)
    assert sum(len(oracle_setup(lib, cs, B=1)[0].sched) >= 2 for cs in ORACLE_CASES) >= len(ORACLE_CASES) - 1


# ------------------------------------------------------------------ 7. calibrate_optimize_clustergraph, MvDiag, p = 2
@pytest.mark.parametrize("backend", BACKENDS)
def test_optimize_clustergraph_mvdiag_objective_is_oracle_factored_energy(backend):
    # the driver's objective at its returned theta == the oracle's factored energy there (bycluster
    # regularisation, calibrate with auto-stop, as in calibrate_optimize_clustergraph!)
    lib = get_lib(backend)
    s = Loopy(lib, "mateescu", "bethe", 2, "diag", "fixed", B=1, seed=3)
    y = s.data[0]
    theta, fe, res = pgbp_b200.calibrate_optimize_clustergraph(s.case.plan, s.sched, y, model="MvDiagBrownianMotion",
                                                               start=(np.ones(2), np.zeros(2)), maxiter=100,
                                                               optim_iterations=10)
    assert np.isfinite(fe) and res.nit >= 1
    R = theta[:4].reshape(2, 2)
    assert R[0, 1] == 0.0 and R[1, 0] == 0.0
    model = M.MvDiagBrownianMotion(np.diag(R), theta[4:6])
    c = s.case.oracle_cgb(tbl=y, model=model)
    OBP.init_messagecalibrationflags_reset(c, True)
    OBP.regularizebeliefs_bycluster(c, s.case.cg)
    assert all(OBP.calibrate(c, s.sched, 100, auto=True))
    ref = OBP.factored_energy(c)[2]
    assert abs(fe / ref - 1) <= TOL, (fe, ref)
