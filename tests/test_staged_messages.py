"""Register-class messages (i >= 1 integrated out, i + s <= 12) run in k_message_staged on the device: their operand
rows are bulk-copied into shared memory one tile of elements at a time, and the arithmetic is message_body_t0
reading them from there.  These tests check that it computes what the unchanged register body computes, bit for bit:
  * against the walk kernel (k_walk runs message_thread_t0, operands from global memory) on clique-tree calibrations
    of the lazaridis graph, with batch sizes that leave a partial tile, residual tracking on and off, a failing
    element, a second calibration (non-zero old sepsets) and the element-chunk pipeline;
  * against the host-emulation build, one message per shape of the register class, with an all-zero sender block
    (missing-data shortcut) and a non-positive-definite sender."""
import json
import os

import numpy as np
import pytest

import pgbp_b200
from harness import Case, get_lib
from oracle import models as M
from pgbp_b200 import _lib as L

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "reference_goldens.json")))
TAXA = ["Mbuti", "Onge", "Karitiana", "MA1", "Loschbour", "European", "Stuttgart"]


def _calibrated(case, B, R, data, walk, pipeline, track):
    bt = pgbp_b200.BatchedClusterGraphBelief(case.plan, B)
    bt.set_walk_mode(walk)
    bt.set_pipeline(pipeline)
    p = R.shape[0]
    bt.assignfactors(pgbp_b200.bm_params([R], np.zeros(p)), data)
    J, h, g = bt.get_belief(10)  # element 5: indefinite precision in a leaf cluster of the clique tree
    J[5] = -np.eye(p)
    bt.set_belief(10, J, h, g)
    succ, iscal = bt.calibrate(case.sched, update_residualnorm=track)
    succ2, iscal2 = bt.calibrate(case.sched, update_residualnorm=track)  # old sepsets are non-zero now
    return dict(succ=succ, iscal=iscal, succ2=succ2, iscal2=iscal2, st=bt.status(),
                beliefs=[bt.get_belief(j) for j in range(1, len(case.b) + 1)],
                res=[bt.get_residual(case.nclusters + 1 + j, case.plan.sepset_clusters[j][s] + 1)
                     for j in range(case.plan.nsepsets) for s in (0, 1)])


@pytest.mark.gpu
@pytest.mark.parametrize("track", [True, False])
@pytest.mark.parametrize("B", [70, 65536 + 37])
@pytest.mark.parametrize("p", [1, 2, 3])
def test_staged_calibration_matches_walk_kernel_bitwise(p, B, track):
    lib = get_lib("cuda")
    rng = np.random.default_rng(200 + p)  # (as in test_parity: element 5 then fails)
    A = rng.normal(size=(p, p))
    R = A @ A.T / p + 0.1 * np.eye(p)
    data = rng.normal(size=(B, 7, p))
    case = Case(GOLD["lazaridis"], "cliquetree", data[0], TAXA, M.MvFullBrownianMotion(R, np.zeros(p)), lib,
                order_hint=GOLD["lazaridis_cluster_labels"])
    ref = _calibrated(case, B, R, data, walk=1, pipeline=1, track=track)
    ok = np.arange(B) != 5
    assert (ref["succ"] == ok).all() and ref["st"][5] != 0
    for pipeline in (1, 4):  # level-parallel launches, in one piece and in four element chunks on four streams
        out = _calibrated(case, B, R, data, walk=0, pipeline=pipeline, track=track)
        for k in ("succ", "iscal", "succ2", "iscal2", "st"):
            assert np.array_equal(out[k], ref[k]), k
        for (J0, h0, g0), (J1, h1, g1) in zip(ref["beliefs"], out["beliefs"]):
            assert np.array_equal(J0[ok], J1[ok]) and np.array_equal(h0[ok], h1[ok]) and np.array_equal(g0[ok], g1[ok])
        for r0, r1 in zip(ref["res"], out["res"]):
            assert np.array_equal(r0[0][ok], r1[0][ok]) and np.array_equal(r0[1][ok], r1[1][ok])
            assert np.array_equal(r0[2][ok], r1[2][ok])


T0_SHAPES = [(i, s) for i in range(1, 13) for s in range(0, 13 - i)]


def _spd(rng, B, m):
    X = rng.normal(size=(B, m, m))
    return X @ X.transpose(0, 2, 1) / max(m, 1) + 0.5 * np.eye(m)


def _one_message(lib, i, s, B, seed):
    """Sender (cluster 1, dimension i + s) -> sepset (dimension s) -> receiver (cluster 2, dimension s + 1), sepset
    positions scattered in both clusters.  Element 3: sender rows of the integrated block all zero; element 5:
    integrated block not positive definite.  The message is sent twice (the second one sees a non-zero old sepset)."""
    rng = np.random.default_rng(seed)
    m = i + s
    ua = sorted(rng.choice(m, size=s, replace=False).tolist())
    ub = sorted(rng.choice(s + 1, size=s, replace=False).tolist())
    plan = pgbp_b200.ClusterGraphPlan(2, [m, s + 1, s], [(0, 1)], [(ua, ub)], [([0], [1])], 1, None, lib)
    bt = pgbp_b200.BatchedClusterGraphBelief(plan, B)
    J0, h0, g0 = _spd(rng, B, m), rng.normal(size=(B, m)), rng.normal(size=B)
    iv = [k for k in range(m) if k not in ua]
    J0[3][iv, :] = 0.0
    J0[3][:, iv] = 0.0
    h0[3][iv] = 0.0
    J0[5][np.ix_(iv, iv)] = -np.eye(i)
    bt.set_belief(1, J0, h0, g0)
    bt.set_belief(2, _spd(rng, B, s + 1), rng.normal(size=(B, s + 1)), rng.normal(size=B))
    bt.set_belief(3, _spd(rng, B, s), rng.normal(size=(B, s)), rng.normal(size=B))
    res = []
    for _ in range(2):
        lib.check(lib.pgbp_propagate(bt.handle, 0, 2, 1, L.CAL_RESIDNORM))
        res.append(bt.get_residual(3, 2))
    return dict(st=bt.status(), beliefs=[bt.get_belief(j) for j in (1, 2, 3)], res=res)


@pytest.mark.gpu
@pytest.mark.parametrize("i,s", T0_SHAPES)
def test_staged_message_matches_host_emulation(i, s):
    B = 70
    emu = _one_message(get_lib("emul"), i, s, B, 7000 + 16 * i + s)
    dev = _one_message(get_lib("cuda"), i, s, B, 7000 + 16 * i + s)
    assert np.array_equal(emu["st"], dev["st"]) and dev["st"][5] != 0 and dev["st"][3] == 0
    for (Je, he, ge), (Jd, hd, gd) in zip(emu["beliefs"], dev["beliefs"]):
        assert np.array_equal(Je, Jd) and np.array_equal(he, hd)
        # g takes a log of the pivots: host and device log may differ in the last bits
        np.testing.assert_allclose(gd, ge, rtol=1e-13, atol=1e-13)
    for re_, rd in zip(emu["res"], dev["res"]):  # dJ, dh, calibration flag of both messages
        for xe, xd in zip(re_[:3], rd[:3]):
            assert np.array_equal(xe, xd)
