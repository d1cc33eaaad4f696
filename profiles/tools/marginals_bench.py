"""Posterior node moments (ancestral state reconstruction) on the C4 network, one B200.

    python profiles/tools/marginals_bench.py [--batch 1024] [--host-batch 128] [--out profiles/marginals_c4.json]

C4 = bench.py's 10,000-tip level-1 network (21,999 nodes, 20,998 clusters), HeterogeneousBrownianMotion p = 8 with
4 rate colours and a fixed root, one shared data set, a grid of `--batch` theta, calibrated in both directions.
Measured:
  device    node_moments_device for every in-scope node (enqueue-only ABI call with prebuilt query arrays), CUDA events
            around >= 0.5 s of back-to-back calls after warm-up; algorithmic bytes = every queried belief read once
            (packed J + h) + the mean rows and packed covariance rows written, per element
  host      one node_moments() call end to end (host arrays out), at --host-batch elements (the host result of the
            full grid is ~13 GB)
  loop      the route without the new call at --host-batch: integratebelief_cov of every home cluster + host extraction
            of each node's block; its result must equal node_moments() bit for bit
The card's name and power limit are read in the same run.  The working set (26 MB of beliefs per element) is far
larger than L2.
"""
import argparse
import json
import os
import subprocess
import sys
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import ctypes as C  # noqa: E402

import numpy as np  # noqa: E402

import bench  # noqa: E402
import pgbp_b200  # noqa: E402


def card_info(torch):
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None, "sm_max_mhz": None}
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                            "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30)
        name, pl, mhz = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        info.update(name=name, power_limit_w=float(pl), sm_max_mhz=float(mhz))
    except Exception as ex:  # noqa: BLE001 -- reported, not fatal
        info["query_error"] = repr(ex)
    return info


def calibrated_batch(w, plan, B, stream):
    params, tips = w.inputs(B, 0)
    bt = pgbp_b200.BatchedClusterGraphBelief(plan, B, factors=False, residuals=False, stream=stream)
    bt.assignfactors(params, tips, ncolors=w.ncolors)
    succ, _ = bt.calibrate(None, 1, update_residualnorm=False)
    assert succ.all() and (bt.status() == 0).all()
    return bt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--host-batch", type=int, default=128)
    ap.add_argument("--seconds", type=float, default=0.6)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "marginals_c4.json"))
    args = ap.parse_args()
    import torch
    ctx = bench.Ctx(SimpleNamespace(gpus=1))  # device, HBM peak (MEASURED_PEAKS.json, else bench.py's fallback)
    card = card_info(torch)
    w = bench.C4()
    d = w.d
    lib = pgbp_b200.default_library()
    plan = pgbp_b200.ClusterGraphPlan(d["nclusters"], d["belief_dim"], d["sepset_clusters"], d["upind"], d["trees"],
                                      d["ntraits"], d["families"], lib)
    stream = torch.cuda.current_stream()
    out = {"workload": "C4: synthetic level-1 network, 10,000 tips, 21,999 nodes, 20,998 clusters, HeterogeneousBM p=8, "
                       "fixed root, calibrated (post + pre order); posterior moments of every in-scope node",
           "card": card}

    # ---- device: every node, full grid
    B = args.batch
    bt = calibrated_batch(w, plan, B, stream.cuda_stream)
    nq = bt.node_queries()
    qs = [(j, pos) for _, _, j, pos in nq]
    (qa, qp), (oa, op), (pa, pp), off = bt._query_arrays(qs)
    ks = np.diff(off)
    nmu, ncov = int(ks.sum()), int((ks * (ks + 1) // 2).sum())
    _, ld, _ = bt.device_view()
    d_mu = torch.empty((nmu, ld), dtype=torch.float64, device="cuda")
    d_cov = torch.empty((ncov, ld), dtype=torch.float64, device="cuda")

    def call():
        lib.check(lib.pgbp_marginal_moments_device(bt.handle, len(ks), qp, op, pp, C.c_void_p(d_mu.data_ptr()),
                                                   C.c_void_p(d_cov.data_ptr())))
    for _ in range(3):
        call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream); call(); e1.record(stream); torch.cuda.synchronize()
    n = max(10, int(np.ceil(args.seconds / max(e0.elapsed_time(e1) * 1e-3, 1e-6))))
    t_host = time.perf_counter()
    e0.record(stream)
    for _ in range(n):
        call()
    e1.record(stream)
    t_host = time.perf_counter() - t_host
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    beliefs = sorted({j for j, _ in qs})
    dims = np.array([plan.belief_dim[j - 1] for j in beliefs])
    read = 8.0 * B * float((dims * (dims + 1) // 2 + dims).sum())
    write = 8.0 * B * float(nmu + ncov)
    gbs = (read + write) / (ms * 1e-3) / 1e9
    # the device rows are the host result's entries
    mu_h, cov_h, ins = bt.node_moments()
    dm = d_mu[:, :B].T.cpu().numpy()
    assert np.array_equal(dm, np.concatenate([mu_h[:, v, tr] for v, tr, _, _ in nq], axis=1))
    del mu_h, cov_h
    out["device"] = {"batch": B, "nodes": len(nq), "queried_beliefs": len(beliefs), "mean_rows": nmu, "cov_rows": ncov,
                     "calls_timed": n, "timed_region_s": ms * n * 1e-3, "ms_per_call": ms,
                     "host_enqueue_ms_per_call": t_host / n * 1e3,
                     "algorithmic_bytes": read + write, "bytes_read": read, "bytes_written": write,
                     "achieved_gbs": gbs, "hbm_peak_gbs": ctx.peak, "peak_source": ctx.peak_src,
                     "fraction_of_peak": gbs / ctx.peak,
                     "basis": "each queried belief read once (packed J + h) + mean and packed covariance rows written"}
    del bt, d_mu, d_cov
    torch.cuda.empty_cache()

    # ---- host: one node_moments() call, and the loop over home clusters, same batch
    Bh = args.host_batch
    bt = calibrated_batch(w, plan, Bh, stream.cuda_stream)
    nq = bt.node_queries()
    bt.node_moments()  # warm-up (scratch growth)
    torch.cuda.synchronize()
    t = time.perf_counter()
    mu_h, cov_h, ins = bt.node_moments()
    t_nm = time.perf_counter() - t
    p = d["ntraits"]
    nn = d["families"]["nnodes"]
    t = time.perf_counter()
    mu_l = np.full((Bh, nn, p), np.nan)
    cov_l = np.full((Bh, nn, p, p), np.nan)
    cur_j, fm, fc = None, None, None
    for v, tr, j, pos in sorted(nq, key=lambda q: q[2]):
        if j != cur_j:
            fm, fc, _ = bt.integratebelief_cov(j)
            cur_j = j
        mu_l[:, v, tr] = fm[:, pos]
        cov_l[:, v, np.asarray(tr)[:, None], np.asarray(tr)[None, :]] = fc[:, pos][:, :, pos]
    t_loop = time.perf_counter() - t
    same = bool(np.array_equal(mu_l, mu_h, equal_nan=True) and np.array_equal(cov_l, cov_h, equal_nan=True))
    out["host"] = {"batch": Bh, "node_moments_call_s": t_nm,
                   "integrate_cov_loop_s": t_loop, "integrate_cov_calls": len({q[2] for q in nq}),
                   "loop_over_call": t_loop / t_nm, "results_bit_identical": same}
    assert same
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
