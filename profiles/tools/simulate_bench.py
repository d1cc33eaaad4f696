"""Forward simulation on the device (pgbp_simulate_device) and the device-resident parametric-bootstrap step.

    python profiles/tools/simulate_bench.py --out DIR [--workloads c2,c4,c5] [--profile]

Workloads (bench.py's networks): c2 = lazaridis clique tree, MvFull p = 3, B = 65,536, one record; c4 = the 10k-tip
network with 4 rate colours, p = 8, 4,096 records (one per element); c5 = the 100k-tip network, p = 16, one record,
1,536 replicates on a shared-precision batch.  Per workload:
  - simulation alone: CUDA events around back-to-back pgbp_simulate_device calls over >= 0.5 s; algorithmic bytes
    (tips written once, internal rows written once, parent rows read, records read) and normals drawn, from shapes;
  - bootstrap step: simulate -> assign_factors_device -> postorder -> integrate(root), replicates/s, against the same
    step fed host tip data (pinned host copy -> device -> assign -> postorder -> integrate, bench.py's e2e arm);
  - with --profile, per-kernel times from torch.profiler in a separate run (simulate only).
Writes DIR/simulate_<workload>.json (and DIR/simulate_<workload>_kernels.txt)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import pgbp_b200  # noqa: E402

HBM = 7.7e12


def with_mem_parent(d):
    """bench's plan dict with the families' mem_parent (the workloads/*.json plans predate the key): per member the
    0-based preorder index of a parent (parents by decreasing index, as the family table lists them), -1 first"""
    fam = d["families"]
    if "mem_parent" not in fam:
        mp = []
        for par in d["simulate"]:
            mp.append(-1)
            mp.extend(sorted((int(q) for q, _, _ in par), reverse=True))
        fam["mem_parent"] = mp
    return d


def levels(fam):
    n, off, mp, row = fam["nnodes"], fam["mem_off"], fam["mem_parent"], fam["node_datarow"]
    lv = [0] * n
    for v in range(1, n):
        lv[v] = 1 + max(lv[mp[k]] for k in range(off[v] + 1, off[v + 1]))
    return len({lv[v] for v in range(n) if row[v] < 0})


def events_time(fn, min_s=0.5):
    import torch
    fn()
    torch.cuda.synchronize()
    reps, total = 1, 0.0
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        b.synchronize()
        total = a.elapsed_time(b) / 1e3
        if total >= min_s:
            return total / reps, reps
        reps = max(reps * 2, int(reps * min_s / max(total, 1e-6) * 1.2) + 1)


def run(key, out, profile):
    import torch
    w = bench.WORKLOADS[key]()
    d = with_mem_parent(w.d)
    fam = d["families"]
    p, nc = d["ntraits"], w.ncolors
    B = {"c2": 65536, "c4": 4096, "c5": 1536}[key]
    shared = key == "c5"
    plan = pgbp_b200.ClusterGraphPlan(d["nclusters"], d["belief_dim"], d["sepset_clusters"], d["upind"], d["trees"], p,
                                      fam)
    rng = np.random.default_rng(1)
    nrec = 4096 if key == "c4" else 1
    if key == "c4":
        params, _ = w.inputs(nrec, 0)
    else:
        A = rng.normal(size=(p, p))
        R = A @ A.T / p + 0.1 * np.eye(p)
        params = pgbp_b200.bm_params([R], np.zeros(p))[None]
    # the batch runs on torch's stream: the events, the tip copies of the host-fed arm and the library's kernels are
    # ordered on one stream
    bt = pgbp_b200.BatchedClusterGraphBelief(plan, B, factors=False, residuals=False,
                                             stream=torch.cuda.current_stream().cuda_stream,
                                             shared_precision_group=B if shared else 0)
    dp = torch.tensor(params, device="cuda")
    ntips, nn = fam["ntips"], fam["nnodes"]
    dt = torch.empty((B, ntips, p), dtype=torch.float64, device="cuda")
    seed = [0]

    def sim():
        seed[0] += 1
        bt.simulate_device(dp.data_ptr(), nrec, seed[0], dt.data_ptr(), None, ncolors=nc)

    t_sim, reps = events_time(sim)
    ninternal = sum(1 for r in fam["node_datarow"] if r < 0)
    npar = fam["mem_off"][nn] - nn
    byts = 8.0 * B * p * (ntips + ninternal + npar) + 8.0 * params.size
    fixed_root = not np.any(params[0, nc * p * p + p:])
    normals = B * p * (nn - (1 if fixed_root else 0))
    res = dict(workload=key, B=B, p=p, ncolors=nc, nparamsets=nrec, shared_precision=shared, nnodes=nn, ntips=ntips,
               ninternal=ninternal, levels=levels(fam), sim_s=t_sim, sim_calls=reps, algorithmic_bytes=byts,
               achieved_TBps=byts / t_sim / 1e12, hbm_share=byts / t_sim / HBM, normals=normals,
               normals_per_s=normals / t_sim, replicates_per_s_sim=B / t_sim,
               launches_per_call=None)
    bt.launch_count(reset=True)
    sim()
    torch.cuda.synchronize()
    res["launches_per_call"] = bt.launch_count()
    # bootstrap step, device-resident and fed from the host
    root = d["root_cluster"] + 1
    norm = torch.empty(B, dtype=torch.float64, device="cuda")

    def step_dev():
        sim()
        bt.assignfactors_device(dp.data_ptr(), nrec, dt.data_ptr(), B, ncolors=nc)
        bt.calibrate_async([0], 1, update_residualnorm=False, direction=1)
        bt.integrate_device(root, norm.data_ptr())

    host = torch.empty((B, ntips, p), dtype=torch.float64, pin_memory=True)
    sim()
    host.copy_(dt)
    torch.cuda.synchronize()

    def step_host():
        dt.copy_(host, non_blocking=True)
        bt.assignfactors_device(dp.data_ptr(), nrec, dt.data_ptr(), B, ncolors=nc)
        bt.calibrate_async([0], 1, update_residualnorm=False, direction=1)
        bt.integrate_device(root, norm.data_ptr())

    t_dev, _ = events_time(step_dev)
    t_host, _ = events_time(step_host)
    assert (bt.status() == 0).all() and torch.isfinite(norm).all()
    res.update(bootstrap_step_s=t_dev, bootstrap_replicates_per_s=B / t_dev, hostfed_step_s=t_host,
               hostfed_replicates_per_s=B / t_host, tip_bytes=8.0 * B * ntips * p)
    if profile:
        from torch.profiler import ProfilerActivity, profile as prof
        with prof(activities=[ProfilerActivity.CUDA]) as pr:
            for _ in range(3):
                sim()
            torch.cuda.synchronize()
        txt = pr.key_averages().table(sort_by="cuda_time_total", row_limit=15)
        open(os.path.join(out, f"simulate_{key}_kernels.txt"), "w").write(txt)
        res["kernels"] = {e.key: e.device_time_total / 3 / 1e3 for e in pr.key_averages() if e.device_time_total > 0}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default="c2,c4,c5")
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "simulate_bench measures on a GPU"
    os.makedirs(a.out, exist_ok=True)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                          capture_output=True, text=True).stdout
    for key in a.workloads.split(","):
        t0 = time.time()
        r = run(key, a.out, a.profile)
        r["card"] = card.strip().splitlines()[-1]
        r["wall_s"] = time.time() - t0
        json.dump(r, open(os.path.join(a.out, f"simulate_{key}.json"), "w"), indent=1)
        print(json.dumps({k: v for k, v in r.items() if k != "kernels"}), flush=True)


if __name__ == "__main__":
    main()
