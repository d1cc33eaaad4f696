#!/usr/bin/env python
"""Benchmark of the batched Gaussian-BP hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--batch B] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): lazaridis_2014 admixture graph, clique
tree (17 clusters / 16 sepsets / 32 messages per calibration), full
multivariate Brownian motion with p = 3 traits, fixed root, 65,536 synthetic
trait replicates per GPU simulated down the network (seed 0xB200 + 2).
Metric: clique-tree calibrations per second, whole job (all ranks).

One step =  beliefs <- factors (init_beliefs_reset_fromfactors!),
            calibrate!(beliefs, [spt]) = 16 postorder + 16 preorder messages with
            residual tracking and the iscalibrated reduction,
            integratebelief! at the root cluster (per-replicate log-likelihood),
            [N > 1: NCCL all-gather of the log-likelihoods]
for all B replicates of the rank.  `value` times that with the factors
resident in HBM; `e2e` times the public host-buffer API per step:
pinned host tip data -> H2D -> assignfactors (K1) -> calibrate -> integratebelief
-> D2H of the log-likelihoods.  The timed region is exactly `--steps` steps.

`--dump-outputs DIR` writes what the last timed step of the headline workload computed, as DIR/<name>.npy
(float64): `loglik` [B] (per-replicate log-likelihood at the root), or for the loopy workloads `factored_energy`
[B, 3] (average energy, approximate entropy, factored energy); with N > 1 also `gathered` [N * B], the
per-element results of all ranks in rank order.  The inputs are seeded, so two builds run with the same arguments
can be compared output for output.  Outputs beyond 64 MB in all are cut to a fixed, seeded sample of rows (the
row indices in DIR/<name>_rows.npy).

`--impl reference`: the reference is Julia (not in this image), so the
reference arm is the C/OpenMP restatement of the reference's algorithm
(oracle/c, kind "port") on all host cores, on a bounded sample per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "clique-tree calibrations/sec (batched replicates)"
SEED = 0xB200
DUMP_BYTES = 64 << 20


class C2:
    """BASELINE configs[1]: lazaridis_2014, MvFullBM p=3, 65,536 trait replicates, clique tree."""
    key = "c2"
    unit = "calibrations/s"
    workload = ("lazaridis_2014 admixture graph, MvFullBrownianMotion p=3, 65,536 synthetic trait replicates per GPU, "
                "clique tree, calibrate! (post+pre order, residual tracking) + integratebelief! [BASELINE configs[1]]")
    default_batch = 65536
    ncolors = 1
    residuals = True
    step_text = "reset_from_factors + calibrate (post+pre, residuals, iscal) + integrate(root)"
    e2e_text = "pinned host tip data -> assignfactors (H2D + K1) -> calibrate -> integratebelief -> D2H loglik"
    kernel_text = "k_message<i,s> family (all 32 messages of a calibration)"
    cpu_text = "assignfactors + calibrate + integratebelief per replicate"

    def __init__(self):
        self.d = json.load(open(os.path.join(ROOT, "workloads", "lazaridis_cliquetree_p3.json")))

    def inputs(self, B, rank):
        """SURVEY 8(d) C2: R = A A'/3 + 0.1 I, mu = 0, fixed root; replicates simulated down the
        network: X_v = sum_k gamma_k X_pa_k + N(0, sum_k gamma_k^2 t_k R).  One theta, B data sets."""
        d = self.d
        rng = np.random.Generator(np.random.PCG64(SEED + 2 + 1000 * rank))
        p = d["ntraits"]
        A = rng.normal(size=(p, p))
        R = A @ A.T / 3 + 0.1 * np.eye(p)
        Lr = np.linalg.cholesky(R)
        n = len(d["simulate"])
        X = np.zeros((n, B, p))
        for v in range(1, n):
            par = d["simulate"][v]
            var = sum(g * g * t for _, t, g in par)
            mean = sum(g * X[q] for q, t, g in par)
            X[v] = mean + np.sqrt(var) * (rng.normal(size=(B, p)) @ Lr.T)
        tips = np.ascontiguousarray(X[d["tip_nodes"]].transpose(1, 0, 2))  # [B][ntips][p]
        params = np.concatenate([R.T.ravel(), np.zeros(p), np.zeros(p * p)])[None]
        return params, tips

    def cost(self, plan):
        by = plan.traversal_cost(0, 0, True)[0] + plan.traversal_cost(0, 1, True)[0]
        fl = plan.traversal_cost(0, 0, True)[1] + plan.traversal_cost(0, 1, True)[1]
        return by, fl

    cpu_kw = dict(post=True, pre=True, residnorm=True)


class C2S(C2):
    """C2 with the shared-precision path (SURVEY 8f-1): the 65,536 elements are trait replicates under ONE
    parameter vector, so every J is stored and updated once; per message and element only h and g move.
    Reported separately, with its own algorithmic-bytes formula (never against the full-J byte count)."""
    key = "c2s"
    shared = True
    workload = ("lazaridis_2014 admixture graph, MvFullBrownianMotion p=3, 65,536 synthetic trait replicates per GPU under "
                "ONE parameter vector, clique tree, SHARED-PRECISION batch (J stored once per group, h and g per element), "
                "calibrate! (post+pre order, residual tracking) + integratebelief! [BASELINE configs[1], shared-J variant "
                "of SURVEY 8f-1: own byte count 8*(m_F + 1 + 4*(s+1) + s) per message]")
    kernel_text = "k_hmsg<I> family (element pass of the 32 messages of a calibration; the group pass k_jmsg runs once per GPU)"

    def cost(self, plan):
        return shared_cost(self, plan, (0, 1))


class C4(C2):
    """BASELINE configs[3]: synthetic 10k-tip level-1 network, HeterogeneousBM p=8, grid of 4,096 theta."""
    key = "c4"
    unit = "likelihood evaluations/s"
    workload = ("synthetic level-1 network, 10,000 tips + 1,000 reticulations (21,999 nodes; clique tree of 20,998 "
                "clusters), HeterogeneousBrownianMotion p=8 with 4 rate colours, one shared data set, batched grid of "
                "parameter vectors; unit = assignfactors! + postorder traversal + integratebelief!(root) "
                "(the optimiser objective, src/calibration.jl:195-221) [BASELINE configs[3]]")
    default_batch = 4096
    ncolors = 4
    residuals = False
    step_text = "assign_factors (K1) + propagate_1traversal_postorder (20,997 messages) + integrate(root)"
    e2e_text = "pinned host theta grid -> assignfactors (H2D + K1) -> postorder -> integratebelief -> D2H loglik"
    kernel_text = "k_message* family (20,997 postorder messages of one likelihood evaluation)"
    cpu_text = "assignfactors + postorder + integratebelief per parameter vector"

    def __init__(self, ntips=10000, nretic=1000, p=8):
        from workloads import synth
        net = synth.level1_network(ntips, nretic, SEED + 4)
        self.col = synth.edge_colors(net, self.ncolors)
        self.d = synth.cliquetree_plan(net, p, True, self.col, name="synthetic_level1_%d" % ntips)
        self.synth = synth

    def inputs(self, B, rank):
        d = self.d
        p, nc = d["ntraits"], self.ncolors
        rng = np.random.Generator(np.random.PCG64(SEED + 4 + 1000 * rank))

        def rate():
            A = rng.normal(size=(p, p))
            return A @ A.T / p + 0.1 * np.eye(p)
        R0 = [rate() for _ in range(nc)]
        # families list parents by decreasing index; simulate lists them in edge order: map through parent id
        par_col = {}
        for v, fam in enumerate(d["simulate"]):
            o = d["families"]["mem_off"][v]
            order = sorted(range(len(fam)), key=lambda k: -fam[k][0])
            for pos, k in enumerate(order):
                par_col[(v, k)] = d["families"]["mem_color"][o + 1 + pos]
        tips = self.synth.simulate_tips(d, lambda v, k: R0[par_col[(v, k)]], 1, SEED + 40)  # one shared data set
        params = np.empty((B, nc * p * p + p + p * p))
        for b in range(B):  # SURVEY 8(d) C4: R_c^(b) = A A'/p + 0.1 I
            A = rng.normal(size=(nc, p, p))
            R = A @ A.transpose(0, 2, 1) / p + 0.1 * np.eye(p)
            params[b, :nc * p * p] = R.reshape(-1)  # symmetric: row- and column-major coincide
            params[b, nc * p * p:] = 0.0
        return params, tips

    def cost(self, plan):
        by, fl = plan.traversal_cost(0, 0, False)
        return by, fl

    cpu_kw = dict(post=True, pre=False, residnorm=False)


class C3(C2):
    """BASELINE configs[2]: muller_2022 network, loopy BP on the Bethe cluster graph with regularisation,
    16,384 replicates, fixed iteration count."""
    key = "c3"
    unit = "calibrations/s"
    niter = 10
    workload = ("muller_2022 network (801 nodes, 40 tips, 361 hybrids), Bethe cluster graph (1557 clusters / 1914 sepsets), "
                "UnivariateBrownianMotion(1, 0) fixed root, 16,384 simulated trait replicates per GPU, "
                "regularizebeliefs_bycluster!, spanningtrees_clusterlist schedule (2 trees), niter = 10 fixed, auto = false; "
                "1 calibration = 1 iteration over all spanning trees (4 x 1556 messages) [BASELINE configs[2]]")
    default_batch = 16384
    ncolors = 1
    residuals = True
    step_text = ("reset_from_factors + regularizebeliefs_bycluster! + calibrate!(niter = 10: 62,240 messages, residuals, "
                 "iscal) + factored_energy; value counts 10 calibrations per element per step")
    e2e_text = ("pinned host tip data -> assignfactors (H2D + K1) -> regularize -> calibrate(niter=10) -> factored_energy "
                "-> D2H")
    kernel_text = "k_message<i,s> family (62,240 messages of the 10 iterations)"
    cpu_text = "assignfactors + regularize + calibrate(niter=10) + factored_energy per replicate"

    def __init__(self):
        self.d = json.load(open(os.path.join(ROOT, "workloads", "muller_bethe_p1.json")))

    def inputs(self, B, rank):
        d = self.d
        rng = np.random.Generator(np.random.PCG64(SEED + 3 + 1000 * rank))
        n = len(d["simulate"])
        X = np.zeros((n, B, 1))
        for v in range(1, n):
            par = d["simulate"][v]
            var = sum(g * g * t for _, t, g in par)
            mean = sum(g * X[q] for q, t, g in par)
            X[v] = mean + np.sqrt(var) * rng.normal(size=(B, 1))
        tips = np.ascontiguousarray(X[d["tip_nodes"]].transpose(1, 0, 2))
        params = np.array([[1.0, 0.0, 0.0]])
        return params, tips

    def cost(self, plan):
        nt = len(self.d["trees"])
        by = sum(plan.traversal_cost(t, dr, True)[0] for t in range(nt) for dr in range(2)) * self.niter
        fl = sum(plan.traversal_cost(t, dr, True)[1] for t in range(nt) for dr in range(2)) * self.niter
        return by, fl

    cpu_kw = dict(post=True, pre=True, residnorm=True, niter=10, reg_bycluster=True)


class C3L(C3):
    """BASELINE configs[2], second cluster graph: LTRIP(net) (the node families as clusters: 801 clusters / 1158
    sepsets, sepsets of up to two nodes)."""
    key = "c3l"
    workload = ("muller_2022 network (801 nodes, 40 tips, 361 hybrids), LTRIP(net) cluster graph (801 clusters / 1158 sepsets), "
                "UnivariateBrownianMotion(1, 0) fixed root, 16,384 simulated trait replicates per GPU, "
                "regularizebeliefs_bycluster!, spanningtrees_clusterlist schedule (2 trees), niter = 10 fixed, auto = false; "
                "1 calibration = 1 iteration over all spanning trees (4 x 800 messages) [BASELINE configs[2], LTRIP variant]")
    step_text = ("reset_from_factors + regularizebeliefs_bycluster! + calibrate!(niter = 10: 32,000 messages, residuals, "
                 "iscal) + factored_energy; value counts 10 calibrations per element per step")
    kernel_text = "k_tilewalk / k_message<i,s> family (32,000 messages of the 10 iterations)"

    def __init__(self):
        self.d = json.load(open(os.path.join(ROOT, "workloads", "muller_ltrip_p1.json")))


class C5(C4):
    """BASELINE configs[4]: synthetic 100k-tip network with 10k reticulations, MvFullBrownianMotion p=16, one
    theta, replicate batch as large as HBM allows per GPU (0.92 GB of state per replicate), sharded by
    replicate across GPUs."""
    key = "c5"
    unit = "calibrations/s"
    default_batch = 128
    ncolors = 1
    residuals = False
    workload = ("synthetic level-1 network, 100,000 tips + 10,000 reticulations (219,999 nodes; clique tree of 209,998 "
                "clusters, sender dimensions 16 / 32 / 48), MvFullBrownianMotion p=16, one parameter vector, 128 simulated "
                "trait replicates per GPU (0.92 GB of state each: 118 GB of the 180 GB), assignfactors! + calibrate! "
                "(post+pre order) + integratebelief!(root) [BASELINE configs[4]]")
    step_text = "assign_factors (K1, generic path: p = 16) + calibrate (419,994 messages) + integrate(root)"
    e2e_text = "pinned host tip data -> assignfactors (H2D + K1) -> calibrate -> integratebelief -> D2H loglik"
    kernel_text = "k_message* family (419,994 messages of one calibration; (16,16) shared-memory kernel, (32,16) generic)"
    cpu_text = "assignfactors + calibrate + integratebelief per replicate"

    def __init__(self, ntips=100000, nretic=10000, p=16):
        from workloads import synth
        net = synth.level1_network(ntips, nretic, SEED + 5)
        self.col = None
        self.d = synth.cliquetree_plan(net, p, True, None, name="synthetic_level1_%d" % ntips)
        self.synth = synth

    def inputs(self, B, rank):
        d = self.d
        p = d["ntraits"]
        rng = np.random.Generator(np.random.PCG64(SEED + 5 + 1000 * rank))
        A = rng.normal(size=(p, p))
        R = A @ A.T / p + 0.1 * np.eye(p)
        tips = self.synth.simulate_tips(d, lambda v, k: R, B, SEED + 50 + rank)
        params = np.concatenate([R.reshape(-1), np.zeros(p), np.zeros(p * p)])[None]
        return params, tips

    def cost(self, plan):
        by = plan.traversal_cost(0, 0, False)[0] + plan.traversal_cost(0, 1, False)[0]
        fl = plan.traversal_cost(0, 0, False)[1] + plan.traversal_cost(0, 1, False)[1]
        return by, fl

    cpu_kw = dict(post=True, pre=True, residnorm=False)


def shared_cost(w, plan, directions):
    """Algorithmic bytes / flops per element of a shared-precision batch: per message and element only h and g move
    (8 (m_F + 1 + 4 (s + 1) [+ s with residuals]) bytes) and w = U^-T h_I, h_K - Z'w are applied
    (i^2 + 2 i s + 2 i flops); the J part is per group and not counted."""
    dims = w.d["belief_dim"]
    by = fl = 0.0
    for dr in directions:
        lv = plan.levels(0, dr)
        for f, sp in zip(lv["frm"], lv["sepset"]):
            mF, s_ = dims[f], dims[sp]
            i_ = mF - s_
            by += 8.0 * (mF + 1 + 4 * (s_ + 1) + (s_ if w.residuals else 0))
            fl += i_ * i_ + 2 * i_ * s_ + 2 * i_ + 4 * s_
    return by, fl


class C5S(C5):
    """BASELINE configs[4] as the reference states it -- ONE parameter vector, the replicate batch sharded across
    GPUs -- on the shared-precision path (SURVEY 8f-1): J once per GPU, h and g per replicate (72 MB instead of
    926 MB of HBM each), so 1,536 replicates fit one GPU instead of 128."""
    key = "c5s"
    shared = True
    default_batch = 1536
    nsim = 32
    workload = ("synthetic level-1 network, 100,000 tips + 10,000 reticulations (219,999 nodes; clique tree of 209,998 "
                "clusters, sender dimensions 16 / 32 / 48), MvFullBrownianMotion p=16, ONE parameter vector, 1,536 trait "
                "replicates per GPU on the SHARED-PRECISION path (J stored and factorised once per GPU, h and g per replicate: "
                "72 MB of HBM each = 111 GB; 32 replicates simulated down the network, the others are rescaled copies "
                "x (1 + 0.001 k)), assignfactors! + calibrate! (post+pre order) + integratebelief!(root) "
                "[BASELINE configs[4], shared-J path of SURVEY 8f-1: own byte count 8*(m_F + 1 + 4*(s+1)) per message]")
    step_text = "assign_factors (K1: J once, h / g per replicate) + calibrate (419,994 messages: group pass + element pass) + integrate(root)"
    kernel_text = "k_hmsg_bulk<I> / k_hmsg<I> family (element pass of the 419,994 messages; the group pass k_jmsg runs once per GPU)"

    def inputs(self, B, rank):
        params, base = C5.inputs(self, min(B, self.nsim), rank)
        if B <= base.shape[0]:
            return params, base
        reps = -(-B // base.shape[0])
        tips = np.concatenate([base * (1.0 + 0.001 * k) for k in range(reps)])[:B]
        return params, np.ascontiguousarray(tips)

    def cost(self, plan):
        return shared_cost(self, plan, (0, 1))


WORKLOADS = {"c2": C2, "c2s": C2S, "c3": C3, "c3l": C3L, "c4": C4, "c5": C5, "c5s": C5S}


# ----------------------------------------------------------------------------- config shared by both arms
def messages_per_unit(w):
    d = w.d
    if w.key in ("c2", "c2s", "c5", "c5s"):
        return 2 * len(d["trees"][0][0])
    if w.key == "c4":
        return len(d["trees"][0][0])
    return 2 * sum(len(t[0]) for t in d["trees"])  # loopy: one iteration over all spanning trees


def state_bytes_per_element(w):
    """HBM bytes of one batch element (beliefs + factor snapshot + residuals), from the belief dimensions."""
    d = w.d
    dims, nc = d["belief_dim"], d["nclusters"]
    slots = sum(m * (m + 1) // 2 + m + 1 for m in dims)
    if w.residuals:
        slots += sum(m * (m + 1) // 2 + m + 1 for m in dims[:nc])           # ClusterFactor snapshot
        slots += 2 * sum(m * (m + 1) // 2 + m for m in dims[nc:])          # MessageResidual per directed message
    return 8 * slots


def make_config(w, B, n_gpus):
    """The `config` object of the JSON line: identical in the GPU arm and in the reference arm."""
    st = state_bytes_per_element(w) * B / 1e9
    gather = ("; the per-replicate results of all ranks are gathered every step (GPU arm: written by the integrate kernel "
              "into every rank's window over NVLink peer stores; checked against one NCCL all_gather)" if n_gpus > 1 else "")
    return {"workload": w.workload, "batch_per_gpu": int(B), "ntraits": int(w.d["ntraits"]),
            "messages_per_unit": int(messages_per_unit(w)), "step": w.step_text + gather,
            "l2": "inputs larger than L2: %.2f GB of beliefs%s per GPU rewritten every step (L2 = 126 MB)"
                  % (st, " + factors + residuals" if w.residuals else ""),
            "parallelism": f"batch sharded over {n_gpus} GPU(s), plan replicated, no data-path collective"}


# ----------------------------------------------------------------------------- reference arm / cpu baseline
def cpu_port_rate(w, params, tips, seconds, nthreads=0, steps=2, warmup=1, min_sample=64):
    """units/s of the C/OpenMP oracle port on a bounded sample of the workload (warmed up, mean of `steps`)."""
    from oracle.cport import COracle, dll
    co = COracle.from_plan_dict(w.d)
    kw = dict(root_belief=w.d["root_cluster"], nthreads=nthreads, ncolors=w.ncolors, want_fe=(w.key in ("c3", "c3l")), **w.cpu_kw)
    B = max(params.shape[0], tips.shape[0])

    def run(n):
        return co.run_batch(params[:n] if params.shape[0] > 1 else params, tips[:n] if tips.shape[0] > 1 else tips,
                            B=n, **kw)
    n0 = min(max(min_sample, B // 32), B)
    run(n0)  # warm-up (thread pool, page faults)
    t = time.perf_counter()
    run(n0)
    r0 = n0 / (time.perf_counter() - t)
    n = int(min(B, max(n0, r0 * seconds)))
    for _ in range(warmup):
        run(n)
    t = time.perf_counter()
    for _ in range(steps):
        out = run(n)
    dt = (time.perf_counter() - t) / steps
    assert (out["status"] == 0).all()
    cores = dll().pgbpo_num_threads() if nthreads <= 0 else nthreads
    return n / dt, cores, n, dt, (out["fe"][:, 2] if w.key in ("c3", "c3l") else out["loglik"])


def host_threads():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def julia_reference(w, B):
    """The reference itself (baseline/julia_threads.jl: Threads.@threads over replicates) when a `julia` executable
    with PhyloGaussianBeliefProp installed exists on this box; None otherwise (the image has no Julia)."""
    import shutil
    jl = shutil.which("julia")
    if jl is None or w.key != "c2":
        return None
    try:
        r = subprocess.run([jl, "--threads=auto", os.path.join(ROOT, "baseline", "julia_threads.jl"), "--replicates", str(B),
                            "--seconds", "3"], capture_output=True, text=True, timeout=900)
        line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
        return json.loads(line)
    except Exception:  # noqa: BLE001  (package not installed, script failed: fall back to the port)
        return None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]()
    B = args.batch or w.default_batch
    jl = julia_reference(w, B)
    if jl is not None:
        value, cores, dt, kind, sample = jl["value"], jl["cores"], jl["seconds_per_step"], "reference", jl["sample"]
    else:
        params, tips = w.inputs(B, 0)
        # all host threads this process may use (torchrun exports OMP_NUM_THREADS=1: override it explicitly)
        value, cores, n, dt, _ = cpu_port_rate(w, params, tips, 3.0, nthreads=host_threads(), steps=args.steps, warmup=args.warmup)
        value *= getattr(w, "niter", 1)
        kind, sample = "port", f"{n} of {B} batch elements per step ({w.cpu_text})"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": w.unit, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": make_config(w, B, args.gpus),
        "reference_note": ("the reference itself: baseline/julia_threads.jl (Threads.@threads over replicates)" if kind == "reference" else
                           "the reference is Julia (absent from the image): C/OpenMP restatement of its algorithm (oracle/c), "
                           "all host threads, bounded sample per step; baseline/julia_threads.jl runs instead wherever julia exists"),
        "cpu_baseline": {"value": value, "unit": w.unit, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": w.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: NVML polled in-process every
    2 ms (the timed region of the small config lasts ~20 ms, shorter than nvidia-smi's period);
    falls back to `nvidia-smi -lms 100` if NVML cannot be loaded."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.nv, self.stop_flag, self.mx = [], None, None, False, None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.h = nv.nvmlDeviceGetHandleByIndex(index)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.nv = nv
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nv
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not self.stop_flag:
            try:
                c = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.rows.append((time.perf_counter(), c, [k for k, b in bits.items() if r & b]))
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                c, m = float(f[0]), float(f[1])
            except (ValueError, IndexError):
                continue
            self.mx = m
            self.rows.append((time.perf_counter(), c, [n for n, v in zip(names, f[3:7]) if v.lower().startswith("active")]))

    def stop(self, t0, t1):
        if self.nv is None and not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML / nvidia-smi"], "samples": 0}
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
        self.stop_flag = True
        inside = [(c, r) for t, c, r in self.rows if t0 <= t <= t1]
        where = "timed region"
        if not inside:  # only possible with the nvidia-smi fallback on a very short region
            inside, where = [(c, r) for t, c, r in self.rows], "whole run (region shorter than the sampling period)"
        sm = [c for c, _ in inside]
        reasons = sorted({x for _, r in inside for x in r})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.mx, "reasons": reasons,
                "samples": len(sm), "sampled": where, "source": "nvml" if self.nv else "nvidia-smi"}


# ----------------------------------------------------------------------------- GPU arm
class Ctx:
    """Process-wide state of the GPU arm (one process per GPU)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        if args.gpus != self.world and self.rank == 0:
            print(f"warning: --gpus {args.gpus} but WORLD_SIZE={self.world}; reporting n_gpus={self.world}", file=sys.stderr)
        self.stream = torch.cuda.current_stream()
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            self.peak, self.peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            self.peak, self.peak_src = 6650.0, "fallback (B200_PROFILING.md)"

    def sync(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]


def dump_outputs(outdir, arrays):
    """Writes every array as <outdir>/<name>.npy in float64, all files together at most DUMP_BYTES.  If the arrays
    do not fit, each keeps a fixed, seeded sample of its rows, whose indices go to <name>_rows.npy (float64, exact
    below 2^53)."""
    os.makedirs(outdir, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_BYTES - 2 * 4096 * len(arrays)  # room for the .npy headers of two files per array
    for name, a in arrays.items():
        rows_path = os.path.join(outdir, name + "_rows.npy")
        if total > budget:
            # half the budget for the sampled rows, at most as much again for their indices (a row is >= 8 bytes)
            keep = max(1, int(a.shape[0] * budget / (2 * total)))
            rows = np.sort(np.random.default_rng(SEED).choice(a.shape[0], size=keep, replace=False))
            np.save(rows_path, rows.astype(np.float64))
            a = a[rows]
        elif os.path.exists(rows_path):
            os.remove(rows_path)  # left by an earlier, sampled dump: these rows are all there is now
        np.save(os.path.join(outdir, name + ".npy"), a)


def measure(w, args, ctx, steps, headline, cpu_seconds, e2e_steps_cap):
    """One workload on this rank's GPU: device-resident arm (value, roofline), end-to-end arm (host buffers), CPU
    check on a bounded sample (rank 0 of a single-GPU run).  Returns the dict of the JSON line (rank 0) or None."""
    import pgbp_b200
    from pgbp_b200 import _lib as L
    from pgbp_b200 import sharding
    torch, dist = ctx.torch, ctx.dist
    rank, world, local, dev, stream = ctx.rank, ctx.world, ctx.local, ctx.dev, ctx.stream
    d = w.d
    B = (args.batch if headline else 0) or w.default_batch
    p = d["ntraits"]
    # host memory guard for the big workloads (c5 / c5s hold GBs of tip data per rank): refuse rather than swap
    need = 8.0 * B * len(d["tip_nodes"]) * p
    if need > 1e9:
        import psutil
        avail = psutil.virtual_memory().available
        if 2.5 * need * world > avail:
            raise RuntimeError("host memory: %.0f GB of tip data per rank x %d ranks, %.0f GB available" % (need / 1e9, world, avail / 1e9))
    params, tips = w.inputs(B, rank)
    if tips.nbytes > 2e9:  # keep ONE host copy of big inputs, in pinned memory (it is also the e2e arm's source buffer)
        pinned_tips = torch.from_numpy(tips).pin_memory()
        tips = pinned_tips.numpy()
    lib = pgbp_b200.default_library()
    plan = pgbp_b200.ClusterGraphPlan(d["nclusters"], d["belief_dim"], d["sepset_clusters"], d["upind"], d["trees"], p,
                                      d["families"], lib)
    group = B if getattr(w, "shared", False) else 0
    bt = pgbp_b200.BatchedClusterGraphBelief(plan, B, device=local, stream=stream.cuda_stream,
                                             factors=w.residuals, residuals=w.residuals, shared_precision_group=group)
    if headline:
        if args.walk is not None:
            bt.set_walk_mode(args.walk)
        if args.pipeline is not None:
            bt.set_pipeline(args.pipeline)
        if args.graph is not None:
            bt.set_graph_mode(args.graph)
        if args.tilewalk is not None:
            bt.set_tilewalk_mode(args.tilewalk)
        if args.coop is not None:
            bt.set_coop_mode(args.coop)
        if args.tw_lanes or args.tw_wide:
            bt.set_tilewalk_params(args.tw_lanes, args.tw_wide)
    root = d["root_cluster"] + 1
    bytes_unit, flops_unit = w.cost(plan)
    nmsg = messages_per_unit(w) * getattr(w, "niter", 1)
    upe = getattr(w, "niter", 1)  # metric units per element per step
    loopy = w.key in ("c3", "c3l")

    # ---- gather of the per-element results (N > 1) ------------------------------------------------
    # Default: fused into the producing kernel -- pgbp_integrate_gather / pgbp_comm_put store every result into
    # row `rank` of every rank's window over NVLink peer stores (no collective launch on the step's critical
    # path).  --gather nccl (or a failed IPC mapping on some rank): asynchronous double-buffered NCCL all-gather.
    _, ld, _ = bt.device_view()
    comm, gather_kind = None, "none"
    if world > 1:
        ok = 1.0
        if args.gather == "peer":
            try:
                comm = sharding.PeerGather(lib, local, rank, world, ld, nbuffers=2)
            except Exception as ex:  # noqa: BLE001
                print(f"rank {rank}: peer windows unavailable ({ex}); falling back to the NCCL all-gather", file=sys.stderr)
                ok = 0.0
        else:
            ok = 0.0
        ok = -ctx.max_over_ranks([-ok])[0]  # min over ranks: every rank must use the same transport
        if ok < 0.5:  # some rank could not map its peers: every rank drops its window (unmap, barrier, free)
            if comm is not None:
                lib.pgbp_comm_disconnect(comm.handle)
            ctx.sync()
            if comm is not None:
                comm.close()
                comm = None
        gather_kind = "peer" if comm is not None else "nccl"
    d_norms = [torch.empty(ld, dtype=torch.float64, device=dev) for _ in range(2)]
    gathered = [torch.empty(world * ld, dtype=torch.float64, device=dev) for _ in range(2)] if gather_kind == "nccl" else None
    pending = [None, None]
    counter = [0]
    d_fe = torch.empty(3 * ld, dtype=torch.float64, device=dev) if loopy else None

    def finish():
        """per-element result of the step (integratebelief! at the root, or the factored energy for loopy BP)
        + (N > 1) its gather."""
        k = counter[0] % 2
        counter[0] += 1
        if pending[k] is not None:
            pending[k].wait()  # stream-level wait: buffer k is free again
            pending[k] = None
        if loopy:
            bt.factored_energy_device(d_fe.data_ptr())
            if comm is not None:
                comm.put(bt, k, d_fe[2 * ld:3 * ld].data_ptr())
            else:
                d_norms[k].copy_(d_fe[2 * ld:3 * ld])
        elif comm is not None:
            comm.integrate_gather(bt, root, k)
        else:
            bt.integrate_device(root, d_norms[k].data_ptr())
        if gather_kind == "nccl":
            pending[k] = dist.all_gather_into_tensor(gathered[k], d_norms[k], async_op=True)

    if w.key in ("c2", "c2s"):
        bt.assignfactors(params, tips)  # factors resident in HBM (K1 is outside the device-resident timed region)

        def step(ev=None):
            bt.init_beliefs_reset_fromfactors()
            if ev:
                ev[0].record(stream)
            bt.calibrate_async(None, 1, update_residualnorm=True)
            if ev:
                ev[1].record(stream)
            finish()
    elif loopy:
        bt.assignfactors(params, tips)

        def step(ev=None):
            bt.init_beliefs_reset_fromfactors()
            bt.init_messagecalibrationflags_reset()
            bt.regularizebeliefs_bycluster()
            if ev:
                ev[0].record(stream)
            bt.calibrate_async(None, w.niter, update_residualnorm=True)
            if ev:
                ev[1].record(stream)
            finish()
    else:
        d_params = torch.from_numpy(params).to(dev)
        d_tips = torch.from_numpy(tips).to(dev)
        direction = L.CAL_BOTH if w.key in ("c5", "c5s") else L.CAL_POSTORDER

        def step(ev=None):
            bt.assignfactors_device(d_params.data_ptr(), params.shape[0], d_tips.data_ptr(), tips.shape[0], ncolors=w.ncolors)
            if ev:
                ev[0].record(stream)
            bt.calibrate_async(None, 1, update_residualnorm=False, direction=direction)
            if ev:
                ev[1].record(stream)
            finish()

    def barrier():
        for k in range(2):
            if pending[k] is not None:
                pending[k].wait()
                pending[k] = None
        ctx.sync()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    barrier()
    sampler = ClockSampler(local) if (rank == 0 and headline) else None
    bt.launch_count(reset=True)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    for k in range(steps):
        step(evs[k])
    e1.record(stream)
    barrier()
    t1 = time.perf_counter()
    launches = bt.launch_count()
    ms_total = e0.elapsed_time(e1)
    ms_msgs = sum(a.elapsed_time(b) for a, b in evs)
    clocks = sampler.stop(t0, t1) if sampler else None
    ms_total, ms_msgs = ctx.max_over_ranks([ms_total, ms_msgs])
    value = world * B * upe * steps / (ms_total * 1e-3)
    st = bt.status()
    assert (st == 0).all(), "numerical failure inside the timed region"
    # the gathered vector of the LAST step: every rank's results in rank order; it must equal an NCCL all-gather of
    # the same values (peer transport) and this rank's own slice (both transports)
    klast = (counter[0] - 1) % 2
    gather_checked = None
    if comm is not None:
        comm.wait(bt, klast)
        comm.check(bt)
        ctx.sync()
        win = comm.read(bt, klast)
        wld = comm.ld
        loglik_dev = win[rank, :B].copy()
        mine = torch.from_numpy(win[rank].copy()).to(dev)
        ref_all = torch.empty(world * wld, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(ref_all, mine)  # NCCL cross-check of the peer-written window
        assert np.array_equal(ref_all.cpu().numpy().reshape(world, wld)[:, :B], win[:, :B]), "peer-gathered window != NCCL all_gather"
        gather_checked = "window of every rank == NCCL all_gather of the same values (bitwise)"
        gathered_last = win[:, :B]
    else:
        loglik_dev = d_norms[klast][:B].cpu().numpy()
        if world > 1:
            gathered_last = gathered[klast].view(world, ld)[:, :B].cpu().numpy()
            assert np.array_equal(gathered_last[rank], loglik_dev)
            gather_checked = "own slice of the NCCL-gathered vector == local result (bitwise)"
    if headline and args.dump_outputs and rank == 0:
        outs = {"factored_energy": d_fe.view(3, ld)[:, :B].T.cpu().numpy()} if loopy else {"loglik": loglik_dev}
        if world > 1:
            outs["gathered"] = gathered_last.reshape(-1)
        dump_outputs(args.dump_outputs, outs)

    # ---- end-to-end arm: public host-buffer API, pinned host inputs, D2H of the result -------
    # Every step = one synchronous sequence of public calls on one batch: H2D of that step's inputs
    # (pinned) + K1, message passing, integratebelief! with the D2H of the result.  When several batches
    # fit in HBM the steps alternate between batches driven by their own host threads (the ABI allows
    # distinct batches on distinct threads): the H2D / D2H of one step overlaps the kernels of the others.
    big = params if w.key == "c4" else tips
    e2e_steps = min(steps, e2e_steps_cap)
    d_params = d_tips = None  # the device-resident arm's input copies are not needed any more (c5s: 20 GB)
    step = finish = None
    torch.cuda.empty_cache()
    free_b, total_b = torch.cuda.mem_get_info()
    # (per extra batch: its state plus the device-side staging of one step's inputs, which device_bytes() may not hold yet)
    nb_e2e = max(1, min(args.e2e_batches, 1 + int(free_b / (bt.device_bytes() * 1.1 + 2.5 * big.nbytes))))
    bts = [bt]
    for _ in range(nb_e2e - 1):
        bts.append(pgbp_b200.BatchedClusterGraphBelief(plan, B, device=local, factors=w.residuals, residuals=w.residuals,
                                                       shared_precision_group=group))
        if headline and args.pipeline is not None:
            bts[-1].set_pipeline(args.pipeline)
    pin_np = [big if (big.nbytes > 2e9 and big is tips) else torch.from_numpy(big.copy()).pin_memory().numpy() for _ in bts]
    results = [None] * len(bts)

    def e2e_step(i):
        b_ = bts[i]
        if w.key in ("c2", "c2s"):
            b_.assignfactors(params, pin_np[i])                 # H2D of this step's inputs + K1
            succ, iscal = b_.calibrate(None, 1)                 # D2H of succ / iscal
        elif loopy:
            b_.assignfactors(params, pin_np[i])
            b_.regularizebeliefs_bycluster()
            succ, iscal = b_.calibrate(None, w.niter)
            results[i] = b_.factored_energy()[:, 2]
            return
        elif w.key in ("c5", "c5s"):
            b_.assignfactors(params, pin_np[i])
            succ, _ = b_.calibrate(None, 1, update_residualnorm=False)
        else:
            b_.assignfactors(pin_np[i], tips, ncolors=w.ncolors)
            succ = b_.propagate_1traversal_postorder(0, update_residualnorm=False)
        results[i] = b_.integratebelief(root, want_mu=False)[1]  # D2H of the result

    errors = []

    def worker(i, n):
        torch.cuda.set_device(local)
        try:
            for _ in range(n):
                e2e_step(i)
        except Exception as ex:  # re-raised on the main thread after the join
            errors.append(ex)

    def run_e2e(n):
        if len(bts) == 1:
            worker(0, n)
            if errors:
                raise errors[0]
            return
        nb = len(bts)
        ths = [threading.Thread(target=worker, args=(i, n // nb + (i < n % nb))) for i in range(nb)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        if errors:
            raise errors[0]
    run_e2e(2 * len(bts))
    barrier()
    t0e = time.perf_counter()
    run_e2e(e2e_steps)
    barrier()
    dte = time.perf_counter() - t0e
    dte = ctx.max_over_ranks([dte])[0]
    e2e_value = world * B * upe * e2e_steps / dte
    h2d = tips.nbytes + params.nbytes
    d2h = results[0].nbytes + (1 if w.key == "c4" else 2) * 4 * B
    for r_ in results:
        assert np.allclose(r_, loglik_dev, rtol=1e-12, atol=0)  # same kernels, same inputs: identical
    del bts[1:]
    if comm is not None:
        comm.close(ctx.sync)
    if rank != 0:
        return None

    # ---- roofline of the dominant kernel family (k_message*): ALGORITHMIC bytes / device time -----------
    achieved = bytes_unit * B * steps / (ms_msgs * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get(w.key, {}).get("dram_bytes_per_unit_per_element")
        if traffic is not None:
            traffic = traffic * B
    roofline = {"bound": "hbm", "achieved": achieved, "peak": ctx.peak, "unit": "GB/s", "frac": achieved / ctx.peak,
                "traffic": traffic, "peak_source": ctx.peak_src, "kernel": w.kernel_text,
                "basis": "algorithmic-bytes roofline: SURVEY 8(d) bytes of every message / CUDA-event time of the message "
                         "kernels; the lazy sepset zero, L2 hits on lines written by the previous level and (c2s) shared J "
                         "rows make the DRAM traffic smaller than the algorithmic count, see dram_gbs_from_traffic",
                "dram_gbs_from_traffic": (traffic * steps / (ms_msgs * 1e-3) / 1e9) if traffic else None,
                "algorithmic_bytes_per_unit_per_element": bytes_unit,
                "algorithmic_flops_per_unit_per_element": flops_unit,
                "fp64_gflops_achieved": flops_unit * B * steps / (ms_msgs * 1e-3) / 1e9,
                "share_of_step": ms_msgs / ms_total}

    # ---- CPU baseline + parity of the results (rank 0, N = 1 only) -------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu:
        rate, cores, n, dt, ll_cpu = cpu_port_rate(w, params, tips, cpu_seconds, nthreads=host_threads(),
                                                   min_sample=64 if headline else 8)
        rate *= upe
        err = float(np.max(np.abs(ll_cpu / loglik_dev[:n] - 1)))
        cpu = {"value": rate, "unit": w.unit, "cores": cores, "kind": "port",
               "sample": f"{n} of {B} batch elements in {dt:.2f} s per pass, warmed up, mean of 2 passes ({w.cpu_text}, "
                         f"C/OpenMP restatement of the Julia reference)",
               "max_rel_err_gpu_vs_cpu_loglik": err}
        # c3 (Bethe): the reference's own algorithm evaluated in binary64 is ~3e-5 away from its exact (binary128)
        # result after 10 loopy iterations (oracle/tools/adjudicate_c3.py, DESIGN.md section 2): stated tolerance 1e-4
        assert err < (1e-4 if w.key == "c3" else 1e-10), err

    line = {
        "metric": METRIC, "value": value, "unit": w.unit, "n_gpus": world, "steps": steps,
        "warmup": warm, "ms_per_step": ms_total / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": make_config(w, B, world),
        "timing": {"passes_timed": steps, "timed_region_ms": ms_total,
                   "note": "`steps` passes inside one CUDA-event pair (max over ranks); ms_per_step is per pass"
                           + ("; device-resident passes start from the factors resident in HBM (factor assignment, K1, is "
                              "outside this arm and inside e2e)" if w.key in ("c2", "c2s", "c3", "c3l") else "")},
        "gather": {"kind": gather_kind, "checked": gather_checked} if world > 1 else None,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "e2e": {"value": e2e_value, "unit": w.unit, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "steps": e2e_steps, "path": w.e2e_text + ((" (%d batches x %d host threads: copies of one step overlap the "
                                                          "kernels of the others)" % (nb_e2e, nb_e2e)) if nb_e2e > 1 else "")},
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    return line


def compact(line):
    """What the headline line keeps of another workload's measurement."""
    r = line["roofline"]
    out = {"workload": line["config"]["workload"], "batch_per_gpu": line["config"]["batch_per_gpu"], "unit": line["unit"],
           "value": line["value"], "ms_per_step": line["ms_per_step"], "passes_timed": line["timing"]["passes_timed"],
           "n_gpus": line["n_gpus"],
           "roofline": {"bound": r["bound"], "achieved": r["achieved"], "peak": r["peak"], "unit": r["unit"], "frac": r["frac"],
                        "traffic": r["traffic"], "kernel": r["kernel"], "share_of_step": r["share_of_step"]},
           "e2e": line["e2e"], "gpu_launches": line["gpu_launches"], "gather": line["gather"]}
    if line["cpu_baseline"]:
        out["cpu_baseline"] = {k: line["cpu_baseline"][k] for k in ("value", "cores", "kind", "sample")}
        out["max_rel_err"] = line["cpu_baseline"]["max_rel_err_gpu_vs_cpu_loglik"]
    return out


def run_gpu(args):
    import gc
    ctx = Ctx(args)
    t_start = time.perf_counter()
    w = WORKLOADS[args.workload]()
    line = measure(w, args, ctx, args.steps, True, args.cpu_seconds, 10 ** 9 if args.workload in ("c2", "c2s") else 5)
    # The other BASELINE configurations, each measured the same way at reduced step counts, so that the driver's
    # own run holds them too (configs[3] = the north-star target: 10k-tip network, p = 8, 4,096 parameter vectors).
    others = {}
    if args.workload == "c2" and not args.no_others:
        plan = [("c4", 3, 3.0), ("c3", 2, 3.0), ("c3l", 2, 3.0), ("c2s", 20, 2.0), ("c5", 2, 4.0), ("c5s", 2, 4.0)]
        for key, k_steps, cpu_s in plan:
            if key in ("c5", "c5s") and (args.no_c5 or time.perf_counter() - t_start > args.others_budget_s):
                if ctx.rank == 0:
                    others[key] = {"skipped": "time budget of the default run" if not args.no_c5 else "--no-c5"}
                continue
            gc.collect()
            ctx.torch.cuda.empty_cache()
            try:
                ww = WORKLOADS[key]()
                ln = measure(ww, args, ctx, k_steps, False, cpu_s, 4)
                if ctx.rank == 0:
                    others[key] = compact(ln)
                del ww
            except AssertionError:
                raise
            except Exception as ex:  # noqa: BLE001  (e.g. out of memory for c5 on a smaller GPU)
                if ctx.rank == 0:
                    others[key] = {"failed": repr(ex)[:300]}
    if ctx.rank == 0:
        if others:
            line["other_workloads"] = others
        print(json.dumps(line))
    if ctx.world > 1:
        ctx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the headline workload")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="batch elements per GPU (default: the workload's)")
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS), help="c2 = BASELINE configs[1] (headline), "
                    "c4 = configs[3] (10k-tip synthetic network, p=8)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="headline workload only (skip the other_workloads block)")
    ap.add_argument("--no-c5", action="store_true", help="skip the 100k-tip workload in the other_workloads block")
    ap.add_argument("--others-budget-s", type=float, default=240.0, help="c5 / c5s are skipped when the run is already older than this")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"], help="N > 1: results gathered through NVLink peer "
                    "windows fused into the integrate kernel (default) or an asynchronous NCCL all-gather per step")
    ap.add_argument("--e2e-batches", type=int, default=4, help="batches (= host threads) alternating in the end-to-end arm")
    ap.add_argument("--pipeline", type=int, default=None, help="element chunks of a calibration (-1 auto, 1 off)")
    ap.add_argument("--tilewalk", type=int, default=None, help="tile-walk kernel (-1 auto, 0 off, 1 on)")
    ap.add_argument("--tw-lanes", type=int, default=0, help="tile-walk message lanes per block (4, 8, 16)")
    ap.add_argument("--tw-wide", type=int, default=0, help="tile-walk: steps wider than this keep their own launches")
    ap.add_argument("--coop", type=int, default=None, help="medium-shape kernel: -1 auto, 1 shared-memory, 8 cooperative, 0 generic")
    ap.add_argument("--graph", type=int, default=None, help="CUDA-graph replay of calibrate (-1 auto, 0 off, 1 on)")
    ap.add_argument("--walk", type=int, default=None, help="kernel strategy override: 0 level-parallel, 1 walk kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the results of the last timed step of the "
                    "headline workload to DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU arm computed; the reference arm has no such step")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
