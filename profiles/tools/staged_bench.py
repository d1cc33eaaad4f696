"""Parent build against this tree's build of the CUDA library, on one GPU, in one session.

    python profiles/tools/staged_bench.py --out DIR --lib parent=PATH --lib new=PATH [--lib NAME=PATH ...]
                                          [--runs 3] [--workloads c2:700,c3:30,...] [--dumps c2,c4,c3]
                                          [--no-profile] [--default-runs]

Every library is an already built libpgbp_b200.so (phylogaussianbeliefprop.jl_b200/build.py); nothing is compiled
here.  The first --lib is the baseline.  Written to DIR:
  card.csv                  nvidia-smi name, power limit and maximum SM clock, read in the same session
  <w>_<lib>_<k>.json        bench.py --workload w --steps K --no-others --no-cpu for every w:K of --workloads (default
                            c2:700), libraries alternated, k = 1..runs
  dump_<w>_<lib>/           bench.py --dump-outputs for --dumps (default c2, c4, c3; same seeded inputs)
  kernels_<lib>.txt / .json torch.profiler per-kernel device time of one C2 step (after warm-up), own process
                            (unless --no-profile)
  default_<lib>.json        (--default-runs) the default bench.py run: other_workloads block and CPU check
  summary.json              per workload: medians, spreads, ratios against the baseline and whether each median lies
                            within the baseline's min..max; byte-identity of every dump
  kernels_<w>_<lib>.txt     (--profiles w:K,...) torch.profiler per-kernel device time of bench.py --workload w --steps K
                            --warmup 1, set-up included, own process per library
Run `--profile-c2 FILE` alone to profile one C2 step with the library PGBP_B200_LIB selects.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def run(cmd, lib, out, err, timeout=900):
    env = dict(os.environ, PGBP_B200_LIB=lib)
    with open(out, "w") as fo, open(err, "w") as fe:
        r = subprocess.run(cmd, cwd=ROOT, env=env, stdout=fo, stderr=fe, timeout=timeout)
    return r.returncode


def last_json(path):
    try:
        lines = [ln for ln in open(path) if ln.strip().startswith("{")]
        return json.loads(lines[-1]) if lines else None
    except (OSError, ValueError):
        return None


def profile_c2(path):
    """One C2 step (bench.py's step: reset from factors + calibrate + integrate at the root) under torch.profiler."""
    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    import pgbp_b200
    w = bench.C2()
    d = w.d
    B = w.default_batch
    params, tips = w.inputs(B, 0)
    lib = pgbp_b200.default_library()
    plan = pgbp_b200.ClusterGraphPlan(d["nclusters"], d["belief_dim"], d["sepset_clusters"], d["upind"], d["trees"],
                                      d["ntraits"], d["families"], lib)
    stream = torch.cuda.current_stream()
    bt = pgbp_b200.BatchedClusterGraphBelief(plan, B, stream=stream.cuda_stream, factors=True, residuals=True)
    bt.assignfactors(params, tips)
    _, ld, _ = bt.device_view()
    norm = torch.empty(ld, dtype=torch.float64, device="cuda")
    root = d["root_cluster"] + 1

    def step():
        bt.init_beliefs_reset_fromfactors()
        bt.calibrate_async(None, 1, update_residualnorm=True)
        bt.integrate_device(root, norm.data_ptr())

    for _ in range(50):
        step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    write_kernel_table(prof, path, "kernel device time of one C2 step (B = %d)" % B, {"B": B})
    assert np.isfinite(norm[:B].cpu().numpy()).all()


def profile_workload(w, steps, path):
    """bench.py --workload w --steps steps --warmup 1 (set-up included) under torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    import bench
    sys.argv = ["bench.py", "--workload", w, "--steps", str(steps), "--warmup", "1", "--no-others", "--no-cpu"]
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        bench.main()
    write_kernel_table(prof, path, "kernel device time of bench.py --workload %s --steps %d --warmup 1 (set-up, warm-up "
                       "and timed steps)" % (w, steps), {"workload": w, "steps": steps})


def write_kernel_table(prof, path, title, extra):
    rows = {}
    for ev in prof.key_averages():
        us = getattr(ev, "self_device_time_total", 0.0)
        if us > 0:
            rows[ev.key] = [ev.count, us]
    total = sum(r[1] for r in rows.values())
    table = sorted(([n, c, us] for n, (c, us) in rows.items()), key=lambda x: -x[2])
    lib = os.environ.get("PGBP_B200_LIB")
    lib = os.path.relpath(lib, ROOT) if lib else "default"
    with open(path, "w") as f:
        f.write("library: %s\n%s, sum %.1f us\n" % (lib, title, total))
        f.write("%10s %6s %7s  %s\n" % ("us", "calls", "share", "kernel"))
        for n, c, us in table:
            f.write("%10.1f %6d %6.1f%%  %s\n" % (us, c, 100.0 * us / total if total else 0.0, n))
    json.dump(dict(extra, library=lib, sum_us=total,
                   kernels=[{"name": n, "calls": c, "us": us} for n, c, us in table]),
              open(os.path.splitext(path)[0] + ".json", "w"), indent=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--lib", action="append", default=[])
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--default-runs", action="store_true")
    ap.add_argument("--workloads", default="c2:700", help="timed workloads, name:steps, comma-separated")
    ap.add_argument("--dumps", default="c2,c4,c3", help="workloads whose outputs are dumped and compared")
    ap.add_argument("--no-profile", action="store_true", help="skip the per-kernel profile of one C2 step")
    ap.add_argument("--profile-c2")
    ap.add_argument("--profile-workload", nargs=3, metavar=("W", "STEPS", "FILE"))
    ap.add_argument("--profiles", default="", help="name:steps, comma-separated: per-kernel table of each workload and "
                    "library, own process each (kernels_<w>_<lib>.txt)")
    args = ap.parse_args()
    if args.profile_c2:
        profile_c2(args.profile_c2)
        return
    if args.profile_workload:
        w, k, f = args.profile_workload
        profile_workload(w, int(k), f)
        return
    libs = [tuple(x.split("=", 1)) for x in args.lib]
    libs = [(n, os.path.abspath(p)) for n, p in libs]
    for n, p in libs:
        if not os.path.exists(p):
            raise SystemExit("missing library %s: %s" % (n, p))
    out = os.path.abspath(args.out)
    os.makedirs(out, exist_ok=True)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                          capture_output=True, text=True)
    open(os.path.join(out, "card.csv"), "w").write(card.stdout + card.stderr)
    py = sys.executable
    workloads = [(w, int(k)) for w, k in (x.split(":") for x in args.workloads.split(",") if x)]
    summary = {"card": card.stdout.strip().splitlines(), "libraries": {n: os.path.relpath(p, ROOT) for n, p in libs},
               "dumps": {}}
    vals = {(w, n): [] for w, _ in workloads for n, _ in libs}
    for k in range(1, args.runs + 1):
        for w, steps in workloads:
            for n, p in libs:
                f = os.path.join(out, "%s_%s_%d.json" % (w, n, k))
                rc = run([py, "bench.py", "--workload", w, "--steps", str(steps), "--no-others", "--no-cpu"], p, f,
                         f[:-5] + ".err")
                j = last_json(f)
                if rc == 0 and j:
                    vals[(w, n)].append(j["value"])
    base = libs[0][0]
    for w, _ in workloads:
        summary[w] = {}
        for n, _ in libs:
            v = vals[(w, n)]
            summary[w][n] = {"values": v, "median": statistics.median(v) if v else None,
                             "min": min(v) if v else None, "max": max(v) if v else None}
        b = summary[w][base]
        for n, _ in libs:
            s = summary[w][n]
            if b["median"] and s["median"]:
                s["median_over_baseline"] = s["median"] / b["median"]
                s["min_over_baseline_max"] = s["min"] / b["max"]
                s["median_within_baseline_spread"] = b["min"] <= s["median"] <= b["max"]
    steps = {"c2": 20, "c4": 3, "c3": 2, "c3l": 2, "c2s": 20, "c5": 1, "c5s": 1}
    for w in filter(None, args.dumps.split(",")):
        st = steps[w]
        for n, p in libs:
            dd = os.path.join(out, "dump_%s_%s" % (w, n))
            f = os.path.join(out, "dump_%s_%s.json" % (w, n))
            run([py, "bench.py", "--workload", w, "--steps", str(st), "--warmup", "1", "--no-others", "--no-cpu",
                 "--dump-outputs", dd], p, f, f[:-5] + ".err")
        ref = os.path.join(out, "dump_%s_%s" % (w, base))
        for n, _ in libs[1:]:
            dd = os.path.join(out, "dump_%s_%s" % (w, n))
            names = sorted(os.listdir(ref)) if os.path.isdir(ref) else []
            same = bool(names) and os.path.isdir(dd) and names == sorted(os.listdir(dd)) and all(
                open(os.path.join(ref, x), "rb").read() == open(os.path.join(dd, x), "rb").read() for x in names)
            summary["dumps"]["%s_%s" % (w, n)] = {"files": names, "byte_identical": same}
    for n, p in libs:
        if args.no_profile:
            break
        f = os.path.join(out, "kernels_%s.txt" % n)
        run([py, os.path.abspath(__file__), "--profile-c2", f], p, f + ".log", f + ".err")
    for w, k in (x.split(":") for x in args.profiles.split(",") if x):
        for n, p in libs:
            f = os.path.join(out, "kernels_%s_%s.txt" % (w, n))
            run([py, os.path.abspath(__file__), "--profile-workload", w, k, f], p, f + ".log", f + ".err", timeout=1800)
    if args.default_runs:
        for n, p in libs:
            f = os.path.join(out, "default_%s.json" % n)
            run([py, "bench.py"], p, f, f[:-5] + ".err", timeout=1800)
            j = last_json(f)
            if j:
                summary.setdefault("default", {})[n] = {
                    "c2": j.get("value"), "cpu_max_rel_err": (j.get("cpu_baseline") or {}).get("max_rel_err_gpu_vs_cpu_loglik"),
                    "other_workloads": {w: o.get("value") for w, o in (j.get("other_workloads") or {}).items()
                                        if isinstance(o, dict)}}
        dflt = summary.get("default", {})
        if base in dflt:
            for n, _ in libs[1:]:
                if n in dflt:
                    dflt[n]["other_over_baseline"] = {
                        w: (v / dflt[base]["other_workloads"][w]) if v and dflt[base]["other_workloads"].get(w) else None
                        for w, v in dflt[n]["other_workloads"].items()}
    json.dump(summary, open(os.path.join(out, "summary.json"), "w"), indent=1)
    print(json.dumps({w: summary[w] for w, _ in workloads}))
    print(json.dumps(summary["dumps"]))


if __name__ == "__main__":
    main()
