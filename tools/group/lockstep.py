"""Lockstep groups against solo runs on one resident Y (vbmf_b200_solver_run_group).

  restarts: c3-shaped synthetic Y (20000 x 200000), four dense H = 16 members with est_covs / est_var
  sweep:    c4-shaped synthetic Y (10000 x 100000), sparse members with H = 8, 16 and 40

For each workload the members run one after another (solo) and together (group), alternated --reps times, eps = 0, --steps
timed iterations after --warmup from the same uploaded state.  Recorded: wall time of each pass, per-model iterations per
second, K1 / K2 milliseconds from the context's profiling counters (a separate profiled pass), each member's largest
normwise field difference between its solo and group results (the split-K plans of the total width differ from the solo
ones, so it is rounding-level, not zero) and, for the sparse sweep, each member's lowerBound.  The card's name, power limit
and clocks are read in the same call.  Writes profiles/r08_group_<workload>.json (or under --out).

usage: python tools/group/lockstep.py [--workload restarts|sweep|both] [--steps 20] [--warmup 3] [--reps 3] [--out DIR]
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import vbmf_b200_loader  # noqa: E402

vb = vbmf_b200_loader.load()

WORKLOADS = {
    "restarts": dict(L=20000, M=200000, rank=32, kind="dense", Hs=[16, 16, 16, 16], opts=dict(est_covs=True, est_var=True)),
    "sweep": dict(L=10000, M=100000, rank=16, kind="sparse", Hs=[8, 16, 40], opts=dict(est_cb=True)),
}


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))
    except (OSError, subprocess.SubprocessError) as e:
        return {"error": str(e)}


class Shape:             # the init functions only read Y.shape
    def __init__(self, L, M):
        self.shape = (L, M)


def members(w, ctx):
    shape = Shape(w["L"], w["M"])
    ps = []
    for i, H in enumerate(w["Hs"]):
        rng = np.random.default_rng(1000 + i)
        ps.append(vb.vbmf_init(shape, H, rng=rng) if w["kind"] == "dense" else vb.vbmf_sparse_init(shape, H, rng=rng, trYTY=ctx.trYTY()))
    return ps


def field_diff(a, b):
    out = 0.0
    for k, v in vars(a).items():
        if isinstance(v, np.ndarray) and v.dtype == np.float64 and v.size:
            w = getattr(b, k)
            out = max(out, float(np.linalg.norm(v - w) / max(np.linalg.norm(w), 1e-300)))
    return out


def solo_pass(ctx, ps, flags, steps, warmup):
    qs = [copy.deepcopy(p) for p in ps]
    t = 0.0
    for q, f in zip(qs, flags):
        s = vb.Solver(ctx, q)
        s.upload(q)
        s.run(warmup, 0.0, f)
        s.upload(q)
        ctx.sync()
        t0 = time.perf_counter()
        it, _ = s.run(steps, 0.0, f)
        ctx.sync()
        t += time.perf_counter() - t0
        assert it == steps
        s.download(q)
        s.close()
    return t, qs


def group_pass(ctx, ps, flags, steps, warmup):
    qs = [copy.deepcopy(p) for p in ps]
    ss = [vb.Solver(ctx, q) for q in qs]
    for s, q in zip(ss, qs):
        s.upload(q)
    vb.run_group(ss, warmup, 0.0, flags)
    for s, q in zip(ss, qs):
        s.upload(q)
    ctx.sync()
    t0 = time.perf_counter()
    res = vb.run_group(ss, steps, 0.0, flags)
    ctx.sync()
    t = time.perf_counter() - t0
    assert all(it == steps for it, _ in res)
    for s, q in zip(ss, qs):
        s.download(q)
        s.close()
    return t, qs


def profiled(ctx, fn, *a):
    ctx.profile(True)
    fn(ctx, *a)
    prof = ctx.profile_read()
    ctx.profile(False)
    return {"k1_ms": prof["k1_ms"], "k1_launches": prof["k1_launches"], "k2_ms": prof["k2_ms"], "k2_launches": prof["k2_launches"]}


def run(name, args):
    w = WORKLOADS[name]
    ctx = vb.Context(device=0)
    ctx.synth(w["L"], w["M"], rank=w["rank"], noise=0.1, seed=20260101)
    ps = members(w, ctx)
    flags = [vb.api._flags(**w["opts"])] * len(ps)
    pairs = []
    for _ in range(args.reps):
        ts, qs_solo = solo_pass(ctx, ps, flags, args.steps, args.warmup)
        tg, qs_group = group_pass(ctx, ps, flags, args.steps, args.warmup)
        pairs.append({"solo_s": ts, "group_s": tg, "ratio_group_over_solo": tg / ts})
    n = len(ps)
    solo_rate = [n * args.steps / p["solo_s"] for p in pairs]
    group_rate = [n * args.steps / p["group_s"] for p in pairs]
    out = {
        "workload": name, "card": card(), "shape": [w["L"], w["M"]], "kind": w["kind"], "H": w["Hs"], "options": w["opts"],
        "steps": args.steps, "warmup": args.warmup, "eps": 0.0,
        "pairs": pairs,
        "median_model_iters_per_s": {"solo": float(np.median(solo_rate)), "group": float(np.median(group_rate))},
        "median_ratio_group_over_solo": float(np.median([p["ratio_group_over_solo"] for p in pairs])),
        "group_faster_in_every_pair": all(p["group_s"] < p["solo_s"] for p in pairs),
        "profile_solo": profiled(ctx, solo_pass, ps, flags, args.steps, 0),
        "profile_group": profiled(ctx, group_pass, ps, flags, args.steps, 0),
        "max_normwise_field_diff_solo_vs_group": [field_diff(a, b) for a, b in zip(qs_solo, qs_group)],
    }
    if w["kind"] != "dense":
        out["lower_bound"] = {"solo": [], "group": []}
        for key, qs in (("solo", qs_solo), ("group", qs_group)):
            for q in qs:
                s = vb.Solver(ctx, q)
                s.upload(q)
                out["lower_bound"][key].append(s.lower_bound())
                s.close()
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--workload", choices=["restarts", "sweep", "both"], default="both")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    for name in (["restarts", "sweep"] if args.workload == "both" else [args.workload]):
        res = run(name, args)
        path = os.path.join(args.out, "r08_group_%s.json" % name)
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps({k: res[k] for k in ("workload", "median_model_iters_per_s", "median_ratio_group_over_solo",
                                                "group_faster_in_every_pair", "profile_solo", "profile_group")}))


if __name__ == "__main__":
    main()
