"""Batched residual norms against the host norms they replace, on the two MIL batch shapes.

Batches: the c2 batch of bench.py (548 bags, L = 38, M = 5..40) and the Musk2-shaped batch of large_bags.py (100 bags,
L = 166, M = 1..1044), dual parameters with H = 20, H0 = 19, each bag against two class models.  Both routes run
mil.classify_bags(class_alg="dual")'s work on fresh copies of the parameters:
  (a) BatchedVbls(yhat=True).run(20, full_cov=True), then norm(YHat - Y, 2)/(L*M) per problem with NumPy on the host;
  (b) BatchedVbls(yhat=False).run(20, full_cov=True), then residual_norm()/(L*M) in one C-ABI call.
They alternate, --reps times each.  The script records the wall time of each route and of its two halves, the residual
call's kernels alone from the profiling K1 slot (so its packing is the call time minus that), and the largest relative
difference of the errors and whether the labels (0 iff err0 < err1) agree.  Writes one JSON file to --out.  Needs a GPU.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools", "batched"))


def copies(vb, ps):
    return [vb.copy(p) for p in ps]


def route(vb, ctx, Ys, ps, on_device):
    """One classification pass over the batch; returns (errors per problem, timings in ms)."""
    import torch
    qs = copies(vb, ps)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    batch = vb.BatchedVbls(Ys, qs, ctx=ctx, yhat=not on_device)
    batch.run(20, full_cov=True)
    batch.readback()
    t1 = time.perf_counter()
    LM = np.array([Y.size for Y in Ys], dtype=np.float64)
    if on_device:
        ctx.profile(True)
        t2 = time.perf_counter()
        err = batch.residual_norm() / LM
        t3 = time.perf_counter()
        prof = ctx.profile_read()
        ctx.profile(False)
        kern = prof["k1_ms"] / max(prof["k1_launches"], 1)
    else:
        t2 = time.perf_counter()
        err = np.array([np.linalg.norm(q.YHat - Y, 2) for q, Y in zip(qs, Ys)]) / LM
        t3 = time.perf_counter()
        kern = None
    return err, {"total_ms": 1e3 * (t3 - t0), "vbls_ms": 1e3 * (t1 - t0), "norm_ms": 1e3 * (t3 - t2), "norm_kernels_ms": kern}


def summary(xs):
    xs = [x for x in xs if x is not None]
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "all": xs} if xs else None


def measure(vb, ctx, name, Ys, ps, reps):
    route(vb, ctx, Ys, ps, True)                 # warm the modules and the staging arena
    route(vb, ctx, Ys, ps, False)
    runs = {"host": [], "device": []}
    errs = {}
    for _ in range(reps):
        for key, dev in (("host", False), ("device", True)):
            e, t = route(vb, ctx, Ys, ps, dev)
            runs[key].append(t)
            errs[key] = e
    out = {"problems": len(Ys), "L": int(Ys[0].shape[0]), "M_max": int(max(Y.shape[1] for Y in Ys)),
           "M_total": int(sum(Y.shape[1] for Y in Ys))}
    for key in runs:
        out[key] = {f: summary([r[f] for r in runs[key]]) for f in runs[key][0]}
    out["device"]["norm_packing_ms"] = summary([r["norm_ms"] - r["norm_kernels_ms"] for r in runs["device"]])
    a, b = errs["host"], errs["device"]
    out["max_rel_err_diff"] = float(np.max(np.abs(a - b) / np.abs(a)))
    la = np.where(a[0::2] < a[1::2], 0, 1)       # problems alternate between the two class models
    lb = np.where(b[0::2] < b[1::2], 0, 1)
    out["labels_equal"] = bool(np.array_equal(la, lb))
    out["label_1_count"] = int(la.sum())
    print(json.dumps({name: {k: out[k] for k in ("max_rel_err_diff", "labels_equal")},
                      "host_total_ms": out["host"]["total_ms"]["median"], "device_total_ms": out["device"]["total_ms"]["median"]}),
          flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("tools/batched/residual.py needs a GPU")
    import vbmf_b200_loader
    from bench import make_mil_problems
    from large_bags import card, make_batch
    vb = vbmf_b200_loader.load()
    ctx = vb.Context(device=0)
    res = {"card": card(), "host_cpus": os.cpu_count(), "H": 20, "H0": 19, "vbls_niter": 20, "full_cov": True, "reps": args.reps,
           "norm": "spectral"}
    res["c2"] = measure(vb, ctx, "c2", *make_mil_problems(vb), args.reps)
    res["musk2"] = measure(vb, ctx, "musk2", *make_batch(vb), args.reps)
    res["card_after"] = card()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
