"""Cost of labels in batched vbls!, and a bitwise check that unlabelled inputs compute what a previous build computes.

Timing (one JSON file to --out, needs a GPU): the Musk2-shaped bag sizes of tools/batched/large_bags.py (100 bags of 1..1044
columns at L = 166, two class models each, H = 20, 20 iterations) as sparse full_cov and as dense problems, each run
alternately without labels and with H1 = 1 and every fourth column of every bag labelled.  Reported per variant: the
kernels alone (the profiling K1 slot, CUDA events) and the wall clock of the C-ABI call, medians over --reps calls after one
warm-up call.  With --parent DIR (a built checkout of the previous version) it also runs `bench.py --workload c2`
alternately in DIR and in this tree, and has both builds dump the outputs of unlabelled batches (the c2 problems, the
sparse and dense Musk2-shaped ones, all with a diagonal invCA) and compares them field by field with np.array_equal.

  python tools/batched/labels.py --out labels.json [--parent DIR]
  python tools/batched/labels.py --dump DIR [--root TREE]      (used by --parent: outputs of TREE's build as .npy files)
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "tools", "batched"))

L, H, NITER = 166, 20, 20


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def musk2_batch(vb, kind, labelled):
    """The bags and class models of large_bags.make_batch as `kind` parameters; labelled: H1 = 1 and columns 1, 5, 9, ..."""
    import large_bags
    Ys, duals = large_bags.make_batch(vb)
    rng = np.random.default_rng(7)
    ps = []
    for Y, d in zip(Ys, duals):
        M = Y.shape[1]
        lab = list(range(1, M + 1, 4)) if labelled else None
        if kind == "sparse":
            p = vb.vbmf_sparse_init(Y, H, H1=1 if labelled else 0, labels=lab, rng=rng)
            p.sigmaHat = d.sigmaHat
        else:
            p = vb.vbmf_init(Y, H, sigma2=0.9, H1=1 if labelled else 0, labels=lab, rng=rng)
        p.BHat, p.SigmaB = d.BHat.copy(), d.SigmaB.copy()
        ps.append(p)
    return Ys, ps


def time_variant(vb, ctx, Ys, ps, reps, full_cov):
    import torch
    wall, kern = [], []
    for r in range(reps + 1):
        qs = [vb.copy(p) for p in ps]
        batch = vb.BatchedVbls(Ys, qs, ctx=ctx, yhat=True)
        ctx.profile(True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        batch.run(NITER, full_cov=full_cov)
        t1 = time.perf_counter()
        prof = ctx.profile_read()
        ctx.profile(False)
        batch.readback()
        if r > 0:                                         # the first call warms the modules and the arena
            wall.append(1e3 * (t1 - t0))
            kern.append(prof["k1_ms"] / max(prof["k1_launches"], 1))
    return wall, kern


DUMP_FIELDS = {"dual": ["AHat", "ATVecHat", "diagSigmaATVec", "SigmaA", "CA", "beta", "sigmaHat", "zeta", "YHat", "A0Hat", "A1Hat",
                        "CA0", "CA1", "beta0", "beta1", "alpha0", "alpha1"],
               "sparse": ["AHat", "ATVecHat", "diagSigmaATVec", "SigmaA", "CA", "beta", "sigmaHat", "zeta", "YHat", "sigmaVecHat",
                          "zetaVec", "SigmaATVec_blocks"],
               "dense": ["AHat", "SigmaA", "CA", "invCA", "sigma2", "YHat"]}


def dump(out):
    import vbmf_b200_loader
    vb = vbmf_b200_loader.load()
    sys.path.append(ROOT)
    import bench
    ctx = vb.Context(device=0)
    os.makedirs(out, exist_ok=True)
    runs = [("c2_dual", "dual", bench.make_mil_problems(vb), dict(full_cov=True)),
            ("musk2_sparse_fullcov_diagvar", "sparse", musk2_batch(vb, "sparse", False), dict(full_cov=True, diag_var=True)),
            ("musk2_sparse_diag", "sparse", musk2_batch(vb, "sparse", False), dict()),
            ("musk2_dense", "dense", musk2_batch(vb, "dense", False), dict())]
    for name, kind, (Ys, ps), kw in runs:
        qs = [vb.copy(p) for p in ps]
        vb.vbls_batched_(Ys, qs, NITER, ctx=ctx, yhat=True, keep_blocks=kw.get("full_cov", False) and kind == "sparse", **kw)
        for f in DUMP_FIELDS[kind]:
            if kind == "sparse" and f == "SigmaATVec_blocks" and not kw.get("full_cov"):
                continue
            np.save(os.path.join(out, "%s.%s.npy" % (name, f)),
                    np.concatenate([np.asarray(getattr(q, f), dtype=np.float64).reshape(-1) for q in qs]))
    ctx.close()


def compare(a, b):
    names = sorted(n for n in os.listdir(a) if n.endswith(".npy"))
    res = {"files": len(names), "identical": [], "different": []}
    if sorted(n for n in os.listdir(b) if n.endswith(".npy")) != names:
        res["different"].append("file lists differ")
    for n in names:
        if os.path.exists(os.path.join(b, n)):
            same = np.array_equal(np.load(os.path.join(a, n)), np.load(os.path.join(b, n)), equal_nan=True)
            res["identical" if same else "different"].append(n[:-4])
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--dump")
    ap.add_argument("--root", default=ROOT, help="with --dump: the tree whose build to load")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent", default=None)
    ap.add_argument("--c2-rounds", type=int, default=3)
    args = ap.parse_args()
    if args.dump:
        sys.path.insert(0, os.path.abspath(args.root))
        dump(args.dump)
        return
    if not args.out:
        ap.error("--out or --dump is required")
    sys.path.insert(0, ROOT)
    import vbmf_b200_loader
    vb = vbmf_b200_loader.load()
    ctx = vb.Context(device=0)
    res = {"card": card(), "bags": 100, "problems": 200, "L": L, "H": H, "niter": NITER,
           "labels": "H1 = 1, columns 1, 5, 9, ... of every bag (about a quarter of them)", "variants": {}}
    for kind, full_cov in (("sparse", True), ("dense", False)):
        batches = {lab: musk2_batch(vb, kind, lab) for lab in (False, True)}
        acc = {False: ([], []), True: ([], [])}
        for _ in range(2):                                # alternate the two variants
            for lab in (False, True):
                w, k = time_variant(vb, ctx, *batches[lab], args.reps, full_cov)
                acc[lab][0].extend(w)
                acc[lab][1].extend(k)
        v = {}
        for lab in (False, True):
            w, k = acc[lab]
            v["labelled" if lab else "unlabelled"] = {"call_ms": float(np.median(w)), "kernels_ms": float(np.median(k)),
                                                      "call_ms_all": w, "kernels_ms_all": k}
        v["kernel_cost_of_labels_pct"] = 100.0 * (v["labelled"]["kernels_ms"] / v["unlabelled"]["kernels_ms"] - 1.0)
        v["call_cost_of_labels_pct"] = 100.0 * (v["labelled"]["call_ms"] / v["unlabelled"]["call_ms"] - 1.0)
        res["variants"]["musk2_%s%s" % (kind, "_fullcov" if full_cov else "")] = v
        print(json.dumps({kind: {k: (x if not isinstance(x, dict) else {a: b for a, b in x.items() if not a.endswith("_all")})
                                 for k, x in v.items()}}), flush=True)
    ctx.close()
    if args.parent:
        runs = []
        cmd = [sys.executable, "bench.py", "--gpus", "1", "--workload", "c2", "--steps", "20", "--warmup", "3", "--no-cpu"]
        for i in range(args.c2_rounds):
            for name, cwd in (("parent", args.parent), ("this", ROOT)):
                r = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True)
                line = [x for x in r.stdout.splitlines() if x.startswith("{")]
                rec = json.loads(line[-1]) if line else {"error": r.stderr[-2000:]}
                runs.append({"build": name, "round": i, "problems_per_s": rec.get("value"), "ms_per_step": rec.get("ms_per_step"),
                             "kernel_ms": (rec.get("roofline") or {}).get("kernel_ms"), "error": rec.get("error")})
                print(json.dumps(runs[-1]), flush=True)
        res["c2_alternated"] = runs
        with tempfile.TemporaryDirectory() as tmp:
            dirs = {}
            for name, tree in (("parent", args.parent), ("this", ROOT)):
                dirs[name] = os.path.join(tmp, name)
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--dump", dirs[name], "--root", tree],
                                   capture_output=True, text=True)
                if r.returncode != 0:
                    res["dump_error_" + name] = r.stderr[-2000:]
            if all(os.path.isdir(d) for d in dirs.values()):
                res["unlabelled_outputs_vs_parent"] = compare(dirs["parent"], dirs["this"])
                print(json.dumps({"unlabelled_outputs_vs_parent": res["unlabelled_outputs_vs_parent"]}), flush=True)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
