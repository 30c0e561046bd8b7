"""Batched lowerBound / lowerBoundTrimmed on the Musk2-shaped batch of tools/batched/large_bags.py.

The batch is the seeded one of large_bags.py: 100 bags of 1..1044 columns at L = 166, dual parameters with H = 20, H0 = 19,
against both class models (200 problems).  Batched vbls! runs first (20 iterations, full_cov), as mil.classify_bags does, and
the script then times
  (a) BatchedVbls.lower_bound() and .lower_bound(0.1) on the structs the vbls call left: wall clock around the C-ABI call and
      the kernels alone (profiling K1 slot);
  (b) the per-problem route: lowerBound / lowerBoundTrimmed once per problem (attach Y, create a solver, upload, three
      kernels, tear down);
and reports the largest relative difference between (a) and (b).  With --parent DIR (a checkout of the previous build, its
library built) it also computes single-solver lowerBound / lowerBoundTrimmed values on seeded sparse, dual and trial states
with the library of DIR and with this tree's, each in a process of its own, and reports whether they are bit-identical.
One JSON file is written to --out.  Needs a GPU.
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
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools", "batched"))


def seeded_states(vb, seed=7):
    """Sparse, dual and trial states straight from the initialisers (host RNG), with non-trivial SigmaB / noise scalars."""
    rng = np.random.default_rng(seed)
    out = []
    for kind, L, M, H in (("sparse", 40, 33, 5), ("sparse", 166, 700, 20), ("dual", 166, 1044, 20), ("dual", 38, 200, 64),
                          ("trial", 60, 90, 7), ("trial", 166, 300, 20)):
        Y = np.asfortranarray(10.0 * (rng.standard_normal((L, 3)) @ rng.standard_normal((3, M)) + 0.1 * rng.standard_normal((L, M))))
        if kind == "sparse":
            p = vb.vbmf_sparse_init(Y, H, rng=rng)
        elif kind == "dual":
            p = vb.vbmf_dual_init(Y, H, H - 1, rng=rng)
        else:
            p = vb.vbmf_trial_init(Y, H, H - 2, M // 3, rng=rng)
        p.SigmaB = np.asfortranarray(np.diag(rng.uniform(1e-3, 1e-2, H)))
        p.sigmaHat = 0.7
        out.append((Y, p))
    return out


def single_values(tree, out_path):
    """lowerBound and lowerBoundTrimmed(0.1) of seeded_states with the package and library of `tree` (float.hex strings)."""
    sys.path.insert(0, tree)
    import vbmf_b200_loader
    assert os.path.dirname(os.path.abspath(vbmf_b200_loader.__file__)) == os.path.abspath(tree)
    vb = vbmf_b200_loader.load()
    ctx = vb.Context(device=0)
    vals = []
    for Y, p in seeded_states(vb):
        vals.append([vb.lowerBound(Y, p, ctx=ctx).hex(), vb.lowerBoundTrimmed(Y, p, 0.1, ctx=ctx).hex()])
    ctx.close()
    with open(out_path, "w") as f:
        json.dump(vals, f)


def maxrel(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent", default=None)
    ap.add_argument("--single-values", nargs=2, metavar=("TREE", "OUT"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.single_values:
        single_values(*args.single_values)
        return
    import torch
    import vbmf_b200_loader
    from large_bags import card, make_batch
    vb = vbmf_b200_loader.load()
    niter = 20
    Ys, ps = make_batch(vb)
    Ms = np.array([Y.shape[1] for Y in Ys], dtype=np.int64)
    ctx = vb.Context(device=0)
    res = {"card": card(), "bags": len(Ys) // 2, "problems": len(Ys), "L": 166, "H": 20, "H0": 19, "vbls_niter": niter,
           "full_cov": True, "M_max": int(Ms.max()), "M_total": int(Ms.sum())}
    batch = vb.BatchedVbls(Ys, ps, ctx=ctx, yhat=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    batch.run(niter, full_cov=True)
    res["vbls_call_ms"] = 1e3 * (time.perf_counter() - t0)
    batch.readback()
    # (a) the batched call, untrimmed and trimmed
    for name, trim in (("lower_bound", None), ("lower_bound_trimmed", 0.1)):
        wall, kern = [], []
        for r in range(args.reps + 1):
            ctx.profile(True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            v = batch.lower_bound(trim)
            t1 = time.perf_counter()
            prof = ctx.profile_read()
            ctx.profile(False)
            if r > 0:                                     # the first call warms the modules and the arena
                wall.append(1e3 * (t1 - t0))
                kern.append(prof["k1_ms"] / max(prof["k1_launches"], 1))
        res[name] = {"call_ms": float(np.median(wall)), "call_ms_all": wall, "kernels_ms": float(np.median(kern)),
                     "finite": bool(np.isfinite(v).all())}
        res[name + "_values"] = v
        print(json.dumps(res[name]), flush=True)
    # (b) one lowerBound call per problem
    for name, fn in (("lower_bound", lambda Y, p: vb.lowerBound(Y, p, ctx=ctx)),
                     ("lower_bound_trimmed", lambda Y, p: vb.lowerBoundTrimmed(Y, p, 0.1, ctx=ctx))):
        fn(Ys[0], ps[0])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loop = np.array([fn(Y, p) for Y, p in zip(Ys, ps)])
        torch.cuda.synchronize()
        res[name]["per_problem_route_ms"] = 1e3 * (time.perf_counter() - t0)
        res[name]["max_rel_batched_vs_per_problem"] = maxrel(res.pop(name + "_values"), loop)
        print(json.dumps({name: res[name]}), flush=True)
    ctx.close()
    if args.parent:
        vals = {}
        with tempfile.TemporaryDirectory() as tmp:
            for name, tree in (("parent", os.path.abspath(args.parent)), ("this", ROOT)):
                path = os.path.join(tmp, name + ".json")
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--single-values", tree, path],
                                   capture_output=True, text=True)
                if r.returncode != 0:
                    raise RuntimeError("single-solver values with %s failed:\n%s" % (tree, r.stderr[-3000:]))
                vals[name] = json.load(open(path))
        res["single_solver_parent"] = vals["parent"]
        res["single_solver_this"] = vals["this"]
        res["single_solver_bit_identical"] = vals["parent"] == vals["this"]
        print(json.dumps({"single_solver_bit_identical": res["single_solver_bit_identical"]}), flush=True)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
