"""Batched vbls! on Musk2-shaped bags, which do not fit the one-CTA-per-problem kernel.

Musk2 has 166 features and bags of up to 1044 instances.  The batch here is synthetic and seeded: 100 bags of 1..1044
columns at L = 166, dual parameters with H = 20, H0 = 19, full_cov, 20 iterations, against both class models, as
mil.classify_bags runs it.  The script times
  (a) the batched C-ABI call (wall clock around the call, and the kernels alone from the profiling K1 slot), once per
      column-share bound of the wide kernel in --cols (VBMF_B200_BATCHED_COLS);
  (b) the only route without the wide kernel: a vbls_ call per (bag, model);
and reports the largest relative difference between (a) and (b).  With --parent DIR it also runs
`bench.py --workload c2` alternately in DIR (a checkout of the previous build) and in this tree.  One JSON file is written
to --out.  Needs a GPU.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def make_batch(vb, nbags=100, L=166, H=20, H0=19, seed=2026):
    rng = np.random.default_rng(seed)
    B = [np.asfortranarray(rng.standard_normal((L, H))) for _ in range(2)]
    SB = [np.asfortranarray(np.diag(rng.uniform(1e-3, 1e-2, H))) for _ in range(2)]
    sizes = np.unique(np.concatenate([[1, 1044], rng.integers(1, 1045, nbags - 2)]))
    while sizes.size < nbags:
        sizes = np.unique(np.concatenate([sizes, rng.integers(1, 1045, nbags - sizes.size)]))
    Ys, ps = [], []
    for M in rng.permutation(sizes):
        Y = np.asfortranarray(10.0 * (rng.standard_normal((L, 3)) @ rng.standard_normal((3, M)) + 0.1 * rng.standard_normal((L, M))))
        for c in range(2):
            p = vb.vbmf_dual_init(Y, H, H0, rng=rng)
            p.BHat, p.SigmaB, p.sigmaHat = B[c].copy(), SB[c].copy(), 0.7
            Ys.append(Y)
            ps.append(p)
    return Ys, ps


def maxrel(qa, qb):
    worst = 0.0
    for f in ("AHat", "SigmaA", "CA", "diagSigmaATVec", "YHat", "sigmaHat", "zeta"):
        for a, b in zip(qa, qb):
            x, y = np.asarray(getattr(a, f), dtype=np.float64), np.asarray(getattr(b, f), dtype=np.float64)
            worst = max(worst, float(np.linalg.norm(x - y) / max(np.linalg.norm(y), 1e-300)))
    return worst


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--cols", default="1000000,256,128,64")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent", default=None)
    ap.add_argument("--c2-rounds", type=int, default=3)
    args = ap.parse_args()
    import torch
    import vbmf_b200_loader
    vb = vbmf_b200_loader.load()
    lib = vb._lib.load()
    niter = 20
    Ys, ps = make_batch(vb)
    Ms = np.array([Y.shape[1] for Y in Ys], dtype=np.int64)
    ctx = vb.Context(device=0)
    res = {"card": card(), "bags": len(Ys) // 2, "problems": len(Ys), "L": 166, "H": 20, "H0": 19, "niter": niter,
           "full_cov": True, "M_max": int(Ms.max()), "M_total": int(Ms.sum()), "batched": []}
    ref = None
    for cols in [int(c) for c in args.cols.split(",")]:
        os.environ["VBMF_B200_BATCHED_COLS"] = str(cols)
        cs = np.zeros(Ms.size, dtype=np.int32)
        vb._lib.check(lib.vbmf_b200_batched_plan(2, 166, 20, 1, 0, Ms.size, Ms.ctypes.data, cs.ctypes.data))
        wall, kern = [], []
        for r in range(args.reps + 1):
            qs = [vb.copy(p) for p in ps]
            batch = vb.BatchedVbls(Ys, qs, ctx=ctx, yhat=True)
            ctx.profile(True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            batch.run(niter, full_cov=True)
            t1 = time.perf_counter()
            prof = ctx.profile_read()
            ctx.profile(False)
            batch.readback()
            if r > 0:                                     # the first call warms the modules and the arena
                wall.append(1e3 * (t1 - t0))
                kern.append(prof["k1_ms"] / max(prof["k1_launches"], 1))
        if ref is None:
            ref = qs
        res["batched"].append({"cols_per_cta": cols, "clusters": {str(c): int(np.sum(cs == c)) for c in (0, 1, 2, 4, 8)},
                               "call_ms": float(np.median(wall)), "call_ms_all": wall, "kernels_ms": float(np.median(kern)),
                               "max_rel_vs_first": maxrel(qs, ref)})
        print(json.dumps(res["batched"][-1]), flush=True)
    os.environ.pop("VBMF_B200_BATCHED_COLS")
    # (b) a vbls_ call per problem
    loop = [vb.copy(p) for p in ps]
    vb.vbls_(Ys[0], vb.copy(ps[0]), niter, full_cov=True, ctx=ctx)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for Y, q in zip(Ys, loop):
        vb.vbls_(Y, q, niter, full_cov=True, ctx=ctx)
    torch.cuda.synchronize()
    res["loop_ms"] = 1e3 * (time.perf_counter() - t0)
    res["max_rel_batched_vs_loop"] = maxrel(ref, loop)
    print(json.dumps({"loop_ms": res["loop_ms"], "max_rel_batched_vs_loop": res["max_rel_batched_vs_loop"]}), flush=True)
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
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
