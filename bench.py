#!/usr/bin/env python
"""bench.py -- VB iterations/s of the dense `vbmf` update loop on synthetic low-rank-plus-noise Y (BASELINE.json configs[2]).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference --gpus 1 --steps K --warmup W      # CPU arm: the oracle restatement on the host cores

One step = one VB iteration (updateA!, updateB!, updateCA!, updateCB!, updateSigma2!, delta; src/vbmf.jl:193-214) over the
resident column shard of Y.  Y is column-sharded across ranks (fixed total problem => strong scaling); the per-iteration
exchange of [Y*AHat | AHat'AHat | ...] runs through peer-mapped memory over NVLink with the library's own kernels (reduce-scatter
of Y*AHat, row-sharded BHat epilogue, all-gather of BHat; world <= 8, H <= 64) or, with VBMF_B200_NO_PX=1 / outside those
limits, as one packed NCCL all-reduce.

Timed region: W untimed warm-up iterations, then exactly K iterations between barrier + synchronize, CUDA events on the
stream the kernels run on, max over ranks.  Y (32 GB at N=1) is far larger than L2, so no explicit L2 flush is needed.
`value` has Y resident in HBM; `e2e` is the same metric through the public API (`vbmf_`) with every input in pinned HOST
memory: upload of Y and of the parameter struct, K iterations, download of the results.
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

WORKLOADS = {
    # name: (L, M, H, kind, flags, description)
    "c3": (20000, 200000, 64, "dense", ("est_covs", "est_var"),
           "configs[2]: synthetic dense Y 20000x200000, rank-32 signal + 0.1 noise, vbmf H=64 with ARD (est_covs, est_var), Float64"),
    # diagnostic only: the per-GPU shard of c3 at 8 GPUs on ONE GPU (no exchange), to separate kernel time from exchange time
    "c3shard8": (20000, 25000, 64, "dense", ("est_covs", "est_var"), "diagnostic: one 25000-column shard of configs[2] (what each of 8 GPUs computes)"),
    # diagnostic only: a quarter of c3's columns; on 2 GPUs every rank holds the 25000-column shard of the 8-GPU run, exchange included
    "c3quarter": (20000, 50000, 64, "dense", ("est_covs", "est_var"), "diagnostic: 50000 columns of configs[2] (25000 per GPU on 2 GPUs)"),
    "c4": (10000, 100000, 32, "sparse", ("est_cb",), "configs[3] (diagonal covariance path): vbmf_sparse 10000x100000 H=32"),
    "c4full": (10000, 100000, 32, "sparse", ("est_cb", "full_cov"), "configs[3]: vbmf_sparse 10000x100000 H=32 full_cov (batched per-row Cholesky)"),
    # configs[4] needs >= 4 GPUs at full size (Y = 400 GB); per SURVEY 8(d) fewer GPUs run M = 125000 columns per GPU
    "c5": (50000, 125000, 128, "dual", ("est_cb", "est_priors"), "configs[4] scaled to 125000 columns per GPU: vbmf_dual 50000x(125000*n)x128, H0=64, diagonal covariance, est_priors"),
}
FP64_PEAK_TFLOPS = 37.0   # measured DMMA issue-rate peak on this pool's B200 (profiles/r01_fp64_peak_microbench.jsonl)
SEED = 20260101
DUMP_BYTES = 60 << 20     # --dump-outputs stays below 64 MB in all (npy headers included)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], None, set(), []
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                clk, mx = float(f[0]), float(f[1])
            except ValueError:
                continue
            smax = mx
            if t0 - 0.05 <= ts <= t1 + 0.05:
                sm.append(clk)
                try:
                    power.append(float(f[2]))
                except ValueError:
                    pass
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        if not sm:   # region shorter than the sampling period: fall back to every sample taken
            for ts, line in self.lines:
                try:
                    sm.append(float(line.split(",")[0]))
                except ValueError:
                    pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# fields indexed by column m of Y: (M, w) matrices and (M*w,) vectors of per-column blocks of w entries
COLUMN_FIELDS = {
    "dense": ("AHat",),
    "sparse": ("AHat", "ATVecHat", "diagSigmaATVec", "CA", "beta"),
    "dual": ("AHat", "ATVecHat", "diagSigmaATVec", "CA", "beta", "A0Hat", "A1Hat", "CA0", "CA1", "beta0", "beta1"),
}


def dump_outputs(out_dir, p, delta, kind):
    """--dump-outputs: every floating-point field of the parameter struct the timed loop hands back, plus its final convergence
    delta, as float64 DIR/<field>.npy (DIR/final_delta.npy for the delta).  The COLUMN_FIELDS of `kind` keep the same fixed,
    seeded subset of columns, as many as DUMP_BYTES allows, so that two builds run with the same arguments can be compared
    output for output."""
    M = p.M
    fields = {n: np.asarray(v, dtype=np.float64) for n, v in vars(p).items()
              if v is not None and np.asarray(v).dtype.kind == "f"}
    fields["final_delta"] = np.asarray(delta, dtype=np.float64)
    cols = COLUMN_FIELDS[kind]
    fixed = sum(a.nbytes for n, a in fields.items() if n not in cols)
    per_col = sum(fields[n].nbytes for n in cols) // M
    k = min(M, (DUMP_BYTES - fixed) // per_col)
    if k < 1:
        raise SystemExit("--dump-outputs: the outputs not indexed by column alone exceed %d bytes" % DUMP_BYTES)
    if k < M:
        idx = np.sort(np.random.default_rng(SEED).choice(M, k, replace=False))
        for n in cols:
            fields[n] = fields[n][idx] if fields[n].ndim == 2 else fields[n].reshape(M, -1)[idx].reshape(-1)
    os.makedirs(out_dir, exist_ok=True)
    for n, a in fields.items():
        np.save(os.path.join(out_dir, n + ".npy"), a)


# ------------------------------------------------------------------------------------------------ CPU arm (oracle)
def cpu_reference(L, M, H, kind, flags, steps, warmup, budget_s):
    """The oracle restatement timed on the host cores on a bounded column sample of the workload (same L and H,
    M_s << M columns; one VB iteration is linear in M, so full-size iterations/s = sample iterations/s * M_s/M)."""
    from oracle import vbmf_oracle as vo
    cores = os.cpu_count() or 1
    try:        # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=cores)
    except Exception:
        pass
    # size the sample from a measured GEMM rate so the whole run fits the budget
    n = 1024
    a = np.random.default_rng(0).standard_normal((n, n))
    t = time.perf_counter(); a @ a; a @ a; rate = 4.0 * n ** 3 / (time.perf_counter() - t)
    per_col = 4.0 * L * H * 1.15
    Ms = int(budget_s * rate / (per_col * max(steps + warmup, 1)))
    Ms = max(256, min(M // 10, (Ms // 256) * 256))
    rng = np.random.default_rng(SEED)
    r = H // 2
    Y = rng.standard_normal((L, r)) @ rng.standard_normal((r, Ms)) + 0.1 * rng.standard_normal((L, Ms))
    if kind == "dense":
        p = vo.vbmf_init(Y, H, rng=np.random.default_rng(SEED + 1))
        step = lambda: vo.vbmf_run(Y, p, 1, eps=0.0, est_covs="est_covs" in flags, est_var="est_var" in flags)
    elif kind == "sparse":
        p = vo.vbmf_sparse_init(Y, H, rng=np.random.default_rng(SEED + 1))
        step = lambda: vo.vbmf_sparse_run(Y, p, 1, eps=0.0, full_cov="full_cov" in flags, est_cb="est_cb" in flags)
    else:
        p = vo.vbmf_dual_init(Y, H, H // 2, rng=np.random.default_rng(SEED + 1))
        step = lambda: vo.vbmf_dual_run(Y, p, 1, eps=0.0, full_cov="full_cov" in flags, est_cb="est_cb" in flags,
                                        est_priors="est_priors" in flags)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    sample_its = steps / dt
    return {"value": sample_its * Ms / M, "unit": "iterations/s", "cores": cores, "kind": "port",
            "sample": "oracle (NumPy/OpenBLAS restatement of src/vbmf*.jl) on L=%d x M_s=%d of the %d columns, H=%d, %d timed iterations: "
                      "%.3f it/s on the sample, scaled by M_s/M (an iteration is linear in M)" % (L, Ms, M, H, steps, sample_its),
            "sample_iterations_per_s": sample_its, "sample_ms_per_iteration": dt / steps * 1e3}


def run_reference(args, L, M, H, kind, flags, desc):
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    cb = cpu_reference(L, M, H, kind, flags, args.steps, args.warmup, budget_s=float(os.environ.get("VBMF_BENCH_CPU_BUDGET_S", 150.0)))
    line = {"impl": "reference", "metric": "VB iterations/s at %dx%dx%d (dense vbmf, Float64)" % (L, M, H) if kind == "dense" else
            "VB iterations/s at %dx%dx%d (%s, Float64)" % (L, M, H, kind),
            "value": cb["value"], "unit": "iterations/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 / cb["value"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "extrapolated": True,
            "config": {"workload": desc, "parallelism": "host cores only",
                       "sample": "timed on L=%d x M_s columns (M_s << M=%d, see cpu_baseline.sample) and scaled by M_s/M: one iteration is "
                                 "linear in M; the full-size CPU iteration would take ~%.0f s" % (L, M, 1.0 / cb["value"])},
            "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ config 2: batched MIL-like problems
def make_mil_problems(vbmod, nbags=548, L=38, H=20, seed=SEED):
    """Synthetic stand-in for the MIL bags (the real .jld datasets are not in the reference repo, examples/mil_data.jl:97):
    548 bags, 38 features, 5-40 instances per bag, two class models (BHat, SigmaB), H = 20, H1 = 1, scale = 10."""
    rng = np.random.default_rng(seed)
    B = [np.asfortranarray(rng.standard_normal((L, H))) for _ in range(2)]
    SB = [np.asfortranarray(np.diag(rng.uniform(1e-3, 1e-2, H))) for _ in range(2)]
    Ys, ps = [], []
    for _ in range(nbags):
        M = int(rng.integers(5, 41))
        Y = np.asfortranarray(10.0 * (rng.standard_normal((L, 3)) @ rng.standard_normal((3, M)) + 0.1 * rng.standard_normal((L, M))))
        for c in range(2):
            p = vbmod.vbmf_dual_init(Y, H, H - 1, rng=rng)
            p.BHat, p.SigmaB, p.sigmaHat = B[c].copy(), SB[c].copy(), 0.7
            Ys.append(Y)
            ps.append(p)
    return Ys, ps


def run_c2(args):
    """`--workload c2`: classify(...; class_alg="dual") pattern = vbls!(Y, params, 20, full_cov=true) on every bag x class
    model (examples/mil_util.jl:504-511), all 1096 problems in one launch of the one-CTA-per-problem kernel."""
    import torch
    import vbmf_b200_loader
    vb = vbmf_b200_loader.load()
    lib = vb._lib.load()
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    ctx = vb.Context(device=0, stream=stream.cuda_stream)
    niter = 20
    Ys, ps = make_mil_problems(vb)
    n = len(ps)
    for _ in range(max(args.warmup, 3)):
        vb.vbls_batched_(Ys, [vb.copy(p) for p in ps], niter, full_cov=True, ctx=ctx, yhat=True)
    sampler = ClockSampler(0); sampler.start(); time.sleep(0.1)
    dev_ms, wall, marshal = [], [], []
    ctx.profile(True)
    n0 = lib.vbmf_b200_launch_count()
    t_start = time.time()
    for _ in range(args.steps):
        qs = [vb.copy(p) for p in ps]                   # fresh parameter objects: every step starts from the same state
        m0 = time.perf_counter()
        batch = vb.BatchedVbls(Ys, qs, ctx=ctx, yhat=True)     # Python-only: ctypes structs + pointer tables
        marshal.append(time.perf_counter() - m0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.perf_counter()
        e0.record(stream)
        batch.run(niter, full_cov=True)                 # the C-ABI call: host arrays in, host arrays out
        e1.record(stream)
        torch.cuda.synchronize()
        batch.readback()
        wall.append(time.perf_counter() - w0)
        dev_ms.append(e0.elapsed_time(e1))
    t_end = time.time()
    launches = lib.vbmf_b200_launch_count() - n0
    prof = ctx.profile_read()
    kernel_ms = prof["k1_ms"] / max(prof["k1_launches"], 1)
    clocks = sampler.stop(t_start, t_end)
    ms = float(np.mean(dev_ms))
    cpu = None
    if not args.no_cpu:
        from oracle import vbmf_oracle as vo
        rngc = np.random.default_rng(SEED)
        k = 24
        t0 = time.perf_counter()
        for Y, p in zip(Ys[:k], ps[:k]):
            po = vo.vbmf_dual_init(np.ascontiguousarray(Y), p.H, p.H0, rng=rngc)
            po.BHat, po.SigmaB, po.sigmaHat = np.array(p.BHat), np.array(p.SigmaB), p.sigmaHat
            vo.vbls(np.ascontiguousarray(Y), po, niter, full_cov=True)
        dt = time.perf_counter() - t0
        cpu = {"value": k / dt, "unit": "problems/s", "cores": os.cpu_count(), "kind": "port",
               "sample": "oracle vbls (20 iterations, full_cov) on the first %d of the %d problems" % (k, n)}
    Mtot = sum(Y.shape[1] for Y in Ys)
    line = {"metric": "vbls! problems/s (MIL pattern: 548 bags x 2 class models, L=38, M=5..40, H=20, 20 iterations, full_cov)",
            "value": n / (ms * 1e-3), "unit": "problems/s", "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[1] stand-in: synthetic MIL bags (real datasets are not in the reference repo), vbmf_dual "
                                   "parameters, one CTA per problem", "problems": n, "l2": "working set (%.1f MB) fits L2; each step re-uploads "
                                   "every input from the host" % (Mtot * 38 * 8 / 1e6)},
            "roofline": {"bound": "latency", "kernel": "batched_vbls_kernel", "kernel_ms": kernel_ms, "kernel_problems_per_s": n / (kernel_ms * 1e-3),
                         "note": "one CTA per problem, state in shared memory/registers for all 20 iterations; `value` brackets the whole C-ABI "
                                 "call with CUDA events (host packing into pinned staging + upload + kernel + download + unpack), "
                                 "kernel_ms is the kernel alone", "python_marshal_ms": 1e3 * float(np.mean(marshal))},
            "cpu_baseline": cpu,
            "e2e": {"value": n / float(np.mean(wall)), "unit": "problems/s", "h2d_bytes_per_step": int(Mtot * 38 * 8 + n * (38 * 20 + 400) * 8 + Mtot * 20 * 8),
                    "d2h_bytes_per_step": int(Mtot * 20 * 8 * 4 + Mtot * 38 * 8), "note": "wall clock of the C-ABI call on host arrays plus the scalar read-back; building the 1096 ctypes structs (python_marshal_ms, a Python-binding cost a Julia ccall does not have) is reported separately"},
            "gpu_launches": int(launches), "clocks": clocks}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ one process, N devices
def run_single_process(args, L, M, H, kind, flags, desc):
    """The same workload through vbmf_b200_mctx_* (one host process, one host thread per GPU inside the library): what a Julia
    caller gets from b200_context(0:N-1).  Each step is one whole-loop call on FULL-SIZE host parameter arrays (scatter of
    AHat to the devices, K iterations, gather), Y resident; timed by the wall clock of the call."""
    import vbmf_b200_loader
    vb = vbmf_b200_loader.load()
    lib = vb._lib.load()
    mc = vb.MultiContext(devices=list(range(args.gpus)))
    mc.synth(L, M, rank=H // 2, noise=0.1, seed=SEED)

    class Shape:
        shape = (L, M)
    rng = np.random.default_rng(SEED + 1)
    if kind == "dense":
        p = vb.vbmf_init(Shape, H, rng=rng)
        call = lambda n: vb.vbmf_(None, p, n, eps=0.0, est_covs="est_covs" in flags, est_var="est_var" in flags, ctx=mc, yhat=False)
    elif kind == "sparse":
        p = vb.vbmf_sparse_init(Shape, H, rng=rng, trYTY=mc.trYTY())
        call = lambda n: vb.vbmf_sparse_(None, p, n, eps=0.0, full_cov="full_cov" in flags, est_cb="est_cb" in flags, ctx=mc, yhat=False)
    else:
        p = vb.vbmf_dual_init(Shape, H, H // 2, rng=rng, trYTY=mc.trYTY())
        call = lambda n: vb.vbmf_dual_(None, p, n, eps=0.0, full_cov="full_cov" in flags, est_cb="est_cb" in flags,
                                       est_priors="est_priors" in flags, ctx=mc, yhat=False)
    call(args.warmup)
    sampler = ClockSampler(0); sampler.start(); time.sleep(0.15)
    n0 = lib.vbmf_b200_launch_count()
    t0 = time.time()
    w0 = time.perf_counter()
    call(args.steps)
    w = time.perf_counter() - w0
    t1 = time.time()
    launches = lib.vbmf_b200_launch_count() - n0
    clocks = sampler.stop(t0, t1)
    state_check = {"iterations": args.warmup + args.steps, "norm_BHat_fro": float(np.linalg.norm(p.BHat)),
                   "norm_AHat_fro": float(np.linalg.norm(p.AHat)), "trace_SigmaB": float(np.trace(p.SigmaB)),
                   "trace_SigmaA": float(np.trace(p.SigmaA)), "noise": float(p.sigma2) if kind == "dense" else float(p.sigmaHat)}
    line = {"metric": "VB iterations/s at %dx%dx%d (%s, Float64)" % (L, M, H, "dense vbmf" if kind == "dense" else "vbmf_" + kind),
            "mode": "single_process", "value": args.steps / w, "unit": "iterations/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": w / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": desc, "global_shape": [L, M, H], "parallelism": "ONE host process, %d devices: vbmf_b200_mctx_* (ncclCommInitAll, "
                       "one host thread per device inside the library)" % args.gpus,
                       "timing": "wall clock of one whole-loop call on full-size host parameter arrays: scatter of AHat, %d iterations, gather; "
                                 "Y resident" % args.steps},
            "iteration_frac_of_peak": 4.0 * L * M * H / (w / args.steps) / (args.gpus * FP64_PEAK_TFLOPS * 1e12),
            "gpu_launches": int(launches), "clocks": clocks, "state_check": state_check}
    print(json.dumps(line), flush=True)
    mc.close()


# ------------------------------------------------------------------------------------------------ our arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS) + ["c2"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--single-process", action="store_true",
                    help="drive --gpus N devices from THIS process through the multi-device context (vbmf_b200_mctx_*), the path a "
                         "one-process Julia caller uses; no torchrun")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--segments", action="store_true",
                    help="diagnosis: CUDA events between the launches of every iteration (adds stream bubbles; not for headline numbers)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed iterations, write the state they leave (rank 0's column shard when N > 1) as DIR/<field>.npy, "
                         "float64, under 64 MB in all; column-indexed fields keep a fixed, seeded sample of the columns.  Not available "
                         "with --workload c2, --single-process or --impl reference")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.single_process or args.workload == "c2"):
        ap.error("--dump-outputs covers the resident-Y timed loop only (--impl ours, no --single-process, not --workload c2)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 0)
    if args.workload == "c2":
        if args.impl == "ours":
            run_c2(args)
        return
    L, M, H, kind, flags, desc = WORKLOADS[args.workload]
    if args.workload == "c5":
        M = M * max(1, env_int("WORLD_SIZE", 1))        # weak-scaled columns (the full 1e6 at 8 GPUs)

    if args.impl == "reference":
        run_reference(args, L, M, H, kind, flags, desc)
        return
    if args.single_process:
        run_single_process(args, L, M, H, kind, flags, desc)
        return

    import torch
    import vbmf_b200_loader
    vb = vbmf_b200_loader.load()          # fails loudly if libvbmf_b200.so is missing: no CPU fallback
    lib = vb._lib.load()

    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local_rank = env_int("LOCAL_RANK", 0)
    if args.gpus > 1 and world != args.gpus:
        raise SystemExit("--gpus %d needs torchrun with --nproc-per-node %d (WORLD_SIZE=%d)" % (args.gpus, args.gpus, world))
    torch.cuda.set_device(local_rank)
    dist = None
    nccl_id = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(vb.Context.nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        nccl_id = bytes(idt.cpu().numpy().tobytes())

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    stream = torch.cuda.Stream()
    ctx = vb.Context(device=local_rank, rank=rank, world=world, nccl_id=nccl_id, stream=stream.cuda_stream)
    off, Mloc = vb.shard_columns(M, world, rank)
    ctx.synth(L, Mloc, M_global=M, col_offset=off, rank=H // 2, noise=0.1, seed=SEED)

    class Shape:           # the init functions only read Y.shape
        shape = (L, M)
    rng = np.random.default_rng(SEED + 1)
    if kind == "dense":
        pg = vb.vbmf_init(Shape, H, rng=rng)
        fl = (vb._lib.EST_COVS if "est_covs" in flags else 0) | (vb._lib.EST_VAR if "est_var" in flags else 0)
    elif kind == "sparse":
        pg = vb.vbmf_sparse_init(Shape, H, rng=rng, trYTY=ctx.trYTY())
        fl = (vb._lib.EST_CB if "est_cb" in flags else 0) | (vb._lib.FULL_COV if "full_cov" in flags else 0)
    else:
        pg = vb.vbmf_dual_init(Shape, H, H // 2, rng=rng, trYTY=ctx.trYTY())
        fl = (vb._lib.EST_CB if "est_cb" in flags else 0) | (vb._lib.FULL_COV if "full_cov" in flags else 0) | \
             (vb._lib.EST_PRIORS if "est_priors" in flags else 0)

    def local_params():
        p = vb.copy(pg)
        p.M = Mloc
        p.AHat = np.asfortranarray(pg.AHat[off:off + Mloc])
        if kind != "dense":
            p.MH = Mloc * H
            sl = slice(off * H, (off + Mloc) * H)
            for f in ("ATVecHat", "diagSigmaATVec", "CA", "beta"):
                setattr(p, f, getattr(pg, f)[sl].copy())
        if kind == "dual":
            p.A0Hat = np.asfortranarray(p.AHat[:, :p.H0]); p.A1Hat = np.asfortranarray(p.AHat[:, p.H0:])
            for f, w in (("CA0", p.H0), ("beta0", p.H0), ("CA1", p.H1), ("beta1", p.H1)):
                setattr(p, f, getattr(pg, f)[off * w:(off + Mloc) * w].copy())
        return p

    p = local_params()
    solver = vb.Solver(ctx, p)
    solver.upload(p)
    it, d = solver.run(args.warmup, eps=0.0, flags=fl)
    assert it == args.warmup, "warm-up ended early (it=%d, d=%r)" % (it, d)

    # ---- timed region: exactly K iterations, Y resident in HBM
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.15)
    barrier()
    ctx.profile(True, segments=args.segments)
    n0 = lib.vbmf_b200_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record(stream)
    it, d = solver.run(args.steps, eps=0.0, flags=fl)
    e1.record(stream)
    barrier()
    t1 = time.time()
    ms = e0.elapsed_time(e1)
    launches = lib.vbmf_b200_launch_count() - n0
    prof = ctx.profile_read()
    ctx.profile(False)
    clocks = sampler.stop(t0, t1)
    if it != args.steps or not np.isfinite(d):
        raise SystemExit("timed region did not run %d iterations (it=%d, d=%r): result invalid" % (args.steps, it, d))
    tms = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = float(tms.item())
    value = args.steps / (ms * 1e-3)

    # ---- state_check: shard-invariant scalars of the state after warm-up + K iterations.  Runs at N = 1/2/4/8 start from the
    # same global initialisation, so these must agree across N to ~1e-10 (driver-visible sharded parity, SURVEY 8e).
    solver.download(p)
    a2 = torch.tensor([float(np.sum(np.asarray(p.AHat) ** 2))], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(a2, op=dist.ReduceOp.SUM)
    state_check = {"iterations": args.warmup + args.steps, "norm_BHat_fro": float(np.linalg.norm(p.BHat)),
                   "norm_AHat_fro": float(np.sqrt(a2.item())), "trace_SigmaB": float(np.trace(p.SigmaB)),
                   "trace_SigmaA": float(np.trace(p.SigmaA)),
                   "noise": float(p.sigma2) if kind == "dense" else float(p.sigmaHat), "delta": float(d)}
    if kind != "dense":
        ca = torch.tensor([float(np.sum(p.CA))], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(ca, op=dist.ReduceOp.SUM)
        state_check["sum_CA"] = float(ca.item())
        state_check["sum_CB"] = float(np.sum(p.CB))
    if kind == "dual":
        state_check.update({"alpha00": float(p.alpha00), "beta00": float(p.beta00), "alpha01": float(p.alpha01), "beta01": float(p.beta01)})
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, p, d, kind)

    # ---- roofline of the dominant kernel (the slower of the two contractions), CUDA events on the launching stream
    k1 = prof["k1_ms"] / max(prof["k1_launches"], 1)
    k2 = prof["k2_ms"] / max(prof["k2_launches"], 1)
    flops_per_launch = 2.0 * L * Mloc * H
    dom, dom_ms = ("K1 gemm_ytb (Y'*BHat)", k1) if k1 >= k2 else ("K2 gemm_ya (Y*AHat)", k2)
    traffic = None
    ncu_path = os.path.join(ROOT, "profiles", "ncu_summary.json")
    if os.path.exists(ncu_path):
        try:
            traffic = json.load(open(ncu_path)).get(args.workload, {}).get("K1" if k1 >= k2 else "K2", {}).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    achieved = flops_per_launch / (dom_ms * 1e-3) * 1e-12
    hbm_peak = None
    try:
        hbm_peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs"))
    except Exception:
        hbm_peak = 6535.7          # B200_PROFILING.md fallback (measured copy bandwidth of this pool)
    roofline = {"bound": "tensor", "kernel": dom, "achieved": achieved, "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s",
                "frac": achieved / FP64_PEAK_TFLOPS, "traffic": traffic, "frac_of_nominal_40_tflops": achieved / 40.0,
                "peak_source": "measured FP64 DMMA issue-rate microbenchmark on this pool's B200 (tools/microbench, profiles/"
                               "r01_fp64_peak_microbench.jsonl); MEASURED_PEAKS.json carries no FP64 figure; cuBLAS DGEMM reaches 35.4",
                "algorithmic_flops_per_launch": flops_per_launch,
                # the other roof, for context: one pass over the Y shard per launch against the measured HBM copy bandwidth
                "algorithmic_bytes_per_launch": 8.0 * L * Mloc, "hbm_gbs": 8.0 * L * Mloc / (dom_ms * 1e-3) * 1e-9,
                "hbm_peak_gbs": hbm_peak, "hbm_frac": (8.0 * L * Mloc / (dom_ms * 1e-3) * 1e-9 / hbm_peak) if hbm_peak else None,
                "k1_ms": k1, "k2_ms": k2, "k1_tflops": flops_per_launch / k1 * 1e-9 if k1 else None,
                "k2_tflops": flops_per_launch / k2 * 1e-9 if k2 else None,
                "iteration_frac_of_peak": 4.0 * L * M * H / (ms / args.steps * 1e-3) / (world * FP64_PEAK_TFLOPS * 1e12),
                "contraction_share_of_step": (k1 + k2) / (ms / args.steps),
                # the per-iteration packed all-reduce (N > 1), CUDA events on the launching stream of rank 0
                # N > 1: CUDA-event time of the exchange per iteration -- the NCCL all-reduce alone, or (peer_exchange) the whole
                # stretch from K2's split-K reduction to the Gram reduction: exchange epilogue on this rank's rows + Gram exchange
                "allreduce_ms": (prof["allreduce_ms"] / prof["allreduce_launches"]) if prof.get("allreduce_launches") else None,
                # CUDA events between the launches of one iteration on the main stream (mean over the timed iterations, this rank)
                "segments_ms": {k: round(v, 5) for k, v in prof.get("segments_ms", {}).items()},
                "peer_exchange": bool(ctx.peer_exchange())}

    # ---- e2e: the public API with every input in pinned host memory (upload Y + params, K iterations, download)
    e2e = None
    if not args.no_e2e:
        solver.close()
        ybytes = L * Mloc * 8
        ypin = torch.empty((Mloc, L), dtype=torch.float64, pin_memory=True)     # (M, L) C-order == L x M column-major
        Yh = ypin.numpy().T
        vb._lib.check(lib.vbmf_b200_download_Y(ctx.h, Yh.ctypes.data_as(vb._lib.p_f64), L))
        p2 = local_params()
        pin = {}
        for f in ("AHat", "BHat"):        # the big parameter arrays come from pinned memory too
            a = getattr(p2, f)
            tpin = torch.empty(a.shape[::-1], dtype=torch.float64, pin_memory=True)
            tpin.numpy().T[...] = a
            setattr(p2, f, tpin.numpy().T)
            pin[f] = tpin
        barrier()
        w0 = time.perf_counter()
        ctx.attach(Yh, M_global=M, col_offset=off, force=True)
        if kind == "dense":
            vb.vbmf_(None, p2, args.steps, eps=0.0, est_covs="est_covs" in flags, est_var="est_var" in flags, ctx=ctx, yhat=False)
            done = p2.iterations
        elif kind == "sparse":
            vb.vbmf_sparse_(None, p2, args.steps, eps=0.0, full_cov="full_cov" in flags, est_cb="est_cb" in flags, ctx=ctx, yhat=False)
            done = p2.iterations
        else:
            vb.vbmf_dual_(None, p2, args.steps, eps=0.0, full_cov="full_cov" in flags, est_cb="est_cb" in flags,
                          est_priors="est_priors" in flags, ctx=ctx, yhat=False)
            done = p2.iterations
        barrier()
        w = time.perf_counter() - w0
        tw = torch.tensor([w], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(tw, op=dist.ReduceOp.MAX)
        w = float(tw.item())
        state_bytes = (Mloc * H + L * H + 6 * H * H) * 8 if kind == "dense" else (5 * Mloc * H + L * H + 3 * L + 2 * H * H + 2 * H) * 8
        out_bytes = state_bytes + (0 if kind != "dense" else 0)
        e2e = {"value": done / w, "unit": "iterations/s", "h2d_bytes_per_step": (ybytes + state_bytes) / args.steps,
               "d2h_bytes_per_step": out_bytes / args.steps, "seconds": w, "iterations": done,
               "note": "one vbmf_ call per %d iterations: Y (%.1f GB) and the parameter struct uploaded from pinned host memory, results "
                       "downloaded; YHat (L x M) not requested" % (args.steps, ybytes / 1e9)}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    cpu = None
    if not args.no_cpu and world == 1:
        cpu = cpu_reference(L, M, H, kind, flags, steps=3, warmup=1, budget_s=25.0)

    line = {
        "metric": "VB iterations/s at %dx%dx%d (%s, Float64)" % (L, M, H, "dense vbmf" if kind == "dense" else "vbmf_" + kind),
        "value": value, "unit": "iterations/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak" if args.workload == "c5" else "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "global_shape": [L, M, H], "columns_per_gpu": Mloc, "parallelism": ("column-sharded Y, dp%d, " % world + (
                       "per-iteration exchange over peer-mapped memory with own kernels (reduce-scatter of Y*AHat, row-sharded BHat epilogue, "
                       "all-gather of BHat over NVLink)" if ctx.peer_exchange() else "one packed NCCL all-reduce per iteration")) if world > 1 else "single GPU", "l2": "inputs larger than L2 (Y shard %.1f GB), no flush"
                   % (L * Mloc * 8 / 1e9), "norm": "spectral", "eps": 0.0},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        "final_delta": d, "state_check": state_check,
    }
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
