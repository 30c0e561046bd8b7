"""Roofs of the INT8 contractions from a bench.py JSON line: INT8 operations and slice bytes over the measured K1 / K2 times.

    python tools/int8gemm/roofline.py profiles/r06_bench_c3_new_1.json

bench.py's roofline.frac and iteration_frac_of_peak are quoted against the FP64 peak and read above 1 on this path.  Here
each kernel is set against the rates it can reach:
  ops   = 28 slice products x 2*L*M*H            (levels 0..6 of 7 x 7 signed radix-256 digits)
  bytes = 7*L*M (seven int8 digit planes of Y, read once) + the operand digits (7*L*H or 7*M*H, L2-resident, not counted)
  INT8 tensor rate: 4.5 POPS dense (B200 data sheet, 1000 W card; not measured here).  HBM: the measured 6.54 TB/s copy rate
  (bench.py hbm_peak_gbs).  The larger of ops/rate and bytes/bandwidth is the least time; share = that / kernel time.
"""
import json
import sys

INT8_OPS = 4.5e15


def main(path):
    d = json.loads([ln for ln in open(path) if ln.lstrip().startswith("{")][-1])
    cfg = d["config"]
    L, H, M = cfg["global_shape"][0], cfg["global_shape"][2], cfg["columns_per_gpu"]
    roof = d["roofline"]
    bw = roof.get("hbm_peak_gbs", 6535.7) * 1e9
    ops, nbytes = 28 * 2.0 * L * M * H, 7.0 * L * M
    out = {"shape": [L, M, H], "clocks": d.get("clocks")}
    for k in ("k1", "k2"):
        t = roof[k + "_ms"] * 1e-3
        tmin = max(ops / INT8_OPS, nbytes / bw)
        out[k] = {"ms": roof[k + "_ms"], "int8_pops": ops / t / 1e15, "frac_of_int8_datasheet": ops / t / INT8_OPS,
                  "slice_tb_s": nbytes / t / 1e12, "frac_of_hbm_copy": nbytes / t / bw, "least_ms": tmin * 1e3,
                  "bound": "int8" if ops / INT8_OPS >= nbytes / bw else "hbm", "share_of_roof": tmin / t}
    print(json.dumps(out))


if __name__ == "__main__":
    main(sys.argv[1])
