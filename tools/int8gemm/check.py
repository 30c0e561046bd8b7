"""INT8-path contractions against NumPy and against the FP64 tensor-core path (VBMF_B200_GEMM=dmma) on the same data.

    python tools/int8gemm/check.py            # small and multi-tile shapes, prints one JSON line per case
Each case: normwise error max|err| / max|ref| of P = Y'B and Q = YA against NumPy (float64 BLAS) for both paths.
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def rel(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def main():
    import vbmf_b200_loader
    vb = vbmf_b200_loader.load()
    path = os.environ.get("VBMF_B200_GEMM", "int8")
    ctx = vb.Context(device=0)
    cases = [(10, 20, 2), (257, 1000, 64), (1000, 3001, 33), (64, 300, 7), (33, 7, 16), (16, 16, 1),
             (3000, 50000, 64), (40000, 300, 64), (2048, 4096, 64)]
    for L, M, H in cases:
        rng = np.random.default_rng(L * 7 + M)
        Y = np.asfortranarray(rng.standard_normal((L, M)))
        B = np.asfortranarray(rng.standard_normal((L, H)))
        A = np.asfortranarray(rng.standard_normal((M, H)))
        ctx.attach(Y, force=True)
        P = ctx.gemm_YtB(B)
        Q = ctx.gemm_YA(A)
        print(json.dumps({"path": path, "L": L, "M": M, "H": H, "errP": rel(P, Y.T @ B), "errQ": rel(Q, Y @ A),
                          "repro": bool(np.array_equal(P, ctx.gemm_YtB(B)) and np.array_equal(Q, ctx.gemm_YA(A)))}), flush=True)


if __name__ == "__main__":
    main()
