"""Worst normwise difference per field between two bench.py --dump-outputs directories: max|a-b| / max|b|."""
import json
import os
import sys

import numpy as np


def main(a, b):
    out = {}
    for f in sorted(os.listdir(b)):
        if f.endswith(".npy"):
            x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
            den = float(np.max(np.abs(y))) if y.size else 0.0
            out[f[:-4]] = float(np.max(np.abs(x - y)) / den) if den > 0 else float(np.max(np.abs(x - y), initial=0.0))
    print(json.dumps({"a": a, "b": b, "worst": max(out.values(), default=0.0), "fields": out}))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
