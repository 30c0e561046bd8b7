"""Decode the reference's own JLD (HDF5) fixtures into plain .npz goldens.

Inputs  (read-only, from a checkout of VBMatrixFactorization.jl named by the environment variable VBMF_REFERENCE_DIR):
    $VBMF_REFERENCE_DIR/examples/data/vbmf_test/{inputs,log}.jld     dense vbmf, 100 iterations
    $VBMF_REFERENCE_DIR/examples/data/sparse_test/{inputs,log}.jld   vbmf_sparse full_cov, 100 iterations
They were written by examples/toy_data.jl:35-36,55-56 through save_log (src/data_manip.jl:53-66).

Outputs (committed): tests/golden/vbmf_test.npz, tests/golden/sparse_test.npz

No HDF5 library exists in this image, so this is a minimal reader for exactly what JLD 0.5-era files
contain: 512-byte user block, v0 superblock, v1 object headers, link messages, contiguous / compact
little-endian f64 / i64 datasets.  Julia arrays are column-major; HDF5 dims are the Julia dims reversed,
so a Julia (d1, d2, T) array is returned here as a C-ordered numpy array of shape (T, d2, d1); consumers
use slice[t].T to get the Julia matrix of iteration t.

Run:  VBMF_REFERENCE_DIR=<checkout> python tests/golden/make_golden.py
"""
import os
import re
import struct
import sys

import numpy as np

OUT = os.path.dirname(os.path.abspath(__file__))


def _messages(buf, addr):
    """Yield (type, data) for every header message of the v1 object header at addr (follows continuations)."""
    ver, _, nmsg, _ref, hsize = struct.unpack_from("<BBHII", buf, addr)
    if ver != 1:
        raise ValueError("object header v%d at 0x%x not supported" % (ver, addr))
    blocks = [(addr + 16, hsize)]
    seen = 0
    while blocks and seen < nmsg:
        pos, size = blocks.pop(0)
        end = pos + size
        while pos + 8 <= end and seen < nmsg:
            mtype, msize, _flags = struct.unpack_from("<HHB", buf, pos)
            data = buf[pos + 8: pos + 8 + msize]
            pos += 8 + msize
            seen += 1
            if mtype == 0x10:  # continuation
                off, length = struct.unpack_from("<QQ", data, 0)
                blocks.append((off, length))
            else:
                yield mtype, data


def _read_dataset(buf, addr):
    dims = None
    dtype = None
    raw = None
    for mtype, data in _messages(buf, addr):
        if mtype == 0x01:  # dataspace
            ver, rank = data[0], data[1]
            off = 8 if ver == 1 else 4
            dims = struct.unpack_from("<%dQ" % rank, data, off) if rank else ()
        elif mtype == 0x03:  # datatype
            cls = data[0] & 0x0F
            size = struct.unpack_from("<I", data, 4)[0]
            if cls == 1 and size == 8:
                dtype = np.dtype("<f8")
            elif cls == 0 and size == 8:
                dtype = np.dtype("<i8")
            else:
                dtype = ("unsupported", cls, size)
        elif mtype == 0x08:  # layout
            ver, lcls = data[0], data[1]
            if ver != 3:
                raise ValueError("layout v%d" % ver)
            if lcls == 1:
                a, s = struct.unpack_from("<QQ", data, 2)
                raw = buf[a: a + s] if a != 0xFFFFFFFFFFFFFFFF else b""
            elif lcls == 0:
                s = struct.unpack_from("<H", data, 2)[0]
                raw = data[4: 4 + s]
            else:
                raise ValueError("chunked layout not supported")
    if not isinstance(dtype, np.dtype) or raw is None or dims is None:
        return None
    n = int(np.prod(dims)) if dims else 1
    arr = np.frombuffer(raw[: n * 8], dtype=dtype).copy()
    return arr.reshape(dims) if dims else arr.reshape(())


def read_jld(path):
    with open(path, "rb") as f:
        buf = f.read()[512:]  # strip the JLD user block; HDF5 base address = 512
    if buf[:8] != b"\x89HDF\r\n\x1a\n":
        raise ValueError("no HDF5 superblock at offset 512 in " + path)
    out = {}
    # link message: version 1, flags 0x10 (charset present, 1-byte name length), charset 1, len, name, address
    for m in re.finditer(rb"\x01\x10\x01([\x01-\x40])", buf):
        ln = m.group(1)[0]
        name = buf[m.end(): m.end() + ln]
        if not re.fullmatch(rb"[A-Za-z_][A-Za-z0-9_]*", name):
            continue
        addr = struct.unpack_from("<Q", buf, m.end() + ln)[0]
        if addr + 16 > len(buf) or buf[addr] != 1:
            continue
        try:
            arr = _read_dataset(buf, addr)
        except Exception:
            continue
        if arr is not None:
            out[name.decode()] = arr
    return out


def main():
    global OUT
    if "--out" in sys.argv:          # write somewhere else (tests/test_oracle_mp.py re-derives the fixtures and compares)
        OUT = sys.argv[sys.argv.index("--out") + 1]
    if not os.environ.get("VBMF_REFERENCE_DIR"):
        return "set VBMF_REFERENCE_DIR to a checkout of VBMatrixFactorization.jl"
    ref = os.path.join(os.environ["VBMF_REFERENCE_DIR"], "examples", "data")
    for case in ("vbmf_test", "sparse_test"):
        inputs = read_jld(os.path.join(ref, case, "inputs.jld"))
        log = read_jld(os.path.join(ref, case, "log.jld"))
        Y = inputs["Y"]  # (M, L) C-order == Julia L x M column-major
        fields = {"Y": np.ascontiguousarray(Y)}
        for k, v in sorted(log.items()):
            if k in ("YHat",):   # constant (never refreshed inside the loop); keep only the first slice
                v = v[:1]
            if k in ("SigmaATVec", "invSigmaATVec"):
                # (T, MH, MH) block-diagonal: keep the M diagonal HxH blocks + the off-block max as a scalar
                T, MH, _ = v.shape
                M = Y.shape[0]
                H = MH // M
                blocks = np.stack([v[:, m * H:(m + 1) * H, m * H:(m + 1) * H] for m in range(M)], axis=1)
                mask = np.kron(np.eye(M), np.ones((H, H))) == 0
                fields[k + "_offblock_max"] = np.array(np.abs(v[:, mask]).max())
                v = blocks  # (T, M, H, H) ; block[t, m] is symmetric up to rounding
            fields["log_" + k] = np.ascontiguousarray(v)
        np.savez_compressed(os.path.join(OUT, case + ".npz"), **fields)
        print(case, {k: v.shape for k, v in fields.items()})


if __name__ == "__main__":
    sys.exit(main())
