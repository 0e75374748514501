"""`zkey contribute` on one GPU: device time of sections 8 (L) and 9 (H), points/s, the achieved Fq-product rate and the
wall time of the whole call.

Two keys:
  nzcp  the NZCP shape (n = 2^20, m = 880 001: 879 487 L points, 2^20 H points), a synthetic circuit set up from known
        toxic waste (api.SynthCircuit, as bench.py);
  2^24  2^24 L and 2^24 H points: pseudo-random group elements (api.synth_points) in the container of a small synthetic
        key whose header is patched to match.  Rescaling does the same work whatever the points are.
The Fq-product count per point is the model of benchmarks/ptau_prepare.py (one signed 4-bit window scalar multiplication
and one affine conversion), divided by the kernel time and set against nzcp_intpipe_bench's dependent-chain Fq Montgomery
product rate measured in the same process.  Prints one JSON line.

    python benchmarks/zkey_contribute.py [--shapes nzcp 24]
"""
import argparse
import json
import os
import struct
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

from nzcp_circom_b200 import api  # noqa: E402
from oracle import formats  # noqa: E402
from ptau_prepare import COST, gpu_info, scalar_mul_cost  # noqa: E402

TOXIC = [0x1234567890ABCDEF1234567, 0xA1FA, 0xBE7A0000001, 0x6A33A, 0xDE17A5]
SEED = bytes(range(32))


def nzcp_key():
    sc = api.SynthCircuit(seed=0xC0FFEE, n_constraints=835000, n_public=513, n_free=45000)
    return bytes(sc.zkey(TOXIC))


def wide_key(log_n):
    """Sections 8 and 9 of 2^log_n pseudo-random points each, around the other sections of a small synthetic key."""
    n = 1 << log_n
    small = bytes(api.SynthCircuit(seed=5, n_constraints=100, n_public=1, n_free=16).zkey(TOXIC))
    _, secs = formats.read_container(small, b"zkey")
    s = {sid: small[v[0][0]:v[0][0] + v[0][1]] for sid, v in secs.items()}
    h = bytearray(s[2])
    struct.pack_into("<III", h, 72, n + 2, 1, n)           # nVars = nPublic + 1 + n, nPublic = 1, domainSize = n
    s[2] = bytes(h)
    s[8] = bytes(api.synth_points(201, n))
    s[9] = bytes(api.synth_points(202, n))
    return formats.write_container(b"zkey", 1, sorted(s.items()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", nargs="+", default=["nzcp", "24"])
    args = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("zkey_contribute benchmark: no CUDA device (there is no CPU fallback)")
    rec = {"op": "zkey_contribute", **gpu_info()}
    pipe = api.intpipe_bench()
    rec["intpipe_fq_mul_per_s"] = pipe["fq_mul_per_s"]
    per_point = scalar_mul_cost(False) + COST[False]["affine"]
    api.zkey_contribute(wide_key(4), seed=SEED)                # module load, first launches
    rec["runs"] = []
    for shape in args.shapes:
        key = nzcp_key() if shape == "nzcp" else wide_key(int(shape))
        timings = {}
        t0 = time.perf_counter()
        api.zkey_contribute(key, seed=SEED, timings=timings)
        wall = (time.perf_counter() - t0) * 1e3
        z, _ = formats.read_zkey_header(key)
        n_vars, n_public, domain = z["nVars"], z["nPublic"], z["domainSize"]
        points = (n_vars - n_public - 1) + domain
        kms = sum(timings.values())
        prods = points * per_point
        rec["runs"].append({"shape": shape, "l_points": n_vars - n_public - 1, "h_points": domain, "wall_ms": round(wall, 1),
                            "section_ms": {str(k): round(v, 2) for k, v in timings.items()}, "kernel_ms": round(kms, 2),
                            "points_per_s": points / (kms * 1e-3), "model_fq_products": prods,
                            "achieved_fq_mul_per_s": prods / (kms * 1e-3),
                            "share_of_intpipe": round(prods / (kms * 1e-3) / pipe["fq_mul_per_s"], 3)})
    print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
