"""`powersoftau contribute` on one GPU: key-kernel device time per section, encode-kernel device time, host BLAKE2b time,
the wall time of the whole call, G1 / G2 points/s and the achieved Fq-product rate.

Inputs are phase-1 containers of pseudo-random points (api.synth_points) with no earlier records, so the call also
computes the first challenge hash (a host BLAKE2b pass over ~384 * 2^power bytes).  What a contribution does to a point
does not depend on the point.  The Fq-product count per point is the model of benchmarks/ptau_prepare.py (one signed 4-bit
window scalar multiplication and one affine conversion; the ~45 Fr products of first * tau^i are left out), divided by the
key-kernel time and set against nzcp_intpipe_bench's dependent-chain Fq Montgomery product rate measured in the same
process.  Prints one JSON line.

    python benchmarks/ptau_contribute.py [--powers 20 22]
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
from oracle.bn254 import Q_MOD, to_le32  # noqa: E402
from ptau_prepare import COST, gpu_info, scalar_mul_cost  # noqa: E402

SEED = bytes(range(32))
G2_SECTIONS = (3, 6)


def random_ptau(power, seed=300):
    n = 1 << power
    secs = [(1, struct.pack("<I", 32) + to_le32(Q_MOD) + struct.pack("<II", power, power))]
    for sid, cnt in ((2, 2 * n - 1), (3, n), (4, n), (5, n), (6, 1)):
        secs.append((sid, bytes(api.synth_points(seed + sid, cnt, g2=sid in G2_SECTIONS))))
    secs.append((7, struct.pack("<I", 0)))
    return formats.write_container(b"ptau", 1, secs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--powers", nargs="+", type=int, default=[20, 22])
    args = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("ptau_contribute benchmark: no CUDA device (there is no CPU fallback)")
    rec = {"op": "ptau_contribute", **gpu_info()}
    pipe = api.intpipe_bench()
    rec["intpipe_fq_mul_per_s"] = pipe["fq_mul_per_s"]
    cost = {g2: scalar_mul_cost(g2) + COST[g2]["affine"] for g2 in (False, True)}
    api.ptau_contribute(random_ptau(4), seed=SEED)                # module load, first launches
    rec["runs"] = []
    for power in args.powers:
        buf = random_ptau(power)
        timings = {}
        t0 = time.perf_counter()
        api.ptau_contribute(buf, seed=SEED, timings=timings)
        wall = (time.perf_counter() - t0) * 1e3
        n = 1 << power
        pts = {2: 2 * n - 1, 3: n, 4: n, 5: n, 6: 1}
        g1_pts = sum(v for k, v in pts.items() if k not in G2_SECTIONS)
        g2_pts = sum(v for k, v in pts.items() if k in G2_SECTIONS)
        g1_ms = sum(timings[k] for k in pts if k not in G2_SECTIONS)
        g2_ms = sum(timings[k] for k in pts if k in G2_SECTIONS)
        prods = g1_pts * cost[False] + g2_pts * cost[True]
        key_ms = g1_ms + g2_ms
        rec["runs"].append({"power": power, "g1_points": g1_pts, "g2_points": g2_pts, "wall_ms": round(wall, 1),
                            "key_kernel_ms": {str(k): round(timings[k], 2) for k in pts},
                            "encode_kernel_ms": round(timings["encode"], 2), "blake2b_ms": round(timings["blake2b"], 1),
                            "g1_points_per_s": g1_pts / (g1_ms * 1e-3), "g2_points_per_s": g2_pts / (g2_ms * 1e-3),
                            "model_fq_products": prods, "achieved_fq_mul_per_s": prods / (key_ms * 1e-3),
                            "share_of_intpipe": round(prods / (key_ms * 1e-3) / pipe["fq_mul_per_s"], 3)})
        del buf
    print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
