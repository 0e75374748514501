"""`powersoftau prepare phase2` on one GPU: per-section kernel time, wall time and the achieved Fq-product rate.

The inputs are pseudo-random group elements (api.synth_points), not real tau powers: the inverse FFT does the same work
whatever the points are.  Power 20 and 22 (the size of powersOfTau28_hez_final_22.ptau, what the NZCP circuit needs).  The
Fq-product count is a model (below), divided by the kernel time and set against nzcp_intpipe_bench's dependent-chain Fq
Montgomery product rate measured in the same process.  Prints one JSON line.

    python benchmarks/ptau_prepare.py [--powers 20 22]
"""
import argparse
import json
import os
import struct
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from nzcp_circom_b200 import api  # noqa: E402
from oracle import formats  # noqa: E402
from oracle.bn254 import Q_MOD, to_le32  # noqa: E402

# Fq products per operation (an Fq2 product = 3, an Fq2 square = 2): XYZZ doubling 6M + 3S, addition 12M + 2S, mixed
# addition 8M + 2S, affine conversion = a division-step inversion (~50 products of issue slots; Fq2: one Fq inversion + 5)
# + 4M.  A butterfly with twiddle w^-k, k != 0: signed 4-bit windows over a ~254-bit scalar, a table of 1..8 * b (one
# affine doubling + 6 mixed additions), 252 doublings and ~60 additions (1/16 of the digits are 0); every butterfly:
# 2 mixed additions + 2 affine conversions.  Twiddle 1 (k = 0) costs no multiplication.
COST = {False: {"dbl": 9, "add": 14, "madd": 10, "affine": 54}, True: {"dbl": 24, "add": 40, "madd": 28, "affine": 70}}


def scalar_mul_cost(g2):
    c = COST[g2]
    return c["dbl"] + 6 * c["madd"] + 252 * c["dbl"] + 60 * c["add"]


def section_model(top, g2):
    """-> (butterflies, Fq products) of one output section with levels 0 .. top (load included)."""
    c = COST[g2]
    bfly = prods = 0
    for s in range(top):
        nb = (1 << top) - (1 << s)                 # levels p > s, 2^(p-1) butterflies each
        nz = nb - sum(1 << (p - 1 - s) for p in range(s + 1, top + 1))  # minus those with k = 0
        bfly += nb
        prods += nz * scalar_mul_cost(g2) + nb * (2 * c["madd"] + 2 * c["affine"])
    slots = (2 << top) - 1
    prods += slots * (scalar_mul_cost(g2) + c["affine"])   # load: 2^-p * P, 2^-0 = 1 aside
    return bfly, prods


def synth_ptau(power):
    n = 1 << power
    secs = [(1, struct.pack("<I", 32) + to_le32(Q_MOD) + struct.pack("<II", power, power)),
            (2, bytes(api.synth_points(101, 2 * n - 1))), (3, bytes(api.synth_points(102, n, g2=True))),
            (4, bytes(api.synth_points(103, n))), (5, bytes(api.synth_points(104, n))),
            (6, bytes(api.synth_points(105, 1, g2=True))), (7, bytes(4))]
    return formats.write_container(b"ptau", 1, secs)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim, clk = [x.strip() for x in out.split(",")]
        return {"device": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:          # the numbers below stay valid; the record says what could not be read
        return {"device": "unknown", "power_limit": "unknown (%s)" % type(e).__name__}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--powers", type=int, nargs="+", default=[20, 22])
    args = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("ptau_prepare benchmark: no CUDA device (there is no CPU fallback)")
    rec = {"op": "ptau_prepare", **gpu_info()}
    pipe = api.intpipe_bench()
    rec["intpipe_fq_mul_per_s"] = pipe["fq_mul_per_s"]
    api.ptau_prepare(synth_ptau(2))                  # module load, first launches
    rec["runs"] = []
    for power in args.powers:
        raw = synth_ptau(power)
        timings = {}
        t0 = time.perf_counter()
        api.ptau_prepare(raw, timings=timings)
        wall = (time.perf_counter() - t0) * 1e3
        run = {"power": power, "wall_ms": round(wall, 1), "section_ms": {str(k): round(v, 1) for k, v in timings.items()}}
        bfly = prods = 0
        for sid, top, g2 in ((12, power + 1, False), (13, power, True), (14, power, False), (15, power, False)):
            b, p = section_model(top, g2)
            bfly += b
            prods += p
        kms = sum(timings.values())
        run.update(kernel_ms=round(kms, 1), butterflies=bfly, model_fq_products=prods,
                   achieved_fq_mul_per_s=prods / (kms * 1e-3),
                   share_of_intpipe=round(prods / (kms * 1e-3) / pipe["fq_mul_per_s"], 3))
        rec["runs"].append(run)
    print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
