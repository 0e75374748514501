"""`powersoftau verify` on one GPU: the wall time of the whole call, each of its timing entries (host point checks, encode
kernels, host BLAKE2b of the next challenge, section MSMs, Lagrange transforms + MSMs) and the CPU pairing time of the
returned claims.

Inputs are ceremonies run inside the library: new -> contribute -> contribute -> beacon -> prepare phase2 at each power,
so the file is prepared and carries three records (the first challenge hash runs beside the section work).  Prints one
JSON line.

    python benchmarks/ptau_verify.py [--powers 20 22]
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

from nzcp_circom_b200 import api  # noqa: E402
from ptau_prepare import gpu_info  # noqa: E402

SEED = bytes(range(32))


def ceremony(power):
    """A prepared file with three records (two contributions, a beacon), built on the GPU."""
    f, _ = api.ptau_new(power, first_challenge=False)
    f, _ = api.ptau_contribute(f, name="alice", seed=SEED)
    f, _ = api.ptau_contribute(f, seed=bytes(32))
    f, _ = api.ptau_beacon(f, bytes.fromhex("0123456789abcdef"), 10, name="final")
    return bytes(api.ptau_prepare(f))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--powers", nargs="+", type=int, default=[20, 22])
    args = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("ptau_verify benchmark: no CUDA device (there is no CPU fallback)")
    rec = {"op": "ptau_verify", **gpu_info(), "runs": []}
    assert api.ptau_verify(ceremony(4), seed=SEED)["ok"]              # module load, first launches
    for power in args.powers:
        buf = ceremony(power)
        timings = {}
        t0 = time.perf_counter()
        res = api.ptau_verify(buf, timings=timings)
        wall = (time.perf_counter() - t0) * 1e3
        assert res["ok"], res["message"]
        rec["runs"].append({"power": power, "prepared": res["prepared"], "records": len(res["contributions"]),
                            "wall_ms": round(wall, 1), **{k: round(v, 2) for k, v in timings.items()}})
        del buf
    print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
