"""`zkey verify` on one GPU at the NZCP shape: where the time of verifyFromR1cs goes.

The ptau is synthetic (power 21, pseudo-random points as benchmarks/ptau_prepare.py builds them: the checks do the same
work whatever the points are), taken through preparePhase2; the circuit is
SynthCircuit(seed=0xC0FFEE, n_constraints=835000, n_public=513, n_free=45000) (n = 2^20, m = 880 001); its key gets
newZKey(circuit_hash=True), one contribution and a beacon.  Reported, in ms: `zkey new` (the newZKey call), the
circuit-hash kernels (H differences and point encoding, device time) and the host BLAKE2b apart, the L MSMs, the H scalar
transform + NTT + MSMs (device time), the CPU pairings, and the wall time of the whole verifyFromR1cs.  Prints one JSON
line.

    python benchmarks/zkey_verify.py
"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

from nzcp_circom_b200 import api  # noqa: E402
from ptau_prepare import gpu_info, synth_ptau  # noqa: E402

SEED = bytes(range(32))


def nzcp_chain(timings=None):
    """-> dict(r1cs, ptau, init, key, hashes): the NZCP-shape chain newZKey(circuit_hash) -> contribute -> beacon."""
    prepared = bytes(api.ptau_prepare(synth_ptau(21)))
    r1cs = bytes(api.SynthCircuit(seed=0xC0FFEE, n_constraints=835000, n_public=513, n_free=45000).r1cs())
    t0 = time.perf_counter()
    init = bytes(api.zkey_new(r1cs, prepared, circuit_hash=True))
    if timings is not None:
        timings["zkey_new_ms"] = (time.perf_counter() - t0) * 1e3
    k1, h1 = api.zkey_contribute(init, name="nzcp", seed=SEED)
    k2, h2 = api.zkey_beacon(k1, bytes.fromhex("deadbeef"), 10, name="final")
    return {"r1cs": r1cs, "ptau": prepared, "init": init, "key": bytes(k2), "hashes": [h1, h2]}


def main():
    if api.device_count() < 1:
        raise SystemExit("zkey_verify benchmark: no CUDA device (there is no CPU fallback)")
    rec = {"op": "zkey_verify", "shape": "nzcp", **gpu_info()}
    t = {}
    ch = nzcp_chain(t)
    api.zkey_verify(ch["key"], ch["ptau"], init=ch["init"])          # module load, first launches
    timings = {}
    t0 = time.perf_counter()
    res = api.zkey_verify(ch["key"], ch["ptau"], r1cs=ch["r1cs"], timings=timings)
    wall = (time.perf_counter() - t0) * 1e3
    if not res["ok"]:
        raise SystemExit("zkey_verify benchmark: the key did not verify: %s" % res["message"])
    rec.update({k + ("" if k.endswith("_ms") else "_ms"): round(v, 1) for k, v in {**t, **timings}.items()})
    rec["verify_from_r1cs_wall_ms"] = round(wall, 1)
    print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
