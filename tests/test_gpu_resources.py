"""Every entry point gives back the device memory it takes, on success and on the error paths that fail after device work
has started.

Each case runs once to warm up (module loads, the context's local-memory reservation), then reads the device's free memory
with torch.cuda.mem_get_info, runs five create/free or call cycles, and reads it again.  A cycle that leaked any of its
buffers would leave the reading lower by at least that buffer; the margin is well below the footprint of one cycle of the
large cases (a 2^20-point MSM plan, a resident key with its provers, the 8 MB encode buffers of every point hasher).

mem_get_info reports the whole device.  If another process allocates or frees on the same GPU while a case runs, the
reading includes that; the cases are short to keep the window small.
"""
import os
import random

import numpy as np
import pytest

from nzcp_circom_b200 import api
from nzcp_circom_b200._lib import NzcpError
from oracle import bn254 as ob
from oracle import formats, ptau, setup
from util import le32

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MARGIN = 4 << 20
CYCLES = 5
N_PLAN = 1 << 20
TOX = {"tau": 0x5EED5EED5EED, "alpha": 0xA1A1A1, "beta": 0xB2B2B2B2}
SEED = bytes(range(32))


def _free_bytes():
    import torch
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info(0)[0]


def _no_leak(fn):
    fn()
    base = _free_bytes()
    for _ in range(CYCLES):
        fn()
    lost = base - _free_bytes()
    assert lost < MARGIN, "%d cycles lost %.1f MB of device memory" % (CYCLES, lost / 2**20)


def _scalars(n, seed):
    """n canonical scalars (top byte < 0x30, so every value is < r) as 32-byte little-endian records."""
    a = np.random.default_rng(seed).integers(0, 256, size=(n, 32), dtype=np.uint8)
    a[:, 31] &= 0x1F
    return a.tobytes()


@pytest.fixture(scope="module")
def golden(lib):
    with open(os.path.join(GOLDEN, "g256.zkey"), "rb") as f:
        zb = f.read()
    with open(os.path.join(GOLDEN, "g256.wtns"), "rb") as f:
        wb = f.read()
    return zb, wb


@pytest.fixture(scope="module")
def plan_inputs(lib):
    return bytes(api.synth_points(7, N_PLAN)), _scalars(N_PLAN, 7)


@pytest.fixture(scope="module")
def ceremony(lib):
    cons, n_vars, _ = setup.random_circuit(random.Random(11), 20, 3, 4)
    r1cs = formats.write_r1cs(n_vars, 3, 0, n_vars - 3 - 1, cons)
    raw = ptau.write_ptau(TOX["tau"], TOX["alpha"], TOX["beta"], 6, prepared=False)
    prepared = bytes(api.ptau_prepare(raw))
    key = bytes(api.zkey_new(r1cs, prepared, circuit_hash=True))
    return {"r1cs": r1cs, "raw": raw, "ptau": prepared, "key": key}


def test_prover_objects(golden):
    zb, wb = golden

    def cycle():
        with api.Zkey(zb) as zk:
            with api.Prover(zk) as pr:
                pr.prove(wb, r=1, s=2)
            with api.ProverPool(zk, n_provers=2) as pool:
                pool.prove_many([wb, wb], r=1, s=2)
            zk.prove_batch([wb, wb], r_list=[1, 1], s_list=[2, 2], n_provers=2)   # provers pooled inside the key
    _no_leak(cycle)


@pytest.mark.parametrize("mode", [0, 1])
def test_msm_plan(plan_inputs, mode):
    bases, sc = plan_inputs

    def cycle():
        with api.MsmPlan(bases, N_PLAN, mode=mode) as plan:
            plan.run(sc)
    _no_leak(cycle)


@pytest.mark.parametrize("entry", ["msm", "msm_var", "ntt", "ntt_coset"])
def test_standalone(plan_inputs, entry):
    n = 1 << 16
    bases, sc = plan_inputs[0][:n * 64], plan_inputs[1][:n * 32]
    data = bytearray(_scalars(1 << 18, 3))
    calls = {"msm": lambda: api.msm(bases, sc, n), "msm_var": lambda: api.msm_var(bases, sc, n),
             "ntt": lambda: api.ntt(data, 18), "ntt_coset": lambda: api.ntt_coset(data, 17, batch=2)}
    _no_leak(calls[entry])


@pytest.mark.parametrize("entry", ["zkey_new", "zkey_contribute", "ptau_prepare", "ptau_contribute", "zkey_verify"])
def test_ceremony(ceremony, entry):
    c = ceremony
    calls = {"zkey_new": lambda: api.zkey_new(c["r1cs"], c["ptau"], circuit_hash=True),
             "zkey_contribute": lambda: api.zkey_contribute(c["key"], seed=SEED),
             "ptau_prepare": lambda: api.ptau_prepare(c["raw"]),
             "ptau_contribute": lambda: api.ptau_contribute(c["raw"], seed=SEED),
             "zkey_verify": lambda: api.zkey_verify(c["key"], c["ptau"], r1cs=c["r1cs"], seed=SEED)}
    _no_leak(calls[entry])


def test_synth_zkey(lib):
    sc = api.SynthCircuit(seed=3, n_constraints=120, n_public=6, n_free=24)
    try:
        _no_leak(lambda: sc.zkey([3, 5, 7, 11, 13]))
    finally:
        sc.close()


def test_plan_run_out_of_range_scalar(plan_inputs):
    bases, sc = plan_inputs
    bad = bytearray(sc)
    bad[32 * 5:32 * 6] = le32(ob.R_MOD)

    def cycle():
        with api.MsmPlan(bases, N_PLAN, mode=1) as plan:
            with pytest.raises(NzcpError) as e:
                plan.run(bad)
            assert e.value.code == -7
    _no_leak(cycle)


def test_prove_non_canonical_witness(golden):
    zb, wb = golden
    bad = bytearray(wb)
    bad[len(bad) - 32:] = le32(ob.R_MOD)

    def cycle():
        with api.Zkey(zb) as zk, api.Prover(zk) as pr:
            with pytest.raises(NzcpError) as e:
                pr.prove(bad, r=1, s=2)
            assert e.value.code == -7
    _no_leak(cycle)
