"""`powersoftau contribute` / `powersoftau beacon` on the GPU (csrc/ptau_contribute.cu).

The device output must equal the host hook (the kernels' per-point code run on the CPU) and the test helper's closed-form
file (tests/ptau_contribution_cases.py: write_ptau with tau t, alpha a, beta b) byte for byte, and every record must pass
the pairing checks `powersoftau verify` runs.  At powers 16 and 20 the sections are checked by sampled points against
Python and, at 20, whole through a random linear combination on the variable-base MSM.  A ceremony run inside the library,
new -> contribute -> contribute -> beacon -> prepare phase2 -> zkey new -> zkey contribute, must give the prepared file of
the product key, a key that verifies, and the closed-form proof.
"""
import hashlib
import random
import struct

import numpy as np
import pytest

import contribution_cases as cc
import ptau_cases
import ptau_contribution_cases as pc
from nzcp_circom_b200 import api, groth16
from oracle import formats, ptau, setup
from oracle import prover as oprover
from oracle.bn254 import G1, G2, R_MOD, g1_from_bytes_mont, g2_from_bytes_mont, to_le32
from test_ptau_contribute_cpu import (ALPHA, BETA, SEED, STEPS, TAU, _with_infinity, apply_and_check, prior_beacon_file,
                                      run_chain, run_host)

pytestmark = pytest.mark.gpu


def run_device(buf, step, host=True):
    timings = {}
    if "beacon_hash" in step:
        out = api.ptau_beacon(buf, step["beacon_hash"], step["exp"], name=step.get("name"), timings=timings)
    else:
        out = api.ptau_contribute(buf, name=step.get("name"), seed=step["seed"], timings=timings)
    assert sorted(map(str, timings)) == sorted(map(str, api.PTAU_CONTRIBUTE_TIMINGS))
    assert all(t >= 0 for t in timings.values())
    if host:
        assert run_host(buf, step) == out
    return out


@pytest.mark.parametrize("step", sorted(STEPS))
def test_device_from_new(lib, step):
    apply_and_check(bytes(api.ptau_new(3)[0]), (1, 1, 1), STEPS[step], runner=run_device)


def test_device_chain(lib):
    run_chain(*prior_beacon_file(), runner=run_device)


def test_device_prepared_and_infinity(lib):
    prepared = ptau_cases.write_prepared(TAU, ALPHA, BETA, 3)
    apply_and_check(prepared, (TAU, ALPHA, BETA), STEPS["contribute_named"], runner=run_device)
    inf = [(5, 2), (3, 5), (2, 14), (6, 0)]
    buf = _with_infinity(ptau.write_ptau(TAU, ALPHA, BETA, 3, prepared=False), inf)
    apply_and_check(buf, (TAU, ALPHA, BETA), STEPS["beacon10"], runner=run_device, infinity=inf)


def test_device_power10(lib):
    buf = ptau.write_ptau(TAU, ALPHA, BETA, 10, prepared=False)
    apply_and_check(buf, (TAU, ALPHA, BETA), STEPS["contribute_named"], runner=lambda b, s: run_device(b, s, host=False))


# ------------------------------------------------------------------------------------------------ large powers
def random_ptau(power, seed):
    """A phase-1 container of pseudo-random points (api.synth_points): what a contribution does to a point does not
    depend on the point."""
    n = 1 << power
    secs = [(1, pc.header(power))]
    for sid, cnt, g2 in ((2, 2 * n - 1, False), (3, n, True), (4, n, False), (5, n, False), (6, 1, True)):
        secs.append((sid, bytes(api.synth_points(seed + sid, cnt, g2=g2))))
    secs.append((7, struct.pack("<I", 0)))
    return formats.write_container(b"ptau", 1, secs)


FIRST = {2: 0, 3: 0, 4: 1, 5: 2, 6: 2}      # which key part is `first` (0: tau, i.e. first = 1)


def _first(key, sid):
    return 1 if FIRST[sid] == 0 else key[FIRST[sid]]["prv"]


def _contribute_big(power, seed):
    buf = random_ptau(power, seed)
    got, h = api.ptau_contribute(buf, name="big", seed=SEED)
    key = pc.create_key(cc.rng_contribute(SEED), pc.first_challenge_hash(power))
    return buf, bytes(got), h, key


def _check_samples(old, new, key, rs, k=256):
    t = key[0]["prv"]
    for sid in range(2, 7):
        g2 = sid in pc.G2_SECTIONS
        sz, dec, grp = (128, g2_from_bytes_mont, G2) if g2 else (64, g1_from_bytes_mont, G1)
        n = len(old[sid]) // sz
        idx = sorted(i for i in {0, 1, n - 1} | set(rs.choice(n, min(n, k), replace=False).tolist()) if i < n)
        for i in idx:
            s = _first(key, sid) * pow(t, i, R_MOD) % R_MOD
            assert dec(new[sid][sz * i:sz * (i + 1)]) == grp.mul(dec(old[sid][sz * i:sz * (i + 1)]), s), (sid, i)


def test_power16_hashes_and_samples(lib):
    buf, got, h, key = _contribute_big(16, 100)
    old, new = pc.sections(buf), pc.sections(got)
    challenge = pc.first_challenge_hash(16)
    response = hashlib.blake2b(challenge + pc.encodings(new, True) + pc.pub_key(key, False), digest_size=64).digest()
    assert h == response
    rec = pc.record_fields(pc.parse_records(new[7])[-1])
    assert rec["next"] == hashlib.blake2b(response + pc.encodings(new, False), digest_size=64).digest()
    assert pc.Blake2b.from_partial(rec["partial"]).update(pc.pub_key(key, False)).digest() == response
    assert pc.parse_records(new[7])[-1][:768] == pc.pub_key(key, True)
    _check_samples(old, new, key, np.random.RandomState(16))


def _scalars(vals):
    return np.frombuffer(b"".join(to_le32(v) for v in vals), dtype=np.uint32)


def test_power20_msm(lib):
    """MSM(rho, new) == MSM(rho_i * first * t^i, old) over every G1 section and tauG2."""
    buf, got, _, key = _contribute_big(20, 200)
    old, new = pc.sections(buf), pc.sections(got)
    rs = np.random.RandomState(20)
    _check_samples(old, new, key, rs, k=64)
    t = key[0]["prv"]
    rnd = random.Random(20)
    for sid in (2, 3, 4, 5):
        g2 = sid in pc.G2_SECTIONS
        n = len(old[sid]) // (128 if g2 else 64)
        rho = [rnd.getrandbits(253) for _ in range(n)]
        scaled, s = [], _first(key, sid)
        for r in rho:
            scaled.append(r * s % R_MOD)
            s = s * t % R_MOD
        lhs, _ = api.msm_var(new[sid], _scalars(rho), n, g2=g2)
        rhs, _ = api.msm_var(old[sid], _scalars(scaled), n, g2=g2)
        assert lhs == rhs, sid


# ------------------------------------------------------------------------------------------------ a whole ceremony
class _Log:
    def __init__(self):
        self.lines = []

    def __getattr__(self, level):
        return lambda msg: self.lines.append((level, msg))


def test_ceremony_to_proof(lib):
    """newAccumulator(6) -> contribute -> contribute -> beacon -> preparePhase2 -> newZKey -> zKey.contribute: the prepared
    file is write_prepared of the product key, the zkey verifies from its r1cs, and a proof with fixed r, s is the closed
    form and verifies."""
    f0 = {"type": "mem"}
    assert groth16.powersOfTau.newAccumulator("bn128", 6, f0) == pc.first_challenge_hash(6)
    state, cur = (1, 1, 1), bytes(f0["data"])
    steps = [("alice", SEED, None), (None, bytes(32), None), ("final", None, "deadbeef")]
    for name, seed, beacon in steps:
        nxt, log = {"type": "mem"}, _Log()
        if beacon is None:
            e = pc.contribution(cur, *state, name=name, seed=seed)
            h = groth16.powersOfTau.contribute({"type": "mem", "data": cur}, nxt, name, "", log, seed=seed)
        else:
            e = pc.contribution(cur, *state, name=name, beacon_hash=bytes.fromhex(beacon), exp=10)
            h = groth16.powersOfTau.beacon({"type": "mem", "data": cur}, nxt, name, beacon, 10, log)
        assert h == e["response"] and bytes(nxt["data"]) == e["file"]
        assert ("info", groth16._format_hash(e["next"], "Next Challenge Hash: ")) in log.lines
        state, cur = (e["tau"], e["alpha"], e["beta"]), bytes(nxt["data"])
    tau, alpha, beta = state
    prepared = bytes(groth16.powersOfTau.preparePhase2(cur, None))
    got, want = pc.sections(prepared), pc.sections(ptau_cases.write_prepared(tau, alpha, beta, 6))
    assert sorted(got) == sorted(want) == [1, 2, 3, 4, 5, 6, 7, 12, 13, 14, 15]
    for sid in want:                     # write_prepared has no records; preparePhase2 carries the three along
        assert got[sid] == (pc.sections(cur)[7] if sid == 7 else want[sid]), sid
    assert len(pc.parse_records(got[7])) == 3

    log = _Log()                                                  # a prepared input: snarkjs's warning, 12-15 dropped
    again = {"type": "mem"}
    groth16.powersOfTau.contribute(prepared, again, None, "", log, seed=SEED)
    assert any(lvl == "warn" and "phase2 calculated" in m for lvl, m in log.lines)
    assert sorted(pc.sections(bytes(again["data"]))) == list(range(1, 8))

    rng = random.Random(9)
    cons, n_vars, defines = setup.random_circuit(rng, 20, 3, 4)
    wit = setup.solve_witness(cons, n_vars, defines, 3, [rng.randrange(R_MOD) for _ in range(4)])
    r1cs = formats.write_r1cs(n_vars, 3, 0, n_vars - 4, cons)
    k0, k1 = {"type": "mem"}, {"type": "mem"}
    groth16.zKey.newZKey(r1cs, prepared, k0, circuit_hash=True)
    e = cc.contribution(bytes(k0["data"]), name="p2", seed=SEED)
    groth16.zKey.contribute(k0, k1, "p2", "", seed=SEED)
    assert groth16.zKey.verifyFromR1cs(r1cs, prepared, k1)
    tox = {"tau": tau, "alpha": alpha, "beta": beta, "gamma": 1, "delta": e["k"]}
    r, s = 0x1357, 0x2468
    out = groth16.prove(k1, {"type": "mem", "data": formats.write_wtns(wit)}, r=r, s=s)
    assert out["proof"] == oprover.proof_to_json(setup.expected_proof(cons, n_vars, 3, tox, wit, r, s))
    assert groth16.verify(groth16.zKey.exportVerificationKey(k1["data"]), out["publicSignals"], out["proof"])
    groth16.terminate()
