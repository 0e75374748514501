"""`zkey contribute` / `zkey beacon` on the GPU (csrc/contribute.cu).

The device output must equal the host hook (the kernel's per-point code run on the CPU) and the test helper's closed-form
key (tests/contribution_cases.py: setup.make_zkey with delta = delta0 * k) byte for byte.  Every section-10 record must
pass the pairing checks `zkey verify` runs.  A key made from a ptau through preparePhase2 -> newZKey -> contribute ->
beacon must prove like the closed form with the contributed delta.  At the NZCP shape the rescaled sections are checked
by sampled points and by a random linear combination through the variable-base MSM, and the key must still prove.
"""
import random

import numpy as np
import pytest

import contribution_cases as cc
from nzcp_circom_b200 import api, groth16, verifier
from oracle import formats, ptau, setup
from oracle import prover as oprover
from oracle.bn254 import G1, G1_GEN, R_MOD, g1_from_bytes_mont
from test_zkey_contribute_cpu import CHAIN, SEED, STEPS, _case, apply_and_check, prior_beacon_key, run_host

pytestmark = pytest.mark.gpu


def run_device(zkey, step):
    timings = {}
    if "beacon_hash" in step:
        out = api.zkey_beacon(zkey, step["beacon_hash"], step["exp"], name=step.get("name"), timings=timings)
    else:
        out = api.zkey_contribute(zkey, name=step.get("name"), seed=step["seed"], timings=timings)
    assert sorted(timings) == [8, 9] and all(t >= 0 for t in timings.values())
    assert run_host(zkey, step) == out
    gs, ws = cc.sections(bytes(out[0])), cc.sections(bytes(zkey))
    for sid in (1, 3, 4, 5, 6, 7):
        assert gs[sid] == ws[sid], sid
    return out


CASES = {"contribute": (3, {}), "contribute_named": (3, {}), "beacon10": (3, {}), "beacon11_named": (3, {}),
         "infinity": (4, dict(unused_wire=True)), "domain1024": (8, dict(n_constraints=1000, n_public=3, n_free=12))}


@pytest.mark.parametrize("name", sorted(CASES))
def test_device_matches_host_and_helper(lib, name):
    seed, kw = CASES[name]
    case = _case(seed, **kw)
    if name == "domain1024":
        assert case["zkey"]["domainSize"] == 1024
    apply_and_check(case, case["zkey_bytes"], case["toxic"]["delta"], STEPS.get(name, STEPS["contribute"]), runner=run_device)


def _pair_eq(p1, q1, p2, q2):
    """e(p1, q1) == e(p2, q2)"""
    return verifier.pairing_product_is_one([(p1, q1), (G1.neg(p2), q2)])


def test_device_chain_records_verify(lib):
    """A chain on a key that already holds a beacon record: bytes as the helper, and every record passes zkey verify's
    pairing checks, starting from the delta1 of the key before the first contribution."""
    case = _case(5)
    zkey, delta = prior_beacon_key(case)
    for step in CHAIN:
        zkey, delta = apply_and_check(case, zkey, delta, step, runner=run_device)
    _, recs = cc.parse_mpc(cc.sections(zkey)[10])
    assert len(recs) == 4
    prev = G1.mul(G1_GEN, case["toxic"]["delta"])
    for rec in recs:
        c = cc.record_points(rec)
        g2_sp = cc.hash_to_g2(c["transcript"])
        assert verifier.g2_in_subgroup(c["g2_spx"])
        assert _pair_eq(c["g1_s"], c["g2_spx"], c["g1_sx"], g2_sp)
        assert _pair_eq(prev, c["g2_spx"], c["deltaAfter"], g2_sp)
        prev = c["deltaAfter"]
    hdr, _ = formats.read_zkey_header(zkey)
    assert prev == hdr["vk_delta_1"]


TOX = {"tau": 0x5EED5EED5EED, "alpha": 0xA1A1A1, "beta": 0xB2B2B2B2, "gamma": 1, "delta": 1}


def test_ptau_to_contributed_key_proves(lib):
    """ptau -> preparePhase2 -> newZKey -> contribute -> beacon: the proof with fixed r, s is the closed form with the
    contributed delta, verifies against the new key's verification key, and the first record starts from the G1
    generator (a `zkey new` key has delta = 1)."""
    rng = random.Random(9)
    cons, n_vars, defines = setup.random_circuit(rng, 20, 3, 4)
    wit = setup.solve_witness(cons, n_vars, defines, 3, [rng.randrange(R_MOD) for _ in range(4)])
    r1cs = formats.write_r1cs(n_vars, 3, 0, n_vars - 4, cons)
    # power 6 > cirPower 5: `zkey new` reads H from an exact Lagrange level (at cirPower = power it reads snarkjs's
    # top tauG1 level, which differs from make_zkey's H and gives the same proofs)
    raw = ptau.write_ptau(TOX["tau"], TOX["alpha"], TOX["beta"], 6, prepared=False)
    prepared = groth16.powersOfTau.preparePhase2(raw, None)
    k0 = {"type": "mem"}
    groth16.zKey.newZKey(r1cs, prepared, k0)
    k1, k2 = {"type": "mem"}, {"type": "mem"}
    e1 = cc.contribution(bytes(k0["data"]), name="alice", seed=SEED)
    h1 = groth16.zKey.contribute(k0, k1, "alice", "", seed=SEED)
    e2 = cc.contribution(bytes(k1["data"]), name="final", beacon_hash=bytes.fromhex("deadbeef"), exp=10)
    h2 = groth16.zKey.beacon(k1, k2, "final", "deadbeef", 10)
    assert (h1, h2) == (e1["hash"], e2["hash"])
    tox = dict(TOX, delta=e1["k"] * e2["k"] % R_MOD)
    want = cc.with_section10(formats.write_zkey(setup.make_zkey(cons, n_vars, 3, tox)), e2["s10"])
    gs, ws = cc.sections(bytes(k2["data"])), cc.sections(want)
    for sid in (2, 3, 5, 6, 7, 8, 9, 10):
        assert gs[sid] == ws[sid], sid
    r, s = 0x1357, 0x2468
    out = groth16.prove(k2, {"type": "mem", "data": formats.write_wtns(wit)}, r=r, s=s)
    assert out["proof"] == oprover.proof_to_json(setup.expected_proof(cons, n_vars, 3, tox, wit, r, s))
    assert groth16.verify(groth16.zKey.exportVerificationKey(k2["data"]), out["publicSignals"], out["proof"])
    rec = cc.record_points(cc.parse_mpc(gs[10])[1][0])
    assert _pair_eq(G1_GEN, rec["g2_spx"], rec["deltaAfter"], cc.hash_to_g2(rec["transcript"]))
    groth16.terminate()


def _rand_scalars(n, rs):
    x = rs.randint(0, 2 ** 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    x[:, 7] &= 0x1FFFFFFF
    return x


def test_nzcp_shape(lib):
    """n = 2^20, m = 880 001: sampled points against Python k^-1 * P, the whole sections through
    k * MSM(rho, L') == MSM(rho, L), and a proof with the contributed key verifies."""
    sc = api.SynthCircuit(seed=0xC0FFEE, n_constraints=835000, n_public=513, n_free=45000)
    zb = bytes(sc.zkey([0x1234567890ABCDEF1234567, 0xA1FA, 0xBE7A0000001, 0x6A33A, 0xDE17A5]))
    assert sc.domain_size == 1 << 20 and sc.n_vars == 880001
    timings = {}
    got, h = api.zkey_contribute(zb, name="nzcp", seed=SEED, timings=timings)
    exp = cc.contribution(zb, name="nzcp", seed=SEED)
    assert h == exp["hash"]
    kinv = pow(exp["k"], -1, R_MOD)
    old, new = cc.sections(zb), cc.sections(bytes(got))
    assert new[10] == exp["s10"]
    rs = np.random.RandomState(5)
    for sid in (8, 9):
        n = len(old[sid]) // 64
        for i in rs.choice(n, 1024, replace=False):
            P = g1_from_bytes_mont(old[sid][64 * i:64 * i + 64])
            assert g1_from_bytes_mont(new[sid][64 * i:64 * i + 64]) == G1.mul(P, kinv), (sid, i)
        rho = _rand_scalars(n, rs)
        lhs, _ = api.msm_var(new[sid], rho, n)
        rhs, _ = api.msm_var(old[sid], rho, n)
        lp = (int.from_bytes(lhs[:32], "little"), int.from_bytes(lhs[32:], "little"))
        rp = (int.from_bytes(rhs[:32], "little"), int.from_bytes(rhs[32:], "little"))
        assert G1.mul(lp, exp["k"]) == rp, sid
    wb = sc.wtns(1)
    out = groth16.prove({"type": "mem", "data": got}, {"type": "mem", "data": wb})
    assert groth16.verify(groth16.exportVerificationKey(got), out["publicSignals"], out["proof"])
    groth16.terminate()
