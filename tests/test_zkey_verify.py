"""`zkey verify` and the circuit hash on the GPU (csrc/verify.cu).

A key taken through preparePhase2 -> newZKey(circuit_hash=True) -> contribute -> contribute -> beacon must verify from
the .r1cs and from the initial key, with the circuit hash of the test helper (tests/verify_cases.py) and the contribution
hashes `zkey contribute` / `zkey beacon` returned.  Every one-change tampering must fail with snarkjs's message, for
several seeds of the random checks.  At the NZCP shape (synthetic ptau, power 21) the chain verifies and an altered L or
H point is caught.
"""
import os
import random
import sys

import pytest

import contribution_cases as cc
import verify_cases as vc
from nzcp_circom_b200 import api, groth16, verifier
from oracle import formats, ptau, setup
from oracle.bn254 import (CURVE_B2, G1, G2, Q_MOD, g1_from_bytes_mont, g1_to_bytes_mont, g2_from_bytes_mont,
                          g2_to_bytes_mont)

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "benchmarks"))
from zkey_verify import nzcp_chain  # noqa: E402  (the chain the benchmark times)

pytestmark = pytest.mark.gpu

SEEDS = [bytes([s]) * 32 for s in (1, 2, 3)]
TOX = {"tau": 0x5EED5EED5EED, "alpha": 0xA1A1A1, "beta": 0xB2B2B2B2}


def _r1cs(seed, n_constraints=20, n_public=3, n_free=4):
    cons, n_vars, _ = setup.random_circuit(random.Random(seed), n_constraints, n_public, n_free)
    return formats.write_r1cs(n_vars, n_public, 0, n_vars - n_public - 1, cons)


def _chain(r1cs, prepared):
    """-> (initial key, [keys after each step], [contribution hashes])"""
    k0 = {"type": "mem"}
    groth16.zKey.newZKey(r1cs, prepared, k0, circuit_hash=True)
    keys, hashes, cur = [], [], k0
    for step in [("alice", bytes(range(32))), (None, bytes(32)), None]:
        nxt = {"type": "mem"}
        if step is None:
            hashes.append(groth16.zKey.beacon(cur, nxt, "final", "deadbeef", 10))
        else:
            hashes.append(groth16.zKey.contribute(cur, nxt, step[0], "", seed=step[1]))
        keys.append(bytes(nxt["data"]))
        cur = nxt
    return bytes(k0["data"]), keys, hashes


@pytest.fixture(scope="module")
def chain(lib):
    r1cs = _r1cs(11)
    raw = ptau.write_ptau(TOX["tau"], TOX["alpha"], TOX["beta"], 6, prepared=False)
    prepared = bytes(groth16.powersOfTau.preparePhase2(raw, None))
    init, keys, hashes = _chain(r1cs, prepared)
    return {"r1cs": r1cs, "ptau": prepared, "init": init, "keys": keys, "hashes": hashes}


def _both(ch, key, seed=None):
    a = api.zkey_verify(key, ch["ptau"], r1cs=ch["r1cs"], seed=seed)
    b = api.zkey_verify(key, ch["ptau"], init=ch["init"], seed=seed)
    return a, b


def test_full_chain_verifies(chain):
    want = vc.circuit_hash(chain["init"], chain["ptau"])
    assert api.zkey_circuit_hash(chain["init"], chain["ptau"]) == want
    assert api.host_zkey_circuit_hash(chain["init"], chain["ptau"]) == want
    assert cc.sections(chain["init"])[10][:64] == want
    final = chain["keys"][-1]
    for res in _both(chain, final):
        assert res["ok"], res["message"]
        assert res["cs_hash"] == want
        assert [c["hash"] for c in res["contributions"]] == chain["hashes"]
        assert [c["name"] for c in res["contributions"]] == ["alice", "", "final"]
        assert res["contributions"][2]["beacon_hash"] == bytes.fromhex("deadbeef")
    assert groth16.zKey.verifyFromR1cs(chain["r1cs"], chain["ptau"], final)
    assert groth16.zKey.verifyFromInit(chain["init"], chain["ptau"], final)
    for res in _both(chain, chain["init"]):       # zero contributions
        assert res["ok"], res["message"]


def test_plain_newzkey_key(chain):
    plain = bytes(api.zkey_new(chain["r1cs"], chain["ptau"]))
    assert cc.sections(plain)[10][:64] == bytes(64)
    res = api.zkey_verify(plain, chain["ptau"], r1cs=chain["r1cs"])
    assert not res["ok"] and res["message"] == "Circuit does not match"


def _edit(key, sid, fn):
    secs = cc.sections(key)
    secs[sid] = bytes(fn(bytearray(secs[sid])))
    return formats.write_container(b"zkey", 1, sorted(secs.items()))


def _rec_off(key, i):
    _, recs = cc.parse_mpc(cc.sections(key)[10])
    return 68 + sum(len(r) for r in recs[:i])


def _dbl_g1(b, off):
    b[off:off + 64] = g1_to_bytes_mont(G1.mul(g1_from_bytes_mont(bytes(b[off:off + 64])), 2))
    return b


def _dbl_g2(b, off):
    b[off:off + 128] = g2_to_bytes_mont(G2.mul(g2_from_bytes_mont(bytes(b[off:off + 128])), 2))
    return b


def _off_subgroup_g2():
    rng = cc.rng_from_digest(bytes(32))
    while True:
        x = (cc.from_rng(rng, Q_MOD), cc.from_rng(rng, Q_MOD))
        y = cc.f2_sqrt(verifier.f2_add(verifier.f2_mul(verifier.f2_sqr(x), x), CURVE_B2))
        if y is not None and not verifier.g2_in_subgroup((x, y)):
            return (x, y)


def _flip(off):
    def f(b):
        b[off] ^= 1
        return b
    return f


def _set(off, data):
    def f(b):
        b[off:off + len(data)] = data
        return b
    return f


def _swap_h(b):
    b[0:64], b[64:128] = b[64:128], b[0:64]
    return b


def _tampered(ch):
    k = ch["keys"][-1]
    r0, r2 = _rec_off(k, 0), _rec_off(k, 2)
    n_params = len(cc.parse_mpc(cc.sections(k)[10])[1][2]) - cc.REC_FIXED
    beacon_off = r2 + cc.REC_FIXED + n_params - 1       # last byte of the beacon hash
    bad = _off_subgroup_g2()
    return [
        ("transcript", _edit(k, 10, _flip(r0 + 320)), "INVALID(0): Inconsistent transcript"),
        ("g1_sx", _edit(k, 10, lambda b: _dbl_g1(b, r0 + 128)), "INVALID(0): Inconsistent transcript"),
        ("deltaAfter", _edit(k, 10, lambda b: _dbl_g1(b, r0)), "INVALID(0): deltaAfter does not fillow the public key"),
        ("beacon hash", _edit(k, 10, _flip(beacon_off)), "INVALID(2): Key of the beacon does not match. g1_s"),
        ("alpha1", _edit(k, 2, lambda b: _dbl_g1(b, 84)), "Invalid alpha1"),
        ("delta1", _edit(k, 2, lambda b: _dbl_g1(b, 468)), "Invalid delta1"),
        ("delta2", _edit(k, 2, lambda b: _dbl_g2(b, 532)), "Invalid delta2"),
        ("delta2 off subgroup", _edit(k, 2, _set(532, g2_to_bytes_mont(bad))),
         "zkey: header delta2 is not in the order-r subgroup of G2"),
        ("g2_spx off subgroup", _edit(k, 10, _set(r0 + 192, g2_to_bytes_mont(bad))),
         "zkey: section 10 record 0 g2_spx is not in the order-r subgroup of G2"),
        ("csHash", _edit(k, 10, _flip(3)), "INVALID(0): Inconsistent transcript"),
        ("csHash, no contributions", _edit(ch["init"], 10, _flip(3)), "Circuit does not match"),
        ("IC", _edit(k, 3, lambda b: _dbl_g1(b, 64)), "IC section is not identical"),
        ("coefficient", _edit(k, 4, _flip(4 + 12)), "Coeffs section is not identical"),
        ("A", _edit(k, 5, _flip(70)), "A section is not identical"),
        ("B1", _edit(k, 6, _flip(70)), "B1 section is not identical"),
        ("B2", _edit(k, 7, _flip(130)), "B2 section is not identical"),
        ("L", _edit(k, 8, lambda b: _dbl_g1(b, 64)), "L section does not match"),
        ("H", _edit(k, 9, _swap_h), "H section does not match"),
    ]


def test_tampered_keys(chain):
    for name, key, msg in _tampered(chain):
        for res in _both(chain, key):
            assert not res["ok"] and res["message"] == msg, (name, res["message"])


def test_key_of_another_r1cs(chain):
    other = _r1cs(12)
    res = api.zkey_verify(chain["keys"][-1], chain["ptau"], r1cs=other)
    assert not res["ok"] and res["message"] in ("Circuit does not match", "Different circuit parameters")


def test_independent_of_the_seed(chain):
    t = {name: key for name, key, _ in _tampered(chain)}
    for seed in SEEDS:
        assert api.zkey_verify(chain["keys"][-1], chain["ptau"], init=chain["init"], seed=seed)["ok"]
        assert not api.zkey_verify(t["L"], chain["ptau"], init=chain["init"], seed=seed)["ok"]
        assert not api.zkey_verify(t["H"], chain["ptau"], init=chain["init"], seed=seed)["ok"]


def test_domain_1024_cir_power_equals_power(lib):
    """cirPower = power = 10 (N <= 2^14: hashHPoints stays inside section 2), H read from snarkjs's top tauG1 level."""
    r1cs = _r1cs(13, n_constraints=1000, n_public=3, n_free=12)
    raw = ptau.write_ptau(TOX["tau"], TOX["alpha"], TOX["beta"], 10, prepared=False)
    prepared = bytes(groth16.powersOfTau.preparePhase2(raw, None))
    init, keys, _ = _chain(r1cs, prepared)
    assert formats.read_zkey_header(init)[0]["domainSize"] == 1024
    assert api.zkey_circuit_hash(init, prepared) == vc.circuit_hash(init, prepared)
    assert api.zkey_verify(keys[-1], prepared, r1cs=r1cs)["ok"]
    assert api.zkey_verify(keys[-1], prepared, init=init)["ok"]


def test_nzcp_shape(lib):
    """ptau power 21 of random points -> preparePhase2 -> newZKey(circuit_hash) -> contribute -> beacon: verifies from the
    r1cs; one altered L point or H point fails."""
    ch = nzcp_chain()
    res = api.zkey_verify(ch["key"], ch["ptau"], r1cs=ch["r1cs"])
    assert res["ok"], res["message"]
    assert [c["hash"] for c in res["contributions"]] == ch["hashes"]
    k = ch["key"]
    for sid, msg in ((8, "L section does not match"), (9, "H section does not match")):
        bad = _edit(k, sid, lambda b: _dbl_g1(b, 64 * 1000))
        res = api.zkey_verify(bad, ch["ptau"], r1cs=ch["r1cs"])
        assert not res["ok"] and res["message"] == msg
    groth16.terminate()
