"""`powersoftau prepare phase2` on the GPU (csrc/ptau.cu) against the oracle's closed forms.

The input ptau is written by the oracle from a KNOWN (tau, alpha, beta) without sections 12-15; the prepared file the
library computes from it must equal, byte for byte, the one the oracle writes with every Lagrange point as a scalar times
the generator (snarkjs's convention for the top tauG1 level: tests/ptau_cases.py write_prepared).  At power 20 the levels are
checked through random linear combinations with the variable-base MSM and the C oracle's NTT, code paths independent of
the new kernels.  Then the prepared file goes through `zkey new` and a proof.
"""
import os
import struct

import numpy as np
import pytest

import ptau_cases
from nzcp_circom_b200 import api, groth16
from oracle import cref, formats, ptau
from oracle.bn254 import FR_W, G1, G1_GEN, Q_MOD, R_MOD, FixedBase, g1_to_bytes_mont, to_le32

pytestmark = pytest.mark.gpu

TOX = {"tau": 0x5EED5EED5EED, "alpha": 0xA1A1A1, "beta": 0xB2B2B2B2, "gamma": 1, "delta": 1}


def _sections(buf, magic=b"ptau"):
    _, secs = formats.read_container(buf, magic)
    order = [sid for sid, _ in sorted(((sid, v[0][0]) for sid, v in secs.items()), key=lambda x: x[1])]
    return {sid: bytes(memoryview(buf)[v[0][0]:v[0][0] + v[0][1]]) for sid, v in secs.items()}, order


@pytest.fixture(scope="module")
def raw11():
    return ptau.write_ptau(TOX["tau"], TOX["alpha"], TOX["beta"], 11, prepared=False)


@pytest.mark.parametrize("power", [1, 2, 5, 8, 11])
def test_prepare_byte_exact(lib, raw11, power):
    raw = raw11 if power == 11 else ptau.write_ptau(TOX["tau"], TOX["alpha"], TOX["beta"], power, prepared=False)
    timings = {}
    got = api.ptau_prepare(raw, timings=timings)
    assert sorted(timings) == [12, 13, 14, 15] and all(t > 0 for t in timings.values())
    gs, order = _sections(got)
    rs, _ = _sections(raw)
    assert order == [1, 2, 3, 4, 5, 6, 7, 12, 13, 14, 15]
    for sid in range(1, 8):
        assert gs[sid] == rs[sid], sid
    if power <= 8:
        assert got == ptau_cases.write_prepared(TOX["tau"], TOX["alpha"], TOX["beta"], power)
    else:
        # power 11: the two largest G1 levels in closed form (the whole file is compared at power <= 8; every level of
        # every section is compared at power 20 below)
        fb = FixedBase(G1, G1_GEN)
        n = 1 << power
        for lg, xs in ((power + 1, ptau_cases.lagrange_top_snarkjs(TOX["tau"], power + 1)),
                       (power, ptau_cases.lagrange_any(TOX["tau"], power))):
            off = ((1 << lg) - 1) * 64
            idx = list(range(0, 1 << lg, 37)) + [(1 << lg) - 1]
            for i in idx:
                assert gs[12][off + 64 * i:off + 64 * i + 64] == g1_to_bytes_mont(fb.mul(xs[i])), (lg, i)
        assert len(gs[13]) == (2 * n - 1) * 128


DEGENERATE = [("tau0", 0, TOX["alpha"]), ("tau1", 1, TOX["alpha"]), ("tau-1", R_MOD - 1, TOX["alpha"]),
              ("omega3", FR_W[3], TOX["alpha"]), ("omega5", FR_W[5], TOX["alpha"]), ("alpha0", TOX["tau"], 0)]


@pytest.mark.parametrize("name,tau,alpha", DEGENERATE)
def test_prepare_degenerate_ceremonies(lib, name, tau, alpha):
    """Infinity inputs, equal operands (doubling) and cancellations inside butterflies."""
    raw = ptau.write_ptau(tau, alpha, TOX["beta"], 5, prepared=False)
    assert api.ptau_prepare(raw) == ptau_cases.write_prepared(tau, alpha, TOX["beta"], 5)


def test_prepare_idempotent(lib):
    raw = ptau.write_ptau(TOX["tau"], TOX["alpha"], TOX["beta"], 5, prepared=False)
    once = api.ptau_prepare(raw)
    assert api.ptau_prepare(once) == once
    # an input whose sections 12-15 are wrong (the exact top level) gives the same bytes too
    assert api.ptau_prepare(ptau.write_ptau(TOX["tau"], TOX["alpha"], TOX["beta"], 5)) == once


def _synth_ptau(power):
    n = 1 << power
    secs = [(1, struct.pack("<I", 32) + to_le32(Q_MOD) + struct.pack("<II", power, power))]
    secs.append((2, bytes(api.synth_points(101, 2 * n - 1))))
    secs.append((3, bytes(api.synth_points(102, n, g2=True))))
    secs.append((4, bytes(api.synth_points(103, n))))
    secs.append((5, bytes(api.synth_points(104, n))))
    secs.append((6, bytes(api.synth_points(105, 1, g2=True))))
    secs.append((7, bytes(4)))
    return formats.write_container(b"ptau", 1, secs)


def _rand_scalars(n, rs):
    x = rs.randint(0, 2 ** 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    x[:, 7] &= 0x1FFFFFFF
    return x


def test_prepare_power20_every_level(lib):
    """msm(level_out, rho) == msm(input prefix, ifft(rho)) for every level of every section (the iDFT matrix is
    symmetric); the top tauG1 prefix carries its infinity pad."""
    power = 20
    raw = _synth_ptau(power)
    got = api.ptau_prepare(raw)
    gs, _ = _sections(got)
    rs_, _ = _sections(raw)
    rs = np.random.RandomState(20)
    thr = cref.max_threads()
    for sid, src, g2, top in ((12, 2, False, power + 1), (13, 3, True, power), (14, 4, False, power), (15, 5, False, power)):
        psz = 128 if g2 else 64
        srcb = rs_[src] + bytes(psz) if sid == 12 else rs_[src]
        for lg in range(top + 1):
            n = 1 << lg
            lvl = gs[sid][(n - 1) * psz:(2 * n - 1) * psz]
            rho = _rand_scalars(n, rs)
            y = rho.copy()
            cref.ntt(y, lg, inverse=True, threads=thr)     # linear: raw integers in, raw integers out
            lhs, _ = api.msm_var(lvl, rho, n, g2=g2)
            rhs, _ = api.msm_var(srcb[:n * psz], y, n, g2=g2)
            assert lhs == rhs, (sid, lg)


def test_prepare_end_to_end_zkey(lib, raw11):
    """Power 11 = cirPower: zkey new reads the snarkjs top level for section 9; proofs do not change.  Power 12: the
    whole key equals the synthetic setup's."""
    sc = api.SynthCircuit(seed=77, n_constraints=1500, n_public=9, n_free=40)
    r1cs = sc.r1cs()
    want = sc.zkey([TOX[k] for k in ("tau", "alpha", "beta", "gamma", "delta")])
    ws, _ = _sections(want, b"zkey")
    prepared = api.ptau_prepare(raw11)
    got = api.zkey_new(r1cs, prepared)
    gs, _ = _sections(got, b"zkey")
    for sid in range(1, 9):
        assert gs[sid] == ws[sid], sid
    n = sc.domain_size
    assert n == 2048
    fb = FixedBase(G1, G1_GEN)
    lp = ptau_cases.lagrange_top_snarkjs(TOX["tau"], 12)
    assert gs[9] == b"".join(g1_to_bytes_mont(fb.mul(lp[2 * i + 1])) for i in range(n))
    wt = sc.wtns(5)
    r, s = 0x1357, 0x2468
    p_got = groth16.prove({"type": "mem", "data": got}, {"type": "mem", "data": wt}, r=r, s=s)
    p_want = groth16.prove({"type": "mem", "data": want}, {"type": "mem", "data": wt}, r=r, s=s)
    assert p_got == p_want
    assert groth16.verify(groth16.exportVerificationKey(got), p_got["publicSignals"], p_got["proof"])
    groth16.terminate()
    raw12 = ptau.write_ptau(TOX["tau"], TOX["alpha"], TOX["beta"], 12, prepared=False)
    g12, _ = _sections(api.zkey_new(r1cs, api.ptau_prepare(raw12)), b"zkey")
    for sid in range(1, 10):
        assert g12[sid] == ws[sid], sid


def test_prepare_phase2_outputs(lib, tmp_path):
    raw = ptau.write_ptau(TOX["tau"], TOX["alpha"], TOX["beta"], 3, prepared=False)
    want = ptau_cases.write_prepared(TOX["tau"], TOX["alpha"], TOX["beta"], 3)
    src = tmp_path / "in.ptau"
    src.write_bytes(raw)
    dst = tmp_path / "out.ptau"
    assert groth16.powersOfTau.preparePhase2(str(src), str(dst)) == want
    assert dst.read_bytes() == want
    mem = {"type": "mem"}
    assert groth16.powersOfTau.preparePhase2({"type": "mem", "data": raw}, mem) == want
    assert mem["data"] == want
    assert groth16.powersOfTau.preparePhase2(raw) == want
    assert os.path.getsize(src) == len(raw)
