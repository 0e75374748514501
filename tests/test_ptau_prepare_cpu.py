"""`powersoftau prepare phase2` without a GPU: the oracle's group ifft against the closed forms, the size function, every
rejection of the input checks, malformed containers, and the kernels' load / stage / butterfly code run on the CPU
(nzcp_host_ptau_prepare) byte for byte against the oracle's prepared file."""
import ctypes as C
import random
import struct

import pytest

import ptau_cases
from nzcp_circom_b200 import _lib, api
from nzcp_circom_b200._lib import NzcpError
from oracle import formats, ptau, setup
from oracle.bn254 import FR_W, G1, G1_GEN, G2, G2_GEN, Q_MOD, R_MOD, fq_to_mont, to_le32

TAU, ALPHA, BETA = 0x5EED5EED5EED, 0xA1A1A1, 0xB2B2B2B2


def _raw(power, tau=TAU, alpha=ALPHA, beta=BETA):
    return ptau.write_ptau(tau, alpha, beta, power, prepared=False)


def _sections(buf, magic=b"ptau"):
    _, secs = formats.read_container(buf, magic)
    return {sid: bytes(memoryview(buf)[v[0][0]:v[0][0] + v[0][1]]) for sid, v in secs.items()}


def _rebuild(buf, edit):
    """Re-write a ptau container with edit(dict of sections) applied; sections keep ascending id order."""
    secs = _sections(buf)
    edit(secs)
    return formats.write_container(b"ptau", 1, sorted(secs.items()))


def _size(buf):
    size = C.c_size_t()
    _lib.check(_lib.load().nzcp_ptau_prepare_size(_lib.addr(buf), len(buf), C.byref(size)))
    return size.value


@pytest.mark.parametrize("log_n", [1, 2, 3])
def test_oracle_ifft_matches_closed_forms(log_n):
    """The definition-level group ifft of tau^j G is the Lagrange basis; with the last power replaced by infinity it is
    snarkjs's L' (the top tauG1 level)."""
    n = 1 << log_n
    pts = [G1.mul(G1_GEN, pow(TAU, j, R_MOD)) for j in range(n)]
    assert ptau_cases.ifft_points(G1, pts) == [G1.mul(G1_GEN, x) for x in ptau_cases.lagrange_any(TAU, log_n)]
    top = [G1.mul(G1_GEN, x) for x in ptau_cases.lagrange_top_snarkjs(TAU, log_n)]
    assert ptau_cases.ifft_points(G1, pts[:-1] + [None]) == top
    if log_n == 1:
        q = [G2.mul(G2_GEN, pow(TAU, j, R_MOD)) for j in range(n)]
        assert ptau_cases.ifft_points(G2, q) == [G2.mul(G2_GEN, x) for x in ptau_cases.lagrange_any(TAU, log_n)]


def test_oracle_lagrange_degenerate_tau():
    w = FR_W[3]
    assert ptau_cases.lagrange_any(pow(w, 5, R_MOD), 3) == [int(i == 5) for i in range(8)]
    assert ptau_cases.lagrange_any(TAU, 3) == setup.lagrange_at(TAU, 3)


@pytest.mark.parametrize("power", [1, 2, 3])
def test_write_prepared_matches_oracle(power):
    """The snarkjs-convention file differs from the oracle's exact prepared file in the top tauG1 level alone."""
    got = _sections(ptau_cases.write_prepared(TAU, ALPHA, BETA, power))
    exact = _sections(ptau.write_ptau(TAU, ALPHA, BETA, power))
    assert sorted(got) == sorted(exact) == [1, 2, 3, 4, 5, 6, 7, 12, 13, 14, 15]
    for sid in got:
        if sid != 12:
            assert got[sid] == exact[sid], sid
    top = ((2 << power) - 1) * 64
    assert got[12][:top] == exact[12][:top]
    assert got[12][top:] != exact[12][top:]


@pytest.mark.parametrize("power", [1, 2, 3, 4, 5, 6])
def test_size_matches_oracle(lib, power):
    raw = _raw(power, tau=3, alpha=5, beta=7)
    want = ptau_cases.write_prepared(3, 5, 7, power)
    assert _size(raw) == len(want)
    assert _size(want) == len(want)          # sections 12-15 of the input are ignored


def _g1_mont(x, y):
    return to_le32(fq_to_mont(x)) + to_le32(fq_to_mont(y))


def _rejections(raw):
    """(name, mutated file, code, message fragment)"""
    out = []
    out.append(("magic", b"zkey" + raw[4:], _lib.NZCP_E_FORMAT, "Invalid File format"))
    secs = _sections(raw)
    h = bytearray(secs[1])
    h[4] ^= 1
    out.append(("curve", _rebuild(raw, lambda s: s.__setitem__(1, bytes(h))), _lib.NZCP_E_CURVE, "curve is not bn128"))
    for pw, code, msg in ((0, _lib.NZCP_E_FORMAT, "power out of range"), (29, _lib.NZCP_E_FORMAT, "power out of range"),
                          (28, _lib.NZCP_E_ARG, "coset")):
        hp = bytearray(secs[1])
        struct.pack_into("<I", hp, 36, pw)
        out.append(("power%d" % pw, _rebuild(raw, lambda s, hp=hp: s.__setitem__(1, bytes(hp))), code, msg))
    out.append(("no header", _rebuild(raw, lambda s: s.pop(1)), _lib.NZCP_E_FORMAT, "missing header"))
    for sid in range(2, 8):
        out.append(("missing%d" % sid, _rebuild(raw, lambda s, sid=sid: s.pop(sid)), _lib.NZCP_E_FORMAT,
                    "Missing section %d" % sid))
    for sid in range(2, 7):
        out.append(("short%d" % sid, _rebuild(raw, lambda s, sid=sid: s.__setitem__(sid, s[sid][:-64])), _lib.NZCP_E_FORMAT,
                    "section %d size does not match" % sid))
        out.append(("long%d" % sid, _rebuild(raw, lambda s, sid=sid: s.__setitem__(sid, s[sid] + bytes(64))),
                    _lib.NZCP_E_FORMAT, "section %d size does not match" % sid))
    # a coordinate >= q (x = q itself, y anything), and a point off the curve (y + 1), in every point section
    for sid, size in ((2, 64), (3, 128), (4, 64), (5, 64), (6, 128)):
        def noncanon(s, sid=sid):
            b = bytearray(s[sid])
            b[0:32] = to_le32(Q_MOD)
            s[sid] = bytes(b)
        out.append(("noncanon%d" % sid, _rebuild(raw, noncanon), _lib.NZCP_E_RANGE,
                    "section %d point 0 has a coordinate >= q" % sid))

        def offcurve(s, sid=sid, size=size):
            b = bytearray(s[sid])
            i = len(b) // size - 1                            # the last point of the section
            P = G1.mul(G1_GEN, 9)
            b[i * size:i * size + 64] = _g1_mont(P[0], (P[1] + 1) % Q_MOD) if size == 64 else b[i * size:i * size + 64]
            if size == 128:
                b[i * size + 64] ^= 1                         # y.c0 of the Montgomery form: still < q, now off the twist
            s[sid] = bytes(b)
        out.append(("offcurve%d" % sid, _rebuild(raw, offcurve), _lib.NZCP_E_RANGE, "is not on the curve"))
    return out


@pytest.mark.parametrize("case", range(32))
def test_rejections(lib, case):
    """Each rejection gives its code and message from the size function, the compute entry and the host hook alike."""
    cases = _rejections(_raw(2))
    assert len(cases) == 32
    name, buf, code, msg = cases[case]
    for fn in (lambda: _size(buf), lambda: api.ptau_prepare(buf), lambda: api.host_ptau_prepare(buf)):
        with pytest.raises(NzcpError) as e:
            fn()
        assert e.value.code == code, (name, e.value.code, str(e.value))
        assert msg in str(e.value), (name, str(e.value))


def test_host_hook_power_limit(lib):
    with pytest.raises(NzcpError) as e:
        api.host_ptau_prepare(_raw(5, tau=3, alpha=5, beta=7))
    assert e.value.code == _lib.NZCP_E_ARG


def test_compute_needs_a_device(lib):
    """No CPU fallback: a valid file reaches the device check and fails there."""
    if api.device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(NzcpError) as e:
        api.ptau_prepare(_raw(2))
    assert e.value.code == _lib.NZCP_E_CUDA


ALLOWED = {_lib.NZCP_OK, -1, -2, -3, -4, -5, -6, -7}


def test_fuzz_ptau_prepare(lib):
    """Truncations, bit flips and poked 32-bit fields never crash the parser; every outcome is a documented code."""
    L = _lib.load()
    rng = random.Random(2024)
    base = _raw(2)
    n = len(base)
    size = C.c_size_t()
    out = bytearray(1 << 16)
    written = C.c_size_t()
    for it in range(400):
        b = bytearray(base)
        kind = it % 4
        if kind == 0:
            b = b[:rng.randrange(0, n)]
        elif kind == 1:
            i = rng.randrange(0, min(n, 400))
            b[i] ^= 1 << rng.randrange(8)
        elif kind == 2:
            i = rng.randrange(0, n - 4)
            struct.pack_into("<I", b, i, rng.choice([0, 1, 27, 28, 0x7FFFFFFF, 0xFFFFFFFF, 0x80000000, n, n + 1]))
        else:
            i = rng.randrange(0, n)
            b[i] ^= 1 << rng.randrange(8)
        b = bytes(b)
        assert L.nzcp_ptau_prepare_size(_lib.addr(b), len(b), C.byref(size)) in ALLOWED
        assert L.nzcp_host_ptau_prepare(_lib.addr(b), len(b), _lib.addr(out), len(out), C.byref(written)) in ALLOWED


DEGENERATE = {"generic": (TAU, ALPHA), "zero": (0, ALPHA), "one": (1, ALPHA), "minus_one": (R_MOD - 1, ALPHA),
              "omega": (FR_W[2], ALPHA), "alpha_zero": (TAU, 0)}


@pytest.mark.parametrize("power", [1, 2, 3, 4])
@pytest.mark.parametrize("name", sorted(DEGENERATE))
def test_host_hook_matches_oracle(lib, power, name):
    """The kernels' code on the CPU gives the oracle's snarkjs-convention prepared file, byte for byte: generic tau and
    the degenerate ceremonies whose butterflies meet infinity, doubling and cancellation."""
    tau, alpha = DEGENERATE[name]
    raw = _raw(power, tau=tau, alpha=alpha)
    got = api.host_ptau_prepare(raw)
    want = ptau_cases.write_prepared(tau, alpha, BETA, power)
    if got != want:
        gs, ws = _sections(got), _sections(want)
        assert sorted(gs) == sorted(ws)
        assert [s for s in gs if gs[s] != ws[s]] == []
    assert got == want
