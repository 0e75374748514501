"""`zkey contribute` / `zkey beacon` without a GPU: the test helper's primitives against RFC 8439 and the curve, the
kernel's per-point code run on the CPU (nzcp_host_zkey_contribute) byte for byte against the helper's closed-form key,
the size function, every rejection through the three entry points, and malformed containers."""
import ctypes as C
import random
import struct

import pytest

import contribution_cases as cc
import util
from nzcp_circom_b200 import _lib, api, groth16, verifier
from nzcp_circom_b200._lib import NzcpError
from oracle import formats, setup
from oracle.bn254 import G1, G1_GEN, Q_MOD, R_MOD, to_le32

SEED = bytes(range(32))
BEACON = bytes.fromhex("0123456789abcdef")


def test_chacha_rfc8439_block():
    """RFC 8439 2.3.2: key 00..1f, counter 1, nonce 00:00:00:09:00:00:00:4a:00:00:00:00."""
    key = [int.from_bytes(bytes(range(4 * i, 4 * i + 4)), "little") for i in range(8)]
    out = cc.chacha_block(cc.CONSTANTS + key + [1, 0x09000000, 0x4A000000, 0])
    assert b"".join(w.to_bytes(4, "little") for w in out).hex() == (
        "10f1e7e4d13b5915500fdd1fa32071c4c7d1f4c733c068030422aa9ac3d46c4e"
        "d2826446079faa0914c2d705d98b02a2b5129cd1de164eb9cbd083e8a2503c4e")


@pytest.mark.parametrize("seed", [SEED, bytes(32), b"\xff" * 32])
def test_helper_points(seed):
    rng = cc.rng_contribute(seed)
    k = cc.from_rng(rng, R_MOD)
    assert 0 < k < R_MOD
    g1_s = cc.g1_from_rng(rng)
    assert G1.on_curve(g1_s)
    g2_sp = cc.hash_to_g2(seed * 2)
    assert verifier.g2_on_curve(g2_sp) and verifier.g2_in_subgroup(g2_sp)


# ------------------------------------------------------------------------------------------------ keys
def _case(seed, n_constraints=12, n_public=2, n_free=4, unused_wire=False):
    c = util.tiny_case(seed, n_constraints, n_public, n_free)
    if unused_wire:       # one more private wire in no constraint: its L point is infinity
        c["n_vars"] += 1
        c["witness"] = c["witness"] + [7]
        c["zkey"] = setup.make_zkey(c["constraints"], c["n_vars"], c["n_public"], c["toxic"])
        c["zkey_bytes"] = formats.write_zkey(c["zkey"])
        assert c["zkey"]["C"][-1] is None
    return c


def expected_key(case, delta, s10):
    tox = dict(case["toxic"], delta=delta)
    return cc.with_section10(formats.write_zkey(setup.make_zkey(case["constraints"], case["n_vars"], case["n_public"], tox)),
                             s10)


def _size(buf, name=None, beacon_len=0):
    size = C.c_size_t()
    _lib.check(_lib.load().nzcp_zkey_contribute_size(_lib.addr(buf), len(buf), name.encode() if name else None, beacon_len,
                                                     C.byref(size)))
    return size.value


STEPS = {"contribute": dict(seed=SEED), "contribute_named": dict(seed=SEED, name="alice"),
         "beacon10": dict(beacon_hash=BEACON, exp=10), "beacon11_named": dict(beacon_hash=BEACON, exp=11, name="final")}


def run_host(zkey, step):
    return api.host_zkey_contribute(zkey, name=step.get("name"), seed=step.get("seed"), beacon_hash=step.get("beacon_hash"),
                                    num_iterations_exp=step.get("exp", 0))


def apply_and_check(case, zkey, delta, step, runner=run_host):
    """Run one step, compare with the helper: bytes, hash, size.  -> (new key, new delta)"""
    exp = cc.contribution(zkey, name=step.get("name"), seed=step.get("seed"), beacon_hash=step.get("beacon_hash"),
                          exp=step.get("exp"))
    got, h = runner(zkey, step)
    delta = delta * exp["k"] % R_MOD
    want = expected_key(case, delta, exp["s10"])
    if bytes(got) != want:
        gs, ws = cc.sections(bytes(got)), cc.sections(want)
        assert [s for s in ws if gs.get(s) != ws[s]] == []
    assert bytes(got) == want
    assert h == exp["hash"]
    assert _size(zkey, step.get("name"), len(step.get("beacon_hash", b""))) == len(want)
    return bytes(got), delta


@pytest.mark.parametrize("step", sorted(STEPS))
def test_host_matches_helper(lib, step):
    case = _case(3)
    apply_and_check(case, case["zkey_bytes"], case["toxic"]["delta"], STEPS[step])


def test_host_l_point_at_infinity(lib):
    case = _case(4, unused_wire=True)
    got, _ = apply_and_check(case, case["zkey_bytes"], case["toxic"]["delta"], STEPS["contribute"])
    assert cc.sections(got)[8][-64:] == bytes(64)


def prior_beacon_key(case):
    """A key that already holds a helper-made named beacon record."""
    exp = cc.contribution(case["zkey_bytes"], name="earlier", beacon_hash=b"\x42" * 5, exp=10)
    delta = case["toxic"]["delta"] * exp["k"] % R_MOD
    return expected_key(case, delta, exp["s10"]), delta


CHAIN = [dict(seed=SEED, name="first"), dict(seed=bytes(range(32, 64))), dict(beacon_hash=BEACON, exp=10, name="beacon")]


def test_host_chain(lib):
    case = _case(5)
    zkey, delta = prior_beacon_key(case)
    for step in CHAIN:
        zkey, delta = apply_and_check(case, zkey, delta, step)
    _, recs = cc.parse_mpc(cc.sections(zkey)[10])
    assert [cc.record_points(r)["type"] for r in recs] == [1, 0, 0, 1]


def test_same_seed_same_bytes(lib):
    zk = _case(3)["zkey_bytes"]
    a, ha = api.host_zkey_contribute(zk, seed=SEED)
    b, hb = api.host_zkey_contribute(zk, seed=SEED)
    c, hc = api.host_zkey_contribute(zk, seed=bytes(32))
    assert a == b and ha == hb
    assert a != c and ha != hc
    d, hd = api.host_zkey_contribute(zk, entropy="some entropy")        # OS randomness: a different key each time
    assert d != a and len(d) == len(a) and hd != ha


# ------------------------------------------------------------------------------------------------ rejections
def _rebuild(buf, edit):
    secs = cc.sections(buf)
    edit(secs)
    return formats.write_container(b"zkey", 1, sorted(secs.items()))


def _set(sid, val):
    return lambda s: s.__setitem__(sid, val)


def _file_rejections(zk):
    """(name, file, code, message fragment): rejected by the size function, both compute entries and the host hook."""
    secs = cc.sections(zk)
    h = secs[2]
    out = [("magic", b"ptau" + zk[4:], _lib.NZCP_E_FORMAT, "Invalid File format"),
           ("no header", _rebuild(zk, lambda s: s.pop(1)), _lib.NZCP_E_FORMAT, "missing header"),
           ("plonk", _rebuild(zk, _set(1, struct.pack("<I", 2))), _lib.NZCP_E_NOT_GROTH16, "zkey file is not groth16"),
           ("header short", _rebuild(zk, _set(2, h[:-4])), _lib.NZCP_E_FORMAT, "not 660 bytes"),
           ("header long", _rebuild(zk, _set(2, h + bytes(4))), _lib.NZCP_E_FORMAT, "not 660 bytes"),
           ("curve", _rebuild(zk, _set(2, h[:4] + bytes([h[4] ^ 1]) + h[5:])), _lib.NZCP_E_CURVE, "curve is not bn128"),
           ("L short", _rebuild(zk, _set(8, secs[8][:-64])), _lib.NZCP_E_FORMAT, "section 8 size"),
           ("H long", _rebuild(zk, _set(9, secs[9] + bytes(64))), _lib.NZCP_E_FORMAT, "section 9 size"),
           ("s10 truncated", _rebuild(zk, _set(10, secs[10][:-1])), _lib.NZCP_E_FORMAT, "section 10 is truncated"),
           ("s10 trailing", _rebuild(zk, _set(10, secs[10] + b"\0")), _lib.NZCP_E_FORMAT, "trailing bytes")]
    for sid in range(2, 11):
        out.append(("missing%d" % sid, _rebuild(zk, lambda s, sid=sid: s.pop(sid)), _lib.NZCP_E_FORMAT,
                    "Missing section %d" % sid))
    # section 10 parameters: a record with hand-made parameter bytes
    cs, recs = cc.parse_mpc(secs[10])
    base = recs[0][:cc.REC_FIXED - 4]
    for nm, params, msg in (("unsorted", bytes([2, 10, 1, 1, 65]), "Parameters in the contribution must be sorted"),
                            ("repeated", bytes([1, 1, 65, 1, 1, 66]), "Parameters in the contribution must be sorted"),
                            ("unknown", bytes([4, 0]), "Parameter not recognized"),
                            ("overrun", bytes([1, 5, 65]), "Parametes do not match")):
        rec = base + struct.pack("<I", len(params)) + params
        tail = bytes(8) if nm == "overrun" else b""       # the name reads past paramLength, not past the section
        out.append((nm, _rebuild(zk, _set(10, cs + struct.pack("<I", 1) + rec + tail)), _lib.NZCP_E_FORMAT, msg))
    # points: a coordinate >= q, a point off the curve, in L, H, delta1 and delta2
    P = G1.mul(G1_GEN, 9)
    off = to_le32(P[0] * (1 << 256) % Q_MOD) + to_le32((P[1] + 1) * (1 << 256) % Q_MOD)
    for sid in (8, 9):
        out.append(("noncanon%d" % sid, _rebuild(zk, _set(sid, to_le32(Q_MOD) + secs[sid][32:])), _lib.NZCP_E_RANGE,
                    "section %d point 0 has a coordinate >= q" % sid))
        out.append(("offcurve%d" % sid, _rebuild(zk, _set(sid, secs[sid][:-64] + off)), _lib.NZCP_E_RANGE,
                    "section %d point %d is not on the curve" % (sid, len(secs[sid]) // 64 - 1)))
    out.append(("delta1", _rebuild(zk, _set(2, h[:468] + off + h[532:])), _lib.NZCP_E_RANGE, "is not on the curve"))
    out.append(("delta2", _rebuild(zk, _set(2, h[:532] + to_le32(Q_MOD) + h[564:])), _lib.NZCP_E_RANGE, ">= q"))
    return out


@pytest.fixture(scope="module")
def named_key():
    return prior_beacon_key(_case(6))[0]


N_FILE = 29


def test_rejection_count(lib, named_key):
    assert len(_file_rejections(named_key)) == N_FILE


def _raises(fn, code, msg):
    with pytest.raises(NzcpError) as e:
        fn()
    assert e.value.code == code, (e.value.code, str(e.value))
    assert msg in str(e.value), str(e.value)


@pytest.mark.parametrize("case", range(N_FILE))
def test_file_rejections(lib, named_key, case):
    """Each rejection gives its code and message through the size function, the compute entries and the host hook,
    before any device work."""
    name, buf, code, msg = _file_rejections(named_key)[case]
    for fn in (lambda: _size(buf), lambda: api.zkey_contribute(buf, seed=SEED), lambda: api.zkey_beacon(buf, BEACON, 10),
               lambda: api.host_zkey_contribute(buf, seed=SEED), lambda: api.host_zkey_contribute(buf, beacon_hash=BEACON,
                                                                                                 num_iterations_exp=10)):
        _raises(fn, code, msg)


ARG_REJECTIONS = [
    ("long name", dict(name="n" * 65), "longer than 64 bytes"),
    ("long name utf8", dict(name="é" * 33), "longer than 64 bytes"),
    ("beacon empty", dict(beacon_hash=b""), "Invalid Beacon Hash. (It must be a valid hexadecimal sequence)"),
    ("beacon 256", dict(beacon_hash=bytes(256)), "Maximum lenght of beacon hash is 255 bytes"),
    ("exp 9", dict(beacon_hash=BEACON, exp=9), "Invalid numIterationsExp. (Must be between 10 and 63)"),
    ("exp 64", dict(beacon_hash=BEACON, exp=64), "Invalid numIterationsExp. (Must be between 10 and 63)"),
]


@pytest.mark.parametrize("case", range(len(ARG_REJECTIONS)))
def test_argument_rejections(lib, named_key, case):
    name, a, msg = ARG_REJECTIONS[case]
    zk = named_key
    fns = [lambda: api.host_zkey_contribute(zk, name=a.get("name"), seed=SEED, beacon_hash=a.get("beacon_hash"),
                                            num_iterations_exp=a.get("exp", 10))]
    if "beacon_hash" in a:
        fns.append(lambda: api.zkey_beacon(zk, a["beacon_hash"], a.get("exp", 10)))
    else:
        fns.append(lambda: api.zkey_contribute(zk, name=a["name"], seed=SEED))
    if "exp" not in a and a.get("beacon_hash") != b"":
        fns.append(lambda: _size(zk, a.get("name"), len(a.get("beacon_hash", b""))))
    for fn in fns:
        _raises(fn, _lib.NZCP_E_ARG, msg)


def test_name_of_64_bytes_is_kept(lib, named_key):
    got, _ = api.host_zkey_contribute(named_key, name="é" * 32, seed=SEED)
    _, recs = cc.parse_mpc(cc.sections(bytes(got))[10])
    assert recs[-1][cc.REC_FIXED:] == bytes([1, 64]) + ("é" * 32).encode()


def test_host_hook_size_limit(lib):
    zk = _case(7, n_constraints=2100, n_public=1, n_free=8)["zkey_bytes"]     # 2^12 H points + L > 4096
    _raises(lambda: api.host_zkey_contribute(zk, seed=SEED), _lib.NZCP_E_ARG, "4096 points")


def test_compute_needs_a_device(lib, named_key):
    """No CPU fallback: a valid key reaches the device check and fails there."""
    if api.device_count() > 0:
        pytest.skip("GPU present")
    _raises(lambda: api.zkey_contribute(named_key, seed=SEED), _lib.NZCP_E_CUDA, "no CUDA device")
    _raises(lambda: api.zkey_beacon(named_key, BEACON, 10), _lib.NZCP_E_CUDA, "no CUDA device")


def test_groth16_beacon_hex_check(lib, named_key):
    for bad in ("", "0", "zz", "12 3"):
        _raises(lambda: groth16.zKey.beacon(named_key, None, "x", bad, 10), _lib.NZCP_E_ARG,
                "Invalid Beacon Hash. (It must be a valid hexadecimal sequence)")


ALLOWED = {_lib.NZCP_OK, -1, -2, -3, -4, -5, -6, -7}


def test_fuzz_zkey_contribute(lib, named_key):
    """Truncations, bit flips and poked 32-bit fields never crash the parser; every outcome is a documented code."""
    L = _lib.load()
    rng = random.Random(2025)
    base = named_key
    n = len(base)
    s10 = formats.read_container(base, b"zkey")[1][10][0][0]
    size, written = C.c_size_t(), C.c_size_t()
    out = bytearray(n + 4096)
    h = bytearray(64)
    for it in range(400):
        b = bytearray(base)
        kind = it % 5
        if kind == 0:
            b = b[:rng.randrange(0, n)]
        elif kind == 1:
            i = rng.randrange(0, min(n, 700))
            b[i] ^= 1 << rng.randrange(8)
        elif kind == 2:
            i = rng.randrange(0, n - 4)
            struct.pack_into("<I", b, i, rng.choice([0, 1, 2, 10, 0x7FFFFFFF, 0xFFFFFFFF, 0x80000000, n, n + 1]))
        elif kind == 3:                                   # inside section 10: counts, lengths, tags
            i = rng.randrange(s10, n)
            b[i] = rng.choice([0, 1, 2, 3, 4, 0xFF, b[i] ^ 0x10])
        else:
            i = rng.randrange(0, n)
            b[i] ^= 1 << rng.randrange(8)
        b = bytes(b)
        assert L.nzcp_zkey_contribute_size(_lib.addr(b), len(b), None, 0, C.byref(size)) in ALLOWED
        assert L.nzcp_host_zkey_contribute(_lib.addr(b), len(b), None, None, 0, SEED, None, 0, 0, _lib.addr(out), len(out),
                                           C.byref(written), _lib.addr(h)) in ALLOWED
