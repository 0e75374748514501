"""`powersoftau new` / `contribute` / `beacon` without a GPU: the test helper's BLAKE2b, first challenge hash and
compressed encoding against hashlib and the curve, the kernels' per-point code run on the CPU (nzcp_host_ptau_contribute)
byte for byte against the helper's closed-form file, the pairing checks `powersoftau verify` runs on every record, the
size functions, every rejection through every entry point, and malformed containers."""
import ctypes as C
import hashlib
import random
import struct

import pytest

import ptau_cases
import ptau_contribution_cases as pc
from nzcp_circom_b200 import _lib, api, groth16, verifier
from nzcp_circom_b200._lib import NzcpError
from oracle import formats, ptau
from oracle.bn254 import G1, G1_GEN, G2, G2_GEN, Q_MOD, to_le32

SEED = bytes(range(32))
BEACON = bytes.fromhex("0123456789abcdef")
TAU, ALPHA, BETA = 0x5EED5EED5EED, 0xA1A1A1, 0xB2B2B2B2


# ------------------------------------------------------------------------------------------------ helper primitives
@pytest.mark.parametrize("n", [0, 1, 127, 128, 129, 256, 1000])
def test_blake2b_matches_hashlib(n):
    data = bytes((7 * i + 3) & 0xFF for i in range(n))
    assert pc.Blake2b().update(data).digest() == hashlib.blake2b(data, digest_size=64).digest()


@pytest.mark.parametrize("cut", [0, 1, 64, 128, 129, 300, 384])
def test_blake2b_resumes_from_partial(cut):
    data = bytes((5 * i + 1) & 0xFF for i in range(700))
    h = pc.Blake2b().update(data[:cut])
    p = h.partial()
    assert len(p) == 216 and struct.unpack_from("<II", p, 208) == (h.c, 64)
    assert pc.Blake2b.from_partial(p).update(data[cut:]).digest() == hashlib.blake2b(data, digest_size=64).digest()


@pytest.mark.parametrize("power", [1, 2, 3, 4])
def test_first_challenge_hash(lib, power):
    n = 1 << power
    g1, g2 = pc.u_g1(G1_GEN), pc.u_g2(G2_GEN)
    want = hashlib.blake2b(hashlib.blake2b(b"", digest_size=64).digest() + g1 * (2 * n - 1) + g2 * n + g1 * n + g1 * n + g2,
                           digest_size=64).digest()
    assert pc.first_challenge_hash(power) == want
    data, h = api.ptau_new(power)
    assert h == want
    assert bytes(data) == pc.new_file(power)
    assert api.ptau_new(power, first_challenge=False) == (data, None)
    size = C.c_size_t()
    _lib.check(_lib.load().nzcp_ptau_new_size(power, C.byref(size)))
    assert size.value == len(data)


def _sqrt_fq(a):
    y = pow(a, (Q_MOD + 1) // 4, Q_MOD)
    return y if y * y % Q_MOD == a else None


def test_compressed_encoding_decodes():
    for k in list(range(1, 40)) + [Q_MOD - 5, 2 ** 200 + 11]:
        P = G1.mul(G1_GEN, k)
        c = pc.c_g1(P)
        assert len(c) == 32 and (c[0] & 0x80 != 0) == (P[1] > (Q_MOD - 1) // 2)
        x = int.from_bytes(bytes([c[0] & 0x3F]) + c[1:], "big")
        y = _sqrt_fq((x ** 3 + 3) % Q_MOD)
        if (y > (Q_MOD - 1) // 2) != bool(c[0] & 0x80):
            y = Q_MOD - y
        assert (x, y) == P
        Q2 = G2.mul(G2_GEN, k)
        c2 = pc.c_g2(Q2)
        assert len(c2) == 64 and c2[:64] == bytes([c2[0]]) + Q2[0][1].to_bytes(32, "big")[1:] + Q2[0][0].to_bytes(32, "big")
        for y2 in (Q2[1], verifier.f2_neg(Q2[1])):
            neg = (y2[1] > (Q_MOD - 1) // 2) if y2[1] else (y2[0] > (Q_MOD - 1) // 2)
            assert (pc.c_g2((Q2[0], y2))[0] & 0x80 != 0) == neg
    assert pc.c_g1(None) == b"\x40" + bytes(31) and pc.c_g2(None) == b"\x40" + bytes(63)


# ------------------------------------------------------------------------------------------------ contributions
STEPS = {"contribute": dict(seed=SEED), "contribute_named": dict(seed=SEED, name="alice"),
         "beacon10": dict(beacon_hash=BEACON, exp=10), "beacon11_named": dict(beacon_hash=BEACON, exp=11, name="final")}


def run_host(buf, step):
    return api.host_ptau_contribute(buf, name=step.get("name"), seed=step.get("seed"), beacon_hash=step.get("beacon_hash"),
                                    num_iterations_exp=step.get("exp", 0))


def _size(buf, name=None, beacon_len=0):
    size = C.c_size_t()
    _lib.check(_lib.load().nzcp_ptau_contribute_size(_lib.addr(buf), len(buf), name.encode() if name else None, beacon_len,
                                                     C.byref(size)))
    return size.value


def apply_and_check(buf, state, step, runner=run_host, infinity=()):
    """Run one step and compare with the helper: bytes, response hash, partialHash, nextChallenge, size.
    state = (tau, alpha, beta) of `buf`.  -> (new file, new state, helper result)"""
    exp = pc.contribution(buf, *state, name=step.get("name"), seed=step.get("seed"), beacon_hash=step.get("beacon_hash"),
                          exp=step.get("exp"), infinity=infinity)
    got, h = runner(buf, step)
    if bytes(got) != exp["file"]:
        gs, ws = pc.sections(bytes(got)), pc.sections(exp["file"])
        assert [s for s in ws if gs.get(s) != ws[s]] == []
    assert bytes(got) == exp["file"]
    assert h == exp["response"]
    rec = pc.record_fields(pc.parse_records(pc.sections(bytes(got))[7])[-1])
    assert (rec["partial"], rec["next"]) == (exp["partial"], exp["next"])
    assert _size(buf, step.get("name"), len(step.get("beacon_hash", b""))) == len(got)
    return bytes(got), (exp["tau"], exp["alpha"], exp["beta"]), exp


@pytest.mark.parametrize("step", sorted(STEPS))
def test_host_from_new_matches_helper(lib, step):
    apply_and_check(bytes(api.ptau_new(3)[0]), (1, 1, 1), STEPS[step])


def prior_beacon_file(power=3):
    """write_ptau(TAU, ALPHA, BETA) after a helper-made named beacon record."""
    e = pc.contribution(ptau.write_ptau(TAU, ALPHA, BETA, power, prepared=False), TAU, ALPHA, BETA, name="earlier",
                        beacon_hash=b"\x42" * 5, exp=10)
    return e["file"], (e["tau"], e["alpha"], e["beta"])


CHAIN = [dict(seed=SEED, name="first"), dict(seed=bytes(range(32, 64))), dict(beacon_hash=BEACON, exp=10, name="beacon")]


def _pair_eq(p1, q1, p2, q2):
    """e(p1, q1) == e(p2, q2)"""
    return verifier.pairing_product_is_one([(p1, q1), (G1.neg(p2), q2)])


def check_record_pairings(prev, rec):
    """powersoftau verify's checks of one record against the previous file's first points `prev`."""
    tau, alpha, beta = rec["key"]
    sp = []
    for k, e in zip(rec["key"], hash_inputs(rec)):
        g2_sp = pc.cc.hash_to_g2(e)
        sp.append(g2_sp)
        assert _pair_eq(k["g1_s"], k["g2_spx"], k["g1_sx"], g2_sp)                  # sameRatio(g1_s, g1_sx, g2_sp, g2_spx)
    assert _pair_eq(prev["tauG1"], tau["g2_spx"], rec["tauG1"], sp[0])
    assert _pair_eq(tau["g1_s"], rec["tauG2"], tau["g1_sx"], prev["tauG2"])
    assert _pair_eq(prev["alphaG1"], alpha["g2_spx"], rec["alphaG1"], sp[1])
    assert _pair_eq(prev["betaG1"], beta["g2_spx"], rec["betaG1"], sp[2])
    assert _pair_eq(beta["g1_s"], rec["betaG2"], beta["g1_sx"], prev["betaG2"])


def hash_inputs(rec):
    return [hashlib.blake2b(bytes([j]) + rec["challenge"] + pc.u_g1(k["g1_s"]) + pc.u_g1(k["g1_sx"]), digest_size=64).digest()
            for j, k in enumerate(rec["key"])]


def first_points(buf):
    s = pc.sections(buf)
    g1, g2 = pc.g1_from_bytes_mont, pc.g2_from_bytes_mont
    return {"tauG1": g1(s[2][64:128]), "tauG2": g2(s[3][128:256]), "alphaG1": g1(s[4][:64]), "betaG1": g1(s[5][:64]),
            "betaG2": g2(s[6][:128])}


def run_chain(buf, state, runner=run_host):
    """CHAIN on `buf`; every record passes the pairing checks.  -> (file, state)"""
    for step in CHAIN:
        prev = first_points(buf)
        buf, state, exp = apply_and_check(buf, state, step, runner)
        rec = pc.record_fields(exp["record"])
        rec["challenge"] = exp["challenge"]
        check_record_pairings(prev, rec)
    types = [pc.record_fields(r)["type"] for r in pc.parse_records(pc.sections(buf)[7])]
    assert types == [1, 0, 0, 1]
    return buf, state


def test_host_chain(lib):
    run_chain(*prior_beacon_file())


def test_host_prepared_input(lib):
    """Sections 12-15 of a prepared input are dropped."""
    prepared = ptau_cases.write_prepared(TAU, ALPHA, BETA, 3)
    assert 12 in pc.sections(prepared)
    got, _, _ = apply_and_check(prepared, (TAU, ALPHA, BETA), STEPS["contribute_named"])
    assert sorted(pc.sections(got)) == list(range(1, 8))


def _with_infinity(buf, points):
    secs = pc.sections(buf)
    for sid, i in points:
        sz = 128 if sid in pc.G2_SECTIONS else 64
        secs[sid] = secs[sid][:sz * i] + bytes(sz) + secs[sid][sz * (i + 1):]
    return formats.write_container(b"ptau", 1, sorted(secs.items()))


def test_host_point_at_infinity(lib):
    inf = [(5, 2), (3, 5), (2, 14)]
    buf = _with_infinity(ptau.write_ptau(TAU, ALPHA, BETA, 3, prepared=False), inf)
    got, _, _ = apply_and_check(buf, (TAU, ALPHA, BETA), STEPS["contribute"], infinity=inf)
    assert pc.sections(got)[5][128:192] == bytes(64)


def test_same_seed_same_bytes(lib):
    f = bytes(api.ptau_new(2)[0])
    a, ha = api.host_ptau_contribute(f, seed=SEED)
    assert api.host_ptau_contribute(f, seed=SEED) == (a, ha)
    c, hc = api.host_ptau_contribute(f, seed=bytes(32))
    assert a != c and ha != hc
    d, hd = api.host_ptau_contribute(f, entropy="some entropy")        # OS randomness: a different key each time
    assert d != a and len(d) == len(a) and hd != ha


# ------------------------------------------------------------------------------------------------ rejections
def _rebuild(buf, edit):
    secs = pc.sections(buf)
    edit(secs)
    return formats.write_container(b"ptau", 1, sorted(secs.items()))


def _set(sid, val):
    return lambda s: s.__setitem__(sid, val)


def _file_rejections(f):
    """(name, file, code, message fragment): rejected by the size function, both compute entries and the host hook."""
    secs = pc.sections(f)
    h = secs[1]
    out = [("magic", b"zkey" + f[4:], _lib.NZCP_E_FORMAT, "Invalid File format"),
           ("no header", _rebuild(f, lambda s: s.pop(1)), _lib.NZCP_E_FORMAT, "missing header"),
           ("header short", _rebuild(f, _set(1, h[:43])), _lib.NZCP_E_FORMAT, "missing header"),
           ("curve", _rebuild(f, _set(1, h[:4] + bytes([h[4] ^ 1]) + h[5:])), _lib.NZCP_E_CURVE, "curve is not bn128"),
           ("n8", _rebuild(f, _set(1, struct.pack("<I", 48) + h[4:])), _lib.NZCP_E_CURVE, "curve is not bn128"),
           ("power 0", _rebuild(f, _set(1, h[:36] + struct.pack("<II", 0, 0))), _lib.NZCP_E_FORMAT, "power out of range"),
           ("power 29", _rebuild(f, _set(1, h[:36] + struct.pack("<II", 29, 29))), _lib.NZCP_E_FORMAT, "power out of range"),
           ("reduced", _rebuild(f, _set(1, h[:40] + struct.pack("<I", 4))), _lib.NZCP_E_ARG,
            "This file has been reduced. You cannot contribute into a reduced file."),
           ("tauG1 short", _rebuild(f, _set(2, secs[2][:-64])), _lib.NZCP_E_FORMAT, "section 2 size"),
           ("tauG2 long", _rebuild(f, _set(3, secs[3] + bytes(128))), _lib.NZCP_E_FORMAT, "section 3 size"),
           ("betaG2 short", _rebuild(f, _set(6, secs[6][:64])), _lib.NZCP_E_FORMAT, "section 6 size"),
           ("s7 truncated", _rebuild(f, _set(7, secs[7][:-1])), _lib.NZCP_E_FORMAT, "section 7 is truncated"),
           ("s7 short count", _rebuild(f, _set(7, secs[7][:3])), _lib.NZCP_E_FORMAT, "section 7 is truncated"),
           ("s7 trailing", _rebuild(f, _set(7, secs[7] + b"\0")), _lib.NZCP_E_FORMAT, "trailing bytes")]
    for sid in range(2, 8):
        out.append(("missing%d" % sid, _rebuild(f, lambda s, sid=sid: s.pop(sid)), _lib.NZCP_E_FORMAT,
                    "Missing section %d" % sid))
    rec = pc.parse_records(secs[7])[0]
    base = rec[:pc.REC_FIXED - 4]
    for nm, params, msg in (("unsorted", bytes([2, 10, 1, 1, 65]), "Parameters in the contribution must be sorted"),
                            ("repeated", bytes([1, 1, 65, 1, 1, 66]), "Parameters in the contribution must be sorted"),
                            ("unknown", bytes([4, 0]), "Parameter not recognized"),
                            ("overrun", bytes([1, 5, 65]), "Parametes do not match")):
        r = base + struct.pack("<I", len(params)) + params
        tail = bytes(8) if nm == "overrun" else b""
        out.append((nm, _rebuild(f, _set(7, struct.pack("<I", 1) + r + tail)), _lib.NZCP_E_FORMAT, msg))
    P = G1.mul(G1_GEN, 9)
    off = to_le32(P[0] * (1 << 256) % Q_MOD) + to_le32((P[1] + 1) * (1 << 256) % Q_MOD)
    for sid in (2, 4, 5):
        out.append(("noncanon%d" % sid, _rebuild(f, _set(sid, to_le32(Q_MOD) + secs[sid][32:])), _lib.NZCP_E_RANGE,
                    "section %d point 0 has a coordinate >= q" % sid))
        out.append(("offcurve%d" % sid, _rebuild(f, _set(sid, secs[sid][:-64] + off)), _lib.NZCP_E_RANGE,
                    "section %d point %d is not on the curve" % (sid, len(secs[sid]) // 64 - 1)))
    for sid in (3, 6):
        out.append(("noncanon%d" % sid, _rebuild(f, _set(sid, secs[sid][:96] + to_le32(Q_MOD) + secs[sid][128:])),
                    _lib.NZCP_E_RANGE, "section %d point 0 has a coordinate >= q" % sid))
        out.append(("offcurve%d" % sid, _rebuild(f, _set(sid, secs[sid][:-32] + to_le32(12345))), _lib.NZCP_E_RANGE,
                    "section %d point %d is not on the curve" % (sid, len(secs[sid]) // 128 - 1)))
    return out


@pytest.fixture(scope="module")
def named_file():
    return prior_beacon_file(2)[0]


N_FILE = 34


def test_rejection_count(lib, named_file):
    assert len(_file_rejections(named_file)) == N_FILE


def _raises(fn, code, msg):
    with pytest.raises(NzcpError) as e:
        fn()
    assert e.value.code == code, (e.value.code, str(e.value))
    assert msg in str(e.value), str(e.value)


@pytest.mark.parametrize("case", range(N_FILE))
def test_file_rejections(lib, named_file, case):
    """Each rejection gives its code and message through the size function, the compute entries and the host hook,
    before any device work."""
    name, buf, code, msg = _file_rejections(named_file)[case]
    for fn in (lambda: _size(buf), lambda: api.ptau_contribute(buf, seed=SEED), lambda: api.ptau_beacon(buf, BEACON, 10),
               lambda: api.host_ptau_contribute(buf, seed=SEED),
               lambda: api.host_ptau_contribute(buf, beacon_hash=BEACON, num_iterations_exp=10)):
        _raises(fn, code, msg)


ARG_REJECTIONS = [
    ("long name", dict(name="n" * 65), "ptau: contribution name longer than 64 bytes"),
    ("long name utf8", dict(name="é" * 33), "longer than 64 bytes"),
    ("beacon empty", dict(beacon_hash=b""), "Invalid Beacon Hash. (It must be a valid hexadecimal sequence)"),
    ("beacon 256", dict(beacon_hash=bytes(256)), "Maximum lenght of beacon hash is 255 bytes"),
    ("exp 9", dict(beacon_hash=BEACON, exp=9), "Invalid numIterationsExp. (Must be between 10 and 63)"),
    ("exp 64", dict(beacon_hash=BEACON, exp=64), "Invalid numIterationsExp. (Must be between 10 and 63)"),
]


@pytest.mark.parametrize("case", range(len(ARG_REJECTIONS)))
def test_argument_rejections(lib, named_file, case):
    name, a, msg = ARG_REJECTIONS[case]
    f = named_file
    fns = [lambda: api.host_ptau_contribute(f, name=a.get("name"), seed=SEED, beacon_hash=a.get("beacon_hash"),
                                            num_iterations_exp=a.get("exp", 10))]
    if "beacon_hash" in a:
        fns.append(lambda: api.ptau_beacon(f, a["beacon_hash"], a.get("exp", 10)))
    else:
        fns.append(lambda: api.ptau_contribute(f, name=a["name"], seed=SEED))
    if "exp" not in a and a.get("beacon_hash") != b"":
        fns.append(lambda: _size(f, a.get("name"), len(a.get("beacon_hash", b""))))
    for fn in fns:
        _raises(fn, _lib.NZCP_E_ARG, msg)


def test_new_rejections(lib):
    for p in (0, 29):
        _raises(lambda: api.ptau_new(p), _lib.NZCP_E_ARG, "power out of range [1, 28]")
    _raises(lambda: groth16.powersOfTau.newAccumulator("bls12381", 2, None), _lib.NZCP_E_CURVE, "Curve not supported")
    assert groth16.powersOfTau.newAccumulator(None, 2, None) == api.ptau_new(2)[1]
    out = {"type": "mem"}
    assert groth16.powersOfTau.newAccumulator("bn128", 2, out) == pc.first_challenge_hash(2)
    assert bytes(out["data"]) == pc.new_file(2)


def test_host_hook_power_limit(lib):
    _raises(lambda: api.host_ptau_contribute(api.ptau_new(5)[0], seed=SEED), _lib.NZCP_E_ARG, "limited to power 4")


def test_compute_needs_a_device(lib, named_file):
    """No CPU fallback: a valid file reaches the device check and fails there."""
    if api.device_count() > 0:
        pytest.skip("GPU present")
    _raises(lambda: api.ptau_contribute(named_file, seed=SEED), _lib.NZCP_E_CUDA, "no CUDA device")
    _raises(lambda: api.ptau_beacon(named_file, BEACON, 10), _lib.NZCP_E_CUDA, "no CUDA device")
    _raises(lambda: groth16.powersOfTau.contribute(named_file, None, "x", "", seed=SEED), _lib.NZCP_E_CUDA, "no CUDA device")


def test_groth16_beacon_hex_check(lib, named_file):
    for bad in ("", "0", "zz", "12 3"):
        _raises(lambda: groth16.powersOfTau.beacon(named_file, None, "x", bad, 10), _lib.NZCP_E_ARG,
                "Invalid Beacon Hash. (It must be a valid hexadecimal sequence)")


ALLOWED = {_lib.NZCP_OK, -1, -2, -4, -7}


def test_fuzz_ptau_contribute(lib, named_file):
    """Truncations, bit flips and poked 32-bit fields never crash the parser; every outcome is a documented code."""
    L = _lib.load()
    rng = random.Random(2026)
    base = named_file
    n = len(base)
    s7 = formats.read_container(base, b"ptau")[1][7][0][0]
    size, written = C.c_size_t(), C.c_size_t()
    out = bytearray(n + 4096)
    h = bytearray(64)
    for it in range(300):
        b = bytearray(base)
        kind = it % 5
        if kind == 0:
            b = b[:rng.randrange(0, n)]
        elif kind == 1:
            i = rng.randrange(0, min(n, 200))
            b[i] ^= 1 << rng.randrange(8)
        elif kind == 2:
            i = rng.randrange(0, n - 4)
            struct.pack_into("<I", b, i, rng.choice([0, 1, 2, 3, 28, 29, 0x7FFFFFFF, 0xFFFFFFFF, 0x80000000, n, n + 1]))
        elif kind == 3:                                   # inside section 7: counts, lengths, tags
            i = rng.randrange(s7, n)
            b[i] = rng.choice([0, 1, 2, 3, 4, 0xFF, b[i] ^ 0x10])
        else:
            i = rng.randrange(0, n)
            b[i] ^= 1 << rng.randrange(8)
        b = bytes(b)
        assert L.nzcp_ptau_contribute_size(_lib.addr(b), len(b), None, 0, C.byref(size)) in ALLOWED
        assert L.nzcp_host_ptau_contribute(_lib.addr(b), len(b), None, None, 0, SEED, None, 0, 0, _lib.addr(out), len(out),
                                           C.byref(written), _lib.addr(h)) in ALLOWED
