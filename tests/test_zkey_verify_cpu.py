"""`zkey verify` and the circuit hash without a GPU: the H-check identity of the test helper at a known tau, the circuit
hash of the host hook (the kernels' per-point code on the CPU) byte for byte against the helper, every rejection through
every entry point, the size function, malformed containers, and no CPU fallback for the compute entries."""
import ctypes as C
import random
import struct

import pytest

import contribution_cases as cc
import util
import verify_cases as vc
from nzcp_circom_b200 import _lib, api
from oracle import formats, ptau
from oracle.bn254 import Q_MOD, R_MOD, to_le32
from test_zkey_contribute_cpu import SEED, _file_rejections, _raises, named_key  # noqa: F401  (fixture)

TOX = {"tau": 0x5EED5EED5EED, "alpha": 0xA1A1A1, "beta": 0xB2B2B2B2, "gamma": 1, "delta": 1}


# ------------------------------------------------------------------------------------------------ the helper
@pytest.mark.parametrize("log_n", [1, 2, 3])
def test_h_identity(log_n):
    """The identity the H check rests on, at a known tau: it holds on the exact Lagrange level for any r, and on snarkjs's
    top tauG1 level exactly when r_(N-1) = 0."""
    rng = random.Random(log_n)
    n = 1 << log_n
    tau = rng.randrange(2, R_MOD)
    r = [rng.randrange(R_MOD) for _ in range(n)]
    assert vc.h_identity_holds(tau, log_n, r)
    assert not vc.h_identity_holds(tau, log_n, r, top_snarkjs=True)
    r[-1] = 0
    assert vc.h_identity_holds(tau, log_n, r)
    assert vc.h_identity_holds(tau, log_n, r, top_snarkjs=True)


def test_h_hash_points():
    assert [vc.h_hash_points(1 << k) for k in (1, 3, 14, 15, 20)] == [1, 7, (1 << 14) - 1, 1 << 15, 1 << 20]


# ------------------------------------------------------------------------------------------------ circuit hash
PTAUS = {}


def ptau_file(power):
    if power not in PTAUS:
        PTAUS[power] = ptau.write_ptau(TOX["tau"], TOX["alpha"], TOX["beta"], power)
    return PTAUS[power]


def init_key(seed, n_constraints, n_public=2, n_free=3):
    return util.tiny_case(seed, n_constraints, n_public, n_free, toxic=TOX)["zkey_bytes"]


# (constraints, public) -> domain 2^3 .. 2^6; ptau power = cirPower (2^4 also at cirPower + 1)
HASH_CASES = [(4, 1, 3, 3), (10, 2, 4, 4), (10, 2, 4, 5), (20, 2, 5, 5), (40, 2, 6, 6)]


@pytest.mark.parametrize("nc,np_,cp,power", HASH_CASES)
def test_host_circuit_hash_matches_helper(lib, nc, np_, cp, power):
    zk = init_key(nc, nc, np_)
    hdr, _ = formats.read_zkey_header(zk)
    assert hdr["domainSize"] == 1 << cp
    pt = ptau_file(power)
    want = vc.circuit_hash(zk, pt)
    assert api.host_zkey_circuit_hash(zk, pt) == want
    assert api.host_zkey_circuit_hash({"type": "mem", "data": zk}, pt) == want


# ------------------------------------------------------------------------------------------------ rejections
def _fake_ptau(power):
    """A prepared ptau of the right layout whose points are all at infinity (valid points: the rejection under test comes
    from the domain alone)."""
    n = 1 << power
    secs = [(1, struct.pack("<I", 32) + to_le32(Q_MOD) + struct.pack("<II", power, power))]
    sizes = {2: (2 * n - 1) * 64, 3: n * 128, 4: n * 64, 5: n * 64, 6: 128, 7: 4,
             12: (4 * n - 1) * 64, 13: (2 * n - 1) * 128, 14: (2 * n - 1) * 64, 15: (2 * n - 1) * 64}
    secs += [(sid, bytes(sz)) for sid, sz in sizes.items()]
    return formats.write_container(b"ptau", 1, secs)


def _with_domain(zk, n):
    """The key with domainSize = n and a section 9 of n points at infinity."""
    secs = cc.sections(zk)
    h = bytearray(secs[2])
    struct.pack_into("<I", h, 80, n)
    secs[2], secs[9] = bytes(h), bytes(64 * n)
    return formats.write_container(b"zkey", 1, sorted(secs.items()))


def _init_and_ptau():
    return init_key(10, 10, 2), ptau_file(4)


def _verify_init(key, init, pt):
    return api.zkey_verify(key, pt, init=init, seed=SEED)


def _hash_entries(init, pt):
    return [lambda: api.host_zkey_circuit_hash(init, pt), lambda: api.zkey_circuit_hash(init, pt)]


def test_rejects_cir_power_equal_power_above_2_14(lib):
    """At cirPower = power and N > 2^14 snarkjs's hashHPoints reads past ptau section 2: rejected, never hashed."""
    init = _with_domain(init_key(10, 10, 2), 1 << 15)
    pt = _fake_ptau(15)
    for fn in [lambda: api.zkey_circuit_hash(init, pt), lambda: _verify_init(init, init, pt)]:
        _raises(fn, _lib.NZCP_E_ARG, "past the end of ptau section 2")


def test_init_and_ptau_rejections(lib):
    init, pt = _init_and_ptau()
    secs = cc.sections(init)
    bad3 = dict(secs)
    bad3[3] = secs[3][:-64]
    short3 = formats.write_container(b"zkey", 1, sorted(bad3.items()))
    odd = _with_domain(init, 24)
    unprepared = ptau.write_ptau(TOX["tau"], TOX["alpha"], TOX["beta"], 4, prepared=False)
    small = ptau_file(3)
    cases = [(short3, pt, _lib.NZCP_E_FORMAT, "section 3 size does not match the header"),
             (odd, pt, _lib.NZCP_E_FORMAT, "domainSize is not a power of two"),
             (init, unprepared, _lib.NZCP_E_FORMAT, "Powers of tau is not prepared."),
             (init, small, _lib.NZCP_E_ARG, "circuit too big for this power of tau ceremony"),
             (init, b"nope" * 8, _lib.NZCP_E_FORMAT, "ptau file: Invalid File format")]
    for i, p, code, msg in cases:
        for fn in _hash_entries(i, p) + [lambda: _verify_init(init, i, p)]:
            _raises(fn, code, msg)
    r1cs = formats.write_r1cs(*_r1cs_args(10))
    _raises(lambda: api.zkey_verify(init, unprepared, r1cs=r1cs), _lib.NZCP_E_FORMAT, "Powers of tau is not prepared.")
    _raises(lambda: api.zkey_verify(init, pt, r1cs=b"r1cs" + bytes(8)), _lib.NZCP_E_FORMAT, "r1cs: missing or short section")


def _r1cs_args(seed, n_constraints=10, n_public=2, n_free=3):
    c = util.tiny_case(seed, n_constraints, n_public, n_free, toxic=TOX)
    return c["n_vars"], c["n_public"], 0, c["n_vars"] - c["n_public"] - 1, c["constraints"]


def test_file_rejections_of_the_key(lib, named_key):
    """The container rejections of `zkey contribute` hold for the key under verification, with their codes and messages,
    through the size function and both verify entries.  Bad points there are a false verdict instead (GPU tests)."""
    init, pt = _init_and_ptau()
    n = 0
    for name, buf, code, msg in _file_rejections(named_key):
        if code == _lib.NZCP_E_RANGE:
            continue
        n += 1
        size = C.c_size_t()
        for fn in (lambda: _lib.check(_lib.load().nzcp_zkey_verify_size(_lib.addr(buf), len(buf), C.byref(size),
                                                                      C.byref(size))),
                   lambda: _verify_init(buf, init, pt)):
            _raises(fn, code, msg)
        for fn in _hash_entries(buf, pt):           # as the initial key
            _raises(fn, code, msg)
    assert n >= 20


def test_beacon_record_without_parameters(lib, named_key):
    """A type-1 record must carry its beacon hash: otherwise the container is malformed."""
    secs = cc.sections(named_key)
    s10 = bytearray(secs[10])
    csh, recs = cc.parse_mpc(bytes(s10))
    rec = bytearray(recs[0][:cc.REC_FIXED])
    struct.pack_into("<II", rec, 384, 1, 0)
    secs[10] = csh + struct.pack("<I", 1) + bytes(rec)
    buf = formats.write_container(b"zkey", 1, sorted(secs.items()))
    init, pt = _init_and_ptau()
    _raises(lambda: _verify_init(buf, init, pt), _lib.NZCP_E_FORMAT, "beacon record without a beacon hash")


def test_verify_size_and_buffers(lib, named_key):
    L = _lib.load()
    n_claims, n_recs = C.c_size_t(), C.c_size_t()
    _lib.check(L.nzcp_zkey_verify_size(_lib.addr(named_key), len(named_key), C.byref(n_claims), C.byref(n_recs)))
    _, recs = cc.parse_mpc(cc.sections(named_key)[10])
    assert (n_claims.value, n_recs.value) == (2 * len(recs) + 3, len(recs))
    init, pt = _init_and_ptau()
    claims = (_lib.VerifyClaim * (n_claims.value - 1))()
    records = (_lib.Contribution * n_recs.value)()
    rep = _lib.VerifyReport()
    code = L.nzcp_zkey_verify_from_init(_lib.addr(init), len(init), _lib.addr(pt), len(pt), _lib.addr(named_key),
                                        len(named_key), None, 0, claims, n_claims.value - 1, records, n_recs.value,
                                        C.byref(rep), None)
    assert code == _lib.NZCP_E_ARG and b"too small" in L.nzcp_last_error()
    assert C.sizeof(_lib.VerifyClaim) == 8 + 2 * 64 + 2 * 128
    assert C.sizeof(_lib.Contribution) == 64 + 16 + 2 * 256
    assert C.sizeof(_lib.VerifyReport) == 8 + 256 + 8 + 64


def test_host_hook_size_limit(lib):
    init = init_key(3, 2100, 1, 8)
    _raises(lambda: api.host_zkey_circuit_hash(init, ptau_file(4)), _lib.NZCP_E_ARG, "")


def test_api_arguments(lib, named_key):
    init, pt = _init_and_ptau()
    _raises(lambda: api.zkey_verify(named_key, pt), _lib.NZCP_E_ARG, "exactly one of r1cs and init")
    _raises(lambda: api.zkey_verify(named_key, pt, init=init, seed=b"x"), _lib.NZCP_E_ARG, "seed must be 32 bytes")


def test_compute_needs_a_device(lib, named_key):
    """No CPU fallback: valid inputs reach the device check and fail there."""
    if api.device_count() > 0:
        pytest.skip("GPU present")
    init, pt = _init_and_ptau()
    r1cs = formats.write_r1cs(*_r1cs_args(10))
    for fn in (lambda: api.zkey_circuit_hash(init, pt), lambda: _verify_init(named_key, init, pt),
               lambda: api.zkey_verify(named_key, pt, r1cs=r1cs), lambda: api.zkey_new(r1cs, pt, circuit_hash=True)):
        _raises(fn, _lib.NZCP_E_CUDA, "no CUDA device")


ALLOWED = {_lib.NZCP_OK, -1, -2, -3, -4, -5, -6, -7}


def test_fuzz_verify_containers(lib, named_key):
    """Truncations, bit flips and poked 32-bit fields of the key and of the initial key never crash the parsers; every
    outcome is a documented code (the compute entries stop at the device check here, or run on a GPU box)."""
    L = _lib.load()
    rng = random.Random(77)
    init, pt = _init_and_ptau()
    h = bytearray(64)
    n_claims, n_recs = C.c_size_t(), C.c_size_t()
    for it in range(300):
        base = named_key if it % 2 else init
        b = bytearray(base)
        n = len(b)
        kind = it % 3
        if kind == 0:
            b = b[:rng.randrange(0, n)]
        elif kind == 1:
            b[rng.randrange(0, n)] ^= 1 << rng.randrange(8)
        else:
            struct.pack_into("<I", b, rng.randrange(0, n - 4), rng.choice([0, 1, 2, 0xFFFFFFFF, 0x80000000, n]))
        b = bytes(b)
        assert L.nzcp_zkey_verify_size(_lib.addr(b), len(b), C.byref(n_claims), C.byref(n_recs)) in ALLOWED
        assert L.nzcp_host_zkey_circuit_hash(_lib.addr(b), len(b), _lib.addr(pt), len(pt), _lib.addr(h)) in ALLOWED
