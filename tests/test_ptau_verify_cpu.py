"""`powersoftau verify` without a GPU: the host hook (the kernels' per-point code and the MSMs' code on the CPU) against the
Python restatement (tests/ptau_verify_cases.py) byte for byte on library-made chains, prepared and not, one tampered file
per verdict message, a reduced file, every input rejection through every entry point, malformed containers, and no CPU
fallback for the device entry."""
import ctypes as C
import random
import struct

import pytest

import ptau_contribution_cases as pc
import ptau_verify_cases as pv
from nzcp_circom_b200 import _lib, api, groth16
from nzcp_circom_b200._lib import NzcpError
from oracle import formats
from oracle.bn254 import G1, G2, Q_MOD, g1_from_bytes_mont, g1_to_bytes_mont, g2_from_bytes_mont, g2_to_bytes_mont, to_le32

SEED = bytes(range(32))
VSEED = bytes([7]) * 32
BEACON = bytes.fromhex("0123456789abcdef")


def chain(power, prepared, host=True):
    """new -> contribute -> contribute -> beacon (-> prepare), built by the host hooks (host=True) or on the device."""
    f = bytes(api.ptau_new(power)[0])
    if host:
        steps = [lambda b: api.host_ptau_contribute(b, name="alice", seed=SEED),
                 lambda b: api.host_ptau_contribute(b, seed=bytes(32)),
                 lambda b: api.host_ptau_contribute(b, name="final", beacon_hash=BEACON, num_iterations_exp=10)]
    else:
        steps = [lambda b: api.ptau_contribute(b, name="alice", seed=SEED), lambda b: api.ptau_contribute(b, seed=bytes(32)),
                 lambda b: api.ptau_beacon(b, BEACON, 10, name="final")]
    hashes = []
    for s in steps:
        f, h = s(f)
        f = bytes(f)
        hashes.append(h)
    if prepared:
        f = bytes(api.host_ptau_prepare(f) if host else api.ptau_prepare(f))
    return f, hashes


CHAINS = {}


def get_chain(power, prepared):
    if (power, prepared) not in CHAINS:
        CHAINS[power, prepared] = chain(power, prepared)
    return CHAINS[power, prepared]


def raw(buf, seed, device=None):
    """nzcp_host_ptau_verify (device None) or nzcp_ptau_verify -> (report bytes, [claim bytes], [record bytes])."""
    L = _lib.load()
    n_claims, n_recs = C.c_size_t(), C.c_size_t()
    _lib.check(L.nzcp_ptau_verify_size(_lib.addr(buf), len(buf), C.byref(n_claims), C.byref(n_recs)))
    claims = (_lib.VerifyClaim * n_claims.value)()
    recs = (_lib.PtauContribution * max(1, n_recs.value))()
    rep = _lib.PtauVerifyReport()
    if device is None:
        _lib.check(L.nzcp_host_ptau_verify(_lib.addr(buf), len(buf), seed, claims, n_claims.value, recs, n_recs.value,
                                           C.byref(rep)))
    else:
        _lib.check(L.nzcp_ptau_verify(_lib.addr(buf), len(buf), seed, device, claims, n_claims.value, recs, n_recs.value,
                                      C.byref(rep), None))
    return bytes(rep), [bytes(c) for c in claims[:rep.n_claims]], [bytes(r) for r in recs[:n_recs.value]]


def check_against_python(buf, seed):
    """Report fields, claim bytes and records of the host hook equal the restatement's."""
    want = pv.expected(buf, seed)
    rep_b, claims, recs = raw(buf, seed)
    rep = _lib.PtauVerifyReport.from_buffer_copy(rep_b)
    assert (rep.failed_step, rep.failed_record, rep.message.decode()) == (want["failed_step"], want["failed_record"],
                                                                          want["message"])
    assert claims == want["claims"]
    assert (rep.n_claims, bool(rep.prepared), bytes(rep.next_challenge)) == (len(want["claims"]), want["prepared"],
                                                                            want["next_challenge"])
    assert rep.n_contributions == len(want["records"]) == len(recs)
    for got, w in zip(recs, want["records"]):
        r = _lib.PtauContribution.from_buffer_copy(got)
        assert (bytes(r.response_hash), bytes(r.next_challenge), r.type) == (w["response_hash"], w["next_challenge"],
                                                                           w["type"])
        assert bytes(r.name[:r.name_len]) == w["name"] and r.num_iterations_exp == w["exp"]
        assert bytes(r.beacon_hash[:r.beacon_hash_len]) == (w["beacon"] or b"")
    return want


@pytest.mark.parametrize("prepared", [False, True])
def test_chain_matches_python(lib, prepared):
    buf, hashes = get_chain(3, prepared)
    want = check_against_python(buf, VSEED)
    assert want["failed_step"] == 0 and len(want["claims"]) == 8 * 3 + 4
    res = api.host_ptau_verify(buf, seed=VSEED)
    assert res["ok"], res["message"]
    assert res["prepared"] == prepared
    assert [c["response_hash"] for c in res["contributions"]] == hashes
    assert [c["name"] for c in res["contributions"]] == ["alice", "", "final"]
    assert res["next_challenge"] == pc.record_fields(pc.parse_records(pc.sections(buf)[7])[-1])["next"]


def test_power4_prepared(lib):
    buf, _ = get_chain(4, True)
    assert check_against_python(buf, bytes(32))["failed_step"] == 0


def test_seed_changes_claims_not_verdict(lib):
    buf, _ = get_chain(2, False)
    a, b = raw(buf, SEED), raw(buf, VSEED)
    # the last record's claims, the four section claims, the earlier records' claims: only the section claims use the seed
    assert a[1][:8] + a[1][12:] == b[1][:8] + b[1][12:] and all(x != y for x, y in zip(a[1][8:12], b[1][8:12]))
    assert api.host_ptau_verify(buf)["ok"]                        # OS randomness


# ------------------------------------------------------------------------------------------------ tampered files
def rebuild(buf, edits):
    secs = pc.sections(buf)
    for sid, fn in edits:
        secs[sid] = bytes(fn(bytearray(secs[sid])))
    return formats.write_container(b"ptau", 1, sorted(secs.items()))


def dbl(off, g2=False):
    def f(b):
        if g2:
            b[off:off + 128] = g2_to_bytes_mont(G2.mul(g2_from_bytes_mont(bytes(b[off:off + 128])), 2))
        else:
            b[off:off + 64] = g1_to_bytes_mont(G1.mul(g1_from_bytes_mont(bytes(b[off:off + 64])), 2))
        return b
    return f


def scale(g2):
    def f(b):
        sz = 128 if g2 else 64
        for off in range(0, len(b), sz):
            dbl(off, g2)(b)
        return b
    return f


def rec_off(buf, i):
    return 4 + sum(len(r) for r in pc.parse_records(pc.sections(buf)[7])[:i])


def flip(off):
    def f(b):
        b[off] ^= 1
        return b
    return f


def _last(buf, power):
    return rec_off(buf, 2)


# (name, edits(buf, power) -> [(section, edit)], message): each file reaches its message first.  buf: a prepared
# 3-record chain, the last a beacon.  "Second element of tau*G2 section ..." cannot come first from any file: tauG2[1] is
# pinned by the powers claims (13 ties the section to last.tauG1, 12 ties last.tauG2 to the tauG1 section) and by the last
# record's claims.  Its tau*G1 twin can: doubling tauG1 in the last two records keeps every claim before it true.
TAMPERED = [
    ("beacon key", lambda b, p: [(7, dbl(_last(b, p)))],
     "BEACON key (tauG1_s) is not generated correctly in challenge #3  final"),
    ("beacon g2", lambda b, p: [(7, dbl(_last(b, p) + 512, True))],
     "BEACON key (alphaG2_spx) is not generated correctly in challenge #3  final"),
    ("key tau", lambda b, p: [(7, dbl(rec_off(b, 1) + 64))], "INVALID key (tau) in challenge #2"),
    ("key alpha", lambda b, p: [(7, dbl(rec_off(b, 1) + 192))], "INVALID key (alpha) in challenge #2"),
    ("key beta", lambda b, p: [(7, dbl(rec_off(b, 1) + 320))], "INVALID key (beta) in challenge #2"),
    ("tauG1", lambda b, p: [(7, dbl(_last(b, p) + 768))],
     "INVALID tau*G1. challenge #3 It does not follow the previous contribution"),
    ("tauG2", lambda b, p: [(7, dbl(_last(b, p) + 832, True))],
     "INVALID tau*G2. challenge #3 It does not follow the previous contribution"),
    ("alphaG1", lambda b, p: [(7, dbl(_last(b, p) + 960))],
     "INVALID alpha*G1. challenge #3 It does not follow the previous contribution"),
    ("betaG1", lambda b, p: [(7, dbl(_last(b, p) + 1024))],
     "INVALID beta*G1. challenge #3 It does not follow the previous contribution"),
    ("betaG2", lambda b, p: [(7, dbl(_last(b, p) + 1088, True))],
     "INVALID beta*G2. challenge #3 It does not follow the previous contribution"),
    ("earlier tauG1", lambda b, p: [(7, dbl(rec_off(b, 0) + 768))],
     "INVALID tau*G1. challenge #2 It does not follow the previous contribution"),
    ("powers 2", lambda b, p: [(2, dbl(64 * 5))], "tauG1 section. Powers do not match"),
    ("powers 3", lambda b, p: [(3, dbl(128 * 3, True))], "tauG2 section. Powers do not match"),
    ("powers 4", lambda b, p: [(4, dbl(64 * 2))], "alphaTauG1 section. Powers do not match"),
    ("powers 5", lambda b, p: [(5, dbl(64 * ((1 << p) - 1)))], "betaTauG1 section. Powers do not match"),
    ("scaled 2", lambda b, p: [(2, scale(False))], "First element of tau*G1 section must be the generator"),
    ("scaled 3", lambda b, p: [(3, scale(True))], "First element of tau*G2 section must be the generator"),
    ("second tauG1", lambda b, p: [(7, lambda s: dbl(rec_off(b, 2) + 768)(dbl(rec_off(b, 1) + 768)(s)))],
     "Second element of tau*G1 section does not match the one in the contribution section"),
    ("scaled 4", lambda b, p: [(4, scale(False))],
     "First element of alpha*tau*G1 section (alpha*G1) does not match the one in the contribution section"),
    ("scaled 5", lambda b, p: [(5, scale(False))],
     "First element of beta*tau*G1 section (beta*G1) does not match the one in the contribution section"),
    ("betaG2 section", lambda b, p: [(6, dbl(0, True))],
     "betaG2 element in betaG2 section does not match the one in the contribution section"),
    ("next challenge", lambda b, p: [(7, flip(_last(b, p) + pc.NEXT_OFF + 5))], pv.NEXT),
    # the last non-infinity slot of the top tauG1 level (level p + 1, which starts at 2^(p+1) - 1)
    ("lagrange 12 top", lambda b, p: [(12, dbl(64 * ((1 << (p + 1)) - 1 + (1 << (p + 1)) - 2)))], pv.LAGRANGE),
    ("lagrange 12", lambda b, p: [(12, dbl(64 * 2))], pv.LAGRANGE),
    ("lagrange 13", lambda b, p: [(13, dbl(128 * 4, True))], pv.LAGRANGE),
    ("lagrange 14", lambda b, p: [(14, dbl(64 * 0))], pv.LAGRANGE),
    ("lagrange 15", lambda b, p: [(15, dbl(64 * (2 * (1 << p) - 2)))], pv.LAGRANGE),
]


def tampered(buf, power, names=None):
    """-> [(name, file, message)] for the TAMPERED cases (all, or those in `names`) applied to `buf` of 2^power."""
    return [(name, rebuild(buf, edits(buf, power)), msg) for name, edits, msg in TAMPERED if names is None or name in names]


@pytest.mark.parametrize("case", [t[0] for t in TAMPERED])
def test_tampered(lib, case):
    buf = get_chain(2, True)[0]
    (name, bad, msg), = tampered(buf, 2, {case})
    want = check_against_python(bad, VSEED)
    res = api.host_ptau_verify(bad, seed=VSEED)
    assert not res["ok"] and res["message"] == msg, (name, res["message"])
    assert want["failed_step"] or want["claims"]      # the library stopped, or the verdict is a claim it returned


def test_off_curve_point_is_a_verdict(lib):
    buf = get_chain(2, True)[0]
    P = g1_from_bytes_mont(pc.sections(buf)[2][192:256])
    off = to_le32(P[0] * (1 << 256) % Q_MOD) + to_le32((P[1] + 1) * (1 << 256) % Q_MOD)
    for sid, at, msg in ((2, 192, "ptau: section 2 point 3 is not on the curve"),
                         (14, 64 * 5, "ptau: section 14 point 5 is not on the curve")):
        bad = rebuild(buf, [(sid, lambda b, at=at: b[:at] + off + b[at + 64:])])
        res = api.host_ptau_verify(bad, seed=VSEED)
        assert not res["ok"] and res["message"] == msg
    r0 = rec_off(buf, 0)
    bad = rebuild(buf, [(7, lambda b: b[:r0 + 768] + off + b[r0 + 832:])])
    res = api.host_ptau_verify(bad, seed=VSEED)
    assert res["message"] == "ptau: section 7 record 0 tauG1 is not a canonical point of G1"


def test_failing_file_does_not_wait_for_the_first_challenge(lib):
    """A verdict before record 0 is checked cancels the first challenge hash; at ceremonyPower 28 that pass alone hashes
    ~100 GB."""
    import time
    buf = reduced(get_chain(3, False)[0], 2)
    secs = pc.sections(buf)
    secs[1] = secs[1][:40] + struct.pack("<I", 28)
    secs[2] = secs[2][:64] + to_le32(Q_MOD) + secs[2][96:]
    bad = formats.write_container(b"ptau", 1, sorted(secs.items()))
    t0 = time.perf_counter()
    res = api.host_ptau_verify(bad, seed=VSEED)
    assert res["message"] == "ptau: section 2 point 1 has a coordinate >= q"
    assert time.perf_counter() - t0 < 30


def test_no_records(lib):
    f = bytes(api.ptau_new(2)[0])
    check_against_python(f, VSEED)
    res = api.host_ptau_verify(f, seed=VSEED)
    assert not res["ok"] and res["message"] == pv.NO_RECORDS and res["contributions"] == []


def reduced(buf, power):
    """snarkjs `powersoftau truncate`'s file: the first 2^power powers, header power < ceremonyPower, the records kept."""
    secs = pc.sections(buf)
    n = 1 << power
    secs[1] = secs[1][:36] + struct.pack("<I", power) + secs[1][40:]
    secs[2], secs[3], secs[4], secs[5] = secs[2][:64 * (2 * n - 1)], secs[3][:128 * n], secs[4][:64 * n], secs[5][:64 * n]
    return formats.write_container(b"ptau", 1, sorted((k, v) for k, v in secs.items() if k <= 7))


def test_reduced_file_skips_the_hash_check(lib):
    buf = reduced(get_chain(3, False)[0], 2)
    want = check_against_python(buf, VSEED)
    assert want["failed_step"] == 0
    res = api.host_ptau_verify(buf, seed=VSEED)
    assert res["ok"], res["message"]
    assert res["next_challenge"] != pc.record_fields(pc.parse_records(pc.sections(buf)[7])[-1])["next"]


class _Log:
    def __init__(self):
        self.lines = []

    def __getattr__(self, level):
        return lambda msg: self.lines.append((level, msg))


def test_groth16_verify_needs_a_device_and_logs(lib):
    buf = get_chain(2, False)[0]
    if api.device_count() > 0:
        log = _Log()
        assert groth16.powersOfTau.verify(buf, log, seed=VSEED)
        assert ("info", "Powers of Tau Ok!") in log.lines
        assert any(lvl == "warn" and "phase2 precalculated values" in m for lvl, m in log.lines)
    else:
        _raises(lambda: groth16.powersOfTau.verify(buf, None, seed=VSEED), _lib.NZCP_E_CUDA, "no CUDA device")


# ------------------------------------------------------------------------------------------------ rejections
def _raises(fn, code, msg):
    with pytest.raises(NzcpError) as e:
        fn()
    assert e.value.code == code, (e.value.code, str(e.value))
    assert msg in str(e.value), str(e.value)


def _set_header(buf, power, cpow):
    secs = pc.sections(buf)
    secs[1] = secs[1][:36] + struct.pack("<II", power, cpow)
    return formats.write_container(b"ptau", 1, sorted(secs.items()))


def _rejections():
    f = get_chain(2, True)[0]
    secs = pc.sections(f)
    r0 = rec_off(f, 0)
    rec0 = pc.parse_records(secs[7])[0]

    def partial(off, val):
        return rebuild(f, [(7, lambda b: b[:r0 + pc.PARTIAL_OFF + off] + struct.pack("<I", val)
                            + b[r0 + pc.PARTIAL_OFF + off + 4:])])
    beacon_bare = struct.pack("<I", 1) + rec0[:pc.REC_FIXED - 8] + struct.pack("<II", 1, 0)
    out = [("magic", b"zkey" + f[4:], _lib.NZCP_E_FORMAT, "Invalid File format"),
           ("missing 7", formats.write_container(b"ptau", 1, sorted((k, v) for k, v in secs.items() if k != 7)),
            _lib.NZCP_E_FORMAT, "Missing section 7"),
           ("tauG1 short", rebuild(f, [(2, lambda b: b[:-64])]), _lib.NZCP_E_FORMAT, "section 2 size"),
           ("section 13 short", rebuild(f, [(13, lambda b: b[:-128])]), _lib.NZCP_E_FORMAT,
            "section size does not match the header power"),
           ("ceremonyPower below power", _set_header(f, 2, 1), _lib.NZCP_E_FORMAT, "ceremonyPower out of range"),
           ("ceremonyPower 29", _set_header(f, 2, 29), _lib.NZCP_E_FORMAT, "ceremonyPower out of range"),
           ("partialHash c", partial(208, 129), _lib.NZCP_E_FORMAT, "malformed partialHash"),
           ("partialHash outlen", partial(212, 32), _lib.NZCP_E_FORMAT, "malformed partialHash"),
           ("partialHash t", partial(200, 1), _lib.NZCP_E_FORMAT, "malformed partialHash"),
           ("s7 truncated", rebuild(f, [(7, lambda b: b[:-1])]), _lib.NZCP_E_FORMAT, "section 7 is truncated"),
           ("beacon without parameters", rebuild(f, [(7, lambda b: beacon_bare)]), _lib.NZCP_E_FORMAT,
            "ptau: beacon record without a beacon hash")]
    # power 28, prepared: rejected from the header and the section table, before any size check
    p28 = formats.write_container(b"ptau", 1, [(1, pc.header(28))] + [(sid, b"") for sid in (2, 3, 4, 5, 6, 7, 12, 13, 14, 15)])
    out.append(("power 28 prepared", p28, _lib.NZCP_E_ARG, "power 28 is not supported"))
    return out


REJECTIONS = ["magic", "missing 7", "tauG1 short", "section 13 short", "ceremonyPower below power", "ceremonyPower 29",
              "partialHash c", "partialHash outlen", "partialHash t", "s7 truncated", "beacon without parameters",
              "power 28 prepared"]


def test_rejection_names(lib):
    assert [r[0] for r in _rejections()] == REJECTIONS


@pytest.mark.parametrize("case", REJECTIONS)
def test_rejections(lib, case):
    """Through the size function, the device entry (before any device work) and the host hook."""
    name, buf, code, msg = next(r for r in _rejections() if r[0] == case)
    size = C.c_size_t()
    for fn in (lambda: _lib.check(_lib.load().nzcp_ptau_verify_size(_lib.addr(buf), len(buf), C.byref(size), C.byref(size))),
               lambda: api.ptau_verify(buf, seed=VSEED), lambda: api.host_ptau_verify(buf, seed=VSEED)):
        _raises(fn, code, msg)


def test_unprepared_power_28_header_is_not_the_power_28_rejection(lib):
    p28 = formats.write_container(b"ptau", 1, [(1, pc.header(28))] + [(sid, b"") for sid in (2, 3, 4, 5, 6, 7)])
    _raises(lambda: api.host_ptau_verify(p28), _lib.NZCP_E_FORMAT, "section 2 size")


def test_buffers_and_arguments(lib):
    buf = get_chain(2, False)[0]
    L = _lib.load()
    n_claims, n_recs = C.c_size_t(), C.c_size_t()
    _lib.check(L.nzcp_ptau_verify_size(_lib.addr(buf), len(buf), C.byref(n_claims), C.byref(n_recs)))
    assert (n_claims.value, n_recs.value) == (28, 3)
    claims = (_lib.VerifyClaim * 27)()
    recs = (_lib.PtauContribution * 3)()
    rep = _lib.PtauVerifyReport()
    for fn in (lambda: L.nzcp_host_ptau_verify(_lib.addr(buf), len(buf), None, claims, 27, recs, 3, C.byref(rep)),
               lambda: L.nzcp_ptau_verify(_lib.addr(buf), len(buf), None, 0, claims, 27, recs, 3, C.byref(rep), None)):
        assert fn() == _lib.NZCP_E_ARG and b"too small" in L.nzcp_last_error()
    assert C.sizeof(_lib.PtauContribution) == 128 + 16 + 512
    assert C.sizeof(_lib.PtauVerifyReport) == 8 + 256 + 12 + 64
    _raises(lambda: api.ptau_verify(buf, seed=b"x"), _lib.NZCP_E_ARG, "seed must be 32 bytes")
    _raises(lambda: api.host_ptau_verify(bytes(api.ptau_new(5)[0])), _lib.NZCP_E_ARG, "limited to power 4")
    assert L.nzcp_ptau_verify(_lib.addr(buf), len(buf), None, -1, claims, 28, recs, 3, C.byref(rep), None) == _lib.NZCP_E_ARG


def test_device_entry_needs_a_device(lib):
    """No CPU fallback: a valid file reaches the device check and fails there."""
    if api.device_count() > 0:
        pytest.skip("GPU present")
    _raises(lambda: api.ptau_verify(get_chain(2, True)[0], seed=VSEED), _lib.NZCP_E_CUDA, "no CUDA device")


ALLOWED = {_lib.NZCP_OK, -1, -2, -4}


def test_fuzz_ptau_verify(lib):
    """Truncations, bit flips and poked 32-bit fields never crash the parser; every outcome is a documented code."""
    L = _lib.load()
    rng = random.Random(2027)
    base = get_chain(1, True)[0]
    n = len(base)
    n_claims, n_recs = C.c_size_t(), C.c_size_t()
    claims = (_lib.VerifyClaim * 64)()
    recs = (_lib.PtauContribution * 8)()
    rep = _lib.PtauVerifyReport()
    for it in range(200):
        b = bytearray(base)
        kind = it % 3
        if kind == 0:
            b = b[:rng.randrange(0, n)]
        elif kind == 1:
            b[rng.randrange(0, n)] ^= 1 << rng.randrange(8)
        else:
            struct.pack_into("<I", b, rng.randrange(0, n - 4), rng.choice([0, 1, 2, 28, 29, 0xFFFFFFFF, 0x80000000, n]))
        b = bytes(b)
        assert L.nzcp_ptau_verify_size(_lib.addr(b), len(b), C.byref(n_claims), C.byref(n_recs)) in ALLOWED
        if it % 10 == 0:      # a full host run (pairings are not part of it)
            assert L.nzcp_host_ptau_verify(_lib.addr(b), len(b), VSEED, claims, 64, recs, 8, C.byref(rep)) in ALLOWED
