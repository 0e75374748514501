"""Every C entry that reads a .zkey or a .ptau before any device work, run on the same single-fault mutants: the error
code each entry returns for each fault is pinned in one table, so the shared container readers cannot drift apart
again.  A structurally valid input gets past every check made before device work: the size functions then return
NZCP_OK, and the entries that need a device return NZCP_E_CUDA on a machine without one (PARSED below; those rows are
skipped where a device is present).

Two rows differ from earlier releases on purpose: `zkey selfcheck` now refuses a container version > 1 and a section 1
shorter than 4 bytes with NZCP_E_FORMAT, as `zkey load` always has (it used to accept the first and call the second
NZCP_E_NOT_GROTH16).
"""
import ctypes as C
import struct

import pytest

from nzcp_circom_b200 import _lib, api
from oracle import formats, ptau
from util import tiny_case

OK, ARG, FMT, G16, CURVE, CUDA = (_lib.NZCP_OK, _lib.NZCP_E_ARG, _lib.NZCP_E_FORMAT, _lib.NZCP_E_NOT_GROTH16,
                                  _lib.NZCP_E_CURVE, _lib.NZCP_E_CUDA)
PARSED = CUDA
POWER = 6


def _sections(buf, magic):
    _, secs = formats.read_container(buf, magic)
    return {sid: bytes(buf[v[0][0]:v[0][0] + v[0][1]]) for sid, v in secs.items()}


def _mutants(buf, magic, required, header_sid):
    """name -> (file) with exactly one fault; "valid" is the unchanged file."""
    secs = _sections(buf, magic)

    def build(edit=None, version=1):
        s = dict(secs)
        if edit:
            edit(s)
        return formats.write_container(magic, version, sorted(s.items()))

    def poke(sid, off, fmt, val):
        def edit(s):
            b = bytearray(s[sid])
            struct.pack_into(fmt, b, off, val)
            s[sid] = bytes(b)
        return edit

    out = {"valid": build(), "version 2": build(version=2), "s1 cut to 2": build(lambda s: s.__setitem__(1, s[1][:2]))}
    for sid in required:
        out["no s%d" % sid] = build(lambda s, sid=sid: s.pop(sid))
    h = secs[header_sid]
    out["n8q 48"] = build(poke(header_sid, 0, "<I", 48))
    out["q flipped"] = build(poke(header_sid, 4, "<B", h[4] ^ 1))
    return out, build, poke


@pytest.fixture(scope="module")
def files():
    c = tiny_case(seed=31, n_constraints=20, n_public=2, n_free=4)
    zk, r1cs = c["zkey_bytes"], formats.write_r1cs(c["n_vars"], c["n_public"], 0, c["n_vars"] - c["n_public"] - 1,
                                                 c["constraints"])
    pt = ptau.write_ptau(11, 22, 33, POWER)

    zm, build, poke = _mutants(zk, b"zkey", range(1, 11), 2)
    h = _sections(zk, b"zkey")[2]
    n_vars = struct.unpack_from("<I", h, 72)[0]
    zm["protocol 2"] = build(poke(1, 0, "<I", 2))
    zm["header 600"] = build(lambda s: s.__setitem__(2, s[2][:600]))
    zm["nPublic = nVars"] = build(poke(2, 76, "<I", n_vars))
    zm["domainSize 3"] = build(poke(2, 80, "<I", 3))

    pm, build, poke = _mutants(pt, b"ptau", list(range(1, 8)) + [12, 13, 14, 15], 1)
    for p in (0, 28, 29):
        pm["power %d" % p] = build(poke(1, 36, "<I", p))
    pm["s3 one point short"] = build(lambda s: s.__setitem__(3, s[3][:-128]))
    return {"zkey": zk, "ptau": pt, "r1cs": r1cs, "zkey_mutants": zm, "ptau_mutants": pm}


def _code(fn):
    return fn(_lib.load())


def _zkey_load(m):
    def call(L):
        h = C.c_void_p()
        rc = L.nzcp_zkey_load(_lib.addr(m), len(m), 0, C.byref(h))
        if rc == OK:
            L.nzcp_zkey_free(h)
        return rc
    return call


def _hash(init, pt):
    return lambda L: L.nzcp_zkey_circuit_hash(_lib.addr(init), len(init), _lib.addr(pt), len(pt), 0, _lib.addr(bytearray(64)),
                                              None)


def zkey_entries(m, f):
    size, n = C.c_size_t(), C.c_size_t()
    return {
        "load": _zkey_load(m),
        "selfcheck": lambda L: L.nzcp_zkey_selfcheck(_lib.addr(m), len(m), 0, C.byref(_lib.ZkeyCheck())),
        "contribute_size": lambda L: L.nzcp_zkey_contribute_size(_lib.addr(m), len(m), None, 0, C.byref(size)),
        "verify_size": lambda L: L.nzcp_zkey_verify_size(_lib.addr(m), len(m), C.byref(size), C.byref(n)),
        "circuit_hash": _hash(m, f["ptau"]),
    }


def ptau_entries(m, f):
    size = C.c_size_t()
    r1cs = f["r1cs"]
    return {
        "zkey_new_size": lambda L: L.nzcp_zkey_new_size(_lib.addr(r1cs), len(r1cs), _lib.addr(m), len(m), C.byref(size)),
        "prepare_size": lambda L: L.nzcp_ptau_prepare_size(_lib.addr(m), len(m), C.byref(size)),
        "contribute_size": lambda L: L.nzcp_ptau_contribute_size(_lib.addr(m), len(m), None, 0, C.byref(size)),
        "circuit_hash": _hash(f["zkey"], m),
    }


#                        load    selfcheck contribute_size verify_size circuit_hash
ZKEY_CODES = {
    "valid":            (PARSED, PARSED,  OK,    OK,    PARSED),
    "version 2":        (FMT,    FMT,     FMT,   FMT,   FMT),       # selfcheck: PARSED before, on purpose
    "s1 cut to 2":      (FMT,    FMT,     FMT,   FMT,   FMT),       # selfcheck: NOT_GROTH16 before, on purpose
    "no s1":            (FMT,    FMT,     FMT,   FMT,   FMT),
    "no s2":            (FMT,    FMT,     FMT,   FMT,   FMT),
    "no s3":            (FMT,    FMT,     FMT,   FMT,   FMT),
    "no s4":            (FMT,    FMT,     FMT,   FMT,   FMT),
    "no s5":            (FMT,    FMT,     FMT,   FMT,   FMT),
    "no s6":            (FMT,    FMT,     FMT,   FMT,   FMT),
    "no s7":            (FMT,    FMT,     FMT,   FMT,   FMT),
    "no s8":            (FMT,    FMT,     FMT,   FMT,   FMT),
    "no s9":            (FMT,    FMT,     FMT,   FMT,   FMT),
    "no s10":           (PARSED, PARSED,  FMT,   FMT,   FMT),
    "n8q 48":           (CURVE,  CURVE,   CURVE, CURVE, CURVE),
    "q flipped":        (CURVE,  CURVE,   CURVE, CURVE, CURVE),
    "protocol 2":       (G16,    G16,     G16,   G16,   G16),
    "header 600":       (FMT,    FMT,     FMT,   FMT,   FMT),
    "nPublic = nVars":  (FMT,    FMT,     FMT,   FMT,   FMT),
    "domainSize 3":     (FMT,    FMT,     FMT,   FMT,   FMT),
}

#                        zkey_new_size prepare_size contribute_size circuit_hash
PTAU_CODES = {
    "valid":              (OK,  OK,  OK,  PARSED),
    "version 2":          (FMT, FMT, FMT, FMT),
    "s1 cut to 2":        (FMT, FMT, FMT, FMT),
    "no s1":              (FMT, FMT, FMT, FMT),
    "no s2":              (FMT, FMT, FMT, FMT),
    "no s3":              (FMT, FMT, FMT, FMT),
    "no s4":              (FMT, FMT, FMT, FMT),
    "no s5":              (FMT, FMT, FMT, FMT),
    "no s6":              (FMT, FMT, FMT, FMT),
    "no s7":              (OK,  FMT, FMT, PARSED),
    "no s12":             (FMT, OK,  OK,  FMT),
    "no s13":             (FMT, OK,  OK,  FMT),
    "no s14":             (FMT, OK,  OK,  FMT),
    "no s15":             (FMT, OK,  OK,  FMT),
    "n8q 48":             (CURVE, CURVE, CURVE, CURVE),
    "q flipped":          (CURVE, CURVE, CURVE, CURVE),
    "power 0":            (FMT, FMT, FMT, FMT),
    "power 28":           (FMT, ARG, FMT, FMT),
    "power 29":           (FMT, FMT, FMT, FMT),
    "s3 one point short": (OK,  FMT, FMT, PARSED),
}


def _check(table, mutants, entries, f):
    assert sorted(table) == sorted(mutants)
    have_device = api.device_count() > 0
    got, want = {}, {}
    for name, m in mutants.items():
        e = entries(m, f)
        for (entry, fn), code in zip(e.items(), table[name]):
            if code == PARSED and have_device:
                continue
            got[name, entry], want[name, entry] = _code(fn), code
    assert {k: v for k, v in got.items() if v != want[k]} == {}


def test_zkey_codes(lib, files):
    _check(ZKEY_CODES, files["zkey_mutants"], zkey_entries, files)


def test_ptau_codes(lib, files):
    _check(PTAU_CODES, files["ptau_mutants"], ptau_entries, files)
