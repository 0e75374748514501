"""CPU: the C-ABI library loads, exports every symbol include/nzcp_prover.h declares, its host-compiled arithmetic
matches the oracle, and every compute entry point fails loudly (NZCP_E_CUDA) on a box without a GPU."""
import os
import random
import re

import pytest

from nzcp_circom_b200 import _lib, api
from nzcp_circom_b200._lib import NzcpError
from oracle import bn254 as ob
from util import g1_plain_bytes, g2_plain_bytes, le32, tiny_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R, Q = ob.R_MOD, ob.Q_MOD


def test_every_declared_symbol_is_exported_and_bound(lib):
    hdr = open(os.path.join(ROOT, "include", "nzcp_prover.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(nzcp_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), "library does not export %s" % name
    assert declared == set(_lib.SIGNATURES), "ctypes table and header differ: %s" % (declared ^ set(_lib.SIGNATURES))


def test_struct_sizes_match_header():
    import ctypes as C
    assert C.sizeof(_lib.Proof) == 256
    assert C.sizeof(_lib.ZkeyInfo) == 4 * 4 + 8 + 3 * 64 + 3 * 128 + 8
    assert C.sizeof(_lib.ProveDebug) == 4 * 64 + 128 + 8 + (8 + 2 + 5 + 2 + 1) * 4


@pytest.mark.parametrize("field,p", [(0, R), (1, Q)])
def test_host_field_ops_vs_oracle(lib, field, p):
    rng = random.Random(field)
    vals = [0, 1, p - 1, (1 << 256) % p] + [rng.randrange(p) for _ in range(500)]
    a = vals
    b = list(reversed(vals))
    ab, bb = b"".join(le32(x) for x in a), b"".join(le32(x) for x in b)
    rinv = pow(1 << 256, -1, p)
    assert api.host_field_op(field, 0, ab, bb, len(a)) == b"".join(le32(x * y * rinv % p) for x, y in zip(a, b))
    assert api.host_field_op(field, 1, ab, bb, len(a)) == b"".join(le32((x + y) % p) for x, y in zip(a, b))
    assert api.host_field_op(field, 2, ab, bb, len(a)) == b"".join(le32((x - y) % p) for x, y in zip(a, b))


def test_host_curve_and_roots_vs_oracle(lib):
    rng = random.Random(4)
    for k in [0, 1, 2, R - 1, rng.randrange(R), rng.randrange(R)]:
        assert api.host_scalar_mul(False, None, k) == g1_plain_bytes(ob.G1.mul(ob.G1_GEN, k))
        assert api.host_scalar_mul(True, None, k) == g2_plain_bytes(ob.G2.mul(ob.G2_GEN, k))
    P = ob.G1.mul(ob.G1_GEN, 77)
    assert api.host_scalar_mul(False, ob.g1_to_bytes_mont(P), 1000) == g1_plain_bytes(ob.G1.mul(P, 1000))
    for k in range(0, 29):
        assert api.host_root_of_unity(k) == ob.FR_W[k]


def test_synthetic_circuit_host_side(lib):
    """r1cs / wtns writers run on the host: the witness satisfies every constraint and has the NZCP value mix."""
    from oracle import formats
    sc = api.SynthCircuit(seed=9, n_constraints=400, n_public=7, n_free=40)
    assert sc.n_vars == 1 + 40 + 400 and sc.domain_size == 512
    r1 = formats.read_r1cs(bytes(sc.r1cs()))
    wt = formats.read_wtns(bytes(sc.wtns(3)))["witness"]
    assert wt[0] == 1 and len(wt) == sc.n_vars
    for (A, B, C) in r1["constraints"]:
        ev = [sum(v * wt[s] for s, v in lc.items()) % R for lc in (A, B, C)]
        assert ev[0] * ev[1] % R == ev[2]
    bits = sum(1 for x in wt if x < 2)
    assert 0.3 < bits / len(wt) < 0.8
    assert wt != formats.read_wtns(bytes(sc.wtns(4)))["witness"]
    assert sc.n_coefs == sum(len(A) + len(B) for A, B, _ in r1["constraints"]) + 7 + 1


def test_no_cpu_fallback(lib):
    """Without a CUDA device every compute entry point returns NZCP_E_CUDA -- nothing silently runs on the CPU."""
    if api.device_count() > 0:
        pytest.skip("GPU present")
    c = tiny_case(1, 4, 1, 3)
    with pytest.raises(NzcpError) as e:
        api.Zkey(c["zkey_bytes"])
    assert e.value.code == _lib.NZCP_E_CUDA and "no CPU fallback" in str(e.value)
    with pytest.raises(NzcpError) as e:
        api.ntt(bytearray(64), 1)
    assert e.value.code == _lib.NZCP_E_CUDA
    with pytest.raises(NzcpError) as e:
        api.msm(bytes(64), bytes(32), 1)
    assert e.value.code == _lib.NZCP_E_CUDA
    with pytest.raises(NzcpError) as e:
        api.selftest()
    assert e.value.code == _lib.NZCP_E_CUDA
    with pytest.raises(NzcpError) as e:
        api.arith_op(2, bytes(128), 1)
    assert e.value.code == _lib.NZCP_E_CUDA
    with pytest.raises(NzcpError) as e:
        api.curve_op(False, 3, bytes(128), None, 1)
    assert e.value.code == _lib.NZCP_E_CUDA


def test_zkey_format_errors_are_reported_before_touching_the_gpu(lib):
    c = tiny_case(2, 4, 1, 3)
    zb = bytearray(c["zkey_bytes"])
    with pytest.raises(NzcpError) as e:
        api.Zkey(b"nope" + bytes(zb[4:]))
    assert e.value.code == _lib.NZCP_E_FORMAT
    z2 = bytearray(zb)
    z2[24] = 2
    with pytest.raises(NzcpError, match="zkey file is not groth16") as e:
        api.Zkey(z2)
    assert e.value.code == _lib.NZCP_E_NOT_GROTH16
    z3 = bytearray(zb)
    z3[12 + 12 + 4 + 12 + 4] ^= 0xFF          # first byte of q in the header
    with pytest.raises(NzcpError) as e:
        api.Zkey(z3)
    assert e.value.code == _lib.NZCP_E_CURVE


def test_null_and_bad_arguments_return_error_codes(lib):
    """Misuse never crashes the host: null pointers / bad sizes come back as NZCP_E_ARG (or FORMAT) with a message."""
    import ctypes as C
    p = C.c_void_p()
    assert lib.nzcp_zkey_load(None, 0, 0, C.byref(p)) == _lib.NZCP_E_ARG
    assert lib.nzcp_zkey_load(b"zkey", 4, 0, None) == _lib.NZCP_E_ARG
    assert lib.nzcp_zkey_load(b"zkey\x01\x00\x00\x00", 8, 0, C.byref(p)) == _lib.NZCP_E_FORMAT
    assert b"Invalid File format" in lib.nzcp_last_error() or b"truncated" in lib.nzcp_last_error()
    assert lib.nzcp_prover_create(None, C.byref(p)) == _lib.NZCP_E_ARG
    assert lib.nzcp_prove(None, b"", 0, None, None, None, None) == _lib.NZCP_E_ARG
    assert lib.nzcp_prove_batch(None, None, None, 0, None, None, None, 0, None) == _lib.NZCP_E_ARG
    assert lib.nzcp_zkey_info_get(None, None) == _lib.NZCP_E_ARG
    assert lib.nzcp_ntt(None, 4, 0, 0, None) == _lib.NZCP_E_ARG
    assert lib.nzcp_msm(None, None, 5, 0, 0, 0, None, None) == _lib.NZCP_E_ARG
    assert lib.nzcp_host_root_of_unity(29, (C.c_uint8 * 32)()) == _lib.NZCP_E_ARG
    assert lib.nzcp_synth_create(1, 0, 0, 0, C.byref(p)) == _lib.NZCP_E_ARG
    lib.nzcp_zkey_free(None)          # no-ops
    lib.nzcp_prover_free(None)
    lib.nzcp_synth_free(None)


def test_arith_and_curve_ops_reject_bad_arguments(lib):
    """The device arithmetic hooks check op, group and operand domain on the host, before any device is touched: a raw
    operand of the wide product >= 2^255, a wide-reduction input >= q 2^256 and a madd operand at infinity never reach a
    kernel.  Inputs just inside the bounds pass the checks (and then need a device)."""
    import ctypes as C
    out = (C.c_uint8 * 512)()
    good = bytes(256)
    for op in (-1, 10):
        assert lib.nzcp_arith_op(op, good, out, 1, 0) == _lib.NZCP_E_ARG
    for g2, op in ((0, -1), (0, 5), (2, 0), (-1, 0)):
        assert lib.nzcp_curve_op(g2, op, good, good, out, 1, 0) == _lib.NZCP_E_ARG
    assert lib.nzcp_arith_op(0, None, out, 1, 0) == _lib.NZCP_E_ARG
    assert lib.nzcp_arith_op(0, good, None, 1, 0) == _lib.NZCP_E_ARG
    assert lib.nzcp_curve_op(0, 0, good, None, out, 1, 0) == _lib.NZCP_E_ARG
    assert lib.nzcp_curve_op(0, 3, None, None, out, 1, 0) == _lib.NZCP_E_ARG

    def arith(op, *vals, width=32):
        return lib.nzcp_arith_op(op, b"".join(v.to_bytes(width, "little") for v in vals), out, 1, 0)
    mont = 1 << 256
    # fp_mul_wide: a, b < 2^255 (either operand, second record of a batch too)
    assert arith(0, 1 << 255, 1) == _lib.NZCP_E_ARG
    assert arith(0, 1, mont - 1) == _lib.NZCP_E_ARG
    assert lib.nzcp_arith_op(0, bytes(64) + le32(1) + le32(1 << 255), out, 2, 0) == _lib.NZCP_E_ARG
    assert arith(0, (1 << 255) - 1, (1 << 255) - 1) != _lib.NZCP_E_ARG
    # fp_redc_wide: T < q 2^256
    assert arith(1, Q * mont, width=64) == _lib.NZCP_E_ARG
    assert arith(1, (1 << 512) - 1, width=64) == _lib.NZCP_E_ARG
    assert arith(1, Q * mont - 1, width=64) != _lib.NZCP_E_ARG
    # xyzz_madd: the affine operand must not be (0, 0); the XYZZ side may be infinity
    for g2, (xs, as_) in enumerate(((128, 64), (256, 128))):
        for op in (1, 2):
            assert lib.nzcp_curve_op(g2, op, bytes(xs), bytes(as_), out, 1, 0) == _lib.NZCP_E_ARG
            assert lib.nzcp_curve_op(g2, op, bytes(xs), b"\x01" + bytes(as_ - 1), out, 1, 0) != _lib.NZCP_E_ARG
