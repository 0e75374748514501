"""Device Fq / Fq2 arithmetic and the XYZZ group law, limb for limb against Python integers and the oracle.

Covers the device-only code under every proof: the 512-bit product and wide reduction behind the lazy-reduction bodies
(f_mulsub on Fq, the default Fq2 product reached through the non-inlined f2_mul_call), the Fq2 square and inversions,
and xyzz_add / xyzz_madd / xyzz_dbl / xyzz_to_affine on G1 and G2 with every special branch.  Operands come from
tests/arith_cases.py: limb patterns, operands solved for a chosen result, and the extremes of the stated bounds.
"""
import random

import numpy as np
import pytest

import arith_cases as ac
from nzcp_circom_b200 import api
from oracle import bn254 as ob
from util import le32

pytestmark = pytest.mark.gpu

Q, MONT, F2 = ob.Q_MOD, ac.MONT, ac.F2


def _rec(vals, width=32):
    return b"".join(int(v).to_bytes(width, "little") for v in vals)


def _ints(buf, width=32):
    return [int.from_bytes(buf[i:i + width], "little") for i in range(0, len(buf), width)]


def _f2_flat(vals):
    return [c for v in vals for c in v]


def _f2_pairs(ints):
    return [(ints[i], ints[i + 1]) for i in range(0, len(ints), 2)]


def _check(op, cases, got_ints, exp):
    bad = [(c, g, e) for c, g, e in zip(cases, got_ints, exp) if g != e]
    assert not bad, "op %d: %d of %d cases differ, first: %r" % (op, len(bad), len(cases), bad[0])


# ------------------------------------------------------------------------------------------------ Fq: wide product, reduction
def test_mul_wide_is_the_exact_product(lib):
    rng = random.Random(1)
    pat = [(ac.limb_pattern(rng) >> 1, ac.limb_pattern(rng) >> 1) for _ in range(3000)]
    pat += [(ac.limb_pattern(rng) & ((1 << 255) - 1), ac.limb_pattern(rng) & ((1 << 255) - 1)) for _ in range(1000)]
    rnd = [(rng.getrandbits(255), rng.getrandbits(255)) for _ in range(1000)]
    cases = ac.mul_wide_extremes() + pat + rnd
    got = _ints(api.arith_op(0, _rec(_f2_flat(cases)), len(cases)), 64)
    _check(0, cases, got, [a * b for a, b in cases])


def test_redc_wide(lib):
    rng = random.Random(2)
    cases = ac.redc_extremes()
    cases += [ac.redc_targeted(rng, y) for y in ac.targets() for _ in range(8)]
    cases += [y * MONT % Q for y in ac.targets()]                                   # k = 0: high half zero
    cases += [y * MONT % Q + (MONT - 1) * Q for y in ac.targets()]                  # largest k
    for _ in range(3000):                                                           # limb patterns, high half < q
        t = ac.limb_pattern(rng, 16)
        cases.append((t >> 256) % Q * MONT + (t & (MONT - 1)))
    assert max(cases) < Q * MONT
    got = _ints(api.arith_op(1, _rec(cases, 64), len(cases)))
    _check(1, cases, got, [t * ac.RINV % Q for t in cases])


# ------------------------------------------------------------------------------------------------ Fq: a b - c d
def _mulsub_cases(rng):
    cases = ac.mulsub_extremes()
    cases += [ac.mulsub_targeted(rng, y) for y in ac.targets() for _ in range(10)]
    v = ac.pattern_values(rng, 4 * 2000)
    cases += [tuple(v[4 * i:4 * i + 4]) for i in range(2000)]
    return cases


@pytest.mark.parametrize("op", [2, 3])    # 2: lazy f_mulsub (one wide reduction), 3: fp_sub(fp_mul, fp_mul)
def test_mulsub(lib, op):
    cases = _mulsub_cases(random.Random(3))
    got = _ints(api.arith_op(op, _rec(_f2_flat(cases)), len(cases)))
    _check(op, cases, got, [ac.mulsub_ref(*c) for c in cases])


# ------------------------------------------------------------------------------------------------ Fq2
def _f2_mul_cases(rng):
    cases = ac.f2_mul_extremes()
    cases += [ac.f2_mul_targeted(rng, y) for y in ac.targets_fq2() for _ in range(2)]
    v = ac.pattern_fq2(rng, 2 * 2000)
    cases += [(v[2 * i], v[2 * i + 1]) for i in range(2000)]
    return cases


@pytest.mark.parametrize("op", [4, 5])    # 4: f_mul(Fq2) as the kernels call it (f2_mul_call), 5: f2_mul_inline
def test_fq2_mul(lib, op):
    cases = _f2_mul_cases(random.Random(4))
    got = _f2_pairs(_ints(api.arith_op(op, _rec(_f2_flat(_f2_flat(cases))), len(cases))))
    _check(op, cases, got, [ac.f2_mont_mul(a, b) for a, b in cases])


def test_fq2_sqr(lib):
    rng = random.Random(6)
    cases = [a for a, _ in ac.f2_mul_extremes()[::8]] + [a for a, _ in _f2_mul_cases(rng)] + ac.pattern_fq2(rng, 2000)
    got = _f2_pairs(_ints(api.arith_op(6, _rec(_f2_flat(cases)), len(cases))))
    _check(6, cases, got, [ac.f2_mont_mul(a, a) for a in cases])


def test_fq2_mulsub(lib):
    rng = random.Random(9)
    cases = ac.f2_mulsub_extremes()
    cases += [ac.f2_mulsub_targeted(rng, y) for y in ac.targets_fq2()]
    v = ac.pattern_fq2(rng, 4 * 1000)
    cases += [tuple(v[4 * i:4 * i + 4]) for i in range(1000)]
    got = _f2_pairs(_ints(api.arith_op(9, _rec(_f2_flat(_f2_flat(cases))), len(cases))))
    _check(9, cases, got, [ac.f2_mulsub_ref(*c) for c in cases])


@pytest.mark.parametrize("op", [7, 8])    # 7: Fermat f_inv(Fq2), 8: f_inv_fast(Fq2) by division steps
def test_fq2_inverse(lib, op):
    rng = random.Random(7)
    edge = ac.inverse_edge_values(Q)
    cases = [(0, 0)] + [(x, 0) for x in edge] + [(0, x) for x in edge] + [(x, x) for x in edge]
    cases += [ac.f2_inv_targeted(y) for y in ac.targets_fq2() if not F2.is_zero(y)]
    cases += ac.pattern_fq2(rng, 2000) + [(rng.randrange(Q), rng.randrange(Q)) for _ in range(1000)]
    out = api.arith_op(op, _rec(_f2_flat(cases)), len(cases))
    got = _f2_pairs(_ints(out))
    _check(op, cases, got, [ac.f2_mont_inv(a) for a in cases])
    # a * a^-1 = 1 (Montgomery one) through the device product, for every a != 0
    nz = [i for i, a in enumerate(cases) if not F2.is_zero(a)]
    pairs = b"".join(_rec(cases[i]) + out[64 * i:64 * i + 64] for i in nz)
    prod = api.arith_op(4, pairs, len(nz))
    assert prod == (le32(MONT % Q) + le32(0)) * len(nz)


# ------------------------------------------------------------------------------------------------ lazy == eager, 2^22 cases
def _random_fq(rng, shape):
    """Uniform-ish canonical Fq limbs: top limb below q's, so every value is < q."""
    x = rng.integers(0, 1 << 32, size=shape + (8,), dtype=np.uint32)
    x[..., 7] = rng.integers(0, 0x30644E72, size=shape, dtype=np.uint32)
    return x


@pytest.mark.parametrize("lazy,eager", [(2, 3), (4, 5)])
def test_lazy_matches_eager_random(lib, lazy, eager):
    n = 1 << 22
    data = _random_fq(np.random.default_rng(lazy), (n, 4))
    a = np.frombuffer(api.arith_op(lazy, data, n), dtype=np.uint32).reshape(n, -1)
    b = np.frombuffer(api.arith_op(eager, data, n), dtype=np.uint32).reshape(n, -1)
    diff = np.flatnonzero((a != b).any(axis=1))
    assert diff.size == 0, "op %d vs op %d: %d of %d differ, first at %d" % (lazy, eager, diff.size, n, diff[0])


# ------------------------------------------------------------------------------------------------ XYZZ group law
def _fenc(g2, v):
    return le32(v[0] * MONT % Q) + le32(v[1] * MONT % Q) if g2 else le32(v * MONT % Q)


def _fdec(g2, b):
    """Montgomery record -> field value; every limb vector the device writes must be canonical (< q)."""
    raw = _ints(b)
    assert all(v < Q for v in raw), "non-canonical coordinate"
    v = [x * ac.RINV % Q for x in raw]
    return tuple(v) if g2 else v[0]


def _lambdas(g2, rng):
    if g2:
        return [(1, 0), (Q - 1, 0), (rng.randrange(1, Q), rng.randrange(Q))]
    return [1, Q - 1, rng.randrange(1, Q)]


def _xyzz(curve, P, lam, garbage=None):
    """(x lam^2, y lam^3, lam^2, lam^3); P = None -> zz = zzz = 0 with x, y = garbage (zeros by default)."""
    F = curve.F
    if P is None:
        return (garbage or (F.zero, F.zero)) + (F.zero, F.zero)
    l2 = F.sqr(lam)
    l3 = F.mul(l2, lam)
    return (F.mul(P[0], l2), F.mul(P[1], l3), l2, l3)


def _check_xyzz(curve, g2, out, exp, what):
    F = curve.F
    w = 64 if g2 else 32
    for i, E in enumerate(exp):
        x, y, zz, zzz = (_fdec(g2, out[(4 * i + k) * w:(4 * i + k + 1) * w]) for k in range(4))
        if E is None:
            assert F.is_zero(zz), (what, i, "expected infinity")
            continue
        assert not F.is_zero(zz), (what, i, "unexpected infinity")
        assert F.mul(F.sqr(zz), zz) == F.sqr(zzz), (what, i, "zz^3 != zzz^2")
        assert x == F.mul(E[0], zz) and y == F.mul(E[1], zzz), (what, i, "wrong point")


@pytest.fixture(scope="module")
def points():
    rng = random.Random(11)
    fbs = ob.FixedBase(ob.G1, ob.G1_GEN), ob.FixedBase(ob.G2, ob.G2_GEN)
    return {g2: [fbs[g2].mul(rng.randrange(1, ob.R_MOD)) for _ in range(24)] for g2 in (False, True)}


@pytest.mark.parametrize("g2", [False, True])
def test_xyzz_add(lib, points, g2):
    curve = ob.G2 if g2 else ob.G1
    rng = random.Random(20 + g2)
    pts = points[g2]
    junk = ((5, 7), (11, 13)) if g2 else (5, 7)
    cases = []   # (P, lamP, garbageP, Q, lamQ, garbageQ)
    for i, P in enumerate(pts):
        la, lb = _lambdas(g2, rng), _lambdas(g2, rng)
        Qp = pts[(i + 1) % len(pts)]
        cases.append((P, la[i % 3], None, Qp, lb[(i + 1) % 3], None))             # random pair
        cases.append((P, la[i % 3], None, P, lb[(i + 2) % 3], None))              # same point, other lambda: doubling
        cases.append((P, la[i % 3], None, P, la[i % 3], None))                    # identical records
        cases.append((P, la[i % 3], None, curve.neg(P), lb[i % 3], None))         # P + (-P): cancellation
    P0, lam = pts[0], _lambdas(g2, rng)[2]
    for g in (None, junk):                                                        # infinity, x = y = 0 and not
        cases.append((None, lam, g, P0, lam, None))
        cases.append((P0, lam, None, None, lam, g))
        cases.append((None, lam, g, None, lam, g))
    a = b"".join(_fenc(g2, v) for P, l, g, _, _, _ in cases for v in _xyzz(curve, P, l, g))
    b = b"".join(_fenc(g2, v) for _, _, _, P, l, g in cases for v in _xyzz(curve, P, l, g))
    out = api.curve_op(g2, 0, a, b, len(cases))
    _check_xyzz(curve, g2, out, [curve.add(c[0], c[3]) for c in cases], "add")


@pytest.mark.parametrize("neg", [False, True])
@pytest.mark.parametrize("g2", [False, True])
def test_xyzz_madd(lib, points, g2, neg):
    curve = ob.G2 if g2 else ob.G1
    rng = random.Random(30 + 2 * g2 + neg)
    pts = points[g2]
    junk = ((5, 7), (11, 13)) if g2 else (5, 7)
    cases = []   # (acc point, lambda, garbage, affine operand)
    for i, P in enumerate(pts):
        lam = _lambdas(g2, rng)[i % 3]
        cases.append((P, lam, None, pts[(i + 5) % len(pts)]))     # random pair
        cases.append((P, lam, None, P))                             # onto itself: doubling (neg: cancellation)
        cases.append((curve.neg(P), lam, None, P))                  # onto its negative: cancellation (neg: doubling)
    for g in (None, junk):
        cases.append((None, 1 if not g2 else (1, 0), g, pts[0]))    # accumulator at infinity
    enc = ob.g2_to_bytes_mont if g2 else ob.g1_to_bytes_mont
    a = b"".join(_fenc(g2, v) for P, l, g, _ in cases for v in _xyzz(curve, P, l, g))
    b = b"".join(enc(c[3]) for c in cases)
    out = api.curve_op(g2, 2 if neg else 1, a, b, len(cases))
    exp = [curve.add(c[0], curve.neg(c[3]) if neg else c[3]) for c in cases]
    _check_xyzz(curve, g2, out, exp, "madd neg=%d" % neg)


@pytest.mark.parametrize("g2", [False, True])
def test_xyzz_dbl_and_to_affine(lib, points, g2):
    curve = ob.G2 if g2 else ob.G1
    rng = random.Random(40 + g2)
    junk = ((5, 7), (11, 13)) if g2 else (5, 7)
    cases = [(P, _lambdas(g2, rng)[i % 3], None) for i, P in enumerate(points[g2])]
    cases += [(P, lam, None) for P in points[g2][:2] for lam in _lambdas(g2, rng)]
    cases += [(None, _lambdas(g2, rng)[0], None), (None, _lambdas(g2, rng)[0], junk)]
    a = b"".join(_fenc(g2, v) for P, l, g in cases for v in _xyzz(curve, P, l, g))
    _check_xyzz(curve, g2, api.curve_op(g2, 3, a, None, len(cases)), [curve.add(c[0], c[0]) for c in cases], "dbl")
    enc = ob.g2_to_bytes_mont if g2 else ob.g1_to_bytes_mont
    assert api.curve_op(g2, 4, a, None, len(cases)) == b"".join(enc(c[0]) for c in cases)
