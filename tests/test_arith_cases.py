"""CPU: the operand generators of the device arithmetic tests hit what they aim at (tests/arith_cases.py)."""
import random

import pytest

import arith_cases as ac
from oracle import bn254 as ob

R, Q, MONT, F2 = ob.R_MOD, ob.Q_MOD, ac.MONT, ac.F2


def test_limb_patterns_reach_every_special_limb_in_every_position():
    rng = random.Random(1)
    for n_limbs in (8, 16):
        xs = [ac.limb_pattern(rng, n_limbs) for _ in range(600)]
        assert all(x < 1 << (32 * n_limbs) for x in xs)
        for k in range(n_limbs):
            seen = {(x >> (32 * k)) & 0xFFFFFFFF for x in xs}
            assert set(ac.SPECIAL_LIMBS) <= seen, k
    v = ac.pattern_values(rng, 1000)
    assert len(v) == 1000 and all(0 <= x < Q for x in v)
    assert all(v[i] + v[i + 1] == Q - 1 for i in range(0, 1000, 2))
    assert any(x >> 224 == Q >> 224 for x in v)               # top limb equal to q's: the full compare decides


def test_targets():
    for p in (R, Q):
        t = ac.targets(p)
        assert all(0 <= y < p for y in t)
        assert {0, 1} | {p - k for k in range(1, 65)} <= set(t)
        assert any(abs(y - (1 << 253)) <= 3 for y in t)
    assert len(ac.targets_fq2()) == 4 * len(ac.targets())


@pytest.mark.parametrize("p", [R, Q])
def test_mul_targeted(p):
    rng = random.Random(2)
    for y in ac.targets(p):
        a, b = ac.mul_targeted(rng, y, p)
        assert 0 <= a < p and 0 <= b < p and ac.mont_mul(a, b, p) == y


def test_redc_targeted_and_extremes():
    rng = random.Random(3)
    ts = []
    for y in ac.targets():
        t = ac.redc_targeted(rng, y)
        assert 0 <= t < Q * MONT and t * ac.RINV % Q == y
        ts.append(t)
    assert any(t >> 256 > Q // 2 for t in ts)                  # the high half spreads over [0, q)
    ex = ac.redc_extremes()
    assert all(0 <= t < Q * MONT for t in ex)
    assert Q * MONT - 1 in ex
    assert any(0 < t < MONT for t in ex) and any(t and t % MONT == 0 for t in ex)


def test_mul_wide_extremes():
    ex = ac.mul_wide_extremes()
    assert all(0 <= a < 1 << 255 and 0 <= b < 1 << 255 for a, b in ex)
    assert ((1 << 255) - 1, (1 << 255) - 1) in ex


def test_mulsub_targeted_and_extremes():
    rng = random.Random(4)
    for y in ac.targets():
        c = ac.mulsub_targeted(rng, y)
        assert all(0 <= x < Q for x in c) and ac.mulsub_ref(*c) == y
    ex = ac.mulsub_extremes()
    assert (Q - 1, Q - 1, 0, 0) in ex and (0, 0, Q - 1, Q - 1) in ex    # a b - c d at both ends
    assert all(0 <= x < Q for c in ex for x in c)


def test_fq2_generators():
    rng = random.Random(5)
    for y in ac.targets_fq2():
        a, b = ac.f2_mul_targeted(rng, y)
        assert ac.f2_mont_mul(a, b) == y
        assert ac.f2_mulsub_ref(*ac.f2_mulsub_targeted(rng, y)) == y
        if not F2.is_zero(y):
            assert ac.f2_mont_inv(ac.f2_inv_targeted(y)) == y
    # Karatsuba sums at 2q - 2: a0 = a1 = b0 = b1 = q - 1
    assert ((Q - 1, Q - 1), (Q - 1, Q - 1)) in ac.f2_mul_extremes()
    m, z = (Q - 1, Q - 1), (0, 0)
    assert (m, m, z, z) in ac.f2_mulsub_extremes() and (z, z, m, m) in ac.f2_mulsub_extremes()
    v = ac.pattern_fq2(rng, 50)
    assert len(v) == 50 and all(0 <= c < Q for x in v for c in x)


def test_montgomery_references():
    """The references the device results are compared with, against the oracle's plain-form field arithmetic."""
    rng = random.Random(6)
    for _ in range(50):
        x, y = (rng.randrange(Q), rng.randrange(Q)), (rng.randrange(Q), rng.randrange(Q))
        xm, ym = F2.muli(x, MONT), F2.muli(y, MONT)                    # Montgomery representatives
        assert ac.f2_mont_mul(xm, ym) == F2.muli(F2.mul(x, y), MONT)
        assert ac.f2_mont_inv(xm) == F2.muli(F2.inv(x), MONT)
    assert ac.f2_mont_inv((0, 0)) == (0, 0)
