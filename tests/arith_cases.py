"""Operand generators for the limb-exact device arithmetic tests.

Carry-chain and conditional-subtraction code fails on operands that uniformly random inputs essentially never produce,
so besides random values there are three kinds of case:
- limb patterns: every 32-bit limb drawn from {0, 1, 2^31 - 1, 2^31, 2^32 - 2, 2^32 - 1, random};
- output-targeted operands: the result is chosen first (0, 1, q-1 .. q-64, values near 2^253 and at limb borrows) and the
  last operand is solved for it, which is what drives a final subtraction's "t >= q" decision to its edge;
- the extremes of the bounds the lazy-reduction code states (Karatsuba sums at 2q - 2, a b - c d at both ends, T at
  q 2^256 - 1 and with either half zero, a = b = 2^255 - 1 for the wide product).

Values are the raw integers a kernel sees: Montgomery representatives where the operation is a Montgomery one.
Fq2 values are pairs (c0, c1), u^2 = -1.
"""
from oracle import bn254 as ob

Q = ob.Q_MOD
MONT = 1 << 256
RINV = pow(MONT, -1, Q)
F2 = ob.G2.F
SPECIAL_LIMBS = (0, 1, (1 << 31) - 1, 1 << 31, (1 << 32) - 2, (1 << 32) - 1)


# ------------------------------------------------------------------------------------------------ references
def mont_mul(a, b, p=Q):
    """Montgomery product of raw representatives: a b / 2^256 mod p."""
    return a * b * pow(MONT, -1, p) % p


def f2_mont(x):
    """The raw Fq2 value x / 2^256 (what a Montgomery reduction leaves of x)."""
    return F2.muli(x, RINV)


def f2_mont_mul(a, b):
    return f2_mont(F2.mul(a, b))


def f2_mont_inv(a):
    """Montgomery-form inverse of a raw representative: 2^512 / a (0 -> 0)."""
    return (0, 0) if F2.is_zero(a) else F2.muli(F2.inv(a), MONT * MONT % Q)


def mulsub_ref(a, b, c, d):
    return (a * b - c * d) * RINV % Q


def f2_mulsub_ref(a, b, c, d):
    return f2_mont(F2.sub(F2.mul(a, b), F2.mul(c, d)))


# ------------------------------------------------------------------------------------------------ generators
def limb_pattern(rng, n_limbs=8):
    x = 0
    for k in range(n_limbs):
        c = rng.randrange(len(SPECIAL_LIMBS) + 1)
        x |= (SPECIAL_LIMBS[c] if c < len(SPECIAL_LIMBS) else rng.getrandbits(32)) << (32 * k)
    return x


def pattern_values(rng, n, p=Q):
    """n values below p: limb patterns reduced mod p, each followed by its mirror p - 1 - x."""
    out = []
    while len(out) < n:
        x = limb_pattern(rng) % p
        out += [x, p - 1 - x]
    return out[:n]


def pattern_fq2(rng, n):
    v = pattern_values(rng, 2 * n)
    return [(v[2 * i], v[2 * i + 1]) for i in range(n)]


def targets(p=Q):
    """Results the output-targeted generators aim at."""
    t = [0, 1, 2] + [p - k for k in range(1, 65)]
    t += [(1 << 253) + d for d in range(-3, 4)]
    t += [p - (1 << (32 * k)) for k in range(1, 8)]          # one limb below p's, the lower limbs equal to p's
    t += [p - (p & ((1 << (32 * k)) - 1)) - 1 for k in range(1, 8)]   # p's upper limbs, then all-ones down to limb 0
    return t


def targets_fq2():
    t = targets()
    return [(y, 0) for y in t] + [(0, y) for y in t] + [(y, y) for y in t] + [(t[i], t[-1 - i]) for i in range(len(t))]


def mul_targeted(rng, y, p=Q):
    """(a, b) whose Montgomery product is y: b = y 2^256 / a mod p."""
    a = rng.randrange(1, p)
    return a, y * MONT * pow(a, -1, p) % p


def redc_targeted(rng, y):
    """T < q 2^256 with T / 2^256 = y mod q: T = (y 2^256 mod q) + k q for a random k."""
    return y * MONT % Q + rng.randrange(MONT) * Q


def mulsub_targeted(rng, y):
    """(a, b, c, d) with (a b - c d) / 2^256 = y mod q: d = (a b - y 2^256) / c."""
    a, b, c = rng.randrange(Q), rng.randrange(Q), rng.randrange(1, Q)
    return a, b, c, (a * b - y * MONT) * pow(c, -1, Q) % Q


def _rand_fq2(rng, nonzero=False):
    while True:
        x = (rng.randrange(Q), rng.randrange(Q))
        if not (nonzero and F2.is_zero(x)):
            return x


def f2_mul_targeted(rng, y):
    """(a, b) whose Montgomery Fq2 product is y: b = y 2^256 / a."""
    a = _rand_fq2(rng, nonzero=True)
    return a, F2.mul(F2.muli(y, MONT % Q), F2.inv(a))


def f2_mulsub_targeted(rng, y):
    a, b, c = _rand_fq2(rng), _rand_fq2(rng), _rand_fq2(rng, nonzero=True)
    return a, b, c, F2.mul(F2.sub(F2.mul(a, b), F2.muli(y, MONT % Q)), F2.inv(c))


def f2_inv_targeted(y):
    """a whose Montgomery-form inverse is y (y != 0): a = 2^512 / y."""
    return f2_mont_inv(y)


# ------------------------------------------------------------------------------------------------ bound extremes
def mul_wide_extremes():
    top = (1 << 255) - 1
    vals = [0, 1, (1 << 32) - 1, 1 << 32, (1 << 224) - 1, 1 << 224, (1 << 254) - 1, 1 << 254, Q - 1, top]
    return [(a, b) for a in vals for b in vals]


def redc_extremes():
    """T = q 2^256 - 1 (largest input), T < 2^256 (high half zero), T = h 2^256 (low half zero), and neighbours."""
    return [Q * MONT - 1, Q * MONT - MONT, (Q - 1) * MONT, MONT, (Q - 1) * MONT + MONT - 1,
            0, 1, Q - 1, Q, MONT - 1, MONT - Q, MONT - 1 - (MONT - 1) % Q,
            (1 << 254) * 2 - 1, Q * Q, 2 * Q * Q - 1, (Q - 1) * (Q - 1) + Q * Q]


def mulsub_extremes():
    m = Q - 1
    return [(m, m, 0, 0), (0, 0, m, m), (m, m, m, m), (0, 0, 0, 0), (m, m, 1, 0), (1, 1, m, m), (m, 1, 1, m),
            (m, m, m, m - 1), (m, m - 1, m, m), (1, 0, 0, 1), (0, 1, 1, 0)]


def f2_mul_extremes():
    m = Q - 1
    vals = [(m, m), (m, 0), (0, m), (0, 0), (1, 0), (0, 1), (m, 1), (1, m)]
    return [(a, b) for a in vals for b in vals]


def f2_mulsub_extremes():
    m, z = (Q - 1, Q - 1), (0, 0)
    return [(m, m, z, z), (z, z, m, m), (m, m, m, m), (z, z, z, z), ((Q - 1, 0), (Q - 1, 0), (0, Q - 1), (0, Q - 1)),
            ((0, Q - 1), (0, Q - 1), (Q - 1, 0), (Q - 1, 0))]


def inverse_edge_values(p):
    """Inputs for the field inversions (raw Montgomery representatives) that sit on the division-step loop's edges."""
    return [0, 1, 2, 3, p - 1, p - 2, (p - 1) // 2, (p + 1) // 2, MONT % p, MONT * MONT % p, 1 << 253, (1 << 30) - 1,
            1 << 30, (1 << 60) + 1, p - (MONT % p)]
