"""groth16.verify -- CPU pairing check (the step after the hot path; SURVEY.md section 8f row 2).

Mirrors snarkjs 0.4.12 src/groth16_verify.js (upstream, not vendored: /root/reference/package.json:12,
yarn.lock:987-999):  e(-A, B) * e(alpha1, beta2) * e(vk_x, gamma2) * e(C, delta2) == 1  with
vk_x = IC[0] + sum_i pub_i * IC[i+1].  snarkjs runs this on the CPU as well (3 pairings + an nPublic-term MSM);
it is host logic here too, in plain Python ints.  The optimal-ate pairing is checked by bilinearity tests
(tests/test_verifier.py); nothing in this file is on the GPU path.
"""

Q = 21888242871839275222246405745257275088696311157297823662689037894645226208583
R = 21888242871839275222246405745257275088548364400416034343698204186575808495617
ATE_LOOP = 29793968203157093288          # 6x + 2, x = 4965661367192848881
XI = (9, 1)                              # Fq6/Fq12 non-residue 9 + u


# ---------------------------------------------------------------------------------------- Fq2
def f2_add(a, b):
    return ((a[0] + b[0]) % Q, (a[1] + b[1]) % Q)


def f2_sub(a, b):
    return ((a[0] - b[0]) % Q, (a[1] - b[1]) % Q)


def f2_mul(a, b):
    return ((a[0] * b[0] - a[1] * b[1]) % Q, (a[0] * b[1] + a[1] * b[0]) % Q)


def f2_sqr(a):
    return ((a[0] + a[1]) * (a[0] - a[1]) % Q, 2 * a[0] * a[1] % Q)


def f2_neg(a):
    return ((-a[0]) % Q, (-a[1]) % Q)


def f2_conj(a):
    return (a[0], (-a[1]) % Q)


def f2_inv(a):
    d = pow(a[0] * a[0] + a[1] * a[1], -1, Q)
    return (a[0] * d % Q, (-a[1]) * d % Q)


def f2_muls(a, k):
    return (a[0] * k % Q, a[1] * k % Q)


def f2_mul_xi(a):
    return ((9 * a[0] - a[1]) % Q, (a[0] + 9 * a[1]) % Q)


def f2_pow(a, e):
    r_ = (1, 0)
    while e:
        if e & 1:
            r_ = f2_mul(r_, a)
        a = f2_sqr(a)
        e >>= 1
    return r_


F2_ZERO, F2_ONE = (0, 0), (1, 0)

# ---------------------------------------------------------------------------------------- Fq12 = Fq2[w]/(w^6 - xi)
F12_ONE = [F2_ONE] + [F2_ZERO] * 5


def f12_mul(a, b):
    acc = [[0, 0] for _ in range(11)]
    for i in range(6):
        ai = a[i]
        if ai[0] == 0 and ai[1] == 0:
            continue
        for j in range(6):
            bj = b[j]
            if bj[0] == 0 and bj[1] == 0:
                continue
            t = acc[i + j]
            t[0] += ai[0] * bj[0] - ai[1] * bj[1]
            t[1] += ai[0] * bj[1] + ai[1] * bj[0]
    out = []
    for k in range(6):
        lo = acc[k]
        if k < 5:
            hi = acc[k + 6]
            out.append(((lo[0] + 9 * hi[0] - hi[1]) % Q, (lo[1] + hi[0] + 9 * hi[1]) % Q))
        else:
            out.append((lo[0] % Q, lo[1] % Q))
    return out


def f12_pow(a, e):
    r_ = F12_ONE
    for bit in bin(e)[2:]:
        r_ = f12_mul(r_, r_)
        if bit == "1":
            r_ = f12_mul(r_, a)
    return r_


FINAL_EXP = (Q ** 12 - 1) // R


# ---------------------------------------------------------------------------------------- curve helpers
def g1_on_curve(P):
    return P is None or (P[1] * P[1] - P[0] * P[0] * P[0] - 3) % Q == 0


_B2 = f2_mul((3, 0), f2_inv(XI))


def g2_on_curve(Pt):
    if Pt is None:
        return True
    x, y = Pt
    return f2_sub(f2_sqr(y), f2_add(f2_mul(f2_sqr(x), x), _B2)) == F2_ZERO


def g1_add(P, S):
    if P is None:
        return S
    if S is None:
        return P
    if P[0] == S[0]:
        if (P[1] + S[1]) % Q == 0:
            return None
        lam = 3 * P[0] * P[0] * pow(2 * P[1], -1, Q) % Q
    else:
        lam = (S[1] - P[1]) * pow(S[0] - P[0], -1, Q) % Q
    x3 = (lam * lam - P[0] - S[0]) % Q
    return (x3, (lam * (P[0] - x3) - P[1]) % Q)


def g1_mul(P, k):
    acc = None
    while k:
        if k & 1:
            acc = g1_add(acc, P)
        P = g1_add(P, P)
        k >>= 1
    return acc


def g1_neg(P):
    return None if P is None else (P[0], (-P[1]) % Q)


def g2_add(P, S):
    if P is None:
        return S
    if S is None:
        return P
    if P[0] == S[0]:
        if f2_add(P[1], S[1]) == F2_ZERO:
            return None
        lam = f2_mul(f2_muls(f2_sqr(P[0]), 3), f2_inv(f2_muls(P[1], 2)))
    else:
        lam = f2_mul(f2_sub(S[1], P[1]), f2_inv(f2_sub(S[0], P[0])))
    x3 = f2_sub(f2_sub(f2_sqr(lam), P[0]), S[0])
    return (x3, f2_sub(f2_mul(lam, f2_sub(P[0], x3)), P[1]))


def g2_mul(P, k):
    acc = None
    while k:
        if k & 1:
            acc = g2_add(acc, P)
        P = g2_add(P, P)
        k >>= 1
    return acc


# Frobenius on the twist: (x, y) -> (conj(x) * xi^((q-1)/3), conj(y) * xi^((q-1)/2))
_G12 = f2_pow(XI, (Q - 1) // 3)
_G13 = f2_pow(XI, (Q - 1) // 2)


def _frob_twist(Pt):
    return (f2_mul(f2_conj(Pt[0]), _G12), f2_mul(f2_conj(Pt[1]), _G13))


def _line(T, S, P):
    """Line through T and S (twist points, affine; T == S -> tangent) evaluated at P in G1, as a sparse Fq12
    element  yP + (-lam xP) w + (lam xT - yT) w^3 ; returns (line, T + S)."""
    if T[0] == S[0] and T[1] == S[1]:
        lam = f2_mul(f2_muls(f2_sqr(T[0]), 3), f2_inv(f2_muls(T[1], 2)))
    elif T[0] == S[0]:
        # vertical line: xP - xT w^2
        return [(P[0], 0), F2_ZERO, f2_neg(T[0]), F2_ZERO, F2_ZERO, F2_ZERO], None
    else:
        lam = f2_mul(f2_sub(S[1], T[1]), f2_inv(f2_sub(S[0], T[0])))
    x3 = f2_sub(f2_sub(f2_sqr(lam), T[0]), S[0])
    y3 = f2_sub(f2_mul(lam, f2_sub(T[0], x3)), T[1])
    line = [(P[1], 0), f2_neg(f2_muls(lam, P[0])), F2_ZERO, f2_sub(f2_mul(lam, T[0]), T[1]), F2_ZERO, F2_ZERO]
    return line, (x3, y3)


def miller_loop(P, Qt):
    """f_{6x+2,Q}(P) times the two Frobenius lines; P in G1 affine, Qt in G2 (twist) affine."""
    if P is None or Qt is None:
        return F12_ONE
    f = F12_ONE
    T = Qt
    for bit in bin(ATE_LOOP)[3:]:
        line, T = _line(T, T, P)
        f = f12_mul(f12_mul(f, f), line)
        if bit == "1":
            line, T = _line(T, Qt, P)
            f = f12_mul(f, line)
    Q1 = _frob_twist(Qt)
    Q2 = _frob_twist(Q1)
    nQ2 = (Q2[0], f2_neg(Q2[1]))
    line, T = _line(T, Q1, P)
    f = f12_mul(f, line)
    line, T = _line(T, nQ2, P)
    f = f12_mul(f, line)
    return f


def final_exp(f):
    return f12_pow(f, FINAL_EXP)


def pairing(P, Qt):
    return final_exp(miller_loop(P, Qt))


def pairing_product_is_one(pairs):
    f = F12_ONE
    for P, Qt in pairs:
        f = f12_mul(f, miller_loop(P, Qt))
    return final_exp(f) == F12_ONE


def same_ratio(a, b, c, d):
    """snarkjs sameRatio(a, b, c, d): e(a, d) == e(b, c) -- the pairing half of `zkey verify` (api.zkey_verify)."""
    return pairing_product_is_one([(a, d), (g1_neg(b), c)])


# ---------------------------------------------------------------------------------------- snarkjs-shaped verify
class _BadPoint(ValueError):
    pass


def _coord(v):
    """Canonical field element: a decimal string / int in [0, Q).  Anything else is rejected, never reduced."""
    x = int(v)
    if not 0 <= x < Q:
        raise _BadPoint("coordinate not in [0, q)")
    return x


def _g1(obj):
    """snarkjs point object [x, y, z] with z in {"0", "1"} (affine; ffjavascript's zero is ["0", "1", "0"])."""
    x, y, z = (_coord(v) for v in obj)
    if z == 0:
        return None
    if z != 1:
        raise _BadPoint("G1 point is not affine")
    return (x, y)


def _g2(obj):
    (x0, x1), (y0, y1), (z0, z1) = ((_coord(a), _coord(b)) for a, b in obj)
    if z0 == 0 and z1 == 0:
        return None
    if (z0, z1) != (1, 0):
        raise _BadPoint("G2 point is not affine")
    return ((x0, x1), (y0, y1))


def g2_in_subgroup(Pt):
    """r * P == O.  The twist E'(Fq2) has order r * (2q - r): a point on the curve is not automatically in G2, and the
    optimal-ate Miller loop is only a pairing on the r-torsion (the invalid-point surface EIP-197 and arkworks close)."""
    return Pt is None or g2_mul(Pt, R) is None


_vk_ok = {}     # content fingerprint of a verification key -> checked once (points on curve, G2 points in the subgroup)


def _check_vk(vk):
    try:
        key = hash(repr((vk["vk_alpha_1"], vk["vk_beta_2"], vk["vk_gamma_2"], vk["vk_delta_2"], vk["IC"])))
    except (KeyError, TypeError):
        return False
    ent = _vk_ok.get(key)
    if ent is not None:
        return ent
    try:
        ic = [_g1(p) for p in vk["IC"]]
        a1 = _g1(vk["vk_alpha_1"])
        g2s = [_g2(vk[k]) for k in ("vk_beta_2", "vk_gamma_2", "vk_delta_2")]
        ok = all(g1_on_curve(p) for p in ic + [a1]) and a1 is not None and \
            all(p is not None and g2_on_curve(p) and g2_in_subgroup(p) for p in g2s)
    except (_BadPoint, ValueError, TypeError, KeyError):
        ok = False
    if len(_vk_ok) > 64:
        _vk_ok.clear()
    _vk_ok[key] = ok
    return ok


def verify(vk, public_signals, proof, logger=None):
    """snarkjs groth16.verify(vk_verifier, publicSignals, proof) -> bool.

    Stricter than snarkjs 0.4.12 on malformed input (which it never checks): coordinates must be canonical (< q, not
    silently reduced), points affine and on the curve, pi_b (and the key's G2 points) in the order-r subgroup."""
    if not _check_vk(vk):
        if logger:
            logger.error("Invalid verification key")
        return False
    ic = [_g1(p) for p in vk["IC"]]
    try:
        pubs = [int(s) for s in public_signals]
    except (ValueError, TypeError):
        return False
    if len(pubs) + 1 != len(ic):
        if logger:
            logger.error("Invalid number of public signals")
        return False
    for s in pubs:
        if not 0 <= s < R:
            if logger:
                logger.error("Public input not in field")
            return False
    try:
        A, B, Cc = _g1(proof["pi_a"]), _g2(proof["pi_b"]), _g1(proof["pi_c"])
    except (_BadPoint, ValueError, TypeError, KeyError):
        if logger:
            logger.error("Invalid proof point")
        return False
    if not (g1_on_curve(A) and g2_on_curve(B) and g1_on_curve(Cc) and g2_in_subgroup(B)):
        if logger:
            logger.error("Invalid proof point")
        return False
    vk_x = ic[0]
    for s, P in zip(pubs, ic[1:]):
        if s:
            vk_x = g1_add(vk_x, g1_mul(P, s))
    ok = pairing_product_is_one([
        (g1_neg(A), B),
        (_g1(vk["vk_alpha_1"]), _g2(vk["vk_beta_2"])),
        (vk_x, _g2(vk["vk_gamma_2"])),
        (Cc, _g2(vk["vk_delta_2"])),
    ])
    if logger:
        (logger.info if ok else logger.error)("OK!" if ok else "Invalid proof")
    return ok
