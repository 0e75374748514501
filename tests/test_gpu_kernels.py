"""GPU parity: field arithmetic, NTT pipeline and MSM kernels vs the CPU oracle -- all through the C ABI.

Bar: bit-exact (integer work).  Sizes are what the pure-Python oracle finishes in seconds; full-size runs are covered
by size-independent properties in test_gpu_prove.py.
"""
import random

import pytest

from arith_cases import inverse_edge_values, mul_targeted, targets
from nzcp_circom_b200 import api
from nzcp_circom_b200._lib import NzcpError
from oracle import bn254 as ob
from oracle import prover as oprover
from util import g1_plain_bytes, g2_plain_bytes, le32

pytestmark = pytest.mark.gpu

R, Q = ob.R_MOD, ob.Q_MOD
MONT = 1 << 256


def _edge_values(p):
    return [0, 1, 2, p - 1, p - 2, MONT % p, (MONT * MONT) % p, (1 << 253), (1 << 224) - 1, 0xFFFFFFFF, 1 << 32]


def test_selftest_device_vs_host(lib):
    assert api.selftest(0, 1, 8192) == 0
    assert api.selftest(0, 99, 257) == 0


@pytest.mark.parametrize("field,p", [(0, R), (1, Q)])
def test_field_ops_limb_exact(lib, field, p):
    rng = random.Random(5 + field)
    ev = _edge_values(p)
    a = [x for x in ev for _ in ev] + [rng.randrange(p) for _ in range(4000)]
    b = [y for _ in ev for y in ev] + [rng.randrange(p) for _ in range(4000)]
    # operands solved so that the Montgomery product lands on 0, 1, p-1 .. p-64, ...: the final subtraction's edge
    tgt = [mul_targeted(rng, y, p) for y in targets(p) for _ in range(4)]
    a += [x for x, _ in tgt]
    b += [y for _, y in tgt]
    ab = b"".join(le32(x) for x in a)
    bb = b"".join(le32(x) for x in b)
    rinv = pow(MONT, -1, p)
    n = len(a)
    for op, fn in ((0, lambda x, y: x * y * rinv % p), (1, lambda x, y: (x + y) % p), (2, lambda x, y: (x - y) % p)):
        exp = b"".join(le32(fn(x, y)) for x, y in zip(a, b))
        assert api.field_op(field, op, ab, bb, n) == exp            # IMAD carry-chain PTX path
        assert api.field_op(field, op + 3, ab, bb, n) == exp        # portable path compiled for the device


@pytest.mark.parametrize("field,p", [(0, R), (1, Q)])
def test_field_inverses_device(lib, field, p):
    """Ops 6 (division steps, what the pair rounds run) and 7 (Fermat ladder, what xyzz_to_affine runs)."""
    rng = random.Random(41 + field)
    vals = inverse_edge_values(p) + [rng.randrange(p) for _ in range(1 << 16)]
    a = b"".join(le32(x) for x in vals)
    # Montgomery in, Montgomery out: x = aR  ->  a^-1 R = R^2 / x
    exp = b"".join(le32(0 if x == 0 else pow(x, -1, p) * MONT * MONT % p) for x in vals)
    assert api.field_op(field, 6, a, a, len(vals)) == exp
    assert api.field_op(field, 7, a, a, len(vals)) == exp


def _mont_bytes(vals):
    return bytearray(b"".join(le32(v * MONT % R) for v in vals))


def _from_mont_bytes(buf):
    rinv = pow(MONT, -1, R)
    return [int.from_bytes(buf[i:i + 32], "little") * rinv % R for i in range(0, len(buf), 32)]


@pytest.mark.parametrize("log_n", [1, 2, 3, 5, 8, 10, 11, 12, 13])
def test_ntt_forward_inverse_vs_oracle(lib, log_n):
    rng = random.Random(log_n)
    n = 1 << log_n
    a = [rng.randrange(R) for _ in range(n)]
    a[0], a[-1] = R - 1, 0
    buf = _mont_bytes(a)
    api.ntt(buf, log_n, inverse=False)
    assert _from_mont_bytes(buf) == ob.ntt(a)
    buf = _mont_bytes(a)
    api.ntt(buf, log_n, inverse=True)
    assert _from_mont_bytes(buf) == ob.ntt(a, inverse=True)


def _coset_oracle(a, log_n):
    inc = 25 if log_n == ob.FR_S else ob.FR_W[log_n + 1]
    coef = ob.ntt(a, inverse=True)
    k, sc = 1, []
    for x in coef:
        sc.append(x * k % R)
        k = k * inc % R
    return ob.ntt(sc)


@pytest.mark.parametrize("log_n,batch", [(1, 1), (2, 3), (4, 3), (9, 3), (10, 2), (11, 3), (13, 3)])
def test_ntt_coset_pipeline_vs_oracle(lib, log_n, batch):
    """iNTT -> x inc^i -> NTT, the per-polynomial H pipeline of groth16_prove.js, batched as the prover runs it."""
    rng = random.Random(100 + log_n)
    n = 1 << log_n
    polys = [[rng.randrange(R) for _ in range(n)] for _ in range(batch)]
    buf = bytearray(b"".join(bytes(_mont_bytes(p)) for p in polys))
    api.ntt_coset(buf, log_n, batch)
    got = _from_mont_bytes(buf)
    for k, p in enumerate(polys):
        assert got[k * n:(k + 1) * n] == _coset_oracle(p, log_n)


@pytest.mark.parametrize("log_n,batch", [(10, 1), (10, 3), (12, 3), (14, 5), (16, 3)])
def test_ntt_coset_tma_and_thread_loaded_low_pass_agree(lib, log_n, batch):
    """Both low-pass kernels -- TMA-staged (bulk copies + mbarrier, shared-memory twiddles; persistent blocks that walk
    several tiles, incl. grids smaller and larger than the tile count) and thread-loaded -- against the C oracle."""
    import numpy as np
    from oracle import cref
    n = 1 << log_n
    rs = np.random.RandomState(log_n * 7 + batch)
    x = rs.randint(0, 2 ** 32, size=(batch * n, 8), dtype=np.uint64).astype(np.uint32)
    x[:, 7] &= 0x1FFFFFFF
    x[0] = 0
    exp = x.copy()
    for k in range(batch):
        e = np.ascontiguousarray(exp[k * n:(k + 1) * n])
        cref.ntt_coset(e, log_n, threads=cref.max_threads())
        exp[k * n:(k + 1) * n] = e
    try:
        for tma in (1, 0):
            api.tuning_set("ntt_tma", tma)
            g = x.copy()
            api.ntt_coset(g, log_n, batch=batch)
            assert np.array_equal(g, exp), "ntt_tma=%d" % tma
    finally:
        api.tuning_set("ntt_tma", 1)


def test_ntt_roundtrip_large(lib):
    """2^20 (the NZCP domain) and 2^22: forward then inverse is the identity; linearity against a second vector."""
    import numpy as np
    for log_n in (20, 22):
        n = 1 << log_n
        rs = np.random.RandomState(log_n)
        x = rs.randint(0, 2 ** 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
        x[:, 7] &= 0x0FFFFFFF                      # < 2^252 < r: canonical
        y = x.copy()
        api.ntt(y, log_n, inverse=False)
        assert not np.array_equal(x, y)
        api.ntt(y, log_n, inverse=True)
        assert np.array_equal(x, y)


def _rand_points(curve, fb, rng, n):
    return [fb.mul(rng.randrange(1, R)) for _ in range(n)]


@pytest.fixture(scope="module")
def fixed_bases():
    return ob.FixedBase(ob.G1, ob.G1_GEN), ob.FixedBase(ob.G2, ob.G2_GEN)


def _msm_case(g2, pts, scalars, window_bits=0):
    curve = ob.G2 if g2 else ob.G1
    enc = ob.g2_to_bytes_mont if g2 else ob.g1_to_bytes_mont
    bases = b"".join(enc(P) for P in pts)
    sc = b"".join(le32(s) for s in scalars)
    got, _ = api.msm(bases, sc, len(pts), g2=g2, window_bits=window_bits)
    exp = curve.to_affine(oprover.multiexp(curve, pts, scalars))
    assert got == (g2_plain_bytes(exp) if g2 else g1_plain_bytes(exp))


@pytest.mark.parametrize("g2", [False, True])
@pytest.mark.parametrize("n", [0, 1, 2, 17, 300])
def test_msm_vs_oracle_uniform(lib, fixed_bases, g2, n):
    rng = random.Random(n * 2 + g2)
    pts = _rand_points(None, fixed_bases[g2], rng, n)
    scalars = [rng.randrange(R) for _ in range(n)]
    _msm_case(g2, pts, scalars)


@pytest.mark.parametrize("g2", [False, True])
def test_msm_edge_cases(lib, fixed_bases, g2):
    """Witness-like scalars (0/1/bytes), r-1, infinity bases, repeated and opposite points (exercise the doubling and
    cancellation branches of the bucket adds)."""
    rng = random.Random(77 + g2)
    fb = fixed_bases[g2]
    curve = ob.G2 if g2 else ob.G1
    P = fb.mul(5)
    pts = [P, P, curve.neg(P), None, fb.mul(9), None, P, fb.mul(11)] + _rand_points(None, fb, rng, 120)
    scalars = [3, 3, 3, 7, 0, 0, R - 1, 1] + [rng.choice([0, 1, 1, rng.randrange(256), rng.randrange(R)])
                                               for _ in range(120)]
    _msm_case(g2, pts, scalars)
    # all points equal with equal scalars: every bucket add after the first is a doubling
    _msm_case(g2, [P] * 64, [1] * 64)
    _msm_case(g2, [P] * 64, [R - 1] * 64)
    # sum is the point at infinity
    _msm_case(g2, [P, curve.neg(P)], [12345, 12345])
    _msm_case(g2, [None] * 10, [rng.randrange(R) for _ in range(10)])


@pytest.mark.parametrize("c", [2, 5, 9, 13, 16, 17, 19])   # <= 16: shared-memory histogram; above: global atomics
def test_msm_window_sizes(lib, fixed_bases, c):
    rng = random.Random(c)
    pts = _rand_points(None, fixed_bases[0], rng, 200)
    scalars = [rng.randrange(R) for _ in range(190)] + [R - 1] * 10
    _msm_case(False, pts, scalars, window_bits=c)


def test_msm_default_window_mid_size(lib):
    """2^13 points with the default window (c = 10) and witness-like scalars: heavy bucket "1", adaptive task length,
    two-stage heavy combine -- against the C oracle (the Python one is too slow here)."""
    from oracle import cref
    n = 1 << 13
    bases = bytes(api.synth_points(9, n))
    rng = random.Random(12)
    sc = [rng.choice([0, 1, 1, 1, rng.randrange(256), rng.randrange(R)]) for _ in range(n)]
    scb = b"".join(le32(x) for x in sc)
    got, _ = api.msm(bases, scb, n)
    assert got == cref.msm(bases, scb, n, False, 4)
    b2 = bytes(api.synth_points(10, 2048, g2=True))
    got2, _ = api.msm(b2, scb[:2048 * 32], 2048, g2=True)
    assert got2 == cref.msm(b2, scb[:2048 * 32], 2048, True, 4)


def test_msm_rejects_non_canonical_scalar(lib, fixed_bases):
    pts = _rand_points(None, fixed_bases[0], random.Random(3), 4)
    bases = b"".join(ob.g1_to_bytes_mont(P) for P in pts)
    sc = le32(1) + le32(R) + le32(2) + le32(3)
    with pytest.raises(NzcpError) as e:
        api.msm(bases, sc, 4)
    assert e.value.code == -7


def test_msm_large_linearity(lib):
    """2^18 points (generated on the GPU by the synthetic setup's fixed-base kernel is not exposed here, so bases are
    small multiples built by doubling on the host): MSM(s) + MSM(t) == MSM(s + t) and MSM(k*1) == k * sum(P)."""
    import numpy as np
    n = 1 << 14
    fb = ob.FixedBase(ob.G1, ob.G1_GEN)
    base_pts = [fb.mul(i + 1) for i in range(64)]
    rng = random.Random(1)
    pts = [base_pts[rng.randrange(64)] for _ in range(n)]
    bases = b"".join(ob.g1_to_bytes_mont(P) for P in pts)
    s = [rng.randrange(R) for _ in range(n)]
    t = [rng.randrange(R) for _ in range(n)]
    st = [(a + b) % R for a, b in zip(s, t)]

    def run(v):
        out, _ = api.msm(bases, b"".join(le32(x) for x in v), n)
        return None if out == bytes(64) else (int.from_bytes(out[:32], "little"), int.from_bytes(out[32:], "little"))
    assert ob.G1.add(run(s), run(t)) == run(st)
    # closed form: every base is k_i * G, so the MSM is (sum s_i k_i) * G
    ks = {id(P): i + 1 for i, P in enumerate(base_pts)}
    tot = sum(x * ks[id(P)] for x, P in zip(s, pts)) % R
    assert run(s) == fb.mul(tot)


@pytest.fixture
def forced_rounds():
    """Force the batched-affine pair rounds on (small inputs would run without them) and restore the defaults after."""
    def force(rounds, k=16):
        api.tuning_set("msm_rounds", rounds)
        api.tuning_set("prover_rounds_w", rounds)
        api.tuning_set("prover_rounds_h", rounds)
        for name in ("pair_k1", "pair_k2", "pair_k3"):
            api.tuning_set(name, k)
    yield force
    for name, v in (("msm_rounds", -1), ("prover_rounds_w", -1), ("prover_rounds_h", -1), ("pair_k1", 16), ("pair_k2", 16),
                    ("pair_k3", 16), ("pair_stage", 0), ("pair_prefetch_fwd", 0), ("pair_prefetch_bwd", 0), ("gather_hint", 0)):
        api.tuning_set(name, v)


@pytest.mark.parametrize("rounds,k", [(1, 16), (2, 16), (3, 16), (3, 32), (2, 8)])
@pytest.mark.parametrize("g2", [False, True])
def test_msm_pair_rounds_forced_edge_cases(lib, fixed_bases, forced_rounds, g2, rounds, k):
    """The edge-case MSMs again with the pair rounds forced on: equal points (tangent pairs), opposite points (infinity
    results carried into the next round), infinity bases, witness-like scalars, several window sizes."""
    forced_rounds(rounds, k)
    rng = random.Random(177 + g2 + rounds)
    fb = fixed_bases[g2]
    curve = ob.G2 if g2 else ob.G1
    P = fb.mul(5)
    pts = [P, P, curve.neg(P), None, fb.mul(9), None, P, fb.mul(11)] + _rand_points(None, fb, rng, 120)
    scalars = [3, 3, 3, 7, 0, 0, R - 1, 1] + [rng.choice([0, 1, 1, rng.randrange(256), rng.randrange(R)])
                                               for _ in range(120)]
    for c in (0, 2, 5):
        _msm_case(g2, pts, scalars, window_bits=c)
    _msm_case(g2, [P] * 64, [1] * 64, window_bits=3)
    _msm_case(g2, [P] * 61, [R - 1] * 61, window_bits=4)
    _msm_case(g2, [P, curve.neg(P)] * 8, [12345] * 16, window_bits=3)
    _msm_case(g2, [None] * 10, [rng.randrange(R) for _ in range(10)])
    _msm_case(g2, [], [])
    _msm_case(g2, [P], [R - 1])


@pytest.mark.parametrize("stage", [1, 0])
@pytest.mark.parametrize("rounds", [1, 2, 3])
def test_msm_pair_rounds_forced_mid_size(lib, forced_rounds, rounds, stage):
    """2^13 points, witness-like scalars (heavy bucket "1"), vs the C oracle, every round count; round 1 with its operands
    gathered twice (default) and staged by the forward pass ("pair_stage" = 1), with and without operand prefetch."""
    from oracle import cref
    forced_rounds(rounds, 32)
    api.tuning_set("pair_stage", stage)
    api.tuning_set("pair_prefetch_fwd", 1 - stage)
    api.tuning_set("pair_prefetch_bwd", 2 * (1 - stage))
    api.tuning_set("gather_hint", 1 - stage)          # the fetch-size-qualified gathers ride along with the second variant
    n = 1 << 13
    bases = bytes(api.synth_points(9, n))
    rng = random.Random(12)
    sc = [rng.choice([0, 1, 1, 1, rng.randrange(256), rng.randrange(R)]) for _ in range(n)]
    scb = b"".join(le32(x) for x in sc)
    got, _ = api.msm(bases, scb, n)
    assert got == cref.msm(bases, scb, n, False, 4)
    b2 = bytes(api.synth_points(10, 2048, g2=True))
    got2, _ = api.msm(b2, scb[:2048 * 32], 2048, g2=True)
    assert got2 == cref.msm(b2, scb[:2048 * 32], 2048, True, 4)
