"""Batched-affine pair rounds (csrc/msm_pair.cuh) and the division-step inversion (csrc/fp.cuh fp_inv_fast), run on the
CPU through the library's host hooks -- the SAME __host__ __device__ code the CUDA kernels execute -- against the oracle.

Covers what the GPU suite cannot reach cheaply: every special pair of the affine addition (infinity operands, P + P,
P + (-P)), odd bucket lengths carried between rounds, threads that start and end in the middle of a bucket, empty
buckets between them, and surplus threads.  No GPU is touched.
"""
import random

import pytest

from arith_cases import inverse_edge_values
from nzcp_circom_b200 import api
from oracle import bn254 as ob
from oracle import prover as oprover
from util import g1_plain_bytes, g2_plain_bytes, le32

R, Q = ob.R_MOD, ob.Q_MOD
MONT = 1 << 256


@pytest.mark.parametrize("field,p", [(0, R), (1, Q)])
def test_inverse_by_division_steps(lib, field, p):
    rng = random.Random(41 + field)
    vals = inverse_edge_values(p) + [rng.randrange(p) for _ in range(3000)]
    a = b"".join(le32(x) for x in vals)
    # Montgomery in, Montgomery out: x = aR  ->  a^-1 R = R^2 / x
    exp = b"".join(le32(0 if x == 0 else pow(x, -1, p) * MONT * MONT % p) for x in vals)
    assert api.host_field_op(field, 3, a, a, len(vals)) == exp      # fp_inv_fast
    assert api.host_field_op(field, 4, a, a, len(vals)) == exp      # Fermat ladder (what the rest of the host glue uses)


@pytest.fixture(scope="module")
def fixed_bases():
    return ob.FixedBase(ob.G1, ob.G1_GEN), ob.FixedBase(ob.G2, ob.G2_GEN)


def _check(g2, pts, scalars, c, rounds, k):
    """Both round-1 variants: operands gathered a second time from the window table by the backward pass (the default), and
    staged by the forward pass / streamed by the backward pass ("pair_stage" = 1)."""
    curve = ob.G2 if g2 else ob.G1
    enc = ob.g2_to_bytes_mont if g2 else ob.g1_to_bytes_mont
    bases = b"".join(enc(P) for P in pts)
    sc = b"".join(le32(s) for s in scalars)
    exp = curve.to_affine(oprover.multiexp(curve, pts, scalars))
    try:
        for stage in (1, 0):
            api.tuning_set("pair_stage", stage)
            got = api.host_msm_sim(bases, sc, len(pts), g2=g2, window_bits=c, rounds=rounds, adds_per_thread=k)
            assert got == (g2_plain_bytes(exp) if g2 else g1_plain_bytes(exp)), (g2, c, rounds, k, stage)
    finally:
        api.tuning_set("pair_stage", 0)


@pytest.mark.parametrize("g2", [False, True])
@pytest.mark.parametrize("rounds,k", [(0, 4), (1, 4), (2, 4), (3, 4), (3, 16), (2, 32), (1, 8)])
def test_pair_rounds_uniform(lib, fixed_bases, g2, rounds, k):
    rng = random.Random(rounds * 10 + k + g2)
    n = 24 if g2 else 60
    pts = [fixed_bases[g2].mul(rng.randrange(1, R)) for _ in range(n)]
    scalars = [rng.randrange(R) for _ in range(n)]
    _check(g2, pts, scalars, 3, rounds, k)      # 4 buckets: long lists, several threads per bucket
    if not g2:
        _check(g2, pts, scalars, 7, rounds, k)  # 64 buckets: short lists, empty buckets, threads spanning many buckets


@pytest.mark.parametrize("g2", [False, True])
@pytest.mark.parametrize("rounds", [1, 2, 3])
def test_pair_rounds_special_pairs(lib, fixed_bases, g2, rounds):
    """Equal points (tangent case), opposite points (sum = infinity), infinity bases, witness-like scalars."""
    rng = random.Random(7 + rounds + g2)
    fb = fixed_bases[g2]
    curve = ob.G2 if g2 else ob.G1
    P, Qp = fb.mul(5), fb.mul(77)
    # all points equal, equal scalars: every pair of every round is a doubling
    _check(g2, [P] * 16, [1] * 16, 2, rounds, 4)
    _check(g2, [P] * 13, [R - 1] * 13, 4, rounds, 4)
    # P, -P adjacent in the same bucket: infinity results feed the next round as operands
    _check(g2, [P, curve.neg(P)] * 6, [3] * 12, 2, rounds, 4)
    _check(g2, [P, curve.neg(P), Qp, Qp, None, P, None, None, curve.neg(Qp), Qp, P], [1] * 11, 2, rounds, 4)
    # everything cancels
    _check(g2, [P, curve.neg(P)], [12345, 12345], 4, rounds, 4)
    _check(g2, [None] * 9, [rng.randrange(R) for _ in range(9)], 3, rounds, 4)
    # mixed
    pts = [P, P, curve.neg(P), None, fb.mul(9), None, P, fb.mul(11)] + [fb.mul(rng.randrange(1, R)) for _ in range(12 if g2 else 30)]
    scalars = [3, 3, 3, 7, 0, 0, R - 1, 1] + [rng.choice([0, 1, 1, rng.randrange(256), rng.randrange(R)]) for _ in range(len(pts) - 8)]
    _check(g2, pts, scalars, 4, rounds, 4)
    _check(g2, pts, scalars, 2, rounds, 16)


def test_pair_rounds_empty_and_single(lib, fixed_bases):
    _check(False, [], [], 4, 2, 4)
    _check(False, [fixed_bases[0].mul(3)], [R - 1], 4, 3, 4)
    _check(False, [fixed_bases[0].mul(3)], [0], 4, 3, 4)
