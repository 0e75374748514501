"""Expected outputs of `zkey contribute` / `zkey beacon`: a second, pure-Python restatement of snarkjs 0.4.12
zkey_contribute.js / zkey_beacon.js (csrc/contribute.cu restates the same steps in C++).

Shared with the library: nothing but the published algorithm.  BLAKE2b-512 and SHA-256 are hashlib's; the ChaCha of
ffjavascript random.js is written out below and tied to RFC 8439 by its block test vector; the square roots, the sign
convention (wasmcurves isNegative: the plain value > (q-1)/2; for Fq2 c1 decides, c0 when c1 = 0) and G1/G2.fromRng
follow the published code; curve arithmetic is oracle/bn254's and verifier.py's.

contribution() returns k, the new section-10 record and the contribution hash for a given input key.  The contributed key
itself is expected in closed form: formats.write_zkey(setup.make_zkey(..., delta = delta0 * k)) with section 10 replaced
(with_section10), which does not depend on any per-point multiplication agreeing.
"""
import hashlib
import struct

from nzcp_circom_b200 import verifier as V
from oracle import formats
from oracle.bn254 import (CURVE_B2, G1, G2, MONT_R, Q_MOD, R_MOD, g1_from_bytes_mont, g1_to_bytes_mont,
                          g2_from_bytes_mont, g2_to_bytes_mont)

M32 = 0xFFFFFFFF


# ------------------------------------------------------------------------------------------------ ChaCha
def _rotl(x, c):
    return ((x << c) | (x >> (32 - c))) & M32


def chacha_block(state):
    """RFC 8439 2.3: 10 double rounds over the 16-word state, plus the input state."""
    x = list(state)

    def qr(a, b, c, d):
        x[a] = (x[a] + x[b]) & M32; x[d] = _rotl(x[d] ^ x[a], 16)
        x[c] = (x[c] + x[d]) & M32; x[b] = _rotl(x[b] ^ x[c], 12)
        x[a] = (x[a] + x[b]) & M32; x[d] = _rotl(x[d] ^ x[a], 8)
        x[c] = (x[c] + x[d]) & M32; x[b] = _rotl(x[b] ^ x[c], 7)

    for _ in range(10):
        qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15)
        qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14)
    return [(a + b) & M32 for a, b in zip(x, state)]


CONSTANTS = [0x61707865, 0x3320646E, 0x79622D32, 0x6B206574]


class ChaCha:
    """ffjavascript ChaCha(seed): seed = 8 u32 words; words 12-15 form a 128-bit block counter starting at 0."""

    def __init__(self, seed_words):
        self.key = list(seed_words)
        self.counter = 0
        self.buf, self.idx = [], 16

    def next_u32(self):
        if self.idx == 16:
            ctr = [(self.counter >> (32 * i)) & M32 for i in range(4)]
            self.buf = chacha_block(CONSTANTS + self.key + ctr)
            self.counter = (self.counter + 1) % (1 << 128)
            self.idx = 0
        self.idx += 1
        return self.buf[self.idx - 1]

    def next_u64(self):
        hi = self.next_u32()
        return hi << 32 | self.next_u32()

    def next_bool(self):
        return self.next_u32() & 1 == 1


def rng_from_digest(d):
    return ChaCha([int.from_bytes(d[4 * i:4 * i + 4], "big") for i in range(8)])


def rng_contribute(seed32):
    """The rng of zkey_contribute with the OS bytes and entropy replaced by a fixed 32-byte digest prefix."""
    return rng_from_digest(seed32)


def rng_beacon(beacon_hash, exp):
    h = bytes(beacon_hash)
    for _ in range(1 << exp):
        h = hashlib.sha256(h).digest()
    return rng_from_digest(h)


# ------------------------------------------------------------------------------------------------ fields and points
def from_rng(rng, p):
    """F.fromRng: 4 x nextU64 little-endian, masked to 254 bits, redrawn while >= p; the value is a Montgomery buffer."""
    while True:
        v = sum(rng.next_u64() << (64 * i) for i in range(4)) & ((1 << 254) - 1)
        if v < p:
            return v * pow(MONT_R, -1, p) % p


def is_negative(a):
    return a > (Q_MOD - 1) // 2


def f2_is_negative(a):
    return is_negative(a[1]) if a[1] else is_negative(a[0])


def f2_sqrt(a):
    """Adj / Rodriguez-Henriquez 2012, Algorithm 9 (q = 3 mod 4); None for a non-square."""
    a1 = V.f2_pow(a, (Q_MOD - 3) // 4)
    alpha = V.f2_mul(V.f2_sqr(a1), a)
    a0 = V.f2_mul(V.f2_conj(alpha), alpha)
    if a0 == (Q_MOD - 1, 0):
        return None
    x0 = V.f2_mul(a1, a)
    if alpha == (Q_MOD - 1, 0):
        x = V.f2_mul((0, 1), x0)
    else:
        x = V.f2_mul(V.f2_pow(V.f2_add((1, 0), alpha), (Q_MOD - 1) // 2), x0)
    assert V.f2_sqr(x) == a
    return x


def g1_from_rng(rng):
    while True:
        x = from_rng(rng, Q_MOD)
        greatest = rng.next_bool()
        y2 = (x * x * x + 3) % Q_MOD
        y = pow(y2, (Q_MOD + 1) // 4, Q_MOD)
        if y * y % Q_MOD == y2:
            break
    if greatest != is_negative(y):
        y = (-y) % Q_MOD
    return (x, y)


H2 = 2 * Q_MOD - R_MOD       # G2 cofactor


def g2_from_rng(rng):
    while True:
        x = (from_rng(rng, Q_MOD), from_rng(rng, Q_MOD))
        greatest = rng.next_bool()
        y = f2_sqrt(V.f2_add(V.f2_mul(V.f2_sqr(x), x), CURVE_B2))
        if y is not None:
            break
    if greatest != f2_is_negative(y):
        y = V.f2_neg(y)
    return G2.mul((x, y), H2)


def hash_to_g2(transcript):
    return g2_from_rng(rng_from_digest(transcript))


# ------------------------------------------------------------------------------------------------ transcript
def u_g1(P):
    return b"\x40" + bytes(63) if P is None else P[0].to_bytes(32, "big") + P[1].to_bytes(32, "big")


def u_g2(P):
    if P is None:
        return b"\x40" + bytes(127)
    return b"".join(c.to_bytes(32, "big") for c in (P[0][1], P[0][0], P[1][1], P[1][0]))


REC_FIXED = 3 * 64 + 128 + 64 + 8


def hash_pub_key(rec):
    """hashPubKey over a record in its zkey layout."""
    return (u_g1(g1_from_bytes_mont(rec[0:64])) + u_g1(g1_from_bytes_mont(rec[64:128]))
            + u_g1(g1_from_bytes_mont(rec[128:192])) + u_g2(g2_from_bytes_mont(rec[192:320])) + rec[320:384])


def parse_mpc(s10):
    """-> (csHash, [record bytes])"""
    n = struct.unpack_from("<I", s10, 64)[0]
    pos, recs = 68, []
    for _ in range(n):
        plen = struct.unpack_from("<I", s10, pos + REC_FIXED - 4)[0]
        recs.append(bytes(s10[pos:pos + REC_FIXED + plen]))
        pos += REC_FIXED + plen
    assert pos == len(s10)
    return bytes(s10[:64]), recs


def record_points(rec):
    return {"deltaAfter": g1_from_bytes_mont(rec[0:64]), "g1_s": g1_from_bytes_mont(rec[64:128]),
            "g1_sx": g1_from_bytes_mont(rec[128:192]), "g2_spx": g2_from_bytes_mont(rec[192:320]),
            "transcript": rec[320:384], "type": struct.unpack_from("<I", rec, 384)[0]}


def sections(buf):
    _, secs = formats.read_container(buf, b"zkey")
    return {sid: bytes(memoryview(buf)[v[0][0]:v[0][0] + v[0][1]]) for sid, v in secs.items()}


def contribution(zkey, name=None, seed=None, beacon_hash=None, exp=None):
    """One contribution (seed: 32 bytes) or beacon (beacon_hash, exp) to the key `zkey`, as snarkjs computes it
    -> dict(k, record, hash, s10 (the new section 10), g2_sp, delta1, delta2)."""
    hdr, _ = formats.read_zkey_header(zkey)
    s10 = sections(zkey)[10]
    cs_hash, recs = parse_mpc(s10)
    rng = rng_beacon(beacon_hash, exp) if beacon_hash is not None else rng_contribute(seed)
    k = from_rng(rng, R_MOD)
    g1_s = g1_from_rng(rng)
    g1_sx = G1.mul(g1_s, k)
    transcript = hashlib.blake2b(cs_hash + b"".join(hash_pub_key(r) for r in recs) + u_g1(g1_s) + u_g1(g1_sx),
                                 digest_size=64).digest()
    g2_sp = hash_to_g2(transcript)
    g2_spx = G2.mul(g2_sp, k)
    d1, d2 = G1.mul(hdr["vk_delta_1"], k), G2.mul(hdr["vk_delta_2"], k)
    params = b""
    if name:
        nb = name.encode()
        params += bytes([1, len(nb)]) + nb
    if beacon_hash is not None:
        params += bytes([2, exp, 3, len(beacon_hash)]) + bytes(beacon_hash)
    rec = (g1_to_bytes_mont(d1) + g1_to_bytes_mont(g1_s) + g1_to_bytes_mont(g1_sx) + g2_to_bytes_mont(g2_spx)
           + transcript + struct.pack("<II", 0 if beacon_hash is None else 1, len(params)) + params)
    new_s10 = cs_hash + struct.pack("<I", len(recs) + 1) + b"".join(recs) + rec
    return {"k": k, "record": rec, "hash": hashlib.blake2b(hash_pub_key(rec), digest_size=64).digest(), "s10": new_s10,
            "g1_s": g1_s, "g2_sp": g2_sp, "delta1": d1, "delta2": d2}


def with_section10(zkey, s10):
    """The key with section 10 replaced; sections in 1..10 order."""
    secs = sections(zkey)
    secs[10] = s10
    return formats.write_container(b"zkey", 1, sorted(secs.items()))
