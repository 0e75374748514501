"""Expected outputs of `powersoftau new` / `contribute` / `beacon`: a second, pure-Python restatement of snarkjs 0.4.12
powersoftau_new.js, powersoftau_contribute.js, powersoftau_beacon.js and keypair.js createPTauKey
(csrc/ptau_contribute.cu restates the same steps in C++).

Shared with the library: nothing but the published algorithm.  ChaCha, F/G.fromRng, hashToG2 and the uncompressed
encoding U are tests/contribution_cases.py's.  The BLAKE2b below is RFC 7693 written out, so that its state (blake2b-wasm's
216-byte context, snarkjs's partialHash) can be read; the tests tie its digest to hashlib.  C is wasmcurves LEMtoC.

contribution() returns the whole expected file in closed form: contributing (t, a, b) to write_ptau(tau, alpha, beta, p)
gives sections 2-6 of write_ptau(tau t, alpha a, beta b, p), which does not depend on any per-point multiplication
agreeing.  `new` is write_ptau(1, 1, 1, p).
"""
import hashlib
import struct

import contribution_cases as cc
from oracle import formats, ptau
from oracle.bn254 import (G1, G1_GEN, G2, G2_GEN, Q_MOD, R_MOD, g1_from_bytes_mont, g1_to_bytes_mont, g2_from_bytes_mont,
                          g2_to_bytes_mont, to_le32)

M64 = (1 << 64) - 1
IV = [0x6a09e667f3bcc908, 0xbb67ae8584caa73b, 0x3c6ef372fe94f82b, 0xa54ff53a5f1d36f1,
      0x510e527fade682d1, 0x9b05688c2b3e6c1f, 0x1f83d9abfb41bd6b, 0x5be0cd19137e2179]
SIGMA = [[0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15], [14, 10, 4, 8, 9, 15, 13, 6, 1, 12, 0, 2, 11, 7, 5, 3],
         [11, 8, 12, 0, 5, 2, 15, 13, 10, 14, 3, 6, 7, 1, 9, 4], [7, 9, 3, 1, 13, 12, 11, 14, 2, 6, 5, 10, 4, 0, 15, 8],
         [9, 0, 5, 7, 2, 4, 10, 15, 14, 1, 11, 12, 6, 8, 3, 13], [2, 12, 6, 10, 0, 11, 8, 3, 4, 13, 7, 5, 15, 14, 1, 9],
         [12, 5, 1, 15, 14, 13, 4, 10, 0, 7, 6, 3, 9, 2, 8, 11], [13, 11, 7, 14, 12, 1, 3, 9, 5, 0, 15, 4, 8, 6, 2, 10],
         [6, 15, 14, 9, 11, 3, 0, 8, 12, 2, 13, 7, 1, 4, 10, 5], [10, 2, 8, 4, 7, 6, 1, 5, 15, 11, 9, 14, 3, 12, 13, 0]]


def _rotr(x, c):
    return ((x >> c) | (x << (64 - c))) & M64


class Blake2b:
    """RFC 7693 BLAKE2b-512, unkeyed, with blake2b_ctx's lazy last block: a full buffer is compressed only when more
    input follows."""

    def __init__(self):
        self.h = list(IV)
        self.h[0] ^= 0x01010000 ^ 64
        self.t, self.b, self.c = 0, bytearray(128), 0

    def _compress(self, last):
        m = struct.unpack("<16Q", bytes(self.b))
        v = self.h + IV
        v[12] ^= self.t & M64
        v[13] ^= self.t >> 64
        if last:
            v[14] ^= M64

        def g(a, b, c, d, x, y):
            v[a] = (v[a] + v[b] + x) & M64; v[d] = _rotr(v[d] ^ v[a], 32)
            v[c] = (v[c] + v[d]) & M64; v[b] = _rotr(v[b] ^ v[c], 24)
            v[a] = (v[a] + v[b] + y) & M64; v[d] = _rotr(v[d] ^ v[a], 16)
            v[c] = (v[c] + v[d]) & M64; v[b] = _rotr(v[b] ^ v[c], 63)

        for r in range(12):
            s = SIGMA[r % 10]
            g(0, 4, 8, 12, m[s[0]], m[s[1]]); g(1, 5, 9, 13, m[s[2]], m[s[3]])
            g(2, 6, 10, 14, m[s[4]], m[s[5]]); g(3, 7, 11, 15, m[s[6]], m[s[7]])
            g(0, 5, 10, 15, m[s[8]], m[s[9]]); g(1, 6, 11, 12, m[s[10]], m[s[11]])
            g(2, 7, 8, 13, m[s[12]], m[s[13]]); g(3, 4, 9, 14, m[s[14]], m[s[15]])
        self.h = [self.h[i] ^ v[i] ^ v[i + 8] for i in range(8)]

    def update(self, data):
        data = memoryview(bytes(data))
        pos = 0
        while pos < len(data):
            if self.c == 128:
                self.t += 128
                self._compress(False)
                self.c = 0
            k = min(128 - self.c, len(data) - pos)
            self.b[self.c:self.c + k] = data[pos:pos + k]
            self.c += k
            pos += k
        return self

    def digest(self):
        t, b = self.t, bytearray(self.b)
        self.t += self.c
        self.b[self.c:] = bytes(128 - self.c)
        self._compress(True)
        out = struct.pack("<8Q", *self.h)
        self.t, self.b = t, b
        return out

    def partial(self):
        """blake2b-wasm getPartialHash: b[128], h[8], t[2] (u64 LE), c, outlen (u32 LE)."""
        return (bytes(self.b) + struct.pack("<8Q", *self.h) + struct.pack("<QQ", self.t & M64, self.t >> 64)
                + struct.pack("<II", self.c, 64))

    @classmethod
    def from_partial(cls, p):
        assert len(p) == 216 and struct.unpack_from("<I", p, 212)[0] == 64
        s = cls()
        s.b = bytearray(p[:128])
        s.h = list(struct.unpack_from("<8Q", p, 128))
        lo, hi = struct.unpack_from("<QQ", p, 192)
        s.t = lo | hi << 64
        s.c = struct.unpack_from("<I", p, 208)[0]
        return s


# ------------------------------------------------------------------------------------------------ encodings
u_g1, u_g2 = cc.u_g1, cc.u_g2
HALF_Q = (Q_MOD - 1) // 2


def c_g1(P):
    """wasmcurves LEMtoC: big-endian x, 0x80 in byte 0 when y > (q-1)/2; infinity 0x40 then zeros."""
    if P is None:
        return b"\x40" + bytes(31)
    b = bytearray(P[0].to_bytes(32, "big"))
    if P[1] > HALF_Q:
        b[0] |= 0x80
    return bytes(b)


def c_g2(P):
    """x.c1 || x.c0; the sign of y: c1 decides, c0 when c1 = 0."""
    if P is None:
        return b"\x40" + bytes(63)
    b = bytearray(P[0][1].to_bytes(32, "big") + P[0][0].to_bytes(32, "big"))
    if cc.f2_is_negative(P[1]):
        b[0] |= 0x80
    return bytes(b)


def first_challenge_hash(power):
    n = 1 << power
    g1, g2 = u_g1(G1_GEN), u_g2(G2_GEN)
    h = hashlib.blake2b(digest_size=64)
    h.update(hashlib.blake2b(digest_size=64).digest())
    h.update(g1 * (2 * n - 1))
    h.update(g2 * n)
    h.update(g1 * n)
    h.update(g1 * n)
    h.update(g2)
    return h.digest()


# ------------------------------------------------------------------------------------------------ the key
def create_key(rng, challenge):
    """keypair.js createPTauKey -> [tau, alpha, beta], each dict(prv, g1_s, g1_sx, g2_sp, g2_spx)."""
    key = [{"prv": cc.from_rng(rng, R_MOD)} for _ in range(3)]
    for pers, k in enumerate(key):
        k["g1_s"] = cc.g1_from_rng(rng)
        k["g1_sx"] = G1.mul(k["g1_s"], k["prv"])
        d = hashlib.blake2b(bytes([pers]) + challenge + u_g1(k["g1_s"]) + u_g1(k["g1_sx"]), digest_size=64).digest()
        k["g2_sp"] = cc.hash_to_g2(d)
        k["g2_spx"] = G2.mul(k["g2_sp"], k["prv"])
    return key


def pub_key(key, montgomery):
    """toPtauPubKeyRpr: tau.g1_s tau.g1_sx alpha.g1_s ... beta.g1_sx, then the three g2_spx."""
    e1, e2 = (g1_to_bytes_mont, g2_to_bytes_mont) if montgomery else (u_g1, u_g2)
    return b"".join(e1(k["g1_s"]) + e1(k["g1_sx"]) for k in key) + b"".join(e2(k["g2_spx"]) for k in key)


# ------------------------------------------------------------------------------------------------ files
PUBKEY_LEN = 768
REC_FIXED = PUBKEY_LEN + 3 * 64 + 2 * 128 + 216 + 64 + 8       # 1504
PARTIAL_OFF, NEXT_OFF = 1216, 1432
G2_SECTIONS = (3, 6)


def sections(buf):
    _, secs = formats.read_container(buf, b"ptau")
    return {sid: bytes(memoryview(buf)[v[0][0]:v[0][0] + v[0][1]]) for sid, v in secs.items()}


def power_of(buf):
    return struct.unpack_from("<I", sections(buf)[1], 36)[0]


def parse_records(s7):
    n = struct.unpack_from("<I", s7, 0)[0]
    pos, recs = 4, []
    for _ in range(n):
        plen = struct.unpack_from("<I", s7, pos + REC_FIXED - 4)[0]
        recs.append(bytes(s7[pos:pos + REC_FIXED + plen]))
        pos += REC_FIXED + plen
    assert pos == len(s7)
    return recs


def record_fields(rec):
    g1 = lambda o: g1_from_bytes_mont(rec[o:o + 64])
    g2 = lambda o: g2_from_bytes_mont(rec[o:o + 128])
    key = [{"g1_s": g1(128 * j), "g1_sx": g1(128 * j + 64), "g2_spx": g2(384 + 128 * j)} for j in range(3)]
    return {"key": key, "tauG1": g1(768), "tauG2": g2(832), "alphaG1": g1(960), "betaG1": g1(1024), "betaG2": g2(1088),
            "partial": rec[PARTIAL_OFF:PARTIAL_OFF + 216], "next": rec[NEXT_OFF:NEXT_OFF + 64],
            "type": struct.unpack_from("<I", rec, 1496)[0], "params": rec[REC_FIXED:]}


def points(sec, g2):
    sz, dec = (128, g2_from_bytes_mont) if g2 else (64, g1_from_bytes_mont)
    return [dec(sec[i:i + sz]) for i in range(0, len(sec), sz)]


def encodings(secs, compressed):
    """C or U of every point of sections 2-6, in order."""
    out = []
    for sid in range(2, 7):
        g2 = sid in G2_SECTIONS
        enc = (c_g2 if g2 else c_g1) if compressed else (u_g2 if g2 else u_g1)
        out.append(b"".join(enc(P) for P in points(secs[sid], g2)))
    return b"".join(out)


def header(power):
    return struct.pack("<I", 32) + to_le32(Q_MOD) + struct.pack("<II", power, power)


def new_file(power):
    return ptau.write_ptau(1, 1, 1, power, prepared=False)


def contribution(ptau_buf, tau, alpha, beta, name=None, seed=None, beacon_hash=None, exp=None, infinity=(),
                 partial=True):
    """One contribution (seed: 32 bytes) or beacon (beacon_hash, exp) to `ptau_buf`, whose sections 2-6 are those of
    write_ptau(tau, alpha, beta) with the points `infinity` ((sid, index) pairs) at infinity, as snarkjs computes it
    -> dict(file, response, partial, next, key, record, tau, alpha, beta (the new totals)).  partial=False hashes the
    response with hashlib and leaves partialHash zero (large powers)."""
    secs = sections(ptau_buf)
    power = struct.unpack_from("<I", secs[1], 36)[0]
    recs = parse_records(secs[7])
    challenge = recs[-1][NEXT_OFF:NEXT_OFF + 64] if recs else first_challenge_hash(power)
    rng = cc.rng_beacon(beacon_hash, exp) if beacon_hash is not None else cc.rng_contribute(seed)
    key = create_key(rng, challenge)
    t, a, b = (k["prv"] for k in key)
    tau, alpha, beta = tau * t % R_MOD, alpha * a % R_MOD, beta * b % R_MOD
    new = sections(ptau.write_ptau(tau, alpha, beta, power, prepared=False))
    for sid, i in infinity:
        sz = 128 if sid in G2_SECTIONS else 64
        new[sid] = new[sid][:sz * i] + bytes(sz) + new[sid][sz * (i + 1):]
    if partial:
        h = Blake2b().update(challenge).update(encodings(new, True))
        part = h.partial()
        response = h.update(pub_key(key, False)).digest()
    else:
        part = bytes(216)
        response = hashlib.blake2b(challenge + encodings(new, True) + pub_key(key, False), digest_size=64).digest()
    nxt = hashlib.blake2b(response + encodings(new, False), digest_size=64).digest()
    params = b""
    if name:
        nb = name.encode()
        params += bytes([1, len(nb)]) + nb
    if beacon_hash is not None:
        params += bytes([2, exp, 3, len(beacon_hash)]) + bytes(beacon_hash)
    rec = (pub_key(key, True) + new[2][64:128] + new[3][128:256] + new[4][:64] + new[5][:64] + new[6]
           + part + nxt + struct.pack("<II", 0 if beacon_hash is None else 1, len(params)) + params)
    s7 = struct.pack("<I", len(recs) + 1) + b"".join(recs) + rec
    out = [(1, header(power))] + [(sid, new[sid]) for sid in range(2, 7)] + [(7, s7)]
    return {"file": formats.write_container(b"ptau", 1, out), "response": response, "partial": part, "next": nxt,
            "key": key, "record": rec, "tau": tau, "alpha": alpha, "beta": beta, "challenge": challenge}
