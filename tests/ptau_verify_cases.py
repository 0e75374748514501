"""Expected outcome of `powersoftau verify`: a pure-Python restatement of snarkjs 0.4.12 powersoftau_verify.js with the
library's random combinations (csrc/ptau_verify.cu restates the same steps in C++), for small powers.

expected(file, seed) returns the report and the claims nzcp_ptau_verify gives for a file whose points are canonical and
on their curves (step 1 is left to the tests): the claims in the C layout, byte for byte, and the first check the library
fails itself.  The scalars are F.fromRng buffers drawn from ChaCha(seed): the N - 1 of sections 2, 3, 4, 5, then the levels of
12, 13, 14, 15 (the top tauG1 level's last scalar is 0, not drawn).  The Lagrange sums use the definition of Fr.fft.
"""
import hashlib
import struct

import contribution_cases as cc
import ptau_contribution_cases as pc
from oracle.bn254 import FR_W, G1, G1_GEN, G2, G2_GEN, R_MOD, to_le32

NO_RECORDS = "This file has no contribution! It cannot be used in production"
LAGRANGE = "Phase2 caclutation does not match with powers of tau"
NEXT = "Hash of the values does not match the next challenge of the last contributor in the contributions section"
POWERS = {2: "tauG1", 3: "tauG2", 4: "alphaTauG1", 5: "betaTauG1"}
BEACON_PARTS = ["tauG1_s", "tauG1_sx", "alphaG1_s", "alphaG1_sx", "betaG1_s", "betaG1_sx", "tauG2_spx", "alphaG2_spx",
                "betaG2_spx"]


class Verdict(Exception):
    def __init__(self, step, record, message):
        super().__init__(message)
        self.step, self.record, self.message = step, record, message


def draw(rng):
    """A scalar: the F.fromRng buffer itself, as the library uses it (plain, < r)."""
    return cc.from_rng(rng, R_MOD) * cc.MONT_R % R_MOD


def claim_bytes(step, record, a, b, c, d):
    """nzcp_zkey_verify_claim: i32 step, i32 record, G1 a, b (plain x, y), G2 c, d (x.c0 x.c1 y.c0 y.c1); infinity = 0."""
    g1 = lambda P: bytes(64) if P is None else to_le32(P[0]) + to_le32(P[1])
    g2 = lambda P: bytes(128) if P is None else to_le32(P[0][0]) + to_le32(P[0][1]) + to_le32(P[1][0]) + to_le32(P[1][1])
    return struct.pack("<ii", step, record) + g1(a) + g1(b) + g2(c) + g2(d)


def params(rec):
    """name, numIterationsExp, beaconHash of a record's parameters."""
    p, out, pos = rec[pc.REC_FIXED:], {"name": b"", "exp": 0, "beacon": None}, 0
    while pos < len(p):
        tag = p[pos]
        if tag == 2:
            out["exp"] = p[pos + 1]
            pos += 2
        else:
            ln = p[pos + 1]
            out["name" if tag == 1 else "beacon"] = p[pos + 2:pos + 2 + ln]
            pos += 2 + ln
    return out


def response_hash(rec):
    f = pc.record_fields(rec)
    return pc.Blake2b.from_partial(f["partial"]).update(pc.pub_key(f["key"], False)).digest()


def msm(curve, pts, scalars):
    acc = None
    for P, s in zip(pts, scalars):
        if P is not None and s:
            acc = curve.add(acc, curve.mul(P, s))
    return acc


def fft(r):
    """Fr.fft: X_i = sum_j r_j w^(ij), w = Fr.w[log2 N]."""
    n = len(r)
    w = FR_W[n.bit_length() - 1]
    return [sum(r[j] * pow(w, i * j, R_MOD) for j in range(n)) % R_MOD for i in range(n)]


def expected(buf, seed):
    """-> dict(failed_step, failed_record, message, claims [bytes], prepared, next_challenge (64 bytes, zero if not
    reached), records [dict(response_hash, next_challenge, type, name, exp, beacon)])."""
    secs = pc.sections(buf)
    power, cpow = struct.unpack_from("<II", secs[1], 36)
    prepared = all(s in secs for s in (12, 13, 14, 15))
    recs = pc.parse_records(secs[7])
    fields = [pc.record_fields(r) for r in recs]
    out = {"failed_step": 0, "failed_record": -1, "message": "", "claims": [], "prepared": prepared,
           "next_challenge": bytes(64),
           "records": [dict(response_hash=response_hash(r), next_challenge=f["next"], type=f["type"], **params(r))
                       for r, f in zip(recs, fields)]}
    claims = out["claims"]
    first = pc.first_challenge_hash(cpow) if recs else None

    def prev(i):
        if i:
            return fields[i - 1]
        return {"tauG1": G1_GEN, "alphaG1": G1_GEN, "betaG1": G1_GEN, "tauG2": G2_GEN, "betaG2": G2_GEN, "next": first}

    def contribution(i):
        cur, pv, rec = fields[i], prev(i), recs[i]
        if cur["type"] == 1:
            p = params(rec)
            bk = pc.create_key(cc.rng_beacon(p["beacon"], p["exp"]), pv["next"])
            want = pc.pub_key(bk, True)
            for q in range(9):
                off, ln = (64 * q, 64) if q < 6 else (384 + 128 * (q - 6), 128)
                if want[off:off + ln] != rec[off:off + ln]:
                    raise Verdict(3, i, "BEACON key (%s) is not generated correctly in challenge #%d  %s"
                                  % (BEACON_PARTS[q], i + 1, p["name"].decode()))
        key = cur["key"]
        sp = [cc.hash_to_g2(hashlib.blake2b(bytes([j]) + pv["next"] + pc.u_g1(k["g1_s"]) + pc.u_g1(k["g1_sx"]),
                                            digest_size=64).digest()) for j, k in enumerate(key)]
        for j in range(3):
            claims.append(claim_bytes(4 + j, i, key[j]["g1_s"], key[j]["g1_sx"], sp[j], key[j]["g2_spx"]))
        claims.append(claim_bytes(7, i, pv["tauG1"], cur["tauG1"], sp[0], key[0]["g2_spx"]))
        claims.append(claim_bytes(8, i, key[0]["g1_s"], key[0]["g1_sx"], pv["tauG2"], cur["tauG2"]))
        claims.append(claim_bytes(9, i, pv["alphaG1"], cur["alphaG1"], sp[1], key[1]["g2_spx"]))
        claims.append(claim_bytes(10, i, pv["betaG1"], cur["betaG1"], sp[2], key[2]["g2_spx"]))
        claims.append(claim_bytes(11, i, key[2]["g1_s"], key[2]["g1_sx"], pv["betaG2"], cur["betaG2"]))

    try:
        if not recs:
            raise Verdict(2, -1, NO_RECORDS)
        n = len(recs)
        contribution(n - 1)
        last = fields[-1]
        rng = cc.rng_contribute(seed)
        rs = {sid: [draw(rng) for _ in range(len(pc.points(secs[sid], sid == 3)) - 1)] for sid in (2, 3, 4, 5)}
        lag_ok = True
        for sid in (2, 3, 4, 5, 6):
            g2 = sid in pc.G2_SECTIONS
            pts = pc.points(secs[sid], g2)
            if sid == 6:
                if pts[0] != last["betaG2"]:
                    raise Verdict(16, -1, "betaG2 element in betaG2 section does not match the one in the contribution section")
                break
            curve = G2 if g2 else G1
            r1, r2 = msm(curve, pts[:-1], rs[sid]), msm(curve, pts[1:], rs[sid])
            if sid == 3:
                claims.append(claim_bytes(13, -1, G1_GEN, last["tauG1"], r1, r2))
            else:
                claims.append(claim_bytes(10 + sid, -1, r1, r2, G2_GEN, last["tauG2"]))
            name = {2: "tau*G1", 3: "tau*G2"}.get(sid)
            if name:
                if pts[0] != (G2_GEN if g2 else G1_GEN):
                    raise Verdict(16, -1, "First element of %s section must be the generator" % name)
                if pts[1] != last["tauG2" if g2 else "tauG1"]:
                    raise Verdict(16, -1, "Second element of %s section does not match the one in the contribution section"
                                  % name)
            else:
                ab = "alpha" if sid == 4 else "beta"
                if pts[0] != last[ab + "G1"]:
                    raise Verdict(16, -1, "First element of %s*tau*G1 section (%s*G1) does not match the one in the "
                                  "contribution section" % (ab, ab))
            if prepared:
                lag_ok &= lagrange_ok(rng, pts, pc.points(secs[sid + 10], g2), curve, power + 1 if sid == 2 else power)
        nxt = hashlib.blake2b(response_hash(recs[-1]) + pc.encodings(secs, False), digest_size=64).digest()
        out["next_challenge"] = nxt
        if power == cpow and nxt != last["next"]:
            raise Verdict(17, -1, NEXT)
        for i in range(n - 2, -1, -1):
            contribution(i)
        if not lag_ok:
            raise Verdict(18, -1, LAGRANGE)
    except Verdict as v:
        out.update(failed_step=v.step, failed_record=v.record, message=v.message)
    return out


def lagrange_ok(rng, tau, lag, curve, top):
    lhs, rhs, off = None, None, 0
    for p in range(top + 1):
        n = 1 << p
        r = [draw(rng) if j < len(tau) else 0 for j in range(n)]
        lhs = curve.add(lhs, msm(curve, tau[:n], r))
        rhs = curve.add(rhs, msm(curve, lag[off:off + n], fft(r)))
        off += n
    return lhs == rhs
