"""Expected results of `zkey verify` and of the circuit hash: a pure-Python restatement of snarkjs 0.4.12 zkey_new.js
(csHasher) and zkey_verify_frominit.js (csrc/verify.cu restates the same steps in C++).

Shared with the library: nothing but the published algorithm.  BLAKE2b-512 is hashlib's, point arithmetic is
oracle/bn254's, the encodings and section-10 records are contribution_cases.py's.

The H check.  With H[j] = L^(2N)_(2j+1)(tau) (times 1 / delta) and r'_j = sum_m a_m w_N^(jm) (Fr.fft), a_m = -2 w_2N^m r_m:
    sum_j r'_j L^(2N)_(2j+1)(x) = (1/2N) sum_m a_m sum_t x^t w_2N^-t sum_j w_N^(j(m-t))
                               = (1/2) sum_m a_m w_2N^-m (x^m - x^(m+N))        (t = m or m + N; w_2N^-N = -1)
                               = sum_m r_m (x^(m+N) - x^m).
It is linear, so it holds point by point for any tauG1 whose Lagrange level is its inverse FFT.  snarkjs's top tauG1
level (cirPower = power) lacks tau^(2N-1) and has the point at infinity in its place: that changes only the x^(2N-1)
term, which belongs to m = N - 1, and r_(N-1) = 0 removes it.  h_identity_holds() checks both claims at a known tau.
"""
import hashlib
import struct

import contribution_cases as cc
import ptau_cases
from oracle import formats
from oracle.bn254 import FR_W, G1, G1_GEN, G2_GEN, R_MOD, g1_from_bytes_mont, g2_from_bytes_mont
from oracle.setup import lagrange_at

H_CHUNK = 1 << 14        # hashHPoints CHUNK_SIZE


def h_hash_points(n):
    """Points hashHPoints passes to the hasher: its chunk loop takes min(N - 1, CHUNK) points for every
    i < N - 1 in steps of CHUNK, so N - 1 points up to N = 2^14 and N points above."""
    return sum(min(n - 1, H_CHUNK) for _ in range(0, n - 1, H_CHUNK))


def _points(buf, size, n):
    dec = g1_from_bytes_mont if size == 64 else g2_from_bytes_mont
    return [dec(buf[size * i:size * i + size]) for i in range(n)]


def circuit_hash(init_zkey, ptau):
    """csHash of zkey_new.js from an initial key and its ptau (section 2 tauG1)."""
    secs = cc.sections(bytes(init_zkey))
    h = secs[2]
    n_vars, n_public, n = struct.unpack_from("<III", h, 72)
    _, psecs = formats.read_container(bytes(ptau), b"ptau")
    off, _ = psecs[2][0]
    n_hash = h_hash_points(n)
    tau = _points(bytes(ptau)[off:off + 64 * (n + n_hash)], 64, n + n_hash)
    out = hashlib.blake2b(digest_size=64)
    out.update(cc.u_g1(g1_from_bytes_mont(h[84:148])) + cc.u_g1(g1_from_bytes_mont(h[148:212])))
    out.update(cc.u_g2(g2_from_bytes_mont(h[212:340])))
    out.update(cc.u_g2(G2_GEN) + cc.u_g1(G1_GEN) + cc.u_g2(G2_GEN))

    def arr(count, pts, u):
        out.update(struct.pack(">I", count))
        for P in pts:
            out.update(u(P))

    arr(n_public + 1, _points(secs[3], 64, n_public + 1), cc.u_g1)
    arr(n - 1, [G1.add(tau[i + n], G1.neg(tau[i])) for i in range(n_hash)], cc.u_g1)
    arr(n_vars - n_public - 1, _points(secs[8], 64, n_vars - n_public - 1), cc.u_g1)
    arr(n_vars, _points(secs[5], 64, n_vars), cc.u_g1)
    arr(n_vars, _points(secs[6], 64, n_vars), cc.u_g1)
    arr(n_vars, _points(secs[7], 128, n_vars), cc.u_g2)
    return out.digest()


def with_cs_hash(zkey, cs_hash):
    """The key with the csHash of section 10 replaced."""
    s10 = cc.sections(bytes(zkey))[10]
    return cc.with_section10(bytes(zkey), bytes(cs_hash) + s10[64:])


def h_scalars(r, log_n):
    """r' = Fr.fft(-2 w_2N^m r_m), w_2N = Fr.w[log_n + 1]; naive transform."""
    n = 1 << log_n
    w2, w = FR_W[log_n + 1], FR_W[log_n]
    a = [-2 * pow(w2, m, R_MOD) * r[m] % R_MOD for m in range(n)]
    return [sum(a[m] * pow(w, j * m, R_MOD) for m in range(n)) % R_MOD for j in range(n)]


def h_identity_holds(tau, log_n, r, top_snarkjs=False):
    """sum_j r'_j L^(2N)_(2j+1)(tau) == sum_m r_m (tau^(m+N) - tau^m), scalars at a known tau; top_snarkjs: the size-2N
    level is snarkjs's top tauG1 level (ptau_cases.lagrange_top_snarkjs)."""
    n = 1 << log_n
    lv = ptau_cases.lagrange_top_snarkjs(tau, log_n + 1) if top_snarkjs else lagrange_at(tau, log_n + 1)
    rp = h_scalars(r, log_n)
    lhs = sum(rp[j] * lv[2 * j + 1] for j in range(n)) % R_MOD
    rhs = sum(r[m] * (pow(tau, m + n, R_MOD) - pow(tau, m, R_MOD)) for m in range(n)) % R_MOD
    return lhs == rhs


def record_claims(zkey):
    """The claims verifyFromInit derives from section 10 and the header, before the L / H checks, as (step, record,
    a, b, c, d) with e(a, d) = e(b, c) claimed: per record steps 3 and 4, then step 8 (delta2)."""
    secs = cc.sections(bytes(zkey))
    _, recs = cc.parse_mpc(secs[10])
    hdr, _ = formats.read_zkey_header(bytes(zkey))
    out, cur = [], G1_GEN
    for i, rec in enumerate(recs):
        c = cc.record_points(rec)
        g2_sp = cc.hash_to_g2(c["transcript"])
        out.append((3, i, c["g1_s"], c["g1_sx"], g2_sp, c["g2_spx"]))
        out.append((4, i, cur, c["deltaAfter"], g2_sp, c["g2_spx"]))
        cur = c["deltaAfter"]
    out.append((8, -1, G1_GEN, cur, G2_GEN, hdr["vk_delta_2"]))
    return out
