"""Expected outputs of `powersoftau prepare phase2`, restated from known toxic waste for the ptau tests.

oracle/ptau.py write_ptau writes a phase-1 file (prepared=False) and, with prepared=True, the exact Lagrange basis on
every level.  snarkjs 0.4.12 powersoftau_preparephase2.js does not produce the exact basis on the top tauG1 level
(p = power+1): section 2 holds only 2^(power+1) - 1 powers, and snarkjs puts the point at infinity in the last slot, so
that level is the ifft of an incomplete vector,
    L'_i(tau) = L_i(tau) - w^i tau^(N-1) / N,   N = 2^(power+1), w = Fr.w[power+1].
write_prepared writes the file snarkjs would write: the phase-1 sections of write_ptau, then sections 12-15 with L' on the
top tauG1 level.  It also takes a tau inside a domain (degenerate ceremonies), where L_i(w^k) = [i == k].

ifft_points is the group ifft by its definition, with no tau: the CPU tests tie it to the closed forms.
"""
from oracle import formats, ptau
from oracle.bn254 import FR_W, G1, G1_GEN, G2, G2_GEN, R_MOD, FixedBase, g1_to_bytes_mont, g2_to_bytes_mont
from oracle.setup import lagrange_at


def lagrange_any(tau, log_n):
    """lagrange_at, also for a tau inside the domain: there L_i(w^k) = [i == k]."""
    n = 1 << log_n
    if pow(tau, n, R_MOD) != 1:
        return lagrange_at(tau, log_n)
    w = FR_W[log_n]
    return [1 if pow(w, i, R_MOD) == tau % R_MOD else 0 for i in range(n)]


def lagrange_top_snarkjs(tau, log_n):
    """L'_i(tau) = L_i(tau) - w^i tau^(N-1) / N: the level snarkjs derives from N - 1 powers and one infinity."""
    n = 1 << log_n
    w = FR_W[log_n]
    corr = pow(tau, n - 1, R_MOD) * pow(n, -1, R_MOD) % R_MOD
    return [(x - pow(w, i, R_MOD) * corr) % R_MOD for i, x in enumerate(lagrange_any(tau, log_n))]


def ifft_points(curve, pts):
    """out_i = (1/N) sum_j w^(-ij) P_j, w = Fr.w[log2 N]; None = infinity."""
    n = len(pts)
    log_n = n.bit_length() - 1
    assert 1 << log_n == n
    winv, ninv = pow(FR_W[log_n], -1, R_MOD), pow(n, -1, R_MOD)
    out = []
    for i in range(n):
        acc = None
        for j, P in enumerate(pts):
            if P is not None:
                acc = curve.add(acc, curve.mul(P, pow(winv, i * j, R_MOD) * ninv % R_MOD))
        out.append(acc)
    return out


def write_prepared(tau, alpha, beta, power):
    """The prepared file snarkjs writes from write_ptau(tau, alpha, beta, power, prepared=False)."""
    raw = ptau.write_ptau(tau, alpha, beta, power, prepared=False)
    _, secs = formats.read_container(raw, b"ptau")
    mv = memoryview(raw)
    out = [(sid, bytes(mv[secs[sid][0][0]:secs[sid][0][0] + secs[sid][0][1]])) for sid in range(1, 8)]
    fb1, fb2 = FixedBase(G1, G1_GEN), FixedBase(G2, G2_GEN)
    lv = [lagrange_any(tau, p) for p in range(power + 1)] + [lagrange_top_snarkjs(tau, power + 1)]
    out.append((12, b"".join(g1_to_bytes_mont(fb1.mul(x)) for p in range(power + 2) for x in lv[p])))
    out.append((13, b"".join(g2_to_bytes_mont(fb2.mul(x)) for p in range(power + 1) for x in lv[p])))
    out.append((14, b"".join(g1_to_bytes_mont(fb1.mul(alpha * x % R_MOD)) for p in range(power + 1) for x in lv[p])))
    out.append((15, b"".join(g1_to_bytes_mont(fb1.mul(beta * x % R_MOD)) for p in range(power + 1) for x in lv[p])))
    return formats.write_container(b"ptau", 1, out)
