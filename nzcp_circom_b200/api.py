"""Object wrappers over the C ABI (include/nzcp_prover.h): Zkey, Prover, and the standalone NTT / MSM calls.

This is the layer a Node N-API addon would sit at (INTEGRATION.md); groth16.py puts the snarkjs-shaped surface on
top of it.  Everything computes on the GPU through libnzcp_prover.so; nothing here falls back to the CPU.
"""
import ctypes as C

from . import _lib
from ._lib import NzcpError, Proof, ProveDebug, ZkeyCheck, ZkeyInfo, addr, check

STAGE_NAMES = ("upload", "r1cs_eval", "ntt_join", "msm_a", "msm_b1", "msm_b2", "msm_c", "msm_h")


def _as_bytes_like(x):
    """Path | bytes-like | {"type": "mem", "data": ...} (fastfile convention) -> bytes-like."""
    if isinstance(x, dict) and x.get("type") == "mem":
        return x["data"]
    if isinstance(x, str) or hasattr(x, "__fspath__"):
        with open(x, "rb") as f:
            return f.read()
    return x


def _nbytes(buf):
    if hasattr(buf, "nbytes"):
        return int(buf.nbytes)
    return len(buf)


def _scalar32(v):
    """int | 32 bytes | None -> 32-byte LE or None."""
    if v is None:
        return None
    if isinstance(v, int):
        return int(v).to_bytes(32, "little")
    b = bytes(v)
    if len(b) != 32:
        raise NzcpError(_lib.NZCP_E_ARG, "blinding scalar must be 32 bytes")
    return b


def device_count():
    return _lib.load().nzcp_device_count()


class Zkey:
    """A proving key resident on one GPU (sections 4-9 parsed and uploaded once)."""

    def __init__(self, zkey, device=0):
        lib = _lib.load()
        data = _as_bytes_like(zkey)
        h = C.c_void_p()
        check(lib.nzcp_zkey_load(addr(data), _nbytes(data), int(device), C.byref(h)))
        self._h = h
        self.device = int(device)
        inf = ZkeyInfo()
        check(lib.nzcp_zkey_info_get(self._h, C.byref(inf)))
        self.n_vars, self.n_public, self.domain_size = inf.n_vars, inf.n_public, inf.domain_size
        self.power, self.n_coefs, self.device_bytes = inf.power, inf.n_coefs, inf.device_bytes
        self._info = inf

    def prove_batch(self, wtns_list, r_list=None, s_list=None, n_provers=0):
        """nzcp_prove_batch: all proofs of the list through the library's own thread pool -> list of 256-byte proofs."""
        n = len(wtns_list)
        datas = [_as_bytes_like(w) for w in wtns_list]
        ptrs = (C.c_void_p * n)(*[addr(d) for d in datas])
        lens = (C.c_size_t * n)(*[_nbytes(d) for d in datas])
        rb = b"".join(_scalar32(x) for x in r_list) if r_list is not None else None
        sb = b"".join(_scalar32(x) for x in s_list) if s_list is not None else None
        proofs = (Proof * n)()
        status = (C.c_int * n)()
        check(_lib.load().nzcp_prove_batch(self._h, ptrs, lens, n, addr(rb), addr(sb), proofs, int(n_provers), status))
        return [bytes(p.pi_a) + bytes(p.pi_b) + bytes(p.pi_c) for p in proofs]

    def header_points(self):
        """alpha1, beta1, delta1 (64 B) and beta2, gamma2, delta2 (128 B): plain affine LE bytes."""
        i = self._info
        return {"alpha1": bytes(i.alpha1), "beta1": bytes(i.beta1), "delta1": bytes(i.delta1),
                "beta2": bytes(i.beta2), "gamma2": bytes(i.gamma2), "delta2": bytes(i.delta2)}

    def close(self):
        if getattr(self, "_h", None):
            _lib.load().nzcp_zkey_free(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Prover:
    """Work buffers + streams for proofs against one Zkey.  One in-flight proof per Prover."""

    def __init__(self, zkey, throughput=False):
        """throughput=False: latency mode (a lone proof at a time).  True: meant to run beside other provers on the same
        GPU (batched-affine pair rounds in the bucket accumulation: more proofs/s, slightly slower alone)."""
        self.zkey = zkey
        h = C.c_void_p()
        check(_lib.load().nzcp_prover_create_mode(zkey._h, 1 if throughput else 0, C.byref(h)))
        self._h = h

    def _finish(self, proof, dbg, want_h, hbuf):
        out = {"proof": bytes(proof.pi_a) + bytes(proof.pi_b) + bytes(proof.pi_c)}
        if dbg is not None:
            out.update(msm_a=bytes(dbg.msm_a), msm_b1=bytes(dbg.msm_b1), msm_b2=bytes(dbg.msm_b2),
                       msm_c=bytes(dbg.msm_c), msm_h=bytes(dbg.msm_h),
                       stage_ms=dict(zip(STAGE_NAMES, [float(x) for x in dbg.stage_ms])),
                       sort_ms={"witness": float(dbg.sort_ms[0]), "h": float(dbg.sort_ms[1])},
                       accumulate_ms=dict(zip(("a", "b1", "b2", "c", "h"), [float(x) for x in dbg.accumulate_ms])),
                       n_entries={"witness": int(dbg.n_entries[0]), "h": int(dbg.n_entries[1])},
                       total_ms=float(dbg.total_ms))
            if want_h:
                out["h"] = bytes(hbuf)
        return out

    def _dbg(self, debug, want_h):
        if not debug and not want_h:
            return None, None, None
        dbg = ProveDebug()
        hbuf = None
        if want_h:
            hbuf = bytearray(self.zkey.domain_size * 32)
            dbg.h_scalars = addr(hbuf)
        return dbg, hbuf, C.byref(dbg)

    def prove(self, wtns, r=None, s=None, debug=False, want_h=False):
        """`wtns`: a complete .wtns image (bytes-like or path).  -> dict(proof=256 bytes, [msm_*, stage_ms, h])."""
        data = _as_bytes_like(wtns)
        proof = Proof()
        dbg, hbuf, ref = self._dbg(debug, want_h)
        rb, sb = _scalar32(r), _scalar32(s)
        check(_lib.load().nzcp_prove(self._h, addr(data), _nbytes(data), addr(rb), addr(sb), C.byref(proof), ref))
        return self._finish(proof, dbg, want_h, hbuf)

    def prove_witness(self, witness, n_witness, r=None, s=None, debug=False, want_h=False):
        """`witness`: n_witness x 32-byte LE plain values in host memory (section 2 of a .wtns)."""
        proof = Proof()
        dbg, hbuf, ref = self._dbg(debug, want_h)
        rb, sb = _scalar32(r), _scalar32(s)
        check(_lib.load().nzcp_prove_witness(self._h, addr(witness), int(n_witness), addr(rb), addr(sb),
                                             C.byref(proof), ref))
        return self._finish(proof, dbg, want_h, hbuf)

    def prove_device(self, d_witness, r=None, s=None, debug=False):
        """`d_witness`: device pointer (int or torch tensor) to n_vars x 32 B already in HBM."""
        proof = Proof()
        dbg, hbuf, ref = self._dbg(debug, False)
        rb, sb = _scalar32(r), _scalar32(s)
        check(_lib.load().nzcp_prove_device(self._h, addr(d_witness), addr(rb), addr(sb), C.byref(proof), ref))
        return self._finish(proof, dbg, False, hbuf)

    def witness_buffer(self):
        return _lib.load().nzcp_prover_witness_buffer(self._h)

    def launch_count(self):
        return int(_lib.load().nzcp_prover_launch_count(self._h))

    def close(self):
        if getattr(self, "_h", None):
            _lib.load().nzcp_prover_free(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ProverPool:
    """Several Provers on one resident Zkey, driven from host threads so that the latency-bound tail of one proof (bucket
    reduction trees, host finalisation) overlaps the integer-pipe-bound kernels of the next.  ctypes drops the GIL inside
    the library calls.  Proof i is independent of proof j: this is the batch mode of SURVEY.md 8e on ONE GPU."""

    def __init__(self, zkey, n_provers=2, throughput=True):
        from concurrent.futures import ThreadPoolExecutor
        self.zkey = zkey
        self.provers = [Prover(zkey, throughput=throughput) for _ in range(max(1, int(n_provers)))]
        self._pool = ThreadPoolExecutor(max_workers=len(self.provers))

    def _run(self, method, items, r, s, kw):
        k = len(self.provers)

        def work(j):
            pr = self.provers[j]
            return [(i, getattr(pr, method)(*items[i], r=r, s=s, **kw)) for i in range(j, len(items), k)]
        out = [None] * len(items)
        for fut in [self._pool.submit(work, j) for j in range(k)]:
            for i, res in fut.result():
                out[i] = res
        return out

    def prove_many(self, wtns_list, r=None, s=None, **kw):
        """.wtns images (host memory) -> list of result dicts, in order."""
        return self._run("prove", [(w,) for w in wtns_list], r, s, kw)

    def prove_device_many(self, d_witness_list, r=None, s=None, **kw):
        return self._run("prove_device", [(d,) for d in d_witness_list], r, s, kw)

    def launch_count(self):
        """Kernel launches issued for ALL provers of the pool so far."""
        return sum(p.launch_count() for p in self.provers)

    def close(self):
        self._pool.shutdown(wait=True)
        for p in self.provers:
            p.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


# ------------------------------------------------------------------------------------------------ standalone kernels
def ntt(data, log_n, inverse=False, device=0):
    """In-place natural-order NTT/iNTT of 2^log_n Montgomery-form Fr values held in a writable buffer.
    Returns kernel milliseconds."""
    ms = C.c_float()
    check(_lib.load().nzcp_ntt(addr(data), int(log_n), int(bool(inverse)), int(device), C.byref(ms)))
    return ms.value


def ntt_coset(data, log_n, batch=1, device=0):
    ms = C.c_float()
    check(_lib.load().nzcp_ntt_coset(addr(data), int(log_n), int(batch), int(device), C.byref(ms)))
    return ms.value


def msm(bases, scalars, n_points, g2=False, window_bits=0, device=0):
    """-> (plain affine point bytes: 64 for G1 / 128 for G2, kernel ms)."""
    out = bytearray(128 if g2 else 64)
    ms = C.c_float()
    check(_lib.load().nzcp_msm(addr(bases), addr(scalars), int(n_points), int(bool(g2)), int(window_bits), int(device),
                               addr(out), C.byref(ms)))
    return bytes(out), ms.value


def msm_var(bases, scalars, n_points, g2=False, window_bits=0, device=0):
    """One-shot variable-base MSM (no window table; ffjavascript multiExpAffine's contract).
    -> (plain affine point bytes, {"wall_ms": whole call incl. uploads, "kernel_ms": sort + accumulate + reduce})."""
    out = bytearray(128 if g2 else 64)
    ms = (C.c_float * 2)()
    check(_lib.load().nzcp_msm_var(addr(bases), addr(scalars), int(n_points), int(bool(g2)), int(window_bits), int(device),
                                   addr(out), ms))
    return bytes(out), {"wall_ms": float(ms[0]), "kernel_ms": float(ms[1])}


XYZZ_BYTES = {False: 128, True: 256}   # one extended-Jacobian point (x, y, zz, zzz; Montgomery) in device memory


class MsmPlan:
    """A base set resident on one GPU (csrc/msm_plan.cu).  mode 0 = fixed-base (window table built once, as the prover
    does per zkey section), mode 1 = variable-base (no table).  `run` returns the plain affine sum; `run_partial` leaves
    the sum in HBM as one XYZZ point at `d_out` (a device pointer / CUDA tensor) for an NCCL all-gather."""

    def __init__(self, bases, n_points, g2=False, window_bits=0, mode=1, device=0):
        h = C.c_void_p()
        ms = C.c_float()
        check(_lib.load().nzcp_msm_plan_create(addr(bases) if n_points else None, int(n_points), int(bool(g2)),
                                               int(window_bits), int(mode), int(device), C.byref(h), C.byref(ms)))
        self._h = h
        self.g2, self.n_points, self.mode, self.device, self.build_ms = bool(g2), int(n_points), int(mode), int(device), ms.value

    def run(self, scalars, n_scalars=None):
        n = self.n_points if n_scalars is None else int(n_scalars)
        out = bytearray(128 if self.g2 else 64)
        ms = C.c_float()
        check(_lib.load().nzcp_msm_plan_run(self._h, addr(scalars) if n else None, n, addr(out), C.byref(ms)))
        return bytes(out), ms.value

    def accumulate_ms(self):
        """Device time of the bucket accumulation alone (pair rounds + XYZZ kernel) in the last run."""
        ms = C.c_float()
        check(_lib.load().nzcp_msm_plan_accumulate_ms(self._h, C.byref(ms)))
        return ms.value

    def run_partial(self, scalars, d_out, n_scalars=None):
        n = self.n_points if n_scalars is None else int(n_scalars)
        ms = C.c_float()
        check(_lib.load().nzcp_msm_plan_run_partial(self._h, addr(scalars) if n else None, n, addr(d_out), C.byref(ms)))
        return ms.value

    def close(self):
        if getattr(self, "_h", None):
            _lib.load().nzcp_msm_plan_free(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def msm_sum_partials(d_partials, count, g2=False, device=0):
    """Sum of `count` XYZZ points in device memory (the gathered per-rank partials) -> plain affine bytes."""
    out = bytearray(128 if g2 else 64)
    check(_lib.load().nzcp_msm_sum_partials(addr(d_partials), int(count), int(bool(g2)), int(device), addr(out)))
    return bytes(out)


def zkey_new(r1cs, ptau, device=0, *, circuit_hash=False):
    """snarkjs `zkey new`: .r1cs + prepared .ptau (path | bytes-like | {"type": "mem"}) -> bytearray with the .zkey image
    (gamma = delta = 1, no contributions).  The sparse point combinations run on `device` (csrc/setup.cu).
    circuit_hash=True stamps the circuit hash snarkjs writes into section 10 (zkey_circuit_hash); only such a key passes
    `zkey verify`.  The default leaves it zero, as before; it is meant to flip to True in a later release."""
    lib = _lib.load()
    rb, pb = _as_bytes_like(r1cs), _as_bytes_like(ptau)
    size = C.c_size_t()
    check(lib.nzcp_zkey_new_size(addr(rb), _nbytes(rb), addr(pb), _nbytes(pb), C.byref(size)))
    out = bytearray(size.value)
    written = C.c_size_t()
    check(lib.nzcp_zkey_new(addr(rb), _nbytes(rb), addr(pb), _nbytes(pb), int(device), addr(out), len(out), C.byref(written)))
    assert written.value == len(out)
    if circuit_hash:
        # section 10 (csHash, u32 0) is the last section zkey_new writes
        out[-68:-4] = zkey_circuit_hash(out, pb, device=device)
    return out


def zkey_circuit_hash(init_zkey, ptau, device=0, timings=None):
    """The circuit hash snarkjs's newZKey writes into section 10 (csrc/verify.cu), from an initial key (`zkey new`
    output) and the prepared ptau it was made from -> 64 bytes.  `timings` receives "hash_kernels" (device ms) and
    "blake2b" (host ms)."""
    lib = _lib.load()
    zb, pb = _as_bytes_like(init_zkey), _as_bytes_like(ptau)
    h, ms = bytearray(64), (C.c_float * 2)()
    check(lib.nzcp_zkey_circuit_hash(addr(zb), _nbytes(zb), addr(pb), _nbytes(pb), int(device), addr(h), ms))
    if timings is not None:
        timings.update(hash_kernels=float(ms[0]), blake2b=float(ms[1]))
    return bytes(h)


def host_zkey_circuit_hash(init_zkey, ptau):
    """zkey_circuit_hash with the kernels' per-point code run on the CPU (domain <= 4096); test hook."""
    zb, pb = _as_bytes_like(init_zkey), _as_bytes_like(ptau)
    h = bytearray(64)
    check(_lib.load().nzcp_host_zkey_circuit_hash(addr(zb), _nbytes(zb), addr(pb), _nbytes(pb), addr(h)))
    return bytes(h)


VERIFY_TIMINGS = ("hash_kernels", "blake2b", "l_msm", "h_ntt_msm")
CLAIM_MESSAGES = {3: "INVALID(%d): public key G1 and G2 do not have the same ration",
                  4: "INVALID(%d): deltaAfter does not fillow the public key",
                  8: "Invalid delta2", 11: "L section does not match", 12: "H section does not match"}


def _plain_g1(b):
    x, y = int.from_bytes(bytes(b[:32]), "little"), int.from_bytes(bytes(b[32:]), "little")
    return None if x == 0 and y == 0 else (x, y)


def _plain_g2(b):
    c = [int.from_bytes(bytes(b[32 * i:32 * i + 32]), "little") for i in range(4)]
    return None if not any(c) else ((c[0], c[1]), (c[2], c[3]))


def zkey_verify(zkey, ptau, *, r1cs=None, init=None, seed=None, device=0, timings=None):
    """snarkjs `zkey verify`: checks `zkey` against the circuit, given as the .r1cs (verifyFromR1cs) or as the initial key
    (verifyFromInit), and the prepared ptau (all: path | bytes-like | {"type": "mem"}).  The library runs every check but
    the pairings on the GPU and returns the pairing claims that precede its first failure; they are checked here, in order,
    on the CPU (verifier.same_ratio).  -> dict(ok, message, cs_hash, contributions=[dict(type, name, hash,
    beacon_hash, num_iterations_exp)]).  `seed` (32 bytes, tests) replaces the OS randomness of the L / H scalars;
    `timings` receives VERIFY_TIMINGS in ms plus "pairings" (host ms)."""
    import time
    from . import verifier
    if (r1cs is None) == (init is None):
        raise NzcpError(_lib.NZCP_E_ARG, "zkey_verify: give exactly one of r1cs and init")
    if seed is not None and len(bytes(seed)) != 32:
        raise NzcpError(_lib.NZCP_E_ARG, "seed must be 32 bytes")
    lib = _lib.load()
    zb, pb = _as_bytes_like(zkey), _as_bytes_like(ptau)
    n_claims, n_recs = C.c_size_t(), C.c_size_t()
    check(lib.nzcp_zkey_verify_size(addr(zb), _nbytes(zb), C.byref(n_claims), C.byref(n_recs)))
    claims = (_lib.VerifyClaim * n_claims.value)()
    recs = (_lib.Contribution * max(1, n_recs.value))()
    rep, ms = _lib.VerifyReport(), (C.c_float * 4)()
    sd = None if seed is None else bytes(seed)
    if r1cs is not None:
        cb = _as_bytes_like(r1cs)
        fn = lib.nzcp_zkey_verify_from_r1cs
    else:
        cb = _as_bytes_like(init)
        fn = lib.nzcp_zkey_verify_from_init
    check(fn(addr(cb), _nbytes(cb), addr(pb), _nbytes(pb), addr(zb), _nbytes(zb), sd, int(device), claims,
             n_claims.value, recs, n_recs.value, C.byref(rep), ms))
    t0 = time.perf_counter()
    message = None
    for k in claims[:rep.n_claims]:
        if not verifier.same_ratio(_plain_g1(k.a), _plain_g1(k.b), _plain_g2(k.c), _plain_g2(k.d)):
            message = CLAIM_MESSAGES[k.step] % k.record if "%d" in CLAIM_MESSAGES[k.step] else CLAIM_MESSAGES[k.step]
            break
    if timings is not None:
        timings.update(zip(VERIFY_TIMINGS, [float(x) for x in ms]))
        timings["pairings"] = (time.perf_counter() - t0) * 1e3
    if message is None and rep.failed_step:
        message = rep.message.decode(errors="replace")
    contributions = [{"type": r.type, "name": bytes(r.name[:r.name_len]).decode(errors="replace"), "hash": bytes(r.hash),
                      "beacon_hash": bytes(r.beacon_hash[:r.beacon_hash_len]), "num_iterations_exp": r.num_iterations_exp}
                     for r in recs[:n_recs.value]]
    return {"ok": message is None, "message": message, "cs_hash": bytes(rep.cs_hash), "contributions": contributions}


PTAU_SECTIONS = (12, 13, 14, 15)


def ptau_prepare(ptau, device=0, timings=None):
    """snarkjs `powersoftau prepare phase2`: a phase-1 .ptau (path | bytes-like | {"type": "mem"}) -> bytearray with the
    prepared file (Lagrange-basis sections 12-15 added; csrc/ptau.cu).  The inverse FFTs run on `device`.  `timings`: a
    dict that receives the device milliseconds of each output section, keyed 12, 13, 14, 15."""
    lib = _lib.load()
    pb = _as_bytes_like(ptau)
    size = C.c_size_t()
    check(lib.nzcp_ptau_prepare_size(addr(pb), _nbytes(pb), C.byref(size)))
    out = bytearray(size.value)
    written = C.c_size_t()
    ms = (C.c_float * 4)()
    check(lib.nzcp_ptau_prepare(addr(pb), _nbytes(pb), int(device), addr(out), len(out), C.byref(written), ms))
    assert written.value == len(out)
    if timings is not None:
        timings.update(zip(PTAU_SECTIONS, [float(x) for x in ms]))
    return out


CONTRIBUTE_SECTIONS = (8, 9)


def _utf8(v):
    if v is None:
        return None
    b = v.encode() if isinstance(v, str) else bytes(v)
    if b"\0" in b:
        raise NzcpError(_lib.NZCP_E_ARG, "zkey: contribution name contains a NUL byte")
    return b


def _contribute_out(lib, zb, name, beacon_len):
    size = C.c_size_t()
    check(lib.nzcp_zkey_contribute_size(addr(zb), _nbytes(zb), name, beacon_len, C.byref(size)))
    return bytearray(size.value)


def zkey_contribute(zkey, name=None, entropy=None, seed=None, device=0, timings=None):
    """snarkjs `zkey contribute`: a Groth16 key (path | bytes-like | {"type": "mem"}) -> (bytearray with the new key,
    64-byte contribution hash).  The random key comes from BLAKE2b(64 OS-random bytes || entropy) (str: UTF-8); `seed`
    (32 bytes, tests) seeds the ChaCha directly instead.  Sections 8 and 9 are rescaled on `device`; `timings` receives
    their device milliseconds, keyed 8 and 9."""
    lib = _lib.load()
    zb = _as_bytes_like(zkey)
    nb, eb = _utf8(name), _utf8(entropy) or b""
    if seed is not None and len(bytes(seed)) != 32:
        raise NzcpError(_lib.NZCP_E_ARG, "seed must be 32 bytes")
    out = _contribute_out(lib, zb, nb, 0)
    written, h, ms = C.c_size_t(), bytearray(64), (C.c_float * 2)()
    check(lib.nzcp_zkey_contribute(addr(zb), _nbytes(zb), nb, addr(eb) if eb else None, len(eb),
                                   None if seed is None else bytes(seed), int(device), addr(out), len(out),
                                   C.byref(written), addr(h), ms))
    assert written.value == len(out)
    if timings is not None:
        timings.update(zip(CONTRIBUTE_SECTIONS, [float(x) for x in ms]))
    return out, bytes(h)


def zkey_beacon(zkey, beacon_hash, num_iterations_exp, name=None, device=0, timings=None):
    """snarkjs `zkey beacon`: as zkey_contribute, with the random key derived from `beacon_hash` (bytes) hashed with
    SHA-256 2^num_iterations_exp times (10..63)."""
    lib = _lib.load()
    zb = _as_bytes_like(zkey)
    nb, hb = _utf8(name), bytes(beacon_hash)
    out = _contribute_out(lib, zb, nb, len(hb))
    written, h, ms = C.c_size_t(), bytearray(64), (C.c_float * 2)()
    check(lib.nzcp_zkey_beacon(addr(zb), _nbytes(zb), nb, hb, len(hb), int(num_iterations_exp), int(device), addr(out),
                               len(out), C.byref(written), addr(h), ms))
    assert written.value == len(out)
    if timings is not None:
        timings.update(zip(CONTRIBUTE_SECTIONS, [float(x) for x in ms]))
    return out, bytes(h)


def ptau_new(power, first_challenge=True):
    """snarkjs `powersoftau new`: a fresh phase-1 .ptau of 2^power (1..28) -> (bytearray, 64-byte first challenge hash, or
    None with first_challenge=False, which skips a BLAKE2b pass over ~384 * 2^power bytes).  Host only."""
    lib = _lib.load()
    size = C.c_size_t()
    check(lib.nzcp_ptau_new_size(int(power), C.byref(size)))
    out = bytearray(size.value)
    written, h = C.c_size_t(), bytearray(64) if first_challenge else None
    check(lib.nzcp_ptau_new(int(power), addr(out), len(out), C.byref(written), addr(h)))
    assert written.value == len(out)
    return out, None if h is None else bytes(h)


PTAU_CONTRIBUTE_TIMINGS = (2, 3, 4, 5, 6, "encode", "blake2b")


def _ptau_contribute_out(lib, pb, name, beacon_len):
    size = C.c_size_t()
    check(lib.nzcp_ptau_contribute_size(addr(pb), _nbytes(pb), name, beacon_len, C.byref(size)))
    return bytearray(size.value)


def ptau_contribute(ptau, name=None, entropy=None, seed=None, device=0, timings=None):
    """snarkjs `powersoftau contribute`: a phase-1 .ptau (path | bytes-like | {"type": "mem"}) -> (bytearray with the new
    file, 64-byte response hash).  The random key comes from BLAKE2b(64 OS-random bytes || entropy) (str: UTF-8); `seed`
    (32 bytes, tests) seeds the ChaCha directly instead.  Sections 2-6 are multiplied on `device`; `timings` receives the
    key-kernel device ms keyed 2..6, "encode" (encode kernels, device ms) and "blake2b" (host ms)."""
    lib = _lib.load()
    pb = _as_bytes_like(ptau)
    nb, eb = _utf8(name), _utf8(entropy) or b""
    if seed is not None and len(bytes(seed)) != 32:
        raise NzcpError(_lib.NZCP_E_ARG, "seed must be 32 bytes")
    out = _ptau_contribute_out(lib, pb, nb, 0)
    written, h, ms = C.c_size_t(), bytearray(64), (C.c_float * 7)()
    check(lib.nzcp_ptau_contribute(addr(pb), _nbytes(pb), nb, addr(eb) if eb else None, len(eb),
                                   None if seed is None else bytes(seed), int(device), addr(out), len(out),
                                   C.byref(written), addr(h), ms))
    assert written.value == len(out)
    if timings is not None:
        timings.update(zip(PTAU_CONTRIBUTE_TIMINGS, [float(x) for x in ms]))
    return out, bytes(h)


def ptau_beacon(ptau, beacon_hash, num_iterations_exp, name=None, device=0, timings=None):
    """snarkjs `powersoftau beacon`: as ptau_contribute, with the random key derived from `beacon_hash` (bytes) hashed
    with SHA-256 2^num_iterations_exp times (10..63)."""
    lib = _lib.load()
    pb = _as_bytes_like(ptau)
    nb, hb = _utf8(name), bytes(beacon_hash)
    out = _ptau_contribute_out(lib, pb, nb, len(hb))
    written, h, ms = C.c_size_t(), bytearray(64), (C.c_float * 7)()
    check(lib.nzcp_ptau_beacon(addr(pb), _nbytes(pb), nb, hb, len(hb), int(num_iterations_exp), int(device), addr(out),
                               len(out), C.byref(written), addr(h), ms))
    assert written.value == len(out)
    if timings is not None:
        timings.update(zip(PTAU_CONTRIBUTE_TIMINGS, [float(x) for x in ms]))
    return out, bytes(h)


def host_ptau_contribute(ptau, name=None, entropy=None, seed=None, beacon_hash=None, num_iterations_exp=0):
    """CPU run of ptau_contribute (beacon_hash None) or ptau_beacon, power <= 4 -> the same (bytearray, hash)."""
    lib = _lib.load()
    pb = _as_bytes_like(ptau)
    nb, eb = _utf8(name), _utf8(entropy) or b""
    hb = None if beacon_hash is None else bytes(beacon_hash)
    out = _ptau_contribute_out(lib, pb, nb, len(hb) if hb else 0)
    written, h = C.c_size_t(), bytearray(64)
    check(lib.nzcp_host_ptau_contribute(addr(pb), _nbytes(pb), nb, addr(eb) if eb else None, len(eb),
                                        None if seed is None else bytes(seed), hb, len(hb) if hb is not None else 0,
                                        int(num_iterations_exp), addr(out), len(out), C.byref(written), addr(h)))
    assert written.value == len(out)
    return out, bytes(h)


def zkey_selfcheck(zkey, device=0):
    """Format self-checks of SURVEY.md 8c-3 on a .zkey image (path | bytes-like | {"type": "mem"}) -> dict; ["ok"] is
    the verdict.  Meant for the first REAL snarkjs-made key: it pins the section-4 `coef * R^2` convention, the moduli
    and that every base point is on its curve, without needing snarkjs."""
    data = _as_bytes_like(zkey)
    rep = ZkeyCheck()
    check(_lib.load().nzcp_zkey_selfcheck(addr(data), _nbytes(data), int(device), C.byref(rep)))
    names = ("A", "B1", "B2", "C", "H", "IC")
    return {"ok": bool(rep.ok), "n_vars": rep.n_vars, "n_public": rep.n_public, "domain_size": rep.domain_size,
            "n_constraints": rep.n_constraints, "n_coefs": rep.n_coefs, "bad_coef_values": rep.bad_coef_values,
            "bad_coef_indices": rep.bad_coef_indices, "off_curve": dict(zip(names, [int(x) for x in rep.off_curve])),
            "infinity": dict(zip(names, [int(x) for x in rep.infinity])), "header_moduli_ok": bool(rep.header_moduli_ok),
            "header_points_ok": bool(rep.header_points_ok), "public_rows_ok": bool(rep.public_rows_ok)}


def selftest(device=0, seed=1, n_cases=4096):
    bad = C.c_uint32()
    check(_lib.load().nzcp_selftest(int(device), int(seed), int(n_cases), C.byref(bad)))
    return bad.value


def field_op(field, op, a, b, n, device=0):
    out = bytearray(32 * n)
    check(_lib.load().nzcp_field_op(int(field), int(op), addr(a), addr(b), addr(out), int(n), int(device)))
    return bytes(out)


# nzcp_arith_op record sizes in bytes, per op: (input, output)
ARITH_IO = ((64, 64), (64, 32), (128, 32), (128, 32), (128, 64), (128, 64), (64, 64), (64, 64), (64, 64), (256, 64))


def arith_op(op, data, n, device=0):
    """Device Fq / Fq2 arithmetic on n little-endian records (include/nzcp_prover.h nzcp_arith_op) -> output records."""
    out = bytearray(ARITH_IO[op][1] * n)
    check(_lib.load().nzcp_arith_op(int(op), addr(data), addr(out), int(n), int(device)))
    return bytes(out)


def curve_op(g2, op, a, b, n, device=0):
    """Device XYZZ group law on n records (include/nzcp_prover.h nzcp_curve_op) -> XYZZ records, affine for op 4."""
    out = bytearray((128 if g2 else 64) * n * (1 if op == 4 else 2))
    check(_lib.load().nzcp_curve_op(int(bool(g2)), int(op), addr(a), addr(b), addr(out), int(n), int(device)))
    return bytes(out)


def intpipe_bench(device=0, iters=4096):
    """-> dict(imad_wide_per_s, imad_lo_per_s, fq_mul_per_s, sm_count): the integer-pipe roofline denominators."""
    out = (C.c_double * 4)()
    check(_lib.load().nzcp_intpipe_bench(int(device), int(iters), out))
    return {"imad_wide_per_s": out[0], "imad_lo_per_s": out[1], "fq_mul_per_s": out[2], "sm_count": int(out[3])}


def intpipe_modes(device=0, iters=4096):
    out = (C.c_double * 10)()
    check(_lib.load().nzcp_intpipe_modes(int(device), int(iters), out))
    names = ("mad_wide", "mad_lo", "fq_mul", "chain2_wide", "chain4_wide", "chain8_wide", "chain2_plus_addc", "addc_only",
             "mad_wide_plus_2addc")
    return dict(zip(names, list(out)[:9]))


def pipe_probe(device=0, iters=4096):
    """Which instructions issue beside IMAD.WIDE: -> dict of per-second rates (csrc/standalone.cu pipeprobe_kernel)."""
    out = (C.c_double * 5)()
    check(_lib.load().nzcp_pipe_probe(int(device), int(iters), out))
    names = ("dfma_alone", "wide_with_dfma_1to1", "wide_with_2xor", "wide_with_2add", "dfma_with_wide_1to1")
    return dict(zip(names, list(out)))


def host_field_op(field, op, a, b, n):
    out = bytearray(32 * n)
    check(_lib.load().nzcp_host_field_op(int(field), int(op), addr(a), addr(b), addr(out), int(n)))
    return bytes(out)


def host_scalar_mul(g2, base_mont, scalar):
    out = bytearray(128 if g2 else 64)
    sb = _scalar32(scalar)
    check(_lib.load().nzcp_host_scalar_mul(int(bool(g2)), addr(base_mont), addr(sb), addr(out)))
    return bytes(out)


def host_msm_sim(bases, scalars, n_points, g2=False, window_bits=8, rounds=1, adds_per_thread=4):
    """CPU run of the MSM data path incl. the batched-affine pair rounds (same code as the kernels) -> plain affine."""
    out = bytearray(128 if g2 else 64)
    check(_lib.load().nzcp_host_msm_sim(addr(bases), addr(scalars), int(n_points), int(bool(g2)), int(window_bits),
                                        int(rounds), int(adds_per_thread), addr(out)))
    return bytes(out)


def host_ptau_prepare(ptau):
    """CPU run of ptau_prepare's load / stage / butterfly code (power <= 4) -> the same bytes."""
    lib = _lib.load()
    pb = _as_bytes_like(ptau)
    size = C.c_size_t()
    check(lib.nzcp_ptau_prepare_size(addr(pb), _nbytes(pb), C.byref(size)))
    out = bytearray(size.value)
    written = C.c_size_t()
    check(lib.nzcp_host_ptau_prepare(addr(pb), _nbytes(pb), addr(out), len(out), C.byref(written)))
    assert written.value == len(out)
    return out


def host_zkey_contribute(zkey, name=None, entropy=None, seed=None, beacon_hash=None, num_iterations_exp=0):
    """CPU run of zkey_contribute (beacon_hash None) or zkey_beacon, sections 8 + 9 of at most 4096 points -> the same
    (bytearray, hash)."""
    lib = _lib.load()
    zb = _as_bytes_like(zkey)
    nb, eb = _utf8(name), _utf8(entropy) or b""
    hb = None if beacon_hash is None else bytes(beacon_hash)
    out = _contribute_out(lib, zb, nb, len(hb) if hb else 0)
    written, h = C.c_size_t(), bytearray(64)
    check(lib.nzcp_host_zkey_contribute(addr(zb), _nbytes(zb), nb, addr(eb) if eb else None, len(eb),
                                        None if seed is None else bytes(seed), hb, len(hb) if hb is not None else 0,
                                        int(num_iterations_exp), addr(out), len(out), C.byref(written), addr(h)))
    assert written.value == len(out)
    return out, bytes(h)


def tuning_set(name, value):
    """Process-wide tuning knob (see include/nzcp_prover.h nzcp_tuning_set)."""
    check(_lib.load().nzcp_tuning_set(name.encode(), int(value)))


def host_root_of_unity(k):
    out = bytearray(32)
    check(_lib.load().nzcp_host_root_of_unity(int(k), addr(out)))
    return int.from_bytes(out, "little")


# ------------------------------------------------------------------------------------------------ synthetic circuits
def synth_points(seed, n_points, g2=False, device=0):
    """n pseudo-random points k_i * G as a bytearray of Montgomery affine coordinates (zkey section format)."""
    out = bytearray(n_points * (128 if g2 else 64))
    check(_lib.load().nzcp_synth_points(int(seed), int(n_points), int(bool(g2)), int(device), addr(out) if n_points else None))
    return out


class SynthCircuit:
    """Random forward-solvable R1CS of the NZCP shape + Groth16 setup from explicit toxic waste (GPU)."""

    def __init__(self, seed, n_constraints, n_public, n_free):
        h = C.c_void_p()
        check(_lib.load().nzcp_synth_create(int(seed), int(n_constraints), int(n_public), int(n_free), C.byref(h)))
        self._h = h
        nv, nc, npub, dom = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()
        ncoef = C.c_uint64()
        check(_lib.load().nzcp_synth_dims(h, C.byref(nv), C.byref(nc), C.byref(npub), C.byref(dom), C.byref(ncoef)))
        self.n_vars, self.n_constraints, self.n_public = nv.value, nc.value, npub.value
        self.domain_size, self.n_coefs = dom.value, ncoef.value

    def zkey(self, toxic, device=0):
        """toxic: 5 ints (tau, alpha, beta, gamma, delta) -> bytearray with the .zkey image."""
        lib = _lib.load()
        tb = b"".join(int(t).to_bytes(32, "little") for t in toxic)
        out = bytearray(lib.nzcp_synth_zkey_size(self._h))
        check(lib.nzcp_synth_write_zkey(self._h, addr(tb), int(device), addr(out), len(out)))
        return out

    def r1cs(self):
        lib = _lib.load()
        out = bytearray(lib.nzcp_synth_r1cs_size(self._h))
        check(lib.nzcp_synth_write_r1cs(self._h, addr(out), len(out)))
        return out

    def wtns(self, witness_seed):
        lib = _lib.load()
        out = bytearray(lib.nzcp_synth_wtns_size(self._h))
        check(lib.nzcp_synth_write_wtns(self._h, int(witness_seed), addr(out), len(out)))
        return out

    def close(self):
        if getattr(self, "_h", None):
            _lib.load().nzcp_synth_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
