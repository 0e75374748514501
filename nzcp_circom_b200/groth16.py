"""snarkjs-shaped surface: groth16.fullProve / groth16.prove / groth16.verify, zKey.exportVerificationKey.

Mirrors snarkjs 0.4.12 main.js `groth16` (upstream, not vendored: /root/reference/package.json:12,
yarn.lock:987-999).  The reference's tests build the prover input at /root/reference/test/nzcp.js:37-38
(`{ toBeSigned: bufferToBitArray(bytes), toBeSignedLen }`) and read public signals as witness[1..513] at
test/nzcp.js:41-48; `publicSignals` below is that same slice, in the same order, as decimal strings.

`zKey` groups newZKey / contribute / beacon / verifyFromR1cs / verifyFromInit / exportVerificationKey the way snarkjs's
main.js does (snarkjs.zKey.newZKey, ...); `powersOfTau` groups newAccumulator / contribute / beacon / preparePhase2
(snarkjs.powersOfTau.*).

Same names, argument meaning and error text as snarkjs:
  prove(zkeyFileName, witnessFileName, logger=None)   file args: path | bytes-like | {"type": "mem", "data": ...}
  fullProve(input, wasmFile, zkeyFileName, logger=None)
  verify(vk_verifier, publicSignals, proof, logger=None)
Extensions (keyword-only): r=, s= inject the blinding scalars (snarkjs draws them with Fr.random() and has no hook --
bit-exact comparison needs one, SURVEY.md 8b); device= picks the GPU.

The Python functions are synchronous (snarkjs returns Promises); the Node wrapper in js/ returns Promises.
The proving key is parsed and uploaded on first use and cached per (source, device): snarkjs re-reads the five point
sections from disk on every call.
"""
import collections
import hashlib
import os
import struct
import threading

from . import _lib, api, verifier
from ._lib import NzcpError

_Q = verifier.Q
_RINV_Q = pow(1 << 256, -1, _Q)

MAX_CACHED_KEYS = 4      # resident proving keys kept by prove() (an NZCP key is ~5.8 GB of HBM); least recently used goes


class _Entry:
    """One resident proving key with its prover.  `lock` serialises proofs: an nzcp_prover carries ONE in-flight proof
    (one stream set, one set of work buffers) and ctypes drops the GIL inside nzcp_prove, so two threads calling
    groth16.prove on the same key must not reach the library at the same time."""

    def __init__(self, zk, pr):
        self.zk, self.pr = zk, pr
        self.lock = threading.Lock()

    def close(self):
        with self.lock:
            self.pr.close()
            self.zk.close()


_cache = collections.OrderedDict()     # key -> _Entry, in least-recently-used order
_cache_lock = threading.Lock()         # guards _cache and makes "load the key once" atomic


def _cache_key(zkey, device):
    """Files are identified by path + mtime + size; in-memory keys by a digest of their CONTENT (an id()-based key
    would go stale when a bytearray is mutated or an address reused)."""
    if isinstance(zkey, dict) and zkey.get("type") == "mem":
        zkey = zkey["data"]
    if isinstance(zkey, str) or hasattr(zkey, "__fspath__"):
        p = os.path.abspath(os.fspath(zkey))
        st = os.stat(p)
        return ("path", p, st.st_mtime_ns, st.st_size, device)
    return ("mem", _fingerprint(zkey), len(zkey), device)


def _fingerprint(buf):
    """Digest of an in-memory key: everything up to 8 MB; beyond that the first and last 64 KB (header, verification-key
    points, section table) plus 256 evenly spaced 4 KB blocks -- two different proving keys differ in delta and hence in
    every C and H point, so sampled blocks tell them apart at ~1 MB hashed per call instead of 0.5 GB."""
    mv = memoryview(buf).cast("B")
    n = len(mv)
    h = hashlib.blake2b(digest_size=16)
    h.update(n.to_bytes(8, "little"))
    if n <= (8 << 20):
        h.update(mv)
    else:
        h.update(mv[:65536])
        h.update(mv[n - 65536:])
        step = n // 256
        for k in range(256):
            h.update(mv[k * step:k * step + 4096])
    return h.digest()


def _get_entry(zkey, device):
    key = _cache_key(zkey, device)
    evicted = []
    with _cache_lock:
        ent = _cache.get(key)
        if ent is None:
            zk = api.Zkey(api._as_bytes_like(zkey), device)      # under the lock: a first-call race must not load it twice
            try:
                ent = _Entry(zk, api.Prover(zk))
            except Exception:
                zk.close()
                raise
            _cache[key] = ent
            while len(_cache) > MAX_CACHED_KEYS:
                evicted.append(_cache.popitem(last=False)[1])
        else:
            _cache.move_to_end(key)
    for e in evicted:
        e.close()          # waits for a proof still running on the evicted key
    return ent


def terminate():
    """snarkjs callers `await curve.terminate()` to stop the worker pool; here it frees the cached GPU state."""
    with _cache_lock:
        ents = list(_cache.values())
        _cache.clear()
    for e in ents:
        e.close()


def _le(b, i):
    return int.from_bytes(b[32 * i:32 * i + 32], "little")


def proof_from_bytes(pb):
    """256-byte C-ABI proof -> snarkjs proof object (decimal strings of plain affine coordinates)."""
    v = [_le(pb, i) for i in range(8)]
    # the point at infinity: ffjavascript's G.zero is [0, 1, 0], and that is what toObject(toAffine(P)) prints
    def g1(x, y):
        return ["0", "1", "0"] if x == 0 and y == 0 else [str(x), str(y), "1"]
    b_inf = all(x == 0 for x in v[2:6])
    return {
        "pi_a": g1(v[0], v[1]),
        "pi_b": [["0", "0"], ["1", "0"], ["0", "0"]] if b_inf else [[str(v[2]), str(v[3])], [str(v[4]), str(v[5])], ["1", "0"]],
        "pi_c": g1(v[6], v[7]),
        "protocol": "groth16",
        "curve": "bn128",
    }


def _public_signals(wtns_bytes, n_public):
    """witness[1 .. nPublic] from section 2 of the .wtns image, as decimal strings."""
    mv = memoryview(wtns_bytes)
    nsec = struct.unpack_from("<I", mv, 8)[0]
    pos = 12
    for _ in range(nsec):
        sid, ln = struct.unpack_from("<IQ", mv, pos)
        pos += 12
        if sid == 2:
            return [str(int.from_bytes(mv[pos + 32 * i:pos + 32 * i + 32], "little")) for i in range(1, n_public + 1)]
        pos += ln
    raise NzcpError(_lib.NZCP_E_FORMAT, "wtns: missing section 2")


def prove(zkeyFileName, witnessFileName, logger=None, *, r=None, s=None, device=0):
    """groth16.prove -> {"proof": {...}, "publicSignals": [...]}"""
    if logger:
        logger.debug("Reading Wtns")
    wt = api._as_bytes_like(witnessFileName)
    if logger:
        logger.debug("Reading zkey")
    ent = _get_entry(zkeyFileName, device)
    zk = ent.zk
    with ent.lock:
        res = ent.pr.prove(wt, r=r, s=s, debug=logger is not None)
    if logger:
        for k, v in res["stage_ms"].items():
            logger.debug("%s: %.3f ms" % (k, v))
    return {"proof": proof_from_bytes(res["proof"]), "publicSignals": _public_signals(wt, zk.n_public)}


_NODE_WTNS_SCRIPT = (
    'const snarkjs = require("snarkjs"); const fs = require("fs");'
    '(async () => { const input = JSON.parse(fs.readFileSync(process.argv[1], "utf8"));'
    ' await snarkjs.wtns.calculate(input, process.argv[2], process.argv[3]); process.exit(0); })()'
    '.catch((e) => { console.error(e && e.message ? e.message : String(e)); process.exit(1); });')


def calculate_witness(input, wasmFile, node=None, cwd=None):
    """snarkjs `wtns.calculate(input, wasmFile, wtns)` -- the step BEFORE the proving path (SURVEY.md 8f-3): it runs the
    circom-generated WASM on the CPU and is out of scope for the GPU work, so it is delegated to the reference's own
    toolchain: a `node` process with snarkjs installed (circom_runtime's WitnessCalculator underneath).  `node`: the
    executable (default: $NZCP_NODE or "node" on PATH); `cwd`: where `require("snarkjs")` resolves (the reference
    checkout with its node_modules).  Returns the .wtns image.  Raises NzcpError(NZCP_E_ARG) when no node is available --
    there is no WASM runtime inside this package."""
    import json
    import shutil
    import subprocess
    import tempfile
    exe = node or os.environ.get("NZCP_NODE") or shutil.which("node")
    if not exe or (os.path.sep in exe and not os.path.exists(exe)):
        raise NzcpError(_lib.NZCP_E_ARG,
                        "fullProve: witness calculation needs node + snarkjs (the reference's own toolchain) and no node "
                        "executable was found; pass a witness-calculator callable as wasmFile, or call prove() with a .wtns")
    wasm = os.fspath(wasmFile)
    if not os.path.exists(wasm):
        raise NzcpError(_lib.NZCP_E_ARG, "fullProve: wasm file not found: %s" % wasm)
    with tempfile.TemporaryDirectory(prefix="nzcp_wtns_") as d:
        inp, out = os.path.join(d, "input.json"), os.path.join(d, "witness.wtns")
        def js_safe(v):   # integers beyond 2^53 travel as decimal strings (JSON.parse would round them; snarkjs accepts strings)
            if isinstance(v, bool) or v is None or isinstance(v, str):
                return v
            if isinstance(v, int):
                return v if -(1 << 53) < v < (1 << 53) else str(v)
            if isinstance(v, dict):
                return {str(k): js_safe(x) for k, x in v.items()}
            if isinstance(v, (list, tuple)):
                return [js_safe(x) for x in v]
            return str(v)
        with open(inp, "w") as f:
            json.dump(js_safe(input), f)
        res = subprocess.run([exe, "-e", _NODE_WTNS_SCRIPT, inp, os.path.abspath(wasm), out], cwd=cwd, capture_output=True, text=True)
        if res.returncode != 0 or not os.path.exists(out):
            raise NzcpError(_lib.NZCP_E_ARG, "fullProve: witness calculation failed: %s" % (res.stderr.strip() or res.stdout.strip()))
        with open(out, "rb") as f:
            return f.read()


def fullProve(input, wasmFile, zkeyFileName, logger=None, *, r=None, s=None, device=0, node=None, node_cwd=None):
    """groth16.fullProve: witness calculation (circom-generated WASM, CPU) followed by prove().

    The witness generator is outside the hot path (SURVEY.md 8f row 3).  `wasmFile` may be
      * a callable `calc(input) -> .wtns bytes` (any binding of circom_runtime's WitnessCalculator), or
      * a path to the circuit's .wasm, as in snarkjs: the witness is then computed by the reference's own toolchain in a
        `node` child process (calculate_witness above); without node this raises -- no WASM runtime ships here.
    """
    if callable(wasmFile):
        wtns = wasmFile(input)
    else:
        if logger:
            logger.debug("Calculating the witness with node + snarkjs")
        wtns = calculate_witness(input, wasmFile, node=node, cwd=node_cwd)
    return prove(zkeyFileName, {"type": "mem", "data": wtns}, logger, r=r, s=s, device=device)


def verify(vk_verifier, publicSignals, proof, logger=None):
    """groth16.verify: CPU pairing check (snarkjs verifies on the CPU as well)."""
    return verifier.verify(vk_verifier, publicSignals, proof, logger)


def newZKey(r1csName, ptauName, zkeyName=None, logger=None, *, device=0, circuit_hash=False):
    """snarkjs zKey.newZKey(r1csName, ptauName, zkeyName): the circuit-specific key from an .r1cs and a prepared .ptau,
    computed on the GPU.  `zkeyName`: a path to write, a {"type": "mem"} object that receives `.data`, or None.
    Returns the .zkey image (snarkjs returns the circuit hash).  circuit_hash=True computes the circuit hash and writes it
    into section 10 as snarkjs does, which `zkey verify` requires; the default still leaves it zero (api.zkey_new)."""
    if logger:
        logger.info("Reading r1cs / ptau, combining points on the GPU")
    data = api.zkey_new(r1csName, ptauName, device=device, circuit_hash=circuit_hash)
    if isinstance(zkeyName, dict):
        zkeyName["data"] = data
    elif zkeyName is not None:
        with open(zkeyName, "wb") as f:
            f.write(data)
    return data


def exportVerificationKey(zkeyFileName):
    """snarkjs zKey.exportVerificationKey: header points + IC (section 3), plain decimal strings."""
    data = api._as_bytes_like(zkeyFileName)
    mv = memoryview(data)
    if bytes(mv[:4]) != b"zkey":
        raise NzcpError(_lib.NZCP_E_FORMAT, "zkey file: Invalid File format")
    nsec = struct.unpack_from("<I", mv, 8)[0]
    pos, secs = 12, {}
    for _ in range(nsec):
        sid, ln = struct.unpack_from("<IQ", mv, pos)
        pos += 12
        secs.setdefault(sid, (pos, ln))
        pos += ln
    if struct.unpack_from("<I", mv, secs[1][0])[0] != 1:
        raise NzcpError(_lib.NZCP_E_NOT_GROTH16, "zkey file is not groth16")
    h = secs[2][0]
    n_vars, n_public, _dom = struct.unpack_from("<III", mv, h + 72)

    def fq(off):
        return int.from_bytes(mv[off:off + 32], "little") * _RINV_Q % _Q

    def g1(off):
        x, y = fq(off), fq(off + 32)
        return ["0", "1", "0"] if x == 0 and y == 0 else [str(x), str(y), "1"]

    def g2(off):
        c = [fq(off + 32 * i) for i in range(4)]
        if all(v == 0 for v in c):
            return [["0", "0"], ["1", "0"], ["0", "0"]]
        return [[str(c[0]), str(c[1])], [str(c[2]), str(c[3])], ["1", "0"]]

    p = h + 84
    vk = {"protocol": "groth16", "curve": "bn128", "nPublic": n_public}
    vk["vk_alpha_1"] = g1(p)
    vk["vk_beta_2"] = g2(p + 128)
    vk["vk_gamma_2"] = g2(p + 256)
    vk["vk_delta_2"] = g2(p + 448)
    ic0 = secs[3][0]
    vk["IC"] = [g1(ic0 + 64 * i) for i in range(n_public + 1)]
    return vk


def _write_out(dest, data):
    if isinstance(dest, dict):
        dest["data"] = data
    elif dest is not None:
        with open(dest, "wb") as f:
            f.write(data)


def _log_sections(logger, timings):
    if logger:
        for sid, ms in timings.items():
            logger.debug("section %d: %.3f ms" % (sid, ms))


def preparePhase2(oldPtauFilename, newPTauFilename=None, logger=None, *, device=0):
    """snarkjs powersOfTau.preparePhase2(oldPtauFilename, newPTauFilename): adds the Lagrange-basis sections 12-15 that
    `zkey new` reads, computed on the GPU.  `newPTauFilename`: a path to write, a {"type": "mem"} object that receives
    `.data`, or None.  Returns the prepared .ptau image."""
    timings = {} if logger else None
    data = api.ptau_prepare(oldPtauFilename, device=device, timings=timings)
    _log_sections(logger, timings)
    _write_out(newPTauFilename, data)
    return data


def newAccumulator(curve, power, fileName=None, logger=None):
    """snarkjs powersOfTau.newAccumulator(curve, power, fileName): a fresh phase-1 file of 2^power (1..28) on the host.
    `curve`: "bn128" / "bn254" or None (bn128).  `fileName`: a path to write, a {"type": "mem"} object that receives
    `.data`, or None.  Returns the 64-byte first challenge hash, as snarkjs does."""
    if curve is not None and str(curve).lower() not in ("bn128", "bn254"):
        raise NzcpError(_lib.NZCP_E_CURVE, "Curve not supported: %s" % curve)
    data, h = api.ptau_new(power)
    if logger:
        logger.debug(_format_hash(hashlib.blake2b(digest_size=64).digest(), "Blank Contribution Hash:"))
        logger.info(_format_hash(h, "First Contribution Hash:"))
    _write_out(fileName, data)
    return h


def _section_ids(buf):
    mv = memoryview(buf).cast("B")
    pos, ids = 12, []
    for _ in range(struct.unpack_from("<I", mv, 8)[0] if len(mv) >= 12 else 0):
        if pos + 12 > len(mv):
            break
        sid, ln = struct.unpack_from("<IQ", mv, pos)
        ids.append(sid)
        pos += 12 + ln
    return ids


def _ptau_step(old, new, logger, run, params_len):
    """Shared tail of powersOfTau.contribute / beacon: the phase-2 warning, the call, snarkjs's log lines, the output."""
    pb = api._as_bytes_like(old)
    if logger and 12 in _section_ids(pb):
        logger.warn("WARNING: Contributing into a file that has phase2 calculated. You will have to prepare phase2 again.")
    timings = {} if logger else None
    data, h = run(pb, timings)
    if logger:
        end = len(data) - params_len - 8     # the new record is last: ... nextChallenge, type, paramLength, parameters
        for k, v in timings.items():
            logger.debug("%s: %.3f ms" % (k if isinstance(k, str) else "section %d" % k, v))
        logger.info(_format_hash(h, "Contribution Response Hash imported: "))
        logger.info(_format_hash(bytes(data[end - 64:end]), "Next Challenge Hash: "))
    _write_out(new, data)
    return h


def ptauContribute(oldPtauFilename, newPTauFilename, name, entropy, logger=None, *, seed=None, device=0):
    """snarkjs powersOfTau.contribute(oldPtauFilename, newPTauFilename, name, entropy): one phase-1 contribution; sections
    2-6 are multiplied on the GPU.  Empty entropy means OS randomness alone (snarkjs would prompt for it).
    `newPTauFilename`: a path to write, a {"type": "mem"} object that receives `.data`, or None.  Returns the 64-byte
    response hash.  `seed` (32 bytes) replaces the randomness: for tests only."""
    nb = api._utf8(name or None)
    return _ptau_step(oldPtauFilename, newPTauFilename, logger,
                      lambda pb, t: api.ptau_contribute(pb, name=name or None, entropy=entropy or None, seed=seed,
                                                        device=device, timings=t),
                      2 + len(nb) if nb else 0)


def _beacon_hash(beaconHashStr):
    try:
        hb = bytes.fromhex(beaconHashStr)
    except (TypeError, ValueError):
        hb = b""
    if not hb or len(hb) * 2 != len(beaconHashStr):
        raise NzcpError(_lib.NZCP_E_ARG, "Invalid Beacon Hash. (It must be a valid hexadecimal sequence)")
    return hb


def ptauBeacon(oldPtauFilename, newPTauFilename, name, beaconHashStr, numIterationsExp, logger=None, *, device=0):
    """snarkjs powersOfTau.beacon(oldPtauFilename, newPTauFilename, name, beaconHashStr, numIterationsExp): the final,
    publicly reproducible phase-1 contribution, its key derived from the hex string beaconHashStr hashed
    2^numIterationsExp times.  Output and return value as ptauContribute."""
    hb = _beacon_hash(beaconHashStr)
    nb = api._utf8(name or None)
    return _ptau_step(oldPtauFilename, newPTauFilename, logger,
                      lambda pb, t: api.ptau_beacon(pb, hb, int(numIterationsExp), name=name or None, device=device,
                                                    timings=t),
                      (2 + len(nb) if nb else 0) + 4 + len(hb))


def contribute(zkeyNameOld, zkeyNameNew, name, entropy, logger=None, *, seed=None, device=0):
    """snarkjs zKey.contribute(zkeyNameOld, zkeyNameNew, name, entropy): one phase-2 contribution to delta; sections 8
    and 9 are rescaled on the GPU.  Empty entropy means OS randomness alone (snarkjs would prompt for it).
    `zkeyNameNew`: a path to write, a {"type": "mem"} object that receives `.data`, or None.  Returns the 64-byte
    contribution hash.  `seed` (32 bytes) replaces the randomness: for tests only."""
    timings = {} if logger else None
    data, h = api.zkey_contribute(zkeyNameOld, name=name or None, entropy=entropy or None, seed=seed, device=device,
                                  timings=timings)
    _log_sections(logger, timings)
    _write_out(zkeyNameNew, data)
    return h


def beacon(zkeyNameOld, zkeyNameNew, name, beaconHashStr, numIterationsExp, logger=None, *, device=0):
    """snarkjs zKey.beacon(zkeyNameOld, zkeyNameNew, name, beaconHashStr, numIterationsExp): the final, publicly
    reproducible contribution, its key derived from the hex string beaconHashStr hashed 2^numIterationsExp times.
    Output and return value as contribute."""
    hb = _beacon_hash(beaconHashStr)
    timings = {} if logger else None
    data, h = api.zkey_beacon(zkeyNameOld, hb, int(numIterationsExp), name=name or None, device=device, timings=timings)
    _log_sections(logger, timings)
    _write_out(zkeyNameNew, data)
    return h


def _format_hash(h, title):
    """misc.js formatHash: the title, then the hash in four lines of four 8-hex-digit groups."""
    hx = h.hex()
    rows = ["\t\t" + " ".join(hx[32 * r + 8 * c:32 * r + 8 * c + 8] for c in range(4)) for r in range(4)]
    return "\n".join([title] + rows)


def _verify(res, logger):
    if logger:
        if not res["ok"]:
            logger.error(res["message"])
        else:
            logger.info(_format_hash(res["cs_hash"], "Circuit Hash: "))
            for i in range(len(res["contributions"]) - 1, -1, -1):
                c = res["contributions"][i]
                logger.info("-------------------------")
                logger.info(_format_hash(c["hash"], "contribution #%d %s:" % (i + 1, c["name"])))
                if c["type"] == 1:
                    logger.info("Beacon generator: %s" % c["beacon_hash"].hex())
                    logger.info("Beacon iterations Exp: %d" % c["num_iterations_exp"])
            logger.info("-------------------------")
            logger.info("ZKey Ok!")
    return res["ok"]


def verifyFromR1cs(r1csFileName, pTauFileName, zkeyFileName, logger=None, *, seed=None, device=0):
    """snarkjs zKey.verifyFromR1cs: rebuilds the initial key (newZKey with its circuit hash) and checks `zkeyFileName`
    against it (verifyFromInit).  Returns a bool; the logger gets snarkjs's messages.  `seed` (32 bytes) replaces the OS
    randomness of the L / H checks: for tests only."""
    return _verify(api.zkey_verify(zkeyFileName, pTauFileName, r1cs=r1csFileName, seed=seed, device=device), logger)


def verifyFromInit(initFileName, pTauFileName, zkeyFileName, logger=None, *, seed=None, device=0):
    """snarkjs zKey.verifyFromInit: every contribution of `zkeyFileName` chains onto the one before, and the key is the
    initial key `initFileName` with the contributed delta (sections 8 and 9 through random linear combinations on the GPU,
    pairings on the CPU).  Returns a bool, as verifyFromR1cs."""
    return _verify(api.zkey_verify(zkeyFileName, pTauFileName, init=initFileName, seed=seed, device=device), logger)


class powersOfTau:
    """snarkjs.powersOfTau namespace: the entries this library computes."""
    newAccumulator = staticmethod(newAccumulator)
    contribute = staticmethod(ptauContribute)
    beacon = staticmethod(ptauBeacon)
    preparePhase2 = staticmethod(preparePhase2)


class zKey:
    """snarkjs.zKey namespace: the setup entries this library computes and the key export."""
    newZKey = staticmethod(newZKey)
    contribute = staticmethod(contribute)
    beacon = staticmethod(beacon)
    verifyFromR1cs = staticmethod(verifyFromR1cs)
    verifyFromInit = staticmethod(verifyFromInit)
    exportVerificationKey = staticmethod(exportVerificationKey)
