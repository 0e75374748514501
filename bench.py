#!/usr/bin/env python
"""bench.py -- Groth16 proofs/s (nzcp, BN254) on N B200s, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--shape live|example|small] [--impl reference]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): the nzcp_liveTest shape -- n = 2^20, 835 000 constraints, 880 001 wires,
513 public signals, ~4.6 M A/B coefficients -- as a SYNTHETIC R1CS + satisfying witnesses (the real circuit cannot be
compiled here: no circom / sha256-var-circom, SURVEY.md F5).  A step = B independent proofs (distinct witnesses, one
resident proving key).  Multi-GPU = batch sharding, no collective (weak scaling: B proofs per rank per step).

`value`  : proofs/s with the witnesses already resident in HBM (nzcp_prove_device).
`e2e`    : proofs/s through the reference-facing call (nzcp_prove_batch: .wtns images in pinned HOST memory in, the
           proofs in host memory out; H2D + D2H inside the timed region, random r/s); `e2e.pageable` = the same from
           ordinary pageable memory.
`extras` : BASELINE configs[2] (1024 exampleTest-shape proofs sharded over the ranks) and configs[4] (one 2^24-point G1
           MSM split over the ranks, NCCL gather of the partial sums) -- skipped with --no-extras.
`roofline`: the dominant kernel of the step, timed live with CUDA events on its own stream inside the library.
`cpu_baseline` / `--impl reference`: the C restatement of snarkjs groth16.prove (oracle/c) on the host cores -- NOT
           snarkjs itself (node is not installed on these boxes); labelled kind="port".
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPES = {
    # name: (n_constraints, n_public, n_free)  -> n_vars = 1 + n_free + n_constraints
    "live": (835000, 513, 45000),       # S_live  (SURVEY.md 8d): m = 880 001, n = 2^20
    "example": (716000, 513, 44000),    # S_ex: m = 760 001, n = 2^20
    "small": (30000, 33, 2000),         # n = 2^15, for quick checks
}
TOXIC = [0x1234567890ABCDEF1234567, 0xA1FA, 0xBE7A0000001, 0x6A33A, 0xDE17A5]
R_FIXED = 0x0123456789ABCDEF0123456789ABCDEF0123456789ABCDEF0123456789ABCD
S_FIXED = 0x0FEDCBA9876543210FEDCBA9876543210FEDCBA9876543210FEDCBA9876543


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU through NVML every 100 ms while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = str(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4,
                 "hw_power_brake": 0x80, "sync_boost": 0x10}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, b in names.items():
                    if bits & b:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def make_workload(shape, device, n_witness, first_seed):
    from nzcp_circom_b200 import api
    nc, npub, nfree = SHAPES[shape]
    sc = api.SynthCircuit(seed=0xC0FFEE, n_constraints=nc, n_public=npub, n_free=nfree)
    zkey = sc.zkey(TOXIC, device=device)
    wtns = [sc.wtns(first_seed + i) for i in range(n_witness)]
    dims = {"n_constraints": nc, "n_vars": sc.n_vars, "n_public": npub, "domain_size": sc.domain_size,
            "n_coefs": sc.n_coefs}
    return zkey, wtns, dims


def workload_cache_dir():
    d = os.environ.get("NZCP_BENCH_CACHE") or os.path.join(os.environ.get("TMPDIR", "/tmp"), "nzcp_bench_cache")
    os.makedirs(d, exist_ok=True)
    return d


def make_workload_files(shape, n_witness, first_seed):
    """The same workload as make_workload, written to files by a SEPARATE process: the reference arm must not map
    libnzcp_prover.so (the synthetic key is made by the library's GPU setup kernel), so it only reads the result.
    -> (zkey bytes, [wtns bytes], dims)."""
    import subprocess
    d = workload_cache_dir()
    tag = "%s_s%d_n%d" % (shape, first_seed, n_witness)
    meta = os.path.join(d, tag + ".json")
    if not os.path.exists(meta):
        code = ("import json,sys; sys.path.insert(0, %r); import bench\n"
                "zkey, wtns, dims = bench.make_workload(%r, 0, %d, %d)\n"
                "open(%r, 'wb').write(zkey)\n"
                "[open(%r %% i, 'wb').write(w) for i, w in enumerate(wtns)]\n"
                "json.dump(dims, open(%r + '.tmp', 'w'))\n"
                % (ROOT, shape, n_witness, first_seed, os.path.join(d, tag + ".zkey"), os.path.join(d, tag + "_%d.wtns"), meta))
        subprocess.check_call([sys.executable, "-c", code], stdout=sys.stderr)
        os.replace(meta + ".tmp", meta)
    dims = json.load(open(meta))
    zkey = open(os.path.join(d, tag + ".zkey"), "rb").read()
    wtns = [open(os.path.join(d, tag + "_%d.wtns" % i), "rb").read() for i in range(n_witness)]
    return zkey, wtns, dims


def config_block(args, world, dims):
    """`config` of the JSON line -- the SAME keys and values on both arms (the driver compares them)."""
    return dict(workload="nzcp_%s shape (BASELINE configs[1]), synthetic R1CS + satisfying witnesses" % args.shape,
                proofs_per_step_per_gpu=args.batch, provers_in_flight=args.provers,
                parallelism="batch-sharded x%d, no collective" % world,
                l2="inputs exceed L2: each proof streams the ~5.8 GB expanded proving key (window tables)", **dims)


def cpu_reference_proofs(zkey, wtns_list, n_proofs, threads=0):
    """Times the C restatement of snarkjs groth16.prove (oracle/c) on the host: -> (seconds per proof list, info)."""
    from oracle import cref
    times, stages = [], None
    for i in range(n_proofs):
        t = time.perf_counter()
        out = cref.prove(zkey, wtns_list[i % len(wtns_list)], R_FIXED, S_FIXED, threads=threads)
        times.append(time.perf_counter() - t)
        stages = out["stage_sec"]
        thr = out["threads"]
    return times, stages, thr, out["proof"]


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (port: oracle/c) on all host threads."""
    if rank != 0:
        return
    # the synthetic key + witnesses come from a separate process (cached on disk): nothing of nzcp_circom_b200 is
    # imported or mapped here, the timed region runs oracle/c alone
    zkey, wtns, dims = make_workload_files(args.shape, 2, 1000)
    assert "nzcp_circom_b200" not in sys.modules
    for _ in range(args.warmup):
        cpu_reference_proofs(zkey, wtns, 1)
    times, stages, thr, _ = cpu_reference_proofs(zkey, wtns, args.steps)
    total = sum(times)
    val = args.steps / total
    line = {
        "impl": "reference", "metric": "groth16_proofs_per_sec", "value": val, "unit": "proofs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u256 (Fr/Fq Montgomery, 4x64-bit limbs)", "data": "synthetic",
        "config": config_block(args, args.gpus, dims),
        "cpu_baseline": {"value": val, "unit": "proofs/s", "cores": thr, "kind": "port",
                         "sample": "%d full proofs (ONE per step, not proofs_per_step_per_gpu) of the same workload; C restatement of snarkjs "
                                   "groth16.prove, OpenMP over ffjavascript's task decomposition; NOT snarkjs itself "
                                   "(node absent)" % args.steps,
                         "stage_sec": stages},
        "e2e": {"value": val, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "p50_latency_ms": 1e3 * statistics.median(times), "gpu_launches": 0,
    }
    emit(line)


_REAL_STDOUT = None


def quiet_stdout():
    """Everything except the final JSON line goes to stderr: NCCL prints its version banner on fd 1, and the driver
    reads ONE JSON line from stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def dump_proofs(out_dir, proofs, prefix=""):
    """--dump-outputs: the B proofs of one step as float64 arrays pi_a (B, 2, 8), pi_b (B, 2, 2, 8) and pi_c (B, 2, 8), in
    the coordinate order of the proof bytes (include/nzcp_prover.h).  Each coordinate is a plain field element split into
    8 little-endian 32-bit limbs, which float64 holds exactly, so two builds can be compared bit for bit.  The inputs
    (synthetic key, witnesses, r, s) are seeded, so the same arguments give the same proofs."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    v = np.frombuffer(b"".join(proofs), dtype="<u4").reshape(len(proofs), 8, 8).astype(np.float64)
    for name, a in (("pi_a", v[:, 0:2]), ("pi_b", v[:, 2:6].reshape(-1, 2, 2, 8)), ("pi_c", v[:, 6:8])):
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.ascontiguousarray(a))


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=12, help="proofs per step per GPU")
    ap.add_argument("--shape", default="live", choices=sorted(SHAPES))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--provers", type=int, default=4, help="concurrent provers (host threads + stream sets) per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--latency-runs", type=int, default=50, help="lone proofs timed for p50_latency_ms")
    ap.add_argument("--no-extras", action="store_true", help="skip the BASELINE configs[2] / configs[4] records")
    ap.add_argument("--extras-proofs", type=int, default=1024, help="configs[2]: proofs in the sharded batch")
    ap.add_argument("--extras-msm-log", type=int, default=24, help="configs[4]: log2 points of the split G1 MSM")
    ap.add_argument("--tune", action="append", default=[], metavar="KNOB=VALUE",
                    help="library tuning knob (include/nzcp_prover.h nzcp_tuning_set), e.g. prover_rounds_h=0")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the proofs of the last timed step to DIR/pi_a.npy, pi_b.npy, pi_c.npy (see dump_proofs)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.warmup < 3:
        args.warmup = 3 if args.steps > 0 else args.warmup

    import torch
    import torch.distributed as dist
    from nzcp_circom_b200 import api

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; nzcp_circom_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B = args.batch
    for kv in args.tune:
        k, v = kv.split("=")
        api.tuning_set(k, int(v))
    zkey, wtns, dims = make_workload(args.shape, local, B, 1 + rank * B)
    zk = api.Zkey(zkey, device=local)
    pool = api.ProverPool(zk, args.provers)     # throughput-mode provers (what nzcp_prove_batch uses as well)
    pr = api.Prover(zk)                         # latency-mode prover: p50 of a lone proof, per-kernel timings
    m = zk.n_vars

    # host side: .wtns images in pinned memory (what the N-API shim hands over); device side: resident witnesses
    pinned = []
    for w in wtns:
        t = torch.empty(len(w), dtype=torch.uint8).pin_memory()
        t.numpy()[:] = memoryview(w)
        pinned.append(t)
    body_off = len(wtns[0]) - m * 32
    d_wit = [p[body_off:].to("cuda", non_blocking=False) for p in pinned]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def step_device():
        last["proofs"] = pool.prove_device_many(d_wit, r=R_FIXED, s=S_FIXED)

    lat = []
    host_wtns = [p.numpy() for p in pinned]

    def step_e2e(record):
        # the reference-facing C-ABI call: host .wtns images in, proofs out, the library's own prover threads, r and s
        # drawn from the OS CSPRNG per proof exactly as groth16.prove does (None = random)
        zk.prove_batch(host_wtns, None, None, n_provers=args.provers)

    # the same call from PAGEABLE host memory (what a Node Buffer or a Python bytes object is): the library copies it
    # through each prover's pinned staging buffer in chunks ("stage_mode" -1); mode 0 hands it to the driver instead
    import numpy as np
    pageable = [np.array(p.numpy(), copy=True) for p in pinned]

    def step_e2e_pageable():
        zk.prove_batch(pageable, None, None, n_provers=args.provers)

    def latency_run(count):
        # p50 per-proof latency: one proof at a time through the host-buffer call, nothing else in flight
        for i in range(count):
            t = time.perf_counter()
            pr.prove(host_wtns[i % B], r=R_FIXED, s=S_FIXED)
            lat.append(time.perf_counter() - t)

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    for _ in range(args.warmup):
        step_device()
    for _ in range(max(1, args.warmup // 3)):
        step_e2e(False)

    sampler = ClockSampler(local)
    sampler.start()
    l0 = pool.launch_count()          # per-prover counters, summed over the pool's provers
    ms_dev = timed(step_device, args.steps)
    launches = pool.launch_count() - l0
    if args.dump_outputs:
        dump_proofs(args.dump_outputs, [o["proof"] for o in last["proofs"]], "rank%d_" % rank if world > 1 else "")
    ms_e2e = timed(lambda: step_e2e(True), args.steps)
    clocks = sampler.stop()
    step_e2e_pageable()
    ms_e2e_pg = timed(step_e2e_pageable, args.steps)
    api.tuning_set("stage_mode", 0)
    step_e2e_pageable()
    ms_e2e_pg_direct = timed(step_e2e_pageable, args.steps)
    api.tuning_set("stage_mode", -1)
    latency_run(5)                      # warm the latency-mode prover (its own work buffers, first-touch of the staging path)
    del lat[:]
    latency_run(args.latency_runs)      # BASELINE configs[1]: one proof at a time, p50 over the runs
    lat_pinned = list(lat)
    del lat[:]
    for i in range(5 + args.latency_runs):          # lone-proof latency from pageable memory (first 5 = warm-up)
        t = time.perf_counter()
        pr.prove(pageable[i % B], r=R_FIXED, s=S_FIXED)
        lat.append(time.perf_counter() - t)
    lat_pageable, lat[:] = list(lat[5:]), lat_pinned

    # per-stage device times + the dominant kernel, from the library's own CUDA events (one extra proof, not timed above)
    dbg = pr.prove(host_wtns[0], r=R_FIXED, s=S_FIXED, debug=True, want_h=True)
    correct = None
    value = world * B * args.steps / (ms_dev / 1e3)
    e2e = world * B * args.steps / (ms_e2e / 1e3)
    n_dig = lambda npts: ((16 if npts >= (1 << 19) else 14 if npts >= (1 << 17) else 12) - 1 + 4) // 5  # noqa: E731
    d2h_per_proof = 3 * (n_dig(m) + 1) * 128 + (n_dig(m) + 1) * 256 + (n_dig(zk.domain_size) + 1) * 128 + 64
    if rank == 0:
        hbm, peak_src = peaks()
        line = {
            "metric": "groth16_proofs_per_sec", "value": value, "unit": "proofs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u256 (Fr/Fq Montgomery, 8x32-bit limbs, IMAD.WIDE carry chains)",
            "data": "synthetic",
            "config": config_block(args, world, dims),
            "e2e": {"value": e2e, "unit": "proofs/s", "h2d_bytes_per_step": B * m * 32,
                    "d2h_bytes_per_step": B * d2h_per_proof, "ms_per_step": ms_e2e / args.steps,
                    "d2h_note": "per proof: 4 G1 + 1 G2 MSM results as (digits + 1) XYZZ points each + 2 x 32 B of sort flags; "
                                "the 256-byte proof itself is assembled on the host",
                    "host_memory": "pinned (cudaHostAlloc) .wtns images, random r/s per proof",
                    "pageable": {"value": world * B * args.steps / (ms_e2e_pg / 1e3), "unit": "proofs/s",
                                 "value_driver_staged": world * B * args.steps / (ms_e2e_pg_direct / 1e3),
                                 "note": "same call with the .wtns images in ordinary pageable memory (a Node Buffer): `value` "
                                         "= through the prover's pinned staging buffer in 1 MiB chunks (default), "
                                         "`value_driver_staged` = cudaMemcpyAsync straight from the pageable buffer"}},
            "p50_latency_ms": 1e3 * statistics.median(lat) if lat else None,
            "latency_ms": {"runs": len(lat), "p50": 1e3 * statistics.median(lat), "min": 1e3 * min(lat), "max": 1e3 * max(lat),
                           "p90": 1e3 * sorted(lat)[int(0.9 * (len(lat) - 1))]} if lat else None,
            "p50_latency_ms_pageable": 1e3 * statistics.median(lat_pageable) if lat_pageable else None,
            "gpu_launches": launches, "clocks": clocks, "stage_ms": dbg["stage_ms"],
        }
        if args.tune:
            line["config"]["tune"] = args.tune
        line.update(roofline_block(dbg, zk, hbm, peak_src, zkey, dbg.pop("h", None)))
        line["roofline_step"] = step_roofline(dbg, zk, value / world, line["roofline"]["peak"] if "roofline" in line else None)
        line["modes"] = ("value / e2e: %d throughput-mode provers in flight (batched-affine pair rounds on); "
                                   "p50_latency_ms, stage_ms, roofline: one latency-mode prover, lone proofs" % args.provers)
        if not args.no_cpu_baseline and world == 1:     # the CPU leg runs at N = 1 only (rank 0's cores are shared at N > 1)
            times, stages, thr, cproof = cpu_reference_proofs(zkey, wtns, 1)
            correct = (cproof == dbg["proof"])
            line["cpu_baseline"] = {"value": 1.0 / times[0], "unit": "proofs/s", "cores": thr, "kind": "port",
                                    "sample": "1 full proof of the same workload (same zkey, witness 0); C restatement "
                                              "of snarkjs groth16.prove (oracle/c), OpenMP; NOT snarkjs itself",
                                    "stage_sec": stages}
            line["proof_matches_cpu_port"] = correct
        # one proof of the timed batch through the independent pairing check (CPU, a few seconds)
        try:
            from nzcp_circom_b200 import groth16
            out = pr.prove(host_wtns[0], r=None, s=None)
            vk = groth16.exportVerificationKey(zkey)
            line["proof_verifies"] = bool(groth16.verify(vk, groth16._public_signals(host_wtns[0], zk.n_public),
                                                         groth16.proof_from_bytes(out["proof"])))
        except Exception as e:  # noqa: BLE001
            line["proof_verifies"] = "error: %s" % e
    extra = None
    if not args.no_extras:
        try:
            pool.close()
            pr.close()
            zk.close()
            extra = run_extras(args, rank, world, local, timed, zkey if args.shape == "example" else None)
        except Exception as e:  # noqa: BLE001
            extra = {"error": repr(e)}
    if rank == 0:
        if extra is not None:
            line["extras"] = extra
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if correct is False:
        raise SystemExit("bench.py: GPU proof differs from the CPU port")


def run_extras(args, rank, world, local, timed, zkey_example):
    """The two other multi-GPU configurations of BASELINE.json, recorded as extra keys of the same JSON line so that the
    driver's --gpus N runs carry them: configs[2] (a fixed batch of nzcp_exampleTest-shape proofs sharded i mod N: STRONG
    scaling) and configs[4] (one 2^24-point G1 MSM split by point range, NCCL all-gather of the partial sums)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from nzcp_circom_b200 import api, parallel
    out = {}
    dev = torch.device("cuda", local)

    def agree(ok):
        """All ranks enter the timed (barrier-bracketed) part of a section, or none does: a rank that failed while
        preparing must not leave the others waiting in a collective."""
        if world == 1:
            return ok
        t = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    # ---- configs[2]
    n_total, n_distinct = args.extras_proofs, 16
    zk, err = None, None
    try:
        nc, npub, nfree = SHAPES["example"]
        sc = api.SynthCircuit(seed=0xC0FFEE, n_constraints=nc, n_public=npub, n_free=nfree)
        if zkey_example is None:
            zkey_example = sc.zkey(TOXIC, device=local)
        wt = []
        for i in range(n_distinct):
            w = sc.wtns(5000 + n_distinct * rank + i)
            t = torch.empty(len(w), dtype=torch.uint8).pin_memory()
            t.numpy()[:] = memoryview(w)
            wt.append(t.numpy())
        mine = parallel.shard_indices(n_total, rank, world)
        zk = api.Zkey(zkey_example, device=local)
        zk.prove_batch([wt[i % n_distinct] for i in range(2 * args.provers)], None, None, n_provers=args.provers)   # warm-up
    except Exception as e:  # noqa: BLE001
        err = repr(e)
    if agree(err is None):
        ms = timed(lambda: zk.prove_batch([wt[i % n_distinct] for i in mine], None, None, n_provers=args.provers), 1)
        out["config2_batch"] = {"workload": "nzcp_example shape, %d proofs sharded i mod %d (%d on rank 0; %d distinct witnesses "
                                            "per rank, cycled; random r/s)" % (n_total, world, len(mine), n_distinct),
                                "proofs": n_total, "n_gpus": world, "seconds": ms / 1e3, "proofs_per_s": n_total / (ms / 1e3),
                                "scaling": "strong", "path": "nzcp_prove_batch, pinned host .wtns in, proofs out"}
    else:
        out["config2_batch"] = {"error": err or "another rank failed"}
    if zk is not None:
        zk.close()
    del zkey_example
    # ---- configs[4]
    log_n = args.extras_msm_log
    n = 1 << log_n
    lo, hi = parallel.shard_range(n, rank, world)
    cnt = hi - lo
    plan, err, kms = None, None, []
    mine_t = torch.zeros(128, dtype=torch.uint8, device=dev)
    try:
        bases = api.synth_points(1000 + rank, cnt, device=local)
        sc_np = np.random.RandomState(rank).randint(0, 2 ** 32, size=(cnt, 8), dtype=np.uint64).astype(np.uint32)
        sc_np[:, 7] &= 0x1FFFFFFF
        plan = api.MsmPlan(bases, cnt, mode=1, device=local)
        kms.append(plan.run_partial(sc_np, mine_t))       # warm-up
    except Exception as e:  # noqa: BLE001
        err = repr(e)
    if agree(err is None):
        def run():
            kms.append(plan.run_partial(sc_np, mine_t))
            if world > 1:
                parts = [torch.empty_like(mine_t) for _ in range(world)]
                dist.all_gather(parts, mine_t)
            else:
                parts = [mine_t]
            run.result = api.msm_sum_partials(torch.cat(parts), world, device=local)
        run()
        ms = timed(run, 2) / 2
        k = torch.tensor([min(kms[1:])], device=dev)
        if world > 1:
            dist.all_reduce(k, op=dist.ReduceOp.MAX)
        out["config4_split_msm"] = {
            "workload": "one 2^%d-point G1 MSM, uniform 253-bit scalars, points range-partitioned over %d GPU(s)" % (log_n, world),
            "n_gpus": world, "points_per_gpu": cnt, "ms": ms, "kernel_ms_max_over_ranks": float(k.item()),
            "Mpoints_per_s": n / ms / 1e3, "plan_build_ms": plan.build_ms,
            "path": "per rank: variable-base plan (bases resident, no window table), scalars uploaded from pageable host memory "
                    "inside the timed region, partial sum left in HBM as one XYZZ point; one all-gather of 128 B per rank over "
                    "NCCL from and into device memory; nzcp_msm_sum_partials adds them on the GPU",
            "result_x_low64": int.from_bytes(run.result[:8], "little")}
    else:
        out["config4_split_msm"] = {"error": err or "another rank failed"}
    if plan is not None:
        plan.close()
    return out


def step_roofline(dbg, zk, proofs_per_s_per_gpu, peak_gmul):
    """The whole proving step against the integer-pipe roofline: CANONICAL field products per proof (SURVEY.md 8d: signed
    c = 16 Pippenger, 10 / 28 Fq products per G1 / G2 bucket addition, per-window bucket reduction 16 x 2 x 2^15 full
    additions at 14 / 40; NTT (n/2) log n per transform; one product per R1CS coefficient and per join element) times the
    measured proofs/s of ONE GPU, over the measured IMAD.WIDE peak / 128.  An implementation that executes fewer products
    (window tables: one bucket set instead of 16; batched-affine additions) is still scored against the canonical count,
    so the fraction may exceed the per-kernel ones."""
    if not peak_gmul:
        return None
    ew, eh = dbg["n_entries"]["witness"], dbg["n_entries"]["h"]
    n = zk.domain_size
    lg = n.bit_length() - 1
    acc = eh * 10 + 3 * ew * 10 + ew * 28
    red = 16 * 2 * (1 << 15) * (4 * 14 + 40)
    ntt = 6 * (n // 2) * lg + 3 * n
    rest = zk.n_coefs + n + 2 * n
    tot = acc + red + ntt + rest
    out = {"bound": "int32-mul-pipe", "unit": "GFqmul/s", "peak": peak_gmul,
           "canonical_fq_mul_per_proof": {"bucket_additions": acc, "per_window_bucket_reduction": red, "ntt": ntt,
                                          "r1cs_and_join": rest, "total": tot},
           "achieved": tot * proofs_per_s_per_gpu / 1e9, "frac": tot * proofs_per_s_per_gpu / 1e9 / peak_gmul,
           "achieved_without_reduction_term": (tot - red) * proofs_per_s_per_gpu / 1e9,
           "frac_without_reduction_term": (tot - red) * proofs_per_s_per_gpu / 1e9 / peak_gmul,
           "note": "per GPU, from `value`; measured pipe occupancy of the same step (ncu, sum of duration x fmaheavy-active "
                   "over one proof's launches / ms per proof): profiles/r02_pipe_summary.txt"}
    return out


def zkey_section(zkey, sid):
    """Payload of section `sid` of a .zkey image (binfileutils container)."""
    import struct
    mv = memoryview(zkey)
    pos = 12
    for _ in range(struct.unpack_from("<I", mv, 8)[0]):
        i, ln = struct.unpack_from("<IQ", mv, pos)
        pos += 12
        if i == sid:
            return mv[pos:pos + ln]
        pos += ln
    raise KeyError(sid)


def h_stage_alone(zkey, zk, h_scalars):
    """The H MSM's bucket accumulation with the GPU to itself: the same kernels the prover runs (fixed-base window table of
    zkey section 9, c = 16; 3 batched-affine pair rounds + XYZZ tail), on the h scalars of a real proof, timed by the
    library's CUDA events around the accumulation on its own stream.  Also the single XYZZ kernel (rounds off)."""
    from nzcp_circom_b200 import api
    n = zk.domain_size
    out = {}
    try:
        for rounds, key in ((3, "pair_rounds"), (0, "xyzz_only")):
            api.tuning_set("msm_rounds", rounds)
            with api.MsmPlan(zkey_section(zkey, 9), n, mode=0, window_bits=16, device=zk.device) as plan:
                plan.run(h_scalars)
                ts = []
                for _ in range(5):
                    plan.run(h_scalars)
                    ts.append(plan.accumulate_ms())
                out[key] = sum(ts) / len(ts)
    finally:
        api.tuning_set("msm_rounds", -1)
    return out


def roofline_block(dbg, zk, hbm, peak_src, zkey=None, h_scalars=None):
    """Roofline of the dominant kernel group -- from the library's live CUDA-event timings on the kernels' own stream.

    The dominant work of the step is the bucket accumulation of the H MSM.  In the default configuration that is three
    batched-affine pair rounds (msm_pair_forward / invert / backward_kernel<Fq>, 9 launches) followed by the XYZZ tail
    (msm_accumulate_pts_kernel<Fq>): ten launches timed as ONE unit.  It is scored against the integer multiply pipe, not
    HBM or the tensor cores (DESIGN.md "Rooflines"): algorithmic work = (non-zero signed digits of the h scalars) x 10 Fq
    products (the CANONICAL 8M + 2S mixed addition of SURVEY.md 8d; the pair rounds execute ~6.3 per addition, so the
    fraction credits that saving, as the survey prescribes).  Peak = the IMAD.WIDE.U32 issue rate measured on this GPU
    by nzcp_intpipe_bench / 128 products per Montgomery multiplication (MEASURED_PEAKS.json has no integer figure).
    `launch_ms` = the unit timed ALONE on the GPU (average of 5; what the ncu launch list shows as well); `in_proof_ms` =
    the same unit inside a lone proof, where it shares the SMs with the four witness MSMs.
    """
    from nzcp_circom_b200 import api
    out = {}
    ip = api.intpipe_bench(zk.device, 4096)
    peak_mul = ip["imad_wide_per_s"] / 128.0
    in_proof_ms = dbg["accumulate_ms"]["h"]
    ent = dbg["n_entries"]["h"]
    alone = h_stage_alone(zkey, zk, h_scalars) if zkey is not None and h_scalars is not None else {}
    acc_ms = alone.get("pair_rounds") or in_proof_ms
    if acc_ms > 0:
        ach = ent * 10 / (acc_ms * 1e-3)
        alg_bytes = ent * (64 + 4) + (ent / 64.0) * 128
        out["roofline"] = {
            "kernel": "H MSM bucket accumulation: 3 batched-affine pair rounds (msm_pair_forward/invert/backward_kernel<Fq>) + "
                      "XYZZ tail (msm_accumulate_pts_kernel<Fq>), 10 launches timed as one unit",
            "bound": "int32-mul-pipe",
            "achieved": ach / 1e9, "peak": peak_mul / 1e9, "unit": "GFqmul/s", "frac": ach / peak_mul,
            "launch_ms": acc_ms, "in_proof_ms": in_proof_ms, "algorithmic_fq_mul": ent * 10,
            "traffic": 7.86e9 * ent / 16776933.0,
            "traffic_source": "recorded, not live: dram__bytes_read.sum + dram__bytes_write.sum of the unit's ten launches in the "
                              "committed ncu launch list profiles/r02_launches_pipe_final.csv (6.54 GB read + 1.32 GB written at "
                              "16 776 933 entries), scaled by this run's entry count; algorithmic bytes: 1.14 GB (68 B/entry) -- "
                              "an affine addition reads each operand twice and the rounds write their sums back",
            "peak_source": "measured here: %.2f T IMAD.WIDE.U32/s (32 per SM per clock, half the 32-bit IMAD rate) / 128 "
                           "32x32 products per 254-bit Montgomery mul; a register-only Fq mul microbenchmark reaches "
                           "%.1f GFqmul/s" % (ip["imad_wide_per_s"] / 1e12, ip["fq_mul_per_s"] / 1e9),
            "hbm_view": {"bound": "hbm", "achieved": 7.86e9 * ent / 16776933.0 / (acc_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                         "frac": 7.86e9 * ent / 16776933.0 / (acc_ms * 1e-3) / 1e9 / hbm,
                         "note": "recorded DRAM traffic of the unit / its live duration; algorithmic bytes (%.2f GB) would give %.0f GB/s; "
                                 "peak %s" % (alg_bytes / 1e9, alg_bytes / (acc_ms * 1e-3) / 1e9, peak_src)},
        }
        if alone.get("xyzz_only"):
            x = alone["xyzz_only"]
            out["roofline"]["xyzz_kernel"] = {
                "kernel": "msm_accumulate_kernel<Fq> (the single-kernel alternative: XYZZ mixed additions only, pair rounds off)",
                "launch_ms": x, "achieved": ent * 10 / (x * 1e-3) / 1e9, "frac": ent * 10 / (x * 1e-3) / peak_mul,
                "note": "executes the canonical 10 products per addition; fmaheavy 85 % active (profiles/r02_ncu_ntt_accumulate_full.md)"}
    # the NTT pipeline: 3 polynomials x (iNTT + NTT) = 6 transforms x 2 x 32 x n bytes
    n = zk.domain_size
    ntt_ms = dbg["stage_ms"].get("ntt_join")
    if ntt_ms:
        alg = 6 * 2 * 32 * n
        lg = n.bit_length() - 1
        muls = 6 * (n // 2) * lg + 4 * n + 2 * n
        # the same three kernels with the GPU to themselves (nzcp_ntt_coset, batch 3, library CUDA events; no join)
        alone_ms = None
        try:
            import numpy as np
            buf = np.random.default_rng(1).integers(0, 256, size=3 * n * 32, dtype=np.uint8)
            buf[31::32] &= 0x1f                               # canonical (< r); the kernels' work is data-independent
            api.ntt_coset(buf, lg, batch=3, device=zk.device)
            alone_ms = min(api.ntt_coset(buf, lg, batch=3, device=zk.device) for _ in range(3))
        except Exception as e:  # noqa: BLE001
            print("standalone NTT timing failed: %s" % e, file=sys.stderr)
        out["roofline_ntt"] = {"bound": "hbm", "achieved": alg / (ntt_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                               "frac": alg / (ntt_ms * 1e-3) / 1e9 / hbm, "traffic": None, "stage_ms": ntt_ms,
                               "int_pipe_view": {"achieved": muls / (ntt_ms * 1e-3) / 1e9, "peak": peak_mul / 1e9,
                                                 "unit": "GFrmul/s", "frac": muls / (ntt_ms * 1e-3) / peak_mul},
                               "note": "H pipeline (3x iNTT+scale+NTT, join) as one stage, other streams running; "
                                       "algorithmic 384*n bytes; peak %s" % peak_src}
        if alone_ms:
            m6 = 6 * (n // 2) * lg + 3 * n
            out["roofline_ntt"]["alone"] = {
                "ms": alone_ms, "hbm_gbs": alg / (alone_ms * 1e-3) / 1e9, "hbm_frac": alg / (alone_ms * 1e-3) / 1e9 / hbm,
                "gfrmul_s": m6 / (alone_ms * 1e-3) / 1e9, "int_pipe_frac": m6 / (alone_ms * 1e-3) / peak_mul,
                "note": "the 3 NTT kernels on an otherwise idle GPU (nzcp_ntt_coset, batch 3): %d Fr products; the "
                        "pipeline is bound by the multiplier, HBM floor %.0f us" % (m6, alg / hbm / 1e3)}
    out["msm"] = {"accumulate_ms": dbg["accumulate_ms"], "sort_ms": dbg["sort_ms"], "n_entries": dbg["n_entries"],
                  "total_ms": dbg["total_ms"]}
    return out


if __name__ == "__main__":
    main()
