#!/usr/bin/env python
"""bench.py -- PLONK proofs/s at 2^20 gates on B200 (BASELINE.json metric), with the roofline of the
dominant kernel and the reference's CPU path timed beside it.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port), rank 0
  python bench.py ... --dump-outputs DIR                   # also write the proofs of the last timed step

A "step" is one full proof (Prover.prove rounds 1-5, 9 KZG commitments) of a synthetic 2^20-gate circuit
(plonkathon_b200/synthetic.py, seeded) under a structured test SRS generated on the device.
  value : proofs/s, wire values already resident in HBM (pb200_prover_prove_device), device-timed.
  e2e   : proofs/s through the reference-facing C ABI call with HOST buffers (pb200_prover_prove): the three
          wire-value vectors are copied host->device from pinned memory and the 768-byte proof is read back
          inside the timed region, every step.
N > 1: one process per GPU (torchrun).  `value` / `e2e`: every rank proves its own copy of the circuit (proofs are
independent units: no data-path collective); value = N*K*lanes proofs / max-over-ranks time ("weak").  The same run
then proves ONE instance across all ranks (plonkathon_b200.parallel.ShardedProver: coset slices, slab-sharded
transforms, bucket-sharded commitments, the library's own NCCL allgathers at the joins), checks it byte for byte
against the single-GPU proof, times it, and does the same for the sharded NTT and the sharded commitment as
operators: `one_proof_sharded`, `sharded_proof_matches_single`, `slab_ntt_matches_single`,
`sharded_msm_matches_single` and `components.sharded_across_N_gpus` in the JSON line."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
from concurrent.futures import ThreadPoolExecutor
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from, which may be read-only

TAU = 0x1234567890ABCDEF1234567890ABCDEF1234567890ABCDEF  # fixed toxic-waste value of the synthetic test SRS


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log-n", type=int, default=20)
    ap.add_argument("--seed", type=int, default=20260924, help="seed of the synthetic circuit (7 with --log-n 22 is the "
                    "circuit of tests/golden/proof_2p22.json)")
    ap.add_argument("--cpu-log-n", type=int, default=8, help="size of the bounded CPU sample (2^k gates)")
    ap.add_argument("--cpu-fit", default="5,7,9", help="reference arm: sample sizes (log2 gates) of the cost fit")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-procs", type=int, default=0,
                    help="reference arm: worker processes proving independent instances side by side "
                         "(0 = one per host core)")
    ap.add_argument("--no-verify", action="store_true", help="skip verifying the benchmarked proof (untimed)")
    ap.add_argument("--inflight", type=int, default=2,
                    help="proofs in flight per GPU: independent provers (own stream + scratch, shared SRS), one host "
                         "thread each; a step is one batch of this many proofs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float64), for comparing builds")
    return ap.parse_args()


def dump_outputs(path, proofs):
    """proofs: the 768-byte proof of every lane (Proof.to_bytes order: 24 big-endian 256-bit words).  Written as
    proof.npy, shape (lanes, 24, 8): each word as eight 32-bit limbs, least significant first (exact in float64)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    words = np.frombuffer(b"".join(proofs), dtype=np.uint8).reshape(len(proofs), 24, 32)[:, :, ::-1]
    limbs = np.ascontiguousarray(words).view("<u4")
    np.save(os.path.join(path, "proof.npy"), limbs.astype(np.float64))


# ----------------------------------------------------------------------------------------------
# the reference's CPU path (oracle port of poly.py / curve.py / prover.py), bounded sample
# ----------------------------------------------------------------------------------------------
def cpu_sample(log_n, steps=1):
    """Times oracle/plonk_oracle.py's Prover.prove (the reference's algorithm: recursive Python FFT, the
    bit-sliced multisubset ec_lincomb with one modular inversion per affine add) on a 2^log_n-gate
    instance of the same synthetic circuit family, single thread (the reference is single-threaded)."""
    from oracle import plonk_oracle as O
    from plonkathon_b200 import synthetic as syn
    c = syn.build_circuit(log_n, seed=20260924, n_public=2)
    S1, S2, S3 = syn.permutation_polys(c.wire_L, c.wire_R, c.wire_O, c.group_order, c.n_constraints)
    pk = O.Preprocessed(c.group_order, c.QM, c.QL, c.QR, c.QO, c.QC, S1, S2, S3)
    n = c.group_order
    pts, cur = [], O.G1  # [tau^i]G by repeated scalar multiplication of the previous power
    for _ in range(n):
        pts.append(cur)
        cur = O.g1_multiply(cur, TAU)
    setup = O.Setup(pts, None)
    A, B, C = c.wires_values()
    prover = O.Prover(setup, pk, check=True)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        prover.prove(A, B, C, c.public_values())
        times.append(time.perf_counter() - t0)
    return n, times


def metric_name(log_n):
    return "plonk_proofs_per_s_2^%d_gates" % log_n


def usable_cores():
    """host threads this process may actually run on: the scheduler affinity mask, capped by the cgroup CPU quota"""
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    cores = min(cores, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    cores = min(cores, max(1, quota // period))
        except Exception:
            pass
    return max(1, cores)


def _reference_worker(job):
    """one host process of the reference arm: per step one proof at every sample size (module level: spawn-safe);
    returns {log_n: [seconds per proof]}"""
    sizes, warmup, steps = job
    if warmup > 0:
        cpu_sample(min(sizes), 1)
    out = {k: [] for k in sizes}
    for _ in range(max(1, steps)):
        for k in sizes:
            out[k].append(cpu_sample(k, 1)[1][0])
    return out


def fit_cost(points):
    """least-squares t(n) = a n + b n log2 n (a, b >= 0) through [(n, seconds)]: the commitments are linear in n, the
    transforms n log n"""
    import numpy as np
    A = np.array([[n, n * np.log2(n)] for n, _ in points], dtype=float)
    y = np.array([t for _, t in points], dtype=float)
    w = 1.0 / y  # relative errors
    sol, *_ = np.linalg.lstsq(A * w[:, None], y * w, rcond=None)
    a, b = float(sol[0]), float(sol[1])
    if a < 0 or b < 0:  # fall back to the one-parameter fits
        a1 = float(np.sum(w * w * A[:, 0] * y) / np.sum(w * w * A[:, 0] ** 2))
        b1 = float(np.sum(w * w * A[:, 1] * y) / np.sum(w * w * A[:, 1] ** 2))
        a, b = (a1, 0.0) if b < 0 else (0.0, b1)
    return a, b


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # The reference is single-threaded Python, but proofs are independent, so "all the host threads it can use" is
    # one process per USABLE core (affinity mask and cgroup quota, not os.cpu_count()), each proving its own
    # instances (the CPU counterpart of replicas / proofs in flight).
    import multiprocessing as mp
    cores = usable_cores()
    procs = min(256, args.cpu_procs if args.cpu_procs > 0 else cores)
    sizes = sorted({int(x) for x in args.cpu_fit.split(",") if x})
    k8 = sizes[len(sizes) // 2]  # the middle sample size: one process alone against all workers running
    t_single = cpu_sample(k8, 1)[1][0] if procs > 1 else None
    job = (sizes, 1 if args.warmup > 0 else 0, args.steps)
    per_proc = None
    if procs > 1:
        try:
            with mp.get_context("spawn").Pool(procs) as pool:
                per_proc = pool.map(_reference_worker, [job] * procs)
        except Exception as e:  # e.g. a sandbox without process spawning: still report the single-process number
            print("reference arm: process pool failed (%r), falling back to one process" % (e,), file=sys.stderr)
            procs = 1
    if per_proc is None:
        per_proc = [_reference_worker(job)]
    # seconds per proof inside one worker at every sample size, all workers running
    mean_t = {k: statistics.mean(x for w in per_proc for x in w[k]) for k in sizes}
    a, b = fit_cost([(1 << k, mean_t[k]) for k in sizes])
    n_full = 1 << args.log_n
    t_full = a * n_full + b * n_full * args.log_n          # seconds per 2^log_n-gate proof in one worker
    value = procs / t_full                                  # all workers
    slowdown = (mean_t[k8] / t_single) if t_single else 1.0
    sample = ("%d worker processes on %d usable host cores (os.cpu_count() = %s), each running the oracle port of "
              "Prover.prove on 2^{%s}-gate instances of the same synthetic circuit family: %s s per proof and worker; "
              "cost model t(n) = a n + b n log2 n fitted to those points (a = %.3e, b = %.3e) and EXTRAPOLATED to "
              "2^%d gates (%.0f s per proof and worker); one worker alone takes %s s at 2^%d gates, i.e. a slowdown "
              "of %.2fx with all workers running"
              % (procs, cores, os.cpu_count(), ",".join(str(k) for k in sizes),
                 ", ".join("%.2f" % mean_t[k] for k in sizes), a, b, args.log_n, t_full,
                 ("%.2f" % t_single) if t_single else "n/a", k8, slowdown))
    line = {
        "impl": "reference", "metric": metric_name(args.log_n), "value": value, "unit": "proofs/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / value, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u256 (BN254 Fr/Fq integers)", "data": "synthetic",
        "extrapolated": True,
        "config": {"workload": "PLONK prove (rounds 1-5, 9 KZG commits), synthetic 2^%d-gate circuit, structured "
                               "test SRS [tau^i]G of 2^%d powers" % (args.log_n, args.log_n),
                   "log_n": args.log_n, "seed": args.seed, "cpu_sample_log_n": sizes},
        "cpu_baseline": {"value": value, "unit": "proofs/s", "cores": procs, "kind": "port", "sample": sample,
                         "usable_cores": cores, "os_cpu_count": os.cpu_count(), "per_worker_slowdown": slowdown,
                         "seconds_per_proof_per_worker": {str(k): mean_t[k] for k in sizes},
                         "fit": {"a_s_per_gate": a, "b_s_per_gate_log_gate": b, "extrapolated_s_per_proof": t_full}},
        "e2e": {"value": value, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock / power / throttle reasons of this rank's GPU sampled during the timed region
    (B200_PROFILING.md).  In-process NVML (no fork, sub-millisecond queries: spawning nvidia-smi from every
    rank stalls CUDA calls on a busy 8-GPU box); falls back to nvidia-smi when pynvml is missing."""
    SMI_Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index = index
        self.period = period
        self.samples = []  # (sm_mhz, sm_max_mhz, power_w, reasons set)
        self.stop_flag = threading.Event()
        self.recording = threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self._sample_nvml()  # the first queries initialise NVML state lazily and can stall CUDA calls for
            self._sample_nvml()  # ~100 ms: take that hit here, long before any timed region
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
        pw = n.nvmlDeviceGetPowerUsage(self.h) / 1000.0
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        return sm, self.sm_max, pw, {name for name, bit in self.BITS if mask & bit}

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.SMI_Q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
        f = [x.strip() for x in out.stdout.strip().split(",")]
        reasons = {name for (name, _), v in zip(self.BITS, f[3:7]) if v.lower().startswith("active")}
        return float(f[0]), float(f[1]), float(f[2]), reasons

    def run(self):
        while not self.stop_flag.is_set():
            if self.recording.is_set():
                try:
                    self.samples.append(self._sample_nvml() if self.nvml else self._sample_smi())
                except Exception:
                    pass
            self.stop_flag.wait(self.period if self.nvml else 0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        reasons = set()
        for s in self.samples:
            reasons |= s[3]
        return {"sm_mhz": statistics.median(s[0] for s in self.samples), "sm_max_mhz": self.samples[0][1],
                "power_w_max": max(s[2] for s in self.samples), "samples": len(self.samples),
                "source": "nvml" if self.nvml else "nvidia-smi", "reasons": sorted(reasons)}


def measured_peaks():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def b200_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import plonkathon_b200 as pb
    from plonkathon_b200 import _lib, synthetic as syn

    L = _lib.lib()
    ctx = _lib.Context(local)
    log_n = args.log_n
    n = 1 << log_n
    t0 = time.time()
    setup = pb.Setup.generate(TAU, n, ctx=ctx)
    circ = syn.build_circuit(log_n, seed=args.seed, n_public=2)
    pk, A, B, C, public = syn.circuit_arrays(circ)
    K = max(1, args.inflight)
    vp = ctypes.c_void_p
    pub = np.frombuffer(b"".join(int(x).to_bytes(32, "little") for x in public), dtype=np.uint8).reshape(-1, 32).copy()
    # one lane per proof in flight: context (stream, scratch, NTT plans), prover, pinned host buffers (e2e) and
    # device-resident copies (value) of the wire values, proof buffer.  Lane 0 uses the setup's own context.
    lanes = []
    for k in range(K):
        lctx = ctx if k == 0 else _lib.Context(local)
        h3 = tuple(torch.from_numpy(x if k == 0 else x.copy()).pin_memory() for x in (A, B, C))
        lanes.append({"ctx": lctx, "prover": pb.Prover.from_arrays(setup, n, pk, ctx=lctx), "h": h3,
                      "d": tuple(x.cuda(non_blocking=False) for x in h3), "proof": ctypes.create_string_buffer(768)})
    setup_s = time.time() - t0
    prover, proof = lanes[0]["prover"], lanes[0]["proof"]
    hA, hB, hC = lanes[0]["h"]
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local))
    pool = ThreadPoolExecutor(K) if K > 1 else None

    def prove_device(lane=lanes[0]):
        _lib.check(L.pb200_prover_prove_device(lane["prover"]._h, *[vp(t.data_ptr()) for t in lane["d"]],
                                               pub.ctypes.data_as(vp), pub.shape[0], lane["proof"]))

    def prove_host(lane=lanes[0]):
        _lib.check(L.pb200_prover_prove(lane["prover"]._h, *[vp(t.data_ptr()) for t in lane["h"]],
                                        pub.ctypes.data_as(vp), pub.shape[0], lane["proof"]))

    def run_lanes(fn, steps, active=None):
        """every active lane proves `steps` times, all lanes concurrently; returns per-lane host milliseconds"""
        def worker(lane):
            t_lane = time.perf_counter()
            marks = []
            for _ in range(steps):
                fn(lane)
                marks.append(time.perf_counter())
            if os.environ.get("PB200_BENCH_STEP_TIMES"):  # debugging aid: host clock of every step
                print("    steps (ms):", [round((b - a) * 1e3, 1) for a, b in zip([t_lane] + marks[:-1], marks)], file=sys.stderr)
            return round((time.perf_counter() - t_lane) * 1e3, 1)
        active = lanes if active is None else active
        return [worker(active[0])] if len(active) == 1 else list(pool.map(worker, active))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, active=None, name=None):
        """device time of `steps` steps; a step = one proof on every active lane.  All lane streams are idle when
        the first event is recorded and again when the second one is (the prove calls return finished proofs)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        per_lane = run_lanes(fn, steps, active)
        e1.record(stream)
        e1.synchronize()
        barrier()
        ms = e0.elapsed_time(e1)
        print("[rank %d] %s: %.2f ms for %d steps x %d lanes (host clock per lane: %s)"
              % (rank, name or getattr(fn, "__name__", "fn"), ms, steps, len(active or lanes), per_lane), file=sys.stderr)
        if world > 1:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    sampler = ClockSampler(local)
    if os.environ.get("PB200_BENCH_NO_SAMPLER"):  # debugging aid: leaves "clocks" unavailable
        sampler.nvml, sampler._sample_smi = None, (lambda: (_ for _ in ()).throw(RuntimeError("disabled")))
    sampler.start()  # started (and NVML initialised) before the warm-up; records only inside the timed regions
    if world > 1:
        # the first collectives on torch's communicator initialise NCCL lazily (channels, proxy threads, buffer
        # registration) and were seen to stall one rank's CUDA calls for ~150 ms afterwards: take that here, not in a
        # timed region
        warm = torch.ones(1, device="cuda")
        dist.all_reduce(warm, op=dist.ReduceOp.MAX)
        barrier()
    run_lanes(prove_device, args.warmup)
    barrier()
    # sampling is already running during this last untimed step: nothing about it is new when the timed region starts
    sampler.recording.set()
    run_lanes(prove_host, 1)
    ref_proof = proof.raw  # the device-buffer path is checked against it after its timed steps (last_proofs)
    assert all(lane["proof"].raw == ref_proof for lane in lanes), "lanes disagree"
    torch.cuda.synchronize()
    sampler.samples.clear()
    launches0 = sum(lane["ctx"].launches for lane in lanes)
    ms_dev = timed(prove_device, args.steps)
    launches = sum(lane["ctx"].launches for lane in lanes) - launches0
    last_proofs = [lane["proof"].raw for lane in lanes]  # the last timed step's results (--dump-outputs)
    ms_e2e = timed(prove_host, args.steps)
    # The device-resident path does strictly less than the host-buffer path.  A reading more than 25 % ABOVE it means the
    # first timed region was hit by a one-off stall (seen once on rank 0 of an 8-GPU run: 369 ms against 219 ms on the
    # other seven ranks and in the e2e region right after): re-measure it once, as for a throttled run, and say so.
    remeasured = None
    if ms_dev > 1.25 * ms_e2e:
        remeasured = {"first_reading_ms": ms_dev, "reason": "device-resident region slower than the host-buffer region"}
        launches0 = sum(lane["ctx"].launches for lane in lanes)
        ms_dev = timed(prove_device, args.steps, name="prove_device (re-measured)")
        launches = sum(lane["ctx"].launches for lane in lanes) - launches0
        last_proofs = [lane["proof"].raw for lane in lanes]
    sampler.recording.clear()
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    assert all(lane["proof"].raw == ref_proof for lane in lanes)
    assert all(p == ref_proof for p in last_proofs), "host- and device-buffer paths disagree"
    # per-kernel durations for the roofline: the same `steps` proofs on lane 0 alone with the library's event pairs
    # around every accumulation launch and NTT pass (alone, so that a duration is the kernel's own and not a share of
    # an SM array it divides with the other lane's kernels)
    _lib.check(L.pb200_ctx_timing(ctx.handle, 1))
    ms_solo = timed(prove_device, args.steps, active=lanes[:1], name="prove_device (one lane, kernel timing)")
    tot, cnt = ctypes.c_double(), ctypes.c_uint64()
    _lib.check(L.pb200_ctx_timing_read(ctx.handle, 0, ctypes.byref(tot), ctypes.byref(cnt)))
    acc_ms, acc_cnt = tot.value, cnt.value
    _lib.check(L.pb200_ctx_timing_read(ctx.handle, 1, ctypes.byref(tot), ctypes.byref(cnt)))
    ntt_ms, ntt_cnt = tot.value, cnt.value
    _lib.check(L.pb200_ctx_timing_read(ctx.handle, 2, ctypes.byref(tot), ctypes.byref(cnt)))
    sort_ms = tot.value
    _lib.check(L.pb200_ctx_timing_read(ctx.handle, 3, ctypes.byref(tot), ctypes.byref(cnt)))
    red_ms = tot.value
    _lib.check(L.pb200_ctx_timing(ctx.handle, 0))
    print("[rank %d] per proof (one lane): %.2f ms; MSM sort %.2f, accumulate %.2f, reduce %.2f; NTT passes (main stream) %.2f"
          % (rank, ms_solo / args.steps, sort_ms / args.steps, acc_ms / args.steps, red_ms / args.steps, ntt_ms / args.steps),
          file=sys.stderr)

    # outside every timed region: byte-for-byte against the oracle's golden proof of this very circuit, when the
    # fixture for this size and seed exists (tests/golden/make_proof_2p20.py; reading a JSON file is not running the
    # oracle).  Reported, not asserted: the parity gate is the test-suite, the bench only says what it saw.
    golden_match = None
    gpath = os.path.join(ROOT, "tests", "golden", "proof_2p%d_seed%d.json" % (log_n, args.seed))
    if args.seed == 7:  # the circuits of tests/test_gpu_parity.py's golden proofs
        gpath = os.path.join(ROOT, "tests", "golden", "proof_2p%d.json" % log_n)
    if os.path.exists(gpath):
        try:
            golden_match = bool(json.load(open(gpath))["proof_hex"] == ref_proof.hex())
        except Exception:
            golden_match = None

    # ---- N > 1: ONE proof across all the GPUs (north_star's sharded path), checked and timed where the driver's
    # scaling run sees it: coset slices + slab-sharded interpolation + bucket-sharded commitments, the library's own
    # NCCL allgathers at the joins (plonkathon_b200/parallel.py, csrc/prover.cu with world > 1)
    shard = None
    if world > 1:
        from plonkathon_b200 import parallel
        sp = parallel.ShardedProver.from_arrays(setup, n, pk)  # every rank holds the same circuit instance
        pA, pB, pC = hA.numpy(), hB.numpy(), hC.numpy()  # views of the pinned buffers
        proof_ok = sp.prove_arrays(pA, pB, pC, public) == ref_proof
        c0 = parallel.comm_info(ctx)
        barrier()
        t0 = time.perf_counter()
        shard_ms = timed(lambda lane: sp.prove_arrays(pA, pB, pC, public), args.steps, active=lanes[:1],
                         name="one proof sharded across the GPUs") / args.steps
        shard_wall_ms = (time.perf_counter() - t0) * 1e3 / args.steps
        c1 = parallel.comm_info(ctx)
        # the two sharded operators of BASELINE.json's metric, against their single-GPU results, then timed
        xs = torch.randint(0, 2 ** 31 - 1, (n, 8), dtype=torch.int32, device="cuda",
                           generator=torch.Generator(device="cuda").manual_seed(1234))  # same vector on every rank
        xs[:, 7] &= 0x0FFFFFFF
        ys, yf = torch.empty_like(xs), torch.empty_like(xs)
        _lib.check(L.pb200_fr_ntt(ctx.handle, vp(xs.data_ptr()), vp(yf.data_ptr()), log_n, 0))
        parallel.sharded_ntt(xs, log_n, False, ctx=ctx, out=ys)
        ctx.sync()
        ntt_ok = bool(torch.equal(ys, yf))
        _lib.check(L.pb200_fr_ntt(ctx.handle, vp(xs.data_ptr()), vp(yf.data_ptr()), log_n, 1))
        parallel.sharded_ntt(xs, log_n, True, ctx=ctx, out=ys)
        ctx.sync()
        ntt_ok = ntt_ok and bool(torch.equal(ys, yf))
        o1, i1 = ctypes.create_string_buffer(64), ctypes.c_int()
        _lib.check(L.pb200_srs_commit_coeffs(ctx.handle, setup._srs, vp(xs.data_ptr()), n, 0, o1, ctypes.byref(i1)))
        one = (int.from_bytes(o1.raw[:32], "little"), int.from_bytes(o1.raw[32:], "little"))
        msm_ok = parallel.sharded_commit(setup, xs, n) == one
        ok_all = torch.tensor([int(proof_ok), int(ntt_ok), int(msm_ok)], device="cuda")
        dist.all_reduce(ok_all, op=dist.ReduceOp.MIN)  # true only if true on every rank
        proof_ok, ntt_ok, msm_ok = (bool(v) for v in ok_all.tolist())

        def ntt_sh(lane=None):
            parallel.sharded_ntt(xs, log_n, False, ctx=ctx, out=ys)
            parallel.sharded_ntt(ys, log_n, True, ctx=ctx, out=ys)
        ntt_sh()
        ntt_sh_ms = timed(ntt_sh, 5, active=lanes[:1], name="sharded NTT forward + inverse") / 5
        msm_sh = lambda lane=None: parallel.sharded_commit(setup, xs, n)  # noqa: E731
        msm_sh()
        msm_sh_ms = timed(msm_sh, 5, active=lanes[:1], name="sharded commitment") / 5
        shard = {"ms": shard_ms, "ms_wall_clock": shard_wall_ms, "proof_ok": proof_ok, "ntt_ok": ntt_ok,
                 "msm_ok": msm_ok, "ntt_pair_ms": ntt_sh_ms, "msm_ms": msm_sh_ms,
                 "collectives_per_proof": (c1[2] - c0[2]) / args.steps,
                 "bytes_received_per_proof": (c1[3] - c0[3]) / args.steps}
        del sp

    # component micro-configs (BASELINE.json configs[1], configs[2], configs[3]), device-timed, rank 0 only
    comp = {}
    if rank == 0:
        hbm_peak = measured_peaks()[0]
        x = torch.randint(0, 2 ** 31 - 1, (n, 8), dtype=torch.int32, device="cuda")
        x[:, 7] &= 0x0FFFFFFF
        y = torch.empty_like(x)

        def ntt_component(k):
            m = 1 << k
            xx = x if m == n else torch.randint(0, 2 ** 31 - 1, (m, 8), dtype=torch.int32, device="cuda")
            yy = y if m == n else torch.empty_like(xx)

            def pair():
                _lib.check(L.pb200_fr_ntt(ctx.handle, vp(xx.data_ptr()), vp(yy.data_ptr()), k, 0))
                _lib.check(L.pb200_fr_ntt(ctx.handle, vp(yy.data_ptr()), vp(yy.data_ptr()), k, 1))
            pair()
            ms = timed_local(torch, stream, pair, 5) / 5
            gbs = 128.0 * m / (ms * 1e-3) / 1e9  # 64 B per element per transform, two transforms
            return {"ms": ms, "elems_per_s": 2 * m / (ms * 1e-3),
                    "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                                 "modmul_ceiling_frac": (2 * (m / 2 * k + m) / (ms * 1e-3)) / 65.4e9}}
        comp["fr_ntt_fwd_plus_inv_2^%d" % log_n] = ntt_component(log_n)
        if log_n + 2 <= 24:
            comp["fr_ntt_fwd_plus_inv_2^%d" % (log_n + 2)] = ntt_component(log_n + 2)
        ident = ctypes.c_int()
        out = ctypes.create_string_buffer(64)

        def commit():
            _lib.check(L.pb200_srs_commit_coeffs(ctx.handle, setup._srs, vp(x.data_ptr()), n, 0, out, ctypes.byref(ident)))
        commit()
        ms = timed_local(torch, stream, commit, 5) / 5
        gbs = 96.0 * n / (ms * 1e-3) / 1e9  # 64 B point + 32 B scalar
        comp["g1_msm_fixed_base_2^%d" % log_n] = {
            "ms": ms, "points_per_s": n / (ms * 1e-3),
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak}}
        # curve.py:38 ec_lincomb as a drop-in: arbitrary (variable) bases, no precomputed table -- the SRS points themselves
        pts_dev = torch.from_numpy(setup.export_points_array(0, n)).cuda() if hasattr(setup, "export_points_array") else None
        if pts_dev is not None:
            def lincomb():
                _lib.check(L.pb200_g1_msm(ctx.handle, vp(pts_dev.data_ptr()), vp(x.data_ptr()), n, out, ctypes.byref(ident)))
            lincomb()
            ms = timed_local(torch, stream, lincomb, 3) / 3
            gbs = 96.0 * n / (ms * 1e-3) / 1e9
            comp["g1_msm_variable_base_2^%d" % log_n] = {
                "ms": ms, "points_per_s": n / (ms * 1e-3),
                "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak}}
            del pts_dev
        # BASELINE.json configs[3]: a full Prover.prove at the size of test/mini_poseidon (n = 1024), host buffers
        small = syn.build_circuit(10, seed=args.seed, n_public=2)
        spk, sA, sB, sC, spub = syn.circuit_arrays(small)
        ssetup = pb.Setup.generate(TAU, 1 << 10, ctx=ctx)  # its own 2^10-power SRS (window table sized for 1024 points)
        sprover = pb.Prover.from_arrays(ssetup, 1 << 10, spk)
        sprover.prove_arrays(sA, sB, sC, spub)
        ms = timed_local(torch, stream, lambda: sprover.prove_arrays(sA, sB, sC, spub), 10) / 10
        comp["prove_2^10_gates_latency"] = {"ms": ms, "proofs_per_s": 1e3 / ms,
                                            "note": "one proof at a time, host buffers, rounds 1-5 + transcript"}
        del sprover, ssetup
        if shard is not None:
            one_ms = ms_solo / args.steps
            base_ntt = comp["fr_ntt_fwd_plus_inv_2^%d" % log_n]["ms"]
            base_msm = comp["g1_msm_fixed_base_2^%d" % log_n]["ms"]
            comp["sharded_across_%d_gpus" % world] = {
                "one_proof_ms": shard["ms"], "one_proof_ms_wall_clock": shard["ms_wall_clock"],
                "one_proof_speedup_vs_1_gpu": one_ms / shard["ms"], "one_proof_efficiency": one_ms / shard["ms"] / world,
                "fr_ntt_fwd_plus_inv_ms": shard["ntt_pair_ms"], "fr_ntt_elems_per_s": 2 * n / (shard["ntt_pair_ms"] * 1e-3),
                "fr_ntt_speedup_vs_1_gpu": base_ntt / shard["ntt_pair_ms"],
                "g1_msm_ms": shard["msm_ms"], "g1_msm_points_per_s": n / (shard["msm_ms"] * 1e-3),
                "g1_msm_speedup_vs_1_gpu": base_msm / shard["msm_ms"],
                "collectives_per_proof": shard["collectives_per_proof"],
                "nvlink_bytes_received_per_proof_and_rank": shard["bytes_received_per_proof"],
                "note": "ONE proof / transform / commitment across all ranks (strong scaling), max over ranks, device "
                        "timed; full-vector in, full-vector out on every rank"}

    # outside every timed region (and after every timed section: it runs on rank 0 only, on the library's default
    # context): the proof that was timed is a valid proof -- the product's verifier (GPU linear
    # combinations + the BN254 pairing against X2 = [tau]_2) accepts it and rejects a tampered copy
    verified = None
    if rank == 0 and not args.no_verify:
        vk = setup.verification_key_arrays(n, pk)
        pf = pb.Proof.from_bytes(ref_proof)
        pub_ints = [int(x) for x in public]
        bad = bytearray(ref_proof)
        bad[32 * 14 + 31] ^= 1  # lowest bit of a_eval
        verified = bool(vk.verify_proof(n, pf, pub_ints) and vk.verify_proof_unoptimized(n, pf, pub_ints)
                        and not vk.verify_proof(n, pb.Proof.from_bytes(bytes(bad)), pub_ints))
        assert verified, "the benchmarked proof does not verify"
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last_proofs)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    hbm_gbs, peak_src = measured_peaks()
    proofs = args.steps * K * world
    value = proofs / (ms_dev * 1e-3)
    e2e = proofs / (ms_e2e * 1e-3)
    # dominant kernel: the MSM bucket accumulation (k_msm_seg_accumulate, one launch per MSM call, bracketed by an
    # event pair; with PB200_MSM_ACC=affine the rounds of batched affine additions of the call instead).  Algorithmic bytes: 96 B per point (64 B
    # affine point + 32 B scalar, SURVEY 8d) x the points of the call.
    xyzz = os.environ.get("PB200_MSM_ACC") != "affine"
    acc_avg_ms = acc_ms / max(1, acc_cnt)
    # 9 commitments x n points per proof go through the accumulation (4 batched MSM calls per proof)
    points_per_launch = 9.0 * n * args.steps / max(1, acc_cnt)
    achieved = 96.0 * points_per_launch / (acc_avg_ms * 1e-3) / 1e9
    windows = -(-256 // min(21, log_n))
    # DRAM traffic of the same launches from the committed ncu --set full capture (profiles/r02_dominant_kernel.json,
    # written by tools/summarize_profiles.py from the .ncu-rep), scaled to this run's average call
    traffic = None
    try:
        dk = json.load(open(os.path.join(ROOT, "profiles", "r02_dominant_kernel.json")))
        if dk.get("log_n") == log_n and xyzz:
            traffic = dk["dram_bytes_per_point"] * points_per_launch
    except Exception:
        pass
    ntt_avg_ms = ntt_ms / max(1, ntt_cnt)
    line = {
        "metric": metric_name(log_n), "value": value, "unit": "proofs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u256 (BN254 Fr/Fq integers, 8x32-bit Montgomery limbs)", "data": "synthetic",
        "config": {"workload": "PLONK prove (rounds 1-5, 9 KZG commits), synthetic 2^%d-gate circuit, structured "
                               "test SRS [tau^i]G of 2^%d powers" % (log_n, log_n),
                   "log_n": log_n, "seed": args.seed,
                   "parallelism": ("%d GPUs, replicas" % world if world > 1 else "1 GPU") + ", %d proofs in flight per GPU" % K,
                   "step": "one batch of %d independent proofs per GPU (%d prover lanes: own stream and scratch, shared "
                           "SRS, one host thread each); one lane alone: %.2f ms per proof" % (K, K, ms_solo / args.steps),
                   "proofs_in_flight_per_gpu": K,
                   "l2": "working set per proof ~3 GB >> 126 MB L2 (no flush needed)",
                   "setup_seconds_untimed": round(setup_s, 1)},
        "e2e": {"value": e2e, "unit": "proofs/s", "h2d_bytes_per_step": K * (3 * n * 32 + 32 * len(public)),
                "d2h_bytes_per_step": K * 768, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "value_remeasured": remeasured,
        "proof_verified": verified,
        "proof_matches_oracle_golden": golden_match,
        "sharded_proof_matches_single": shard["proof_ok"] if shard else None,
        "slab_ntt_matches_single": shard["ntt_ok"] if shard else None,
        "sharded_msm_matches_single": shard["msm_ok"] if shard else None,
        "one_proof_sharded": ({"n_gpus": world, "ms": shard["ms"], "proofs_per_s": 1e3 / shard["ms"],
                               "one_gpu_ms": ms_solo / args.steps,
                               "speedup": ms_solo / args.steps / shard["ms"],
                               "strong_scaling_efficiency": ms_solo / args.steps / shard["ms"] / world} if shard else None),
        "roofline": {"bound": "hbm",
                     "kernel": "k_msm_seg_accumulate" if xyzz else "k_aff_round0 + k_aff_round (the accumulation rounds of one MSM call)",
                     "achieved": achieved, "peak": hbm_gbs,
                     "unit": "GB/s", "frac": achieved / hbm_gbs, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": 96.0 * points_per_launch,
                     "modmul_ceiling_frac": ((10.0 if xyzz else 6.0) * windows * points_per_launch / (acc_avg_ms * 1e-3)) / 65.4e9,
                     "launches": int(acc_cnt), "avg_launch_ms": acc_avg_ms,
                     "share_of_step": acc_ms / ms_solo if ms_solo else None,
                     "msm_ms_per_proof": {"sort": sort_ms / args.steps, "accumulate": acc_ms / args.steps,
                                          "reduce": red_ms / args.steps},
                     "note": "a 'launch' is one MSM call's accumulation (event pair around its rounds), timed in a pass with "
                             "one lane (see config.step); integer-pipe bound, not HBM bound (ncu: profiles/); "
                             "modmul_ceiling_frac = field products/s (10 per XYZZ += affine addition -- 6 with "
                             "PB200_MSM_ACC=affine --, one addition per point and window) / 65.4e9 measured peak; traffic exceeds the algorithmic bytes because every point "
                             "is gathered once per window from the fixed-base table: see DESIGN.md"},
        "roofline_ntt": {"bound": "hbm", "kernel": "k_ntt_pass", "launches": int(ntt_cnt), "avg_launch_ms": ntt_avg_ms,
                         "achieved": comp["fr_ntt_fwd_plus_inv_2^%d" % log_n]["roofline"]["achieved"], "peak": hbm_gbs,
                         "unit": "GB/s", "frac": comp["fr_ntt_fwd_plus_inv_2^%d" % log_n]["roofline"]["frac"],
                         "note": "achieved = 64 B per element and transform / duration of a 2^%d forward + inverse pair "
                                 "(components); launches / avg_launch_ms: main-stream passes of the timed proofs (the coset "
                                 "extensions issued on the side stream are not timed)" % log_n,
                         "share_of_step": ntt_ms / ms_solo if ms_solo else None},
        "components": comp,
        "clocks": sampler.summary(),
    }
    if not args.no_cpu_baseline:
        try:
            ncpu, times = cpu_sample(args.cpu_log_n, 1)
            t = times[0]
            scale = n / ncpu
            line["cpu_baseline"] = {
                "value": 1.0 / (t * scale), "unit": "proofs/s", "cores": 1, "kind": "port",
                "sample": "oracle port of the reference's Python path: Prover.prove at 2^%d gates took %.2f s on one "
                          "host core, scaled linearly in gates to 2^%d (%d usable host cores; the reference is "
                          "single-threaded; --impl reference runs one worker per usable core)"
                          % (args.cpu_log_n, t, log_n, usable_cores())}
        except Exception as e:  # the bench line must still print
            line["cpu_baseline"] = {"value": None, "unit": "proofs/s", "cores": 1, "kind": "port", "sample": "failed: %r" % e}
    if not args.no_cpu_baseline:
        # a competent single-threaded CPU implementation for scale (NOT the reference): the C restatement of the
        # two cores (oracle/c/plonk_oracle.c) on one host core
        try:
            from oracle import c_oracle as CO
            rs = np.random.default_rng(3)
            v = rs.integers(0, 1 << 32, size=(1 << 18, 8), dtype=np.uint64).astype(np.uint32)
            v[:, 7] &= 0x0FFFFFFF
            t0 = time.perf_counter()
            CO.fft(v.view(np.uint8).reshape(-1, 32))
            t_fft = time.perf_counter() - t0
            m = 1 << 14
            pts = np.frombuffer(b"".join(p[0].n.to_bytes(32, "little") + p[1].n.to_bytes(32, "little")
                                         for p in setup.export_points(0, m)), dtype=np.uint8).reshape(m, 64)
            t0 = time.perf_counter()
            CO.g1_lincomb(pts, v[:m].view(np.uint8).reshape(-1, 32))
            t_msm = time.perf_counter() - t0
            line["cpu_c_restatement_1core"] = {
                "fr_ntt_2^18": {"s": t_fft, "elems_per_s": (1 << 18) / t_fft},
                "g1_msm_2^14": {"s": t_msm, "points_per_s": m / t_msm},
                "note": "oracle/c/plonk_oracle.c, one core; a competent-CPU scale line, not the reference's path"}
        except Exception as e:
            line["cpu_c_restatement_1core"] = {"error": repr(e)}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def timed_local(torch, stream, fn, steps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        reference_arm(a)
    else:
        b200_arm(a)
