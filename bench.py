#!/usr/bin/env python
"""bench.py -- IQ Msamples/s through the 32-PRN x 41-Doppler acquisition grid (BASELINE.json config 2), plus one sub-line
per other BASELINE configuration.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm (numpy) on the host cores
    python bench.py ... --dump-outputs DIR                   # also the records of the last timed step, DIR/<field>.npy

One STEP = one pass of the hot path over one batch of synthetic input: `calls_per_step` x `blocks_per_call` independent
1-ms IQ blocks @ 2.046 Msps (default 12 x 256 = 3072 blocks, 6.3 Msamples, ~25 ms of GPU work), each searched over the full
32 PRN x 41 Doppler (+-10 kHz / 500 Hz) grid with 1 ms of non-coherent integration -- i.e. 3072 x (BASELINE config 2).
The metric is per input sample, so the batch only sets how much work one step carries.

  value : steps timed with CUDA events on the launching stream, inputs already in HBM (an IQ ring larger than L2, fresh
          blocks every call), per-cell records left on the device.
  e2e   : the same steps through the public host API, copies inside the timed region.
          N = 1: pinned host IQ -> GridStream.submit / collect (pipelined copies) -> per-cell records in host memory.
          N > 1: ALL the step's IQ starts in rank 0's host memory and ALL per-cell records end there:
                 ShardedBlockStream = one H2D on rank 0, one NCCL scatter of block shares, the grid on every rank, one NCCL
                 gather of the records, one D2H on rank 0 (north_star's "single broadcast ... final gather"), two steps in
                 flight so that rank 0's copies run under the kernels; the one-call (unpipelined) figure is reported beside it.
  N > 1 : one process per GPU (torchrun); `value` = every rank searching its own resident blocks (weak scaling, no
          data-path collective); time = max over ranks.
  configs: config3 / config4 / config5 sub-objects (N = 1), and at N > 1 config5 as a STRONG-scaling job (1000 blocks
          @ 16.368 Msps scattered from rank 0, records gathered back) beside the weak numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N = 2046
WORKLOAD = "config2: 32 PRN x 41 Doppler (+-10 kHz / 500 Hz) x 1 ms non-coherent @ 2.046 Msps complex64"  # both arms
FS = 2046000
N_PRN = 32
DOPPLERS = np.arange(-10000.0, 10001.0, 500.0)  # 41 bins
DOPPLERS_81 = np.arange(-10000.0, 10001.0, 250.0)  # config 5
N_MS = 1
METRIC = "IQ Msamples/s through 32-PRN x 41-Doppler acquisition (1 ms non-coherent, 2.046 Msps complex64)"
L2_BYTES = 126 << 20
PLANTED = [(3, -3000.0, 5, 1.0, 0.3), (11, 4500.0, 1234, 2.0, 0.3), (25, 1500.0, 777, 0.3, 0.3), (32, -9500.0, 2045, 2.5, 0.3)]
MAG_TOL = 1e-5  # DESIGN.md section 6
DUMP_BYTES = 63_000_000  # --dump-outputs stays under 64 MB, .npy headers included


def dump_outputs(out_dir: str, blocks: np.ndarray, records: dict) -> None:
    """--dump-outputs: per-cell records of the last timed step as <field>.npy, each [blocks, 32 PRN, D Doppler] in float32 or
    float64, plus block.npy, the index of each block in the IQ the step read.  The inputs are seeded, so two builds run with the
    same arguments can be compared file for file; blocks beyond the size budget are dropped by a fixed, seeded choice."""
    per_block = 8 + sum(a[0].nbytes for a in records.values())
    keep = np.arange(len(blocks))
    if per_block * len(blocks) > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(len(blocks), DUMP_BYTES // per_block, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "block.npy"), blocks[keep].astype(np.float64))
    for name, a in records.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a[keep])


def alg_bytes(n: int, n_dop: int, m: int, n_blocks: int = 1) -> float:
    """SURVEY.md 8(d): P*D*M*16N + 32*P*D per block (IQ chunk + replica spectrum per cell-ms, one 32-byte record per cell)."""
    return n_blocks * (N_PRN * n_dop * m * 16 * n + 32 * N_PRN * n_dop)


def noise_blocks(n_blocks: int, n: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    out = np.empty((n_blocks, n), dtype=np.complex64)
    step = max(1, (1 << 22) // n)
    for b0 in range(0, n_blocks, step):
        nb = min(step, n_blocks - b0)
        z = rng.standard_normal((nb, n), dtype=np.float32) + 1j * rng.standard_normal((nb, n), dtype=np.float32)
        out[b0:b0 + nb] = z * np.float32(1 / np.sqrt(2))
    return out


def make_ring(n_blocks: int, seed: int, n: int = N, fs: int = FS, m: int = 1, planted=PLANTED) -> np.ndarray:
    """complex64[n_blocks, m * n]: seeded gaussian noise with planted satellites (SURVEY.md 8d)."""
    from gypsum_b200 import synth as o  # product-side generator (the oracle is only used by the CPU legs below)

    ring = noise_blocks(n_blocks, m * n, seed)
    ring += o.synth_iq(seed, n, m, fs, planted, sigma=0.0)
    return ring


# ----------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def window(self, t0: float, t1: float) -> dict:
        sm, mx, reasons, power = [], [], set(), []
        for t, line in list(self.rows):
            if not (t0 <= t <= t1):
                continue
            p = [x.strip() for x in line.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1])); power.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}

    def stop(self) -> None:
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()


# ----------------------------------------------------------------------------------------------------------------
# CPU legs: the reference algorithm (numpy restatement in oracle/), cells spread over ALL host cores
# ----------------------------------------------------------------------------------------------------------------
def _cpu_cells_worker(args):
    """One process's share of a grid: cells = [(block, sv, doppler index)], reduced like acquisition.py:180-189."""
    blocks, fs, n, dop, cells = args
    from oracle import gypsum_oracle as o  # the CPU legs are the one place bench.py may execute the oracle

    out = np.zeros((len(cells), 4))
    reps = {}
    for i, (b, sv, d) in enumerate(cells):
        prn = reps.get(sv)
        if prn is None:
            prn = reps[sv] = o.replica(sv, n)
        prof = o.integrate(o.NON_COHERENT, blocks[b], fs, n, dop[d], prn)
        mx = prof.max()
        out[i] = (mx, int(np.argmax(prof)), prof.sum(), int(np.count_nonzero(prof == mx)))
    return out


def _cpu_track_worker(args):
    x, ch, init, fs, n, n_ms = args
    from oracle import tracker_oracle as t

    tr = t.TrackerOracle(ch[0], init[0], init[1], init[2], fs, n)
    sym = []
    for k in range(n_ms):
        a, b = t.chunk_times(k, fs, n)
        sym.append(tr.step(x[k * n:(k + 1) * n], a, b)["symbol"])
    return sym


def usable_cores() -> int:
    """Host threads this process may actually run on: the affinity mask, capped by a cgroup CPU quota when there is one."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return n


def _cpu_acquire_worker(args):
    x, fs, n, sv = args
    from oracle import gypsum_oracle as o

    r = o.acquire_sv(sv, x, fs, n)
    return sv, r.doppler, r.code_phase, r.strength


class CpuPool:
    """Fork pools created BEFORE CUDA is initialised in this process.  The box reports more hardware threads than the
    numpy path can use (SMT siblings share one FFT unit; a container quota may sit below the thread count), so the pool
    size is CALIBRATED: the same two-block grid is timed at several process counts and the fastest one is kept -- the CPU
    leg is given every host thread that helps it."""

    def __init__(self, calibrate: bool = True):
        import multiprocessing as mp

        self.avail = usable_cores()
        cands = sorted({c for c in (self.avail, self.avail // 2, self.avail // 4, 32, 16) if 1 <= c <= self.avail})
        self.calibration = {}
        best = None
        blocks = noise_blocks(2, N, 7)
        for c in (cands if calibrate else [self.avail]):
            pool = mp.get_context("fork").Pool(c)
            pool.map(_warm, range(c))
            self.cores, self.pool = c, pool
            sec = min(self.grid(blocks, FS, N, DOPPLERS)[1] for _ in range(2)) if calibrate else 0.0
            self.calibration[c] = sec
            if best is None or sec < best[0]:
                if best is not None:
                    best[2].terminate()
                best = (sec, c, pool)
            else:
                pool.terminate()
        _, self.cores, self.pool = best

    def grid(self, blocks: np.ndarray, fs: int, n: int, dop: np.ndarray):
        """Full 32 x D grid of every block in `blocks` [nb, M*n].  Returns (records [nb, 32, D, 4], seconds)."""
        nb, nd = blocks.shape[0], len(dop)
        cells = [(b, sv, d) for b in range(nb) for sv in range(1, N_PRN + 1) for d in range(nd)]
        # contiguous shares: a process sees few distinct (block, PRN) pairs, so its replica spectra stay in cache
        bounds = [len(cells) * i // self.cores for i in range(self.cores + 1)]
        parts = [cells[bounds[i]:bounds[i + 1]] for i in range(self.cores)]
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_cells_worker, [(blocks, fs, n, dop, p) for p in parts if p], chunksize=1)
        sec = time.perf_counter() - t0
        flat = np.concatenate(res, axis=0)
        return flat.reshape(nb, N_PRN, nd, 4), sec

    def describe(self) -> str:
        cal = ", ".join(f"{c}: {1e3 * s:.0f} ms" for c, s in sorted(self.calibration.items()))
        return f"{self.cores} processes (fastest of the calibrated counts; two-block grid: {cal}; {self.avail} host threads usable)"

    def close(self):
        self.pool.terminate()


def _warm(_):
    from oracle import gypsum_oracle as o

    o.integrate(o.NON_COHERENT, np.zeros(N, np.complex64), FS, N, 0.0, o.replica(1, N))
    return 0


def check_records(rec, ref, x_blocks, fs, n, dop, what) -> int:
    """GPU records [nb, 32, D] (RECORD_DTYPE) vs the CPU grid [nb, 32, D, 4]: magnitudes to 1e-5 of the largest, count
    exact, code phase exact unless the float64 profile itself ties to within the tolerance at the GPU's index."""
    from oracle import gypsum_oracle as o

    peak, arg, total, count = ref[..., 0], ref[..., 1].astype(np.int64), ref[..., 2], ref[..., 3].astype(np.int64)
    assert np.abs(rec["peak"] - peak).max() <= MAG_TOL * peak.max(), f"{what}: peak mismatch vs the CPU reference"
    assert np.abs(rec["sum"] - total).max() <= MAG_TOL * total.max(), f"{what}: sum mismatch vs the CPU reference"
    assert np.array_equal(rec["count"], count), f"{what}: count mismatch vs the CPU reference"
    for b, a, d in np.argwhere(rec["argmax"] != arg):
        prof = o.integrate(o.NON_COHERENT, x_blocks[b], fs, n, dop[d], o.replica(a + 1, n))
        assert prof.max() - prof[rec["argmax"][b, a, d]] <= MAG_TOL * prof.max(), f"{what}: code phase mismatch at {(b, a, d)}"
    return int(peak.size)


def run_reference(args, rank: int, world: int) -> None:
    """--impl reference: the reference's own CPU implementation of the path.  gypsum is pure Python + numpy and
    /root/reference does not exist on the GPU box, so this is the oracle port (numpy, same pocketfft calls), the cells of
    each step's blocks spread over ALL host cores.  Rank 0 only."""
    if rank != 0:
        return
    t_start = time.perf_counter()
    pool = CpuPool()
    nb = args.cpu_blocks_per_step
    blocks = make_ring(nb * 2, seed=1)
    times = []
    for k in range(args.warmup + args.steps):
        ref, sec = pool.grid(blocks[(k % 2) * nb:(k % 2 + 1) * nb], FS, N, DOPPLERS)
        times.append(sec)
    pool.close()
    per_step = times[args.warmup:]
    total = sum(per_step)
    value = args.steps * nb * N / total / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "blocks_per_step": nb,
                   "sample": f"each step = the full 32x41 grid over {nb} 1-ms blocks (bounded sample of the GPU arm's step)"},
        "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": pool.cores, "kind": "port",
                         "sample": f"{args.steps} steps x {nb} blocks x 1312 cells over {pool.describe()}"},
        "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t_start,
    }
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, (k % 2) * nb + np.arange(nb),
                     {f: ref[..., i] for i, f in enumerate(("peak", "argmax", "sum", "count"))})


# ----------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------
class Gpu:
    """Shared plumbing of the GPU measurements: stream, barrier, event timing with max over ranks."""

    def __init__(self, rank, local_rank, world):
        import torch

        self.torch = torch
        self.rank, self.local_rank, self.world = rank, local_rank, world
        torch.cuda.set_device(local_rank)
        self.dist = None
        if world > 1:
            import torch.distributed as dist

            # NCCL announces its version on stdout when the communicator comes up; keep stdout to the one JSON line
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
                dist.barrier()
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)
            self.dist = dist
        self.stream = torch.cuda.Stream()  # a real (non-legacy) stream: the engine launches on it, the events time it
        torch.cuda.set_stream(self.stream)

    def engine(self, fs, n):
        from gypsum_b200 import _native
        from gypsum_b200.gps_ca_prn_codes import ca_code_chips

        eng = _native.Engine(fs, n, device=self.local_rank)
        eng.set_replicas(np.stack([ca_code_chips(sv) for sv in range(1, 33)]).astype(np.uint8))
        eng.set_stream(self.stream.cuda_stream)
        return eng

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v: float) -> float:
        if self.dist is None:
            return v
        t = self.torch.tensor([v], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps: int, first: int = 0) -> float:
        """ms for `steps` calls of fn(k), CUDA events on the launching stream, max over ranks."""
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record(self.stream)
        for k in range(first, first + steps):
            fn(k)
        e1.record(self.stream)
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1))

    def wall(self, fn, steps: int, first: int = 0, drain=None) -> float:
        """seconds for `steps` host-to-host calls of fn(k) (+ drain), barrier on both sides, max over ranks."""
        self.barrier()
        t0 = time.perf_counter()
        for k in range(first, first + steps):
            fn(k)
        if drain is not None:
            drain()
        self.torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        self.barrier()
        return self.max_over_ranks(sec)


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured)"
    return 6650.0, "B200_PROFILING.md fallback"


def kernel_times(eng, fn, reps: int):
    """(doppler_spectra ms per launch, launches, correlate ms per launch, launches) over `reps` calls of fn(k)."""
    eng.enable_kernel_timing(True)
    for k in range(reps):
        fn(k)
    ks, ns = eng.kernel_timing(0)
    kc, nc = eng.kernel_timing(1)
    eng.enable_kernel_timing(False)
    return ks / max(ns, 1), ns, kc / max(nc, 1), nc


def traffic_for(key: str):
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        return json.load(open(tp)).get(key)
    return None


def run_ours(args, rank: int, local_rank: int, world: int) -> None:
    cpu = CpuPool() if rank == 0 else None  # fork before CUDA comes up
    import torch

    from gypsum_b200 import _native

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU leg)")
    g = Gpu(rank, local_rank, world)
    peak_gbs, peak_src = peak_hbm()

    B, C = args.blocks_per_call, args.calls_per_step
    block_bytes = N * 8
    ring_blocks = max(args.ring_blocks, (L2_BYTES // block_bytes // B + 2) * B)
    ring_blocks -= ring_blocks % B
    ring_host = torch.from_numpy(make_ring(ring_blocks, seed=1000 + rank)).pin_memory()
    ring_dev = ring_host.to("cuda", non_blocking=False)
    n_slots = ring_blocks // B
    n_cells = N_PRN * len(DOPPLERS)
    rec_dev = torch.empty((4, B * n_cells * 32), dtype=torch.uint8, device="cuda")
    eng = g.engine(FS, N)
    prn = np.arange(N_PRN, dtype=np.int32)
    dop = np.ascontiguousarray(DOPPLERS, dtype=np.float64)

    def device_call(j: int) -> None:
        slot = j % n_slots
        eng.bind_iq_device(ring_dev.data_ptr() + slot * B * block_bytes, B * N)
        eng.acquire_grid_device(B, N_MS, prn, dop, _native.NON_COHERENT, rec_dev[j % 4].data_ptr())

    def device_step(k: int) -> None:
        for c in range(C):
            device_call(k * C + c)

    # ---- warm-up, then the timed device-resident region (clock sampler running) ----
    for k in range(max(args.warmup, 3)):
        device_step(k)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    time.sleep(0.15)
    t_clock0 = time.perf_counter()
    launches0 = eng.launch_count
    ms_total = g.timed(device_step, args.steps, first=args.warmup)
    launches = eng.launch_count - launches0
    if args.dump_outputs and rank == 0:
        # the record ring has 4 slots: it still holds the last min(C, 4) calls of the last timed step
        last = [(args.warmup + args.steps - 1) * C + c for c in range(max(0, C - 4), C)]
        rec = np.concatenate([rec_dev[j % 4].cpu().numpy().view(_native.RECORD_DTYPE).reshape(B, N_PRN, len(DOPPLERS))
                              for j in last])
        dump_outputs(args.dump_outputs, np.concatenate([(j % n_slots) * B + np.arange(B) for j in last]),
                     {"peak": rec["peak"], "argmax": rec["argmax"].astype(np.float32), "sum": rec["sum"],
                      "count": rec["count"].astype(np.float32)})
    t_end = time.perf_counter() + 0.3  # continuation of the same loop so that short runs still get clock samples under load
    k = args.warmup + args.steps
    while time.perf_counter() < t_end:
        device_step(k)
        k += 1
        torch.cuda.synchronize()
    t_clock1 = time.perf_counter()
    clocks = sampler.window(t_clock0, t_clock1) if sampler else None
    if clocks is not None:
        clocks["window"] = "timed region plus a 0.3 s continuation of the same step loop"

    samples_per_step = C * B * N
    value = world * args.steps * samples_per_step / (ms_total * 1e-3) / 1e6

    # ---- per-kernel device time (second pass, event-bracketed launches) for the roofline ----
    spec_ms, spec_n, corr_ms, corr_n = kernel_times(eng, device_call, 3 * C)

    # ---- end to end through the public host API ----
    depth = 3
    rec_pinned = [torch.empty(B * n_cells * 32, dtype=torch.uint8).pin_memory() for _ in range(depth)]
    rec_host = [r.numpy().view(_native.RECORD_DTYPE).reshape(B, N_PRN, len(DOPPLERS)) for r in rec_pinned]
    e2e = {}
    if world == 1:
        gs = _native.GridStream(eng, B, N_MS, prn, dop, _native.NON_COHERENT, depth=depth)
        collected = [0]
        last = [None]

        def e2e_step(k: int) -> None:
            for c in range(C):
                j = k * C + c
                if gs.in_flight == depth:
                    last[0] = gs.collect()
                    collected[0] += 1
                gs.submit(ring_host.data_ptr() + (j % n_slots) * B * block_bytes, rec_host[j % depth])

        def drain() -> None:
            while gs.in_flight:
                last[0] = gs.collect()
                collected[0] += 1

        e2e_step(0)
        drain()
        collected[0] = 0
        sec = g.wall(e2e_step, args.steps, first=1, drain=drain)
        assert collected[0] == args.steps * C, "every submitted batch must come back inside the timed region"
        rec = last[0]
        assert int(rec["argmax"][0, 24, int(np.argmax(rec["peak"][0, 24]))]) == 777, "planted SV25 not at code phase 777"
        gs.close()
        e2e = {"value": args.steps * samples_per_step / sec / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": C * B * block_bytes, "d2h_bytes_per_step": C * B * n_cells * 32,
               "api": f"GridStream.submit / collect, depth {depth}, {C} batches of {B} blocks per step"}

        def e2e_sync_call(j: int) -> None:
            eng.upload_iq_ptr(ring_host.data_ptr() + (j % n_slots) * B * block_bytes, B * N)
            eng.acquire_grid(B, N_MS, prn, dop, _native.NON_COHERENT, out=rec_host[0])

        for j in range(3):
            e2e_sync_call(j)
        n_sync = min(args.steps * C, 256)
        e2e["synchronous_call_value"] = n_sync * B * N / g.wall(e2e_sync_call, n_sync, first=3) / 1e6
    else:
        e2e = multi_gpu_e2e(g, eng, args, prn, dop)

    # ---- single-block latency: one 32x41 grid over ONE 1-ms block (what config 2 literally names) ----
    one_rec = torch.empty(n_cells * 32, dtype=torch.uint8, device="cuda")

    def one_block_step(k: int) -> None:
        eng.bind_iq_device(ring_dev.data_ptr() + (k % ring_blocks) * block_bytes, N)
        eng.acquire_grid_device(1, N_MS, prn, dop, _native.NON_COHERENT, one_rec.data_ptr())

    for k in range(5):
        one_block_step(k)
    one_block_ms = g.timed(one_block_step, 500, first=5) / 500
    one_out = rec_host[0][:1]
    lat = []
    for k in range(400):
        t1 = time.perf_counter()
        eng.acquire_grid_host(ring_host.data_ptr() + (k % ring_blocks) * block_bytes, 1, N_MS, prn, dop, _native.NON_COHERENT,
                              out=one_out)
        lat.append(time.perf_counter() - t1)
    single_us = 1e6 * float(np.median(lat[20:]))
    assert int(one_out["argmax"][0, 24, int(np.argmax(one_out["peak"][0, 24]))]) == 777
    single_block = {"note": "the same grid with ONE 1-ms block per call",
                    "device_Msamples_per_s": N / (one_block_ms * 1e-3) / 1e6, "device_us_per_block": 1e3 * one_block_ms,
                    "e2e_us_per_block": single_us, "e2e_Msamples_per_s": N / (single_us * 1e-6) / 1e6,
                    "e2e_api": "gb200_acquire_grid_host: {copy-in, 2 kernels} replayed as one CUDA graph, records stored by the kernel into the caller's pinned buffer, one host sync"}

    line = None
    if rank == 0:
        alg = alg_bytes(N, len(DOPPLERS), N_MS, B)
        achieved = alg / (corr_ms * 1e-3) / 1e9
        traffic = traffic_for("correlate_cells_dram_bytes_per_launch")

        # ---- parity of this run's own output: the CPU reference grid of `cpu_blocks` of the GPU arm's blocks, cell for cell
        cpu_blocks = ring_host.numpy()[: args.cpu_blocks]
        ref, _ = cpu.grid(cpu_blocks, FS, N, DOPPLERS)  # also warms the pool for the timed repeats below
        eng.upload_iq(cpu_blocks.reshape(-1))
        got = eng.acquire_grid(args.cpu_blocks, N_MS, prn, dop, _native.NON_COHERENT)
        parity_cells = check_records(got, ref, cpu_blocks, FS, N, DOPPLERS, "config 2")
        cpu_secs = [cpu.grid(cpu_blocks, FS, N, DOPPLERS)[1] for _ in range(3)]
        cpu_sps = args.cpu_blocks * N / float(np.median(cpu_secs))
        t_single = time.perf_counter()
        _cpu_cells_worker((cpu_blocks[:1], FS, N, DOPPLERS, [(0, sv, d) for sv in range(1, 9) for d in range(len(DOPPLERS))]))
        single_sps = N / ((time.perf_counter() - t_single) * 4)  # a quarter of the grid, one process, one thread

        line = {
            "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": WORKLOAD, "blocks_per_step": C * B, "calls_per_step": C, "blocks_per_call": B, "cells_per_block": n_cells,
                "parallelism": (f"value: blocks sharded over {world} GPU(s), no collective; "
                                + ("e2e: one process" if world == 1 else "e2e: rank-0 host -> NCCL scatter -> grid per rank -> NCCL gather -> rank-0 host")),
                "l2": f"inputs larger than L2: IQ ring of {ring_blocks} distinct blocks = {ring_blocks * block_bytes >> 20} MiB per GPU, "
                      f"fresh blocks every call; the spectra scratch ({B * 1.34:.0f} MB per call) is written and re-read by the two kernels of a call",
            },
            "e2e": e2e,
            "single_block": single_block,
            "gpu_launches": int(launches),
            "parity_checked_cells": parity_cells,
            "parity": f"{parity_cells} cells of {args.cpu_blocks} of the timed blocks == CPU reference (peak/sum 1e-5 of max, count and code phase exact bar float64 near-ties)",
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "k_correlate_w2048 (correlate_cells, one warp per transform)", "achieved": achieved,
                         "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg, "kernel_ms_per_launch": corr_ms, "launches_timed": int(corr_n),
                         "kernel_share_of_step": corr_ms * corr_n / max(corr_ms * corr_n + spec_ms * spec_n, 1e-12),
                         "other_kernels_ms_per_launch": {"k_doppler_spectra": spec_ms},
                         "secondary": secondary_rooflines(traffic, corr_ms, ms_total / args.steps / C, B, n_cells, clocks),
                         "note": "algorithmic bytes are on-chip reuse traffic (each IQ byte feeds 1312 cells); DRAM traffic is near the compulsory minimum, the kernel is FP32-issue / shared-memory bound"},
            "cpu_baseline": {"value": cpu_sps / 1e6, "unit": "Msamples/s", "cores": cpu.cores, "kind": "port",
                             "single_thread_value": single_sps / 1e6,
                             "sample": f"{args.cpu_blocks} of the GPU arm's 1-ms blocks x full 32x41 grid, median of 3, cells over {cpu.describe()}"},
        }
    eng.close()
    del ring_dev, rec_dev

    configs = {}
    if world == 1 and not args.no_configs:
        configs["config3"] = bench_config3(g, cpu, peak_gbs, sampler)
        configs["config5"] = bench_config5(g, cpu, peak_gbs, sampler, None)
        configs["config4"] = bench_config4(g, cpu, peak_gbs, sampler)
        configs["detector"] = bench_detector(g, cpu, sampler)
    elif world > 1 and not args.no_configs:
        configs["config5"] = bench_config5(g, cpu, peak_gbs, sampler, args)
        configs["sharded_single_block"] = bench_sharded_single_block(g)
    if sampler:
        sampler.stop()
    if cpu:
        cpu.close()
    if rank == 0:
        line["configs"] = configs
        print(json.dumps(line), flush=True)
    if g.dist is not None:
        g.dist.destroy_process_group()


def multi_gpu_e2e(g, eng, args, prn, dop) -> dict:
    """N > 1: one step's IQ (world x C x B blocks) starts in rank 0's pinned host memory, the per-cell records of all of it
    end in rank 0's host memory; ShardedBlockSearch moves them with one scatter and one gather per step."""
    from gypsum_b200 import _native
    from gypsum_b200.distributed import ShardedBlockSearch

    torch = g.torch
    B, C, world = args.blocks_per_call, args.calls_per_step, g.world
    per_rank = B * C
    total_blocks = per_rank * world
    host = None
    if g.rank == 0:
        host = torch.from_numpy(make_ring(total_blocks, seed=77)).pin_memory().numpy().reshape(-1)
    search = ShardedBlockSearch(eng, torch.device("cuda", g.local_rank))
    out = {}
    for key, mode in (("per_cell", None), ("best_bin", "best")):
        res = [None]

        def step(k: int) -> None:
            res[0] = search.acquire_blocks(host, total_blocks, N_MS, prn, dop, _native.NON_COHERENT, reduce=mode, copy=False)

        step(0)
        steps = max(3, min(args.steps, 10))
        sec = g.wall(step, steps, first=1) / steps
        if g.rank == 0:
            r = res[0]
            if mode is None:
                assert r.shape == (total_blocks, N_PRN, len(dop))
                for b in (0, total_blocks // 2, total_blocks - 1):
                    assert int(r["argmax"][b, 24, int(np.argmax(r["peak"][b, 24]))]) == 777
            else:
                assert (r["doppler"][total_blocks - 1, 24], r["code_phase"][total_blocks - 1, 24]) == (1500.0, 777)
        out[key] = {"value": total_blocks * N / sec / 1e6, "seconds_per_step": sec, "steps": steps, **search.last_bytes}
    # the same steps as a pipelined stream: two steps in flight, rank 0's copies on the copy engines under the kernels
    from gypsum_b200.distributed import ShardedBlockStream

    for key, mode in (("per_cell_stream", None), ("best_bin_stream", "best")):
        st = ShardedBlockStream(eng, torch.device("cuda", g.local_rank), total_blocks, N_MS, prn, dop, _native.NON_COHERENT, reduce=mode)
        last = [None]

        def sstep(k: int) -> None:
            if st.in_flight == 2:
                last[0] = st.collect()
            st.submit(host)

        def sdrain() -> None:
            while st.in_flight:
                last[0] = st.collect()

        sstep(0)
        sdrain()
        steps = max(4, min(args.steps, 12))
        sec = g.wall(sstep, steps, first=1, drain=sdrain) / steps
        if g.rank == 0:
            r = last[0]
            if mode is None:
                for b in (0, total_blocks // 2, total_blocks - 1):
                    assert int(r["argmax"][b, 24, int(np.argmax(r["peak"][b, 24]))]) == 777
            else:
                assert (r["doppler"][total_blocks - 1, 24], r["code_phase"][total_blocks - 1, 24]) == (1500.0, 777)
        out[key] = {"value": total_blocks * N / sec / 1e6, "seconds_per_step": sec, "steps": steps, **st.bytes_per_job}
        del st
    ps, pc = out["per_cell_stream"], out["per_cell"]
    return {"value": ps["value"], "unit": "Msamples/s", "h2d_bytes_per_step": ps["h2d"], "d2h_bytes_per_step": ps["d2h"],
            "nccl_scatter_bytes_per_step": ps["scatter"], "nccl_gather_bytes_per_step": ps["gather"],
            "blocks_per_step": total_blocks, "seconds_per_step": ps["seconds_per_step"],
            "api": "ShardedBlockStream.submit / collect (two steps in flight): rank-0 pinned host IQ -> H2D (copy stream) -> ONE NCCL scatter -> "
                   "grid on every rank -> ONE NCCL gather -> D2H (copy stream) -> rank-0 host records",
            "synchronous_call_value": pc["value"], "synchronous_call_seconds_per_step": pc["seconds_per_step"],
            "with_on_device_best_bin_reduction": {"value": out["best_bin_stream"]["value"], "seconds_per_step": out["best_bin_stream"]["seconds_per_step"],
                                                  "synchronous_call_value": out["best_bin"]["value"],
                                                  "d2h_bytes_per_step": out["best_bin"]["d2h"],
                                                  "nccl_gather_bytes_per_step": out["best_bin"]["gather"],
                                                  "note": "acquisition.py:179-189 per (block, PRN) row on the device: 32 B per row instead of 32 B per cell"},
            "limiter": "rank 0's return path: the NCCL gather of every rank's per-cell records (42 KB per block) sits between the kernel "
                       "phases (NCCL's kernels cannot co-reside with the persistent full-shared-memory correlate CTAs: overlapping them "
                       "was measured and is slower, profiles/ablation_r2.md), and the ONE device->host copy over rank 0's PCIe link "
                       "(688 MB per step at 8 GPUs) only hides under the next step's kernels while it is shorter than them; "
                       "the best-bin reduction removes 40/41 of both"}


def secondary_rooflines(traffic, corr_ms, call_ms, blocks, n_cells, clocks):
    """DRAM GB/s of the dominant kernel (ncu bytes / live duration) and the nominal algorithmic flop rate of one call
    (SURVEY.md 8d: 2 * 5 N log2 N + 16 N flops per cell-ms) against the FP32 FMA peak at the observed SM clock."""
    flops = float((2 * 5 * N * np.log2(N) + 16 * N) * N_MS * n_cells * blocks)
    sm_mhz = float((clocks or {}).get("sm_mhz") or 1965.0)
    fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12  # TFLOP/s: 148 SMs x 128 FMA lanes
    out = {"algorithmic_tflops": flops / (call_ms * 1e-3) / 1e12, "fp32_fma_peak_tflops": fp32_peak,
           "algorithmic_flop_frac": flops / (call_ms * 1e-3) / 1e12 / fp32_peak,
           "flop_note": "nominal radix-2 count incl. the forward transforms the de-duplicated design computes once per Doppler, "
                        "not 32 times; FFT butterflies are mostly FADD/FMUL, so 50 % of the FMA peak is the practical ceiling"}
    if traffic:
        out["dram_gbs"] = traffic / (corr_ms * 1e-3) / 1e9
    return out


# ----------------------------------------------------------------------------------------------------------------
# the other BASELINE configurations
# ----------------------------------------------------------------------------------------------------------------
def bench_config3(g, cpu, peak_gbs, sampler) -> dict:
    """32 PRN x 41 Doppler, 10 ms non-coherent @ 4.092 Msps: one 10-ms window per call (what receiver.py:219 hands over)."""
    from gypsum_b200 import _native

    torch = g.torch
    n, fs, m = 4092, 4092000, 10
    planted = [(3, -3000.0, 5, 1.0, 0.1), (11, 4500.0, 2500, 2.0, 0.1), (25, 1500.0, 4091, 0.3, 0.08), (32, -9500.0, 2045, 2.5, 0.1)]
    win_bytes = m * n * 8
    n_win = L2_BYTES // win_bytes + 2
    host = torch.from_numpy(make_ring(n_win, seed=3, n=n, fs=fs, m=m, planted=planted)).pin_memory()
    dev = host.to("cuda")
    eng = g.engine(fs, n)
    prn = np.arange(N_PRN, dtype=np.int32)
    dop = np.ascontiguousarray(DOPPLERS)
    n_cells = N_PRN * len(dop)
    rec_dev = torch.empty(n_cells * 32, dtype=torch.uint8, device="cuda")

    def call(k):
        eng.bind_iq_device(dev.data_ptr() + (k % n_win) * win_bytes, m * n)
        eng.acquire_grid_device(1, m, prn, dop, _native.NON_COHERENT, rec_dev.data_ptr())

    for k in range(5):
        call(k)
    reps = 1500
    t0 = time.perf_counter()
    ms = g.timed(call, reps, first=5) / reps
    t1 = time.perf_counter()
    spec_ms, spec_n, corr_ms, corr_n = kernel_times(eng, call, 50)
    out_host = (torch.empty(n_cells * 32, dtype=torch.uint8).pin_memory().numpy().view(_native.RECORD_DTYPE)
                .reshape(1, N_PRN, len(dop)))
    for k in range(5):
        eng.acquire_grid_host(host.data_ptr() + (k % n_win) * win_bytes, 1, m, prn, dop, _native.NON_COHERENT, out=out_host)

    def e2e_call(k):
        eng.acquire_grid_host(host.data_ptr() + (k % n_win) * win_bytes, 1, m, prn, dop, _native.NON_COHERENT, out=out_host)

    n_e2e = 1000
    sec = g.wall(e2e_call, n_e2e, first=5)
    # parity + CPU baseline on one of the timed windows
    x0 = host.numpy()[:1]
    ref, cpu_sec = cpu.grid(x0, fs, n, DOPPLERS)
    eng.upload_iq(x0.reshape(-1))
    got = eng.acquire_grid(1, m, prn, dop, _native.NON_COHERENT)
    cells = check_records(got, ref, x0, fs, n, DOPPLERS, "config 3")
    alg = alg_bytes(n, len(dop), m)
    res = {"workload": "config3: 32 PRN x 41 Doppler x 10 ms non-coherent @ 4.092 Msps, one 10-ms window per call",
           "value": m * n / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "device_ms_per_window": ms, "calls_timed": reps,
           "e2e": {"value": m * n * n_e2e / sec / 1e6, "unit": "Msamples/s", "h2d_bytes_per_call": win_bytes, "d2h_bytes_per_call": n_cells * 32,
                   "us_per_window": 1e6 * sec / n_e2e, "api": "gb200_acquire_grid_host: DMA from the caller's pinned window, 2 kernels, records stored into the caller's pinned buffer"},
           "roofline": {"bound": "hbm", "kernel": "k_correlate_cells<8, non-coherent> (warp pair per transform, 10-ms accumulation)",
                        "achieved": alg / (corr_ms * 1e-3) / 1e9, "peak": peak_gbs, "unit": "GB/s", "frac": alg / (corr_ms * 1e-3) / 1e9 / peak_gbs,
                        "algorithmic_bytes_per_launch": alg, "kernel_ms_per_launch": corr_ms, "other_kernels_ms_per_launch": {"k_doppler_spectra": spec_ms},
                        "traffic": traffic_for("config3_correlate_dram_bytes_per_launch")},
           "cpu_baseline": {"value": m * n / cpu_sec / 1e6, "unit": "Msamples/s", "cores": cpu.cores, "kind": "port",
                            "sample": "one of the timed 10-ms windows, full 32x41 grid, cells over all cores"},
           "parity_checked_cells": cells,
           "l2": f"ring of {n_win} distinct windows = {n_win * win_bytes >> 20} MiB (> L2)",
           "clocks": sampler.window(t0, t1) if sampler else None}
    eng.close()
    return res


def bench_config5(g, cpu, peak_gbs, sampler, args) -> dict:
    """32 PRN x 81 Doppler @ 16.368 Msps over 1000 independent 1-ms blocks.  N = 1: the whole job on one GPU.  N > 1: the
    same FIXED job, IQ on rank 0's host, sharded with one scatter + one gather (strong scaling)."""
    from gypsum_b200 import _native

    torch = g.torch
    n, fs, nb = 16368, 16368000, 1000
    planted = [(3, -3000.0, 5, 1.0, 0.12), (11, 4500.0, 12345, 2.0, 0.12), (25, 1500.0, 16367, 0.3, 0.1)]
    prn = np.arange(N_PRN, dtype=np.int32)
    dop = np.ascontiguousarray(DOPPLERS_81)
    n_cells = N_PRN * len(dop)
    eng = g.engine(fs, n)
    host = None
    if g.rank == 0:
        host = torch.from_numpy(make_ring(nb, seed=5, n=n, fs=fs, planted=planted)).pin_memory()
    res = {"workload": "config5: 32 PRN x 81 Doppler (+-10 kHz / 250 Hz) x 1 ms @ 16.368 Msps, 1000 independent blocks",
           "unit": "Msamples/s", "blocks": nb, "job_samples": nb * n, "job_cells": nb * n_cells}
    if g.world == 1:
        dev = host.to("cuda")
        rec_dev = torch.empty(nb * n_cells * 32, dtype=torch.uint8, device="cuda")

        def job(k):
            eng.bind_iq_device(dev.data_ptr(), nb * n)
            eng.acquire_grid_device(nb, 1, prn, dop, _native.NON_COHERENT, rec_dev.data_ptr())

        job(0)
        t0 = time.perf_counter()
        ms = g.timed(job, 2, first=1) / 2
        t1 = time.perf_counter()

        per_launch = 24  # what the 512 MB spectra scratch holds at this rate (21 MB per block)

        def part(k):  # per-kernel timing on a slice (event-bracketed launches)
            eng.bind_iq_device(dev.data_ptr() + (k % 10) * 2 * per_launch * n * 8, 2 * per_launch * n)
            eng.acquire_grid_device(2 * per_launch, 1, prn, dop, _native.NON_COHERENT, rec_dev.data_ptr())

        spec_ms, spec_n, corr_ms, corr_n = kernel_times(eng, part, 3)
        blocks_per_launch = 2 * per_launch * 3 / max(corr_n, 1)
        # host to host: pipelined batches (41 x 24 blocks + one of 16)
        bb, rem = per_launch, nb % per_launch
        gs = _native.GridStream(eng, bb, 1, prn, dop, _native.NON_COHERENT, depth=3)
        gs_rem = _native.GridStream(eng, rem, 1, prn, dop, _native.NON_COHERENT, depth=1) if rem else None
        outs = [torch.empty(bb * n_cells * 32, dtype=torch.uint8).pin_memory() for _ in range(3)]
        outs_np = [o_.numpy().view(_native.RECORD_DTYPE).reshape(bb, N_PRN, len(dop)) for o_ in outs]
        out_rem = np.empty((max(rem, 1), N_PRN, len(dop)), dtype=_native.RECORD_DTYPE)

        def e2e_job(k):
            for j in range(nb // bb):
                if gs.in_flight == 3:
                    gs.collect()
                gs.submit(host.data_ptr() + j * bb * n * 8, outs_np[j % 3])
            while gs.in_flight:
                gs.collect()
            if gs_rem is not None:
                gs_rem.submit(host.data_ptr() + (nb - rem) * n * 8, out_rem)
                gs_rem.collect()

        e2e_job(0)
        sec = g.wall(e2e_job, 2, first=1) / 2
        gs.close()
        if gs_rem is not None:
            gs_rem.close()
        x2 = host.numpy()[:2]
        ref, cpu_sec = cpu.grid(x2, fs, n, DOPPLERS_81)
        eng.upload_iq(x2.reshape(-1))
        got = eng.acquire_grid(2, 1, prn, dop, _native.NON_COHERENT)
        cells = check_records(got, ref, x2, fs, n, DOPPLERS_81, "config 5")
        alg = alg_bytes(n, len(dop), 1, 1) * blocks_per_launch
        res.update({
            "value": nb * n / (ms * 1e-3) / 1e6, "device_ms_per_job": ms,
            "e2e": {"value": nb * n / sec / 1e6, "unit": "Msamples/s", "h2d_bytes_per_job": nb * n * 8, "d2h_bytes_per_job": nb * n_cells * 32,
                    "seconds_per_job": sec, "api": f"GridStream, batches of {bb} blocks, depth 3"},
            "roofline": {"bound": "hbm", "kernel": "k_correlate_w2048 (16 polyphase branches per cell)", "achieved": alg / (corr_ms * 1e-3) / 1e9,
                         "peak": peak_gbs, "unit": "GB/s", "frac": alg / (corr_ms * 1e-3) / 1e9 / peak_gbs,
                         "algorithmic_bytes_per_launch": alg, "blocks_per_launch": blocks_per_launch, "kernel_ms_per_launch": corr_ms,
                         "other_kernels_ms_per_launch": {"k_doppler_spectra": spec_ms}, "traffic": traffic_for("config5_correlate_dram_bytes_per_launch")},
            "cpu_baseline": {"value": 2 * n / cpu_sec / 1e6, "unit": "Msamples/s", "cores": cpu.cores, "kind": "port",
                             "sample": "2 of the 1000 blocks, full 32x81 grid, cells over all cores (the job's CPU time is this x 500, extrapolated)"},
            "parity_checked_cells": cells, "l2": "job input 125 MiB (~L2); 509 MB of spectra scratch written and re-read per 24-block launch pair (far beyond L2)",
            "clocks": sampler.window(t0, t1) if sampler else None})
    else:
        from gypsum_b200.distributed import ShardedBlockSearch

        search = ShardedBlockSearch(eng, torch.device("cuda", g.local_rank))
        flat = host.numpy().reshape(-1) if g.rank == 0 else None
        out = {}
        for key, mode in (("per_cell", None), ("best_bin", "best")):
            got = [None]

            def job(k):
                got[0] = search.acquire_blocks(flat, nb, 1, prn, dop, _native.NON_COHERENT, reduce=mode, copy=False)

            job(0)
            sec = g.wall(job, 3, first=1) / 3
            if g.rank == 0:
                r = got[0]
                if mode is None:
                    for b in (0, nb // 2, nb - 1):
                        assert int(r["argmax"][b, 24, int(np.argmax(r["peak"][b, 24]))]) == 16367
                else:
                    assert (r["doppler"][nb - 1, 24], r["code_phase"][nb - 1, 24]) == (1500.0, 16367)
            out[key] = {"value": nb * n / sec / 1e6, "seconds_per_job": sec, **search.last_bytes}
        pc = out["per_cell"]
        res.update({"scaling": "strong", "value": pc["value"],
                    "e2e": {"value": pc["value"], "unit": "Msamples/s", "seconds_per_job": pc["seconds_per_job"],
                            "h2d_bytes_per_job": pc["h2d"], "d2h_bytes_per_job": pc["d2h"],
                            "nccl_scatter_bytes": pc["scatter"], "nccl_gather_bytes": pc["gather"],
                            "api": "ShardedBlockSearch: rank-0 host -> one scatter -> grid per rank -> one gather -> rank-0 host"},
                    "with_on_device_best_bin_reduction": out["best_bin"],
                    "note": "fixed 1000-block job; compare `value` across N for strong-scaling efficiency; the N = 1 figure is configs.config5.e2e of the 1-GPU run"})
    eng.close()
    return res


def bench_config4(g, cpu, peak_gbs, sampler) -> dict:
    """32-channel E/P/L tracking over 60 s of streaming IQ @ 2.046 Msps."""
    from gypsum_b200 import _native
    from gypsum_b200 import synth
    from gypsum_b200.antenna_sample_provider import AntennaSampleChunk, SampleProviderAttributes
    from gypsum_b200.gps_ca_prn_codes import GpsSatelliteId, generate_replica_prn_signals
    from gypsum_b200.satellite import GpsSatellite
    from gypsum_b200.tracker import GpsSatelliteTracker, GpsSatelliteTrackingParameters, TrackerBank

    torch = g.torch
    n, fs, n_ch, n_ms = 2046, 2046000, 32, 60000
    chans = [(sv, 1000.0 + 37.3 * sv, 0.0, (53 * sv) % n, 0.1 * sv, 0.004) for sv in range(1, n_ch + 1)]
    base_ms = 1000
    base = synth.synth_tracking_iq(5, n, base_ms, fs, chans)
    host = torch.empty(n_ms * n * 2, dtype=torch.float32).pin_memory()
    x = host.numpy().view(np.complex64)
    for k in range(n_ms // base_ms):  # periodic stream: the noise repeats every second, which tracking does not care about
        x[k * base_ms * n:(k + 1) * base_ms * n] = base
    times = np.array([round(k * n / fs, 6) for k in range(n_ms)])
    eng = g.engine(fs, n)
    seeds = ([c[0] - 1 for c in chans], [c[1] for c in chans], [0.0] * n_ch, [c[3] for c in chans])
    dev = host.to("cuda")
    out = torch.empty(n_ch * n_ms * _native.TRACK_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    trk = _native.Tracker(eng, *seeds)
    eng.bind_iq_device(dev.data_ptr(), n_ms * n)
    trk.process_device(200, times[:200], out.data_ptr())  # warm-up
    trk.close()
    trk = _native.Tracker(eng, *seeds)
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g.barrier()
    e0.record(g.stream)
    trk.process_device(n_ms, times, out.data_ptr())
    e1.record(g.stream)
    g.barrier()
    dev_s = e0.elapsed_time(e1) * 1e-3
    t1 = time.perf_counter()
    rec = out.cpu().numpy().view(_native.TRACK_DTYPE).reshape(n_ch, n_ms)
    locked = float(rec["locked"][:, -1000:].mean())
    lost = int((rec["lost"] > 0).any(axis=1).sum())
    trk.close()
    # capacity: one channel per SM on the same stream (every satellite tracked by 4-5 channels), 10 s
    n_cap, cap_ms = int(torch.cuda.get_device_properties(g.local_rank).multi_processor_count), 10000
    cap_seeds = ([chans[i % n_ch][0] - 1 for i in range(n_cap)], [chans[i % n_ch][1] for i in range(n_cap)], [0.0] * n_cap,
                 [chans[i % n_ch][3] for i in range(n_cap)])
    out_cap = torch.empty(n_cap * cap_ms * _native.TRACK_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    trk = _native.Tracker(eng, *cap_seeds)
    trk.process_device(200, times[:200], out_cap.data_ptr())
    trk.close()
    trk = _native.Tracker(eng, *cap_seeds)
    g.barrier()
    e0.record(g.stream)
    trk.process_device(cap_ms, times[:cap_ms], out_cap.data_ptr())
    e1.record(g.stream)
    g.barrier()
    cap_s = e0.elapsed_time(e1) * 1e-3
    cap_rec = out_cap.cpu().numpy().view(_native.TRACK_DTYPE).reshape(n_cap, cap_ms)
    assert np.array_equal(cap_rec["symbol"][:n_ch], rec["symbol"][:, :cap_ms])  # a channel's result does not depend on its neighbours
    trk.close()
    del dev, out, out_cap, cap_rec
    # host to host: the whole stream from pinned host memory, records back
    trk = _native.Tracker(eng, *seeds)
    g.barrier()
    t2 = time.perf_counter()
    eng.upload_iq_ptr(host.data_ptr(), n_ms * n)
    rec2 = trk.process(n_ms, times)
    e2e_s = time.perf_counter() - t2
    bits_t = time.perf_counter()
    bits = trk.integrate_bits(n_ms, times, times + n / fs)
    bits_s = time.perf_counter() - bits_t
    assert np.array_equal(rec2["symbol"], rec["symbol"])
    trk.close()
    # the drop-in path: 32 GpsSatelliteTracker objects, one process_samples call per object per millisecond
    attrs = SampleProviderAttributes(fs, n)
    codes = generate_replica_prn_signals()
    objs = []
    for c in chans:
        sat = GpsSatellite(GpsSatelliteId(c[0]), codes[GpsSatelliteId(c[0])], 2)
        p = GpsSatelliteTrackingParameters(satellite=sat, current_doppler_shift=c[1], current_carrier_wave_phase_shift=0.0,
                                           current_prn_code_phase_shift=c[3], doppler_shifts=[])
        objs.append(GpsSatelliteTracker(p, attrs, keep_correlation_profiles=False))
    drop_ms = 1500
    for phase, lo, hi in (("warm", 0, 100), ("timed", 100, 100 + drop_ms)):
        tt = time.perf_counter()
        for k in range(lo, hi):
            chunk = AntennaSampleChunk(times[k], round((k + 1) * n / fs, 6), x[k * n:(k + 1) * n])
            for o_ in objs:
                o_.process_samples(chunk)
        drop_s = time.perf_counter() - tt
    drop_sym = np.array([[1 if s > 0 else -1 for s in (v.real for v in list(o_.tracking_params.correlation_peaks_rolling_buffer))] for o_ in objs])
    for o_ in objs:
        o_.close()
    # CPU: the tracker oracle, 4 channels x 2 s, one process per channel
    cpu_ms = 2000
    tcpu = time.perf_counter()
    cpu.pool.map(_cpu_track_worker, [(x[: cpu_ms * n], chans[i], (chans[i][1], 0.0, chans[i][3]), fs, n, cpu_ms) for i in range(4)])
    cpu_s = time.perf_counter() - tcpu
    alg = n_ch * n_ms * 16 * n + n_ch * n_ms * _native.TRACK_DTYPE.itemsize
    res = {"workload": "config4: 32-channel E/P/L tracking loop, 60 s of streaming IQ @ 2.046 Msps",
           "value": n_ms * n / dev_s / 1e6, "unit": "Msamples/s (stream samples; every sample is consumed by 32 channels)",
           "device_seconds": dev_s, "realtime_factor": (n_ms / 1000) / dev_s, "channel_ms_per_s": n_ch * n_ms / dev_s,
           "us_per_stream_ms": dev_s / n_ms * 1e6, "locked_fraction_last_second": locked, "lost_channels": lost,
           "e2e": {"value": n_ms * n / e2e_s / 1e6, "unit": "Msamples/s", "seconds": e2e_s, "realtime_factor": (n_ms / 1000) / e2e_s,
                   "h2d_bytes": n_ms * n * 8, "d2h_bytes": n_ch * n_ms * _native.TRACK_DTYPE.itemsize,
                   "api": "gb200_upload_iq + gb200_tracker_process: 60 s of pinned host IQ in, 1.92 M millisecond records out, one launch"},
           "capacity": {"channels": n_cap, "stream_ms": cap_ms, "device_seconds": cap_s, "us_per_stream_ms": cap_s / cap_ms * 1e6,
                        "channel_ms_per_s": n_cap * cap_ms / cap_s, "realtime_factor": (cap_ms / 1000) / cap_s,
                        "note": "one persistent CTA per SM: the per-millisecond latency is the same with every SM busy, so a GPU tracks 148 channels at the 32-channel rate"},
           "navigation_bits": {"seconds": bits_s, "bits": int(sum(len(b) for b in bits))},
           "drop_in_per_ms": {"api": "32 GpsSatelliteTracker.process_samples calls per millisecond (one pooled launch per millisecond)",
                              "ms_timed": drop_ms, "us_per_stream_ms": drop_s / drop_ms * 1e6, "realtime_factor": (drop_ms / 1000) / drop_s,
                              "symbols_equal_bank": bool(np.array_equal(drop_sym[:, -1000:], rec["symbol"][:, 100 + drop_ms - 1000:100 + drop_ms]))},
           "roofline": {"bound": "hbm", "kernel": "k_track_channels<2> (one persistent CTA per channel; feedback makes time sequential)",
                        "achieved": alg / dev_s / 1e9, "peak": peak_gbs, "unit": "GB/s", "frac": alg / dev_s / 1e9 / peak_gbs,
                        "algorithmic_bytes": alg, "note": "latency-bound by construction: 60,000 dependent steps per channel on 32 of 148 SMs; the figure that matters is us per stream-ms"},
           "cpu_baseline": {"value": 4 * cpu_ms / cpu_s / 1000, "unit": "channel-seconds per second (4 processes)", "cores": 4, "kind": "port",
                            "channel_ms_per_s": 4 * cpu_ms / cpu_s, "sample": "TrackerOracle, 4 of the 32 channels x the first 2 s of the same stream, one process per channel"},
           "clocks": sampler.window(t0, t1) if sampler else None}
    eng.close()
    return res


def bench_detector(g, cpu, sampler) -> dict:
    """The receiver's real acquisition scan (receiver.py:219-224): GpsSatelliteDetector.detect_satellites_in_antenna_data for all
    32 satellites over a 10-ms window -- per satellite ten refinement passes (222 Doppler bins, acquisition.py:70-152) and one
    coherent integration -- through the drop-in class, host array in, result objects out."""
    from gypsum_b200 import synth
    from gypsum_b200.acquisition import GpsSatelliteDetector
    from gypsum_b200.antenna_sample_provider import AntennaSampleChunk, DeviceSampleRing, SampleProviderAttributes
    from gypsum_b200.gps_ca_prn_codes import GpsSatelliteId, generate_replica_prn_signals
    from gypsum_b200.satellite import GpsSatellite

    attrs = SampleProviderAttributes(FS, N)
    planted = [(25, 1504.0, 777, 0.3, 0.12), (3, -3250.0, 5, 1.0, 0.1), (32, 4875.5, 2045, 2.5, 0.15)]
    x = synth.synth_iq(7, N, 10, FS, planted)
    codes = generate_replica_prn_signals()
    det = GpsSatelliteDetector({sid: GpsSatellite(sid, c, 2) for sid, c in codes.items()})
    ids = [GpsSatelliteId(i) for i in range(1, 33)]
    for _ in range(3):
        found = det.detect_satellites_in_antenna_data(ids, x, attrs)
    t0 = time.perf_counter()
    reps = 50
    for _ in range(reps):
        found = det.detect_satellites_in_antenna_data(ids, x, attrs)
    sec = (time.perf_counter() - t0) / reps
    t1 = time.perf_counter()
    # the same scan with the window already on the device (DeviceSampleRing: one upload per millisecond, none per scan)
    ring = DeviceSampleRing(attrs, 10)
    for k in range(10):
        ring.append(AntennaSampleChunk(k * 0.001, (k + 1) * 0.001, x[k * N:(k + 1) * N]))
    det.detect_satellites_in_antenna_data(ids, ring.window(), attrs)
    t2 = time.perf_counter()
    for _ in range(reps):
        found_ring = det.detect_satellites_in_antenna_data(ids, ring.window(), attrs)
    sec_ring = (time.perf_counter() - t2) / reps
    ring.native.close()
    all_results = {r.satellite_id.id: r for r in det._acquire_many(ids, x, attrs)}
    # CPU: the oracle's acquire_sv for every satellite, one process per satellite at a time over the pool
    tc = time.perf_counter()
    cpu_res = {sv: (d, c, st) for sv, d, c, st in cpu.pool.map(_cpu_acquire_worker, [(x, FS, N, sv) for sv in range(1, 33)], chunksize=1)}
    cpu_sec = time.perf_counter() - tc
    detected = sorted(r.satellite_id.id for r in found)
    assert detected == sorted(sv for sv, v in cpu_res.items() if v[2] > 3) == sorted(r.satellite_id.id for r in found_ring)
    for sv in detected:  # detected satellites: the reference's (Doppler, code phase) exactly, strength to 1e-4
        r = all_results[sv]
        assert (r.doppler_shift, r.prn_phase_shift) == cpu_res[sv][:2], sv
        assert abs(r.correlation_strength - cpu_res[sv][2]) <= 1e-4 * cpu_res[sv][2], sv
    same = sum((all_results[sv].doppler_shift, all_results[sv].prn_phase_shift) == cpu_res[sv][:2] for sv in range(1, 33))
    cell_ms = 32 * 223 * 10
    return {"workload": "real detector: 32 satellites x (222 non-coherent bins in 10 passes + 1 coherent) x 10 ms @ 2.046 Msps",
            "seconds_per_scan": sec, "scans_per_second": 1.0 / sec, "cell_ms_per_second": cell_ms / sec,
            "value": 10 * N / sec / 1e6, "unit": "Msamples/s (the 10-ms window per scan)",
            "e2e": {"value": 10 * N / sec / 1e6, "unit": "Msamples/s", "h2d_bytes_per_scan": 10 * N * 8, "d2h_bytes_per_scan": 32 * 32,
                    "api": "GpsSatelliteDetector.detect_satellites_in_antenna_data(ids, ndarray, attrs): upload + gb200_detect (all passes on the device)"},
            "from_device_ring": {"seconds_per_scan": sec_ring, "note": "window read in place from DeviceSampleRing (no upload in the scan)"},
            "detected": detected, "satellites_identical_to_cpu_reference": same,
            "parity": "detected satellites: (Doppler, code phase) exact, strength 1e-4; noise-only satellites may take another branch of the search at float64 near-ties (tests prove those per satellite)",
            "cpu_baseline": {"seconds_per_scan": cpu_sec, "cores": cpu.cores, "kind": "port", "value": 10 * N / cpu_sec / 1e6, "unit": "Msamples/s",
                             "sample": "oracle acquire_sv for all 32 satellites, one satellite per process"},
            "clocks": sampler.window(t0, t1) if sampler else None}


def bench_sharded_single_block(g) -> dict:
    """north_star's literal shape for ONE 1-ms block: broadcast the IQ block, every rank searches its PRN rows, all-gather
    the per-cell records.  Reported because it is SLOWER than one GPU (two collectives around ~30 us of work)."""
    from gypsum_b200 import _native
    from gypsum_b200.distributed import ShardedGridSearch

    torch = g.torch
    eng = g.engine(FS, N)
    search = ShardedGridSearch(eng, torch.device("cuda", g.local_rank))
    x = make_ring(1, seed=9)[0] if g.rank == 0 else None
    prn = np.arange(N_PRN, dtype=np.int32)
    got = [None]

    def call(k):
        got[0] = search.acquire_grid(x, 1, 1, prn, DOPPLERS, _native.NON_COHERENT)

    for k in range(5):
        call(k)
    sec = g.wall(call, 100, first=5) / 100
    full = got[0]
    assert int(full["argmax"][0, 24, int(np.argmax(full["peak"][0, 24]))]) == 777
    eng.close()
    return {"workload": "config 2, ONE 1-ms block, PRN rows sharded over the ranks", "us_per_block": sec * 1e6,
            "Msamples_per_s": N / sec / 1e6, "api": "ShardedGridSearch: NCCL broadcast of 16 KB + all-gather of 42 KB",
            "note": "compare single_block.e2e_us_per_block of the 1-GPU line: sharding one short block over GPUs loses to one GPU"}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--blocks-per-call", type=int, default=256)
    ap.add_argument("--calls-per-step", type=int, default=12)
    ap.add_argument("--ring-blocks", type=int, default=0)
    ap.add_argument("--cpu-blocks", type=int, default=4)
    ap.add_argument("--cpu-blocks-per-step", type=int, default=8)
    ap.add_argument("--no-configs", action="store_true", help="skip the config 3 / 4 / 5 sub-lines")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's per-cell records of the last timed step to DIR/<field>.npy (see dump_outputs)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
