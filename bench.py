#!/usr/bin/env python3
"""bench.py — HBM scrub-and-verify throughput of the CC-transition hot path on B200.

Contract (driver):  python bench.py --gpus N --steps K --warmup W      [--impl reference]
  N>1 is launched by the driver as torchrun with one rank per GPU (NCCL is used ONLY
  for the barrier and the max/sum/gather of the timings: the path is per-GPU independent,
  no data-path collective — SURVEY.md §8e).

A "step" = one pass of the hot path over one region: the scrub kernel zero-fills
every byte of the arena, then the verify kernel reads it back and counts non-zero
bytes.  Workload = BASELINE.json configs[1]: one B200, all the HBM a CUDA context can
map (~190.8 GB of 191.5 GB), poisoned with 0xA5 before the first step.

  value     whole-job GB/s with the region resident in HBM: (bytes zeroed + bytes read
            back) over all ranks / max-over-ranks CUDA-event time of the K steps.
  e2e       the same metric through the public API a manager calls
            (k8s_cc_manager_b200.devices.Gpu.scrub_and_verify -> ccm_scrub_verify): a COLD
            call maps all free HBM, scrubs and reads back chunk by chunk, copies the 8-byte
            count to the host and hands the HBM back.  >= 15 calls; every call starts on a
            barrier over the ranks.  `value` counts the WHOLE cycle (call -> HBM back with
            the driver); `verdict_s` is the part a transition waits for (the release runs on
            libccm's reaper thread, off the critical path).  Median / p10 / p90 over calls of
            the max over ranks.  No host-resident input exists on this path (it takes a device
            index): h2d_bytes_per_step = 0, d2h_bytes_per_step = 8.
  roofline  scrub kernel (HBM write bound): R bytes / mean CUDA-event duration of the scrub
            launches inside the timed region, vs MEASURED_PEAKS.json hbm_gbs; plus the
            library write bar (cudaMemsetAsync) and a library read-only pass (torch sum)
            timed in the SAME run.
  checks    hardware proof at every N: k = 7 bytes injected at seeded offsets (first, last,
            unaligned) are counted exactly, on every rank; after the ranks are done, ONE process
            drives all N GPUs through the concurrent launcher (clean + coverage + a dirt drill).
  transition  BASELINE metric 1 at every N: CCManager.set_cc_mode off->on->devtools->off,
            eviction-gated, on the first N GPUs from one process — once with the daemon's
            defaults (CUDA contexts released after every gate) and once with contexts kept;
            constructed baselines B1/B2 (BASELINE.md §3) in the same run.
  cpu_baseline  the oracle's C port (memset + byte-wise count) on the box's host cores,
            NUMA-local first touch, pinned threads.

Other modes:  --sweep  region sweep 1 GB -> max (BASELINE configs[4]) on this rank's GPU.

--dump-outputs DIR  after the timed steps, runs the step once more on a seeded dirty input and
            writes what it computed to DIR as .npy (see dump_outputs), so that two builds can be
            compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "HBM scrub-and-verify throughput (bytes zeroed + bytes read back per second, whole job)"
UNIT = "GB/s"
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
DATASHEET_HBM_GBS = 8000.0  # HBM3e nominal, B200


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy, read+write)"
        except Exception:  # noqa: BLE001
            pass
    return FALLBACK_HBM_GBS, "fallback 6.65 TB/s (B200_PROFILING.md)"


def pct(xs, q):
    xs = sorted(xs)
    return xs[min(len(xs) - 1, max(0, round(q * (len(xs) - 1))))] if xs else float("nan")


def stats(xs):
    return {"median": statistics.median(xs), "p10": pct(xs, 0.1), "p90": pct(xs, 0.9), "min": min(xs), "max": max(xs),
            "n": len(xs)}


# ------------------------------------------------------------------ clock sampler
class ClockSampler:
    """Samples SM clock + throttle reasons of one GPU during the timed region (NVML)."""

    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int, period_s: float = 0.02):
        self.index, self.period = index, period_s
        self.samples, self.reason_bits = [], 0
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self.error = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception as exc:  # noqa: BLE001
            self.error = f"nvml unavailable: {exc}"
            return self
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def _run(self):
        nv = self._nvml
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
            except Exception as exc:  # noqa: BLE001
                self.error = str(exc)
                return
            self._stop.wait(self.period)

    def stop(self) -> dict:
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=2)
        reasons = [name for bit, name in self.REASONS.items() if self.reason_bits & bit and name != "gpu_idle"]
        out = {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
               "reasons": reasons, "samples": len(self.samples)}
        if self.error:
            out["error"] = self.error
        return out


# ------------------------------------------------------------------- CPU baseline
def host_threads() -> int:
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_arm(sample_gib: float, passes: int, warm: int, probe: bool = False):
    """oracle/scrub_oracle.c (scrub + byte-wise non-zero count) on the host cores — the ONLY place
    bench.py executes oracle code, and only as the baseline.  The baseline gets every help a careful CPU
    implementation would take (a straw man inflates the headline ratio — VERDICT r1 weak #3): a
    persistent pool, thread i pinned to the i-th allowed CPU, first-touching and then streaming its OWN
    slice (NUMA-local; round 1 first-touched from one thread: 26 GB/s on one box, 112 on another), and the
    faster of {libc memset, non-temporal stores} x {all hardware threads, one per core} picked in the
    untimed warm-up."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import numpy as np
    import scrub_oracle as SO

    hw = host_threads()
    nbytes = int(sample_gib * 2**30)
    buf = np.empty(nbytes, dtype=np.uint8)
    candidates = []
    for threads in sorted({hw, max(1, hw // 2)}, reverse=True):
        with SO.Pool(buf, threads, pin=True) as pool:
            assert pool.poison() == nbytes                              # parallel first touch (untimed)
            for stream in (False, True):
                assert pool.scrub_verify(stream) == 0
                ts = []
                for _ in range(max(2, warm)):
                    t0 = time.perf_counter()
                    assert pool.scrub_verify(stream) == 0
                    ts.append(time.perf_counter() - t0)
                candidates.append({"threads": threads, "scrub": "nt-stores" if stream else "memset",
                                   "gbs_best": 2.0 * nbytes / min(ts) / 1e9, "gbs_median": 2.0 * nbytes / statistics.median(ts) / 1e9})
    pick = max(candidates, key=lambda c: c["gbs_median"])
    threads, stream = pick["threads"], pick["scrub"] == "nt-stores"
    with SO.Pool(buf, threads, pin=True) as pool:
        assert pool.poison() == nbytes                                  # slices re-touched by THESE threads
        assert pool.scrub_verify(stream) == 0
        times = []
        for _ in range(passes):
            t0 = time.perf_counter()
            nz = pool.scrub_verify(stream)
            times.append(time.perf_counter() - t0)
            assert nz == 0
    rates = [2.0 * nbytes / t / 1e9 for t in times]
    sample = (f"{sample_gib:g} GiB host buffer, {passes} timed passes of scrub ({pick['scrub']}) + byte-wise count on a "
              f"persistent pool of {threads} pinned pthreads (of {hw} hardware threads), each first-touching and then "
              f"streaming its own slice (oracle/scrub_oracle.c; the reference has no scrub to time); {SO.numa_layout()}")
    out = {"value": 2.0 * nbytes * passes / sum(times) / 1e9, "best": max(rates), "median": statistics.median(rates),
           "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "seconds": sum(times),
           "bytes_per_pass": nbytes, "passes": passes, "tuning": candidates}
    if probe:
        print(json.dumps(out), flush=True)
    return out


def run_reference_arm(args):
    """--impl reference: the CPU statement of the path on the host cores (the reference
    itself has no implementation of it — SURVEY.md §0 — and no compilable sources for
    an oracle/_ref, so this is the oracle port, kind='port')."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_arm(args.cpu_sample_gib, passes=args.steps, warm=max(1, args.warmup))
    value = cb["value"]
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["seconds"] / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": "configs[1] CPU statement: scrub + read-back verify of a host buffer",
                       "sample": cb["sample"], "same_config": False,
                       "note": f"bounded sample: {args.cpu_sample_gib:g} GiB per step instead of the GPU arm's ~190.8 GB per GPU "
                               "(a bandwidth-bound loop: GB/s does not depend on the length)"},
            "cpu_baseline": {k: cb[k] for k in ("value", "best", "median", "unit", "cores", "kind", "sample", "tuning")},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------- our arm
def check(rc, what):
    from k8s_cc_manager_b200 import _native as N
    if rc != 0:
        raise RuntimeError(f"{what}: {N.strerror(rc)}: {N.last_error()}")


def injected_count_check(L, N, dev, R, vv, sptr):
    """k = 7 bytes at seeded offsets — first byte, last byte, one non-16-aligned offset, four random
    ones — must be counted exactly; after a scrub the count is 0 again (tests/test_scrub_gpu.py
    :134-163 at full size, on every rank)."""
    import numpy as np
    rng = np.random.default_rng(1234 + dev)
    offs = {0, R - 1, 16 * 1000 + 3}
    while len(offs) < 7:
        offs.add(int(rng.integers(0, R)))
    nz = C.c_uint64()
    for o in sorted(offs):
        check(L.ccm_arena_write(dev, o, (C.c_uint8 * 1)(int(rng.integers(1, 256))), 1), "arena_write")
    check(L.ccm_arena_verify(dev, vv, None, sptr, C.byref(nz), None), "verify injected")
    found = nz.value
    check(L.ccm_arena_scrub(dev, N.SCRUB_AUTO, None, sptr, None), "scrub")
    check(L.ccm_arena_verify(dev, vv, None, sptr, C.byref(nz), None), "verify after scrub")
    ok = found == 7 and nz.value == 0
    if not ok:
        raise RuntimeError(f"injected 7 bytes, verify counted {found}; after scrub {nz.value}")
    return {"injected": 7, "counted": found, "after_scrub": nz.value, "offsets_include": ["first byte", "last byte", "unaligned"]}


DUMP_WINDOWS, DUMP_WINDOW_BYTES, DUMP_SEED = 64, 16 << 10, 42


def dump_outputs(L, dev, R, vv, sptr, step, out_dir, rank=None):
    """Runs the timed step once more on a seeded input and writes what it computed to out_dir.

    A correct step always ends with a zeroed arena and a count of 0, so the timed steps' own results
    cannot tell a verify kernel that counts from one that always says 0.  The step is therefore given
    dirt it must see: the arena is filled with the seeded xorshift pattern (ccm_arena_fill_random,
    seed 42; the same arguments give the same input on every run), counted with the step's verify
    kernel, and then scrubbed and verified by the timed call itself.  Files (.npy):
      input_nonzero_bytes  non-zero bytes the verify kernel counts in the seeded input (float64)
      nonzero_bytes        the count the step hands its caller (ccm_arena_fetch_count; float64)
      arena_sample         the scrubbed arena, float32, one row per window: the first and last
                           16 KiB and 64 windows of 16 KiB at offsets drawn with seed 0
    Under torchrun every rank writes its own files, suffixed _rank<r>."""
    import numpy as np
    nz = C.c_uint64()
    check(L.ccm_arena_fill_random(dev, DUMP_SEED, sptr), "fill seeded input")
    check(L.ccm_arena_verify(dev, vv, None, sptr, C.byref(nz), None), "verify seeded input")
    dirty = nz.value
    step()
    check(L.ccm_arena_fetch_count(dev, sptr, C.byref(nz)), "fetch_count")
    if dirty == 0 or nz.value != 0:
        raise RuntimeError(f"seeded input counted {dirty} non-zero bytes, {nz.value} after the step")
    w = min(DUMP_WINDOW_BYTES, R)
    rng = np.random.default_rng(0)
    offsets = [0, R - w] + sorted(int(x) for x in rng.integers(0, R - w + 1, size=DUMP_WINDOWS))
    sample = np.empty((len(offsets), w), dtype=np.uint8)
    for row, off in zip(sample, offsets):
        check(L.ccm_arena_read(dev, off, row.ctypes.data, w), "arena_read")
    suffix = "" if rank is None else f"_rank{rank}"
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / f"input_nonzero_bytes{suffix}.npy", np.array([dirty], dtype=np.float64))
    np.save(out_dir / f"nonzero_bytes{suffix}.npy", np.array([nz.value], dtype=np.float64))
    np.save(out_dir / f"arena_sample{suffix}.npy", sample.astype(np.float32))


def run_ours(args):
    import torch

    from k8s_cc_manager_b200 import _native as N
    from k8s_cc_manager_b200 import devices as D
    from k8s_cc_manager_b200.aggregate import aggregate_cold_calls, aggregate_job, gather_rows as gather_rows_

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the scrub path has no host fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(x, op):
        if not dist:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
        return float(t.item())

    def gather_rows(rows):
        return gather_rows_(dist, "cuda", rows)

    if dist:
        # NCCL allocates its communicator buffers lazily: touch every collective used below
        # BEFORE the arena takes all free HBM, and leave it headroom.
        barrier()
        reduce(0.0, "MAX")
        reduce(0.0, "SUM")
        gather_rows([[0.0, 0.0]])
        os.environ.setdefault("CCM_ARENA_RESERVE_MB", "1024")

    L = N.lib()
    check(L.ccm_init(N.BACKEND_CUDASIM), "ccm_init")
    dev = local
    sv = N.SCRUB_VARIANTS[args.scrub]
    vv = N.VERIFY_VARIANTS[args.verify]
    k_scrub, k_verify = N.default_kernels()

    # ---- resident region: everything the context can map (or --gib) -------------------
    ai = N.ArenaInfo()
    check(L.ccm_arena_acquire(dev, int(args.gib * 2**30) if args.gib > 0 else 0, C.byref(ai)), "arena_acquire")
    R = int(ai.bytes)
    # A dedicated non-default stream: its handle is what the C ABI launches on (a NULL
    # handle would mean "the library's own stream"), and the torch events below are
    # recorded on the same stream, so they bracket exactly these kernels.
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sptr = C.c_void_p(stream.cuda_stream)
    assert stream.cuda_stream != 0
    nz = C.c_uint64()
    check(L.ccm_arena_fill(dev, 0xA5, sptr), "poison")          # untimed: pre-scrub content
    check(L.ccm_arena_verify(dev, vv, None, sptr, C.byref(nz), None), "verify poison")
    if nz.value != R:
        raise RuntimeError(f"poisoned arena must read back {R} non-zero bytes, got {nz.value}")
    checks = {"poison_counted": nz.value == R}
    check(L.ccm_arena_scrub(dev, sv, None, sptr, None), "scrub")
    checks["injection"] = injected_count_check(L, N, dev, R, vv, sptr)
    check(L.ccm_arena_fill(dev, 0xA5, sptr), "re-poison")       # the timed steps start from dirty memory

    def step():
        check(L.ccm_arena_scrub_verify_async(dev, sv, vv, None, None, sptr), "scrub_verify_async")

    for _ in range(max(3, args.warmup)):
        step()
    check(L.ccm_arena_fetch_count(dev, sptr, C.byref(nz)), "fetch_count")
    if nz.value != 0:
        raise RuntimeError(f"scrub left {nz.value} non-zero bytes")
    L.ccm_arena_step_times(dev, 0, None, None, None)             # drop warm-up step events

    # ---- timed region: exactly K steps, device-timed, max over ranks ------------------
    sampler = ClockSampler(local).start()
    launches0 = L.ccm_kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    ms_local = e0.elapsed_time(e1)
    clocks = sampler.stop()
    launches = L.ccm_kernel_launches() - launches0
    check(L.ccm_arena_fetch_count(dev, sptr, C.byref(nz)), "fetch_count")   # D2H of the step result
    if nz.value != 0:
        raise RuntimeError(f"verify found {nz.value} non-zero bytes inside the timed region")
    s_ms, v_ms, nsteps = (C.c_float * 64)(), (C.c_float * 64)(), C.c_int()
    check(L.ccm_arena_step_times(dev, 64, s_ms, v_ms, C.byref(nsteps)), "step_times")
    scrub_ms = statistics.mean(s_ms[:nsteps.value]) if nsteps.value else float("nan")
    verify_ms = statistics.mean(v_ms[:nsteps.value]) if nsteps.value else float("nan")
    if args.dump_outputs:                                       # after the step times: its step is not timed
        dump_outputs(L, dev, R, vv, sptr, step, Path(args.dump_outputs), rank if world > 1 else None)

    # ---- same-run peaks: the library write bar over the same arena ... ------------------
    peaks = {}
    ms = C.c_float()
    best = 1e30
    for _ in range(4):
        check(L.ccm_arena_scrub(dev, N.SCRUB_MEMSET, None, sptr, C.byref(ms)), "memset pass")
        best = min(best, ms.value)
    peaks["peak_write_same_run"] = R / best / 1e6
    peaks["peak_write_how"] = "cudaMemsetAsync over the same arena, best of 4 (CUDA events)"
    check(L.ccm_arena_release(dev), "arena_release")
    # ... and a library read-only pass (torch reduction over 32 GiB, >> L2)
    try:
        n_read = min(32 << 30, R // 2) // 8
        t = torch.zeros(n_read, dtype=torch.int64, device="cuda")
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        best = 1e30
        for _ in range(4):
            a.record(stream)
            t.sum()
            b.record(stream)
            b.synchronize()
            best = min(best, a.elapsed_time(b))
        peaks["peak_read_same_run"] = n_read * 8 / best / 1e6
        peaks["peak_read_how"] = f"torch.sum over {n_read * 8 >> 30} GiB of int64 (library reduction kernel), best of 4"
        del t
    except Exception as exc:  # noqa: BLE001
        peaks["peak_read_error"] = str(exc)
    torch.cuda.empty_cache()

    agg = aggregate_job(dist, "cuda", region_bytes=R, steps=args.steps, elapsed_ms=ms_local, launches=launches)
    ms_total, value, total_launches = agg["ms"], agg["value_gbs"], agg["launches"]

    # ---- e2e: the public API, cold; every call starts on a barrier over the ranks -------
    gpu = [d for d in D.find_gpus()[0] if d.is_gpu()][dev]
    want = int(args.gib * 2**30) if args.gib > 0 else 0
    e2e_steps = max(1, args.e2e_steps)
    for _ in range(max(3, args.warmup)):                                     # same W as the kernel arm
        gpu.scrub_and_verify(want)
    gpu.wait_scrub_released()
    rows, reports = [], []
    barrier()
    t_loop = time.perf_counter()
    for _ in range(e2e_steps):
        barrier()
        t0 = time.perf_counter()
        rep = gpu.scrub_and_verify(want)                # returns with the verdict (8-byte count on the host)
        t1 = time.perf_counter()
        ms_rel, _waited = gpu.wait_scrub_released()     # HBM back with the driver
        t2 = time.perf_counter()
        reports.append(rep)
        rows.append([t1 - t0, t2 - t0, float(rep.bytes_scrubbed), rep.ms_acquire, rep.ms_gpu_span, rep.ms_scrub,
                     rep.ms_verify, ms_rel])
    barrier()
    loop_s = reduce(time.perf_counter() - t_loop, "MAX")
    all_rows = gather_rows(rows)                        # [rank][call][col]
    cold = aggregate_cold_calls(all_rows)
    verdict, cycle, e2e_value = cold["verdict_s_each"], cold["cycle_s_each"], cold["value_gbs"]
    phase_names = ["acquire_host_ms", "gpu_span_ms", "scrub_kernels_ms", "verify_kernels_ms", "release_ms"]
    phases = {name: {"median_of_max_over_ranks": statistics.median(
        max(all_rows[r][i][3 + j] for r in range(world)) for i in range(e2e_steps))}
        for j, name in enumerate(phase_names)}
    last = reports[-1]

    # ---- informational: the same kernels driven with a HOST buffer (ccm_host_roundtrip:
    # H2D of dirty bytes, count, scrub, count, D2H of the zeroed bytes).  Not how a manager
    # calls the path (it passes a device index, not a buffer) — reported so that a number
    # with host<->device copies inside the timed region exists too.  PCIe-bound by nature.
    host_rt = None
    if not args.no_host_roundtrip:
        hb = 1 << 30
        pinned = torch.empty(hb, dtype=torch.uint8, pin_memory=True)
        pre, post = C.c_uint64(), C.c_uint64()
        times = []
        for i in range(4):
            pinned.fill_(0xA5)
            t0 = time.perf_counter()
            check(L.ccm_host_roundtrip(dev, C.c_void_p(pinned.data_ptr()), hb, 0, sv, vv, C.byref(pre), C.byref(post)),
                  "host_roundtrip")
            dt = time.perf_counter() - t0
            if pre.value != hb or post.value != 0 or int(pinned[:4096].sum()) != 0:
                raise RuntimeError("host round trip returned wrong counts/bytes")
            if i:
                times.append(dt)
        host_rt = {"value": 2.0 * hb * len(times) / sum(times) / 1e9, "unit": UNIT, "h2d_bytes_per_step": hb,
                   "d2h_bytes_per_step": hb + 16, "steps": len(times), "seconds_per_step": sum(times) / len(times),
                   "api": "ccm_host_roundtrip (C ABI): pinned host buffer -> device -> count, scrub, count -> host",
                   "note": "PCIe-bound; informational — the manager's call takes no host buffer"}
        del pinned

    all_checks = gather_rows([[1.0 if checks["poison_counted"] else 0.0, float(checks["injection"]["counted"]),
                               float(checks["injection"]["after_scrub"])]])
    if dist:
        dist.destroy_process_group()
    if rank != 0:
        return                                            # the node leg needs the other GPUs idle

    peak, peak_src = measured_peak()
    # DRAM traffic per launch: from the committed ncu capture (never measured under this run), scaled to
    # this run's region size — and only if the capture is of the kernels this library launches today.
    traffic_s = traffic_v = None
    traffic_src = "profiles/traffic.json (ncu dram__bytes_read+write of one full-arena launch)"
    try:
        tr = json.loads((ROOT / "profiles" / "traffic.json").read_text())
        k = R / tr["region_bytes"]
        traffic_s = int(k * (tr["kernels"][k_scrub]["dram_bytes_read"] + tr["kernels"][k_scrub]["dram_bytes_write"]))
        traffic_v = int(k * (tr["kernels"][k_verify]["dram_bytes_read"] + tr["kernels"][k_verify]["dram_bytes_write"]))
    except KeyError:
        traffic_src = "profiles/traffic.json is STALE: it does not hold the kernels libccm launches now"
    except Exception:  # noqa: BLE001
        traffic_src = "profiles/traffic.json unreadable"
    scrub_gbs, verify_gbs = R / scrub_ms / 1e6, R / verify_ms / 1e6
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {
            "workload": "BASELINE configs[1]: B200 off->on transition scrub over all mappable HBM, "
                        "read-back verify all-zero (pre-scrub content: 0xA5 poison)",
            "region_bytes_per_gpu": R, "coverage_of_device_total": R / ai.device_total_bytes,
            "arena_segments": ai.segments, "scrub_variant": args.scrub, "verify_variant": args.verify,
            "l2": "no flush needed: region (>=190 GB) is >1000x the 126 MB L2; every step re-streams it",
            "parallelism": f"{world} independent GPU(s), one process per GPU, no data-path collective",
        },
        "per_gpu": {"scrub_gbs": scrub_gbs, "verify_gbs": verify_gbs, "scrub_ms": scrub_ms, "verify_ms": verify_ms,
                    "step_gbs": 2.0 * R * args.steps / ms_local / 1e6},
        "roofline": {"bound": "hbm", "kernel": f"{k_scrub} (HBM write)", "achieved": scrub_gbs,
                     "peak": peak, "unit": "GB/s", "frac": scrub_gbs / peak, "traffic": traffic_s,
                     "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": R, "note": "of measured" if "MEASURED" in peak_src else "of fallback",
                     **peaks,
                     "frac_vs_write_peak": scrub_gbs / peaks["peak_write_same_run"],
                     "frac_vs_datasheet": scrub_gbs / DATASHEET_HBM_GBS},
        "roofline_verify": {"bound": "hbm", "kernel": f"{k_verify} (HBM read)", "achieved": verify_gbs,
                            "peak": peak, "unit": "GB/s", "frac": verify_gbs / peak, "traffic": traffic_v,
                            "algorithmic_bytes_per_launch": R,
                            "frac_vs_read_peak": verify_gbs / peaks["peak_read_same_run"] if "peak_read_same_run" in peaks else None,
                            "frac_vs_datasheet": verify_gbs / DATASHEET_HBM_GBS},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 8,
                "steps": e2e_steps, "warmup": max(3, args.warmup),
                "seconds_per_step": statistics.median(cycle),
                "cycle_s": cold["cycle_s"], "verdict_s": cold["verdict_s"],
                "value_mean": cold["value_mean_gbs"], "verdict_value": cold["verdict_value_gbs"],
                "loop_wall_s": loop_s,
                "phases": phases,
                "ms_verdict_each_step": [round(x * 1e3, 2) for x in verdict],
                "ms_cycle_each_step": [round(x * 1e3, 2) for x in cycle],
                "breakdown_ms_last_step_rank0": {"acquire_host": last.ms_acquire, "gpu_span": last.ms_gpu_span,
                                                 "scrub_kernels": last.ms_scrub, "verify_kernels": last.ms_verify,
                                                 "to_verdict": last.ms_total, "chunks": last.segments,
                                                 "bytes_unreached": last.bytes_unreached, "coverage": last.coverage},
                "api": "k8s_cc_manager_b200.devices.Gpu.scrub_and_verify -> ccm_scrub_verify (C ABI); "
                       "Gpu.wait_scrub_released -> ccm_scrub_release_wait",
                "note": "value = 2 x bytes of one call (all ranks) / MEDIAN over calls of the max-over-ranks CYCLE time (call "
                        "start -> verdict -> HBM handed back; value_mean uses the sum instead); every call starts on a "
                        "barrier.  verdict_s is what a transition waits "
                        "for: the unmap/release runs on libccm's reaper thread.  Back-to-back cold calls are the "
                        "driver's worst case (it re-allocates memory it is still scrubbing after the last free).  "
                        "No host-resident input exists on this path."},
        "gpu_launches": total_launches,
        "clocks": clocks,
        "checks": {"per_rank": {"poison_counted": [bool(r[0][0]) for r in all_checks],
                                "injected_7_counted": [int(r[0][1]) for r in all_checks],
                                "after_scrub": [int(r[0][2]) for r in all_checks]},
                   "ok": all(r[0][0] == 1.0 and r[0][1] == 7.0 and r[0][2] == 0.0 for r in all_checks)},
    }
    if host_rt:
        line["e2e_host_buffers"] = host_rt
    if not args.no_node_leg:
        node = run_node_leg(world, args)
        for key in ("node_checks", "node_gate", "transition", "baselines"):
            if key in node:
                if key == "node_checks":
                    line["checks"]["node"] = node[key]
                    line["checks"]["ok"] = bool(line["checks"]["ok"] and node[key].get("ok"))
                else:
                    line[key] = node[key]
        if "error" in node:
            line["node_leg_error"] = node["error"]
    if world == 1 and not args.no_cpu_baseline:
        cb = cpu_arm(args.cpu_sample_gib, passes=args.cpu_passes, warm=2)
        line["cpu_baseline"] = cb
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------ node leg
def wait_for_idle_gpus(n, timeout_s=60.0):
    """The other ranks exit after the per-rank phases; wait until their processes are gone."""
    try:
        import pynvml
        pynvml.nvmlInit()
        me = os.getpid()
        deadline = time.time() + timeout_s
        while time.time() < deadline:
            busy = 0
            for i in range(n):
                h = pynvml.nvmlDeviceGetHandleByIndex(i)
                busy += sum(1 for p in pynvml.nvmlDeviceGetComputeRunningProcesses(h) if p.pid != me)
            if busy == 0:
                return True
            time.sleep(0.1)
        return False
    except Exception:  # noqa: BLE001
        time.sleep(3.0)
        return True


def run_node_leg(n_gpus, args):
    """ONE fresh process drives the first N GPUs (node-level checks, constructed baselines, the
    manager's transitions).  A subprocess, because the release-context policy resets CUDA primary
    contexts, which this process still shares with torch."""
    idle = wait_for_idle_gpus(n_gpus)
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "CCM_ARENA_RESERVE_MB"):
        env.pop(k, None)
    cmd = [sys.executable, str(ROOT / "bench.py"), "--node-leg", "--gpus", str(n_gpus),
           "--node-gate-calls", str(args.node_gate_calls), "--fresh-context-calls", str(args.fresh_context_calls),
           "--b1-sample-gib", str(args.b1_sample_gib)]
    if args.no_transition:
        cmd.append("--no-transition")
    if args.no_baselines:
        cmd.append("--no-baselines")
    try:
        proc = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=args.node_leg_timeout_s)
        lines = [ln for ln in proc.stdout.splitlines() if ln.startswith("NODE_LEG ")]
        if not lines:
            return {"error": f"node leg exit {proc.returncode}: {proc.stderr.strip()[-800:]}"}
        out = json.loads(lines[-1][9:])
        out.setdefault("node_checks", {})["other_ranks_gone_before_start"] = idle
        return out
    except Exception as exc:  # noqa: BLE001
        return {"error": f"node leg failed: {exc}"}


def node_leg(args):
    n = args.gpus
    sys.path.insert(0, str(ROOT / "tests" / "fakes"))
    os.environ["CCM_ALLOW_SIM"] = "1"
    # rank 0's parent process is still alive with its own CUDA context (~0.8 GiB) on GPU 0, so that
    # GPU reaches ~99.2 % instead of the 99.66 % of a GPU with no other tenant: keep a margin under it
    os.environ.setdefault("CC_SCRUB_MIN_COVERAGE", "0.985")
    import logging

    from k8s_cc_manager_b200 import _native as N
    from k8s_cc_manager_b200 import devices as D
    L = N.lib()
    check(L.ccm_init(N.BACKEND_CUDASIM), "ccm_init")
    out = {}
    gpus = [d for d in D.find_gpus()[0] if d.is_gpu()][:n]
    if len(gpus) < n:
        raise SystemExit(f"node leg wants {n} GPUs, sees {len(gpus)}")

    # ---- hardware proof for the in-process N-GPU launcher (tests/test_scrub_gpu.py:325-352) ----
    t0 = time.perf_counter()
    reports, wall_ms = D.scrub_and_verify_many(gpus, 0)
    clean = all(r.clean for r in reports)
    cov = [r.coverage for r in reports]
    victim = gpus[-1]
    # 3 bytes: first, an unaligned and the middle byte of the first chunk — valid for both launch shapes of the
    # product call (pipelined: 4 candidates per chunk; mapped-first, which n > 1 uses: 4 for the whole range)
    L.ccm_sim_set(victim.index, b"scrub_inject", 3)
    drill, _ = D.scrub_and_verify_many(gpus, 2 << 30)
    L.ccm_sim_set(victim.index, b"scrub_inject", 0)
    drill_ok = all((r.status == N.ERR_DIRTY and r.nonzero_bytes == 3) if r.bdf == victim.bdf else r.clean for r in drill)
    out["node_checks"] = {
        "gpus": n, "all_clean": clean, "coverage_min": min(cov), "coverage_max": max(cov),
        "bytes_unreached_max": max(r.bytes_unreached for r in reports),
        "first_gate_incl_context_creation_ms": (time.perf_counter() - t0) * 1e3, "first_gate_wall_ms": wall_ms,
        "dirt_drill": {"victim": victim.bdf, "injected": 3, "statuses": [r.status for r in drill],
                       "victim_counted": [r.nonzero_bytes for r in drill if r.bdf == victim.bdf][0], "ok": drill_ok},
        "ok": bool(clean and min(cov) >= 0.99 and drill_ok)}
    for g in gpus:
        g.wait_scrub_released()

    # ---- the node-level cold gate (one process, N threads), statistics ---------------------
    v, c = [], []
    for _ in range(args.node_gate_calls):
        t0 = time.perf_counter()
        reps, _ = D.scrub_and_verify_many(gpus, 0)
        v.append(time.perf_counter() - t0)
        for g in gpus:
            g.wait_scrub_released()
        c.append(time.perf_counter() - t0)
        assert all(r.clean for r in reps)
    out["node_gate"] = {"gpus": n, "launcher": "ONE process, one thread per GPU (ccm_scrub_verify_many; maps first when N > 1)"}
    out["node_gate"]["warm_contexts"] = {
        "verdict_s": stats(v), "cycle_s": stats(c), "bytes_total": sum(r.bytes_scrubbed for r in reps),
        "acquire_host_ms_max": max(r.ms_acquire for r in reps), "gpu_span_ms_max": max(r.ms_gpu_span for r in reps)}

    # ---- the same gate on FRESH contexts: what a daemon that drops its contexts after every gate (the default)
    # pays before the first byte is scrubbed — context creation is part of the time to the verdict --------------
    fv, fc = [], []
    for _ in range(args.fresh_context_calls):
        D.release_cuda_contexts(gpus)                                  # untimed: contexts gone, HBM back
        t0 = time.perf_counter()
        reps, _ = D.scrub_and_verify_many(gpus, 0)                     # creates N primary contexts, then the gate
        fv.append(time.perf_counter() - t0)
        assert all(r.clean for r in reps)
        D.release_cuda_contexts(gpus)                                  # joins the HBM give-back, resets the contexts
        fc.append(time.perf_counter() - t0)
    if fv:
        out["node_gate"]["fresh_contexts"] = {
            "verdict_s": stats(fv), "cycle_incl_context_reset_s": stats(fc),
            "what": "per call: N primary contexts created + full-HBM gate (verdict), then HBM handed back + contexts reset"}

    logging.disable(logging.CRITICAL)
    try:
        if not args.no_transition:
            out["transition"] = {"contexts_kept": measure_transitions(L, N, n, release_contexts=False)}
        if not args.no_baselines:
            out["baselines"] = constructed_baselines(L, N, n, args)
        if not args.no_transition:
            # LAST: this policy resets the CUDA primary contexts (torch, used by B2 above, is dead afterwards)
            out["transition"]["daemon_default_release_contexts"] = measure_transitions(L, N, n, release_contexts=True)
            out["transition"]["simulated"] = ["CC mode registers (cudasim backend; the box's driver-bound GPUs cannot be reset)",
                                             "reset/boot latency = 0 ms", "kubernetes API (in-memory fake, 0 ms RTT)"]
            out["transition"]["real"] = ["full-HBM scrub-and-verify gate on every GPU", "CUDA context creation / reset",
                                         "driver memory management (cuMemCreate/Map/SetAccess/Unmap/Release)"]
    finally:
        logging.disable(logging.NOTSET)
    print("NODE_LEG " + json.dumps(out), flush=True)
    sys.stdout.flush()
    os._exit(0)   # contexts may have been reset under torch: skip interpreter teardown


def measure_transitions(L, N, n_gpus, release_contexts):
    """BASELINE metric 1: wall-clock of CCManager.set_cc_mode off->on->devtools->off on the first N
    GPUs, eviction-gated.  Simulated and reported as such: CC registers, reset/boot latency (0 ms),
    the k8s API server (in-memory).  Real: the full-HBM scrub gate, CUDA contexts, driver memory work."""
    import kubernetes
    from k8s_cc_manager_b200 import devices as D
    from k8s_cc_manager_b200 import manager
    from k8s_cc_manager_b200.drain_gate import COMPONENT_LABELS
    L.ccm_sim_set(-1, b"cc_mode", 0)
    c = kubernetes.reset_cluster()
    c.add_node("bench-node", {k: "true" for k in COMPONENT_LABELS})
    os.environ["EVICT_OPERATOR_COMPONENTS"] = "true"
    os.environ["CC_RELEASE_CUDA_CONTEXT"] = "true" if release_contexts else "false"
    first_n = lambda: tuple(x[:n_gpus] if isinstance(x, list) else n_gpus for x in D.find_gpus())  # noqa: E731
    mgr = manager.CCManager("bench-node", "on", True, device_source=first_n)
    out = {"policy": "CC_RELEASE_CUDA_CONTEXT=" + ("true (daemon default)" if release_contexts else "false (contexts kept)"),
           "gpus": n_gpus}
    walls = []
    for mode in ("on", "devtools", "off", "on", "off"):
        t0 = time.perf_counter()
        okay = mgr.set_cc_mode(mode)
        dt = time.perf_counter() - t0
        reps = mgr.last_transition.get("scrub") or []
        key = f"to_{mode}" if f"to_{mode}" not in out else f"to_{mode}_again"
        out[key] = {"ok": bool(okay), "wall_s": dt,
                    "seconds_to_verdict": mgr.last_transition.get("seconds_to_verdict"),
                    "state_label": c.labels("bench-node").get("nvidia.com/cc.mode.state"),
                    "phase_seconds": mgr.last_transition.get("phase_seconds"),
                    "scrubbed_bytes": [r.bytes_scrubbed for r in reps] if isinstance(reps, list) else reps,
                    "coverage_min": min((r.coverage for r in reps), default=None) if isinstance(reps, list) else None}
        walls.append(dt)
    out["wall_s"] = stats(walls)
    out["all_ok"] = all(v["ok"] for k, v in out.items() if k.startswith("to_"))
    return out


def constructed_baselines(L, N, n_gpus, args):
    """BASELINE.md §3: the reference has no scrub, so the baselines mirror its STRUCTURE (one Python
    thread, GPUs one after another like reference main.py:504-529) with library calls only."""
    import numpy as np
    import torch
    out = {}
    # B2: serial cudaMemsetAsync + torch.count_nonzero per GPU (library-only GPU path)
    t0 = time.perf_counter()
    total = 0
    for g in range(n_gpus):
        torch.cuda.set_device(g)
        free, _ = torch.cuda.mem_get_info(g)
        want = (free - (4 << 30)) // (2 << 20) * (2 << 20)
        buf = torch.empty(want, dtype=torch.uint8, device=f"cuda:{g}")
        check(L.ccm_region_scrub(g, C.c_void_p(buf.data_ptr()), want, N.SCRUB_MEMSET, None, None, None), "memset")
        torch.cuda.synchronize(g)
        nz, step = 0, 256 << 20     # torch.count_nonzero on uint8 materialises an 8x temporary
        for off in range(0, want, step):
            nz += int(torch.count_nonzero(buf[off:off + step]))
        assert nz == 0
        total += want
        del buf
        torch.cuda.empty_cache()
    dt = time.perf_counter() - t0
    out["B2"] = {"wall_s": dt, "bytes_total": total, "value_gbs": 2.0 * total / dt / 1e9, "gpus": n_gpus,
                 "what": "constructed: GPUs one after another, cudaMemsetAsync + torch.count_nonzero (256 MiB slices)"}
    # B1: serial cudaMemset, verify on the HOST (256 MiB pinned D2H chunks + np.count_nonzero), bounded sample
    sample = int(args.b1_sample_gib * 2**30)
    chunk = 256 << 20
    pinned = torch.empty(chunk, dtype=torch.uint8, pin_memory=True)
    host = pinned.numpy()
    t0 = time.perf_counter()
    for g in range(n_gpus):
        torch.cuda.set_device(g)
        buf = torch.empty(sample, dtype=torch.uint8, device=f"cuda:{g}")
        check(L.ccm_region_scrub(g, C.c_void_p(buf.data_ptr()), sample, N.SCRUB_MEMSET, None, None, None), "memset")
        torch.cuda.synchronize(g)
        nz = 0
        for off in range(0, sample, chunk):
            k = min(chunk, sample - off)
            pinned[:k].copy_(buf[off:off + k])
            torch.cuda.synchronize(g)
            nz += int(np.count_nonzero(host[:k]))
        assert nz == 0
        del buf
        torch.cuda.empty_cache()
    dt = time.perf_counter() - t0
    out["B1"] = {"wall_s": dt, "bytes_total": sample * n_gpus, "value_gbs": 2.0 * sample * n_gpus / dt / 1e9,
                 "sample_bytes_per_gpu": sample,
                 "what": "constructed: GPUs one after another, cudaMemset + host verify over PCIe "
                         "(256 MiB pinned D2H + np.count_nonzero, one thread); bounded sample, throughput extrapolates linearly"}
    out["B0_get_only"] = b0_get_only(L, N, n_gpus)
    return out


def b0_get_only(L, N, n_gpus, reps=200):
    """B0: the get-only plumbing path (BASELINE configs[0]) through the product — set_cc_mode(mode) with every
    GPU already in `mode` (reference main.py:232-258): N register reads + the state label."""
    from k8s_cc_manager_b200 import devices as D
    from k8s_cc_manager_b200 import manager
    import kubernetes
    c = kubernetes.reset_cluster()
    c.add_node("bench-node", {})
    L.ccm_sim_set(-1, b"cc_mode", 1)
    os.environ["EVICT_OPERATOR_COMPONENTS"] = "false"
    first_n = lambda: tuple(x[:n_gpus] if isinstance(x, list) else n_gpus for x in D.find_gpus())  # noqa: E731
    mgr = manager.CCManager("bench-node", "on", True, device_source=first_n, scrub_mode="skip")
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        assert mgr.set_cc_mode("on") is True
        ts.append(time.perf_counter() - t0)
    ref = None
    for name in ("r2_config1_get_only.json", "r1_config1_get_only.json"):
        try:
            ref = json.loads((ROOT / "profiles" / name).read_text())
            break
        except Exception:  # noqa: BLE001
            pass
    result = {"product_us_median": statistics.median(ts) * 1e6, "gpus": n_gpus,
                          "what": "configs[0]: set_cc_mode(mode) with every GPU already in `mode` (reference main.py:232-258): "
                                  "N register reads + state label; sim registers, in-memory API",
                          "reference_main_py_committed": ref and {k: (v if not isinstance(v, dict) else v.get("median_us")) for k, v in ref.items()},
                          "reference_note": "the unmodified reference cannot run on the GPU box (/root/reference is not there); "
                                            "its numbers (median us per call) were taken in the dev container by benchmarks/config1_get_only.py: profiles/r2_config1_get_only.json"}
    L.ccm_sim_set(-1, b"cc_mode", 0)
    return result


# --------------------------------------------------------------------------- sweep
def run_sweep(args):
    """BASELINE configs[4]: region sweep 1 GB -> max on this rank's GPU (all ranks concurrently under
    torchrun): resident-kernel rates (CUDA events, best and median of 5) and the cold product call."""
    import torch
    from k8s_cc_manager_b200 import _native as N
    from k8s_cc_manager_b200 import devices as D
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
        os.environ.setdefault("CCM_ARENA_RESERVE_MB", "1024")
    L = N.lib()
    check(L.ccm_init(N.BACKEND_CUDASIM), "ccm_init")
    dev = local
    gpu = [d for d in D.find_gpus()[0] if d.is_gpu()][dev]
    sizes = [int(x * 1e9) // (2 << 20) * (2 << 20) for x in (1, 2, 4, 8, 16, 32, 64, 128)] + [0]
    rows = []
    ms, nz = C.c_float(), C.c_uint64()
    for want in sizes:
        ai = N.ArenaInfo()
        check(L.ccm_arena_acquire(dev, want, C.byref(ai)), "arena_acquire")
        R = int(ai.bytes)
        s_t, v_t, m_t = [], [], []
        for i in range(7):
            check(L.ccm_arena_fill(dev, 0xA5, None), "poison")
            check(L.ccm_arena_scrub(dev, N.SCRUB_AUTO, None, None, C.byref(ms)), "scrub")
            if i >= 2:
                s_t.append(ms.value)
            check(L.ccm_arena_verify(dev, N.VERIFY_AUTO, None, None, C.byref(nz), C.byref(ms)), "verify")
            assert nz.value == 0
            if i >= 2:
                v_t.append(ms.value)
            check(L.ccm_arena_scrub(dev, N.SCRUB_MEMSET, None, None, C.byref(ms)), "memset")
            if i >= 2:
                m_t.append(ms.value)
        check(L.ccm_arena_release(dev), "release")
        cold = []
        for i in range(6):
            if dist:
                dist.barrier()
            t0 = time.perf_counter()
            rep = gpu.scrub_and_verify(want)
            t1 = time.perf_counter()
            gpu.wait_scrub_released()
            if i:
                cold.append((t1 - t0, time.perf_counter() - t0))
        row = [float(R), R / min(s_t) / 1e6, R / statistics.median(s_t) / 1e6, R / min(v_t) / 1e6,
               R / statistics.median(v_t) / 1e6, R / min(m_t) / 1e6, statistics.median(x[0] for x in cold) * 1e3,
               statistics.median(x[1] for x in cold) * 1e3]
        rows.append(row)
    if dist:
        t = torch.tensor(rows, dtype=torch.float64, device="cuda")
        g = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(g, t)
        allr = [x.cpu().tolist() for x in g]
        dist.destroy_process_group()
    else:
        allr = [rows]
    if rank != 0:
        return
    table = []
    for i in range(len(sizes)):
        per = [allr[r][i] for r in range(world)]
        table.append({"region_bytes_per_gpu": int(per[0][0]), "gpus": world,
                      "scrub_gbs_per_gpu_best_min_over_gpus": min(p[1] for p in per),
                      "scrub_gbs_per_gpu_median": statistics.median(p[2] for p in per),
                      "verify_gbs_per_gpu_best_min_over_gpus": min(p[3] for p in per),
                      "verify_gbs_per_gpu_median": statistics.median(p[4] for p in per),
                      "memset_gbs_per_gpu_best": statistics.median(p[5] for p in per),
                      "aggregate_scrub_gbs": sum(p[2] for p in per), "aggregate_verify_gbs": sum(p[4] for p in per),
                      "cold_call_verdict_ms_max_over_gpus": max(p[6] for p in per),
                      "cold_call_cycle_ms_max_over_gpus": max(p[7] for p in per)})
    print(json.dumps({"sweep": table, "n_gpus": world, "unit": "GB/s", "kernels": list(N.default_kernels()),
                      "how": "resident kernels: CUDA events around ONE launch, 5 timed passes after 2 warm passes, region "
                             "re-poisoned before every scrub; memset = cudaMemsetAsync over the same region; cold call = "
                             "Gpu.scrub_and_verify(bytes) wall-clock to verdict / to HBM handed back, median of 5"}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=("ours", "reference"))
    ap.add_argument("--gib", type=float, default=0.0, help="region per GPU in GiB (0 = all mappable HBM)")
    ap.add_argument("--scrub", default="auto", choices=("auto", "st128", "st256", "tma", "memset"))
    ap.add_argument("--verify", default="auto", choices=("auto", "ld128", "ld256"))
    ap.add_argument("--e2e-steps", type=int, default=15)
    ap.add_argument("--cpu-sample-gib", type=float, default=8.0)
    ap.add_argument("--cpu-passes", type=int, default=40)
    ap.add_argument("--b1-sample-gib", type=float, default=2.0)
    ap.add_argument("--node-gate-calls", type=int, default=7)
    ap.add_argument("--fresh-context-calls", type=int, default=4)
    ap.add_argument("--node-leg-timeout-s", type=float, default=600.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-transition", action="store_true")
    ap.add_argument("--no-baselines", action="store_true")
    ap.add_argument("--no-node-leg", action="store_true")
    ap.add_argument("--no-host-roundtrip", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/*.npy")
    ap.add_argument("--sweep", action="store_true", help="region sweep 1 GB -> max instead of the bench line")
    ap.add_argument("--cpu-probe", action="store_true", help="only the CPU arm, with its tuning table")
    ap.add_argument("--node-leg", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.cpu_probe:
        cpu_arm(args.cpu_sample_gib, passes=args.cpu_passes, warm=3, probe=True)
    elif args.node_leg:
        node_leg(args)
    elif args.sweep:
        run_sweep(args)
    elif args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
