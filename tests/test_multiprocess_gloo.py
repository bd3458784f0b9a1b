"""N>1 host logic of bench.py on CPU: world_size 2 over gloo (127.0.0.1).  The data path
has no collective; ranks only agree on max(time) and sum(bytes), and the reference arm
lets rank 0 alone print."""
from __future__ import annotations

import json
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]

WORKER = r"""
import os, sys, json
import torch, torch.distributed as dist
sys.path.insert(0, os.environ["REPO"])
from k8s_cc_manager_b200.aggregate import aggregate_job
dist.init_process_group("gloo")
rank = dist.get_rank()
# rank r pretends: region (r+1)*1000 bytes, 4 steps in (10 + 5r) ms, 8 launches
out = aggregate_job(dist, device="cpu", region_bytes=(rank + 1) * 1000, steps=4,
                    elapsed_ms=10.0 + 5.0 * rank, launches=8)
if rank == 0:
    print(json.dumps(out))
dist.destroy_process_group()
"""


def test_two_rank_aggregation_over_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, REPO=str(ROOT), MASTER_ADDR="127.0.0.1")
    proc = subprocess.run(
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
         "--master-addr", "127.0.0.1", "--master-port", "29571", str(script)],
        capture_output=True, text=True, env=env, timeout=240)
    assert proc.returncode == 0, proc.stderr[-2000:]
    line = [l for l in proc.stdout.splitlines() if l.startswith("{")][-1]
    out = json.loads(line)
    assert out["world"] == 2
    assert out["ms"] == 15.0                        # MAX over ranks, never the mean
    assert out["total_region_bytes"] == 3000        # SUM over ranks (weak scaling: per-GPU work fixed)
    assert out["launches"] == 16
    # whole-job value: (bytes zeroed + bytes read back) * steps / max time
    assert abs(out["value_gbs"] - 2 * 3000 * 4 / 15e-3 / 1e9) < 1e-12


def test_reference_arm_prints_once_under_torchrun(tmp_path):
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    proc = subprocess.run(
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
         "--master-addr", "127.0.0.1", "--master-port", "29572", str(ROOT / "bench.py"),
         "--impl", "reference", "--gpus", "2", "--steps", "2", "--warmup", "1", "--cpu-sample-gib", "0.125"],
        capture_output=True, text=True, env=env, timeout=240)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [json.loads(l) for l in proc.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    ref = lines[0]
    assert ref["impl"] == "reference" and ref["n_gpus"] == 2 and ref["unit"] == "GB/s"
    assert ref["e2e"]["h2d_bytes_per_step"] == 0 and ref["cpu_baseline"]["kind"] == "port"
    assert ref["value"] > 0


COLD_WORKER = r"""
import os, sys, json
import torch, torch.distributed as dist
sys.path.insert(0, os.environ["REPO"])
from k8s_cc_manager_b200.aggregate import aggregate_cold_calls, gather_rows
dist.init_process_group("gloo")
rank = dist.get_rank()
# three cold calls; rank 1 is slower to the verdict in call 0 and slower to release in call 2
rows = [[0.050 + 0.030 * rank, 0.120 + 0.010 * rank, 100.0 * (rank + 1)],
        [0.055, 0.125, 100.0 * (rank + 1)],
        [0.060 - 0.005 * rank, 0.130 + 0.200 * rank, 100.0 * (rank + 1)]]
allr = gather_rows(dist, "cpu", rows)
if rank == 0:
    print(json.dumps(aggregate_cold_calls(allr)))
dist.destroy_process_group()
"""


def test_cold_call_statistics_take_the_slowest_rank_per_call(tmp_path):
    script = tmp_path / "cold_worker.py"
    script.write_text(COLD_WORKER)
    env = dict(os.environ, REPO=str(ROOT), MASTER_ADDR="127.0.0.1")
    proc = subprocess.run(
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
         "--master-addr", "127.0.0.1", "--master-port", "29573", str(script)],
        capture_output=True, text=True, env=env, timeout=240)
    assert proc.returncode == 0, proc.stderr[-2000:]
    out = json.loads([l for l in proc.stdout.splitlines() if l.startswith("{")][-1])
    assert out["world"] == 2 and out["calls"] == 3 and out["bytes_total"] == 900.0
    assert [round(x, 3) for x in out["verdict_s_each"]] == [0.080, 0.055, 0.060]      # max over ranks, per call
    assert [round(x, 3) for x in out["cycle_s_each"]] == [0.130, 0.125, 0.330]
    assert abs(out["verdict_s"]["median"] - 0.060) < 1e-12 and abs(out["cycle_s"]["max"] - 0.330) < 1e-12
    assert out["cycle_s"]["n"] == 3
    assert abs(out["value_mean_gbs"] - 2 * 900.0 / (0.130 + 0.125 + 0.330) / 1e9) < 1e-15
    assert abs(out["value_gbs"] - 2 * 300.0 / 0.130 / 1e9) < 1e-15                   # median cycle, robust to the outlier


def test_single_process_aggregation_needs_no_process_group():
    from k8s_cc_manager_b200.aggregate import aggregate_cold_calls, gather_rows, spread
    allr = gather_rows(None, "cpu", [[0.05, 0.12, 10], [0.07, 0.11, 10]])
    out = aggregate_cold_calls(allr)
    assert out["world"] == 1 and abs(out["verdict_s"]["median"] - 0.06) < 1e-12
    assert abs(out["value_mean_gbs"] - 2 * 20 / 0.23 / 1e9) < 1e-18 and abs(out["value_gbs"] - 2 * 10 / 0.115 / 1e9) < 1e-18
    assert spread([3, 1, 2])["median"] == 2 and spread([1, 2, 3, 4])["median"] == 2.5
    assert spread(list(range(1, 12)))["p10"] == 2 and spread(list(range(1, 12)))["p90"] == 10


def test_cpu_arm_reports_best_and_median_with_numa_layout():
    sys.path.insert(0, str(ROOT))
    import bench
    cb = bench.cpu_arm(0.03125, passes=3, warm=1)
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["passes"] == 3
    assert cb["best"] >= cb["median"] > 0 and cb["value"] > 0
    assert "NUMA" in cb["sample"] and "pinned" in cb["sample"]
    assert {c["scrub"] for c in cb["tuning"]} == {"memset", "nt-stores"}


def test_bench_b0_get_only_runs_on_the_sim_backend(native, cluster):
    """bench.py's node leg, the part that needs no GPU: configs[0] through the product on simulated registers."""
    sys.path.insert(0, str(ROOT))
    import bench
    L = native.lib()
    assert L.ccm_sim_topology(8, 0) == 0
    out = bench.b0_get_only(L, native, 4, reps=20)
    assert out["gpus"] == 4 and 1.0 < out["product_us_median"] < 5000.0
    ref = out["reference_main_py_committed"]
    assert ref and ref["reference_fake_devices"] > 0 and ref["product_serial"] > 0


def test_bench_dump_outputs_runs_the_step_on_a_seeded_input(tmp_path):
    """--dump-outputs: seeded dirt counted by the step's verify kernel, the step's own count, and the same
    seeded windows of the scrubbed arena on every run, well under 64 MB; a verify that sees no dirt fails."""
    import ctypes as C

    import numpy as np
    import pytest
    sys.path.insert(0, str(ROOT))
    import bench
    R = (3 << 30) + 5

    class FakeArena:
        """Arena of R bytes: the seeded fill makes it (offset % 251), the step zeroes it."""

        def __init__(self, verify_sees_dirt=True):
            self.calls, self.dirty, self.sees = [], False, verify_sees_dirt

        def ccm_arena_fill_random(self, dev, seed, stream):
            self.calls.append(("fill", seed))
            self.dirty = True
            return 0

        def ccm_arena_verify(self, dev, variant, cfg, stream, nz, ms):
            self.calls.append(("verify", variant))
            nz._obj.value = R - R // 251 - 1 if self.dirty and self.sees else 0
            return 0

        def step(self):
            self.calls.append(("step",))
            self.dirty = False

        def ccm_arena_fetch_count(self, dev, stream, nz):
            nz._obj.value = 0
            return 0

        def ccm_arena_read(self, dev, off, dst, n):
            self.calls.append(("read", off))
            assert 0 <= off and off + n <= R
            C.memmove(dst, bytes((off + i) % 251 if self.dirty else 0 for i in range(n)), n)
            return 0

    arenas = {d: FakeArena() for d in ("a", "b", "r")}
    for d in ("a", "b"):
        bench.dump_outputs(arenas[d], 0, R, 7, None, arenas[d].step, tmp_path / d)
    bench.dump_outputs(arenas["r"], 1, R, 7, None, arenas["r"].step, tmp_path / "r", rank=1)
    a = arenas["a"]
    assert a.calls[:3] == [("fill", bench.DUMP_SEED), ("verify", 7), ("step",)]
    load = lambda d, n: np.load(tmp_path / d / f"{n}.npy")  # noqa: E731
    assert load("a", "input_nonzero_bytes").dtype == np.float64
    assert load("a", "input_nonzero_bytes").tolist() == [R - R // 251 - 1] and load("a", "nonzero_bytes").tolist() == [0.0]
    sample = load("a", "arena_sample")
    assert sample.dtype == np.float32 and sample.shape == (bench.DUMP_WINDOWS + 2, bench.DUMP_WINDOW_BYTES)
    assert not sample.any()                                          # read back after the step's scrub
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) < 64 << 20
    for n in ("input_nonzero_bytes", "nonzero_bytes", "arena_sample"):
        assert np.array_equal(load("a", n), load("b", n))
    offs = [c[1] for c in a.calls if c[0] == "read"]
    assert offs == [c[1] for c in arenas["b"].calls if c[0] == "read"]
    assert offs[:2] == [0, R - bench.DUMP_WINDOW_BYTES] and len(set(offs)) == len(offs) == bench.DUMP_WINDOWS + 2
    assert load("r", "input_nonzero_bytes_rank1").tolist() == [R - R // 251 - 1]
    blind = FakeArena(verify_sees_dirt=False)
    with pytest.raises(RuntimeError, match="seeded input counted 0"):
        bench.dump_outputs(blind, 0, R, 7, None, blind.step, tmp_path / "blind")
