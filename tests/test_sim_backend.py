"""Register-level semantics of the shim's backends (CPU only): stage/reset/boot
contract, fault injection, the concurrent batched transition, sysfs enumeration."""
from __future__ import annotations

import ctypes as C
import time

import pytest

from helpers import sim_get, sim_set, sim_trace, sim_trace_clear
from k8s_cc_manager_b200 import _native as N
from k8s_cc_manager_b200 import devices as D


@pytest.fixture()
def sim():
    lib = N.lib()
    assert lib.ccm_sim_topology(8, 4) == 0
    sim_set(-1, "cuda_ordinal", -1)
    sim_trace_clear()
    return lib


def test_enumeration_shape(sim):
    devs, n = D.find_gpus()
    assert n == 12 and len(devs) == 12
    gpus = [d for d in devs if d.is_gpu()]
    sw = [d for d in devs if d.is_nvswitch()]
    assert len(gpus) == 8 and len(sw) == 4
    assert gpus[0].bdf == "0000:1b:00.0" and sw[0].bdf == "0000:05:00.0"
    assert all(g.is_cc_query_supported and g.is_ppcie_query_supported for g in gpus)
    assert all((not s.is_cc_query_supported) and s.is_ppcie_query_supported for s in sw)
    assert isinstance(gpus[0].is_cc_query_supported, bool)  # attribute, not method (main.py:186)


def test_set_stages_reset_applies_wait_boots(sim):
    sim_set(0, "boot_ms", 300)
    g = D.find_gpus()[0][0]
    assert g.query_cc_mode() == "off"
    g.set_cc_mode("on")
    assert g.query_cc_mode() == "off"          # staged only (main.py:455-459)
    g.reset_with_os()
    with pytest.raises(D.GpuError) as e:        # not usable until it has booted
        g.query_cc_mode()
    assert e.value.status == N.ERR_NOT_BOOTED
    g.wait_for_boot()
    assert g.query_cc_mode() == "on"
    sim_set(0, "boot_ms", 0)
    g.set_cc_mode("devtools"); g.reset_with_os()
    assert g.query_cc_mode() == "devtools"     # boot time elapsed: the device is back on its own
    g.wait_for_boot()
    assert sim_trace()[:3] == ["0000:1b:00.0 query_cc_mode off", "0000:1b:00.0 set_cc_mode on",
                               "0000:1b:00.0 query_cc_mode off"]


def test_state_survives_reenumeration(sim):
    g = D.find_gpus()[0][3]
    g.set_ppcie_mode("on"); g.reset_with_os(); g.wait_for_boot()
    again = D.find_gpus()[0][3]
    assert again.bdf == g.bdf and again.query_ppcie_mode() == "on"


def test_invalid_arguments(sim):
    g, s = D.find_gpus()[0][0], D.find_gpus()[0][8]
    with pytest.raises(D.GpuError):
        g.set_cc_mode("maybe")
    with pytest.raises(D.GpuError) as e:
        s.query_cc_mode()
    assert e.value.status == N.ERR_UNSUPPORTED
    assert N.lib().ccm_query_cc_mode(99, C.byref(C.c_int())) == N.ERR_NO_DEVICE
    assert N.lib().ccm_set_cc_mode(0, 7) == N.ERR_INVALID


@pytest.mark.parametrize("op,call", [("query_cc_mode", lambda g: g.query_cc_mode()),
                                     ("set_cc_mode", lambda g: g.set_cc_mode("on")),
                                     ("reset_with_os", lambda g: g.reset_with_os()),
                                     ("wait_for_boot", lambda g: g.wait_for_boot())])
def test_fault_injection_raises_gpuerror(sim, op, call):
    from helpers import OP_BITS
    sim_set(2, "fail_op", OP_BITS[op])
    g = D.find_gpus()[0][2]
    with pytest.raises(D.GpuError) as e:
        call(g)
    assert e.value.status == N.ERR_FAULT and g.bdf in str(e.value)
    D.find_gpus()[0][1].query_cc_mode()  # other devices unaffected


def test_stuck_device_reads_back_old_mode(sim):
    sim_set(5, "stuck", 1)
    g = D.find_gpus()[0][5]
    g.set_cc_mode("on"); g.reset_with_os(); g.wait_for_boot()
    assert g.query_cc_mode() == "off"


def test_boot_timeout(sim):
    sim_set(0, "boot_ms", 400)
    g = D.find_gpus()[0][0]
    g.reset_with_os()
    with pytest.raises(D.GpuError) as e:
        g.wait_for_boot(timeout_ms=50)
    assert e.value.status == N.ERR_TIMEOUT
    g.wait_for_boot()
    assert g.query_cc_mode() == "off"


def test_python_manager_wallclock_scales_with_max_not_sum(sim, monkeypatch):
    """The concurrent launcher: per-GPU reset/boot latencies overlap (SURVEY.md §8e)."""
    import kubernetes
    from k8s_cc_manager_b200 import manager
    c = kubernetes.reset_cluster()
    c.add_node("n", {})
    monkeypatch.setenv("EVICT_OPERATOR_COMPONENTS", "false")
    sim_set(-1, "reset_ms", 60)
    sim_set(-1, "boot_ms", 90)
    par = manager.CCManager("n", "on", True, scrub_mode="skip", max_parallel=0)
    t0 = time.perf_counter(); assert par.set_cc_mode("on") is True; t_par = time.perf_counter() - t0
    ser = manager.CCManager("n", "on", True, scrub_mode="skip", max_parallel=1)
    t0 = time.perf_counter(); assert ser.set_cc_mode("off") is True; t_ser = time.perf_counter() - t0
    assert t_ser > 8 * 0.06 * 0.9          # serial: resets add up (boots overlap the later resets)
    assert t_par < t_ser / 2.5, (t_par, t_ser)
    assert set(par.last_transition["phase_seconds"]) >= {"stage", "reset", "boot"}


def test_sysfs_backend_enumerates_fake_tree(tmp_path, monkeypatch):
    # PCI domain fffe: no host puts a real GPU there, so no CUDA device matches these addresses
    root = tmp_path / "devices"

    def dev(bdf, vendor, cls, device="0x2901"):
        d = root / bdf
        d.mkdir(parents=True)
        (d / "vendor").write_text(vendor + "\n")
        (d / "class").write_text(cls + "\n")
        (d / "device").write_text(device + "\n")
        (d / "reset").write_text("")

    dev("fffe:1b:00.0", "0x10de", "0x030200")
    dev("fffe:43:00.0", "0x10de", "0x030000")
    dev("fffe:05:00.0", "0x10de", "0x068000", "0x22a3")
    dev("fffe:00:1f.0", "0x8086", "0x060100")
    dev("fffe:aa:00.0", "0x10de", "0x0c0330")  # NVIDIA USB controller: not a GPU
    monkeypatch.setenv("CCM_SYSFS_ROOT", str(root))
    try:
        D.select_backend("sysfs")
        devs, n = D.find_gpus()
        assert [(d.bdf, d.is_gpu()) for d in devs] == [("fffe:05:00.0", False), ("fffe:1b:00.0", True),
                                                       ("fffe:43:00.0", True)]
        gpu = devs[1]
        with pytest.raises(D.GpuError) as e:   # register map is not part of this build
            gpu.set_cc_mode("on")
        assert e.value.status == N.ERR_UNSUPPORTED
        gpu.reset_with_os()
        assert (root / "fffe:1b:00.0" / "reset").read_text() == "1"
        gpu.wait_for_boot(timeout_ms=200)
        with pytest.raises(D.GpuError) as e:   # no CUDA device behind it here
            gpu.scrub_and_verify(1 << 20)
        assert e.value.status == N.ERR_NO_CUDA
    finally:
        D.select_backend("sim")
