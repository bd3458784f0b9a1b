"""The gpu-admin-tools-shaped shim: the UNMODIFIED reference main.py runs on libccm.so.

What the reference calls through the shim, and what each call returned, is recorded in
tests/golden/reference_shim_calls.json (oracle/gen_shim_calls.py); the test replays it against the
shim.  The CLI twin (reference scripts/cc-manager.sh:127,389) is tested as well."""
from __future__ import annotations

import json
import sys
from pathlib import Path

import pytest

import scenarios as SC
from helpers import build_native_world, registers, sim_trace, sim_trace_clear

ROOT = Path(__file__).resolve().parents[1]
COMPAT = ROOT / "k8s_cc_manager_b200" / "compat" / "gpu-admin-tools"
GOLDEN = {s["name"]: s for s in json.loads((ROOT / "tests/golden/transitions.json").read_text())["scenarios"]}
SHIM_CALLS = {s["name"]: s for s in json.loads((ROOT / "tests/golden/reference_shim_calls.json").read_text())["scenarios"]}


def test_cli_twin_prints_what_the_shell_engine_parses(capsys):
    """scripts/cc-manager.sh:_parse_mode greps 'CC mode is <mode>'."""
    sys.path.insert(0, str(COMPAT))
    try:
        import nvidia_gpu_tools as cli
        build_native_world(SC.scenario("cli", gpus_=SC.gpus(2), modes=[]))
        assert cli.main(["--query-cc-mode", "--gpu-bdf=0000:1b:00.0"]) == 0
        assert "CC mode is off" in capsys.readouterr().out
        assert cli.main(["--set-cc-mode=devtools", "--reset-after-cc-mode-switch", "--gpu-bdf=0000:43:00.0"]) == 0
        assert "CC mode is devtools" in capsys.readouterr().out
        assert registers()["0000:43:00.0"]["cc"] == "devtools" and registers()["0000:1b:00.0"]["cc"] == "off"
        assert cli.main(["--query-cc-mode", "--gpu-bdf=0000:ff:00.0"]) == 1
    finally:
        sys.path.remove(str(COMPAT))
        sys.modules.pop("nvidia_gpu_tools", None)


@pytest.mark.parametrize("name", ["off_to_on_evict_pods_gone", "roundtrip_on_devtools_off", "cc_on_with_ppcie_active",
                                  "ppcie_from_off", "fault_set_gpuerror_gpu3", "fault_stuck_mode_gpu5",
                                  "get_only_8gpu_on"])
def test_unmodified_reference_runs_on_libccm(name, monkeypatch):
    """Drop-in check: the reference main.py's calls into the shim (device enumeration, attribute
    reads, register ops), replayed in order against compat shim -> ctypes -> libccm.so (sim
    registers), must return or raise what they did for the reference, and leave the same register
    trace and end registers as the fake gpu-admin-tools the goldens were recorded with."""
    sc = next(s for s in SC.transition_scenarios() if s["name"] == name)
    shim_modules = ("nvidia_gpu_tools", "pci", "pci.devices", "gpu")
    for mod in shim_modules:
        sys.modules.pop(mod, None)
    monkeypatch.syspath_prepend(str(COMPAT))
    try:
        from gpu import GpuError
        from nvidia_gpu_tools import Gpu  # noqa: F401 - imported by the reference (main.py:38)
        from pci.devices import find_gpus
        build_native_world(sc)
        steps = SHIM_CALLS[name]["steps"]
        assert [s["mode"] for s in steps] == sc["modes"]
        for step, want in zip(steps, GOLDEN[name]["steps"]):
            sim_trace_clear()
            devices, finds = {}, 0
            for entry in step["calls"]:
                if entry[0] == "find_gpus":
                    devs, n = find_gpus()
                    assert [len(devs), n] == entry[1:]
                    devices.update({f"{finds}:{i}": d for i, d in enumerate(devs)})
                    finds += 1
                elif entry[1].endswith("()"):
                    handle, method, args, outcome = entry
                    try:
                        got = {"return": getattr(devices[handle], method[:-2])(*args)}
                    except GpuError as exc:
                        got = {"raise": type(exc).__name__}
                    assert got == outcome, (step["mode"], entry)
                else:
                    handle, attr, value = entry
                    assert getattr(devices[handle], attr) == value, (step["mode"], entry)
            assert sim_trace() == want["device_trace"]
            assert registers() == want["registers"]
    finally:
        for mod in shim_modules:
            sys.modules.pop(mod, None)
