#!/usr/bin/env python3
"""Records tests/golden/reference_shim_calls.json: every call the UNMODIFIED reference main.py
makes into the gpu-admin-tools shim (k8s_cc_manager_b200/compat/gpu-admin-tools) for a set of
transition scenarios, with what each call returned or raised.

ORACLE / TEST INFRASTRUCTURE.  Needs a checkout of the reference (--reference DIR, or
CCM_REFERENCE_DIR) and libccm.so; the test that replays the transcript
(tests/test_compat_shim.py) needs neither the reference nor this script.

The reference is run exactly as tests/golden/transitions.json was recorded (oracle/gen_golden.py),
except that its device layer is the shim over libccm's simulated registers instead of the fake
gpu-admin-tools.  Before anything is written, every step's libccm register trace, end registers,
Kubernetes calls, labels and return value are checked against transitions.json, so a transcript
is only ever recorded from a run that matches the reference's own goldens.

Usage:  python oracle/gen_shim_calls.py --reference DIR [--check]
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import logging
import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
COMPAT = ROOT / "k8s_cc_manager_b200" / "compat" / "gpu-admin-tools"
OUT = ROOT / "tests" / "golden" / "reference_shim_calls.json"
SCENARIOS = ["off_to_on_evict_pods_gone", "roundtrip_on_devtools_off", "cc_on_with_ppcie_active", "ppcie_from_off",
             "fault_set_gpuerror_gpu3", "fault_stuck_mode_gpu5", "get_only_8gpu_on"]

for p in (ROOT, ROOT / "tests", ROOT / "tests" / "fakes", ROOT / "oracle"):
    sys.path.insert(0, str(p))


class Recorder:
    """Stands in for `pci.devices.find_gpus` inside the reference; hands out recording device proxies.

    Transcript entries: ["find_gpus", len(devices), n], [handle, attribute, value] for an attribute
    read, [handle, "method()", args, {"return": value} | {"raise": exception type}] for a call.
    A handle is "<find_gpus call>:<index in its list>"."""

    def __init__(self, find_gpus):
        self._find, self._finds, self.calls = find_gpus, 0, []

    def find_gpus(self):
        devs, n = self._find()
        k, self._finds = self._finds, self._finds + 1
        self.calls.append(["find_gpus", len(devs), n])
        return [_Recorded(self, f"{k}:{i}", d) for i, d in enumerate(devs)], n


class _Recorded:
    def __init__(self, rec, handle, dev):
        self._rec, self._handle, self._dev = rec, handle, dev

    def __getattr__(self, name):
        value = getattr(self._dev, name)
        if not callable(value):
            self._rec.calls.append([self._handle, name, value])
            return value

        def call(*args, **kwargs):
            assert not kwargs, f"{name}: keyword arguments are not recorded"
            entry = [self._handle, name + "()", list(args)]
            self._rec.calls.append(entry)
            try:
                out = value(*args)
            except Exception as exc:
                entry.append({"raise": type(exc).__name__})
                raise
            entry.append({"return": out})
            return out
        return call


def record(reference: Path):
    from helpers import build_cluster, build_native_world, k8s_trace, registers, sim_trace, sim_trace_clear
    import scenarios as SC

    golden = {s["name"]: s for s in json.loads((ROOT / "tests/golden/transitions.json").read_text())["scenarios"]}
    sys.path.insert(0, str(reference))
    sys.path.insert(0, str(COMPAT))
    spec = importlib.util.spec_from_file_location("reference_main_on_libccm", reference / "main.py")
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    import gpu_operator_eviction as ref_evict
    assert Path(ref_evict.__file__).parent == reference
    logging.disable(logging.CRITICAL)
    shim_find = ref.find_gpus
    out = []
    for name in SCENARIOS:
        sc = next(s for s in SC.transition_scenarios() if s["name"] == name)
        build_native_world(sc)
        c = build_cluster(sc)
        ref_evict.time = c.clock
        os.environ["EVICT_OPERATOR_COMPONENTS"] = "true" if sc["evict"] else "false"
        os.environ["OPERATOR_NAMESPACE"] = SC.NAMESPACE
        mgr = ref.CCManager(node_name=SC.NODE, default_mode="on", host_cc=sc["host_cc"])
        steps = []
        for mode, want in zip(sc["modes"], golden[name]["steps"]):
            rec = Recorder(shim_find)
            ref.find_gpus = rec.find_gpus
            n_k8s = len(c.calls)
            sim_trace_clear()
            assert mgr.set_cc_mode(mode) == want["result"], (name, mode)
            assert sim_trace() == want["device_trace"], (name, mode)
            assert k8s_trace(c)[n_k8s:] == want["k8s"], (name, mode)
            assert c.labels(SC.NODE) == want["labels"], (name, mode)
            assert registers() == want["registers"], (name, mode)
            steps.append({"mode": mode, "calls": rec.calls})
        out.append({"name": name, "steps": steps})
    ref.find_gpus = shim_find
    return {"generated_by": "oracle/gen_shim_calls.py", "reference": "NVIDIA/k8s-cc-manager@09cd768c main.py",
            "scenarios": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", type=Path, default=os.environ.get("CCM_REFERENCE_DIR"),
                    help="checkout of the reference (its main.py and gpu_operator_eviction.py)")
    ap.add_argument("--check", action="store_true", help="fail if the committed transcript differs")
    args = ap.parse_args()
    if args.reference is None or not (args.reference / "main.py").exists():
        raise SystemExit("--reference DIR (or CCM_REFERENCE_DIR) must name a checkout of the reference")
    os.environ.setdefault("CCM_ALLOW_SIM", "1")
    from k8s_cc_manager_b200 import build
    build.build()
    text = json.dumps(record(args.reference.resolve()), indent=1, sort_keys=True) + "\n"
    if args.check:
        if not OUT.exists() or OUT.read_text() != text:
            print(f"DIFFERS: {OUT}")
            sys.exit(1)
        return
    OUT.write_text(text)
    print(f"wrote {OUT} ({len(text)} bytes)")


if __name__ == "__main__":
    main()
