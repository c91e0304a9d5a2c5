#!/usr/bin/env python3
"""Record what the original extension answers in the differential tests (tests/recorded_reference.py).

Needs oracle/_ref, the original compiled by `make -C oracle ref` (REF=<checkout of WojciechMula/pyahocorasick>).

    python tests/golden/record_reference.py [pytest arguments, default: tests]

Runs the given tests with the live original, keeps every call's answer and merges the traces into
tests/golden/reference/<test module>.pkl.xz.  Without a GPU, the gpu-marked tests that talk to the original call by
call run on the emulated device of tests/emul.py (the original's answers do not depend on the device); the ones that
only keep record digests (tests/test_gpu_parity.py) need a GPU to be recorded.
"""
from __future__ import annotations

import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import oracle  # noqa: E402
import recorded_reference as rr  # noqa: E402


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


class _RecordOnCpu:
    """without a GPU: run the gpu-marked tests that use the `reference` fixture on the emulated device"""

    @pytest.hookimpl(trylast=True)
    def pytest_collection_modifyitems(self, config, items):
        for it in items:
            if "gpu" in it.keywords and "reference" in getattr(it, "fixturenames", ()):
                it.own_markers = [m for m in it.own_markers if m.name != "skip"]

    @pytest.fixture(autouse=True)
    def _emulated_device(self, request, monkeypatch):
        if request.node.get_closest_marker("gpu"):
            import emul
            emul.install(monkeypatch, "filter")


def main():
    if not oracle.ref_available("bytes") or not oracle.ref_available("unicode"):
        raise SystemExit("oracle/_ref is not built: make -C oracle ref REF=<checkout of the original>")
    rr.RECORDING = {}
    plugins = [] if _has_gpu() else [_RecordOnCpu()]
    args = sys.argv[1:] or [os.path.join(ROOT, "tests")]
    rc = pytest.main(["-q", "-p", "no:cacheprovider", *args], plugins=plugins)
    if rc not in (0, 5):
        raise SystemExit(f"pytest failed ({rc}): nothing written")
    for module, traces in sorted(rr.RECORDING.items()):
        merged = rr.load_traces(module)
        merged.update(traces)
        rr.save_traces(module, merged)
        size = os.path.getsize(os.path.join(rr._DIR, module + ".pkl.xz"))
        print(f"{module}: {len(traces)} recorded, {len(merged)} in the file, {size} bytes")


if __name__ == "__main__":
    main()
