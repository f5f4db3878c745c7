import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _has_gpu():
    try:
        from sdrplusplus_b200 import lib
        return lib.load().b200_device_count() > 0
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device: the product has no CPU fallback")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def oracle():
    """The CPU checker (plain-C restatement of the reference path)."""
    from oracle.oracle import Oracle, available
    if not available("restatement"):
        import subprocess
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), os.path.join(ROOT, "oracle", "liboracle.so")])
    return Oracle("restatement")


_REPORT = {}


@pytest.fixture(scope="session")
def report():
    """Collects measured parity errors; written to gpurun_out/parity_report.json at session end."""
    yield _REPORT
    out = os.path.join(ROOT, "gpurun_out")
    try:
        os.makedirs(out, exist_ok=True)
        path = os.path.join(out, "parity_report.json")
        merged = {}
        if os.path.exists(path):
            try:
                with open(path) as f:
                    merged = json.load(f)
            except ValueError:
                merged = {}
        merged.update(_REPORT)
        with open(path, "w") as f:
            json.dump(merged, f, indent=1, sort_keys=True)
    except OSError:
        pass
