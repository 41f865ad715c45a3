import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _host_cpu_budget() -> int:
    """Usable cores: scheduler affinity clamped by the cgroup quota (same rule as bench.py's CPU arm)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return max(1, n)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    # the CPU oracle legs: a thread pool larger than the usable cores (128 threads on a small quota) is 10-50x slower
    import torch
    torch.set_num_threads(min(32, _host_cpu_budget()))


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN
