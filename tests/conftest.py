import importlib
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_addoption(parser):
    parser.addoption("--record-ref-kernels", metavar="DIR", default=None,
                     help="run the reference's own kernels (oracle/_ref/libref_ops.so) where the tests call them and write "
                          "their outputs to DIR/<test>.npz, instead of replaying tests/golden/ref_kernels/")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def pkg():
    """The product package (directory name starts with a digit, hence importlib)."""
    return importlib.import_module("3dssd_b200")


@pytest.fixture(scope="session")
def oracle_ops():
    from oracle import ops
    ops.build()
    return ops


@pytest.fixture(scope="session")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="session")
def _ref_recordings(request):
    recordings = {}
    yield recordings
    if recordings:
        from oracle import ref_golden
        ref_golden.write(recordings, request.config.getoption("--record-ref-kernels"))


@pytest.fixture
def ref_ops(request, cuda, _ref_recordings):
    """The reference's own kernels: their outputs stored under tests/golden/ref_kernels/ for the calls this test makes
    (oracle/ref_golden.py), or, with --record-ref-kernels, the live oracle/_ref/libref_ops.so, recorded."""
    from oracle import ref_golden
    name = request.node.originalname
    if request.config.getoption("--record-ref-kernels"):
        from oracle import ref_ops as live
        if not live.available():
            raise RuntimeError("--record-ref-kernels needs oracle/_ref/libref_ops.so (make -C oracle ref)")
        return ref_golden.Recording(live, _ref_recordings.setdefault(name, {}))
    return ref_golden.Stored(os.path.join(ROOT, "tests", "golden", "ref_kernels", name + ".npz"))
