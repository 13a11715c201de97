import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# compiled patch kernels of the test runs stay inside the repository (the library's default is ~/.cache/maxib200); the directory does not
# travel to the GPU box (.gpurunignore), so the run-time compiler is exercised there
os.environ.setdefault("MXB_PATCH_CACHE", os.path.join(ROOT, ".mxb_cache"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def port():
    """The plain-C restatement oracle (always buildable: gcc only)."""
    from oracle import oracle_py
    oracle_py.build("port")
    return oracle_py


@pytest.fixture(scope="session")
def reference_traces():
    """The stored reference traces, and the compiled reference where oracle/Makefile can build it or it was built before."""
    import reference_trace
    from oracle import oracle_py
    oracle_py.build("reference")                      # leaves oracle/_ref/ as it is where the reference sources are absent
    store = reference_trace.Store()
    yield store, (oracle_py if oracle_py.available("reference") else None)
    store.save()


@pytest.fixture
def reference(request, port, reference_traces):
    """The compiled reference's side of a bit-for-bit pin (tests/reference_trace.py): reference.check(run) compares run("port")
    with the stored trace of run("reference"), and with a live run of the reference where it is built."""
    import reference_trace
    store, live = reference_traces
    return reference_trace.Trace(reference_trace.key(request.node), store, live)


@pytest.hookimpl(tryfirst=True)
def pytest_collection_modifyitems(items):
    """Every pinned test collected, before -k / -m deselect any: recording drops the stored traces of pins that no longer exist."""
    import reference_trace
    reference_trace.COLLECTED.update(reference_trace.key(it) for it in items if "reference" in getattr(it, "fixturenames", ()))
