"""pytest configuration: the `gpu` marker, import paths and shared fixtures.

`-m "not gpu"` runs here (no GPU): oracle vs the compiled reference and the golden vectors, host logic, C-ABI
export checks.  `-m gpu` runs on a B200: the parity tests proper, all through the C ABI of libavifgpu.so.
"""
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for path in (os.path.join(ROOT, "avif-format_b200", "python"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), ROOT):
    if path not in sys.path:
        sys.path.insert(0, path)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on a B200)")


@pytest.fixture(scope="session")
def port():
    import oracle
    return oracle.load_restatement()


@pytest.fixture(scope="session")
def ref():
    """The compiled reference (oracle/_ref) where it is built; elsewhere the restatement held to the reference's recorded
    results (oracle.RecordedReference).  AVIFGPU_RECORD_REFERENCE=<file> records those results from the compiled reference."""
    import oracle
    compiled = oracle.load_reference()
    record_to = os.environ.get("AVIFGPU_RECORD_REFERENCE")
    if compiled is None:
        if record_to:
            pytest.fail("AVIFGPU_RECORD_REFERENCE needs the compiled reference (oracle/_ref/libavifref.so)")
        recorded = oracle.load_recorded_reference()
        if recorded is None:
            pytest.skip("the reference's results were recorded with another libm and oracle/_ref is not built")
        yield recorded
    elif record_to:
        recorder = oracle.ReferenceRecorder(compiled)
        yield recorder
        recorder.save(record_to)
    else:
        yield compiled


@pytest.fixture(scope="session")
def checker():
    """The strongest CPU checker available: the compiled reference, else the restatement."""
    import oracle
    return oracle.best_checker()


@pytest.fixture(scope="session")
def gpu_exact():
    """A context that never builds step tables: float encodes run the exact kernel (glibc-identical powf per sample)."""
    import avifgpu
    ctx = avifgpu.Context(0)
    ctx.set_table_autobuild(-1)
    yield ctx
    ctx.close()


@pytest.fixture(scope="session")
def gpu():
    import avifgpu
    ctx = avifgpu.Context(0)
    ctx.set_table_autobuild(0)  # the tests exercise the step tables: build them at first use, whatever the image size
    yield ctx
    ctx.close()
