import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _have_gpu():
    try:
        import nlopt_b200
        return nlopt_b200.device_count() > 0
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    import reference_runs
    if reference_runs.RECORDING:
        # only the comparisons with the reference run; on a machine without a device the GPU-marked ones skip after
        # their reference side has been recorded (fixture `reference`)
        keep = [it for it in items if "reference" in getattr(it, "fixturenames", ())]
        config.hook.pytest_deselected(items=[it for it in items if it not in keep])
        items[:] = keep
        return
    # GPU tests are selected with `-m gpu` on the GPU box; if they get collected on a machine
    # without a device (plain `pytest tests/`), skip rather than fail.
    if _have_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device visible")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def built():
    """Make sure the product library and the oracle are built (no-op when up to date)."""
    import __graft_entry__ as g
    if not os.path.exists(g.LIB):
        g.build_library()
    port = os.path.join(ROOT, "oracle", "liboracle_port.so")
    if not os.path.exists(port):
        g.build_oracle()
    return g


@pytest.fixture(scope="session")
def reflib(built):
    """The unmodified reference as a Library (oracle/_ref), or skip if it was never built."""
    import oracle_bindings as ob
    from nlopt_b200 import Library
    if not os.path.exists(ob.REF_SO):
        pytest.skip("oracle/_ref/libnlopt_ref.so not built (needs /root/reference at build time)")
    return Library(ob.REF_SO, extensions=False)


@pytest.fixture(scope="session")
def _reference_store(built):
    import reference_runs
    lib = None
    if reference_runs.RECORDING:
        import oracle_bindings as ob
        from nlopt_b200 import Library
        lib = Library(ob.REF_SO, extensions=False)
    store = reference_runs.Store(lib)
    yield store
    store.save()


@pytest.fixture
def reference(request, _reference_store):
    """reference(key, compute) -> the unmodified reference's result of one run, stored under tests/golden
    (tests/reference_runs.py); compute(lib) produces it from the reference library when the results are regenerated."""
    def get(key, compute):
        result = _reference_store.get(key, compute)
        if _reference_store.lib is not None and request.node.get_closest_marker("gpu") and not _have_gpu():
            pytest.skip("reference side recorded; the comparison needs a CUDA device")
        return result
    return get


@pytest.fixture(scope="session")
def hosttest_lib(built):
    """The product's host-side sources (API + CCSA driver + dual optimiser) linked against the
    oracle-backed CPU backend of tests/cpp/oracle_backend.cpp -- host logic without a GPU."""
    from nlopt_b200 import Library
    out = os.path.join(ROOT, "tests", "_build", "libnlopt_hosttest.so")
    srcs = [os.path.join(ROOT, "nlopt_b200", "csrc", f) for f in ("nlopt_api.cpp", "ccsa_driver.cpp")]
    srcs.append(os.path.join(ROOT, "tests", "cpp", "oracle_backend.cpp"))
    deps = srcs + [os.path.join(ROOT, "nlopt_b200", "csrc", f) for f in os.listdir(os.path.join(ROOT, "nlopt_b200", "csrc"))]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        port_o = os.path.join(ROOT, "tests", "_build", "ccsa_port.o")
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-c",
                               os.path.join(ROOT, "oracle", "ccsa_port.c"), "-o", port_o])
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared",
                               "-I/usr/local/cuda/include", *srcs, port_o, "-o", out, "-lm"])
    return Library(out, extensions=False)
