import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    # @pytest.mark.timeout comes from pytest-timeout (tests/requirements.txt); without the plugin the marker would be
    # silently ignored and a hang would hang the suite, so a SIGALRM stand-in takes over
    if not config.pluginmanager.hasplugin("timeout"):
        config.addinivalue_line("markers", "timeout(seconds): fail the test after this long (stand-in for pytest-timeout)")


@pytest.hookimpl(hookwrapper=True)
def pytest_runtest_call(item):
    marker = item.get_closest_marker("timeout")
    if marker is None or item.config.pluginmanager.hasplugin("timeout"):
        yield
        return
    import signal

    def _expired(signum, frame):
        raise TimeoutError(f"test exceeded {marker.args[0]} s (conftest stand-in for pytest-timeout)")
    old = signal.signal(signal.SIGALRM, _expired)
    signal.alarm(int(marker.args[0]))
    try:
        yield
    finally:
        signal.alarm(0)
        signal.signal(signal.SIGALRM, old)


def _ensure_built():
    import harness
    need = [harness.ORACLE_SO, harness.HOSTSIM_SO, os.path.join(ROOT, "linne_b200", "liblinne_b200.so")]
    if not all(os.path.exists(p) for p in need):
        import __graft_entry__
        __graft_entry__.build()


@pytest.fixture(scope="session", autouse=True)
def built_libraries():
    _ensure_built()


@pytest.fixture(scope="session")
def oracle():
    import harness
    return harness.Oracle()


@pytest.fixture(scope="session")
def ref():
    import harness
    if not harness.have_ref():
        pytest.skip("oracle/_ref/liblinne_ref.so not present (built only where /root/reference exists)")
    return harness.Ref()


@pytest.fixture(scope="session")
def reference():
    """The reference's answers: live from oracle/_ref where it was built (and checked against the stored ones), else
    the stored ones (tests/golden/reference_record.json)."""
    import harness
    return harness.ReferenceRecord(harness.Ref() if harness.have_ref() else None)


@pytest.fixture(scope="session")
def hostsim():
    import harness
    return harness.HostSim()


@pytest.fixture(scope="session")
def gpu():
    from linne_b200 import Product
    codec = Product()
    if not codec.device_available():
        pytest.fail("no CUDA device: the product has no CPU fallback, gpu tests cannot run")
    return codec
