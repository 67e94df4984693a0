"""pytest configuration: marker registration and shared fixtures.

``-m "not gpu"`` runs here (no GPU): oracle vs. golden vectors / reference, host
logic, C-ABI symbol checks.  ``-m gpu`` runs on a B200 and is the parity suite
proper (CUDA path vs. oracle through the C ABI).
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# Stable small argsort + libm transcendentals in NumPy (see oracle/ref_loader.py).
# Must happen before NumPy is first imported by the test process.
from oracle import ref_loader  # noqa: E402

# NumPy reads the pin once, when it is first imported.  pytest.ini disables the plugins
# that import it before this file runs; when they load anyway (settings overridden, or a
# plugin given on the command line), pytest_configure restarts the session with the pin
# in its environment, because the goldens hold argsort tie orders and float32 libm
# results that NumPy's AVX paths do not reproduce.  A NPY_DISABLE_CPU_FEATURES of the
# caller's own is kept; if NumPy was imported first under it, tests that compare NumPy-oracle
# floats bit-for-bit fall back to a 1e-6 tolerance.
_PIN_EFFECTIVE = ref_loader.numpy_is_pinned() or "numpy" not in sys.modules
ref_loader.pin_numpy_env()
os.environ["MGD_NUMPY_PIN_EFFECTIVE"] = "1" if _PIN_EFFECTIVE else "0"

import pytest  # noqa: E402


def _restart_with_numpy_pin(config):
    """Replace this process by the same command, now with NPY_DISABLE_CPU_FEATURES set
    (ref_loader.pin_numpy_env put it in os.environ), so NumPy starts pinned.  The restarted
    process sees the pin and does not restart again.  The whole program is executed anew: for
    `pytest` / `python -m pytest` that is the session itself; a program that calls
    pytest.main() is run again from its start, with the pin already set from then on."""
    capman = config.pluginmanager.getplugin("capturemanager")
    if capman is not None:
        capman.stop_global_capturing()
    sys.stdout.flush()
    sys.stderr.flush()
    os.execv(sys.executable, [sys.executable, *sys.orig_argv[1:]])


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    # only when the pin is ours: a NPY_DISABLE_CPU_FEATURES the caller set is left alone
    if not _PIN_EFFECTIVE and ref_loader.numpy_is_pinned():
        _restart_with_numpy_pin(config)


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def c_oracle():
    from oracle import c_oracle as co
    co.build()
    return co
