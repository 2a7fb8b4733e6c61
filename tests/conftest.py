import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def pytest_sessionstart(session):
    """Make sure the native pieces exist before any test imports them: libvdl2gpu.so (nvcc cross-compiles without
    a GPU) and the oracle."""
    try:
        from dumpvdl2_b200.build import build_native
        build_native()
    except Exception as e:          # on a box without nvcc the prebuilt .so that travelled with the repo is used
        print(f"[conftest] libvdl2gpu.so not rebuilt: {e}", file=sys.stderr)
    try:
        from oracle import pyoracle
        pyoracle.build()
    except Exception as e:
        print(f"[conftest] oracle not rebuilt: {e}", file=sys.stderr)
