"""pytest configuration: markers and import paths.

CPU suite:  python -m pytest tests -x -q -m "not gpu"
GPU suite:  python -m pytest tests -x -q -m gpu      (on a B200)
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")
    config.addinivalue_line("markers", "live_reference: needs INVERSUS_REFERENCE_ROOT, a checkout of the original project")
