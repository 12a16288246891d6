import os, sys, subprocess
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session", autouse=True)
def _build_oracle():
    """The CPU restatement is test infrastructure: build it if the prebuilt file did not travel."""
    if not os.path.exists(os.path.join(ROOT, "oracle", "liboracle.so")):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "oracle"])
