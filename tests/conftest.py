import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def orc():
    from tests.checker import get_checker, have
    if not have("orc"):
        import subprocess
        subprocess.check_call(["make", "-s", "-C", str(ROOT / "oracle"), "-f", "Makefile", "oracle"])
    return get_checker("orc")


@pytest.fixture(scope="session")
def engine():
    from openpano_b200.capi import Engine
    eng = Engine(0)
    yield eng
    eng.close()
