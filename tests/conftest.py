"""pytest configuration: registers the `gpu` marker and builds native artefacts once per session."""
import os
import pathlib
import shutil
import subprocess
import sys
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with `pytest -m gpu` on the GPU box)")


@pytest.fixture
def tmp_path(tmp_path):
    """pytest's tmp_path, or a shorter directory when that one is too deep for the Unix sockets the agent tests bind in it (a long
    TMPDIR, user name or --basetemp would otherwise fail them with "AF_UNIX path too long")."""
    from container_engine_accelerators_b200.agent import testing
    if len(str(tmp_path)) <= testing.SOCKET_DIR_MAX:
        yield tmp_path
        return
    short = tempfile.mkdtemp(prefix="b200-test-", dir=testing.socket_tmp_root())
    yield pathlib.Path(short)
    shutil.rmtree(short, ignore_errors=True)


@pytest.fixture(scope="session")
def native_build():
    """Build the native artefacts once per session (g++ / nvcc cross-compile; no GPU needed)."""
    san = os.environ.get("B200_NATIVE_SAN", "")          # "thread" or "address": run the suite against instrumented binaries
    subprocess.run(["make", "-C", os.path.join(ROOT, "agent", "native"), "-j4"] + ([f"SAN={san}"] if san else []), check=True, capture_output=True)
    return os.path.join(ROOT, "build", "agent" + (f"-{san}" if san else ""))


@pytest.fixture(scope="session")
def coll_lib():
    lib = os.path.join(ROOT, "coll", "lib", "libb200coll.so")
    if not os.path.exists(lib):
        subprocess.run(["make", "-C", os.path.join(ROOT, "coll")], check=True, capture_output=True)
    return lib
