import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle_mod():
    """The parity oracle (test infrastructure).  Builds the C restatement on first use."""
    import oracle
    if not os.path.exists(oracle.PORT_LIB):
        oracle.build()
    return oracle


@pytest.fixture(scope="session")
def gpu_ctx():
    import defuse_b200
    return defuse_b200.default_context(0)


@pytest.fixture(scope="session")
def device_double(tmp_path_factory):
    """tests/device_double built into a temporary directory: the eight C-ABI entry points the tools call, answered by
    the parity oracle, for running the tools with LD_PRELOAD where there is no GPU."""
    out = tmp_path_factory.mktemp("device_double")
    obj, lib = str(out / "dp_oracle.o"), str(out / "libdevice_double.so")
    subprocess.run(["gcc", "-O2", "-fPIC", "-c", os.path.join(ROOT, "oracle", "dp_oracle.c"), "-o", obj], check=True)
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "include"), "-o", lib,
                    os.path.join(ROOT, "tests", "device_double", "device_double.cpp"), obj, "-lpthread", "-Wl,--no-undefined"],
                   check=True)
    return lib
