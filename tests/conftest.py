import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")
    # build the CPU checkers (oracle restatement always; compiled reference when its tree exists)
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "all"], check=False,
                   capture_output=True)
    shim = os.path.join(ROOT, "tests", "host_shim")
    subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o",
                    os.path.join(shim, "librules_host.so"), os.path.join(shim, "rules_host.cpp")],
                   check=False, capture_output=True)


@pytest.fixture(scope="session")
def oracle():
    from oracle.pyoracle import OracleLib
    return OracleLib()


@pytest.fixture(scope="session")
def ref():
    from oracle.pyoracle import RefLib, have_ref
    if not have_ref():
        pytest.skip("oracle/_ref not built: set CORINTHO_AI_REFERENCE to a checkout of the original project")
    return RefLib()
