"""Shared fixtures. `-m "not gpu"` runs here (no GPU); `-m gpu` runs on a B200 box.

Only tests (and smoke / bench's cpu_baseline leg) may execute anything under oracle/.
"""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

GOLDEN = os.path.join(ROOT, "tests", "golden")
ORACLE_BIN = os.path.join(ROOT, "oracle", "gaml_oracle")
REF_HARNESS = os.path.join(ROOT, "oracle", "_ref", "ref_harness")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session", autouse=True)
def built():
    """Builds the CUDA library, the oracle and (when /root/reference exists) oracle/_ref once per session."""
    import __graft_entry__ as entry
    entry.build()
    return True


def run_scorer(binary, wl_or_path, tmp_path, name="case", dump=True):
    """Runs oracle/gaml_oracle or oracle/_ref/ref_harness on a workload, returns the parsed results."""
    from gaml_b200 import workload
    if isinstance(wl_or_path, str):
        wp = wl_or_path
    else:
        wp = os.path.join(str(tmp_path), name + ".wl")
        workload.write_workload(wp, wl_or_path)
    rp = os.path.join(str(tmp_path), name + "." + os.path.basename(binary) + ".res")
    subprocess.run([binary, wp, rp, "1" if dump else "0"], check=True, cwd=str(tmp_path), stdout=subprocess.DEVNULL,
                   stderr=subprocess.DEVNULL)
    return workload.read_results(rp)


@pytest.fixture
def oracle(tmp_path):
    def _run(wl, name="case", dump=True):
        return run_scorer(ORACLE_BIN, wl, tmp_path, name, dump)
    return _run
