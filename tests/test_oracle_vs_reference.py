"""CPU: the oracle against the UNMODIFIED original project on the cases of oracle/check_vs_reference.py (fresh seeds and
shapes that the fixtures of oracle/make_golden.py do not use).  Every run compares the oracle with the expected outputs
stored in tests/golden/live_check.npz; where ref_shim finds the original, the script also runs it live and checks both
the oracle and the stored outputs against it."""
import os
import subprocess
import sys

import pytest

import check_vs_reference as C
import ref_shim
from conftest import ROOT


def test_oracle_matches_stored_live_check_outputs():
    inp, expected, source = C.load_fixture()
    C.compare(C.oracle_outputs(inp), expected, f"oracle vs stored ({source})")


@pytest.mark.skipif(not ref_shim.reference_available(), reason="the original project is not available to ref_shim")
def test_oracle_matches_live_reference():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "check_vs_reference.py")], capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert r.stdout.count("ok ") >= 3, r.stdout
