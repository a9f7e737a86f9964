"""INTEGRATION.md section 1, executed: the reference's own data and plot mixins composed with MarginalB200.

Needs the reference's sources, which are not part of this repository: set DISCONTINUUM_REFERENCE to the src/ directory of a
discontinuum checkout to run it; without it this test reports "skipped".  The scenario lives in
tests/reference_integration_check.py and runs in a fresh process, because it installs stand-in `xarray` / `matplotlib`
modules before anything else is imported."""
import os
import subprocess
import sys

import pytest

REF = os.environ.get("DISCONTINUUM_REFERENCE", "")


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "loadest_gp")),
                    reason="set DISCONTINUUM_REFERENCE to the reference's src/ directory to run this")
def test_reference_mixins_run_unchanged_on_marginal_b200():
    here = os.path.dirname(os.path.abspath(__file__))
    r = subprocess.run([sys.executable, os.path.join(here, "reference_integration_check.py")], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "INTEGRATION OK" in r.stdout
    assert "plot_ratings_in_time" in r.stdout and "contourf ok" in r.stdout
