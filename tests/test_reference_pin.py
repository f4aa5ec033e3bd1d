"""The reference-run pin (SURVEY section 8c, item 3): when a Fortran compiler and the reference sources are available,
build the REAL reference and compare its test/test1 output with the golden vectors the oracle produced
(scripts/pin_against_reference.sh).  Skipped - loudly - where that is impossible (this image has no Fortran compiler):
every 'identical to the reference' claim then means 'identical to the oracle's reading of the reference'."""
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCRIPT = os.path.join(ROOT, "scripts", "pin_against_reference.sh")


def test_pin_kit_is_in_place():
    assert os.access(SCRIPT, os.X_OK) and os.path.exists(os.path.join(ROOT, "scripts", "pin_check.py"))


def test_oracle_is_pinned_against_the_compiled_reference():
    fc = next((c for c in ("gfortran", "flang", "nvfortran") if shutil.which(c)), None)
    ref = os.environ.get("REF")
    if fc is None or not ref or not os.path.exists(os.path.join(ref, "src", "diagnose", "main.f90")):
        pytest.skip("PARITY UNPINNED: needs a Fortran compiler (gfortran/flang/nvfortran) and REF=<XLab-EE-fortran checkout> - "
                    "run scripts/pin_against_reference.sh on a machine that has both")
    r = subprocess.run([SCRIPT], capture_output=True, text=True, timeout=3600)
    assert r.returncode == 0, r.stdout + r.stderr
