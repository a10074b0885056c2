"""CPU test (no GPU): the fast feature tier's "%.4g" decision table, looked up by exponent byte and one comparison, gives
the same decimal exponent, scale factors and rounded value as the multiply-shift formula, for all 2^32 float bit patterns."""
import os
import subprocess

from conftest import ROOT


def test_round4_table_matches_the_formula_for_every_float(tmp_path):
    exe = str(tmp_path / "r4c")
    subprocess.run(["/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++", "-O2", "-ffp-contract=off", "-pthread", "-o", exe,
                    os.path.join(ROOT, "tests", "round4_table_check.cpp"), "-lm"], check=True)
    out = subprocess.run([exe, str(max(1, min(16, os.cpu_count() or 1)))], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout
    assert "mismatches=0 checked=4294967296" in out.stdout, out.stdout
