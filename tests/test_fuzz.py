"""Short runs of the two differential fuzzers (scripts/fuzz_oracle.py, scripts/fuzz_readers.py) against the answers the
unmodified reference binary gave for the same seeded cases (tests/golden/fuzz_*.json, written by their --record mode)."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def test_restatement_against_reference_random_cases(built):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "fuzz_oracle.py"), "40", "101",
                        "--replay", os.path.join(GOLDEN, "fuzz_oracle_40_101.json")],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    assert r.returncode == 0, r.stdout.decode()[-3000:]


def test_host_readers_against_reference_tools_random_databases(built):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "fuzz_readers.py"), "10", "102",
                        "--replay", os.path.join(GOLDEN, "fuzz_readers_10_102.json")],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    assert r.returncode == 0, r.stdout.decode()[-3000:]
