"""The device-only prover session with the part-wise quotient (tests/cpp/test_quotient_parts.cpp), after a check of the part
forms of the C++ host mirrors against the full coset: at 2^18 rows (extended
2^20) the proofs of two circuits are accepted by both verifiers, and the quotient step never held a column at extended size --
its peak device bytes stay within (2 * columns + J + 1) * n * 32 (coefficient columns, their per-part scratch, one part buffer)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "test_quotient_parts.cpp")


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("quotient_parts") / "test_quotient_parts")
    lib, orc = os.path.join(ROOT, "scroll-prover_b200"), os.path.join(ROOT, "oracle")
    subprocess.check_call(["make", "-s", "-C", orc, "liboracle.so"])
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", out, SRC, "-L" + lib, "-lb200zk", "-Wl,-rpath," + lib, "-L" + orc, "-loracle",
                           "-Wl,-rpath," + orc])
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [1, 2])
def test_device_session_builds_the_quotient_by_parts(driver, variant):
    r = subprocess.run([driver, "18", "3", str(variant)], capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout[-2000:] + r.stderr[-2000:]
    assert "host mirrors: parts, part evaluation and recombination agree" in r.stdout
    line = [l.split() for l in r.stdout.splitlines() if l.startswith("quotient_peak_bytes")][0]
    peak, columns, parts, n = int(line[1]), int(line[3]), int(line[5]), int(line[7])
    assert parts == 4 and n == 1 << 18
    assert 0 < peak <= (2 * columns + parts + 1) * n * 32
