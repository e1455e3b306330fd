"""RNG fast paths of rm_math.h (tan_ft_fast, sincos_ft_fast, log_ft_fast) against the pinned functions on the host.

tools/rng_sweep.cpp is built with the oracle's flags, so it evaluates the same binary64 operations as the device.
Here it checks every 97th float of each fast path's domain, the domain's last float, and the specials, subnormals
and binade edges of every sign and exponent (which covers NaN, +-inf, zero, negative and large arguments outside
the domains): the fast result must equal the pinned one bit for bit, and the measured |F - P| must stay at most a
quarter of the bound the rounding test assumes.  tools/rng_sweep.py runs the same checks on every float of each
domain; tests/test_rng_fast_paths_gpu.py does so on the device.
"""
import json
import os
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
DEVICE_SRC = ROOT / "raymarching_engine_b200" / "csrc" / "device_src"


@pytest.fixture(scope="module")
def sweep(tmp_path_factory):
    exe = tmp_path_factory.mktemp("rng_sweep") / "rng_sweep"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-mfma", "-pthread", f"-I{DEVICE_SRC}", "-o", str(exe),
                    str(ROOT / "tools" / "rng_sweep.cpp")], check=True)

    def run(*args):
        p = subprocess.run([str(exe), *map(str, args)], capture_output=True, text=True)
        assert p.returncode in (0, 1), p.stderr
        return [json.loads(line) for line in p.stdout.splitlines()]
    return run


def _check(r):
    assert r["mismatches"] == 0, r
    assert r["checked"] > 0
    assert 4 * r["max_ulps"] <= r["bound_ulps"], r


@pytest.mark.parametrize("fn", ["tan", "sincos", "log"])
def test_strided_domain(sweep, fn):
    (r,) = sweep(fn, 97, os.cpu_count() or 1)
    _check(r)
    assert r["checked"] > 10_000_000
    assert r["fallback_rate"] < 1e-5, r


def test_edges_and_outside_the_domains(sweep):
    rs = sweep("edges")
    assert [r["fn"] for r in rs] == ["tan", "sincos", "log"]
    for r in rs:
        _check(r)
