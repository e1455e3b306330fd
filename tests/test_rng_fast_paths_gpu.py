"""RNG fast paths of rm_math.h on the device: tools/rng_probe.cu, built here with nvcc for sm_100a, compares
tan_ft_fast, sincos_ft_fast and log_ft_fast with the pinned functions on every float of each fast path's domain
and on the specials, subnormals and binade edges of all signs and exponents, bit for bit.  It is built twice: with
--fmad=false and --fmad=true, the flags of the exact and the fast flavour, so a contraction or reordering by the
compiler in either would show.
"""
import json
import os
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
DEVICE_SRC = ROOT / "raymarching_engine_b200" / "csrc" / "device_src"
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


@pytest.mark.gpu
@pytest.mark.parametrize("fmad", ["false", "true"])
def test_every_float_of_each_domain_on_the_device(tmp_path, fmad):
    exe = tmp_path / "rng_probe"
    subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", f"--fmad={fmad}", f"-I{DEVICE_SRC}",
                    "-o", str(exe), str(ROOT / "tools" / "rng_probe.cu")], check=True)
    p = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert p.returncode in (0, 1), p.stdout + p.stderr
    rs = [json.loads(line) for line in p.stdout.splitlines()]
    assert [(r["fn"], r["set"]) for r in rs] == [(f, s) for f in ("tan", "sincos", "log") for s in ("domain", "edges")]
    for r in rs:
        assert r["mismatches"] == 0, r
    assert sum(r["checked"] for r in rs if r["set"] == "domain") > 3_000_000_000
    assert p.returncode == 0
