#!/usr/bin/env python3
"""Exhaustive host check of the RNG fast paths of rm_math.h (tan_ft_fast, sincos_ft_fast, log_ft_fast): builds
tools/rng_sweep.cpp with the oracle's flags and, for every float of each fast path's domain, compares the fast
result with the pinned function's bit for bit; reports the largest |F - P| in ulps of P against the bound the
rounding test uses, and the fallback rate.  --sass adds the per-call SASS instruction counts of pinned and fast
path (nvcc -arch=sm_100a, tools/rng_probe.cu).

  python tools/rng_sweep.py [--stride 1] [--threads N] [--fn tan sincos log] [--sass] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
DEVICE_SRC = ROOT / "raymarching_engine_b200" / "csrc" / "device_src"
CXXFLAGS = ["-std=c++17", "-O2", "-ffp-contract=off", "-mfma", "-pthread"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def build(tmp: Path) -> Path:
    exe = tmp / "rng_sweep"
    subprocess.run(["g++", *CXXFLAGS, f"-I{DEVICE_SRC}", "-o", str(exe), str(ROOT / "tools" / "rng_sweep.cpp")], check=True)
    return exe


def run(exe: Path, *args) -> list[dict]:
    p = subprocess.run([str(exe), *map(str, args)], capture_output=True, text=True)
    if p.returncode not in (0, 1):
        raise SystemExit(p.stderr)
    return [json.loads(line) for line in p.stdout.splitlines() if line.strip()]


def sass_counts(tmp: Path) -> list[str]:
    """static instructions of one call: each probe kernel's body up to its EXIT, minus that of the copy kernel.
    Out-of-line code after the EXIT - the slow path of the pinned functions' division, the pinned function a
    fast path falls back to - runs only in rare cases and is listed apart."""
    cubin = tmp / "rng_probe.cubin"
    subprocess.run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-cubin", "-O3", "--fmad=false", f"-I{DEVICE_SRC}",
                    "-o", str(cubin), str(ROOT / "tools" / "rng_probe.cu")], check=True)
    out = subprocess.run(["cuobjdump", "-sass", str(cubin)], capture_output=True, text=True, check=True).stdout
    ops, cur = {}, None
    for line in out.splitlines():
        if "Function :" in line:
            cur = line.split("Function :")[1].strip()
            ops[cur] = []
        elif cur and re.match(r"\s+/\*[0-9a-f]{4}\*/", line):
            op = line.split("*/", 1)[1].split(";")[0].strip()
            if op and not op.startswith("NOP"):
                ops[cur].append(op)
    def body(k):
        return next(i for i, o in enumerate(ops[k]) if o.startswith("EXIT")) + 1
    base = body("probe_copy")
    return [f"{k}: {body(k) - base} instructions inline per call, {len(ops[k]) - body(k)} out of line"
            for k in sorted(ops) if k.startswith("probe_") and k != "probe_copy"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--stride", type=int, default=1)
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 1)
    ap.add_argument("--fn", nargs="*", default=["tan", "sincos", "log"])
    ap.add_argument("--sass", action="store_true")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    lines = [f"# tools/rng_sweep.py --stride {a.stride}: g++ {' '.join(CXXFLAGS)}, {a.threads} threads"]
    bad = False
    with tempfile.TemporaryDirectory() as d:
        exe = build(Path(d))
        for fn in a.fn:
            t0 = time.time()
            (r,) = run(exe, fn, a.stride, a.threads)
            r["seconds"] = round(time.time() - t0, 1)
            lines.append(json.dumps(r))
            bad |= r["mismatches"] != 0
        for r in run(exe, "edges"):
            lines.append(json.dumps(r))
            bad |= r["mismatches"] != 0
        if a.sass:
            lines += ["", "# per-call SASS, nvcc -gencode arch=compute_100a,code=sm_100a -O3 --fmad=false (cuobjdump -sass)"]
            lines += sass_counts(Path(d))
    text = "\n".join(lines) + "\n"
    print(text, end="")
    if a.out:
        Path(a.out).write_text(text)
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
