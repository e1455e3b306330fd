#!/usr/bin/env python3
"""One-process sweep of RMB_MARCH_PLAN (rmb_api.cpp "march stage": budget:threads:ctas_per_sm:pause per pass) on the
default bench workload: frames of the orbit path, one context, L2 flushed per frame, march-kernel time from the
library's CUDA-event timer and frame time from events around the whole sequence.  The plan is read at every draw, so
no recompilation is needed between rows.  Before a plan is timed, frame 0 of the orbit is rendered under it and its
RGBA8, depth bits and SDF evaluation count are compared with the first plan's: a plan that differs (lost or repeated
rays) prints MISMATCH instead of a timing row.

  python tools/sweep_plan.py [--width 1920 --height 1080] [--mode preview] [--steps 12] plan [plan ...]
"""
import argparse
import os
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--mode", default="preview")
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--flavour", default="exact")
    ap.add_argument("--ranks", type=int, default=1, help="emulate one rank of an N-rank row-tile split (rank 0's tiles only): the per-GPU work of --shard tiles")
    ap.add_argument("plans", nargs="+")
    a = ap.parse_args()
    import numpy as np
    import torch
    import bench
    import raymarching_engine_b200 as rm
    L = rm._lib.lib
    flavour = rm.FLAVOUR_FAST if a.flavour == "fast" else rm.FLAVOUR_EXACT
    ctx = rm.load_render_job_context(device=0, rank=0, n_ranks=a.ranks, tile_rows=16, flavour=flavour, specialize="always")
    src = (ROOT / "scenes" / "guide.glsl").read_text()
    custom = rm.default_custom_settings(src)
    prog = ctx.program_cache.get_program(src, None, custom)
    assert isinstance(prog, rm.Program), prog
    stream = torch.cuda.ExternalStream(ctx.stream())
    flush = torch.empty(160 << 20, dtype=torch.uint8, device="cuda")
    W, H = a.width, a.height
    frame = [10]

    def step(pose):
        with torch.cuda.stream(stream):
            flush.zero_()
        frame[0] += 1
        s = bench.make_schema(rm, src, custom, W, H, a.mode, pose, frame[0])
        fb = ctx.fbo.create(W, H, s.render.frameid)
        rm.upload_sample_uniforms(prog, s, (0.5, 1.0 / 3.0))
        assert L.rmb_render_sample(ctx.handle, prog.handle, fb.handle, 0, 0, W, H) == 0, ctx.last_error()
        assert L.rmb_present_device(ctx.handle, fb.handle, 1.0) == 0
        ctx.fbo.delete(W, H, s.render.frameid)

    def frame0():
        """RGBA8, depth bits and SDF evaluations of orbit frame 0 under the current plan"""
        frame[0] += 1
        s = bench.make_schema(rm, src, custom, W, H, a.mode, 0, frame[0])
        fb = ctx.fbo.create(W, H, s.render.frameid)
        rm.upload_sample_uniforms(prog, s, (0.5, 1.0 / 3.0))
        ctx.counters_all(reset=True)
        assert L.rmb_render_sample(ctx.handle, prog.handle, fb.handle, 0, 0, W, H) == 0, ctx.last_error()
        rgba, depth = ctx.present(fb, 1.0)
        out = (rgba.copy(), depth.view(np.uint32).copy(), ctx.counters_all(reset=True)[0])
        ctx.fbo.delete(W, H, s.render.frameid)
        return out

    print(f"# {W}x{H} {a.mode} {a.flavour}; ms per frame incl. a 160 MiB L2 flush (~0.05 ms); march = all march launches of a frame")
    want = None
    for plan in a.plans:
        os.environ["RMB_MARCH_PLAN"] = plan
        got = frame0()
        if want is None:
            want = got
        elif not (np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[2] == want[2]):
            px = int(np.any(got[0] != want[0], axis=-1).sum())
            print(f"{plan:44s} MISMATCH with {a.plans[0]}: {px} RGBA8 pixels and {int((got[1] != want[1]).sum())} depth values "
                  f"differ, {got[2]} SDF evaluations against {want[2]}", flush=True)
            continue
        for i in range(4):
            step(i)
        ctx.sync()
        ctx.timing(True)
        ctx.counters3(reset=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(a.steps):
            step(5 + i)
        e1.record(stream)
        ctx.sync()
        hot_ms, n = ctx.timing(False)
        call = ctx.counters_all(reset=True)
        ev, px, far = call[0], call[1], call[2]
        tot = e0.elapsed_time(e1) / a.steps
        frac = (ev - far) * 282.0 / (hot_ms * 1e-3) / 1e12 / 74.45 if hot_ms else 0
        print(f"{plan:44s} frame {tot:7.4f} ms  march {hot_ms / a.steps:7.4f} ms ({n // a.steps} launches)  march frac {frac:.3f}  Mpx/s {W * H / tot / 1e3:8.1f}", flush=True)
        if call[7]:     # RMB_PROFILE=1: per-warp timeline of the march kernel, summed over launches and frames
            warps, bulk_ns, drain_ns, it_b, it_d, mx, ln_b, ln_d = call[7], call[3], call[4], call[5], call[6], call[8], call[9], call[10]
            print(f"    per warp: bulk {bulk_ns / warps / 1e3:7.1f} us ({it_b / warps:6.1f} iterations, {bulk_ns / max(it_b, 1):6.0f} ns each, {ln_b / max(it_b, 1):4.1f} lanes live)   "
                  f"drain {drain_ns / warps / 1e3:7.1f} us ({it_d / warps:6.1f} iterations, {drain_ns / max(it_d, 1):6.0f} ns each, {ln_d / max(it_d, 1):4.1f} lanes live)   "
                  f"longest warp {mx / 1e3:7.1f} us   warps/frame {warps / a.steps:.0f}", flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
