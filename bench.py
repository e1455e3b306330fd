#!/usr/bin/env python3
"""bench.py -- headline benchmark of the hot path (BASELINE.json: megapixels/s and Msteps/s on the
default scene at 1080p, 1/2/4/8 B200, against the reference shader run on the CPU).

A "step" is a BATCH of `--frames-per-step` (default 32) consecutive frames of the synthetic camera path: each frame is
one raymarch sample of the default scene (scenes/guide.glsl - byte-identical to the reference's - with its @default
uniforms, reference-default preview mode) at 1920x1080 into a fresh framebuffer, followed by the display pass.  Pose 0
of the path is the reference's start-up view (camera at the origin looking down +z, SURVEY.md 8d config 1/2); pose k
orbits bigSphereCenter at radius 10 by 2*pi*k/256 (config 5).

  value      frames resident in HBM (no host copies in the timed region), CUDA events on the library's streams over
             all K steps, max over ranks
  e2e        the same frames through the public API (raymarching_engine_b200.render_frames = do_render_job +
             presenter per frame): uniforms from host memory, RGBA8 read back to pinned host memory every frame
             (the reference's canvas; `--e2e-depth` adds the fp32 depth plane), host wall clock, max over ranks
  roofline   the march kernel against the FP32 FMA pipe (this path is FP32-bound, not HBM- or tensor-bound:
             SURVEY.md 8d): executed full SDF evaluations (counted by the kernel) x 282 algorithmic flop per preview
             step / the kernel's own time, measured in a separate pass on ONE context with CUDA events around every
             march launch
  --impl reference   the CPU restatement of the reference shader (oracle/, see its header: the reference itself needs
             a browser WebGL stack that does not exist here) on all host cores; loads nothing of the product

N > 1 (torchrun): the headline keeps BASELINE.json's metric - 1080p frames of the path dealt to the ranks (independent
units, no data-path collective, weak scaling) - and the same JSON line carries `config3_tiles`: BASELINE.json config 3,
3840x2160 frames split into interleaved 16-row tiles across the ranks with the gather fused into the display kernel's
stores (peer memory over NVLink), strong scaling; at N = 1 `config3_tiles` holds the single-GPU 4K figure the N > 1
runs are compared with.

--dump-outputs DIR   after the timed steps, what the device-resident loop (rank 0's) computed in its last step: per
             frame the arrays run_job hands a caller, DIR/rgba8.npy [frames, pixels, 4] and DIR/depth.npy [frames,
             pixels] (float32), so that two builds can be compared output for output.  The frames of that step are
             copied device to device right after their display pass (inside the timed region: 8 B/px for those frames
             only); when they exceed DUMP_BYTES, the same fixed, seeded sample of pixels (row-major index into the
             W x H frame, row 0 at the bottom) is kept from every frame.  The inputs depend on the arguments only.
"""
from __future__ import annotations

import argparse
import importlib
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time
import types
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

FLOP_PER_PREVIEW_STEP = 282.0   # SURVEY.md 8d: 272 per SDF evaluation + 10 for advance/depth/compares
FLOP_PER_CASTRAY_STEP = 278.0
# a far-field step of a carved scene (include/rmb.h rmb_program_has_carve) evaluates only the outer shape:
# length(p - c) - R = 3 sub + 5 (dot) + 1 sqrt + 1 sub, plus the same 10 / 6 for advance, depth and compares
FLOP_PER_FAR_PREVIEW_STEP = 20.0
FLOP_PER_FAR_CASTRAY_STEP = 16.0
# BASELINE.json config 4 (scenes/mandelbulb.glsl, synthetic - SURVEY.md 8d has no count for it; same convention: FMA = 2,
# every other operation and every transcendental = 1, uniform-only sub-expressions hoisted).  One trip of the DE loop:
# length 6 + bailout compare 1 + z.z / r 1 + acos 1 + atan 1 + (pow, * power, fma) 4 + pow 1 + 2 angle products 2 +
# 2 sin + 2 cos 4 + 2 products 2 + zr * v + position (3 fma) 6 = 29 flop, 9 of them transcendental (in the fast flavour
# 11 MUFU operations: rsq, rcp, 2 x (lg2 + ex2), 2 sin, 2 cos, rsq of acos); per evaluation the trip that bails out
# (length + compare, 7) and the tail 0.5 * log(r) * r / dr (4).  The trips per evaluation are data-dependent: measured
# by the oracle on the workload's own rays (pyoracle.executed_work, cpu_baseline leg), else the pinned figure below
# (oracle, 320x180, poses 0 / 37 / 101 / 200 of the orbit: 2.44 trips per executed evaluation, 29 evaluations per pixel).
MANDELBULB_FLOP_PER_DE_TRIP = 29.0
MANDELBULB_FLOP_PER_EVAL_TAIL = 11.0
MANDELBULB_MUFU_PER_DE_TRIP = 11.0
MANDELBULB_DE_TRIPS_PER_EVAL_PINNED = 2.44
N_POSES = 256
FLUSH_BYTES = 160 << 20   # > the 126 MB L2 of a B200
DUMP_BYTES = 48 << 20     # --dump-outputs: float32 bytes written at most


# orbit centre and radius of the synthetic camera path per scene (default: the guide scene's
# bigSphereCenter = (0,0,10), radius 10, so that pose 0 is the reference's start-up view at the origin)
SCENE_ORBITS = {"mandelbulb": ((0.0, 0.0, 0.0), 3.0)}


def orbit_pose(k: int, scene: str = "guide"):
    """Pose k of the synthetic camera path: a circle in the XZ plane around the scene's centre, looking
    at the centre.  rotation = gl-matrix mat4.fromYRotation(-theta), column-major."""
    (cx, cy, cz), radius = SCENE_ORBITS.get(scene, ((0.0, 0.0, 10.0), 10.0))
    theta = 2.0 * math.pi * (k % N_POSES) / N_POSES
    c, s = math.cos(theta), math.sin(theta)
    position = (cx + radius * s, cy, cz - radius * c)
    phi = -theta
    cp, sp = math.cos(phi), math.sin(phi)
    rotation = (cp, 0.0, -sp, 0.0, 0.0, 1.0, 0.0, 0.0, sp, 0.0, cp, 0.0, 0.0, 0.0, 0.0, 1.0)
    # forward = rotation * (0,0,1) = (sp, 0, cp) = (-sin theta, 0, cos theta): towards the centre
    return position, rotation


def make_schema(rm, src, custom, W, H, mode, pose, frameid, scene="guide", step_counts=None, spp=1):
    """`rm`: anything with default_schema / default_light (the product package, or the host-only modules)"""
    s = rm.default_schema(src, custom, width=W, height=H, renderMode=mode, frameid=frameid, samplesPerPixel=spp)
    s.camera.position, s.camera.rotation = orbit_pose(pose, scene)
    if step_counts:
        s.reflectionIterationCounts = list(step_counts)
    if mode == "full":
        s.lights = [rm.default_light()]
        if scene in SCENE_ORBITS:       # the default light sits at the origin: move it outside this scene's object
            s.lights[0].position = (2.0, 3.0, -4.0)
    return s


def host_only_modules():
    """schema.py / params.py of the product WITHOUT the package __init__ (which loads libraymarch_b200.so): the
    reference arm and the cpu_baseline leg describe the workload with the same dataclasses but must not map the
    product library (VERDICT r1: the reference arm's `native_so_loaded` listed it)."""
    name = "rmb_hostonly"
    if name not in sys.modules:
        pkg = types.ModuleType(name)
        pkg.__path__ = [str(ROOT / "raymarching_engine_b200")]
        sys.modules[name] = pkg
    ns = types.SimpleNamespace()
    schema = importlib.import_module(name + ".schema")
    params = importlib.import_module(name + ".params")
    ns.default_schema, ns.default_light, ns.default_custom_settings = schema.default_schema, schema.default_light, params.default_custom_settings
    return ns


class ClockSampler:
    """Samples nvidia-smi clocks and throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_sample(W, H, mode, band_rows, nthreads=None, scene="guide", counts=None):
    """Times the CPU restatement of the reference shader (oracle/) on a band of `band_rows` rows of
    one W x H frame (every pixel costs the same in the reference: no early exit), plus the display
    pass scaled to the band.  Returns (Mpx/s, seconds, cores, description).  Loads oracle/liboracle.so and the
    host-only schema/params modules - nothing else of the product."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import pyoracle
    ho = host_only_modules()
    src = (ROOT / "scenes" / f"{scene}.glsl").read_text()
    custom = ho.default_custom_settings(src)
    s = make_schema(ho, src, custom, W, H, mode, 0, 0, scene, counts)
    cores = nthreads or os.cpu_count() or 1
    acc = pyoracle.Accumulators(W, H)
    U = pyoracle.uniforms_from_schema(s, (0.5, 1.0 / 3.0))
    y0 = max(0, (H - band_rows) // 2)
    t0 = time.perf_counter()
    pyoracle.render_sample(scene, custom, U, acc, (0, y0, W, band_rows), cores)
    t1 = time.perf_counter()
    pyoracle.display(acc, 1.0, cores)
    t2 = time.perf_counter()
    px = W * min(band_rows, H)
    secs = (t1 - t0) + (t2 - t1) * (px / (W * H))
    return px / secs / 1e6, secs, cores, f"{W}x{min(band_rows, H)} band of one {W}x{H} {mode}-mode frame, raymarch + display, {cores} threads"


def mandelbulb_de_trips_per_eval(counts):
    """DE-loop trips per executed SDF evaluation of the config-4 workload, from the oracle's early-out analysis of the
    workload's own camera rays (part of the cpu_baseline leg: loads oracle/liboracle.so)."""
    sys.path.insert(0, str(ROOT / "oracle"))
    import pyoracle
    ho = host_only_modules()
    src = (ROOT / "scenes" / "mandelbulb.glsl").read_text()
    custom = ho.default_custom_settings(src)
    evals = trips = 0
    for pose in (0, 37, 101, 200):
        s = make_schema(ho, src, custom, 320, 180, "preview", pose, 0, "mandelbulb", counts or [512.0])
        e, t = pyoracle.executed_work("mandelbulb", s)
        evals, trips = evals + e, trips + t
    return trips / max(evals, 1)


def _json_safe(x):
    if isinstance(x, float) and (math.isnan(x) or math.isinf(x)):
        return None
    if isinstance(x, dict):
        return {k: _json_safe(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_json_safe(v) for v in x]
    return x


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The reference cannot be
    executed here (TypeScript + GLSL in a browser; no Node, browser or GL stack in this image), so this
    arm times oracle/ - the CPU restatement of its shader - on all host cores (kind "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    W, H = args.width, args.height
    band = args.ref_band_rows
    vals = []
    for i in range(args.warmup + args.steps):
        mpx, secs, cores, desc = cpu_reference_sample(W, H, args.mode, band, None, args.scene, step_counts_of(args) if args.step_counts else None)
        if i >= args.warmup:
            vals.append((mpx, secs))
    total_s = sum(s for _, s in vals)
    px = W * min(band, H) * len(vals)
    value = px / total_s / 1e6
    line = {
        "impl": "reference", "metric": metric_name(args), "value": value, "unit": "Mpx/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_s / max(len(vals), 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": "Mpx/s", "cores": cores, "kind": "port", "sample": "each step: " + desc},
        "e2e": {"value": value, "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "extra": {"msteps_per_s_ref_equiv": value * ref_steps_per_px(args),
                  "product_library_loaded": any("libraymarch_b200" in ln for ln in open("/proc/self/maps"))},
    }
    print(json.dumps(_json_safe(line)), flush=True)


def step_counts_of(args):
    return [float(x) for x in args.step_counts.split(",")] if args.step_counts else [128.0, 128.0, 64.0, 32.0, 32.0]   # index.tsx:321


def ref_steps_per_px(args) -> float:
    """SDF evaluations per pixel-sample the reference executes (SURVEY.md section 3.3): preview steps[0];
    full sum(steps) * (1 + lights) + 5 per bounce (4 normal probes + the subsurface probe), 1 light."""
    c = step_counts_of(args)
    return c[0] if args.mode == "preview" else sum(c) * 2 + 5.0 * len(c)


def metric_name(args) -> str:
    what = "default scene (guide.glsl)" if args.scene == "guide" else f"{args.scene}.glsl"
    return f"megapixels/s, {what} {args.width}x{args.height}, {args.mode} mode" + (f", {args.spp} spp" if args.spp > 1 else "")


def workload_config(args) -> dict:
    what = "guide.glsl default scene" if args.scene == "guide" else f"{args.scene}.glsl"
    return {"workload": f"{what}, {args.width}x{args.height}, {args.mode} mode, {args.spp} spp/frame, steps {step_counts_of(args)}, "
                        f"256-pose orbit camera path (pose 0 = reference start-up view), fresh framebuffer per frame; "
                        f"one step = a batch of {args.frames_per_step} consecutive frames",
            "frames_per_step": args.frames_per_step,
            "flavour": args.flavour, "pipeline": args.pipeline, "shard": args.shard if args.gpus > 1 else "none",
            "contexts_per_gpu": args.contexts, "gather": args.gather if (args.gpus > 1 and args.shard == "tiles") else "none",
            "l2": "flushed between timed iterations: a 160 MiB in-stream device memset (the L2 is shared by all streams) before each "
                  "step (= batch of frames), inside the timed region; within a step the frames rotate through the contexts' "
                  "framebuffer sets and ray planes (72 B/px per frame in flight); the kernel-alone roofline pass flushes before "
                  "every frame; e2e alternates two framebuffer sets per context (40 B/px each) and reads every frame back",
            "steps_per_px_reference": ref_steps_per_px(args)}


class OutputDump:
    """--dump-outputs: device copies of the RGBA8 and depth planes of the `frames` frames of the last timed step."""

    def __init__(self, torch, frames, W, H):
        import numpy as np
        self.rgba8 = torch.empty((frames, H * W, 4), dtype=torch.uint8, device="cuda")
        self.depth = torch.empty((frames, H * W), dtype=torch.float32, device="cuda")
        keep = min(H * W, DUMP_BYTES // (frames * 5 * 4))
        # RandomState: its stream is frozen across numpy versions, so every build samples the same pixels
        index = np.arange(H * W) if keep == H * W else np.sort(np.random.RandomState(0).permutation(H * W)[:keep])
        self.index = torch.from_numpy(index).to("cuda")

    def slot(self, k):
        """(RGBA8, depth) device addresses for frame k of the step"""
        return self.rgba8[k].data_ptr(), self.depth[k].data_ptr()

    def write(self, directory):
        import numpy as np
        os.makedirs(directory, exist_ok=True)
        np.save(os.path.join(directory, "rgba8.npy"), self.rgba8[:, self.index].float().cpu().numpy())
        np.save(os.path.join(directory, "depth.npy"), self.depth[:, self.index].cpu().numpy())


class Rig:
    """The contexts, programs and streams of one workload shape on this rank: (W, H, mode, tiles?)."""

    def __init__(self, rm, torch, args, W, H, tiles, dist, rank, world, local, nctx):
        self.rm, self.torch, self.args, self.W, self.H, self.tiles, self.dist = rm, torch, args, W, H, tiles, dist
        self.rank, self.world, self.local, self.nctx = rank, world, local, nctx
        self.L = rm._lib.lib
        flavour = rm.FLAVOUR_FAST if args.flavour == "fast" else rm.FLAVOUR_EXACT
        dev = torch.device("cuda", local)
        self.ctxs = []
        for _ in range(nctx):
            c = rm.load_render_job_context(device=local, rank=rank if tiles else 0, n_ranks=world if tiles else 1, tile_rows=16,
                                           flavour=flavour, pipeline=args.pipeline)
            if c is None:
                raise SystemExit("bench.py: " + rm.context_error())
            self.ctxs.append(c)
        self.src = (ROOT / "scenes" / f"{args.scene}.glsl").read_text()
        self.custom = rm.default_custom_settings(self.src)
        self.counts = step_counts_of(args) if args.step_counts else None
        h2, h3 = rm.halton(2), rm.halton(3)
        self.sample_noise = [(next(h2), next(h3)) for _ in range(args.spp)]   # every frame restarts the sequence
        self.streams = [torch.cuda.ExternalStream(c.stream(), device=dev) for c in self.ctxs]
        self.flush_bufs = [torch.empty(FLUSH_BYTES, dtype=torch.uint8, device="cuda") for _ in self.ctxs]
        self.progs = []
        for c in self.ctxs:
            prog = c.program_cache.get_program(self.src, None, self.custom)
            if not isinstance(prog, rm.Program):
                raise SystemExit("bench.py: program failed to compile: " + prog.infoLog)
            self.progs.append(prog)
        self.frame_counter = [1 + (7 if tiles else 0) * 1000000]
        self.gather_state = {}
        self.fused = None
        if tiles and world > 1 and args.gather in ("fused", "fused-nccl"):
            from raymarching_engine_b200.sharding import FusedTileGather
            self.fused = FusedTileGather(self.ctxs, W, H, dist, slots=2 * nctx, blur=(args.mode == "full"),
                                         sync="nccl" if args.gather == "fused-nccl" else "flags")

    def pose_of(self, frame):   # weak scaling: rank r renders poses r, r+world, ...; tiles: everyone renders pose `frame`
        return frame if self.tiles else frame * self.world + self.rank

    def schema(self, frame):
        self.frame_counter[0] += 1
        a = self.args
        return make_schema(self.rm, self.src, self.custom, self.W, self.H, a.mode, self.pose_of(frame), self.frame_counter[0], a.scene, self.counts, a.spp)

    def _gather_tiles(self, ctx, stream, fb):
        # NCCL gather of each rank's RGBA8 rows to rank 0 (SURVEY.md 8e): equal-sized padded buffers (ranks own 1..2
        # tiles more or less), issued in the library's stream order; the comparison arm of the fused gather
        torch, W, H, world = self.torch, self.W, self.H, self.world
        g = self.gather_state.setdefault(id(ctx), {})
        if "send" not in g:
            max_rows = -(-H // (16 * world)) * 16
            g["send"] = torch.zeros(max_rows * W * 4, dtype=torch.uint8, device="cuda")
            g["recv"] = [torch.empty_like(g["send"]) for _ in range(world)] if self.rank == 0 else None
        n = fb.local_rows * W * 4
        st = self.L.rmb_fb_copy_to_device(ctx.handle, fb.handle, 4, g["send"].data_ptr(), n)
        assert st == 0, ctx.last_error()
        with torch.cuda.stream(stream):
            self.dist.gather(g["send"], g["recv"], dst=0)

    def flush_l2(self, nctx=None):
        """160 MiB device memset (> the 126 MB L2, which all streams share) on the stream the step's first frame goes to"""
        with self.torch.cuda.stream(self.streams[0]):
            self.flush_bufs[0].zero_()

    def device_frame(self, frame, flush=False, nctx=None, capture=None):
        """one frame, everything resident in HBM (async): [L2 flush], uniforms, raymarch, display[, gather][, copy of the
        presented RGBA8 and depth planes to the device addresses `capture`]"""
        k = frame % (nctx or self.nctx)
        ctx, prog, stream = self.ctxs[k], self.progs[k], self.streams[k]
        L, W, H, rm = self.L, self.W, self.H, self.rm
        if flush:
            with self.torch.cuda.stream(stream):
                self.flush_bufs[k].zero_()
        s = self.schema(frame)
        fb = ctx.fbo.create(W, H, s.render.frameid)
        for noise in self.sample_noise:
            rm.upload_sample_uniforms(prog, s, noise)
            st = L.rmb_render_sample(ctx.handle, prog.handle, fb.handle, 0, 0, W, H)
            assert st == 0, ctx.last_error()
        fused = self.fused
        if fused and fused.blur:
            # full mode: the display blur reads neighbour tiles, so the accumulator rows go to rank 0's
            # full-frame planes (peer stores) and rank 0 presents the assembled frame
            fused.scatter(ctx, fb, frame)
            fused.complete(ctx)
            if self.rank == 0:
                fused.display_assembled(ctx, frame, 1.0)
        else:
            if fused:
                fused.aim(ctx, frame)      # the display kernel also stores into rank 0's frame `frame % slots`
            st = L.rmb_present_device(ctx.handle, fb.handle, 1.0)
            assert st == 0, ctx.last_error()
            if fused:
                fused.complete(ctx)       # completion flag in stream order (or a one-element all-reduce): every rank has presented
            elif self.tiles and self.world > 1:
                self._gather_tiles(ctx, stream, fb)
        if capture:
            for which, dst in zip((4, 3), capture):
                st = L.rmb_fb_copy_to_device(ctx.handle, fb.handle, which, dst, fb.local_rows * W * 4)
                assert st == 0, ctx.last_error()
        ctx.fbo.delete(W, H, s.render.frameid)
        return k

    def barrier(self):
        if self.dist:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if not self.dist:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def measure_device(self, first_frame, n_frames, frames_per_step=1, dump=None):
        """n_frames enqueued back to back (the host runs ahead of the GPU); before every step (frames_per_step frames)
        an in-stream 160 MiB L2 flush, INSIDE the timed region; one start event (GPU idle,
        recorded on every stream) to the last end event.  `dump` (OutputDump) receives the frames of the last step.
        Returns (total ms max over ranks, launches, (evals, pixel-samples, far evals))."""
        torch = self.torch
        for c in self.ctxs:
            c.sync()
            c.counters(reset=True)
        self.barrier()
        launches0 = sum(c.launch_count() for c in self.ctxs)
        starts = [torch.cuda.Event(enable_timing=True) for _ in self.ctxs]
        ends = [torch.cuda.Event(enable_timing=True) for _ in self.ctxs]
        for e, st_ in zip(starts, self.streams):
            e.record(st_)
        last_step = n_frames - max(1, frames_per_step)
        for i in range(n_frames):
            if i % max(1, frames_per_step) == 0:
                self.flush_l2()
            self.device_frame(first_frame + i, capture=dump.slot(i - last_step) if dump and i >= last_step else None)
        for e, st_ in zip(ends, self.streams):
            e.record(st_)
        self.barrier()
        for c in self.ctxs:
            c.sync()
        launches = sum(c.launch_count() for c in self.ctxs) - launches0
        total_ms = self.max_over_ranks(max(starts[0].elapsed_time(e) for e in ends))
        cnt = [c.counters3(reset=True) for c in self.ctxs]
        return total_ms, launches, tuple(sum(x[j] for x in cnt) for j in range(3))

    def measure_e2e(self, first_frame, n_frames, want_depth, readback=True):
        """the same frames end to end through the public API, host wall clock (max over ranks).  Poses: rm.render_frames
        (do_render_job per frame with a pipelined presenter), uniforms from host memory every frame, every frame's
        RGBA8 (+ depth) read back to pinned host memory and touched by the host.  Tiles: every rank renders + presents
        its rows, the frame is assembled on rank 0 (fused peer stores, or NCCL gather) and rank 0 reads it back."""
        torch, rm = self.torch, self.rm
        checksum = 0
        if self.tiles and self.world > 1:
            slots = 2 * self.nctx
            H, W = self.H, self.W
            pinned = torch.empty((slots, H, W, 4), dtype=torch.uint8, pin_memory=True) if self.rank == 0 else None
            import raymarching_engine_b200.sharding as sh

            def run(first, count):
                nonlocal checksum
                pending = []
                for i in range(count):
                    k = self.device_frame(first + i)
                    if self.rank == 0:
                        with torch.cuda.stream(self.streams[k]):
                            if self.fused:
                                pinned[(first + i) % slots].copy_(self.fused.frame_tensor(first + i), non_blocking=True)
                            else:
                                flat = pinned[(first + i) % slots].view(-1)
                                off = 0
                                for r in range(self.world):
                                    n = len(sh.owned_rows(H, 16, self.world, r)) * W * 4
                                    flat[off:off + n].copy_(self.gather_state[id(self.ctxs[k])]["recv"][r][:n], non_blocking=True)
                                    off += n
                        ev = torch.cuda.Event()
                        ev.record(self.streams[k])
                        pending.append((ev, (first + i) % slots))
                        while len(pending) >= slots:
                            e, sl = pending.pop(0)
                            e.synchronize()
                            checksum += int(pinned[sl, 0, 0, 0]) + int(pinned[sl, -1, -1, 3])
                for e, sl in pending:
                    e.synchronize()
                    checksum += int(pinned[sl, 0, 0, 0]) + int(pinned[sl, -1, -1, 3])
            run(0, 2 * self.nctx + 1)
            self.barrier()
            t0 = time.perf_counter()
            run(first_frame, n_frames)
        elif not readback:
            for i in range(2 * self.nctx + 1):
                self.device_frame(i)
            self.barrier()
            t0 = time.perf_counter()
            for i in range(n_frames):
                self.device_frame(first_frame + i)
        else:
            for _i, res in rm.render_frames([self.schema(i) for i in range(2 * self.nctx + 1)], self.ctxs, want_depth=want_depth):
                assert res["success"], res["why"]
            jobs = [self.schema(first_frame + i) for i in range(n_frames)]      # the job descriptions are the host-side inputs
            self.barrier()
            t0 = time.perf_counter()
            for _i, res in rm.render_frames(jobs, self.ctxs, want_depth=want_depth):
                assert res["success"], res["why"]
                checksum += int(res["rgba8"][0, 0, 0]) + int(res["rgba8"][-1, -1, 3])   # the host reads the result
        torch.cuda.synchronize()
        secs = time.perf_counter() - t0
        self.barrier()
        return self.max_over_ranks(secs), checksum

    def close(self):
        if self.fused:
            self.fused.close()
        for c in self.ctxs:
            c.close()


def run_b200(args):
    import torch
    import raymarching_engine_b200 as rm

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)
    W, H = args.width, args.height
    tiles = world > 1 and args.shard == "tiles"
    F = max(1, args.frames_per_step)
    nctx = max(1, args.contexts)
    rig = Rig(rm, torch, args, W, H, tiles, dist, rank, world, local, nctx)
    wavefront = args.pipeline == "wavefront"
    regs = rig.progs[0].kernel_attr((2 if args.mode == "preview" else 3) if wavefront else (0 if args.mode == "preview" else 1))

    # ---- warm-up (also compiles the program variant): W >= 3 steps' worth of frames, capped so that a huge batch
    # size does not make the warm-up the longest part of the run
    warm_frames = min(max(args.warmup, 3) * F, 64 * nctx)
    for i in range(warm_frames):
        rig.device_frame(i, flush=True)

    if args.dump_outputs and tiles:
        raise SystemExit("bench.py: --dump-outputs needs whole frames on every rank (--shard poses)")
    dump = OutputDump(torch, F, W, H) if args.dump_outputs and rank == 0 else None

    sampler = ClockSampler(local)
    sampler.start()

    # ---- timed: device-resident, K steps of F frames
    n_frames = args.steps * F
    total_ms, gpu_launches, (evals, pxs, far_evals) = rig.measure_device(args.warmup * F, n_frames, F, dump)
    if dump:
        dump.write(args.dump_outputs)
    frames_all = n_frames * (1 if tiles else world)
    value = frames_all * W * H * args.spp / (total_ms * 1e-3) / 1e6     # pixel-samples per second, whole job

    # ---- timed: end to end through the public API
    e2e_s, _cs = rig.measure_e2e(args.warmup * F, n_frames, args.e2e_depth)
    e2e_value = frames_all * W * H * args.spp / e2e_s / 1e6
    d2h_bytes = W * H * (8 if (args.e2e_depth and not tiles) else 4)
    e2e = {"value": e2e_value, "unit": "Mpx/s", "h2d_bytes_per_step": 712 * F * args.spp, "d2h_bytes_per_step": d2h_bytes * F,
           "ms_per_step": 1e3 * e2e_s / max(args.steps, 1),
           "readback": "RGBA8 + fp32 depth" if (args.e2e_depth and not tiles) else "RGBA8 (the reference's canvas; --e2e-depth adds the fp32 depth plane)"}
    if not tiles and not args.quick:
        # where the end-to-end time goes: the same public-API loop without the device->host copies (host + launch
        # overhead only), and the D2H ceiling of this box for the same bytes from the same pinned buffers
        nr_s, _ = rig.measure_e2e(args.warmup * F, n_frames, False, readback=False)
        buf = torch.empty(d2h_bytes, dtype=torch.uint8, device="cuda")
        pin = torch.empty(d2h_bytes, dtype=torch.uint8, pin_memory=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(32):
            pin.copy_(buf, non_blocking=True)
        torch.cuda.synchronize()
        d2h_gbs = 32 * d2h_bytes / (time.perf_counter() - t0) / 1e9
        e2e["breakdown"] = {"no_readback_mpx_s": frames_all * W * H * args.spp / rig.max_over_ranks(nr_s) / 1e6,
                            "d2h_ceiling_gb_s_this_rank": d2h_gbs,
                            "d2h_ceiling_mpx_s_this_rank": d2h_gbs * 1e9 / (d2h_bytes / (W * H)) / 1e6,
                            "note": "no_readback = the same API loop with the display pass but no device->host copy; the ceiling = "
                                    "cudaMemcpyAsync of one frame's readback bytes into pinned memory, back to back"}
    clocks = sampler.stop()

    # ---- roofline of the hot kernel (the persistent march kernel), timed ALONE: with several contexts the march
    # kernels of different frames overlap each other's drain phase, which is good for the job but inflates each
    # kernel's own duration, so the kernel-level figure comes from a second pass on one context (CUDA events
    # around every march launch, L2 flushed before every frame).
    solo_frames = min(n_frames, 64)
    c0 = rig.ctxs[0]
    c0.sync()
    c0.timing(True)
    c0.counters(reset=True)
    for i in range(solo_frames):
        rig.device_frame(args.warmup * F + i, flush=True, nctx=1)
    for c in rig.ctxs:
        c.sync()
    hot_ms, hot_launches = c0.timing(False)
    evals_solo, _px_solo, far_solo = c0.counters3(reset=True)
    for c in rig.ctxs[1:]:
        c.counters(reset=True)
    fp32_measured = c0.measure_fp32_peak(0.5)
    fp32x2_measured = c0.measure_fp32_peak(0.3, packed=True)
    sm_count = torch.cuda.get_device_properties(local).multi_processor_count
    sm_max = clocks.get("sm_max_mhz") or 1965.0
    nominal_peak = sm_count * 128 * 2 * sm_max * 1e6 / 1e12
    flop_per_step = FLOP_PER_PREVIEW_STEP if args.mode == "preview" else FLOP_PER_CASTRAY_STEP
    de_trips, de_trips_source = None, None
    if args.scene == "mandelbulb":
        de_trips, de_trips_source = MANDELBULB_DE_TRIPS_PER_EVAL_PINNED, "pinned (bench.py header)"
        if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.quick:
            try:
                de_trips = mandelbulb_de_trips_per_eval(rig.counts)
                de_trips_source = "oracle, this run: 320x180 preview, poses 0 / 37 / 101 / 200 of the orbit"
            except Exception as e:   # noqa: BLE001 - keep the pinned figure
                de_trips_source += f" (oracle measurement failed: {str(e)[:80]})"
        flop_per_step = MANDELBULB_FLOP_PER_DE_TRIP * de_trips + MANDELBULB_FLOP_PER_EVAL_TAIL + (10.0 if args.mode == "preview" else 6.0)
    elif args.scene != "guide":
        flop_per_step = float("nan")    # the algorithmic flop count (SURVEY.md 8d) is defined for the default scene only
    flop_per_far_step = FLOP_PER_FAR_PREVIEW_STEP if args.mode == "preview" else FLOP_PER_FAR_CASTRAY_STEP
    kernel_s = hot_ms * 1e-3
    # the march kernel executes the full SDF evaluations only (the far-field steps of a carved scene run in the
    # setup kernel's approach and in the far pass, which the library's kernel timer leaves out)
    kernel_flop = (evals_solo - far_solo) * flop_per_step
    achieved = kernel_flop / kernel_s / 1e12 if kernel_s > 0 else 0.0
    if wavefront:
        hot_kernel = "rm_wf_march_preview_kernel" if args.mode == "preview" else "rm_wf_march_cast_kernel"
    else:
        hot_kernel = "rm_preview_kernel" if args.mode == "preview" else "rm_full_kernel"
    traffic = None
    try:
        tj = json.loads((ROOT / "profiles" / "traffic.json").read_text())
        traffic = tj.get(f"{hot_kernel}:{W}x{H}:{args.flavour}")
    except (OSError, ValueError):
        pass
    solo_on_ctx0 = solo_frames                 # the solo pass runs every frame on context 0
    roofline = {
        "bound": "fp32", "achieved": achieved, "peak": nominal_peak, "unit": "TFLOP/s", "frac": achieved / nominal_peak, "traffic": traffic,
        "peak_source": f"derived: {sm_count} SMs x 128 FP32 lanes x 2 x {sm_max:.0f} MHz (MEASURED_PEAKS.json has no FP32 figure; BASELINE.md section 2)",
        "peak_measured_ffma": fp32_measured, "peak_measured_ffma2_packed": fp32x2_measured, "frac_of_measured_ffma": achieved / fp32_measured if fp32_measured else None,
        "kernel": hot_kernel, "kernel_launches_per_frame": hot_launches / max(solo_on_ctx0, 1),
        "kernel_ms_per_frame": 1e3 * kernel_s / max(solo_on_ctx0, 1), "kernel_ms_avg": 1e3 * kernel_s / max(hot_launches, 1),
        "kernel_share_of_frame": min(1.0, (kernel_s / max(solo_on_ctx0, 1)) / (total_ms * 1e-3 / max(n_frames, 1))),
        "whole_step_frac": (((evals - far_evals) * flop_per_step + far_evals * flop_per_far_step) / (total_ms * 1e-3) / 1e12) / nominal_peak,
        "far_field_evals_share": far_solo / max(evals_solo, 1), "flop_per_far_field_step": flop_per_far_step,
        # the whole step priced as the reference prices it (every SDF value at the full evaluation's cost): what the
        # far-field pipeline saves, not a utilisation figure
        "reference_equivalent_whole_step_frac": (evals * flop_per_step / (total_ms * 1e-3) / 1e12) / nominal_peak,
        "executed_sdf_evals_per_frame": evals / max(n_frames, 1), "flop_per_step": flop_per_step,
        "executed_steps_per_px": evals / max(pxs, 1), "registers_per_thread": regs[0], "local_bytes": regs[1],
        "note": "timed alone: a separate pass of frames on ONE context, CUDA events around every march launch, L2 flushed before every frame",
    }
    if de_trips is not None:
        # config 4 is transcendental-bound, not FMA-bound: the FP32 figure above is reported for uniformity, the ceiling
        # that matters is the XU pipe (16 MUFU lanes per SM per clock) in the fast flavour and the fp64 pipe in the exact
        # one, whose transcendentals are evaluated in binary64 (profiles/r2_ncu_config4_*.txt)
        mufu_per_eval = MANDELBULB_MUFU_PER_DE_TRIP * de_trips + 2.0      # + log and the division of the tail
        xu_peak = sm_count * 16 * sm_max * 1e6 / 1e12
        xu_achieved = (evals_solo - far_solo) * mufu_per_eval / kernel_s / 1e12 if kernel_s > 0 else 0.0
        roofline["config4"] = {"de_trips_per_eval": de_trips, "de_trips_source": de_trips_source,
                               "flop_per_de_trip": MANDELBULB_FLOP_PER_DE_TRIP, "flop_per_eval_tail": MANDELBULB_FLOP_PER_EVAL_TAIL,
                               "mufu_per_de_trip_fast_flavour": MANDELBULB_MUFU_PER_DE_TRIP,
                               "xu_bound": {"achieved": xu_achieved, "peak": xu_peak, "unit": "T MUFU lane-ops/s", "frac": xu_achieved / xu_peak,
                                            "applies_to": "fast flavour (the exact flavour evaluates transcendentals in binary64 on the fp64 pipe)"}}

    line = {
        "metric": metric_name(args), "value": value, "unit": "Mpx/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / max(args.steps, 1), "higher_is_better": True, "scaling": "strong" if tiles else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args),
        "roofline": roofline, "e2e": e2e,
        "gpu_launches": gpu_launches,   # counted by the library: every kernel it launched in the device-resident timed loop
        "clocks": clocks,
        "extra": {"ms_per_frame": total_ms / max(n_frames, 1), "timed_region_ms": total_ms,
                  "msteps_per_s_ref_equiv": value * ref_steps_per_px(args), "e2e_msteps_per_s_ref_equiv": e2e_value * ref_steps_per_px(args),
                  "msteps_per_s_executed": evals / (total_ms * 1e-3) / 1e6 * (world if not tiles else 1)},
    }
    rig.close()

    # ---- BASELINE.json config 3 beside the headline: 3840x2160 row tiles across the ranks, fused gather (N = 1: the
    # single-GPU figure the N > 1 runs are compared with)
    if not args.quick and args.scene == "guide" and args.mode == "preview" and not tiles and (W, H) == (1920, 1080) and args.config3_steps > 0:
        try:
            a3 = argparse.Namespace(**vars(args))
            a3.width, a3.height, a3.shard, a3.gpus = 3840, 2160, "tiles", world
            r3 = Rig(rm, torch, a3, 3840, 2160, world > 1, dist, rank, world, local, nctx)
            f3 = max(4, F // 4)
            for i in range(3 * nctx + 2):
                r3.device_frame(i, flush=True)
            n3 = args.config3_steps * f3
            ms3, launches3, _c3 = r3.measure_device(16, n3, f3)
            e3_s, _ = r3.measure_e2e(16, n3, False)
            line["config3_tiles"] = {
                "workload": f"guide.glsl 3840x2160 preview, interleaved 16-row tiles over {world} GPU(s), gather fused into the display kernel's stores "
                            f"(peer memory over NVLink; completion ordered by "
                            f"{'stream-ordered flags in shared pinned memory, no collective' if (r3.fused and r3.fused.sync == 'flags') else 'a one-element all-reduce per frame'}); strong scaling",
                "value": n3 * 3840 * 2160 / (ms3 * 1e-3) / 1e6, "unit": "Mpx/s", "ms_per_frame": ms3 / n3, "frames": n3, "gather": args.gather if world > 1 else "none",
                "e2e": {"value": n3 * 3840 * 2160 / e3_s / 1e6, "unit": "Mpx/s", "d2h_bytes_per_frame": 3840 * 2160 * 4, "readback": "RGBA8 on rank 0"},
                "gpu_launches": launches3, "n_gpus": world, "scaling": "strong",
                "completion": (r3.fused.sync if r3.fused else "none")}
            r3.close()
        except Exception as e:   # noqa: BLE001 - the headline must not depend on the extra configuration
            line["config3_tiles"] = {"error": str(e)[:300]}

    if rank == 0 and world == 1 and args.flavour == "exact" and not args.no_second_flavour and not args.quick:
        # the tolerance-checked fast flavour of the same workload, measured the same way in a child
        # process and reported beside the headline (DESIGN.md section 2: it is not the parity path)
        cmd = [sys.executable, os.fspath(ROOT / "bench.py"), "--flavour", "fast", "--quick",
               "--steps", str(args.steps), "--warmup", str(args.warmup), "--width", str(W), "--height", str(H), "--mode", args.mode,
               "--scene", args.scene, "--spp", str(args.spp), "--contexts", str(args.contexts), "--pipeline", args.pipeline,
               "--frames-per-step", str(F)]
        if args.step_counts:
            cmd += ["--step-counts", args.step_counts]
        try:
            out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
            f = json.loads(out.stdout.strip().splitlines()[-1])
            tol = None
            try:
                tol = json.loads((ROOT / "profiles" / "flavour_tolerance.json").read_text())
            except (OSError, ValueError):
                pass
            line["extra"]["fast_flavour"] = {
                "value": f["value"], "unit": f["unit"], "ms_per_step": f["ms_per_step"], "e2e": f["e2e"]["value"],
                "roofline_frac": f["roofline"]["frac"], "roofline_achieved": f["roofline"]["achieved"], "kernel": f["roofline"]["kernel"],
                "parity": "tolerance-checked, not bit-exact; see profiles/flavour_tolerance.json", "measured_tolerance": tol}
        except Exception as e:   # noqa: BLE001 - the headline must not depend on the optional second arm
            line["extra"]["fast_flavour"] = {"error": str(e)[:200]}
        if roofline.get("far_field_evals_share", 0) > 0:
            # context for the roofline figure: the same workload with the far-field pipeline off (every ray marched by the
            # one kernel, RMB_CARVE=0), measured the same way in a child process
            cmd[3] = "exact"
            try:
                out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=dict(os.environ, RMB_CARVE="0"))
                f = json.loads(out.stdout.strip().splitlines()[-1])
                line["extra"]["far_field_pipeline_off"] = {
                    "value": f["value"], "unit": f["unit"], "ms_per_step": f["ms_per_step"], "e2e": f["e2e"]["value"],
                    "roofline_frac": f["roofline"]["frac"], "roofline_achieved": f["roofline"]["achieved"],
                    "kernel_ms_per_frame": f["roofline"]["kernel_ms_per_frame"],
                    "note": "RMB_CARVE=0: bit-identical frames; the march kernel then also executes the 87 % of SDF evaluations whose value is the outer shape alone"}
            except Exception as e:   # noqa: BLE001 - context only
                line["extra"]["far_field_pipeline_off"] = {"error": str(e)[:200]}
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not args.quick:
        mpx, secs, cores, desc = cpu_reference_sample(W, H, args.mode, args.cpu_band_rows, None, args.scene, rig.counts)
        line["cpu_baseline"] = {"value": mpx, "unit": "Mpx/s", "cores": cores, "kind": "port", "sample": desc, "seconds": secs}
    if rank == 0:
        print(json.dumps(_json_safe(line)), flush=True)
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames-per-step", type=int, default=32, help="frames of the camera path per step (the timed region is steps x this many frames)")
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--mode", default="preview", choices=["preview", "full"])
    ap.add_argument("--scene", default="guide", help="scenes/<name>.glsl (BASELINE.json config 4: mandelbulb)")
    ap.add_argument("--step-counts", default="", help="comma-separated reflectionIterationCounts (config 4: 512)")
    ap.add_argument("--spp", type=int, default=1, help="samples per pixel per frame (config 5: 16)")
    ap.add_argument("--flavour", default="exact", choices=["exact", "fast"])
    ap.add_argument("--shard", default="poses", choices=["poses", "tiles"])
    ap.add_argument("--gather", default="fused", choices=["fused", "fused-nccl", "nccl"],
                    help="--shard tiles: fused = display kernel stores into rank 0's frame over NVLink (CUDA IPC), completion by stream-ordered "
                         "flags; fused-nccl = the same stores, completion by a one-element all-reduce; nccl = torch.distributed.gather of the rows")
    ap.add_argument("--pipeline", default="wavefront", choices=["wavefront", "megakernel"])
    ap.add_argument("--contexts", type=int, default=4, help="contexts (streams) per GPU the independent frames are dealt to")
    ap.add_argument("--e2e-depth", action="store_true", help="the end-to-end arm also reads the fp32 depth plane back (8 B/px instead of 4)")
    ap.add_argument("--config3-steps", type=int, default=4, help="steps of the 4K row-tile configuration measured beside the headline (0 = skip)")
    ap.add_argument("--cpu-band-rows", type=int, default=360)
    ap.add_argument("--ref-band-rows", type=int, default=120)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-second-flavour", action="store_true", help="do not also measure --flavour fast / far-field off beside an exact-flavour headline")
    ap.add_argument("--quick", action="store_true", help="headline + roofline only: no cpu baseline, second flavour, e2e breakdown or config 3")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the RGBA8 and depth of the last timed step's frames to DIR/*.npy (see the header)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.steps < 1):
        ap.error("--dump-outputs needs --impl b200 and --steps >= 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
