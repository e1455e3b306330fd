"""Render-job host layer: the Python mirror of the reference's TypeScript renderer, with the
WebGL2 calls replaced by the C ABI of libraymarch_b200.so.

Mirrors (paths under /root/reference/client/src):
  renderer/LoadRenderJobContext.tsx:268-287   loadRenderJobContext      -> load_render_job_context
  renderer/LoadRenderJobContext.tsx:162-250   fbo.create / fbo.delete   -> RenderJobContext.fbo
  renderer/ShaderCache.tsx:91-119             programCache.getProgram   -> RenderJobContext.program_cache
  renderer/RenderJobExecutor.tsx:77-341       doRenderJob               -> do_render_job
  index.tsx:25-59                             makePresenter             -> make_presenter
Names, argument meaning, loop order and error behaviour follow the reference; errors are values
(`{"success": False, "why": {"type": ..., "infoLog": ...}}`), never exceptions.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass
from typing import Callable, Dict, Generator, Optional

import numpy as np

from . import _lib
from .halton import halton
from .schema import RenderJobSchema
from .uniforms import UniformData, set_uniform_array, set_uniform_matrix4, set_uniforms, u

L = _lib.lib


@dataclass
class ShaderError:                       # ShaderCache.tsx:8-11 (+ "general", RenderJobExecutor.tsx:73-75)
    type: str                            # "vertex" | "fragment" | "program" | "general"
    infoLog: str


class Program:
    def __init__(self, context: "RenderJobContext", handle: int):
        self.context, self.handle = context, handle

    def source(self) -> str:
        return L.rmb_program_source(self.handle).decode()

    def has_carve(self) -> bool:
        """True when the march kernels take the far-field shortcut of a carved scene (include/rmb.h)"""
        return bool(L.rmb_program_has_carve(self.handle))

    def kernel_attr(self, kernel: int):
        r, l = C.c_int(-1), C.c_int(-1)
        L.rmb_program_kernel_attr(self.handle, kernel, C.byref(r), C.byref(l))
        return r.value, l.value


class FramebufferInfo:                   # RenderJobFramebufferInfo, RenderJobExecutor.tsx:14-30
    def __init__(self, context: "RenderJobContext", handle: int, width: int, height: int, frameid: int):
        self.context, self.handle = context, handle
        self.width, self.height, self.frameid = width, height, frameid
        self.local_rows = L.rmb_fb_local_rows(handle)

    def global_rows(self) -> np.ndarray:
        return np.array([L.rmb_fb_global_row(self.handle, r) for r in range(self.local_rows)], dtype=np.int64)

    _PLANES = {"color": (0, np.float32, 4), "normalAndDofRadius": (1, np.uint16, 4), "albedoAndDepth": (2, np.uint16, 4),
               "depth": (3, np.float32, 1), "rgba8": (4, np.uint8, 4)}

    def read(self, plane: str) -> np.ndarray:
        which, dt, ch = self._PLANES[plane]
        shape = (self.local_rows, self.width, ch) if ch > 1 else (self.local_rows, self.width)
        out = np.empty(shape, dtype=dt)
        st = L.rmb_fb_read(self.context.handle, self.handle, which, out.ctypes.data_as(C.c_void_p), out.nbytes)
        if st != _lib.RMB_OK:
            raise RuntimeError(self.context.last_error())
        return out

    def write(self, plane: str, arr: np.ndarray) -> None:
        which, dt, ch = self._PLANES[plane]
        a = np.ascontiguousarray(arr, dtype=dt)
        st = L.rmb_fb_write(self.context.handle, self.handle, which, a.ctypes.data_as(C.c_void_p), a.nbytes)
        if st != _lib.RMB_OK:
            raise RuntimeError(self.context.last_error())

    def device_ptr(self, plane: str) -> int:
        return L.rmb_fb_device_ptr(self.handle, self._PLANES[plane][0])


class _Fbo:
    """context.fbo of the reference (LoadRenderJobContext.tsx:184-249); pool semantics live in C."""

    def __init__(self, context: "RenderJobContext"):
        self._c = context

    def create(self, width: int, height: int, frameid: int) -> Optional[FramebufferInfo]:
        h = L.rmb_fb_acquire(self._c.handle, int(width), int(height), int(frameid))
        if not h:
            return None
        return FramebufferInfo(self._c, h, int(width), int(height), int(frameid))

    def delete(self, width: int, height: int, frameid: int) -> None:
        L.rmb_fb_release(self._c.handle, int(width), int(height), int(frameid))


class _ProgramCache:
    """context.programCache (ShaderCache.tsx:91-119).  `getProgram` returns a Program or a ShaderError."""

    def __init__(self, context: "RenderJobContext"):
        self._c = context
        self._hits: dict = {}          # (source, flavour, baked values) -> Program: the per-job lookup without an FFI crossing

    def get_program(self, scene_source: str, flavour: Optional[int] = None, spec: Optional[Dict[str, UniformData]] = None):
        flavour = self._c.flavour if flavour is None else flavour
        key = (scene_source, flavour, tuple(sorted((k, v.type, tuple(v.data)) for k, v in spec.items())) if spec else None)
        hit = self._hits.get(key)
        if hit is not None and L.rmb_program_is_live(hit.handle):
            return hit
        prog = self._get_program(scene_source, flavour, spec)
        if isinstance(prog, Program):
            if len(self._hits) >= 64:
                self._hits.pop(next(iter(self._hits)))
            self._hits[key] = prog
        return prog

    def _get_program(self, scene_source: str, flavour: int, spec: Optional[Dict[str, UniformData]]):
        arr, n = _lib.make_spec_array(spec)
        out = C.c_void_p()
        etype = C.create_string_buffer(16)
        log = C.create_string_buffer(1 << 16)
        src = scene_source.encode()
        st = L.rmb_program_get(self._c.handle, src, len(src), flavour, arr, n, C.byref(out), etype, log, len(log))
        if st != _lib.RMB_OK:
            return ShaderError(etype.value.decode() or "general", log.value.decode())
        return Program(self._c, out.value)


class RenderJobContext:                  # RenderJobExecutor.tsx:32-54
    def __init__(self, handle: int, device: int, rank: int, n_ranks: int, tile_rows: int, flavour: int, specialize):
        self.handle = handle
        self.device, self.rank, self.n_ranks, self.tile_rows = device, rank, n_ranks, tile_rows
        self.flavour, self.specialize = flavour, specialize
        self.fbo = _Fbo(self)
        self.program_cache = _ProgramCache(self)
        self._pinned_cache: dict = {}

    def last_error(self) -> str:
        return (L.rmb_last_error(self.handle) or b"").decode()

    def stream(self) -> int:
        return L.rmb_ctx_stream(self.handle)

    def sync(self) -> None:
        L.rmb_sync(self.handle)

    def timing(self, enable: bool):
        """(hot-kernel milliseconds, launches) accumulated since the last call; then turns collection on/off"""
        ms, n = C.c_double(0.0), C.c_uint64(0)
        if L.rmb_ctx_timing(self.handle, 1 if enable else 0, C.byref(ms), C.byref(n)) != _lib.RMB_OK:
            raise RuntimeError(self.last_error())
        return ms.value, int(n.value)

    def launch_count(self) -> int:
        return int(L.rmb_ctx_launch_count(self.handle))

    def counters(self, reset: bool = False):
        """(SDF evaluations, pixel-samples)"""
        return tuple(self.counters_all(reset)[:2])

    def counters3(self, reset: bool = False):
        """(SDF evaluations, pixel-samples, evaluations that took the far-field shortcut)"""
        return tuple(self.counters_all(reset)[:3])

    def counters_all(self, reset: bool = False):
        """all 16 counter slots (rmb_counters_read_all; slots 3.. are filled by RMB_PROFILE=1 programs only)"""
        out = (C.c_uint64 * 16)()
        L.rmb_counters_read_all(self.handle, out, 1 if reset else 0)
        return [int(v) for v in out]

    def probe_carve(self, program, points) -> np.ndarray:
        """n x 4: sdf as the march kernels evaluate it, outer shape A, bound U, guarded sdf (rmb_probe_carve)"""
        pts = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
        out = np.zeros((len(pts), 4), np.float32)
        if L.rmb_probe_carve(self.handle, program.handle, pts.ctypes.data_as(C.c_void_p), len(pts), out.ctypes.data_as(C.c_void_p)) != 0:
            raise RuntimeError(self.last_error())
        return out

    def _pinned(self, key, shape, dtype) -> np.ndarray:
        """numpy view of a cached pinned host buffer (rmb_host_alloc) for readbacks"""
        k = (key, tuple(shape), np.dtype(dtype).str)
        buf = self._pinned_cache.get(k)
        if buf is None:
            nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
            ptr = L.rmb_host_alloc(max(nbytes, 1))
            if not ptr:
                raise MemoryError("rmb_host_alloc failed")
            arr = np.ctypeslib.as_array((C.c_uint8 * max(nbytes, 1)).from_address(ptr))[:nbytes].view(dtype).reshape(shape)
            buf = (ptr, arr)
            self._pinned_cache[k] = buf
        return buf[1]

    def render_sample(self, program: Program, fb: FramebufferInfo, x: int, y: int, w: int, h: int) -> int:
        """gl.scissor(x, y, w, h) + the raymarcher draw + blit of one sample (RenderJobExecutor.tsx:181-326); status"""
        return L.rmb_render_sample(self.handle, program.handle, fb.handle, x, y, w, h)

    def present(self, fb: FramebufferInfo, brightness: float, want_depth: bool = True, readback: bool = True):
        """display pass (+ readback into pinned host memory): (rgba8[local_rows, W, 4] uint8,
        depth[local_rows, W] float32 | None).  The arrays are views of buffers reused by the next
        present of the same size - copy them to keep them.  readback=False runs the display pass
        only (the canvas of the reference is never read back either) and returns (None, None)."""
        if not readback:
            st = L.rmb_present_device(self.handle, fb.handle, float(np.float32(brightness)))
            if st != _lib.RMB_OK:
                raise RuntimeError(self.last_error())
            return None, None
        rgba = self._pinned("rgba", (fb.local_rows, fb.width, 4), np.uint8)
        depth = self._pinned("depth", (fb.local_rows, fb.width), np.float32) if want_depth else None
        st = L.rmb_present(self.handle, fb.handle, float(np.float32(brightness)), rgba.ctypes.data_as(C.c_void_p),
                           depth.ctypes.data_as(C.c_void_p) if want_depth else None)
        if st != _lib.RMB_OK:
            raise RuntimeError(self.last_error())
        return rgba, depth

    def present_async(self, fb: FramebufferInfo, brightness: float, want_depth: bool = True, slot: int = 0):
        """Non-blocking present (rmb_present_async): display pass on the context's stream, readback on
        the copy stream into the pinned buffers of ring slot `slot`.  Returns the (rgba8, depth) views,
        valid after present_wait(fb)."""
        rgba = self._pinned(("rgba", slot), (fb.local_rows, fb.width, 4), np.uint8)
        depth = self._pinned(("depth", slot), (fb.local_rows, fb.width), np.float32) if want_depth else None
        st = L.rmb_present_async(self.handle, fb.handle, float(np.float32(brightness)), rgba.ctypes.data_as(C.c_void_p),
                                 depth.ctypes.data_as(C.c_void_p) if want_depth else None)
        if st != _lib.RMB_OK:
            raise RuntimeError(self.last_error())
        return rgba, depth

    def present_wait(self, fb: FramebufferInfo) -> None:
        if L.rmb_present_wait(self.handle, fb.handle) != _lib.RMB_OK:
            raise RuntimeError(self.last_error())

    def measure_fp32_peak(self, seconds: float = 0.5, packed: bool = False) -> float:
        out = C.c_double(0.0)
        fn = L.rmb_measure_fp32x2_peak if packed else L.rmb_measure_fp32_peak
        if fn(self.handle, seconds, C.byref(out)) != _lib.RMB_OK:
            raise RuntimeError(self.last_error())
        return out.value

    def close(self) -> None:
        if self.handle:
            L.rmb_ctx_destroy(self.handle)
            self.handle = None
            for ptr, _arr in self._pinned_cache.values():
                L.rmb_host_free(ptr)
            self._pinned_cache.clear()


def load_render_job_context(device: int = 0, rank: int = 0, n_ranks: int = 1, tile_rows: int = 16,
                            flavour: int = _lib.FLAVOUR_EXACT, specialize=None,
                            pipeline: str = "wavefront") -> Optional[RenderJobContext]:
    """loadRenderJobContext(gl) (LoadRenderJobContext.tsx:268-287): returns None when any piece
    of the context cannot be created (the reference returns undefined).

    specialize: how do_render_job treats schema.customShaderParameters (in the reference a free gl.uniform call,
    RenderJobExecutor.tsx:266).  "auto" (default): plain dynamic uniforms until the same values have been submitted
    for SPECIALIZE_AFTER consecutive jobs of that scene, then a program variant with the values baked in (loops
    unroll, pow(uniform, i) folds); a value that changes - a slider being dragged, an animated parameter - falls
    back to the dynamic variant at once and never costs a compile.  True / "always": bake from the first job on.
    False / "never": always dynamic.  None: the RMB_SPECIALIZE environment variable (auto | always | never), default
    "auto".  The library keeps at most RMB_VARIANT_CAP variants per scene (LRU)."""
    if specialize is None:
        specialize = os.environ.get("RMB_SPECIALIZE", "auto")
    if specialize not in (True, False, "auto", "always", "never"):
        raise ValueError(f"specialize={specialize!r}: expected auto | always | never")
    h = L.rmb_ctx_create(device, rank, n_ranks, tile_rows)
    if not h:
        return None
    # "wavefront": setup -> persistent march -> shade kernels when the scene allows it (default);
    # "megakernel": one thread per pixel always
    L.rmb_ctx_set_pipeline(h, {"wavefront": 0, "megakernel": 1}[pipeline])
    return RenderJobContext(h, device, rank, n_ranks, tile_rows, flavour, specialize)


def context_error() -> str:
    return (L.rmb_last_error(None) or b"").decode()


# RenderJobExecutor.tsx:70-71: module-level generators that are never reset
_render_job_halton2 = halton(2)
_render_job_halton3 = halton(3)


def reset_halton() -> None:
    """Test hook: restart the two module-level Halton generators (a page reload in the reference)."""
    global _render_job_halton2, _render_job_halton3
    _render_job_halton2, _render_job_halton3 = halton(2), halton(3)


def _gen_err(info_log: str) -> ShaderError:      # RenderJobExecutor.tsx:73-75
    return ShaderError("general", info_log)


def builtin_uniforms(schema: RenderJobSchema, rand_noise) -> Dict[str, UniformData]:
    """The uniform record of RenderJobExecutor.tsx:212-264."""
    mode = schema.camera.mode
    mode_index = ["perspective", "orthographic", "panoramic"].index(mode.type) if mode.type in ("perspective", "orthographic", "panoramic") else -1
    counts = schema.reflectionIterationCounts
    return {
        "blendWithPreviousFactor": u.float(schema.render.blendWithPreviousFrameFactor),
        "previousColor": u.int(0),
        "previousNormalAndDofRadius": u.int(1),
        "previousAlbedoAndDepth": u.int(2),
        "randNoise": u.vec2(rand_noise[0], rand_noise[1]),
        "position": u.vec3(*schema.camera.position),
        "dofAmount": u.float(schema.dof.amount),
        "dofFocalPlaneDistance": u.float(schema.dof.distance),
        "cameraMode": u.int(mode_index),
        "fov": u.float(mode.fov if mode.type == "perspective" else mode.size if mode.type == "orthographic" else 1),
        "reflections": u.float(len(counts)),
        "raymarchingSteps": u.float(counts[0] if counts else math.nan),
        "indirectLightingRaymarchingSteps": u.float(counts[1] if len(counts) > 1 else (counts[0] if counts else math.nan)),
        "aspect": u.float(schema.render.width / schema.render.height),
        "fogDensity": u.float(schema.fogDensity),
        "exposure": u.float(schema.render.exposure / schema.render.samplesPerPixel),
        "blendMode": u.int(1 if schema.render.blendMode == "additive" else 0),
        "renderMode": u.int(1 if schema.render.renderMode == "preview" else 0),
        "lightCount": u.int(len(schema.lights)),
        "showDofFocalPlane": u.int(1 if schema.dof.showFocusedArea else 0),
    }


def frame_uniforms(schema: RenderJobSchema, rand_noise) -> "_lib.FrameUniforms":
    """The same record as builtin_uniforms + the array / matrix uploads of RenderJobExecutor.tsx:268-297, as the POD block
    of rmb_uniforms_set_frame (include/rmb.h): one FFI crossing per sample instead of ~25."""
    r, cam, mode = schema.render, schema.camera, schema.camera.mode
    counts = schema.reflectionIterationCounts
    b = _lib.FrameUniforms()
    b.blendWithPreviousFactor = r.blendWithPreviousFrameFactor
    b.randNoise[0], b.randNoise[1] = rand_noise[0], rand_noise[1]
    b.position[0], b.position[1], b.position[2] = cam.position
    b.rotation[:] = list(cam.rotation)
    b.dofAmount, b.dofFocalPlaneDistance = schema.dof.amount, schema.dof.distance
    b.cameraMode = ["perspective", "orthographic", "panoramic"].index(mode.type) if mode.type in ("perspective", "orthographic", "panoramic") else -1
    b.fov = mode.fov if mode.type == "perspective" else mode.size if mode.type == "orthographic" else 1
    b.reflections = len(counts)
    b.raymarchingSteps = counts[0] if counts else math.nan
    b.indirectLightingRaymarchingSteps = counts[1] if len(counts) > 1 else (counts[0] if counts else math.nan)
    b.aspect = r.width / r.height
    b.fogDensity = schema.fogDensity
    b.exposure = r.exposure / r.samplesPerPixel
    b.blendMode = 1 if r.blendMode == "additive" else 0
    b.renderMode = 1 if r.renderMode == "preview" else 0
    n = min(len(counts), 10)
    b.stepCountsLength = n
    b.raymarchingStepCountsArray[:n] = list(counts[:n])
    lights = schema.lights
    b.lightCount = len(lights)
    for k, l in enumerate(lights[:10]):
        b.lightPositions[3 * k:3 * k + 3] = list(l.position if l.type == "point" else l.direction)
        b.lightColors[3 * k:3 * k + 3] = list(l.color)
        b.lightSizes[k] = l.size if l.type == "point" else 0
    b.showDofFocalPlane = 1 if schema.dof.showFocusedArea else 0
    return b


def upload_sample_uniforms(program: Program, schema: RenderJobSchema, rand_noise) -> None:
    """Everything RenderJobExecutor.tsx:212-297 uploads before the draw call: the built-in record, arrays and matrix as
    one block (rmb_uniforms_set_frame applies them in the reference's order), then the scene's custom uniforms (:266)."""
    fn = L.rmb_group_uniforms_set_frame if getattr(program, "is_group", False) else L.rmb_uniforms_set_frame
    if fn(program.handle, C.byref(frame_uniforms(schema, rand_noise))) != _lib.RMB_OK:
        raise RuntimeError(f"uniform upload: {program.context.last_error()}")
    set_uniforms(program, schema.customShaderParameters)                                   # :266


PresentFn = Callable[[RenderJobContext, RenderJobSchema, FramebufferInfo, int], None]

# "auto" specialisation: jobs of a scene whose custom parameters have not changed for this many consecutive jobs
# (counted over all contexts of the process: stability is a property of the job stream) get the baked variant
SPECIALIZE_AFTER = 3
_spec_streak: Dict[int, list] = {}       # hash(scene source) -> [signature of the custom values, consecutive jobs]


def reset_specialization_history() -> None:
    """Test hook: forget which custom-parameter values have been seen."""
    _spec_streak.clear()


def _specialize_now(context: RenderJobContext, schema: RenderJobSchema) -> bool:
    mode = context.specialize
    if mode is True or mode == "always":
        return True
    if mode is False or mode == "never" or mode is None:
        return False
    sig = tuple(sorted((name, d.type, tuple(float(v) for v in d.data)) for name, d in schema.customShaderParameters.items()))
    key = hash(schema.sdfShaderSource)
    st = _spec_streak.get(key)
    if st is None or st[0] != sig:
        st = _spec_streak[key] = [sig, 0]
        if len(_spec_streak) > 64:
            _spec_streak.pop(next(iter(_spec_streak)))
    st[1] += 1
    return st[1] >= SPECIALIZE_AFTER


def do_render_job(schema: RenderJobSchema, context: RenderJobContext):
    """doRenderJob (RenderJobExecutor.tsx:77-341).  Returns a function that takes the `present`
    callback and returns a generator; the generator yields None every `sampleYieldInterval`
    samples and returns {"success": bool, "why": ShaderError | None}."""
    framebuffers = context.fbo.create(schema.render.width, schema.render.height, schema.render.frameid)   # :106-110
    if framebuffers is None:
        def failed(_present):
            return {"success": False, "why": _gen_err("Failed to load framebuffers.")}       # :112-119
            yield  # pragma: no cover
        return failed

    spec = dict(schema.customShaderParameters) if _specialize_now(context, schema) else None
    program = context.program_cache.get_program(schema.sdfShaderSource, None, spec)          # :121-127
    if isinstance(program, ShaderError):
        def failed(_present):
            return {"success": False, "why": program}                                        # :129-136
            yield  # pragma: no cover
        return failed

    def run(present: PresentFn) -> Generator[None, None, dict]:
        samples_rendered_so_far = 0
        r = schema.render
        for y_partitions in range(r.subdivisions):                                           # :148-162
            for x_partitions in range(r.subdivisions):
                for _sample_index in range(r.samplesPerPixel):
                    if samples_rendered_so_far % r.sampleYieldInterval == 0:                 # :163-166
                        present(context, schema, framebuffers, samples_rendered_so_far)
                        yield
                    x1 = math.floor((r.width / r.subdivisions) * x_partitions)               # :167-180
                    y1 = math.floor((r.height / r.subdivisions) * y_partitions)
                    x2 = math.ceil((r.width / r.subdivisions) * (x_partitions + 1))
                    y2 = math.ceil((r.height / r.subdivisions) * (y_partitions + 1))
                    rand_noise = (next(_render_job_halton2), next(_render_job_halton3))      # :219-222
                    upload_sample_uniforms(program, schema, rand_noise)
                    # gl.scissor(x1, y1, x2, y2): the reference passes the far corner where GL expects
                    # width/height (RenderJobExecutor.tsx:182); reproduced as is.
                    st = context.render_sample(program, framebuffers, x1, y1, x2, y2)                         # :299 + blit :301-326
                    if st != _lib.RMB_OK:
                        return {"success": False, "why": _gen_err(context.last_error())}
                    samples_rendered_so_far += 1
        context.fbo.delete(r.width, r.height, r.frameid)                                     # :333-337
        present(context, schema, framebuffers, samples_rendered_so_far)                      # :338
        return {"success": True, "why": None}

    return run


def make_presenter(samples_up_to_this_point: int, sink: Optional[dict] = None, want_depth: bool = True,
                   readback: str = "always", slot: int = 0) -> PresentFn:
    """makePresenter (index.tsx:25-59): display pass with brightness = 1 / samplesUpToThisPoint (the
    host's own counter; the generator's samplesSoFar argument is ignored for the brightness, as in
    the reference).  The canvas is replaced by `sink`: the latest frame lands in sink["rgba8"],
    sink["depth"] (views of pinned buffers).  readback="final" copies to the host only on the last
    present of a job (the intermediate presents still run the display pass, like canvas redraws).
    readback="async" does the same without blocking (present_async into pinned ring slot `slot`); the
    caller waits with context.present_wait(sink["framebuffers"])."""
    def present(context: RenderJobContext, schema: RenderJobSchema, framebuffers: FramebufferInfo, samples_so_far: int) -> None:
        brightness = 1 / samples_up_to_this_point if samples_up_to_this_point else math.inf
        total = schema.render.samplesPerPixel * schema.render.subdivisions ** 2
        rb = readback == "always" or samples_so_far >= total
        if readback == "async" and rb:
            rgba, depth = context.present_async(framebuffers, brightness, want_depth, slot)
            if sink is not None:
                sink["framebuffers"] = framebuffers
        else:
            rgba, depth = context.present(framebuffers, brightness, want_depth, readback=rb)
        if sink is not None:
            if rb:
                sink["rgba8"], sink["depth"] = rgba, depth
            sink["presents"] = sink.get("presents", 0) + 1
    return present


def run_job(schema: RenderJobSchema, context: RenderJobContext, samples_up_to_this_point: Optional[int] = None) -> dict:
    """Convenience: pump a job to completion like the rAF loop of index.tsx:236-263 and return
    {"success", "why", "rgba8", "depth"}."""
    sink: dict = {}
    n = samples_up_to_this_point if samples_up_to_this_point is not None else schema.render.samplesPerPixel * schema.render.subdivisions ** 2
    gen = do_render_job(schema, context)(make_presenter(n, sink, readback="final"))
    result = None
    try:
        while True:
            next(gen)
    except StopIteration as stop:
        result = stop.value
    out = dict(result or {"success": False, "why": _gen_err("generator ended without a result")})
    out.update(sink)
    return out


def render_frames(schemas, context, depth: int = 2, want_depth: bool = True):
    """Pipelined pump for a sequence of jobs (a camera path, BASELINE.json config 5): every job runs
    through do_render_job exactly like run_job, but its final present is non-blocking and the result
    is handed out later, so the device->host readback of frame k overlaps the kernels of frame k+1.
    `context` may be a list of contexts on the same device (each has its own stream, program modules
    and scratch): frames are dealt round-robin, so that the drain phase of one frame's persistent
    march kernel overlaps the next frame's kernels.  Yields (index, result dict) in order;
    result["rgba8"] / ["depth"] are views of a pinned ring buffer that stay valid until
    `depth * len(contexts)` more frames have been rendered."""
    schemas = list(schemas)
    contexts = list(context) if isinstance(context, (list, tuple)) else [context]
    nctx = len(contexts)
    window = depth * nctx
    pending = []      # (index, result, context, fb)
    for k, schema in enumerate(schemas):
        ctx = contexts[k % nctx]
        if k + nctx < len(schemas):
            nxt = schemas[k + nctx].render
            # acquire this context's next framebuffer set before this job releases its own, so that two
            # sets alternate and a set is never redrawn while it is being read back
            ctx.fbo.create(nxt.width, nxt.height, nxt.frameid)
        sink: dict = {}
        n = schema.render.samplesPerPixel * schema.render.subdivisions ** 2
        gen = do_render_job(schema, ctx)(make_presenter(n, sink, want_depth, readback="async", slot=(k // nctx) % depth))
        result = None
        try:
            while True:
                next(gen)
        except StopIteration as stop:
            result = dict(stop.value or {"success": False, "why": _gen_err("generator ended without a result")})
        fb = sink.pop("framebuffers", None)
        result.update(sink)
        pending.append((k, result, ctx, fb))
        while len(pending) >= window:
            i, res, c, f = pending.pop(0)
            if f is not None:
                c.present_wait(f)
            yield i, res
    for i, res, c, f in pending:
        if f is not None:
            c.present_wait(f)
        yield i, res
