"""ctypes wrapper of oracle/liboracle.so -- TEST INFRASTRUCTURE ONLY (see oracle/oracle.cpp header).

Importable only from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs.  The product package never imports this module.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "liboracle.so"


def build(force: bool = False) -> Path:
    if force or not LIB_PATH.exists() or LIB_PATH.stat().st_mtime < max(
            (_HERE / "oracle.cpp").stat().st_mtime,
            (_HERE.parent / "raymarching_engine_b200/csrc/device_src/glsl_rt.h").stat().st_mtime,
            (_HERE.parent / "raymarching_engine_b200/csrc/device_src/rm_math.h").stat().st_mtime):
        subprocess.run(["make", "-C", os.fspath(_HERE), "-B", "liboracle.so"], check=True, capture_output=True)
    return LIB_PATH


class Uniforms(C.Structure):   # OrcUniforms of oracle.cpp
    _fields_ = [("blendWithPreviousFactor", C.c_float), ("randNoise", C.c_float * 2), ("position", C.c_float * 3),
                ("rotation", C.c_float * 16), ("dofAmount", C.c_float), ("dofFocalPlaneDistance", C.c_float),
                ("cameraMode", C.c_int), ("fov", C.c_float), ("reflections", C.c_float), ("aspect", C.c_float),
                ("fogDensity", C.c_float), ("exposure", C.c_float), ("raymarchingStepCountsArray", C.c_float * 10),
                ("blendMode", C.c_int), ("renderMode", C.c_int), ("lightPositions", C.c_float * 30),
                ("lightColors", C.c_float * 30), ("lightSizes", C.c_float * 10), ("lightCount", C.c_int),
                ("showDofFocalPlane", C.c_int)]


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(os.fspath(LIB_PATH))
        assert L.orc_uniforms_size() == C.sizeof(Uniforms)
        L.orc_sdf.restype = C.c_float
        L.orc_sdf.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_float]
        L.orc_sdbox.restype = C.c_float
        L.orc_sdbox.argtypes = [C.c_float] * 6
        L.orc_gold_noise.restype = C.c_float
        L.orc_gold_noise.argtypes = [C.c_float] * 3
        L.orc_builtin.restype = C.c_float
        L.orc_builtin.argtypes = [C.c_int, C.c_float, C.c_float]
        L.orc_f16_to_f32.restype = C.c_float
        L.orc_f16_to_f32.argtypes = [C.c_uint16]
        L.orc_f32_to_f16.restype = C.c_uint16
        L.orc_f32_to_f16.argtypes = [C.c_float]
        L.orc_sdf_evals_reset.restype = C.c_ulonglong
        L.orc_de_iterations_reset.restype = C.c_ulonglong
        L.orc_scene_name.restype = C.c_char_p
        L.orc_materials.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_float, C.c_void_p]
        L.orc_materials_n.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
        L.orc_render_sample.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.orc_display.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_int]
        L.orc_uniform_samples.argtypes = [C.c_float, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.orc_preview_exit_steps.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.orc_trace_pixel.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        _lib = L
    return _lib


# declaration order of each scene's custom uniforms (flat float array handed to the oracle)
SCENE_UNIFORM_ORDER = {
    "guide": ["bigSphereSize", "fractalColor", "fractalIterations", "gridScaleFactor", "bigSphereCenter"],
    "fractal1": ["bigSphereSize", "fractalIterations", "gridScaleFactor", "bigSphereCenter"],
    "menger-sponge": ["fractalIterations"],
    "tree": ["fractalIterations", "scaleFactor", "angles", "offset"],
    "smooth-tree": ["fractalIterations", "scaleFactor", "angles", "offset", "smoothen"],
    "rotation-fractal": ["fractalIterations", "scaleFactor", "angles", "offset"],
    "sphere-grid": [],
    "inline-default": [],
    "mandelbulb": ["power", "bailout", "maxIterations"],
}


def flatten_custom(scene: str, custom: dict | None) -> np.ndarray:
    """dict name -> UniformData-like (.data) or sequence  ->  flat float32 array in oracle order"""
    vals = []
    if custom:
        for name in SCENE_UNIFORM_ORDER[scene]:
            v = custom[name]
            data = getattr(v, "data", v)
            vals += [float(x) for x in (data if hasattr(data, "__len__") else [data])]
    return np.asarray(vals, dtype=np.float32)


def uniforms_from_schema(schema, rand_noise) -> Uniforms:
    """The uniform derivations of RenderJobExecutor.tsx:212-297, restated for the oracle
    (independently of raymarching_engine_b200.executor.builtin_uniforms)."""
    U = Uniforms()
    r = schema.render
    U.blendWithPreviousFactor = r.blendWithPreviousFrameFactor
    U.randNoise[0], U.randNoise[1] = rand_noise
    for i in range(3):
        U.position[i] = schema.camera.position[i]
    for i in range(16):
        U.rotation[i] = schema.camera.rotation[i]
    U.dofAmount = schema.dof.amount
    U.dofFocalPlaneDistance = schema.dof.distance
    t = schema.camera.mode.type
    U.cameraMode = {"perspective": 0, "orthographic": 1, "panoramic": 2}.get(t, -1)
    U.fov = schema.camera.mode.fov if t == "perspective" else schema.camera.mode.size if t == "orthographic" else 1
    U.reflections = len(schema.reflectionIterationCounts)
    U.aspect = r.width / r.height
    U.fogDensity = schema.fogDensity
    U.exposure = r.exposure / r.samplesPerPixel
    for i, c in enumerate(schema.reflectionIterationCounts[:10]):
        U.raymarchingStepCountsArray[i] = c
    U.blendMode = 1 if r.blendMode == "additive" else 0
    U.renderMode = 1 if r.renderMode == "preview" else 0
    U.lightCount = len(schema.lights)
    for j, l in enumerate(schema.lights[:10]):
        p = l.position if l.type == "point" else l.direction
        for k in range(3):
            U.lightPositions[3 * j + k] = p[k]
            U.lightColors[3 * j + k] = l.color[k]
        U.lightSizes[j] = l.size if l.type == "point" else 0
    U.showDofFocalPlane = 1 if schema.dof.showFocusedArea else 0
    return U


class Accumulators:
    """Host copies of the three accumulators + the fp32 depth plane, row 0 = bottom."""

    def __init__(self, W: int, H: int):
        self.W, self.H = W, H
        self.color = np.zeros((H, W, 4), np.float32)
        self.nd = np.zeros((H, W, 4), np.uint16)
        self.ad = np.zeros((H, W, 4), np.uint16)
        self.depth = np.zeros((H, W), np.float32)


def render_sample(scene: str, custom, U: Uniforms, acc: Accumulators, scissor=None, nthreads: int | None = None) -> None:
    sx, sy, sw, sh = scissor if scissor is not None else (0, 0, acc.W, acc.H)
    cu = flatten_custom(scene, custom)
    nthreads = nthreads or os.cpu_count() or 1
    st = lib().orc_render_sample(scene.encode(), cu.ctypes.data_as(C.c_void_p) if cu.size else None, int(cu.size), C.byref(U),
                                 acc.W, acc.H, int(sx), int(sy), int(sw), int(sh), acc.color.ctypes.data_as(C.c_void_p),
                                 acc.nd.ctypes.data_as(C.c_void_p), acc.ad.ctypes.data_as(C.c_void_p),
                                 acc.depth.ctypes.data_as(C.c_void_p), nthreads)
    if st != 0:
        raise RuntimeError(f"oracle render_sample({scene}) failed: {st}")


def display(acc: Accumulators, brightness: float, nthreads: int | None = None) -> np.ndarray:
    out = np.zeros((acc.H, acc.W, 4), np.uint8)
    lib().orc_display(acc.color.ctypes.data_as(C.c_void_p), acc.nd.ctypes.data_as(C.c_void_p), acc.W, acc.H,
                      C.c_float(float(np.float32(brightness))), out.ctypes.data_as(C.c_void_p), nthreads or os.cpu_count() or 1)
    return out


def executed_work(scene: str, schema, rand_noise=(0.5, 1.0 / 3.0)):
    """Workload analysis of one preview-mode sample (orc_preview_exit_steps): (SDF evaluations a bit-exact early-out
    kernel executes, Mandelbulb DE-loop trips inside them - 0 for the other scenes)."""
    r = schema.render
    U = uniforms_from_schema(schema, rand_noise)
    cu = flatten_custom(scene, schema.customShaderParameters)
    out = np.zeros((r.height, r.width), np.int32)
    L = lib()
    L.orc_de_iterations_reset()
    st = L.orc_preview_exit_steps(scene.encode(), cu.ctypes.data_as(C.c_void_p) if cu.size else None, int(cu.size), C.byref(U), r.width, r.height,
                                  out.ctypes.data_as(C.c_void_p))
    if st != 0:
        raise RuntimeError(f"oracle exit_steps({scene}) failed: {st}")
    return int(out.sum()), int(L.orc_de_iterations_reset())


def materials(scene: str, custom, points) -> np.ndarray:
    """orc_materials at every point: n x 17 (the layout of the device probe kernel rmb_probe)"""
    pts = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
    out = np.zeros((len(pts), 17), np.float32)
    cu = flatten_custom(scene, custom)
    st = lib().orc_materials_n(scene.encode(), cu.ctypes.data_as(C.c_void_p) if cu.size else None, int(cu.size),
                               pts.ctypes.data_as(C.c_void_p), len(pts), out.ctypes.data_as(C.c_void_p))
    if st != 0:
        raise RuntimeError(f"oracle materials({scene}) failed: {st}")
    return out


def halton_seq(base: int, n: int) -> list:
    out = (C.c_double * n)()
    lib().orc_halton(base, n, out)
    return list(out)


def run_job(scene: str, schema, halton_start: int = 0, acc: Accumulators | None = None, nthreads: int | None = None):
    """Oracle-side restatement of the doRenderJob loop (RenderJobExecutor.tsx:148-331) followed by the
    final present (index.tsx:25-59) with brightness 1/(spp*subdivisions^2).  Sample k (0-based count of
    samples since the Halton generators were created) uses halton index halton_start + k."""
    r = schema.render
    acc = acc or Accumulators(r.width, r.height)
    total = r.subdivisions * r.subdivisions * r.samplesPerPixel
    h2 = halton_seq(2, halton_start + total)
    h3 = halton_seq(3, halton_start + total)
    k = halton_start
    for yp in range(r.subdivisions):
        for xp in range(r.subdivisions):
            for _ in range(r.samplesPerPixel):
                x1 = math.floor((r.width / r.subdivisions) * xp)
                y1 = math.floor((r.height / r.subdivisions) * yp)
                x2 = math.ceil((r.width / r.subdivisions) * (xp + 1))
                y2 = math.ceil((r.height / r.subdivisions) * (yp + 1))
                U = uniforms_from_schema(schema, (h2[k], h3[k]))
                render_sample(scene, schema.customShaderParameters, U, acc, (x1, y1, x2, y2), nthreads)   # gl.scissor(x1,y1,x2,y2) quirk
                k += 1
    rgba = display(acc, 1.0 / total, nthreads)
    return acc, rgba
