"""ctypes binding of libraymarch_b200.so (C ABI: include/rmb.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``csrc/Makefile``.  There is no
fallback: if the shared object is missing, importing this module raises, and every rendering
entry point fails loudly when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libraymarch_b200.so"

RMB_OK, RMB_ERR_FRAGMENT, RMB_ERR_PROGRAM, RMB_ERR_GENERAL, RMB_ERR_INVALID = range(5)
FLAVOUR_EXACT, FLAVOUR_FAST, FLAVOUR_EXACT_ALT = 0, 1, 2
UNIFORM_F, UNIFORM_I, UNIFORM_UI = 0, 1, 2

# every symbol include/rmb.h declares; tests check that the library exports all of them
EXPORTED_SYMBOLS = [
    "rmb_abi_version", "rmb_ctx_create", "rmb_ctx_destroy", "rmb_last_error", "rmb_ctx_stream", "rmb_sync", "rmb_ctx_set_pipeline", "rmb_ctx_launch_count", "rmb_ctx_timing", "rmb_ctx_set_gather_target", "rmb_fb_scatter_rows", "rmb_display_planes", "rmb_ipc_export", "rmb_ipc_open", "rmb_ipc_close",
    "rmb_program_get", "rmb_program_is_live", "rmb_program_source", "rmb_program_kernel_attr", "rmb_uniform_set", "rmb_uniform_set_array",
    "rmb_uniform_matrix4", "rmb_fb_acquire", "rmb_fb_release", "rmb_fb_local_rows", "rmb_fb_global_row",
    "rmb_render_sample", "rmb_present", "rmb_present_device", "rmb_present_async", "rmb_present_wait", "rmb_fb_device_ptr", "rmb_fb_plane_bytes",
    "rmb_fb_read", "rmb_fb_write", "rmb_fb_copy_to_device", "rmb_counters_read_all", "rmb_program_has_carve", "rmb_probe_carve", "rmb_probe", "rmb_compile_only", "rmb_translate_only", "rmb_host_alloc", "rmb_device_alloc", "rmb_device_free",
    "rmb_host_free", "rmb_measure_fp32_peak", "rmb_measure_fp32x2_peak", "rmb_owned_rows_below",
    "rmb_uniforms_set_frame", "rmb_host_register", "rmb_host_unregister", "rmb_stream_write_u32", "rmb_stream_wait_geq_u32", "rmb_ctx_wait_ctx",
    "rmb_group_create", "rmb_group_destroy", "rmb_group_last_error", "rmb_group_size", "rmb_group_ctx", "rmb_group_sync", "rmb_group_program_get",
    "rmb_group_program_member", "rmb_group_uniform_set", "rmb_group_uniform_set_array", "rmb_group_uniform_matrix4", "rmb_group_uniforms_set_frame", "rmb_group_fb_acquire",
    "rmb_group_fb_release", "rmb_group_fb_member", "rmb_group_render_sample", "rmb_group_present", "rmb_group_present_device",
]


class SpecData(C.Union):
    _fields_ = [("f", C.c_float * 4), ("i", C.c_int32 * 4), ("u", C.c_uint32 * 4)]


class SpecUniform(C.Structure):
    _fields_ = [("name", C.c_char_p), ("type", C.c_int), ("count", C.c_int), ("data", SpecData)]


class FrameUniforms(C.Structure):        # rmb_frame_uniforms (include/rmb.h)
    _fields_ = [("blendWithPreviousFactor", C.c_float), ("randNoise", C.c_float * 2), ("position", C.c_float * 3),
                ("rotation", C.c_float * 16), ("dofAmount", C.c_float), ("dofFocalPlaneDistance", C.c_float),
                ("cameraMode", C.c_int32), ("fov", C.c_float), ("reflections", C.c_float), ("raymarchingSteps", C.c_float),
                ("indirectLightingRaymarchingSteps", C.c_float), ("aspect", C.c_float), ("fogDensity", C.c_float),
                ("exposure", C.c_float), ("blendMode", C.c_int32), ("renderMode", C.c_int32), ("stepCountsLength", C.c_int32),
                ("raymarchingStepCountsArray", C.c_float * 10), ("lightCount", C.c_int32), ("lightPositions", C.c_float * 30),
                ("lightColors", C.c_float * 30), ("lightSizes", C.c_float * 10), ("showDofFocalPlane", C.c_int32)]


def _load() -> C.CDLL:
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C raymarching_engine_b200/csrc`). There is no CPU fallback."
        )
    lib = C.CDLL(os.fspath(LIB_PATH))
    vp, cp, i, sz, f = C.c_void_p, C.c_char_p, C.c_int, C.c_size_t, C.c_float
    proto = {
        "rmb_abi_version": (i, []),
        "rmb_ctx_create": (vp, [i, i, i, i]),
        "rmb_ctx_destroy": (None, [vp]),
        "rmb_last_error": (cp, [vp]),
        "rmb_ctx_stream": (vp, [vp]),
        "rmb_sync": (i, [vp]),
        "rmb_ctx_set_pipeline": (i, [vp, i]),
        "rmb_ctx_launch_count": (C.c_uint64, [vp]),
        "rmb_ctx_timing": (i, [vp, i, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
        "rmb_ctx_set_gather_target": (i, [vp, vp, sz]),
        "rmb_fb_scatter_rows": (i, [vp, vp, i, vp]),
        "rmb_display_planes": (i, [vp, vp, vp, vp, i, i, f]),
        "rmb_ipc_export": (i, [vp, C.c_char_p]),
        "rmb_ipc_open": (i, [vp, C.c_char_p, C.POINTER(vp)]),
        "rmb_ipc_close": (i, [vp, vp]),
        "rmb_program_get": (i, [vp, cp, sz, i, C.POINTER(SpecUniform), i, C.POINTER(vp), cp, cp, sz]),
        "rmb_program_is_live": (i, [vp]),
        "rmb_program_source": (cp, [vp]),
        "rmb_program_kernel_attr": (i, [vp, i, C.POINTER(i), C.POINTER(i)]),
        "rmb_uniform_set": (i, [vp, cp, i, i, vp]),
        "rmb_uniform_set_array": (i, [vp, cp, i, i, i, vp]),
        "rmb_uniform_matrix4": (i, [vp, cp, C.POINTER(f)]),
        "rmb_fb_acquire": (vp, [vp, i, i, C.c_int64]),
        "rmb_fb_release": (None, [vp, i, i, C.c_int64]),
        "rmb_fb_local_rows": (i, [vp]),
        "rmb_fb_global_row": (i, [vp, i]),
        "rmb_render_sample": (i, [vp, vp, vp, i, i, i, i]),
        "rmb_present": (i, [vp, vp, f, vp, vp]),
        "rmb_present_device": (i, [vp, vp, f]),
        "rmb_present_async": (i, [vp, vp, f, vp, vp]),
        "rmb_present_wait": (i, [vp, vp]),
        "rmb_fb_device_ptr": (vp, [vp, i]),
        "rmb_fb_plane_bytes": (sz, [vp, i]),
        "rmb_fb_read": (i, [vp, vp, i, vp, sz]),
        "rmb_fb_write": (i, [vp, vp, i, vp, sz]),
        "rmb_fb_copy_to_device": (i, [vp, vp, i, vp, sz]),
        "rmb_counters_read_all": (i, [vp, C.POINTER(C.c_uint64), i]),
        "rmb_program_has_carve": (i, [vp]),
        "rmb_probe_carve": (i, [vp, vp, vp, i, vp]),
        "rmb_probe": (i, [vp, vp, vp, i, vp]),
        "rmb_compile_only": (i, [cp, sz, i, C.POINTER(SpecUniform), i, cp, sz, vp, sz, C.POINTER(sz), cp, sz]),
        "rmb_translate_only": (i, [cp, sz, i, C.POINTER(SpecUniform), i, cp, sz, cp, sz]),
        "rmb_measure_fp32_peak": (i, [vp, C.c_double, C.POINTER(C.c_double)]),
        "rmb_measure_fp32x2_peak": (i, [vp, C.c_double, C.POINTER(C.c_double)]),
        "rmb_owned_rows_below": (i, [i, i, i, i, i]),
        "rmb_host_alloc": (vp, [sz]),
        "rmb_device_alloc": (vp, [vp, sz]),
        "rmb_device_free": (None, [vp, vp]),
        "rmb_host_free": (None, [vp]),
        "rmb_uniforms_set_frame": (i, [vp, C.POINTER(FrameUniforms)]),
        "rmb_host_register": (i, [vp, sz]),
        "rmb_host_unregister": (i, [vp]),
        "rmb_stream_write_u32": (i, [vp, vp, C.c_uint32]),
        "rmb_stream_wait_geq_u32": (i, [vp, vp, C.c_uint32]),
        "rmb_ctx_wait_ctx": (i, [vp, vp]),
        "rmb_group_create": (vp, [C.POINTER(i), i, i]),
        "rmb_group_destroy": (None, [vp]),
        "rmb_group_last_error": (cp, [vp]),
        "rmb_group_size": (i, [vp]),
        "rmb_group_ctx": (vp, [vp, i]),
        "rmb_group_sync": (i, [vp]),
        "rmb_group_program_get": (i, [vp, cp, sz, i, C.POINTER(SpecUniform), i, C.POINTER(vp), cp, cp, sz]),
        "rmb_group_program_member": (vp, [vp, i]),
        "rmb_group_uniform_set": (i, [vp, cp, i, i, vp]),
        "rmb_group_uniform_set_array": (i, [vp, cp, i, i, i, vp]),
        "rmb_group_uniform_matrix4": (i, [vp, cp, C.POINTER(f)]),
        "rmb_group_uniforms_set_frame": (i, [vp, C.POINTER(FrameUniforms)]),
        "rmb_group_fb_acquire": (vp, [vp, i, i, C.c_int64]),
        "rmb_group_fb_release": (None, [vp, i, i, C.c_int64]),
        "rmb_group_fb_member": (vp, [vp, i]),
        "rmb_group_render_sample": (i, [vp, vp, vp, i, i, i, i]),
        "rmb_group_present": (i, [vp, vp, f, vp, vp]),
        "rmb_group_present_device": (i, [vp, vp, f, C.POINTER(vp)]),
    }
    for name, (res, args) in proto.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.rmb_abi_version() != 1:
        raise ImportError("libraymarch_b200.so ABI version mismatch")
    return lib


lib = _load()


def make_spec_array(spec: dict | None):
    """dict name -> UniformData-like (type 'f'|'i'|'ui', data sequence)  ->  (ctypes array, n)"""
    if not spec:
        return None, 0
    arr = (SpecUniform * len(spec))()
    for k, (name, ud) in enumerate(sorted(spec.items())):
        arr[k].name = name.encode()
        t = {"f": UNIFORM_F, "i": UNIFORM_I, "ui": UNIFORM_UI}[ud.type]
        arr[k].type = t
        arr[k].count = ud.count
        for j, v in enumerate(ud.data):
            if t == UNIFORM_F:
                arr[k].data.f[j] = float(v)
            elif t == UNIFORM_I:
                arr[k].data.i[j] = int(v)
            else:
                arr[k].data.u[j] = int(v)
    return arr, len(spec)
