"""GLSL -> CUDA lowering and NVRTC compilation for sm_100a, exercised without a GPU
(NVRTC is a compiler; rmb_compile_only never touches a device)."""
import ctypes as C
import re

import pytest

import raymarching_engine_b200 as rm
from raymarching_engine_b200 import _lib
from conftest import SCENES, scene_source

L = _lib.lib


def compile_only(src, flavour=_lib.FLAVOUR_EXACT, spec=None, want_source=True):
    log = C.create_string_buffer(1 << 16)
    n = C.c_size_t(0)
    out = C.create_string_buffer(1 << 20) if want_source else None
    arr, ns = _lib.make_spec_array(spec)
    b = src.encode()
    st = L.rmb_compile_only(b, len(b), flavour, arr, ns, log, len(log), None, 0, C.byref(n), out, len(out) if out else 0)
    return st, log.value.decode(), n.value, (out.value.decode() if out else "")


@pytest.mark.parametrize("name", SCENES)
def test_every_bundled_scene_compiles_for_sm100a(name):
    src = scene_source(name)
    st, log, nbytes, tu = compile_only(src, _lib.FLAVOUR_EXACT, rm.default_custom_settings(src))
    assert st == _lib.RMB_OK, log
    assert nbytes > 10000
    assert "rm_preview_kernel" in tu and "rm_full_kernel" in tu


def test_fast_flavour_and_generic_variant_compile():
    src = scene_source("guide")
    st, log, nbytes, tu = compile_only(src, _lib.FLAVOUR_FAST, rm.default_custom_settings(src))
    assert st == _lib.RMB_OK, log
    assert "#define RM_FLAVOUR_FAST 1" in tu
    st, log, nbytes, tu = compile_only(src, _lib.FLAVOUR_EXACT, None)
    assert st == _lib.RMB_OK, log
    assert "__constant__ float fractalIterations;" in tu and "__constant__ vec3 bigSphereCenter;" in tu


def test_uniform_extraction_baking_and_defaults():
    src = scene_source("fractal1")          # defines only sdf(): all seven material functions are injected
    st, log, _, tu = compile_only(src, spec={"fractalIterations": rm.u.float(8), "bigSphereCenter": rm.u.vec3(0, 0, 10)})
    assert st == _lib.RMB_OK, log
    assert "const float fractalIterations = __int_as_float(0x41000000)" in tu
    assert "const vec3 bigSphereCenter = vec3(" in tu
    assert "__constant__ float bigSphereSize;" in tu          # not baked -> stays dynamic
    assert "uniform" not in tu.split('#line 1 "scene.glsl"')[1].split("#line")[0]
    for fn in ("sceneDiffuseColor", "sceneSpecularColor", "sceneSpecularRoughness", "sceneSubsurfaceScattering",
               "sceneSubsurfaceScatteringColor", "sceneIOR", "sceneEmission"):
        assert tu.count(f" {fn}(vec3 position)") == 1, fn
    # a constant-trip loop over a baked uniform is marked for unrolling; one over a dynamic uniform is not
    assert '_Pragma("unroll 32") for (float i = -1.0f; i < fractalIterations; i++)' in tu
    st, log, _, tu2 = compile_only(src, spec=None)
    assert st == _lib.RMB_OK and "_Pragma" not in tu2.split('#line 1 "scene.glsl"')[1].split("#line")[0]


def test_guide_defines_all_materials_so_none_are_injected():
    st, log, _, tu = compile_only(scene_source("guide"))
    assert st == _lib.RMB_OK, log
    assert tu.count("vec3 sceneEmission(vec3 position)") == 1


def test_literals_qualifiers_and_keywords():
    src = """
precision highp float;
uniform highp float k;
const float A = 1.;
float helper(in float a, out float b, inout vec3 c) { b = a * .5 + 1e-3; c *= 2.0; return 3; }
float new(float not) { return not + 1.0; }
float sdf(vec3 p) {
  float o; vec3 q = p;
  float r = helper(p.x, o, q) + new(2.0) + A;
  bvec3 m = lessThan(p, vec3(0.0));
  if (any(not(m)) ^^ false) r += 0.5;
  return length(q.zyx) - o * k - r * 0.0;
}
"""
    st, log, _, tu = compile_only(src)
    assert st == _lib.RMB_OK, log
    body = tu.split('#line 1 "scene.glsl"')[1].split("#line")[0]
    assert "precision" not in body and "highp" not in body and "uniform" not in body
    assert "1.f" in body and ".5f" in body and "1e-3f" in body and "2.0f" in body
    flat = " ".join(body.split())
    assert "( float a, float& b, vec3& c)" in flat
    assert "new_rmk(float not_)" in flat and "not_(m)" in flat
    assert "return 3;" in body                      # integer literals are left alone


def test_purity_analysis_disables_early_exit():
    pure = "float sdf(vec3 p) { return length(p) - 1.0; }"
    rng = "float sdf(vec3 p) { return length(p) - 1.0 + 0.001 * uniformSample(); }"
    glob = "float counter = 0.0;\nfloat sdf(vec3 p) { counter += 1.0; return length(p) - 1.0; }"
    const_glob = "const float R = 1.0;\nfloat sdf(vec3 p) { return length(p) - R; }"
    for src, want in ((pure, 1), (rng, 0), (glob, 0), (const_glob, 1)):
        st, log, _, tu = compile_only(src)
        assert st == _lib.RMB_OK, log
        assert f"#define RM_PURE_SDF {want}" in tu


def test_compile_errors_are_values_with_gl_style_lines():
    # scene line numbers are offset by 145 like the spliced reference shader (GLSLEditor.tsx:134-136)
    st, log, _, _ = compile_only("float sdf(vec3 p) {\n  return lenght(p) - 1.0;\n}\n")
    assert st == _lib.RMB_ERR_FRAGMENT
    assert log.startswith("ERROR: 0:147:") and "lenght" in log
    st, log, _, _ = compile_only("vec3 sceneEmission(vec3 p) { return vec3(0.0); }\n")     # no sdf()
    assert st == _lib.RMB_ERR_FRAGMENT and "'sdf'" in log
    st, log, _, _ = compile_only("uniform sampler2D tex;\nfloat sdf(vec3 p) { return 1.0; }")
    assert st == _lib.RMB_ERR_FRAGMENT and "0:146" in log and "sampler" in log
    st, log, _, _ = compile_only("float sdf(vec3 p) { return 1.0; ")
    assert st == _lib.RMB_ERR_FRAGMENT


def test_translate_only_reports_scene_level_errors_without_compiling():
    """rmb_translate_only: the lowering alone (milliseconds) gives the scene-level diagnostics and the translation unit;
    errors only the C++ compiler can see (an undeclared identifier) need rmb_compile_only.  The march has one
    implementation with fixed tunables: the translation unit carries no switch for them."""
    def translate(src):
        log = C.create_string_buffer(1 << 16)
        out = C.create_string_buffer(2 << 20)
        b = src.encode()
        st = L.rmb_translate_only(b, len(b), _lib.FLAVOUR_EXACT, None, 0, log, len(log), out, len(out))
        return st, log.value.decode(), out.value.decode()
    st, log, tu = translate(scene_source("guide"))
    assert st == _lib.RMB_OK and "rm_wf_march_preview_kernel" in tu and "__constant__ float fractalIterations;" in tu
    for name in ("RM_DUAL", "scene_packed.glsl", "RM_FLOOR_FP_COMPONENTS", "RM_WF_CHUNK", "RM_REFILL_MIN", "RM_MARCH_MIN_BLOCKS",
                 "RM_BOUNCE_MIN_BLOCKS", "RM_USE_F32X2"):
        assert name not in tu, name
    assert set(re.findall(r"\bRMB_\w+", tu)) <= {"RMB_PROFILE"}    # the kernel text names only the profiling switch
    st, log, _ = translate("vec3 sceneEmission(vec3 p) { return vec3(0.0); }\n")
    assert st == _lib.RMB_ERR_FRAGMENT and "'sdf'" in log
    st, log, _ = translate("uniform sampler2D tex;\nfloat sdf(vec3 p) { return 1.0; }")
    assert st == _lib.RMB_ERR_FRAGMENT and "0:146" in log and "sampler" in log
    st, log, _ = translate("float sdf(vec3 p) { return 1.0; ")
    assert st == _lib.RMB_ERR_FRAGMENT
    st, log, _ = translate("float sdf(vec3 p) {\n  return lenght(p) - 1.0;\n}\n")
    assert st == _lib.RMB_OK          # not a lowering error
    assert L.rmb_translate_only(None, 0, _lib.FLAVOUR_EXACT, None, 0, None, 0, None, 0) == _lib.RMB_ERR_INVALID


def test_uniform_arrays_matrices_and_int_vectors():
    src = """
uniform float weights[4];
uniform ivec3 cell;
uniform mat3 basis;
uniform bool flip;
float sdf(vec3 p) {
  vec3 q = basis * p + vec3(cell);
  float s = 0.0;
  for (int i = 0; i < 4; i++) s += weights[i];
  return (flip ? -1.0 : 1.0) * (length(q) - s);
}
"""
    st, log, _, tu = compile_only(src)
    assert st == _lib.RMB_OK, log
    assert "__constant__ float weights[4];" in tu and "__constant__ ivec3 cell;" in tu and "__constant__ mat3 basis;" in tu


def test_preprocessor_directives_are_sandboxed():
    """ADVICE r1: the scene is sandboxed GLSL ES in the reference.  #include (NVRTC would read host files and quote them
    in the info log) and any non-GLSL directive are compile errors; macros may not take the names of the pipeline the
    scene is spliced into; and a legal scene macro ends with the scene text (it is #undef'd before the kernels)."""
    def translate(src):
        log = C.create_string_buffer(1 << 16)
        out = C.create_string_buffer(2 << 20)
        b = src.encode()
        st = L.rmb_translate_only(b, len(b), _lib.FLAVOUR_EXACT, None, 0, log, len(log), out, len(out))
        return st, log.value.decode(), out.value.decode()
    sdf = "float sdf(vec3 p) { return length(p) - 1.0; }\n"
    st, log, _ = translate('#include "/etc/passwd"\n' + sdf)
    assert st == _lib.RMB_ERR_FRAGMENT and log.startswith("ERROR: 0:146:") and "include" in log and "root:" not in log
    st, log, _ = translate(sdf + "#  include </etc/hostname>\n")
    assert st == _lib.RMB_ERR_FRAGMENT and "include" in log
    for bad in ("#import x", "#warning hello", "#include_next <x>", "#assert x"):
        assert translate(bad + "\n" + sdf)[0] == _lib.RMB_ERR_FRAGMENT, bad
    for name in ("sdfAt", "g_fma", "rm_carve_outer", "RM_BLOCK_THREADS", "GLSL_FAST", "__launch_bounds__", "gl_FragCoord"):
        st, log, _ = translate(f"#define {name} 1\n" + sdf)
        assert st == _lib.RMB_ERR_FRAGMENT and name in log and "reserved" in log, name
        assert translate(f"#undef {name}\n" + sdf)[0] == _lib.RMB_ERR_FRAGMENT, name
    # legal directives pass through, and the macro does not outlive the scene
    src = "#define RADIUS 1.5\n#define lane 7\n#ifdef RADIUS\nfloat sdf(vec3 p) { return length(p) - RADIUS; }\n#else\n#error no radius\n#endif\n"
    st, log, tu = translate(src)
    assert st == _lib.RMB_OK, log
    scene_at, undef_at, kernels_at = tu.index("#define RADIUS 1.5"), tu.index("#undef RADIUS"), tu.rindex("rm_wf_march_preview_kernel")
    assert scene_at < undef_at < kernels_at and "#undef lane" in tu
    st, log, _, _ = compile_only(src, want_source=False)      # `lane` is a variable of the march kernel: still compiles
    assert st == _lib.RMB_OK, log
