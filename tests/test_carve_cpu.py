"""Far-field shortcut for carved scenes (lower_glsl.cpp pass 1b, include/rmb.h rmb_program_has_carve).

The product has no CPU path, so the claim "sdf(P) == A(P) bit for bit wherever A(P) > U" is checked here
on the LOWERED TEXT itself: the scene functions and the two helpers the lowering emits are cut out of the
translation unit rmb_compile_only returns, compiled with g++ against the shared deterministic math
(glsl_rt.h, exact policy, the oracle's flags) and evaluated at a few hundred thousand positions, including
the non-finite ones escaping rays reach.  The GPU side of the same claim is tests/test_parity_gpu.py
(test_carve_*: probe kernel, far-field on/off frames, oracle parity of every scene with the shortcut on) and, at the
settings-tab value sets of tests/slider_cases.py that both files also run here, tests/test_slider_values_gpu.py.
"""
import ctypes as C
import os
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

import raymarching_engine_b200 as rm
from raymarching_engine_b200 import _lib
import slider_cases
from conftest import scene_source

L = _lib.lib
ROOT = Path(__file__).resolve().parent.parent
DEVICE_SRC = ROOT / "raymarching_engine_b200" / "csrc" / "device_src"


def translation_unit(src, spec=None, flavour=_lib.FLAVOUR_EXACT, compile=False):
    log = C.create_string_buffer(1 << 16)
    n = C.c_size_t(0)
    out = C.create_string_buffer(2 << 20)
    arr, ns = _lib.make_spec_array(spec)
    b = src.encode()
    if compile:       # through NVRTC for sm_100a as well
        st = L.rmb_compile_only(b, len(b), flavour, arr, ns, log, len(log), None, 0, C.byref(n), out, len(out))
    else:
        st = L.rmb_translate_only(b, len(b), flavour, arr, ns, log, len(log), out, len(out))
    assert st == _lib.RMB_OK, log.value.decode()
    return out.value.decode()


def has_carve(src, spec=None, compile=False):
    tu = translation_unit(src, spec, compile=compile)
    on = "#define RM_HAS_CARVE 1" in tu
    assert on == ("float rm_carve_outer(" in tu) == ("float rm_carve_bound(" in tu)
    return on


SDF = """
uniform float R;
uniform float s0;
float sdf(vec3 p) {
  float m = 1000.0;
  for (float i = 0.0; i < 4.0; i++) {
    float sf = pow(s0, i);
    vec3 d = mod(p + vec3(0.5 * sf), sf) - vec3(sf / 2.0);
    %s
  }
  %s
}
"""


def _scene(loop_tail="float dist = length(d) - 0.3 * sf; m = min(dist, m);", end="return max(length(p) - R, -m);"):
    return SDF % (loop_tail, end)


def test_accepted_shapes():
    assert has_carve(scene_source("guide"))
    assert has_carve(scene_source("guide"), rm.default_custom_settings(scene_source("guide")))
    assert has_carve(scene_source("inline-default"))
    assert has_carve(scene_source("fractal1"))
    assert has_carve(_scene())
    assert has_carve(_scene("m = min(m, length(d) - 0.3 * sf);"))                       # inline term, M first
    assert has_carve(_scene(end="m = max(-m, length(p) - R); return m;"), compile=True)  # operands swapped, assigned; NVRTC takes it
    assert has_carve(_scene(end="float r = max(length(p) - R, -m); return r;"))
    assert has_carve(_scene("float k = 0.3 * sf / 2.0; float dist = length(d) - k; m = min(dist, m);"))
    for name in ("sphere-grid", "mandelbulb", "tree", "smooth-tree", "rotation-fractal"):
        assert not has_carve(scene_source(name)), name                                    # not of that form
    # pattern B: boxes carved out of an outer shape level by level (X = max(X, -E), E a min() tree of sdBox calls)
    assert has_carve(scene_source("menger-sponge"), compile=True)
    assert has_carve(scene_source("menger-sponge"), rm.default_custom_settings(scene_source("menger-sponge")))
    assert has_carve(_boxes())
    assert has_carve(_boxes("x = max(-sdBox(g, vec3(sf)), x);"))                          # operands swapped, a single box
    assert has_carve(_boxes(init="length(p) - R"))                                         # any outer shape of the position


BOXES = """
uniform float R;
uniform float s0;
float sdf(vec3 p) {
  float x = %s;
  for (float i = 1.0; i < 4.0; i++) {
    float sf = pow(s0, i);
    vec3 g = mod(p, sf * 3.0) - sf * 1.5;
    %s
  }
  return x;
}
"""


def _boxes(stmt="x = max(x, -min(sdBox(g, vec3(sf * 1.5, sf * 0.5, sf * 0.5)), sdBox(g.zxy, vec3(sf * 0.5, sf * 1.5, sf * 0.5))));",
           init="sdBox(p + vec3(0.5), vec3(R))"):
    return BOXES % (init, stmt)


@pytest.mark.parametrize("stmt,init", [
    ("x = max(x, -sdBox(g, vec3(sf * p.x)));", None),                        # half-extents depend on the position
    ("x = max(x, -sdBox(g, g));", None),
    ("x = max(x, sdBox(g, vec3(sf)));", None),                               # not a difference
    ("x = max(x, -sdBox(g, vec3(sf)) * 2.0);", None),
    ("x = max(x, -max(sdBox(g, vec3(sf)), sdBox(g, vec3(sf * 0.5))));", None),   # an intersection inside: no lower bound from the boxes alone
    ("x = max(x, -(length(g) - sf));", None),                                # not a box (pattern A handles spheres in its own form)
    ("x = min(x, -sdBox(g, vec3(sf)));", None),
    ("x = max(x, -sdBox(g, vec3(sf))); x += 0.01;", None),                   # the accumulator is touched some other way
    ("x = max(x, -sdBox(g, vec3(sf))) - 0.01;", None),
    ("float y = x; x = max(x, -sdBox(g, vec3(sf)));", None),
    ("if (p.x > 0.0) x = max(x, -sdBox(g, vec3(sf)));", None),
    ("x = max(x, -sdBox(g, vec3(sf = sf * 2.0)));", None),                   # side effect inside
    ("x = max(x, -sdBox(g * x, vec3(sf)));", None),                          # the accumulator feeds its own term
    (None, "sdBox(p, vec3(R)) + s0 * sdfFractal(p)"),                        # outer shape calls something the analysis does not know
    (None, "1.0"),                                                           # (accepted shape, but see below: must still be exact)
])
def test_rejected_box_shapes(stmt, init):
    kw = {}
    if stmt is not None:
        kw["stmt"] = stmt
    if init is not None:
        kw["init"] = init
    if init == "1.0":
        assert has_carve(_boxes(**kw))           # a constant outer shape is a (useless but valid) function of the position
        return
    assert not has_carve(_boxes(**kw))


def test_box_scene_with_its_own_sdBox_is_rejected():
    assert not has_carve("float sdBox(vec3 p, vec3 b) { return length(p) - b.x - 10.0; }\n" + _boxes())
    assert not has_carve(_boxes() + "\nfloat rm_box0(vec3 b) { return 0.0; }\n")


@pytest.mark.parametrize("loop_tail,end", [
    # a term whose offset depends on the position
    ("float dist = length(d) - 0.3 * sf * p.x; m = min(dist, m);", None),
    ("float k = d.x; float dist = length(d) - k; m = min(dist, m);", None),
    # not `length - K`
    ("float dist = length(d) * 0.5 - 0.3 * sf; m = min(dist, m);", None),
    ("float dist = length(d) - 0.3 * sf + p.y; m = min(dist, m);", None),
    ("float dist = -length(d) - 0.3 * sf; m = min(dist, m);", None),
    ("float dist = d.x - 0.3 * sf; m = min(dist, m);", None),
    ("float dist = length(d) - 0.3 * sf; m = max(dist, m);", None),
    # control flow the analysis does not follow
    ("float dist = length(d) - 0.3 * sf; if (p.x > 0.0) m = min(dist, m);", None),
    ("float dist = length(d) - 0.3 * sf; m = p.x > 0.0 ? min(dist, m) : m;", None),
    ("float dist = length(d) - 0.3 * sf; m = min(dist, m); if (m < 0.0) break;", None),
    ("float dist = length(d) - 0.3 * sf; m = min(dist, m); if (m < 0.0) return m;", None),
    # the accumulator or the term is touched some other way
    ("float dist = length(d) - 0.3 * sf; m = min(dist, m); m -= 0.1;", None),
    ("float dist = length(d) - 0.3 * sf; dist -= p.x; m = min(dist, m);", None),
    ("float dist = length(d) - 0.3 * sf; m = min(dist, m) - 0.1;", None),
    ("float dist = length(d) - 0.3 * sf; float q = m; m = min(dist, m);", None),
    ("sf = sf * p.x; float dist = length(d) - 0.3 * sf; m = min(dist, m);", None),
    ("i += p.x; float dist = length(d) - 0.3 * sf; m = min(dist, m);", None),
    ("p = p * 2.0; float dist = length(d) - 0.3 * sf; m = min(dist, m);", None),
    # the result is not max(A, -M), or A is not a function of the position and uniforms alone
    (None, "return max(length(p) - R, m);"),
    (None, "return max(length(p) - R, -m) + 0.1;"),
    (None, "return min(length(p) - R, -m);"),
    (None, "return max(length(p) - R, -m * 2.0);"),
    (None, "float t = m * 0.5; return max(length(p) - t, -m);"),
    (None, "return max(length(p) - R, max(-m, 0.0));"),
])
def test_rejected_shapes(loop_tail, end):
    kw = {}
    if loop_tail is not None:
        kw["loop_tail"] = loop_tail
    if end is not None:
        kw["end"] = end
    assert not has_carve(_scene(**kw))


def test_rejected_contexts():
    good = _scene()
    assert has_carve(good)
    assert not has_carve("#define OFF 0.3\n" + good)                                          # macros can hide anything
    assert not has_carve(good.replace("float m = 1000.0;", "float m = R;"))                 # not a literal
    assert not has_carve(good.replace("float sdf(vec3 p) {", "float sdf(vec3 p) {\n  p = p.zyx;"))
    assert not has_carve(good + "\nvoid twist(inout vec3 q) { q = q.zyx; }\n")              # reference parameters anywhere
    assert not has_carve(good.replace("for (float i = 0.0; i < 4.0; i++)", "for (float i = 0.0; i < p.x; i++)"))
    assert not has_carve(good.replace("float sf = pow(s0, i);", "float sf = pow(s0, i); float R = 1.0;"))   # shadows a uniform
    assert not has_carve("float seedy = 0.0;\n" + good)                                       # impure scene: no wavefront pipeline at all
    assert not has_carve("float length(vec3 v) { return -1.0; }\n" + good)                   # a scene function named like a built-in
    assert not has_carve("float pow(float a, float b) { return a; }\n" + good)
    assert not has_carve(good + "\nfloat rm_len0(vec3 v) { return 1.0; }\n")                 # the helper names must be free
    assert not has_carve(good.replace("float dist", "float rm_carve_outer = 0.0; float dist"))
    # the switch
    os.environ["RMB_CARVE"] = "0"
    try:
        assert not has_carve(good)
    finally:
        del os.environ["RMB_CARVE"]


HARNESS = r"""
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <vector>
#define GLSL_NS xg
#define GLSL_FAST 0
#include "glsl_rt.h"
namespace xg {
%(uniforms)s
struct Frag {
    vec2 texcoord;
    ivec2 rm_texSize;
    template <class V> static float rm_len0(const V&) { return 0.0f; }
    float rm_box0(const vec3& b) { return -max(0.0f, max(b.x, max(b.y, b.z))); }
    float sdBox(vec3 p, vec3 b) { vec3 q = abs(p) - b; return length(max(q, 0.0f)) + min(max(q.x, max(q.y, q.z)), 0.0f); }
    float sdfSphere(vec3 position, vec3 center, float radius) { return distance(position, center) - radius; }
%(scene)s
};
}
int main(int argc, char** argv) {
    // stdin: n, then n * 3 floats; stdout: n * 3 floats (sdf, A, U), all binary
    uint32_t n = 0;
    if (fread(&n, 4, 1, stdin) != 1) return 2;
    std::vector<float> in(3 * (size_t)n), out(3 * (size_t)n);
    if (fread(in.data(), 4, in.size(), stdin) != in.size()) return 2;
    xg::Frag f;
    f.texcoord = xg::vec2(0.5f, 0.5f);
    f.rm_texSize = xg::ivec2(1, 1);
    const float U = f.rm_carve_bound();
    for (uint32_t i = 0; i < n; i++) {
        const xg::vec3 p(in[3 * i], in[3 * i + 1], in[3 * i + 2]);
        out[3 * i] = f.sdf(p);
        out[3 * i + 1] = f.rm_carve_outer(p);
        out[3 * i + 2] = U;
    }
    fwrite(out.data(), 4, out.size(), stdout);
    return 0;
}
"""


def _cxx_value(v):
    # bit-pattern literals, as rmb_api.cpp float_literal bakes them: NaN and +-inf uniforms compile too
    a = np.atleast_1d(np.asarray(v, dtype=np.float32))
    lit = ["__builtin_bit_cast(float, 0x%08xu)" % b for b in a.view(np.uint32)]
    return lit[0] if len(lit) == 1 else "vec%d(%s)" % (len(lit), ", ".join(lit))


def _build_harness(tmp_path, src, values):
    tu = translation_unit(src)                                    # generic variant: every scene uniform dynamic
    m = re.search(r'#line 1 "scene.glsl"\n(.*?)\n#line \d+ "raymarch_kernel.cuh"', tu, re.S)
    assert m
    scene = m.group(1)
    assert "rm_carve_outer" in scene and ("rm_len0" in scene or "rm_box0" in scene)
    decls = re.findall(r"^__constant__ (\w+) (\w+);$", tu, re.M)
    uniforms = "".join("static %s %s = %s;\n" % (t, nme, _cxx_value(values[nme])) for t, nme in decls if nme in values)
    assert len(uniforms.splitlines()) == len(values)
    cpp = tmp_path / "carve_harness.cpp"
    cpp.write_text(HARNESS % {"uniforms": uniforms, "scene": scene})
    exe = tmp_path / "carve_harness"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-mfma", "-Wno-unknown-pragmas", "-I", str(DEVICE_SRC),
                    str(cpp), "-o", str(exe)], check=True)
    return exe


def _points(rng, centre, radius):
    c = np.asarray(centre, np.float32)
    near = c + rng.uniform(-1.3, 1.3, (120000, 3)).astype(np.float32) * np.float32(radius)
    shell = c + (rng.normal(size=(60000, 3)) * 1.0).astype(np.float32)
    shell = c + (shell - c) / np.linalg.norm(shell - c, axis=1, keepdims=True).astype(np.float32) * \
        (np.float32(radius) + rng.uniform(-0.1, 1.5, (60000, 1)).astype(np.float32))
    with np.errstate(over="ignore"):        # overflow to +-inf is wanted
        far = (rng.normal(size=(60000, 3)) * 10.0 ** rng.uniform(0, 38.5, (60000, 1))).astype(np.float32)
    tiny = (rng.normal(size=(2000, 3)) * 10.0 ** rng.uniform(-45, -30, (2000, 1))).astype(np.float32)
    special = np.array([[np.inf, 0, 0], [0, -np.inf, 1], [np.inf, np.inf, -np.inf], [np.nan, 1, 2], [1, np.nan, np.inf],
                        [3.4e38, 3.4e38, 3.4e38], [-3.4e38, 1, 1], [0, 0, 0], [-0.0, -0.0, -0.0], [1e19, 1e19, 1e19], [2e19, 0, 0]], np.float32)
    with np.errstate(all="ignore"):
        return np.ascontiguousarray(np.concatenate([near, shell, far, tiny, special]).astype(np.float32))


def _run(exe, pts):
    blob = np.uint32(len(pts)).tobytes() + pts.tobytes()
    r = subprocess.run([str(exe)], input=blob, stdout=subprocess.PIPE, check=True)
    return np.frombuffer(r.stdout, np.float32).reshape(-1, 3)


SLIDER_CASES = ["%s/%s" % sc for sc in slider_cases.all_cases(slider_cases.CARVED)]


def _slider_case(case):
    """(source, plain uniform values, scene, case name) of a tests/slider_cases.py entry `scene/case`"""
    scene, name = case.split("/")
    src = scene_source(scene)
    return src, slider_cases.plain(slider_cases.custom(rm, src, scene, name)), scene, name


@pytest.mark.parametrize("case", ["guide-defaults", "guide-varied", "inline-default", "menger-sponge", "boxes-varied"] + SLIDER_CASES)
def test_far_field_value_is_the_outer_shape_bit_for_bit(tmp_path, case):
    rng = np.random.default_rng(20261017)
    if "/" in case:         # the settings-tab value sets: U as tabulated, the claim everywhere, no non-vacuity bar
        src, values, scene, name = _slider_case(case)
        exe = _build_harness(tmp_path, src, values)
        out = _run(exe, _points(rng, *slider_cases.region(scene, values)))
        sdf, A, U = out[:, 0], out[:, 1], out[:, 2]
        assert np.all(U.view(np.uint32) == U[0].view(np.uint32))
        assert U[0].view(np.uint32) == slider_cases.expected_U(scene, name).view(np.uint32), U[0]
        with np.errstate(invalid="ignore"):
            far = A > U[0]
        np.testing.assert_array_equal(sdf[far].view(np.uint32), A[far].view(np.uint32))
        return
    if case == "menger-sponge":
        src = scene_source("menger-sponge")
        values = {k: (v.data[0] if v.count == 1 else tuple(v.data)) for k, v in rm.default_custom_settings(src).items()}
        centre, radius, expect_U = (-0.5, -0.5, -0.5), 0.9, None
    elif case == "boxes-varied":
        src, values, centre, radius, expect_U = _boxes(), {"R": 0.8, "s0": 0.41}, (-0.5, -0.5, -0.5), 1.4, None
    elif case == "inline-default":
        src, values, centre, radius = scene_source("inline-default"), {}, (0, 0, 0), 5.0
        expect_U = np.float32(0.21) * np.float32(3.0)
    else:
        src = scene_source("guide")
        values = {k: (v.data[0] if v.count == 1 else tuple(v.data)) for k, v in rm.default_custom_settings(src).items()}
        values = {k: v for k, v in values.items() if k in ("bigSphereSize", "fractalIterations", "gridScaleFactor", "bigSphereCenter", "fractalColor")}
        expect_U = np.float32(0.21) * np.float32(3.0)
        if case == "guide-varied":
            values.update(bigSphereSize=2.37, fractalIterations=5.0, gridScaleFactor=0.41, bigSphereCenter=(1.5, -0.25, 3.0))
            expect_U = None
        centre, radius = values["bigSphereCenter"], values["bigSphereSize"]
    exe = _build_harness(tmp_path, src, values)
    pts = _points(rng, centre, radius)
    out = _run(exe, pts)
    sdf, A, U = out[:, 0], out[:, 1], out[:, 2]
    assert np.all(U == U[0]) and np.isfinite(U[0])
    if expect_U is not None:
        assert U[0] == expect_U                                   # 0.21 * sf of the coarsest grid (sf = 1/gridScaleFactor)
    with np.errstate(invalid="ignore"):
        far = A > U[0]
    # the claim
    np.testing.assert_array_equal(sdf[far].view(np.uint32), A[far].view(np.uint32))
    # and it is not vacuous: both sides of the bound are well populated, the near side really differs
    assert far.sum() > 50000 and (~far).sum() > 50000
    near_differs = (sdf[~far].view(np.uint32) != A[~far].view(np.uint32)).mean()
    # (spheres carved out of a sphere change most of the near field; the sponge's holes only the inside of its cube)
    assert near_differs > (0.05 if case in ("menger-sponge", "boxes-varied") else 0.2)
    # non-finite positions included
    assert np.isinf(A[far]).any()


# ---- guard-free floor at the bounded repetition sites (lower_glsl.cpp pass 2, glsl_rt.h "bounded-floor sites") ----
# The march kernels evaluate floor() of `mod(position + H1, S)` as (q +RD 1.5*2^23) - 1.5*2^23 with no range test
# once max|position| <= rm_floor_plim().  Checked here on the lowered text, on the CPU: the same g++ harness with
# rm_rep_b overridden by that arithmetic (round-down add through fesetround) must reproduce sdf() bit for bit at
# every position inside the limit, and every floor argument it sees there must lie within 2^22.
NF_HARNESS = r"""
#include <cfenv>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <vector>
#define GLSL_NS xg
#define GLSL_FAST 0
#include "glsl_rt.h"
namespace xg {
%(uniforms)s
static float fadd_rd(float a, float b) {
    volatile float x = a, y = b;
    const int old = fegetround();
    fesetround(FE_DOWNWARD);
    volatile float r = x + y;
    fesetround(old);
    return r;
}
static float g_max_q = 0.0f;
template <bool NF>
struct FragT {
    vec2 texcoord;
    ivec2 rm_texSize;
    template <class V> static float rm_len0(const V&) { return 0.0f; }
    float rm_box0(const vec3& b) { return -max(0.0f, max(b.x, max(b.y, b.z))); }
    float sdBox(vec3 p, vec3 b) { vec3 q = abs(p) - b; return length(max(q, 0.0f)) + min(max(q.x, max(q.y, q.z)), 0.0f); }
    float sdfSphere(vec3 position, vec3 center, float radius) { return distance(position, center) - radius; }
    static float floor_nf(float q, float h2) {
        const float M = 12582912.0f;
        if (std::fabs(q) > g_max_q) g_max_q = std::fabs(q);
        float r = fadd_rd(q, M) + (-M);
        if (!(h2 != 0.0f) || !(h2 == h2)) { uint32_t rb, qb; memcpy(&rb, &r, 4); memcpy(&qb, &q, 4); rb |= qb & 0x80000000u; memcpy(&r, &rb, 4); }
        return r;
    }
    static float rep1_nf(float x, float h1, float s, float h2) {
        const float a = g_add(x, h1);
        return g_sub(g_fma(-s, floor_nf(g_mul(a, g_rcp(s)), h2), a), h2);
    }
    template <class H1, class S, class H2> vec3 rm_rep_b(const vec3& x, const H1& h1, const S& s, const H2& h2) {
        if (!NF) return rm_rep(x, h1, s, h2);
        return vec3(rep1_nf(x.x, rm_c(h1, 0), rm_c(s, 0), rm_c(h2, 0)), rep1_nf(x.y, rm_c(h1, 1), rm_c(s, 1), rm_c(h2, 1)),
                    rep1_nf(x.z, rm_c(h1, 2), rm_c(s, 2), rm_c(h2, 2)));
    }
%(scene)s
};
}
int main(int argc, char** argv) {
    // stdin: n, then n * 3 floats; stdout: n * 3 floats (sdf guarded, sdf with the guard-free floor, plim) + max |q| seen inside the limit
    uint32_t n = 0;
    if (fread(&n, 4, 1, stdin) != 1) return 2;
    std::vector<float> in(3 * (size_t)n), out(3 * (size_t)n + 1);
    if (fread(in.data(), 4, in.size(), stdin) != in.size()) return 2;
    xg::FragT<false> f;
    xg::FragT<true> g;
    f.texcoord = g.texcoord = xg::vec2(0.5f, 0.5f);
    f.rm_texSize = g.rm_texSize = xg::ivec2(1, 1);
    const float plim = f.rm_floor_plim();
    float max_q_inside = 0.0f;
    for (uint32_t i = 0; i < n; i++) {
        const xg::vec3 p(in[3 * i], in[3 * i + 1], in[3 * i + 2]);
        out[3 * i] = f.sdf(p);
        xg::g_max_q = 0.0f;
        out[3 * i + 1] = g.sdf(p);
        const bool inside = std::fmax(std::fmax(std::fabs(p.x), std::fabs(p.y)), std::fabs(p.z)) <= plim;
        if (inside && xg::g_max_q > max_q_inside) max_q_inside = xg::g_max_q;
        out[3 * i + 2] = plim;
    }
    out[3 * (size_t)n] = max_q_inside;
    fwrite(out.data(), 4, out.size(), stdout);
    return 0;
}
"""


def _build_nf_harness(tmp_path, src, values):
    tu = translation_unit(src)
    assert "#define RM_HAS_FLOOR_PLIM 1" in tu and "rm_rep_b(" in tu and "float rm_floor_plim()" in tu
    m = re.search(r'#line 1 "scene.glsl"\n(.*?)\n#line \d+ "raymarch_kernel.cuh"', tu, re.S)
    scene = m.group(1)
    decls = re.findall(r"^__constant__ (\w+) (\w+);$", tu, re.M)
    uniforms = "".join("static %s %s = %s;\n" % (t, nme, _cxx_value(values[nme])) for t, nme in decls if nme in values)
    cpp = tmp_path / "nf_harness.cpp"
    cpp.write_text(NF_HARNESS % {"uniforms": uniforms, "scene": scene})
    exe = tmp_path / "nf_harness"
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-frounding-math", "-mfma", "-Wno-unknown-pragmas", "-I", str(DEVICE_SRC),
                    str(cpp), "-o", str(exe)], check=True)
    return exe


@pytest.mark.parametrize("case", ["guide-defaults", "guide-varied", "guide-tiny-cells", "inline-default"] + SLIDER_CASES)
def test_guard_free_floor_is_floorf_inside_the_proven_range(tmp_path, case):
    rng = np.random.default_rng(7)
    scene = None
    if "/" in case:
        src, values, scene, _name = _slider_case(case)
        centre, radius = slider_cases.region(scene, values)
    elif case == "inline-default":
        src, values, centre, radius = scene_source("inline-default"), {}, (0, 0, 0), 5.0
    else:
        src = scene_source("guide")
        values = {k: (v.data[0] if v.count == 1 else tuple(v.data)) for k, v in rm.default_custom_settings(src).items()}
        if case == "guide-varied":
            values.update(bigSphereSize=2.37, fractalIterations=5.0, gridScaleFactor=0.41, bigSphereCenter=(1.5, -0.25, 3.0))
        if case == "guide-tiny-cells":       # the finest grid is 0.2^13 ~ 8e-10: the limit drops to ~0.003 and most positions fall outside
            values.update(fractalIterations=13.0, gridScaleFactor=0.2)
        centre, radius = values["bigSphereCenter"], values["bigSphereSize"]
    exe = _build_nf_harness(tmp_path, src, values)
    pts = _points(rng, centre, radius)
    # plus positions on and around cell boundaries, negative zero and tiny negatives (the floor's own edge cases)
    if scene is None:
        cells = (rng.integers(-40, 40, (20000, 3)) * np.float32(1.0 / 3.0) ** rng.integers(0, 8, (20000, 1))).astype(np.float32)
        cells = np.concatenate([cells, np.nextafter(cells, np.float32(-np.inf)), np.nextafter(cells, np.float32(np.inf)), -cells])
    else:                   # the case's own cell sizes, and the band where the proven range ends
        cells = np.concatenate([slider_cases.cell_points(rng, scene, values), slider_cases.band_points(rng)])
    edge = np.array([[-0.0, -0.0, -0.0], [-1e-45, 1e-45, -1e-40], [-0.5, -0.5, -0.5], [-1.5, -0.16666667, -0.055555556]], np.float32)
    pts = np.ascontiguousarray(np.concatenate([pts, cells, edge]).astype(np.float32))
    blob = np.uint32(len(pts)).tobytes() + pts.tobytes()
    r = subprocess.run([str(exe)], input=blob, stdout=subprocess.PIPE, check=True)
    raw = np.frombuffer(r.stdout, np.float32)
    out, max_q = raw[:-1].reshape(-1, 3), raw[-1]
    plim = out[0, 2]
    with np.errstate(invalid="ignore"):
        inside = np.nanmax(np.abs(pts), axis=1) <= plim
    inside &= ~np.isnan(pts).all(axis=1)
    if scene is not None:   # a NaN or zero cell gives -1 (never fast), a loop that does not run 3e38
        assert plim == -1.0 or (np.isfinite(plim) and plim > 0), plim
    else:
        assert np.isfinite(plim) and plim > 0
        if case != "guide-tiny-cells":
            assert inside.sum() > 200000
        assert inside.sum() > 1000 and (~inside).sum() > 1000
    np.testing.assert_array_equal(out[inside, 0].view(np.uint32), out[inside, 1].view(np.uint32))
    assert max_q <= 4194304.0
    # not vacuous: where the limit is smaller than the carved sphere the guard-free floor really goes wrong outside it
    # (with the default cells the limit is ~600 units: everything beyond is far field, whose value is the outer shape)
    if case == "guide-tiny-cells":
        o = ~inside & np.isfinite(pts).all(axis=1)
        assert (out[o, 0].view(np.uint32) != out[o, 1].view(np.uint32)).any()
