"""Host-side mirror of the reference's TypeScript renderer: Halton, parameter annotations, uniform
derivations, row-tile sharding arithmetic (no GPU needed)."""
import itertools
import math

import numpy as np
import pytest

import pyoracle
import raymarching_engine_b200 as rm
from raymarching_engine_b200 import sharding
from conftest import SCENES, scene_source, ROOT


def test_halton_matches_oracle_and_known_values():
    for b in (2, 3, 5):
        got = list(itertools.islice(rm.halton(b), 200))
        assert got == pyoracle.halton_seq(b, 200)
    assert list(itertools.islice(rm.halton(2), 4)) == [0.5, 0.25, 0.75, 0.125]


def test_guide_defaults_from_annotations():
    # SURVEY.md 8c: bigSphereSize=4, fractalColor=(.5,.5,.5), fractalIterations=8, gridScaleFactor=0.33333333333, bigSphereCenter=(0,0,10)
    d = rm.default_custom_settings(scene_source("guide"))
    assert d["bigSphereSize"] == rm.u.float(4.0)
    assert d["fractalColor"] == rm.u.vec3(0.5, 0.5, 0.5)
    assert d["fractalIterations"] == rm.u.float(8.0)
    assert d["gridScaleFactor"] == rm.u.float(0.33333333333)
    assert d["bigSphereCenter"] == rm.u.vec3(0.0, 0.0, 10.0)
    assert rm.default_custom_settings(scene_source("smooth-tree"))["smoothen"] == rm.UniformData("i", 1, (1,))


def test_annotation_parser_records_metadata_and_errors():
    src = """uniform vec3 tint;
//@name="Tint colour" @format=color/bogus @default=1,2
uniform float gain; /* @min=0 @max=abc @scale=log @step=0.5 */
//@tooltip="how \\"bright\\"" @sensitivity=0.01 @default=2.5
float sdf(vec3 p) { return 1.0; }
"""
    ps = rm.get_custom_shader_params(src)
    ok = [p for p in ps if p.success]
    errs = [p for p in ps if not p.success]
    assert [p.internalName for p in ok] == ["tint", "gain"]
    assert ok[0].name == "Tint colour" and ok[0].formats == ["color"] and ok[0].quantity == 3
    assert ok[1].min == 0 and ok[1].scale == "log" and ok[1].step == 0.5 and ok[1].defaultValue == [2.5]
    reasons = " | ".join(e.reason for e in errs)
    assert "Unknown input format 'bogus'" in reasons
    assert "requires 3 default values, but 2 were supplied" in reasons
    assert "Expected property 'max' to be a number" in reasons


# sha256 of the reference's example scenes (client/public/examples/*.glsl, client/dist/examples/sphere-grid.glsl):
# the bundled copies are byte-identical (scenes/README.md), so the annotation parser and the lowering are
# tested on the reference's own text
REFERENCE_SCENE_SHA256 = {
    "guide": "0f2900dd06904709fce54c84f1e3b7a098a185c5041fd45cef6612b4e3014c37",
    "sphere-grid": "63d2ec34eba260e1821923851bb3ba50d6e05f9655f0a953a429b0ad79b57de1",
    "fractal1": "53e424a43cf768007b725870052f71ecf858fc4f2cd763356bb45f3b0df09b92",
    "menger-sponge": "ba317b8e6f4443fa83f72edf62d8e993bde6fdf3339890cc682024a94edd0d8e",
    "rotation-fractal": "870ca32c26b5afb4f80ae35213aa974cb22537a9063ae1ae150183bec5f068ba",
    "smooth-tree": "31b672f0b6182fdfed8ddb67a84b0ff5228d1c635595ade1628e46e2584ad1d5",
    "tree": "5e4cdbbef90d34b558cdeddaa729b176b6718bbe0c69e008210dccb0c346b92b",
}


@pytest.mark.parametrize("name", sorted(REFERENCE_SCENE_SHA256))
def test_bundled_scenes_are_verbatim(name):
    import hashlib
    for d in (ROOT / "scenes", ROOT / "tests" / "fixtures" / "scenes"):
        if (d / f"{name}.glsl").exists():
            data = (d / f"{name}.glsl").read_bytes()
    assert hashlib.sha256(data).hexdigest() == REFERENCE_SCENE_SHA256[name]


@pytest.mark.parametrize("name", sorted(REFERENCE_SCENE_SHA256))
def test_annotation_parser_on_the_reference_text(name):
    """(f1) on the verbatim reference scenes: every declared uniform parses without an error record and
    gets a default of the right arity (CustomShaderParamParser.tsx:91-165)."""
    src = scene_source(name)
    ps = rm.get_custom_shader_params(src)
    assert all(p.success for p in ps), [p.reason for p in ps if not p.success]
    d = rm.default_custom_settings(src)
    declared = [ln.split()[2].rstrip(";") for ln in src.splitlines() if ln.startswith("uniform ")]
    assert sorted(d) == sorted(declared)


def test_builtin_uniform_derivations():
    # RenderJobExecutor.tsx:212-264
    s = rm.default_schema("float sdf(vec3 p){return 1.0;}", {}, width=1920, height=1080, samplesPerPixel=16, exposure=0.5)
    s.camera.mode = rm.Orthographic(7.5)
    s.lights = [rm.default_light(), rm.SunLight(direction=(0, 1, 0), color=(1, 1, 1))]
    u = rm.builtin_uniforms(s, (0.5, 1 / 3))
    assert u["exposure"].data == (0.5 / 16,)
    assert u["aspect"].data == (1920 / 1080,)
    assert u["cameraMode"].data == (1,) and u["fov"].data == (7.5,)
    assert u["reflections"].data == (5,) and u["raymarchingSteps"].data == (128,) and u["indirectLightingRaymarchingSteps"].data == (128,)
    assert u["renderMode"].data == (1,) and u["blendMode"].data == (1,) and u["lightCount"].data == (2,)
    assert u["randNoise"].data == (0.5, 1 / 3)
    s.camera.mode = rm.Panoramic()
    assert rm.builtin_uniforms(s, (0, 0))["fov"].data == (1,) and rm.builtin_uniforms(s, (0, 0))["cameraMode"].data == (2,)
    # the oracle-side restatement derives the same numbers
    U = pyoracle.uniforms_from_schema(s, (0.5, 1 / 3))
    assert U.exposure == np.float32(0.5 / 16) and U.aspect == np.float32(1920 / 1080) and U.cameraMode == 2 and U.lightCount == 2
    assert U.lightSizes[1] == 0.0 and tuple(U.lightPositions[3:6]) == (0.0, 1.0, 0.0)      # sun light -> point at `direction`, size 0


def test_default_light_colour():
    # index.tsx:174 with LightSettings.tsx:82-87 (rgb 255, strength 3)
    assert rm.default_light().color == (255 * 3 / 256,) * 3


def test_row_tile_ownership_arithmetic():
    for H, T, G in [(1080, 16, 8), (2160, 16, 8), (72, 16, 3), (50, 7, 4), (5, 16, 2), (16, 16, 1)]:
        rows = [sharding.owned_rows(H, T, G, r) for r in range(G)]
        assert (np.sort(np.concatenate(rows)) == np.arange(H)).all()
        for r in range(G):
            assert (rows[r] // T % G == r).all()
            for g in [0, 1, T - 1, T, T + 1, H // 2, H - 1, H, H + 9]:
                assert sharding.owned_rows_below(g, H, T, G, r) == int((rows[r] < g).sum())
    assert sharding.owned_rows_below(3, 10, 16, 2, 5) == -1


def test_orbit_path_pose_zero_is_the_reference_view():
    import bench
    pos, rot = bench.orbit_pose(0)
    assert pos == (0.0, 0.0, 0.0) and rot == rm.schema.IDENTITY4
    pos, rot = bench.orbit_pose(64)                       # quarter turn: camera at (10, 0, 10) looking along -x
    assert np.allclose(pos, (10, 0, 10)) and np.allclose((rot[8], rot[9], rot[10]), (-1, 0, 0), atol=1e-12)
    for k in (1, 37, 200):
        pos, rot = bench.orbit_pose(k)
        fwd = np.array([rot[8], rot[9], rot[10]])
        to_centre = np.array([0, 0, 10]) - np.array(pos)
        assert np.allclose(fwd, to_centre / np.linalg.norm(to_centre)) and abs(np.linalg.norm(to_centre) - 10) < 1e-9


def test_frame_uniform_block_carries_the_same_record_as_the_per_name_uploads():
    """rmb_uniforms_set_frame's POD block (executor.frame_uniforms) against builtin_uniforms + the array / matrix uploads of
    RenderJobExecutor.tsx:212-297, value by value after the float32 conversion both paths apply."""
    import ctypes as C
    from raymarching_engine_b200 import executor as ex
    src = scene_source("guide")
    f32 = lambda v: C.c_float(v).value                                    # noqa: E731
    for mode, cam in (("preview", rm.Perspective(1.5)), ("full", rm.Orthographic(2.25)), ("full", rm.Panoramic())):
        s = rm.default_schema(src, rm.default_custom_settings(src), width=640, height=360, renderMode=mode, samplesPerPixel=3,
                              blendMode="mix" if mode == "full" else "additive")
        s.camera.mode = cam
        s.camera.position = (0.1, -2.5, 3.75)
        s.camera.rotation = tuple(0.01 * k for k in range(16))
        s.dof.showFocusedArea = mode == "full"
        s.fogDensity = 0.125
        s.reflectionIterationCounts = [96, 48, 24]
        if mode == "full":
            s.lights = [rm.default_light(), rm.SunLight(direction=(0.0, -1.0, 0.5), color=(1.0, 0.5, 0.25))]
        noise = (0.625, 1.0 / 9.0)
        rec = ex.builtin_uniforms(s, noise)
        b = ex.frame_uniforms(s, noise)
        for name, u in rec.items():
            if name in ("previousColor", "previousNormalAndDofRadius", "previousAlbedoAndDepth"):
                continue                                                   # sampler units: constants inside the library
            got = getattr(b, name)
            got = list(got) if hasattr(got, "__len__") else [got]
            want = [f32(v) if u.type == "f" else int(v) for v in u.data]
            if any(isinstance(w, float) and math.isnan(w) for w in want):
                assert all(math.isnan(g) for g in got), name
            else:
                assert got == want, (name, got, want)
        assert list(b.rotation) == [f32(v) for v in s.camera.rotation]
        assert b.stepCountsLength == 3 and list(b.raymarchingStepCountsArray)[:3] == [96.0, 48.0, 24.0]
        assert b.lightCount == len(s.lights)
        for k, l in enumerate(s.lights):
            v = l.position if l.type == "point" else l.direction
            assert list(b.lightPositions)[3 * k:3 * k + 3] == [f32(x) for x in v]
            assert list(b.lightColors)[3 * k:3 * k + 3] == [f32(x) for x in l.color]
            assert b.lightSizes[k] == f32(l.size if l.type == "point" else 0)
