"""Edge cases of the far-field step loop (farRun: the camera rays' approach in the setup kernel, the far pass and the
march kernel's last-pass retire block) against the one-thread-per-pixel megakernel, which steps every ray through the
plain march loop.  Every case renders the same job on the wavefront pipeline with the scene's custom uniforms baked
(the bound U folds to a literal), on the wavefront pipeline with them dynamic (U is evaluated on the device) and on the
megakernel, and requires the same accumulators, bytes and SDF-evaluation counts from all three.

The cases are where the loop leaves its common step: trip counts of 0, 1, 2 and around the ~35 steps a sky ray takes
to freeze at 1e11 (so that some rays freeze in their last allowed step or run out one step before it), bounds U below
the 1e-4 stepsTaken threshold, directions with subnormal and zero components, and full mode, where castRay's far steps
run until the escaping rays overflow.
"""
import math

import numpy as np
import pytest

import raymarching_engine_b200 as rm
from conftest import scene_source
from raymarching_engine_b200.schema import IDENTITY4, Orthographic
from raymarching_engine_b200.uniform_types import UniformData

pytestmark = pytest.mark.gpu

PLANES = ("color", "normalAndDofRadius", "albedoAndDepth", "depth")
_FRAME = [860000]


@pytest.fixture(scope="module")
def contexts(ctx):
    gen = rm.load_render_job_context(device=0, specialize=False)
    mega = rm.load_render_job_context(device=0, pipeline="megakernel")
    if gen is None or mega is None:
        pytest.fail("no CUDA context: " + rm.context_error())
    yield {"baked": ctx, "dynamic": gen, "megakernel": mega}
    gen.close()
    mega.close()


def _custom(src, overrides):
    values = dict(rm.default_custom_settings(src))
    for name, v in overrides.items():
        d = values[name]
        values[name] = UniformData(d.type, d.count, (v,))
    return values


def _schema(scene, mode, W, H, steps=None, overrides=None, lights=1):
    src = scene_source(scene)
    s = rm.default_schema(src, _custom(src, overrides or {}), width=W, height=H, renderMode=mode)
    if steps is not None:
        s.reflectionIterationCounts = list(steps)
    if mode == "full":
        s.lights = [rm.default_light() for _ in range(lights)]
    return s


def _render(c, schema):
    _FRAME[0] += 1
    schema.render.frameid = _FRAME[0]
    rm.reset_halton()
    c.counters3(reset=True)
    fb = c.fbo.create(schema.render.width, schema.render.height, schema.render.frameid)
    got = rm.run_job(schema, c)
    assert got["success"], got["why"]
    out = {p: fb.read(p) for p in PLANES} | {"rgba8": got["rgba8"].copy()}
    return out, c.counters3(reset=True)


def _bits(a):
    return a.view(np.uint32) if a.dtype == np.float32 else a


def _check(contexts, make_schema, far_expected=True):
    """renders make_schema() on every context; returns the wavefront's (evaluations, pixels, far-field evaluations)"""
    ref, ref_counts = _render(contexts["megakernel"], make_schema())
    for name in ("baked", "dynamic"):
        got, counts = _render(contexts[name], make_schema())
        for p in PLANES:
            np.testing.assert_array_equal(_bits(got[p]), _bits(ref[p]), err_msg=f"{name} {p}")
        np.testing.assert_array_equal(got["rgba8"], ref["rgba8"], err_msg=f"{name} rgba8")
        assert counts[:2] == ref_counts[:2], (name, counts, ref_counts)
        if far_expected:
            assert counts[2] > 0, (name, counts)
    return counts


@pytest.mark.parametrize("steps", [0, 1, 2, 2.5, 3, 31, 33, 34, 35, 36, 37, 38, 40])
def test_preview_trip_counts(contexts, steps):
    _check(contexts, lambda: _schema("guide", "preview", 160, 90, steps=[steps]), far_expected=steps > 0)


@pytest.mark.parametrize("steps", [[1], [2], [3, 2], [36, 1], [128, 128], [160]])
def test_full_trip_counts_and_overflow(contexts, steps):
    """castRay has no freeze: a sky ray doubles its distance until length() overflows (~125 steps), then goes on
    with +inf / NaN positions"""
    _check(contexts, lambda: _schema("guide", "full", 64, 36, steps=steps))


@pytest.mark.parametrize("mode", ["preview", "full"])
@pytest.mark.parametrize("overrides", [{"fractalIterations": -1.0}, {"gridScaleFactor": math.nan}],
                         ids=["no-level", "nan-cells"])
def test_bound_below_stepstaken_threshold(contexts, overrides, mode):
    """U = -9999.9 < 1e-4 (no fractal level runs, or every cell is NaN and min() drops it): a far-field step with
    a <= 1e-4 must leave stepsTaken alone.  The whole scene is then the outer sphere, so rays also reach their fixed
    point on its surface inside the far field."""
    _check(contexts, lambda: _schema("guide", mode, 96, 54, overrides=overrides))


@pytest.mark.parametrize("mode", ["preview", "full"])
@pytest.mark.parametrize("column", [(1e-39, -0.0, 1.0), (-2e-38, 1e-45, -1.0), (0.0, 0.0, 1.0)],
                         ids=["subnormal-x-negzero-y", "subnormal-xy-backwards", "zero-xy"])
def test_subnormal_and_zero_direction_components(contexts, column, mode):
    """An orthographic camera sends every primary ray along the rotation's third column (normalised): components of
    d and of d * s that are subnormal or zero"""
    def make():
        s = _schema("guide", mode, 96, 54)
        s.camera.mode = Orthographic(12.0)
        s.camera.position = (0.0, 0.0, 10.0 - 20.0 * column[2])
        rot = list(IDENTITY4)
        rot[8:11] = column
        s.camera.rotation = rot
        return s
    _check(contexts, make)


@pytest.mark.parametrize("mode", ["preview", "full"])
def test_pattern_b_scene(contexts, mode):
    """the sponge's outer shape is a box (rm_carve_outer of the other lowering pattern)"""
    _check(contexts, lambda: _schema("menger-sponge", mode, 96, 54, steps=[40, 36] if mode == "full" else [36]))
