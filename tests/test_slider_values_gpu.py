"""Every bundled scene against the CPU oracle at the settings-tab slider values of tests/slider_cases.py, in both program
variants: custom uniforms baked into the program (NVRTC folds them, U = rm_carve_bound() becomes a literal that can be
+inf) and dynamic (__constant__ memory, U and rm_floor_plim() evaluated on the device).

Per case: the probe kernel (sdf and the seven material functions) at near, far, overflowing, non-finite and tiny
positions, on and beside the cell boundaries and in the band where the guard-free floor's proven range ends; for the
carved scenes the march kernels' own evaluation (far-field shortcut, guard-free floor, sticky square-root guard and
their guarded fallbacks) against the guarded sdf; a preview and a full-mode frame against the oracle, bit for bit.
Then the queue extremes of the far-field pipeline at the benchmark's 1080p size, and a slider drag through the
pipelined render_frames with specialize="auto".
"""
import ctypes as C

import numpy as np
import pytest

import bench
import pyoracle
import raymarching_engine_b200 as rm
import slider_cases
from conftest import scene_source
from raymarching_engine_b200 import executor as ex
from test_parity_gpu import _canon, _carve_points

pytestmark = pytest.mark.gpu

_FRAME = [740000]
PLANES = ("color", "normalAndDofRadius", "albedoAndDepth", "depth")


@pytest.fixture(scope="module")
def dyn_ctx():
    """a context whose jobs always run on the dynamic variant"""
    c = rm.load_render_job_context(device=0, specialize=False)
    if c is None:
        pytest.fail("no CUDA context: " + rm.context_error())
    yield c
    c.close()


def _diff(label, got, want):
    """None, or a line naming how many entries differ and the first of them (NaN payloads canonicalised)"""
    bad = _canon(got) != _canon(want) if got.dtype == np.float32 else got != want
    if not bad.any():
        return None
    i = tuple(np.argwhere(bad)[0])
    return f"{label}: {int(bad.sum())} of {bad.size} differ, first at {i}: {got[i]!r} vs {want[i]!r}"


def _probe(ctx, prog, pts):
    out = np.zeros((len(pts), 17), np.float32)
    st = rm._lib.lib.rmb_probe(ctx.handle, prog.handle, pts.ctypes.data_as(C.c_void_p), len(pts), out.ctypes.data_as(C.c_void_p))
    assert st == 0, ctx.last_error()
    return out


def _frame(c, schema):
    """render one job on context c: the four accumulator planes and the RGBA8, copied"""
    _FRAME[0] += 1
    schema.render.frameid = _FRAME[0]
    rm.reset_halton()
    fb = c.fbo.create(schema.render.width, schema.render.height, schema.render.frameid)
    got = rm.run_job(schema, c)
    assert got["success"], got["why"]
    return {p: fb.read(p) for p in PLANES} | {"rgba8": got["rgba8"].copy()}


def _oracle_frame(scene, schema, halton_start=0):
    acc, want = pyoracle.run_job(scene, schema, halton_start=halton_start)
    return {"color": acc.color, "normalAndDofRadius": acc.nd, "albedoAndDepth": acc.ad, "depth": acc.depth, "rgba8": want}


def _frame_diffs(label, got, want):
    return [d for p in PLANES + ("rgba8",) if (d := _diff(f"{label} {p}", got[p], want[p])) is not None]


def _schemas(src, custom):
    pre = rm.default_schema(src, custom, width=96, height=54, renderMode="preview")
    full = rm.default_schema(src, custom, width=64, height=36, renderMode="full")
    full.lights = [rm.default_light()]
    return {"preview": pre, "full": full}


@pytest.mark.parametrize("scene,case", slider_cases.all_cases(), ids=["%s/%s" % sc for sc in slider_cases.all_cases()])
def test_slider_values_match_the_oracle(ctx, dyn_ctx, scene, case):
    src = scene_source(scene)
    custom = slider_cases.custom(rm, src, scene, case)
    values = slider_cases.plain(custom)
    carved = scene in slider_cases.CARVED
    problems = []

    # both variants of the case, finished with before the next case asks for its own (RMB_VARIANT_CAP per scene)
    baked = ctx.program_cache.get_program(src, rm.FLAVOUR_EXACT, custom)
    dyn = ctx.program_cache.get_program(src, rm.FLAVOUR_EXACT, None)
    assert isinstance(baked, rm.Program), baked
    assert isinstance(dyn, rm.Program), dyn
    rm.set_uniforms(dyn, custom)
    variants = {"baked": baked, "dynamic": dyn}
    for name, prog in variants.items():          # a carved case cannot pass because the shortcut was dropped
        assert prog.has_carve() == carved, name

    rng = np.random.default_rng(20261020)
    pts = np.ascontiguousarray(np.concatenate([_carve_points(rng, *slider_cases.region(scene, values)),
                                               slider_cases.cell_points(rng, scene, values),
                                               slider_cases.band_points(rng)]).astype(np.float32))

    # probe: sdf and the material functions, all 17 outputs
    want = pyoracle.materials(scene, custom, pts)
    for name, prog in variants.items():
        if (d := _diff(f"probe {name}", _probe(ctx, prog, pts), want)) is not None:
            problems.append(d)

    # far field: the march kernels' evaluation is the guarded sdf everywhere; U as tabulated in both variants
    if carved:
        U_want = slider_cases.expected_U(scene, case)
        for name, prog in variants.items():
            out = ctx.probe_carve(prog, pts)
            via_march, U, guarded = out[:, 0], out[:, 2], out[:, 3]
            if (d := _diff(f"far field {name}: march evaluation vs guarded sdf", via_march, guarded)) is not None:
                problems.append(d + f" at position {pts[np.flatnonzero(_canon(via_march) != _canon(guarded))[0]]}")
            if not np.all(U.view(np.uint32) == U_want.view(np.uint32)):
                problems.append(f"far field {name}: U = {np.unique(U)} instead of {U_want!r}")

    # frames: baked against the oracle bit for bit, dynamic against baked; the far pass used where the table says
    far_evals = 0
    for mode, schema in _schemas(src, custom).items():
        ctx.counters3(reset=True)
        got = _frame(ctx, schema)
        far_evals += ctx.counters3(reset=True)[2]
        problems += _frame_diffs(f"{mode} frame baked vs oracle", got, _oracle_frame(scene, schema))
        problems += _frame_diffs(f"{mode} frame dynamic vs baked", _frame(dyn_ctx, schema), got)
    if carved:
        expect_far = slider_cases.CASES[scene][case][2]
        if (far_evals > 0) != expect_far:
            problems.append(f"far-field evaluations {far_evals}, expected {'some' if expect_far else 'none'}")

    assert not problems, "\n".join(problems)


@pytest.mark.parametrize("case", ["grid-0", "iterations-negative", "iterations-20"])
def test_far_field_queue_extremes_at_bench_size(ctx, case):
    """The bench's 1080p preview frame (pose 0) where the far pass never receives a ray (U = +inf), where every ray is
    parked as far field (U = -9999.9) and where the finest cells push most evaluations out of line (20 iterations)."""
    src = scene_source("guide")
    custom = slider_cases.custom(rm, src, "guide", case)
    s = bench.make_schema(rm, src, custom, 1920, 1080, "preview", 0, 0)
    ctx.counters3(reset=True)
    got = _frame(ctx, s)
    far = ctx.counters3(reset=True)[2]
    diffs = _frame_diffs("1080p frame vs oracle", got, _oracle_frame("guide", s))
    assert not diffs, "\n".join(diffs)
    assert (far == 0) if case == "grid-0" else (far > 0), far


def _drag_jobs():
    """about ten guide jobs: a slider moves on every job except a stretch of SPECIALIZE_AFTER + 1 held values"""
    src = scene_source("guide")
    base = rm.default_custom_settings(src)
    steps = [("gridScaleFactor", 0.34), ("gridScaleFactor", 0.36), ("bigSphereSize", 3.7)] + \
        [("bigSphereSize", 3.5)] * (ex.SPECIALIZE_AFTER + 1) + [("gridScaleFactor", 0.3), ("bigSphereSize", 4.2), ("gridScaleFactor", 0.5)]
    custom, jobs = dict(base), []
    for name, v in steps:
        custom = dict(custom, **{name: rm.u.float(v)})
        jobs.append(rm.default_schema(src, custom, width=96, height=54, renderMode="preview"))
    return jobs


@pytest.mark.parametrize("n_contexts", [1, 2])
def test_slider_drag_through_render_frames(n_contexts):
    """specialize="auto" while a slider is dragged: the moving jobs run on the dynamic variant, the held ones switch to a
    freshly baked variant, and the next move goes back - each uniform upload queued while the previous frame is still
    in flight.  Every frame equals the oracle's for its own values; job k draws Halton sample k."""
    contexts = [rm.load_render_job_context(device=0, specialize="auto") for _ in range(n_contexts)]
    try:
        assert all(c is not None for c in contexts), rm.context_error()
        jobs = _drag_jobs()
        for k, s in enumerate(jobs):
            s.render.frameid = 750000 + 100 * n_contexts + k
        want = [_oracle_frame("guide", s, halton_start=k) for k, s in enumerate(jobs)]
        ex.reset_specialization_history()
        rm.reset_halton()
        seen = []
        for i, r in rm.render_frames(jobs, contexts if n_contexts > 1 else contexts[0], depth=2):
            assert r["success"], r["why"]
            np.testing.assert_array_equal(r["rgba8"], want[i]["rgba8"], err_msg=f"job {i}")
            np.testing.assert_array_equal(_canon(r["depth"]), _canon(want[i]["depth"]), err_msg=f"job {i}")
            seen.append(i)
        assert seen == list(range(len(jobs)))
        for c in contexts:          # the held values did run on a baked variant
            assert any(key[2] is not None for key in c.program_cache._hits), "no baked variant was used"
    finally:
        ex.reset_specialization_history()
        for c in contexts:
            if c is not None:
                c.close()
