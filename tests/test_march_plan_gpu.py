"""Every march pass plan renders the oracle's frame with the same work.

A march stage of the wavefront pipeline runs as a sequence of passes of the persistent march kernel, described by the
plan RMB_MARCH_PLAN = "budget:threads:ctas_per_sm:pause[,...]" (rmb_api.cpp render_wavefront, DESIGN.md section 4).
Between two passes a ray travels as a 48-byte record; in a carved scene a far pass steps the parked rays in between.
How the work is split into passes changes nothing a ray computes, so for every plan and every case:

1. exact flavour: the four accumulator planes and the RGBA8 frame are the oracle's, bit for bit;
2. every flavour: the frame is bit-identical to the default plan's;
3. counter slot 0 (SDF evaluations, far-field steps included) and slot 1 (pixel-samples) equal the default plan's, and
   slot 0 equals the megakernel's (one thread per pixel, no passes): a lost ray lowers slot 0, a ray marched twice raises
   it, even where the image survives.  Slot 2 counts the far-field steps run outside the march loop (approach, far
   pass, last pass), which legitimately depends on the plan: it is only bounded by slot 0, and 0 without far field;
4. one draw launches exactly what the parsed and truncated plan implies (at most 4 passes for a carved program, 8
   otherwise; the last pass ignores its budget and pause).

The library reads RMB_MARCH_PLAN at every draw, so one context and one program per scene serve every plan.
"""
from dataclasses import dataclass
from typing import Optional

import numpy as np
import pytest

import pyoracle
import raymarching_engine_b200 as rm
from conftest import scene_source

pytestmark = pytest.mark.gpu

PLANES = ("color", "normalAndDofRadius", "albedoAndDepth", "depth")
CARVED_SCENES = ("guide", "menger-sponge")      # the scenes of this file whose programs take the far-field path


def _repeat(entry, n):
    return ",".join([entry] * (n - 1) + ["0:256:2:0"])


# (RMB_MARCH_PLAN, None = unset; march passes a program without / with the far-field pipeline runs; test id)
PLANS = [
    # the shipped plan below 4 M rays (0:256:2:8,0:256:1:0): the reference of invariants 2 and 3
    (None, 2, 2, "default"),
    # every live ray parked after one step and resumed once
    ("1:256:2:0,0:256:2:0", 2, 2, "budget1-2pass"),
    # four passes, the maximum for a carved program: three park / far pass / resume cycles
    ("1:256:2:0,1:256:2:0,1:256:2:0,0:256:2:0", 4, 4, "budget1-4pass"),
    # eight passes, the maximum without far field; a carved program keeps the first four (the last of them unbudgeted)
    (_repeat("2:256:2:0", 8), 8, 4, "budget2-8pass"),
    # ten entries: truncated to eight passes (four carved), the last pass kept ignores its budget
    (_repeat("2:256:2:0", 10), 8, 4, "budget2-10entries"),
    # budget at trips - 1, trips and trips + 1 of the 128-step preview march and of the first two castRay stages
    ("127:256:2:0,0:256:1:0", 2, 2, "budget127"),
    ("128:256:2:0,0:256:1:0", 2, 2, "budget128"),
    ("129:256:2:0,0:256:1:0", 2, 2, "budget129"),
    # the same edge for the 32-step bounces 3 and 4 of the default step counts [128, 128, 64, 32, 32] (full mode)
    ("31:256:2:0,0:256:1:0", 2, 2, "budget31"),
    ("32:256:2:0,0:256:1:0", 2, 2, "budget32"),
    ("33:256:2:0,0:256:1:0", 2, 2, "budget33"),
    # odd budgets; 64-, 96- and 32-thread CTAs (grid clamped to the draw's 32-ray chunks); a warp that runs dry hands
    # over everything it holds (31) and its last ray (1)
    ("7:64:1:31,13:96:4:1,0:32:1:0", 3, 3, "odd-shapes"),
    # 32 CTAs per SM, clamped to the useful grid on small draws
    ("0:256:32:0,0:32:1:0", 2, 2, "32ctas"),
    # the shipped plan above 4 M rays, on the small draws it never serves
    ("0:256:3:12,0:256:2:0", 2, 2, "large-draw-plan"),
    # the parser: no entry parses -> one pass of 256 threads x 2 CTAs per SM
    ("", 1, 1, "empty"),
    ("abc", 1, 1, "unparsable"),
    # empty entries are skipped; a single entry is the last pass, whose budget and pause are ignored
    (",,5:256:2:31", 1, 1, "empty-entries"),
    # threads clamped to 256, CTAs per SM to 1, pause to 31 (then ignored: last pass)
    ("5:1000:0:99", 1, 1, "clamp-high"),
    # negative budget / CTAs / pause clamped to 0 / 1 / 0, 31 threads rounded down and clamped to 32
    ("-3:31:-1:-1", 1, 1, "clamp-low"),
    # a lone budgeted entry with the largest hand-over threshold: both ignored
    ("50:256:2:31", 1, 1, "single-entry"),
]


@dataclass(frozen=True)
class Case:
    scene: str
    mode: str
    width: int
    height: int
    lights: int = 0
    spp: int = 1
    subdivisions: int = 1
    flavour: str = "exact"
    carve: bool = True          # False: the program is built with RMB_CARVE=0
    tile: bool = False          # True: rank 1 of 2, 16-row tiles

    @property
    def context_key(self):
        return (self.flavour, self.carve, self.tile)

    @property
    def oracle_key(self):
        """what the oracle frame depends on (not the flavour-independent pipeline switches)"""
        return (self.scene, self.mode, self.width, self.height, self.lights, self.spp, self.subdivisions)


CASES = {
    # preview: carve patterns A (guide) and B (menger-sponge), and two scenes without far field; 203x117 pads the
    # 8x4 ray tiles in both directions, 7x3 is less than one tile (21 rays, 11 padding lanes), 1x1 a single ray
    "guide-preview-203x117": Case("guide", "preview", 203, 117),
    "guide-preview-7x3": Case("guide", "preview", 7, 3),
    "guide-preview-1x1": Case("guide", "preview", 1, 1),
    "menger-sponge-preview-203x117": Case("menger-sponge", "preview", 203, 117),
    "menger-sponge-preview-7x3": Case("menger-sponge", "preview", 7, 3),
    "sphere-grid-preview-203x117": Case("sphere-grid", "preview", 203, 117),
    "sphere-grid-preview-1x1": Case("sphere-grid", "preview", 1, 1),
    # (the exact flavour's Mandelbulb loop is long: a small frame)
    "mandelbulb-preview-51x27": Case("mandelbulb", "preview", 51, 27),
    # full mode: 5 bounce stages plus a shadow stage per light and bounce, each a multi-pass march in one draw
    "guide-full-2lights-203x117": Case("guide", "full", 203, 117, lights=2),
    "guide-full-2lights-7x3": Case("guide", "full", 7, 3, lights=2),
    "guide-full-2lights-1x1": Case("guide", "full", 1, 1, lights=2),
    "tree-full-1light-203x117": Case("tree", "full", 203, 117, lights=1),
    # the same scene without the far-field pipeline: a program that may run 8 passes
    "guide-nocarve-preview-203x117": Case("guide", "preview", 203, 117, carve=False),
    "guide-nocarve-full-2lights-203x117": Case("guide", "full", 203, 117, lights=2, carve=False),
    # scissored draws (x0 != 0) accumulating into one frame
    "guide-preview-subdiv3-spp2-203x117": Case("guide", "preview", 203, 117, spp=2, subdivisions=3),
    # one rank of a row-tile split: the rays of the draw cover the rank's rows only
    "guide-preview-tile-rank1of2-160x90": Case("guide", "preview", 160, 90, tile=True),
    # fast flavour: no oracle; every plan must give the fast flavour's own default-plan frame
    "guide-fast-preview-203x117": Case("guide", "preview", 203, 117, flavour="fast"),
    "guide-fast-full-2lights-203x117": Case("guide", "full", 203, 117, lights=2, flavour="fast"),
}


def _schema(case: Case):
    src = scene_source(case.scene)
    s = rm.default_schema(src, rm.default_custom_settings(src), width=case.width, height=case.height, renderMode=case.mode,
                          samplesPerPixel=case.spp, subdivisions=case.subdivisions)
    s.lights = [rm.default_light() for _ in range(case.lights)]
    if case.lights > 1:
        s.lights[1].position = (1.0, 2.0, 3.0)
        s.lights[1].size = 0.3
    return s


def _canon(a):
    """fp32 array -> uint32 bit patterns with every NaN mapped to one pattern: x86 and sm_100 produce
    different default-NaN payloads (0xffc00000 vs 0x7fffffff), and GLSL does not define one"""
    bits = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32).copy()
    bits[np.isnan(a)] = 0x7fc00000
    return bits


def _diff(label, got, want):
    """None, or a line naming how many entries differ and the first of them (NaN payloads canonicalised)"""
    bad = _canon(got) != _canon(want) if got.dtype == np.float32 else got != want
    if not bad.any():
        return None
    i = tuple(int(x) for x in np.argwhere(bad)[0])
    return f"{label}: {int(bad.sum())} of {bad.size} differ, first at {i}: {got[i]!r} vs {want[i]!r}"


def _frame_diffs(label, got, want):
    """the five-plane bit-exact comparison: colour and depth with NaNs canonicalised, the half-float planes and RGBA8 as is"""
    return [d for p in PLANES + ("rgba8",) if (d := _diff(f"{label} {p}", got[p], want[p])) is not None]


# ---- contexts, programs and the per-case references (computed once, shared by every plan) ----------------------------

_CONTEXTS = {}
_ORACLE = {}
_DEFAULT = {}
_MEGAKERNEL = {}
_FRAME = [770000]


@pytest.fixture(scope="module")
def contexts(ctx):
    """one wavefront context per (flavour, RMB_CARVE, tiling): the suite's own for the exact flavour"""
    _CONTEXTS[("exact", True, False)] = ctx
    yield _CONTEXTS
    for c in list(_CONTEXTS.values()):
        if c is not ctx:
            c.close()
    _CONTEXTS.clear()


def _context(contexts, case: Case):
    c = contexts.get(case.context_key)
    if c is None:
        flavour = rm.FLAVOUR_FAST if case.flavour == "fast" else rm.FLAVOUR_EXACT
        c = rm.load_render_job_context(device=0, rank=1 if case.tile else 0, n_ranks=2 if case.tile else 1, tile_rows=16,
                                       flavour=flavour, specialize="always")
        assert c is not None, rm.context_error()
        contexts[case.context_key] = c
    return c


def _program(c, case: Case, schema):
    """the program run_job uses for this case (custom uniforms baked), built under the case's RMB_CARVE"""
    with pytest.MonkeyPatch.context() as mp:
        if case.carve:
            mp.delenv("RMB_CARVE", raising=False)
        else:
            mp.setenv("RMB_CARVE", "0")
        prog = c.program_cache.get_program(schema.sdfShaderSource, None, dict(schema.customShaderParameters))
    assert isinstance(prog, rm.Program), prog
    # a lowering change that un-carves a scene must fail here, not silently lose the phased path
    assert prog.has_carve() == (case.carve and case.scene in CARVED_SCENES)
    return prog


def _render(c, schema):
    """one job: the four accumulator planes (local rows), RGBA8, the rows drawn and counter slots 0-2"""
    _FRAME[0] += 1
    schema.render.frameid = _FRAME[0]
    rm.reset_halton()
    c.counters_all(reset=True)
    fb = c.fbo.create(schema.render.width, schema.render.height, schema.render.frameid)
    got = rm.run_job(schema, c)
    assert got["success"], got["why"]
    out = {p: fb.read(p) for p in PLANES} | {"rgba8": got["rgba8"].copy(), "rows": fb.global_rows()}
    out["counters"] = tuple(c.counters_all(reset=True)[:3])
    return out


def _draw_launches(c, prog, schema):
    """kernel launches of one full-frame rmb_render_sample draw"""
    _FRAME[0] += 1
    W, H = schema.render.width, schema.render.height
    fb = c.fbo.create(W, H, _FRAME[0])
    rm.upload_sample_uniforms(prog, schema, (0.5, 1.0 / 3.0))
    n0 = c.launch_count()
    assert c.render_sample(prog, fb, 0, 0, W, H) == 0, c.last_error()
    n = c.launch_count() - n0
    c.sync()
    c.fbo.delete(W, H, _FRAME[0])
    return n


def _expected_launches(schema, passes, carved):
    """setup, per march stage its passes (and a far pass between two passes of a carved program), the stage kernels"""
    stage = passes + (passes - 1 if carved else 0)
    if schema.render.renderMode == "preview":
        return 1 + stage + 1                                        # setup, march stage, shade
    bounces = min(len(schema.reflectionIterationCounts), 10)
    lights = min(len(schema.lights), 10)
    return 1 + bounces * (stage + 1 + lights * (stage + 1)) + 1     # setup, (cast, bounce, (shadow, light) x L) x B, final


def _oracle(case: Case):
    key = case.oracle_key
    if key not in _ORACLE:
        acc, want = pyoracle.run_job(case.scene, _schema(case))
        _ORACLE[key] = {"color": acc.color, "normalAndDofRadius": acc.nd, "albedoAndDepth": acc.ad, "depth": acc.depth,
                        "rgba8": want}
    return _ORACLE[key]


def _default_frame(c, case: Case):
    if case not in _DEFAULT:
        with pytest.MonkeyPatch.context() as mp:
            mp.delenv("RMB_MARCH_PLAN", raising=False)
            _DEFAULT[case] = _render(c, _schema(case))
    return _DEFAULT[case]


def _megakernel_evals(c, case: Case):
    """slot 0 of the same job through the megakernel: the switch load_render_job_context(pipeline="megakernel") sets,
    on the same context and program"""
    if case not in _MEGAKERNEL:
        assert rm._lib.lib.rmb_ctx_set_pipeline(c.handle, 1) == 0
        try:
            frame = _render(c, _schema(case))
        finally:
            rm._lib.lib.rmb_ctx_set_pipeline(c.handle, 0)
        _MEGAKERNEL[case] = frame["counters"]
    return _MEGAKERNEL[case]


# ---- the test ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", list(CASES.values()), ids=list(CASES))
@pytest.mark.parametrize("plan,passes_pure,passes_carved", [pytest.param(p, a, b, id=i) for p, a, b, i in PLANS])
def test_march_plan_renders_the_same_frame_with_the_same_work(contexts, monkeypatch, plan: Optional[str], passes_pure,
                                                               passes_carved, case):
    c = _context(contexts, case)
    schema = _schema(case)
    prog = _program(c, case, schema)
    carved = prog.has_carve()
    ref = _default_frame(c, case)

    if plan is None:
        monkeypatch.delenv("RMB_MARCH_PLAN", raising=False)
    else:
        monkeypatch.setenv("RMB_MARCH_PLAN", plan)
    got = _render(c, schema)
    problems = []

    # 1. exact flavour: the oracle's frame (the rows this context owns)
    if case.flavour == "exact":
        rows = got["rows"]
        want = {k: v[rows] for k, v in _oracle(case).items()}
        problems += _frame_diffs("vs oracle:", got, want)
    # 2. the default plan's frame
    problems += _frame_diffs("vs default plan:", got, ref)

    # 3. the same work
    evals, pixels, far = got["counters"]
    if (evals, pixels) != ref["counters"][:2]:
        problems.append(f"(evaluations, pixel-samples) = {(evals, pixels)}, default plan {ref['counters'][:2]}")
    if case.flavour == "exact":
        # (the fast flavour contracts differently in the megakernel's inlined copies of the scene: its rays may take
        # other steps there, so only the exact flavour has the megakernel's count)
        mega = _megakernel_evals(c, case)
        if (evals, pixels) != mega[:2]:
            problems.append(f"(evaluations, pixel-samples) = {(evals, pixels)}, megakernel {mega[:2]}")
    if far > evals:
        problems.append(f"far-field steps {far} > evaluations {evals}")
    if not carved and far != 0:
        problems.append(f"far-field steps {far} in a program without far field")

    # 4. the plan that ran
    passes = passes_carved if carved else passes_pure
    launches = _draw_launches(c, prog, schema)
    want_launches = _expected_launches(schema, passes, carved)
    if launches != want_launches:
        problems.append(f"one draw launched {launches} kernels, {passes} march passes per stage imply {want_launches}")

    assert not problems, "\n".join(problems)
