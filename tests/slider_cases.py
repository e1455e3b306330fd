"""Named custom-uniform value sets of the bundled scenes: the settings-tab sliders away from their annotation defaults.

Shared by tests/test_carve_cpu.py (lowered text on the host) and tests/test_slider_values_gpu.py (device against the
oracle).  Each case overrides some of the scene's @default values.  For the carved scenes (far-field shortcut,
lower_glsl.cpp pass 1b) a case also carries

  U    the value rm_carve_bound() folds to: 0.21 * the coarsest cell for the guide grids (sf = 1 / gridScaleFactor
       at i = -1, whatever the iteration count), -9999.9 when the loop does not run at all or every cell is NaN
       (the scene's min() drops NaN operands), +inf for gridScaleFactor = 0 (pow(0, -1)); for the sponge the
       largest half-extent of its coarsest box triple (1.51 / 3), -3e38 when the loop does not run;
  far  whether the shortcut applies to some of the rays of a frame from the default camera (False where U is +inf,
       where the outer shape is -inf everywhere: bigSphereSize = +inf, and where the camera sits so deep inside the
       big sphere that no ray leaves it within its steps).

The last three guide cases lie outside the annotations' ranges but are reachable through set_uniforms and a
schema's customShaderParameters.
"""
import math

import numpy as np

PI = float(np.float32(math.pi))

# scene -> case name -> (overrides, U, far);  U and far are None for scenes without the shortcut
CASES = {
    "guide": {
        "iterations-0": ({"fractalIterations": 0.0}, 0.63, True),
        "iterations-1": ({"fractalIterations": 1.0}, 0.63, True),
        "iterations-2.5": ({"fractalIterations": 2.5}, 0.63, True),
        "iterations-20": ({"fractalIterations": 20.0}, 0.63, True),
        "grid-1": ({"gridScaleFactor": 1.0}, 0.21, True),
        "grid-0.9": ({"gridScaleFactor": 0.9}, 0.23333333, True),
        "grid-0.5-iterations-12": ({"gridScaleFactor": 0.5, "fractalIterations": 12.0}, 0.42, True),
        "grid-0": ({"gridScaleFactor": 0.0}, math.inf, False),
        "size-0": ({"bigSphereSize": 0.0}, 0.63, True),
        "size-30": ({"bigSphereSize": 30.0}, 0.63, False),                 # the camera at the origin is inside the
        # sphere in these two cases: no ray leaves it within its steps
        "size-negative": ({"bigSphereSize": -2.0}, 0.63, True),
        "centre-moved": ({"bigSphereCenter": (1.5, -0.25, 3.0)}, 0.63, False),
        "colour": ({"fractalColor": (1.0, 0.0, 0.25)}, 0.63, True),
        # outside the annotations
        "iterations-negative": ({"fractalIterations": -1.0}, -9999.9, True),
        "grid-nan": ({"gridScaleFactor": math.nan}, -9999.9, True),       # min() drops the NaN cells
        "size-inf": ({"bigSphereSize": math.inf}, 0.63, False),
    },
    "fractal1": {
        "grid-0.9": ({"gridScaleFactor": 0.9}, 0.23333333, True),
        "grid-0": ({"gridScaleFactor": 0.0}, math.inf, False),
        "iterations-0": ({"fractalIterations": 0.0}, 0.63, True),
        "iterations-20": ({"fractalIterations": 20.0}, 0.63, True),
    },
    "menger-sponge": {
        "iterations-0": ({"fractalIterations": 0.0}, -3.0e38, True),
        "iterations-1": ({"fractalIterations": 1.0}, -3.0e38, True),
        "iterations-2": ({"fractalIterations": 2.0}, 0.50333333, True),
        "iterations-3.5": ({"fractalIterations": 3.5}, 0.50333333, True),
        "iterations-20": ({"fractalIterations": 20.0}, 0.50333333, True),
    },
    "mandelbulb": {
        "power-2": ({"power": 2.0}, None, None),
        "power-3.5": ({"power": 3.5}, None, None),
        "power-16": ({"power": 16.0}, None, None),
        "bailout-1": ({"bailout": 1.0}, None, None),
        "bailout-8": ({"bailout": 8.0}, None, None),
        "iterations-1": ({"maxIterations": 1.0}, None, None),
        "iterations-32": ({"maxIterations": 32.0}, None, None),
    },
}

_TREE = {
    "iterations-0": ({"fractalIterations": 0.0}, None, None),
    "iterations-1": ({"fractalIterations": 1.0}, None, None),
    "iterations-20": ({"fractalIterations": 20.0}, None, None),
    "scale-0": ({"scaleFactor": 0.0}, None, None),
    "scale-1": ({"scaleFactor": 1.0}, None, None),
    "scale-1.5": ({"scaleFactor": 1.5}, None, None),
    "angles-0": ({"angles": (0.0, 0.0, 0.0)}, None, None),
    "angles-pi": ({"angles": (PI, PI / 2, -PI)}, None, None),
    "offset-0": ({"offset": 0.0}, None, None),
}
CASES["tree"] = dict(_TREE)
CASES["smooth-tree"] = dict(_TREE, **{"smoothen-0": ({"smoothen": 0}, None, None)})
CASES["rotation-fractal"] = dict(_TREE, **{"iterations-7.5": ({"fractalIterations": 7.5}, None, None)})   # its round()

CARVED = ("guide", "fractal1", "menger-sponge")


def all_cases(scenes=None):
    """[(scene, case name)] in table order"""
    return [(s, c) for s in CASES if scenes is None or s in scenes for c in CASES[s]]


def custom(rm, src, scene, case):
    """the scene's @default custom uniforms (UniformData) with the case's overrides applied"""
    from raymarching_engine_b200.uniform_types import UniformData
    values = dict(rm.default_custom_settings(src))
    for name, v in CASES[scene][case][0].items():
        d = values[name]
        data = tuple(v) if isinstance(v, tuple) else (v,)
        assert len(data) == d.count, (scene, case, name)
        values[name] = UniformData(d.type, d.count, tuple(int(x) for x in data) if d.type == "i" else data)
    return values


def plain(custom_values):
    """UniformData dict -> name -> float or tuple (the form the host harnesses take)"""
    return {k: (v.data[0] if v.count == 1 else tuple(v.data)) for k, v in custom_values.items()}


def expected_U(scene, case):
    """the table's U as float32, or None"""
    U = CASES[scene][case][1]
    return None if U is None else np.float32(U)


def region(scene, values):
    """(centre, radius) around which a scene's shape lies, for the near-field point sets"""
    if scene in ("guide", "fractal1"):
        r = float(values["bigSphereSize"])
        return tuple(values["bigSphereCenter"]), (min(abs(r), 30.0) if math.isfinite(r) and r != 0.0 else 4.0)
    if scene == "menger-sponge":
        return (-0.5, -0.5, -0.5), 0.9
    if scene == "mandelbulb":
        return (0.0, 0.0, 0.0), 1.5
    return (0.0, 0.0, 0.0), 4.0


def cell_points(rng, scene, values, n=20000):
    """positions on and one ulp either side of the cell boundaries of the scene's repetition grids (multiples of half
    a cell of every level), and their negations; grids other than the guide's use the sponge's 1/3 levels"""
    g = float(values["gridScaleFactor"]) if scene in ("guide", "fractal1") else 1.0 / 3.0
    if not 0.0 < g < 1.0:
        g = 1.0 / 3.0
    sizes = np.float32(g) ** np.arange(-1, 21, dtype=np.float32)
    cells = (rng.integers(-80, 80, (n, 3)) * sizes[rng.integers(0, len(sizes), (n, 1))] * np.float32(0.5)).astype(np.float32)
    return np.concatenate([cells, np.nextafter(cells, np.float32(-np.inf)), np.nextafter(cells, np.float32(np.inf)), -cells])


def band_points(rng, n=20000):
    """positions whose largest |coordinate| is log-uniform in [1e3, 1e8]: where the guard-free floor's proven range
    (rm_floor_plim) ends for every table case"""
    d = rng.normal(size=(n, 3))
    d /= np.abs(d).max(axis=1, keepdims=True)
    return (d * 10.0 ** rng.uniform(3.0, 8.0, (n, 1))).astype(np.float32)
