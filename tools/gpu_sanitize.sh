#!/bin/bash
# usage: bash tools/gpu_sanitize.sh [tag] : compute-sanitizer memcheck + racecheck over small preview + full renders through the
# public API, once per build / launch switch that changes which kernels or buffers are in play: defaults, RMB_CARVE=0 (no
# far-field pipeline), a multi-pass march plan with step budgets, a
# device group of two members on this GPU (tile contexts, fused gather store, row scatter), and frame sizes that make the ray
# planes / record lists grow between draws.  Logs -> gpurun_out/sanitizer_<tag>_<case>_<tool>.log
TAG=${1:-r2}
O=gpurun_out; mkdir -p $O
cat > /tmp/san.py <<'PY'
import os, sys; sys.path.insert(0, ".")
os.environ.setdefault("RMB_SPECIALIZE", "always")
import raymarching_engine_b200 as rm
group = os.environ.get("SAN_GROUP") == "1"
ctx = rm.load_render_job_group([0, 0]) if group else rm.load_render_job_context(device=0)
assert ctx is not None
src = open("scenes/guide.glsl").read(); custom = rm.default_custom_settings(src)
fid = 0
for (W, H) in ((40, 24), (77, 45), (130, 70), (64, 36)):       # growing, then shrinking: wf_reserve reallocates, pools reuse
    for mode in ("preview", "full"):
        fid += 1
        s = rm.default_schema(src, custom, width=W, height=H, renderMode=mode, samplesPerPixel=2, subdivisions=2 if W == 77 else 1, frameid=fid)
        if mode == "full":
            s.lights = [rm.default_light()]; s.dof.amount = 0.05
            s.reflectionIterationCounts = [48, 32, 16]
        r = rm.run_job(s, ctx); assert r["success"], r["why"]
if not group:
    sg = open("scenes/sphere-grid.glsl").read()      # a scene without the far-field shortcut
    s = rm.default_schema(sg, rm.default_custom_settings(sg), width=64, height=36, renderMode="preview", frameid=99)
    r = rm.run_job(s, ctx); assert r["success"], r["why"]
ctx.close(); print("sanitize run ok")
PY
run() {   # name, env...
  name=$1; shift
  for tool in memcheck racecheck; do
    env "$@" compute-sanitizer --tool $tool --error-exitcode 9 python /tmp/san.py > $O/sanitizer_${TAG}_${name}_${tool}.log 2>&1
    echo "$name $tool rc=$? : $(grep -E 'ERROR SUMMARY|RACECHECK SUMMARY' $O/sanitizer_${TAG}_${name}_${tool}.log | tail -1) $(grep -c 'sanitize run ok' $O/sanitizer_${TAG}_${name}_${tool}.log) ok-line(s)"
  done
}
run defaults SAN_X=0
run no_carve RMB_CARVE=0
run plan_budget RMB_MARCH_PLAN=24:256:2:8,0:128:1:0
run group2 SAN_GROUP=1
