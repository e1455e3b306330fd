/* rmb.h -- C ABI of libraymarch_b200.so, the B200-native replacement for the WebGL2 layer under
 * radian628/raymarching-engine's render-job API (SURVEY.md section 8b).
 *
 * The reference's TypeScript host (the .tsx files of client/src/renderer) talks to the GPU only through a
 * WebGL2RenderingContext.  Each entry point below replaces one group of those calls; the
 * reference interface it stands in for is cited as file:line under /root/reference/client/src.
 * An N-API addon (INTEGRATION.md) maps these 1:1 into JavaScript; the tests drive the same
 * symbols through Python ctypes.
 *
 * Conventions: plain pointers and sizes only; no exceptions cross the boundary; every function
 * that can fail returns an rmb_status and leaves a message retrievable with rmb_last_error().
 * Images are row-major with row 0 at the BOTTOM (OpenGL convention), RGBA interleaved.
 * One context drives one GPU (one process per GPU; multi-GPU jobs shard rows, see rank/n_ranks).
 * All calls are asynchronous on the context's stream except rmb_present, rmb_fb_read,
 * rmb_counters_read_all, rmb_sync and rmb_ctx_destroy.
 */
#ifndef RMB_H_
#define RMB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RMB_ABI_VERSION 1

typedef struct rmb_ctx rmb_ctx;         /* RenderJobContext            renderer/RenderJobExecutor.tsx:32-54 */
typedef struct rmb_program rmb_program; /* WebGLProgram (raymarcher)   renderer/ShaderCache.tsx:91-119      */
typedef struct rmb_fb rmb_fb;           /* RenderJobFramebufferInfo    renderer/RenderJobExecutor.tsx:14-30 */

typedef enum rmb_status {
    RMB_OK = 0,
    RMB_ERR_FRAGMENT = 1, /* scene failed to compile: ShaderError{type:"fragment"}  ShaderCache.tsx:8-11, :26-33 */
    RMB_ERR_PROGRAM = 2,  /* module load / link failure: ShaderError{type:"program"} ShaderCache.tsx:66-73      */
    RMB_ERR_GENERAL = 3,  /* {type:"general"} e.g. "Failed to load framebuffers."   RenderJobExecutor.tsx:73-75 */
    RMB_ERR_INVALID = 4   /* bad argument (null handle, unknown enum)                                           */
} rmb_status;

/* rmb_program_get flavours */
#define RMB_FLAVOUR_EXACT 0 /* scene arithmetic = unfused IEEE fp32, bit-identical to the CPU oracle */
#define RMB_FLAVOUR_FAST 1  /* scene arithmetic may use FMA contraction and approximate intrinsics   */
/* Measurement aid, not a product mode: the exact flavour with ONE implementation-defined GLSL choice
 * flipped - mod(x,y) = x - y*floor(x/y) with a true division and no fused multiply-add, as the GLSL ES
 * 3.00 text writes it - i.e. a second conforming implementation of the reference shader.  Comparing it
 * with RMB_FLAVOUR_EXACT shows how far two legal implementations drift apart on the same inputs. */
#define RMB_FLAVOUR_EXACT_ALT 2

/* uniform base types, renderer/Uniforms.tsx:7-9 ("f" | "i" | "ui") */
#define RMB_UNIFORM_F 0
#define RMB_UNIFORM_I 1
#define RMB_UNIFORM_UI 2

/* A scene uniform whose value is baked into the compiled program (uniform specialisation,
 * SURVEY.md H3).  `data` holds `count` values of the given base type. */
typedef struct rmb_spec_uniform {
    const char* name;
    int type;  /* RMB_UNIFORM_* */
    int count; /* 1..4 */
    union {
        float f[4];
        int32_t i[4];
        uint32_t u[4];
    } data;
} rmb_spec_uniform;

int rmb_abi_version(void);

/* ---- context -------------------------------------------------------------------------------
 * replaces loadRenderJobContext(gl)                     renderer/LoadRenderJobContext.tsx:268-287
 * and canvas.getContext("webgl2")                       index.tsx:106-108
 * device: CUDA ordinal.  rank/n_ranks/tile_rows: this context renders the row tiles t (of
 * tile_rows rows each) with t % n_ranks == rank (SURVEY.md 8e); n_ranks = 1 renders everything.
 * Returns NULL on failure (the reference returns undefined); rmb_last_error(NULL) explains. */
rmb_ctx* rmb_ctx_create(int device, int rank, int n_ranks, int tile_rows);
void rmb_ctx_destroy(rmb_ctx* ctx);
const char* rmb_last_error(rmb_ctx* ctx);
/* Draw pipeline: 0 (default) = wavefront kernels (setup -> persistent march -> shade) whenever the
 * scene's code is free of per-invocation mutable state, 1 = one-thread-per-pixel megakernel always.
 * Both produce identical accumulators in the exact flavour (tests cross-check them). */
rmb_status rmb_ctx_set_pipeline(rmb_ctx* ctx, int pipeline);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t rmb_ctx_launch_count(rmb_ctx* ctx);
/* Device timing of the hot kernel (the persistent march kernel of the wavefront pipeline, or the
 * megakernel): returns the CUDA-event time and launch count accumulated since the previous call, then
 * switches the collection on or off.  Synchronises the stream.  Used by bench.py's roofline. */
rmb_status rmb_ctx_timing(rmb_ctx* ctx, int enable, double* hot_kernel_ms, uint64_t* hot_kernel_launches);
/* cudaStream_t all work of this context is enqueued on (for CUDA-event timing by the caller) */
void* rmb_ctx_stream(rmb_ctx* ctx);
rmb_status rmb_sync(rmb_ctx* ctx);

/* ---- programs ------------------------------------------------------------------------------
 * replaces programCache.getProgram(vsrc, fsrc.replace("//SCENESDFHERE", addDefaultFunctions(scene)))
 *                                                       renderer/RenderJobExecutor.tsx:121-127
 *          addDefaultFunctionsToShaderCode              settings/shader-editor/Validate.tsx:8-57
 *          createShaderFromSource / createProgram...    renderer/ShaderCache.tsx:13-119
 * Lowers the scene GLSL to CUDA C++, NVRTC-compiles it for sm_100a and caches the result by
 * (source, flavour, baked uniform values).  Compile errors are VALUES: the call returns
 * RMB_ERR_FRAGMENT / RMB_ERR_PROGRAM, writes "fragment" / "program" / "general" to err_type
 * (>= 16 bytes) and a GL-style info log ("ERROR: 0:<line>: ...", line numbered like the spliced
 * reference shader so that the editor's `line - 145` mapping, GLSLEditor.tsx:134-136, holds) to
 * infolog.  The program handle is owned by the context. */
rmb_status rmb_program_get(rmb_ctx* ctx, const char* scene_glsl, size_t scene_len, int flavour,
                           const rmb_spec_uniform* spec, int n_spec, rmb_program** out_program,
                           char* err_type, char* infolog, size_t infolog_cap);
/* 0 once the variant has been unloaded by the per-scene variant cap (RMB_VARIANT_CAP, least recently used first): the
 * handle stays valid memory, every call on it reports an error, rmb_program_get rebuilds the variant */
int rmb_program_is_live(rmb_program* prog);
/* generated CUDA C++ translation unit (debugging / tests); owned by the program */
const char* rmb_program_source(rmb_program* prog);
/* registers per thread / local-memory bytes of a kernel: 0 preview megakernel, 1 full megakernel,
 * 2 preview march, 3 castRay march, 4 setup, 5 bounce (2..5: wavefront, pure scenes only); -1 if unknown */
int rmb_program_kernel_attr(rmb_program* prog, int kernel, int* regs, int* local_bytes);

/* ---- uniforms ------------------------------------------------------------------------------
 * replaces setUniforms(gl, program, {name: UniformData}) renderer/Uniforms.tsx:34-46
 *          gl.uniform1fv / uniform3fv on arrays          renderer/RenderJobExecutor.tsx:268-291
 *          gl.uniformMatrix4fv(loc, false, m)            renderer/RenderJobExecutor.tsx:293-297
 * Unknown names are ignored like a null uniform location (returns RMB_OK).  Values persist per
 * program until overwritten, as GL uniform state does (SURVEY.md H7); they reach __constant__
 * memory asynchronously before the next rmb_render_sample.  Setting a baked uniform to a value
 * different from the baked one returns RMB_ERR_INVALID (ask rmb_program_get for a new variant). */
rmb_status rmb_uniform_set(rmb_program* prog, const char* name, int type, int count, const void* data);
rmb_status rmb_uniform_set_array(rmb_program* prog, const char* name, int type, int components,
                                 int n_elements, const void* data);
rmb_status rmb_uniform_matrix4(rmb_program* prog, const char* name, const float* m16_column_major);
/* The whole built-in uniform record of one sample in ONE call: the values RenderJobExecutor.tsx:212-297 uploads before every
 * draw (setUniforms record :212-264, the step-count / light arrays :268-291, uniformMatrix4fv :293-297), applied in that
 * order with the semantics of the single calls above.  SURVEY.md 8b's "one POD FrameUniforms struct"; a host that sets ~25
 * uniforms per sample through an FFI pays for one crossing instead.  Scene-declared custom uniforms still go by name. */
typedef struct rmb_frame_uniforms {
    float blendWithPreviousFactor;
    float randNoise[2];
    float position[3];
    float rotation[16];                 /* column-major, transpose = false */
    float dofAmount, dofFocalPlaneDistance;
    int32_t cameraMode;                 /* 0 perspective, 1 orthographic, 2 panoramic */
    float fov;
    float reflections, raymarchingSteps, indirectLightingRaymarchingSteps;
    float aspect, fogDensity, exposure;
    int32_t blendMode, renderMode;      /* 1 additive; 1 preview */
    int32_t stepCountsLength;           /* entries of raymarchingStepCountsArray to upload (the reference uploads counts.length) */
    float raymarchingStepCountsArray[10];
    int32_t lightCount;
    float lightPositions[30], lightColors[30], lightSizes[10];
    int32_t showDofFocalPlane;
} rmb_frame_uniforms;
rmb_status rmb_uniforms_set_frame(rmb_program* prog, const rmb_frame_uniforms* u);

/* ---- framebuffer pool ----------------------------------------------------------------------
 * replaces context.fbo.create / context.fbo.delete       renderer/LoadRenderJobContext.tsx:184-249
 * Same semantics: get-or-create by (w, h, frameid); a released set waits in a 3-entry
 * "purgatory" and is reused for the next acquire of the same size, cleared to zero iff the
 * frameid differs; new sets start zeroed.  Accumulator formats follow
 * LoadRenderJobContext.tsx:50-124: colour RGBA32F, normal+dofRadius RGBA16F, albedo+depth RGBA16F.
 * Returns NULL when allocation fails ("Failed to load framebuffers."). */
rmb_fb* rmb_fb_acquire(rmb_ctx* ctx, int width, int height, int64_t frameid);
void rmb_fb_release(rmb_ctx* ctx, int width, int height, int64_t frameid);
/* number of rows this rank owns (== height when n_ranks == 1) and their global row indices */
int rmb_fb_local_rows(rmb_fb* fb);
int rmb_fb_global_row(rmb_fb* fb, int local_row);

/* ---- draw ----------------------------------------------------------------------------------
 * replaces gl.scissor + the raymarcher drawArrays + the blit drawArrays of one sample
 *                                                       renderer/RenderJobExecutor.tsx:181-326
 * (sx, sy, sw, sh) is a GL scissor box: x, y, WIDTH, HEIGHT, clipped to the framebuffer.  The
 * kernel accumulates in place, which equals draw-into-curr followed by blit-to-prev. */
rmb_status rmb_render_sample(rmb_ctx* ctx, rmb_program* prog, rmb_fb* fb, int sx, int sy, int sw, int sh);

/* ---- present / readback --------------------------------------------------------------------
 * replaces present(): display.frag drawn to the canvas   index.tsx:25-59, shader/display.frag:20-61
 *          canvas.toDataURL capture                      index.tsx:470-476
 * Runs the display pass (DoF blur, brightness, gamma 1/2.2) over this rank's rows and copies
 * local_rows*width*4 bytes of RGBA8 to rgba8_host and, if depth_host != NULL, local_rows*width
 * floats of hit depth (fp32, latest sample; SURVEY.md H5).  Blocking. */
rmb_status rmb_present(rmb_ctx* ctx, rmb_fb* fb, float brightness, uint8_t* rgba8_host, float* depth_host);
/* display pass only; the RGBA8 result stays in device memory (rmb_fb_device_ptr(fb, 4)) */
rmb_status rmb_present_device(rmb_ctx* ctx, rmb_fb* fb, float brightness);
/* Non-blocking present, the shape of the reference's own present (WebGL draws are asynchronous,
 * index.tsx:25-59; only toDataURL, index.tsx:470-476, waits): display pass on the context's stream,
 * then the readbacks on a second stream so that they overlap the next frame's kernels.  The host
 * buffers (pinned: rmb_host_alloc) are valid after rmb_present_wait(ctx, fb).  A later draw into the
 * same framebuffer set waits for the readback on the device, never on the host. */
rmb_status rmb_present_async(rmb_ctx* ctx, rmb_fb* fb, float brightness, uint8_t* rgba8_host, float* depth_host);
rmb_status rmb_present_wait(rmb_ctx* ctx, rmb_fb* fb);

/* ---- multi-GPU tile gather, fused into the display pass --------------------------------------
 * (SURVEY.md 8e; the reference has one WebGL context and no counterpart.)  With a gather target set,
 * the display kernel of rmb_present* stores every RGBA8 pixel a second time, at its GLOBAL row, into
 * `rgba8_full_frame` (width*height*4 bytes, row 0 = bottom).  Pointing every rank's context at ONE
 * buffer - rank 0's, mapped into the other processes with rmb_ipc_export / rmb_ipc_open (CUDA IPC,
 * peer access over NVLink) - assembles the frame with coalesced peer stores and no separate collective;
 * the caller only orders "all ranks have presented" (e.g. one NCCL all-reduce of a flag per frame on
 * the contexts' streams).  NULL switches the second store off. */
rmb_status rmb_ctx_set_gather_target(rmb_ctx* ctx, void* rgba8_full_frame, size_t bytes);
/* Frames whose display pass blurs (full mode with depth of field: display.frag:25-55 reads up to 16 rows
 * either side, REPEAT-wrapped) cannot be presented tile by tile: every rank scatters its rows of the
 * colour (which 0) and normal+dofRadius (which 1) accumulators into full-frame planes on one rank
 * (peer memory), which then runs the display pass over the assembled planes. */
rmb_status rmb_fb_scatter_rows(rmb_ctx* ctx, rmb_fb* fb, int which, void* dst_full_plane);
rmb_status rmb_display_planes(rmb_ctx* ctx, const void* color_full, const void* nd_full, void* rgba8_out, int width, int height, float brightness);
rmb_status rmb_ipc_export(void* device_ptr, unsigned char handle64[64]);
rmb_status rmb_ipc_open(rmb_ctx* ctx, const unsigned char handle64[64], void** device_ptr);
rmb_status rmb_ipc_close(rmb_ctx* ctx, void* device_ptr);

/* Completion flags for that gather (the alternative to a per-frame collective): 32-bit counters in memory every process of
 * the box can see - e.g. a POSIX shared-memory segment each process maps and registers with rmb_host_register - written
 * and awaited IN STREAM ORDER (cuStreamWriteValue32 / cuStreamWaitValue32): a rank's "my rows of frame f are stored" follows
 * its display kernel, rank 0's stream waits for every rank's counter before it touches the assembled frame, and the other
 * ranks wait for rank 0's "consumed" counter before they overwrite a frame slot.  No host synchronisation, no NCCL.
 * `flag`: registered host memory or device memory.  RMB_ERR_GENERAL when the driver lacks stream memory operations. */
rmb_status rmb_host_register(void* host_ptr, size_t bytes);
rmb_status rmb_host_unregister(void* host_ptr);
rmb_status rmb_stream_write_u32(rmb_ctx* ctx, void* flag, uint32_t value);
/* work enqueued on `ctx` from now on runs after everything enqueued on `other` so far (event record + stream wait) */
rmb_status rmb_ctx_wait_ctx(rmb_ctx* ctx, rmb_ctx* other);
rmb_status rmb_stream_wait_geq_u32(rmb_ctx* ctx, void* flag, uint32_t value);

/* ---- inspection (tests, benchmarks) --------------------------------------------------------- */
/* which: 0 colour (float4), 1 normal+dofRadius (4 x binary16), 2 albedo+depth (4 x binary16),
 *        3 depth (float), 4 RGBA8 of the last present */
void* rmb_fb_device_ptr(rmb_fb* fb, int which);
size_t rmb_fb_plane_bytes(rmb_fb* fb, int which);
rmb_status rmb_fb_read(rmb_ctx* ctx, rmb_fb* fb, int which, void* host, size_t bytes);
rmb_status rmb_fb_write(rmb_ctx* ctx, rmb_fb* fb, int which, const void* host, size_t bytes);
/* asynchronous device-to-device copy of a plane on the context's stream (multi-GPU tile gather:
 * the caller hands the destination to NCCL in the same stream order) */
rmb_status rmb_fb_copy_to_device(rmb_ctx* ctx, rmb_fb* fb, int which, void* dst_device, size_t bytes);
/* all 16 counter slots, since the last reset: out[0] = SDF evaluations executed, out[1] = pixel-samples rendered,
 * out[2] = how many of out[0] took the far-field shortcut of a carved scene (below); [3..11] are filled only by programs
 * built with RMB_PROFILE=1 in the environment (a measurement aid of the march kernel, see tools/march_timeline.py):
 * warp-nanoseconds and warp-iterations before / after the work queue ran dry, warps, the longest warp, live lanes per
 * iteration */
rmb_status rmb_counters_read_all(rmb_ctx* ctx, uint64_t out[16], int reset);
/* evaluates the scene's sdf() and material functions at n points: in n*3 floats, out n*17 floats
 * (diffuse rgb, specular rgb, roughness, subsurface, subsurfaceColor rgb, IOR, emission rgb, sdf, 0) */
rmb_status rmb_probe(rmb_ctx* ctx, rmb_program* prog, const float* points_xyz, int n, float* out17);
/* Far-field shortcut ("carve").  When the scene's sdf() has the form max(A, -M) with M a union of
 * `length(..) - K` shapes whose K do not depend on the position (the reference's default scene,
 * client/public/examples/guide.glsl:91-102, and its start-up placeholder, client/src/index.tsx:374-388),
 * -M <= U for a constant U, so sdf(P) == A bit for bit wherever A > U and the march kernels skip the
 * union loop there.  rmb_program_has_carve: 1 when the program was built with it (RMB_CARVE=0 in the
 * environment builds without).  rmb_probe_carve: n points in, n*4 floats out: sdf(P) as the march
 * kernels evaluate it, A(P), U, and sdf(P) as the guarded reference evaluation (rmb_probe's). */
int rmb_program_has_carve(rmb_program* prog);
rmb_status rmb_probe_carve(rmb_ctx* ctx, rmb_program* prog, const float* points_xyz, int n, float* out4);
/* Lowering + NVRTC compile for sm_100a without touching a GPU (build checks, offline SASS
 * inspection).  cubin_out/source_out may be NULL. */
rmb_status rmb_compile_only(const char* scene_glsl, size_t scene_len, int flavour, const rmb_spec_uniform* spec,
                            int n_spec, char* infolog, size_t infolog_cap, void* cubin_out, size_t cubin_cap,
                            size_t* cubin_bytes, char* source_out, size_t source_cap);
/* The lowering alone (GLSL scene -> the CUDA C++ translation unit NVRTC would be given), no compile:
 * scene-level diagnostics (missing sdf, unsupported uniform types; Validate.tsx:8-57 asks the GLSL
 * compiler the same questions) in milliseconds, and the text the CPU tests inspect. */
rmb_status rmb_translate_only(const char* scene_glsl, size_t scene_len, int flavour, const rmb_spec_uniform* spec,
                              int n_spec, char* infolog, size_t infolog_cap, char* source_out, size_t source_cap);
/* FP32 FMA throughput of this GPU in TFLOP/s (register-only FFMA kernel, best of `seconds` of
 * launches): the roofline denominator for this FP32-bound path (SURVEY.md 8d). */
rmb_status rmb_measure_fp32_peak(rmb_ctx* ctx, double seconds, double* tflops);
/* the same probe issued as packed FFMA2 (fma.rn.f32x2, 4 flop per lane-instruction): tells whether
 * packing raises the FP32 ceiling or only saves issue slots */
rmb_status rmb_measure_fp32x2_peak(rmb_ctx* ctx, double seconds, double* tflops);
/* host-only helper: rows with global index < g owned by `rank` under the round-robin row-tile
 * deal (tile t -> rank t % n_ranks).  -1 on bad arguments.  Needs no GPU. */
int rmb_owned_rows_below(int g, int height, int tile_rows, int n_ranks, int rank);
/* plain device allocations (a whole cudaMalloc each, so they can be exported with rmb_ipc_export) */
void* rmb_device_alloc(rmb_ctx* ctx, size_t bytes);
void rmb_device_free(rmb_ctx* ctx, void* p);
/* pinned host memory for the caller's readback buffers */
void* rmb_host_alloc(size_t bytes);
void rmb_host_free(void* p);

/* ---- device groups: all GPUs of one box behind one handle -------------------------------------
 * SURVEY.md 8b: `ctx_create(device_ids[], n)` - one context that owns the streams, program cache and buffer pool of
 * every device, reachable from a single-threaded host (client/src/index.tsx:236-263 pumps ONE doRenderJob generator;
 * renderer/RenderJobExecutor.tsx:77-341).  A group is n member contexts in ONE process - member i renders the row
 * tiles t (tile_rows rows each) with t % n == i (SURVEY.md 8e; the reference's own image-space split is the
 * `subdivisions` scissor loop, RenderJobExecutor.tsx:148-182) - and each call below is the single-device call of the
 * same name fanned out to the members.  No torch, no NCCL: the assembled RGBA8 frame lives on member 0's device, the
 * other devices store into it from their display kernels through peer access (cudaDeviceEnablePeerAccess, NVLink),
 * and completion is ordered by cross-device events.  Frames that may blur (some sample drawn with renderMode != 1)
 * scatter their colour / normal+dofRadius rows to member 0, which runs the display pass over the assembled planes.
 * `devices` may name one device more than once (two members on one GPU: the same code path, without peer traffic).
 * rmb_group_create returns NULL on failure; rmb_group_last_error(NULL) explains. */
typedef struct rmb_group rmb_group;
typedef struct rmb_group_program rmb_group_program;
typedef struct rmb_group_fb rmb_group_fb;
rmb_group* rmb_group_create(const int* devices, int n, int tile_rows);
void rmb_group_destroy(rmb_group* group);
const char* rmb_group_last_error(rmb_group* group);
int rmb_group_size(rmb_group* group);
/* member context i (borrowed): per-device inspection, counters, timing */
rmb_ctx* rmb_group_ctx(rmb_group* group, int member);
rmb_status rmb_group_sync(rmb_group* group);
/* rmb_program_get on every member (one host thread per device); errors are values exactly as there */
rmb_status rmb_group_program_get(rmb_group* group, const char* scene_glsl, size_t scene_len, int flavour,
                                 const rmb_spec_uniform* spec, int n_spec, rmb_group_program** out_program,
                                 char* err_type, char* infolog, size_t infolog_cap);
rmb_program* rmb_group_program_member(rmb_group_program* prog, int member);
rmb_status rmb_group_uniform_set(rmb_group_program* prog, const char* name, int type, int count, const void* data);
rmb_status rmb_group_uniform_set_array(rmb_group_program* prog, const char* name, int type, int components,
                                       int n_elements, const void* data);
rmb_status rmb_group_uniform_matrix4(rmb_group_program* prog, const char* name, const float* m16_column_major);
rmb_status rmb_group_uniforms_set_frame(rmb_group_program* prog, const rmb_frame_uniforms* u);
/* fbo.create / fbo.delete on every member (each keeps its own rows; pool semantics as rmb_fb_acquire) */
rmb_group_fb* rmb_group_fb_acquire(rmb_group* group, int width, int height, int64_t frameid);
void rmb_group_fb_release(rmb_group* group, int width, int height, int64_t frameid);
rmb_fb* rmb_group_fb_member(rmb_group_fb* fb, int member);
/* one sample: every member draws its rows of the scissor box (asynchronous) */
rmb_status rmb_group_render_sample(rmb_group* group, rmb_group_program* prog, rmb_group_fb* fb, int sx, int sy, int sw, int sh);
/* present(): display pass on every member + assembly on member 0; rgba8_host receives the WHOLE frame
 * (width*height*4 bytes, row 0 = bottom), depth_host (optional) width*height floats.  Blocking, like rmb_present. */
rmb_status rmb_group_present(rmb_group* group, rmb_group_fb* fb, float brightness, uint8_t* rgba8_host, float* depth_host);
/* the same without the readback (asynchronous): *rgba8_device = the assembled frame on member 0's device, complete
 * after rmb_group_sync and valid until the next present of this group */
rmb_status rmb_group_present_device(rmb_group* group, rmb_group_fb* fb, float brightness, void** rgba8_device);

#ifdef __cplusplus
}
#endif
#endif /* RMB_H_ */
