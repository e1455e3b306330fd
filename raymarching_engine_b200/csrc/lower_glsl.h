// lower_glsl.h -- GLSL ES 3.00 scene source -> CUDA C++ member declarations for struct Frag
// (device_src/raymarch_kernel.cuh).  Replaces the role the browser's GLSL compiler plays for
// the scene splice at /root/reference/client/public/shader/raymarcher.frag:146, and the
// "which material functions are missing" probe of
// /root/reference/client/src/settings/shader-editor/Validate.tsx:8-57.
#pragma once
#include <set>
#include <string>
#include <vector>

namespace rmb {

struct UniformDecl {
    std::string type;   // GLSL type name: float, int, uint, bool, vec2.., ivec2.., uvec2.., mat2..
    std::string name;
    int array_size = 0; // 0 = not an array
    int line = 0;       // 1-based line in the scene source
};

struct LowerResult {
    bool ok = false;
    std::string error;                  // GL-style message when !ok
    std::string body;                   // lowered scene text, same line structure as the input
    std::vector<UniformDecl> uniforms;  // scene-declared uniforms, removed from `body`
    std::set<std::string> functions;    // functions DEFINED at global scope
    std::set<std::string> macros;       // names the scene #defines: the translation unit #undefs them after the scene text,
                                        // so that they cannot reach the pipeline code spliced after it
    bool pure = true;                   // no mutable per-invocation state reachable from scene code
    std::string carve_text;             // non-empty when sdf() is a union of `length(..) - K` shapes carved out
                                        // of an outer shape (max(A, -M)): definitions of rm_carve_outer(P) = A
                                        // and rm_carve_bound() = an upper bound of -M valid at every position,
                                        // so that sdf(P) == A bit for bit wherever A > bound (lower_glsl.cpp 1b)
    int floor_sites = 0;                // > 0: carve_text also defines rm_floor_plim(), and that many domain repetitions of
                                        // sdf() are emitted as rm_rep_b / rm_rep0_b (floor() without a range guard while
                                        // every |position coordinate| <= rm_floor_plim(); lower_glsl.cpp pass 2)
};

// `constant_names`: uniforms that will be compile-time constants in this program variant (baked).
// A `for` loop whose header mentions only its own loop variable, literals and such constants gets
// `_Pragma("unroll 32")`, so that specialised programs fully unroll short fractal loops and fold the
// uniform-only sub-expressions (pow(), reciprocals) at compile time (SURVEY.md H3).
// `heavy_transcendentals`: the flavour evaluates sin / pow / acos ... in binary64 (exact): loops with several such calls on
// non-constant arguments are NOT unrolled (instruction-cache footprint).
LowerResult lower_scene(const std::string& glsl, const std::set<std::string>& constant_names = {}, bool heavy_transcendentals = false);

// The seven material functions every program must define and their default bodies
// (Validate.tsx:18-51), already in lowered form.
struct DefaultFunction {
    const char* name;
    const char* text;
};
const std::vector<DefaultFunction>& default_material_functions();

// GLSL type -> (base type: 'f','i','u','b', component count, is matrix columns)
bool uniform_type_info(const std::string& type, char* base, int* components);

}  // namespace rmb
