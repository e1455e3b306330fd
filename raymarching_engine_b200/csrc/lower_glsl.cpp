// lower_glsl.cpp -- token-level lowering of a GLSL ES 3.00 scene to C++ that compiles against
// device_src/glsl_rt.h inside `struct Frag`.  See lower_glsl.h.
//
// What the lowering does (everything else in GLSL's expression/statement syntax is already
// valid C++ given the vector types, swizzle proxies and built-ins of glsl_rt.h):
//   * comments are blanked, line structure is preserved (diagnostics keep scene line numbers);
//   * `uniform T name[N];` declarations at global scope are collected and removed;
//   * floating literals get an `f` suffix (GLSL `1.0` is fp32, C++ `1.0` is double);
//   * `precision ...;` statements, precision qualifiers and `layout(...)` are dropped;
//   * parameter qualifiers: `in` is dropped, `out`/`inout` turn the parameter into a reference;
//   * identifiers that are C++ keywords but legal GLSL names are renamed (`not` -> `not_`);
//   * `#version` / `#extension` lines are dropped, other preprocessor lines pass through;
//   * functions defined at global scope are recorded (for default-function injection);
//   * purity analysis: a scene that declares mutable globals or touches the RNG state
//     (`seed`, uniformSample, ...) may not use the fixed-point early exit.
#include "lower_glsl.h"

#include <cctype>
#include <algorithm>
#include <cstring>
#include <functional>
#include <map>

namespace rmb {

namespace {

enum Kind { kIdent, kNumber, kPunct, kPP };

struct Token {
    Kind kind;
    std::string text;
    std::string ws;   // whitespace (incl. newlines and blanked comments) preceding the token
    int line;
    bool drop = false;
};

bool is_ident_start(char c) { return std::isalpha((unsigned char)c) || c == '_'; }
bool is_ident_char(char c) { return std::isalnum((unsigned char)c) || c == '_'; }

// Splits the source into tokens; comments become whitespace (newlines kept).
std::vector<Token> tokenize(const std::string& s, std::string* trailing_ws) {
    std::vector<Token> out;
    std::string ws;
    int line = 1;
    size_t i = 0, n = s.size();
    bool line_start = true;
    while (i < n) {
        char c = s[i];
        if (c == '\n') { ws += '\n'; line++; i++; line_start = true; continue; }
        if (c == ' ' || c == '\t' || c == '\r' || c == '\f' || c == '\v') { ws += (c == '\r' ? ' ' : c); i++; continue; }
        if (c == '/' && i + 1 < n && s[i + 1] == '/') {
            while (i < n && s[i] != '\n') i++;
            continue;
        }
        if (c == '/' && i + 1 < n && s[i + 1] == '*') {
            i += 2;
            while (i < n && !(s[i] == '*' && i + 1 < n && s[i + 1] == '/')) {
                if (s[i] == '\n') { ws += '\n'; line++; }
                i++;
            }
            i = (i + 2 <= n) ? i + 2 : n;
            ws += ' ';
            continue;
        }
        Token t;
        t.line = line;
        t.ws = ws;
        ws.clear();
        if (c == '#' && line_start) {
            // whole preprocessor line (with backslash continuations)
            size_t j = i;
            while (j < n) {
                if (s[j] == '\n') {
                    if (j > 0 && s[j - 1] == '\\') { line++; j++; continue; }
                    break;
                }
                j++;
            }
            t.kind = kPP;
            t.text = s.substr(i, j - i);
            i = j;
            out.push_back(t);
            continue;
        }
        line_start = false;
        if (is_ident_start(c)) {
            size_t j = i;
            while (j < n && is_ident_char(s[j])) j++;
            t.kind = kIdent;
            t.text = s.substr(i, j - i);
            i = j;
        } else if (std::isdigit((unsigned char)c) || (c == '.' && i + 1 < n && std::isdigit((unsigned char)s[i + 1]))) {
            size_t j = i;
            bool is_float = false, is_hex = false;
            if (c == '0' && j + 1 < n && (s[j + 1] == 'x' || s[j + 1] == 'X')) {
                is_hex = true;
                j += 2;
                while (j < n && std::isxdigit((unsigned char)s[j])) j++;
            } else {
                while (j < n && std::isdigit((unsigned char)s[j])) j++;
                if (j < n && s[j] == '.') { is_float = true; j++; while (j < n && std::isdigit((unsigned char)s[j])) j++; }
                if (j < n && (s[j] == 'e' || s[j] == 'E')) {
                    size_t k = j + 1;
                    if (k < n && (s[k] == '+' || s[k] == '-')) k++;
                    if (k < n && std::isdigit((unsigned char)s[k])) {
                        is_float = true;
                        j = k;
                        while (j < n && std::isdigit((unsigned char)s[j])) j++;
                    }
                }
            }
            std::string num = s.substr(i, j - i);
            // suffixes: f/F (float), u/U (unsigned)
            if (j < n && (s[j] == 'f' || s[j] == 'F') && !is_hex) { is_float = true; j++; }
            else if (j < n && (s[j] == 'u' || s[j] == 'U')) { num += 'u'; j++; }
            if (is_float) {
                // "1." is valid in both languages; make sure the result is an fp32 literal
                num += 'f';
            }
            t.kind = kNumber;
            t.text = num;
            i = j;
        } else {
            // multi-character operators are kept together only where it matters for pasting
            static const char* ops[] = {"<<=", ">>=", "++", "--", "+=", "-=", "*=", "/=", "%=", "&=", "|=", "^=",
                                        "==", "!=", "<=", ">=", "&&", "||", "^^", "<<", ">>", nullptr};
            t.kind = kPunct;
            t.text = std::string(1, c);
            for (int k = 0; ops[k]; k++) {
                size_t L = strlen(ops[k]);
                if (s.compare(i, L, ops[k]) == 0) { t.text = ops[k]; break; }
            }
            i += t.text.size();
        }
        out.push_back(t);
    }
    *trailing_ws = ws;
    return out;
}

const std::set<std::string>& precision_words() {
    static const std::set<std::string> s = {"highp", "mediump", "lowp"};
    return s;
}

// C++ keywords / alternative tokens that GLSL ES 3.00 does not reserve
const std::map<std::string, std::string>& renames() {
    static const std::map<std::string, std::string> m = {
        {"not", "not_"},           {"and", "and_rmk"},         {"or", "or_rmk"},         {"xor", "xor_rmk"},
        {"bitand", "bitand_rmk"},  {"bitor", "bitor_rmk"},     {"compl", "compl_rmk"},   {"and_eq", "and_eq_rmk"},
        {"or_eq", "or_eq_rmk"},    {"xor_eq", "xor_eq_rmk"},   {"not_eq", "not_eq_rmk"}, {"new", "new_rmk"},
        {"delete", "delete_rmk"},  {"try", "try_rmk"},         {"catch", "catch_rmk"},   {"throw", "throw_rmk"},
        {"char", "char_rmk"},      {"auto", "auto_rmk"},       {"register", "register_rmk"}, {"explicit", "explicit_rmk"},
        {"mutable", "mutable_rmk"}, {"friend", "friend_rmk"},  {"virtual", "virtual_rmk"}, {"private", "private_rmk"},
        {"protected", "protected_rmk"}, {"operator", "operator_rmk"}, {"typename", "typename_rmk"},
        {"wchar_t", "wchar_t_rmk"}, {"nullptr", "nullptr_rmk"}, {"alignas", "alignas_rmk"}, {"alignof", "alignof_rmk"},
        {"decltype", "decltype_rmk"}, {"constexpr", "constexpr_rmk"}, {"noexcept", "noexcept_rmk"},
        {"static_assert", "static_assert_rmk"}, {"thread_local", "thread_local_rmk"}, {"signed", "signed_rmk"},
        {"char16_t", "char16_t_rmk"}, {"char32_t", "char32_t_rmk"}, {"char8_t", "char8_t_rmk"},
        {"concept", "concept_rmk"}, {"requires", "requires_rmk"}, {"consteval", "consteval_rmk"},
        {"constinit", "constinit_rmk"}, {"co_await", "co_await_rmk"}, {"co_return", "co_return_rmk"},
        {"co_yield", "co_yield_rmk"}, {"reinterpret_cast", "reinterpret_cast_rmk"}, {"static_cast", "static_cast_rmk"},
        {"dynamic_cast", "dynamic_cast_rmk"}, {"const_cast", "const_cast_rmk"}, {"typeid", "typeid_rmk"},
        {"asm", "asm_rmk"}, {"export", "export_rmk"}, {"final", "final"}, {"override", "override"},
    };
    return m;
}

const std::set<std::string>& rng_state_words() {
    static const std::set<std::string> s = {"seed", "uniformSample", "boxMullerTransform", "sphereSample", "circleSample"};
    return s;
}

}  // namespace

bool uniform_type_info(const std::string& type, char* base, int* components) {
    struct E { const char* n; char b; int c; };
    static const E table[] = {
        {"float", 'f', 1}, {"vec2", 'f', 2},  {"vec3", 'f', 3},  {"vec4", 'f', 4},  {"int", 'i', 1},   {"ivec2", 'i', 2},
        {"ivec3", 'i', 3}, {"ivec4", 'i', 4}, {"uint", 'u', 1},  {"uvec2", 'u', 2}, {"uvec3", 'u', 3}, {"uvec4", 'u', 4},
        {"bool", 'b', 1},  {"bvec2", 'b', 2}, {"bvec3", 'b', 3}, {"bvec4", 'b', 4}, {"mat2", 'f', 4},  {"mat3", 'f', 9},
        {"mat4", 'f', 16},
    };
    for (const E& e : table)
        if (type == e.n) { *base = e.b; *components = e.c; return true; }
    return false;
}

const std::vector<DefaultFunction>& default_material_functions() {
    // Restated from Validate.tsx:18-51 (the reference appends these GLSL bodies when the scene
    // does not define the function).
    static const std::vector<DefaultFunction> v = {
        {"sceneDiffuseColor",
         "vec3 sceneDiffuseColor(vec3 position) { if (length(position) > 35.0f) return vec3(0.0f); return vec3(0.6f); }\n"},
        {"sceneSpecularColor",
         "vec3 sceneSpecularColor(vec3 position) { if (length(position) > 35.0f) return vec3(0.0f); return vec3(0.6f); }\n"},
        {"sceneSpecularRoughness", "float sceneSpecularRoughness(vec3 position) { return 0.2f; }\n"},
        {"sceneSubsurfaceScattering", "float sceneSubsurfaceScattering(vec3 position) { return 11111115.0f; }\n"},
        {"sceneSubsurfaceScatteringColor",
         "vec3 sceneSubsurfaceScatteringColor(vec3 position) { if (length(position) > 30.0f) return vec3(1.0f); return vec3(1.0f); }\n"},
        {"sceneIOR", "float sceneIOR(vec3 position) { return 100.0f; }\n"},
        {"sceneEmission",
         "vec3 sceneEmission(vec3 position) { float d = max(normalize(position).y, 0.2f); "
         "vec3 brightColor = vec3(0.7f, 0.8f, 1.0f) * d * 1.0f; "
         "return (length(position) > 36.0f) ? (brightColor * 2.00f) : vec3(0.0f); }\n"},
    };
    return v;
}

LowerResult lower_scene(const std::string& glsl, const std::set<std::string>& constant_names, bool heavy_transcendentals) {
    LowerResult R;
    std::string trailing;
    std::vector<Token> T = tokenize(glsl, &trailing);
    const size_t n = T.size();

    auto fail = [&](int line, const std::string& msg) {
        R.ok = false;
        R.error = "ERROR: 0:" + std::to_string(line) + ": " + msg;
        return R;
    };

    // ---- pass 1: structural walk at global scope ------------------------------------------
    int brace = 0, paren = 0;
    size_t i = 0;
    // statement_start: index of the first token of the current global-scope declaration
    bool at_decl_start = true;
    while (i < n) {
        Token& t = T[i];
        if (t.kind == kPP) {
            // #version / #extension are GLSL-only.  The other directives are handed to NVRTC, but only the ones GLSL ES
            // 3.00 itself has (section 3.4): anything else - #include above all, which would make NVRTC read host files
            // and quote them in the info log - is the compile error it is in the reference's sandboxed GLSL.  A #define /
            // #undef may not touch the names the pipeline splices around the scene (rm_*, g_*, RM_*, GLSL_*, __*): a
            // scene macro could otherwise rewrite the hand-written kernels and silently break their parity.
            size_t p = 1;
            while (p < t.text.size() && (t.text[p] == ' ' || t.text[p] == '\t')) p++;
            size_t q = p;
            while (q < t.text.size() && (isalpha((unsigned char)t.text[q]) || t.text[q] == '_')) q++;
            const std::string d = t.text.substr(p, q - p);
            static const std::set<std::string> allowed = {"", "define", "undef", "if", "ifdef", "ifndef", "else", "elif", "endif",
                                                          "error", "pragma", "line", "version", "extension"};
            if (!allowed.count(d)) return fail(t.line, "'#" + d + "' : invalid directive name");
            if (d == "version" || d == "extension") t.drop = true;
            if (d == "define" || d == "undef") {
                size_t a = q;
                while (a < t.text.size() && (t.text[a] == ' ' || t.text[a] == '\t')) a++;
                size_t b = a;
                while (b < t.text.size() && (isalnum((unsigned char)t.text[b]) || t.text[b] == '_')) b++;
                const std::string name = t.text.substr(a, b - a);
                auto starts = [&](const char* pre) { return name.compare(0, strlen(pre), pre) == 0; };
                if (starts("rm_") || starts("g_") || starts("RM_") || starts("GLSL_") || starts("__") || starts("gl_") || starts("GL_") ||
                    name == "sdfAt" || name == "S" || renames().count(name))
                    return fail(t.line, "'" + name + "' : reserved built-in macro name");
                if (d == "define" && !name.empty()) R.macros.insert(name);
            }
            i++;
            continue;
        }
        if (t.kind == kIdent) {
            if (precision_words().count(t.text)) { t.drop = true; i++; continue; }
            if (t.text == "precision") {
                // precision <qual> <type> ;
                size_t j = i;
                while (j < n && !(T[j].kind == kPunct && T[j].text == ";")) { T[j].drop = true; j++; }
                if (j < n) T[j].drop = true;
                i = j + 1;
                continue;
            }
            auto rn = renames().find(t.text);
            if (rn != renames().end()) t.text = rn->second;
            if (rng_state_words().count(t.text)) R.pure = false;
        }
        if (t.kind == kIdent && t.text == "for" && brace > 0 && i + 1 < n && T[i + 1].text == "(") {
            // constant-trip-count loop?  identifiers allowed in the header: type names, the loop
            // variable(s) declared in the init clause, and baked uniforms
            size_t k = i + 1;
            int d = 0;
            size_t close = 0;
            while (k < n) {
                if (T[k].text == "(") d++;
                if (T[k].text == ")") { d--; if (d == 0) { close = k; break; } }
                k++;
            }
            if (close) {
                std::set<std::string> locals;
                bool ok = true, init = true;
                char bt; int bc;
                for (size_t q = i + 2; q < close && ok; q++) {
                    if (T[q].text == ";") init = false;
                    if (T[q].kind != kIdent) continue;
                    const std::string& w = T[q].text;
                    if (uniform_type_info(w, &bt, &bc) || precision_words().count(w) || w == "const") continue;
                    if (init && q > i + 2 && T[q - 1].kind == kIdent && uniform_type_info(T[q - 1].text, &bt, &bc)) { locals.insert(w); continue; }
                    if (locals.count(w) || constant_names.count(w)) continue;
                    ok = false;
                }
                // Unrolling is what folds pow(uniform, i) / reciprocals of a specialised program at compile time - but in the
                // exact flavour every transcendental whose argument is NOT such a constant inlines 40-150 instructions of
                // binary64 arithmetic: a 12-trip Mandelbulb DE unrolled 12 times is a 39 000-instruction kernel that runs
                // out of the instruction cache (ncu: 16 "no instruction" stalls per issue, 18 % issue utilisation).  Loops
                // with three or more such calls keep their loop form there.
                int heavy_calls = 0;
                if (ok && !locals.empty() && heavy_transcendentals) {
                    static const std::set<std::string> tr = {"sin", "cos", "tan", "asin", "acos", "atan", "sinh", "cosh", "tanh", "asinh", "acosh",
                                                             "atanh", "pow", "exp", "log", "exp2", "log2"};
                    size_t b0 = close + 1, b1 = b0;
                    if (b0 < n && T[b0].text == "{") {
                        int bd = 0;
                        for (b1 = b0; b1 < n; b1++) {
                            if (T[b1].text == "{") bd++;
                            if (T[b1].text == "}") { bd--; if (bd == 0) break; }
                        }
                    } else {
                        while (b1 < n && T[b1].text != ";") b1++;
                    }
                    for (size_t q = b0; q < b1 && q + 1 < n; q++) {
                        if (T[q].kind != kIdent || !tr.count(T[q].text) || T[q + 1].text != "(") continue;
                        // arguments made of literals, loop variables and baked uniforms only: folds once unrolled
                        bool foldable = true;
                        int pd = 0;
                        for (size_t a = q + 1; a < b1; a++) {
                            if (T[a].text == "(") pd++;
                            if (T[a].text == ")") { pd--; if (pd == 0) break; }
                            if (T[a].kind == kIdent && !locals.count(T[a].text) && !constant_names.count(T[a].text) &&
                                !uniform_type_info(T[a].text, &bt, &bc))
                                foldable = false;
                        }
                        if (!foldable) heavy_calls++;
                    }
                }
                if (ok && !locals.empty()) t.text = heavy_calls >= 3 ? "_Pragma(\"unroll 1\") for" : "_Pragma(\"unroll 32\") for";
            }
        }
        if (brace == 0 && paren == 0 && t.kind == kIdent && at_decl_start) {
            // ---- global-scope declaration ----
            if (t.text == "layout") {
                t.drop = true;
                size_t j = i + 1;
                if (j < n && T[j].text == "(") {
                    int d = 0;
                    while (j < n) {
                        if (T[j].text == "(") d++;
                        if (T[j].text == ")") d--;
                        T[j].drop = true;
                        j++;
                        if (d == 0) break;
                    }
                }
                i = j;
                continue;   // still at declaration start
            }
            if (t.text == "uniform") {
                size_t j = i + 1;
                t.drop = true;
                while (j < n && T[j].kind == kIdent && (precision_words().count(T[j].text))) { T[j].drop = true; j++; }
                if (j >= n || T[j].kind != kIdent) return fail(t.line, "'uniform' : syntax error");
                std::string type = T[j].text;
                char b; int c;
                if (!uniform_type_info(type, &b, &c)) {
                    if (type.compare(0, 7, "sampler") == 0 || type.compare(0, 8, "isampler") == 0 || type.compare(0, 8, "usampler") == 0)
                        return fail(T[j].line, "'" + type + "' : sampler uniforms are not available to scene code");
                    return fail(T[j].line, "'" + type + "' : unsupported uniform type");
                }
                T[j].drop = true;
                j++;
                for (;;) {
                    if (j >= n || T[j].kind != kIdent) return fail(t.line, "'uniform' : expected identifier");
                    UniformDecl u;
                    u.type = type;
                    u.name = T[j].text;
                    u.line = T[j].line;
                    T[j].drop = true;
                    j++;
                    if (j < n && T[j].text == "[") {
                        T[j].drop = true;
                        j++;
                        if (j >= n || T[j].kind != kNumber) return fail(u.line, "'" + u.name + "' : array size must be an integer literal");
                        u.array_size = std::atoi(T[j].text.c_str());
                        if (u.array_size <= 0) return fail(u.line, "'" + u.name + "' : array size must be positive");
                        T[j].drop = true;
                        j++;
                        if (j >= n || T[j].text != "]") return fail(u.line, "'" + u.name + "' : expected ']'");
                        T[j].drop = true;
                        j++;
                    }
                    R.uniforms.push_back(u);
                    if (j < n && T[j].text == ",") { T[j].drop = true; j++; continue; }
                    break;
                }
                if (j >= n || T[j].text != ";") return fail(t.line, "'uniform' : expected ';'");
                T[j].drop = true;
                i = j + 1;
                continue;
            }
            if (t.text == "in" || t.text == "out" || t.text == "inout" || t.text == "flat" || t.text == "smooth" || t.text == "centroid" || t.text == "invariant") {
                // interface qualifiers make no sense in spliced scene code; treat as plain global
                t.drop = true;
                i++;
                continue;
            }
            // function definition / prototype:  [const] type name ( ... ) { | ;
            size_t j = i;
            bool is_const = false;
            if (T[j].text == "const") { is_const = true; j++; }
            if (T[j].text == "struct") {
                // struct definition: skip to the matching close brace at this level (members are
                // plain declarations, valid C++)
                at_decl_start = false;
                i++;
                continue;
            }
            if (j + 2 < n && T[j].kind == kIdent && T[j + 1].kind == kIdent && T[j + 2].text == "(") {
                // find matching ')'
                size_t k = j + 2;
                int d = 0;
                size_t close = 0;
                while (k < n) {
                    if (T[k].text == "(") d++;
                    if (T[k].text == ")") { d--; if (d == 0) { close = k; break; } }
                    k++;
                }
                if (!close) return fail(t.line, "'" + T[j + 1].text + "' : unbalanced parentheses");
                // parameter qualifiers
                for (size_t q = j + 3; q < close; q++) {
                    if (T[q].kind != kIdent) continue;
                    bool param_start = (q == j + 3) || T[q - 1].text == "," || (T[q - 1].kind == kIdent && (T[q - 1].text == "const" || T[q - 1].drop));
                    if (!param_start) continue;
                    if (T[q].text == "in") { T[q].drop = true; }
                    else if (T[q].text == "out" || T[q].text == "inout") {
                        T[q].drop = true;
                        size_t ty = q + 1;
                        while (ty < close && T[ty].kind == kIdent && precision_words().count(T[ty].text)) ty++;
                        if (ty < close && T[ty].kind == kIdent) T[ty].text += "&";
                    }
                }
                if (close + 1 < n && T[close + 1].text == "{") R.functions.insert(T[j + 1].text);
                // `void f(void)` is fine in C++ too
                at_decl_start = false;
                i++;
                continue;
            }
            // otherwise a global variable declaration
            if (!is_const) R.pure = false;
            at_decl_start = false;
            i++;
            continue;
        }
        if (t.kind == kPunct) {
            if (t.text == "{") brace++;
            else if (t.text == "}") { brace--; if (brace < 0) return fail(t.line, "'}' : syntax error"); if (brace == 0 && paren == 0) at_decl_start = true; }
            else if (t.text == "(") paren++;
            else if (t.text == ")") { paren--; if (paren < 0) return fail(t.line, "')' : syntax error"); }
            else if (t.text == ";" && brace == 0 && paren == 0) at_decl_start = true;
            else if (t.text == "^^") t.text = "!=";   // logical xor on bools
        }
        i++;
    }
    if (brace != 0) return fail(n ? T[n - 1].line : 1, "unexpected end of source: unbalanced '{'");


    // ---- pass 1b: "carve" analysis --------------------------------------------------------------
    // Recognises   float sdf(vec3 P) { float M = <literal>; ... M = min(length(..) - K, M); ...
    //                                  [V =] max(A, -M); return .. }
    // i.e. a union of shapes M carved out of an outer shape A (max(A, -M), the CSG difference).  When every
    // term of the union is `length(..) - K` with K independent of the position, -M can never exceed
    // U = max(-<literal>, max K) whatever the position is (length() >= 0 and rounding is monotonic; NaN
    // terms are dropped by min), so wherever A > U the function returns A bit for bit.  The march
    // kernels use that for the far field (raymarch_kernel.cuh, RM_HAS_CARVE): A costs ~10 instructions,
    // the union loop hundreds.  Two helper functions are emitted after the scene: rm_carve_outer(P) = A
    // and rm_carve_bound() = U, the latter being the scene's own sdf body with each accepted length()
    // replaced by zero and the final max() by (-M), so that U is computed by the same arithmetic, from
    // the same uniforms, as the terms it bounds.  Anything the analysis does not fully understand
    // (branches, early returns, macros, shadowing, a K that mentions position-dependent values, ...)
    // leaves the scene without the helpers.
    struct Carve {
        bool ok = false;
        size_t body_open = 0, body_close = 0;       // '{' and '}' of sdf
        std::string param, m_name;
        size_t ea_first = 0, ea_last = 0;           // token range of A
        size_t max_first = 0, max_close = 0;        // `max` .. its ')'
        std::vector<size_t> len_tokens;             // the accepted `length` identifiers
        // pattern B ("iterated difference", see below): X = max(X, -E) with E a min() tree of sdBox(.., B) calls
        bool boxes = false;
        size_t x_init_first = 0, x_init_last = 0;   // initialiser of X (= A)
        std::map<size_t, size_t> box_sites;         // `sdBox` token -> the ',' that ends its first argument
        // bounded-floor analysis (pass 2): position-independent names of sdf's body, the return statement, and the
        // domain-repetition call sites whose operand is the position parameter itself
        std::set<std::string> clean;
        size_t ret_tok = 0, ret_semi = 0;
        std::vector<size_t> rep_sites;
    } carve;
    static const std::set<std::string> pure_builtins = {
        "pow", "exp", "exp2", "log", "log2", "sqrt", "inversesqrt", "abs", "sign", "floor", "ceil", "fract", "mod", "min", "max",
        "clamp", "mix", "step", "smoothstep", "sin", "cos", "tan", "asin", "acos", "atan", "radians", "degrees", "length",
        "distance", "dot", "cross", "normalize", "round", "trunc"};
    std::set<std::string> uniform_names;
    for (const UniformDecl& u : R.uniforms) uniform_names.insert(u.name);
    if (R.pure) {
        auto live = [&](size_t k) { return k < n && !T[k].drop && T[k].kind != kPP; };
        auto next_live = [&](size_t k) { k++; while (k < n && !live(k)) k++; return k; };
        auto prev_live = [&](size_t k) -> size_t { while (k > 0) { k--; if (live(k)) return k; } return n; };
        auto match_close = [&](size_t open) -> size_t {
            int d = 0;
            for (size_t k = open; k < n; k++) {
                if (!live(k)) continue;
                const std::string& w = T[k].text;
                if (w == "(" || w == "[" || w == "{") d++;
                else if (w == ")" || w == "]" || w == "}") { d--; if (d == 0) return k; }
            }
            return n;
        };
        auto is_for = [&](size_t k) { const std::string& w = T[k].text; return T[k].kind == kIdent && w.size() >= 3 && w.compare(w.size() - 3, 3, "for") == 0 && (w.size() == 3 || w[w.size() - 4] == ' '); };
        static const std::set<std::string> assign_ops = {"=", "+=", "-=", "*=", "/=", "%=", "&=", "|=", "^=", "<<=", ">>=", "++", "--"};
        static const std::set<std::string> banned = {"if", "else", "while", "do", "switch", "case", "default", "break", "continue", "discard", "goto", "struct"};
        char bt; int bc;
        bool has_pp = false, has_ref_params = false, name_clash = false;
        for (size_t k = 0; k < n; k++) {
            if (T[k].kind == kPP && !T[k].drop) has_pp = true;
            if (live(k) && T[k].kind == kIdent && !T[k].text.empty() && T[k].text.back() == '&') has_ref_params = true;
            // the helper names must be free
            if (live(k) && T[k].kind == kIdent && (T[k].text.compare(0, 8, "rm_carve") == 0 || T[k].text == "rm_len0" || T[k].text == "rm_box0" || T[k].text.compare(0, 7, "rm_plim") == 0 ||
                                                       T[k].text.compare(0, 8, "rm_floor") == 0 || T[k].text.compare(0, 6, "rm_rep") == 0)) name_clash = true;
        }
        // the analysis reasons about the built-ins: a scene function of the same name (GLSL ES 3.00 forbids it, C++
        // member lookup would allow it) voids that
        for (const std::string& f : R.functions)
            if (pure_builtins.count(f) || uniform_type_info(f, &bt, &bc)) name_clash = true;
        // locate `float sdf ( [const] vec3 P ) {` at global scope (exactly one definition)
        size_t fn = n; int defs = 0;
        {
            int depth = 0;
            for (size_t k = 0; k < n; k++) {
                if (!live(k)) continue;
                if (T[k].text == "{") depth++;
                else if (T[k].text == "}") depth--;
                else if (depth == 0 && T[k].kind == kIdent && T[k].text == "sdf") {
                    size_t o = next_live(k);
                    if (o < n && T[o].text == "(") { defs++; fn = k; }
                }
            }
        }
        do {
            if (has_pp || has_ref_params || name_clash || defs != 1) break;
            size_t ty = prev_live(fn);
            if (ty == n || T[ty].text != "float") break;
            size_t o = next_live(fn), q = next_live(o);
            if (q < n && T[q].text == "const") q = next_live(q);
            if (q >= n || T[q].text != "vec3") break;
            size_t pn = next_live(q);
            if (pn >= n || T[pn].kind != kIdent) break;
            size_t cp = next_live(pn);
            if (cp >= n || T[cp].text != ")") break;
            size_t ob = next_live(cp);
            if (ob >= n || T[ob].text != "{") break;
            size_t cb = match_close(ob);
            if (cb == n) break;
            carve.param = T[pn].text;
            carve.body_open = ob; carve.body_close = cb;

            // ---- declarations, control flow, assignments
            struct Local { size_t decl = 0; std::string type; size_t init_first = 0, init_last = 0; bool has_init = false; int depth = 0; bool counter = false; bool assigned = false; };
            std::map<std::string, Local> locals;
            std::vector<std::pair<size_t, size_t> > for_headers;   // '(' and ')' of each loop header
            bool bad = false;
            int returns = 0; size_t ret_tok = n;
            {
                int depth = 1;
                for (size_t k = next_live(ob); k < cb && !bad; k = next_live(k)) {
                    const std::string& w = T[k].text;
                    if (w == "{") { depth++; continue; }
                    if (w == "}") { depth--; continue; }
                    if (w == "?") { bad = true; break; }
                    if (T[k].kind != kIdent) continue;
                    { size_t pv = prev_live(k); if (pv != n && T[pv].text == ".") continue; }   // field / swizzle
                    if (banned.count(w)) { bad = true; break; }
                    if (w == "return") { returns++; ret_tok = k; if (depth != 1) bad = true; continue; }
                    if (is_for(k)) {
                        size_t ho = next_live(k);
                        if (ho >= cb || T[ho].text != "(") { bad = true; break; }
                        size_t hc = match_close(ho);
                        if (hc == n || hc >= cb) { bad = true; break; }
                        for_headers.push_back({ho, hc});
                        continue;
                    }
                    if (uniform_type_info(w, &bt, &bc)) {
                        size_t nx = next_live(k);
                        if (nx >= cb || T[nx].kind != kIdent) continue;           // constructor call etc.
                        // declaration: TYPE NAME [= init] ;   (one declarator, no arrays)
                        Local L;
                        L.decl = nx; L.type = w; L.depth = depth;
                        const std::string name = T[nx].text;
                        if (locals.count(name) || name == carve.param || uniform_names.count(name)) { bad = true; break; }
                        size_t a = next_live(nx);
                        if (a >= cb) { bad = true; break; }
                        if (T[a].text == "=") {
                            L.has_init = true;
                            L.init_first = next_live(a);
                            int d = 0; size_t e = L.init_first;
                            for (; e < cb; e = next_live(e)) {
                                const std::string& x = T[e].text;
                                if (x == "(" || x == "[") d++;
                                else if (x == ")" || x == "]") d--;
                                else if (d == 0 && x == ",") { bad = true; break; }
                                else if (d == 0 && x == ";") break;
                                if (d < 0) { bad = true; break; }
                            }
                            if (bad || e >= cb || e == L.init_first) { bad = true; break; }
                            L.init_last = prev_live(e);
                        } else if (T[a].text != ";") { bad = true; break; }
                        locals[name] = L;
                        k = nx;
                        continue;
                    }
                }
            }
            if (bad || returns != 1) break;
            // writes to locals / the parameter other than the declaration itself
            std::map<std::string, std::vector<size_t> > writes;
            for (size_t k = next_live(ob); k < cb; k = next_live(k)) {
                if (T[k].kind != kIdent) continue;
                { size_t pv = prev_live(k); if (pv != n && T[pv].text == ".") continue; }
                const std::string& w = T[k].text;
                const bool is_local = locals.count(w) != 0;
                if (!is_local && w != carve.param) continue;
                if (is_local && locals[w].decl == k) continue;
                size_t e = k, nx = next_live(k);
                while (nx < cb && (T[nx].text == "." || T[nx].text == "[")) {
                    if (T[nx].text == ".") { e = next_live(nx); } else { e = match_close(nx); if (e == n) { bad = true; break; } }
                    nx = next_live(e);
                }
                if (bad) break;
                size_t pv = prev_live(k);
                if ((nx < cb && assign_ops.count(T[nx].text)) || (pv != n && (T[pv].text == "++" || T[pv].text == "--"))) writes[w].push_back(k);
            }
            if (bad || writes.count(carve.param)) break;
            // loop headers: only type names, the loop's own counter, uniforms and literals
            for (auto& h : for_headers) {
                std::string counter;
                for (size_t k = next_live(h.first); k < h.second && !bad; k = next_live(k)) {
                    if (T[k].kind != kIdent) continue;
                    const std::string& w = T[k].text;
                    if (uniform_type_info(w, &bt, &bc) || w == "const") continue;
                    auto L = locals.find(w);
                    if (L != locals.end() && L->second.decl > h.first && L->second.decl < h.second) {
                        if (!counter.empty() && counter != w) bad = true;
                        counter = w;
                        continue;
                    }
                    if (uniform_names.count(w)) continue;
                    bad = true;
                }
                if (bad || counter.empty()) { bad = true; break; }
                for (size_t wtok : writes[counter]) if (!(wtok > h.first && wtok < h.second)) bad = true;
                locals[counter].counter = true;
            }
            if (bad) break;
            // position-independent locals, in declaration order
            std::set<std::string> clean;
            for (auto& kv : locals) if (kv.second.counter) clean.insert(kv.first);
            auto idents_clean = [&](size_t first, size_t last) {
                for (size_t k = first; k <= last && k < n; k = next_live(k)) {
                    if (T[k].kind != kIdent) continue;
                    size_t pv = prev_live(k);
                    if (pv != n && T[pv].text == ".") continue;
                    const std::string& w = T[k].text;
                    if (uniform_type_info(w, &bt, &bc)) continue;
                    size_t nx = next_live(k);
                    const bool call = nx < n && T[nx].text == "(";
                    if (call) { if (pure_builtins.count(w)) continue; return false; }
                    if (clean.count(w) || uniform_names.count(w)) continue;
                    return false;
                }
                return true;
            };
            {
                std::vector<std::pair<size_t, std::string> > order;
                for (auto& kv : locals) order.push_back({kv.second.decl, kv.first});
                std::sort(order.begin(), order.end());
                for (auto& o2 : order) {
                    Local& L = locals[o2.second];
                    if (L.counter || !L.has_init || writes.count(o2.second)) continue;
                    if (idents_clean(L.init_first, L.init_last)) clean.insert(o2.second);
                }
            }
            // `length ( ... ) - K` with K a product/quotient of position-independent primaries
            auto accept_len = [&](size_t first, size_t last) -> size_t {     // returns the `length` token or n
                if (T[first].kind != kIdent || T[first].text != "length") return n;
                size_t o2 = next_live(first);
                if (o2 > last || T[o2].text != "(") return n;
                size_t c2 = match_close(o2);
                if (c2 == n || c2 >= last) return n;
                size_t minus = next_live(c2);
                if (minus >= last + 1 || T[minus].text != "-") return n;
                size_t kf = next_live(minus);
                if (kf > last) return n;
                int d = 0;
                for (size_t k = kf; k <= last; k = next_live(k)) {
                    const std::string& x = T[k].text;
                    if (x == "(" || x == "[") d++;
                    else if (x == ")" || x == "]") d--;
                    else if (d == 0 && T[k].kind == kPunct && x != "*" && x != "/" && x != ".") return n;
                    if (d < 0) return n;
                }
                if (d != 0 || !idents_clean(kf, last)) return n;
                return first;
            };
            // ---- pattern B: the iterated difference
            //     float X = A;  ...  X = max(X, -E);  ...  return X;
            // with every E a tree of min() over sdBox(<anything>, B) calls whose half-extents B do not depend on the
            // position (the Menger sponge of the reference's examples: crosses of boxes carved out of a cube, level by
            // level).  The prelude's sdBox (raymarcher.frag:108-112) is length(max(q, 0)) + min(max(q.x, max(q.y, q.z)), 0)
            // with q = abs(p) - b: the first term is >= 0, and every non-NaN q_j >= -b_j (abs() >= 0, rounding is
            // monotonic), so with the NaN-dropping min / max of the pinned semantics the second term is
            // >= min(0, -max_j b_j) whatever p is - NaN and infinite positions included - and so is the rounded sum.
            // Hence -E <= rm_box0-bound U_E = max over its boxes of max(0, max_j b_j) (a NaN E is dropped by the outer
            // max), X never exceeds max(A, U) through these statements, and wherever A > U every max() returns A itself.
            // rm_carve_bound() is sdf's body with X initialised to -3e38 and each sdBox(.., B) replaced by its lower bound
            // rm_box0(B): the same statements then compute U with the scene's own arithmetic for B.
            {
                size_t semi_b = prev_live(cb);
                size_t rxb = next_live(ret_tok);
                const bool ret_is_local = semi_b != n && T[semi_b].text == ";" && rxb < cb && T[rxb].kind == kIdent && locals.count(T[rxb].text) &&
                                          next_live(rxb) == semi_b && !R.functions.count("sdBox");
                bool okB = ret_is_local;
                std::string x = okB ? T[rxb].text : std::string();
                std::map<size_t, size_t> sites;
                if (okB) {
                    Local& XL = locals[x];
                    okB = XL.type == "float" && XL.depth == 1 && XL.has_init && !XL.counter;
                    if (okB) {
                        // A: the parameter, uniforms, literals, pure built-ins and the prelude's sdBox
                        std::set<std::string> saved = clean;
                        clean.clear();
                        clean.insert(carve.param);
                        for (size_t k = XL.init_first; k <= XL.init_last && k < n && okB; k = next_live(k)) {
                            if (T[k].kind != kIdent) continue;
                            size_t pv = prev_live(k);
                            if (pv != n && T[pv].text == ".") continue;
                            const std::string& w = T[k].text;
                            if (uniform_type_info(w, &bt, &bc)) continue;
                            size_t nx = next_live(k);
                            const bool call = nx < n && T[nx].text == "(";
                            if (call) { if (!(pure_builtins.count(w) || w == "sdBox")) okB = false; continue; }
                            if (!(w == carve.param || uniform_names.count(w))) okB = false;
                        }
                        clean = saved;
                    }
                    // E := min ( E , E ) | sdBox ( <expr> , B )        (token range, inclusive)
                    std::function<bool(size_t, size_t)> accept_e = [&](size_t first, size_t last) -> bool {
                        if (first >= n || last >= n || first > last || T[first].kind != kIdent) return false;
                        size_t o2 = next_live(first);
                        if (o2 > last || T[o2].text != "(" || match_close(o2) != last) return false;
                        size_t cm = n; int cms = 0, d = 0;
                        for (size_t q2 = next_live(o2); q2 < last; q2 = next_live(q2)) {
                            const std::string& t2 = T[q2].text;
                            if (t2 == "(" || t2 == "[") d++;
                            else if (t2 == ")" || t2 == "]") d--;
                            else if (d == 0 && t2 == ",") { cms++; cm = q2; }
                            if (assign_ops.count(t2)) return false;                    // no side effects inside
                            if (T[q2].kind == kIdent && t2 == x) return false;
                        }
                        if (cms != 1) return false;
                        if (T[first].text == "min") return accept_e(next_live(o2), prev_live(cm)) && accept_e(next_live(cm), prev_live(last));
                        if (T[first].text != "sdBox") return false;
                        if (!idents_clean(next_live(cm), prev_live(last))) return false;   // B: position-independent
                        sites[first] = cm;
                        return true;
                    };
                    // every other mention of X:  X = max ( X , - E ) ;   or   X = max ( - E , X ) ;
                    for (size_t k = next_live(ob); k < cb && okB; k = next_live(k)) {
                        if (T[k].kind != kIdent || T[k].text != x || k == locals[x].decl || k == rxb) continue;
                        { size_t pvf = prev_live(k); if (pvf != n && T[pvf].text == ".") { okB = false; break; } }
                        size_t pv = prev_live(k);
                        if (pv == n || !(T[pv].text == ";" || T[pv].text == "{" || T[pv].text == "}" || T[pv].text == ")")) { okB = false; break; }
                        if (T[pv].text == ")") {
                            bool hdr = false;
                            for (auto& h : for_headers) if (h.second == pv) hdr = true;
                            if (!hdr) { okB = false; break; }
                        }
                        size_t eq = next_live(k), mx = next_live(eq), o2 = next_live(mx);
                        if (o2 >= cb || T[eq].text != "=" || T[mx].text != "max" || T[o2].text != "(") { okB = false; break; }
                        size_t c2 = match_close(o2);
                        if (c2 == n || c2 >= cb || T[next_live(c2)].text != ";") { okB = false; break; }
                        size_t cm = n; int cms = 0;
                        { int d = 0; for (size_t q2 = next_live(o2); q2 < c2; q2 = next_live(q2)) { const std::string& t2 = T[q2].text; if (t2 == "(" || t2 == "[") d++; else if (t2 == ")" || t2 == "]") d--; else if (d == 0 && t2 == ",") { cms++; cm = q2; } } }
                        if (cms != 1) { okB = false; break; }
                        size_t x1f = next_live(o2), x1l = prev_live(cm), x2f = next_live(cm), x2l = prev_live(c2);
                        size_t ef, el;
                        if (x1f == x1l && T[x1f].text == x) { ef = x2f; el = x2l; }
                        else if (x2f == x2l && T[x2f].text == x) { ef = x1f; el = x1l; }
                        else { okB = false; break; }
                        if (T[ef].text != "-") { okB = false; break; }
                        if (!accept_e(next_live(ef), el)) { okB = false; break; }
                        k = c2;
                    }
                    if (okB && sites.empty()) okB = false;
                    if (okB && writes.count(x)) {
                        // (every write found above is one of the accepted statements: anything else failed the walk)
                        for (size_t wtok : writes[x]) {
                            size_t eq = next_live(wtok);
                            if (eq >= cb || T[eq].text != "=") okB = false;
                        }
                    }
                }
                if (okB) {
                    carve.ok = true;
                    carve.boxes = true;
                    carve.clean = clean;
                    carve.ret_tok = ret_tok; carve.ret_semi = semi_b;
                    carve.m_name = x;
                    carve.ea_first = locals[x].init_first; carve.ea_last = locals[x].init_last;
                    carve.x_init_first = locals[x].init_first; carve.x_init_last = locals[x].init_last;
                    carve.box_sites = sites;
                    break;
                }
            }
            // ---- the return statement
            size_t semi_end = prev_live(cb);
            if (semi_end == n || T[semi_end].text != ";") break;
            size_t rx = next_live(ret_tok);
            size_t max_tok = n, stmt_semi = semi_end;
            std::string assigned_to;
            if (rx < cb && T[rx].text == "max") {
                max_tok = rx;
            } else if (rx < cb && T[rx].kind == kIdent && next_live(rx) == semi_end) {
                // V = max(..); return V;
                assigned_to = T[rx].text;
                size_t ps = prev_live(ret_tok);
                if (ps == n || T[ps].text != ";") break;
                stmt_semi = ps;
                // walk back to the start of that statement
                size_t st = ps; int d = 0; bool found = false;
                while (true) {
                    size_t pv = prev_live(st);
                    if (pv == n || pv <= ob) { found = (pv == ob); break; }
                    const std::string& x = T[pv].text;
                    if (x == ")" || x == "]") d++;
                    else if (x == "(" || x == "[") d--;
                    else if (d == 0 && (x == ";" || x == "{" || x == "}")) { found = true; break; }
                    st = pv;
                }
                if (!found) break;
                size_t a = st;
                if (T[a].text == "float") a = next_live(a);
                if (T[a].text != assigned_to) break;
                size_t eq = next_live(a);
                if (T[eq].text != "=") break;
                max_tok = next_live(eq);
                if (max_tok >= cb || T[max_tok].text != "max") break;
                // that statement must sit at the function's top level
                int depth = 1; bool top = true;
                for (size_t k = next_live(ob); k < st; k = next_live(k)) { if (T[k].text == "{") depth++; else if (T[k].text == "}") depth--; }
                top = depth == 1;
                if (!top) break;
            } else break;
            size_t mo = next_live(max_tok);
            if (mo >= cb || T[mo].text != "(") break;
            size_t mc = match_close(mo);
            if (mc == n || next_live(mc) != stmt_semi) break;
            if (assigned_to.empty() && stmt_semi != semi_end) break;
            size_t comma = n; int commas = 0;
            { int d = 0; for (size_t k = next_live(mo); k < mc; k = next_live(k)) { const std::string& x = T[k].text; if (x == "(" || x == "[") d++; else if (x == ")" || x == "]") d--; else if (d == 0 && x == ",") { commas++; comma = k; } } }
            if (commas != 1) break;
            size_t a1f = next_live(mo), a1l = prev_live(comma), a2f = next_live(comma), a2l = prev_live(mc);
            auto neg_ident = [&](size_t f, size_t l) -> std::string { return (T[f].text == "-" && next_live(f) == l && T[l].kind == kIdent) ? T[l].text : std::string(); };
            std::string m = neg_ident(a2f, a2l);
            size_t eaf = a1f, eal = a1l;
            if (m.empty() || !locals.count(m)) { m = neg_ident(a1f, a1l); eaf = a2f; eal = a2l; }
            if (m.empty() || !locals.count(m)) break;
            Local& ML = locals[m];
            if (ML.type != "float" || ML.depth != 1 || !ML.has_init) break;
            {   // initialiser: [+-] literal
                size_t v = ML.init_first;
                if (T[v].text == "-" || T[v].text == "+") v = next_live(v);
                if (v != ML.init_last || T[v].kind != kNumber) break;
            }
            // A: the parameter, uniforms, literals and pure built-ins only
            {
                std::set<std::string> saved = clean;
                clean.clear();
                clean.insert(carve.param);
                const bool ok = idents_clean(eaf, eal);
                clean = saved;
                if (!ok) break;
            }
            // ---- every other mention of M: `M = min(X, M);` / `M = min(M, X);`
            std::set<size_t> accounted;
            accounted.insert(ML.decl);
            for (size_t k = next_live(mo); k < mc; k = next_live(k)) if (T[k].kind == kIdent && T[k].text == m) accounted.insert(k);
            if (assigned_to == m) { accounted.insert(prev_live(prev_live(max_tok))); accounted.insert(rx); }
            for (size_t k = next_live(ob); k < cb && !bad; k = next_live(k)) {
                if (T[k].kind != kIdent || T[k].text != m || accounted.count(k)) continue;
                size_t pv = prev_live(k);
                if (pv == n || !(T[pv].text == ";" || T[pv].text == "{" || T[pv].text == "}" || T[pv].text == ")")) { bad = true; break; }
                if (T[pv].text == ")") {
                    // only as the un-braced body of a loop:  for (...) M = min(..);
                    bool hdr = false;
                    for (auto& h : for_headers) if (h.second == pv) hdr = true;
                    if (!hdr) { bad = true; break; }
                }
                size_t eq = next_live(k), mn = next_live(eq), o2 = next_live(mn);
                if (o2 >= cb || T[eq].text != "=" || T[mn].text != "min" || T[o2].text != "(") { bad = true; break; }
                size_t c2 = match_close(o2);
                if (c2 == n || c2 >= cb || T[next_live(c2)].text != ";") { bad = true; break; }
                size_t cm = n; int cms = 0;
                { int d = 0; for (size_t q2 = next_live(o2); q2 < c2; q2 = next_live(q2)) { const std::string& x = T[q2].text; if (x == "(" || x == "[") d++; else if (x == ")" || x == "]") d--; else if (d == 0 && x == ",") { cms++; cm = q2; } } }
                if (cms != 1) { bad = true; break; }
                size_t x1f = next_live(o2), x1l = prev_live(cm), x2f = next_live(cm), x2l = prev_live(c2);
                size_t xf, xl, mtok;
                if (x2f == x2l && T[x2f].text == m) { xf = x1f; xl = x1l; mtok = x2f; }
                else if (x1f == x1l && T[x1f].text == m) { xf = x2f; xl = x2l; mtok = x1f; }
                else { bad = true; break; }
                for (size_t q2 = xf; q2 <= xl; q2 = next_live(q2)) if (T[q2].kind == kIdent && T[q2].text == m) bad = true;
                if (bad) break;
                size_t len_tok = n;
                if (xf == xl && T[xf].kind == kIdent && locals.count(T[xf].text)) {
                    Local& X = locals[T[xf].text];
                    if (X.type == "float" && X.has_init && !writes.count(T[xf].text) && !X.counter) len_tok = accept_len(X.init_first, X.init_last);
                } else len_tok = accept_len(xf, xl);
                if (len_tok == n) { bad = true; break; }
                carve.len_tokens.push_back(len_tok);
                accounted.insert(k);
                accounted.insert(mtok);
            }
            if (bad) break;
            if (writes.count(m)) {
                // every write to M is one of the accepted statements (or the final assignment)
                for (size_t wtok : writes[m]) if (!accounted.count(wtok)) bad = true;
            }
            if (bad) break;
            carve.ok = true;
            carve.clean = clean;
            carve.ret_tok = ret_tok; carve.ret_semi = semi_end;
            carve.m_name = m;
            carve.ea_first = eaf; carve.ea_last = eal;
            carve.max_first = max_tok; carve.max_close = mc;
        } while (false);
    }

    // ---- pass 2: domain-repetition idiom -----------------------------------------------------
    // `mod(X + H1, S) - H2` -> rm_rep(X, H1, S, H2) and `mod(X, S) - H2` -> rm_rep0(X, S, H2), where the
    // whole pattern is one operand of nothing tighter than the binary minus.  glsl_rt.h defines both
    // helpers: the exact policy evaluates the expression exactly as written (same operations, same
    // order), the fast policy turns a centred cell (H2 == S/2) into a centred remainder.
    {
        auto live = [&](size_t k) { return k < n && !T[k].drop && T[k].kind != kPP; };
        auto next_live = [&](size_t k) { k++; while (k < n && !live(k)) k++; return k; };
        auto prev_live = [&](size_t k) -> size_t { while (k > 0) { k--; if (live(k)) return k; } return n; };
        auto match_close = [&](size_t open) -> size_t {   // index of the ')' / ']' matching T[open]
            int d = 0;
            for (size_t k = open; k < n; k++) {
                if (!live(k)) continue;
                if (T[k].text == "(" || T[k].text == "[") d++;
                else if (T[k].text == ")" || T[k].text == "]") { d--; if (d == 0) return k; }
            }
            return n;
        };
        // primary: number | identifier [call] | parenthesised, each followed by .swizzle / [index]
        auto parse_primary = [&](size_t k) -> size_t {   // returns index of the last token, or n
            if (!live(k)) return n;
            size_t last;
            if (T[k].kind == kNumber) last = k;
            else if (T[k].kind == kIdent) {
                last = k;
                size_t q = next_live(k);
                if (q < n && T[q].text == "(") { last = match_close(q); if (last == n) return n; }
            } else if (T[k].text == "(") { last = match_close(k); if (last == n) return n; }
            else return n;
            for (;;) {
                size_t q = next_live(last);
                if (q < n && T[q].text == ".") { size_t f = next_live(q); if (f < n && T[f].kind == kIdent) { last = f; continue; } return n; }
                if (q < n && T[q].text == "[") { size_t c = match_close(q); if (c == n) return n; last = c; continue; }
                break;
            }
            return last;
        };
        static const std::set<std::string> ok_before = {"(", ",", "=", "return", "?", ":", ";", "{", "}", "+=", "-=", "*=", "/="};
        static const std::set<std::string> low_prec = {"<", ">", "<=", ">=", "==", "!=", "&&", "||", "!=", "?", ":", "=", "&", "|", "^", "<<", ">>",
                                                        "+=", "-=", "*=", "/="};
        for (size_t m = 0; m < n; m++) {
            if (!live(m) || T[m].kind != kIdent || T[m].text != "mod") continue;
            size_t open = next_live(m);
            if (open >= n || T[open].text != "(") continue;
            size_t pv = prev_live(m);
            if (pv != n && !ok_before.count(T[pv].text)) continue;
            if (pv != n && T[pv].text == "(") {
                // `f(mod(..) - h)` is fine, `(mod(..)) - h` is handled as written; but `x.f(mod` cannot occur in GLSL
            }
            size_t close = match_close(open);
            if (close == n) continue;
            // split the two arguments at the top-level comma
            size_t comma = n; int d = 0; bool bad = false; int commas = 0;
            size_t last_add = n;      // last top-level binary + or - of argument 1
            for (size_t k = next_live(open); k < close; k = next_live(k)) {
                const std::string& w = T[k].text;
                if (w == "(" || w == "[") d++;
                else if (w == ")" || w == "]") d--;
                else if (d == 0 && w == ",") { commas++; if (comma == n) comma = k; }
                else if (d == 0 && comma == n) {
                    if (low_prec.count(w)) bad = true;
                    if (w == "+" || w == "-") {
                        size_t b = prev_live(k);
                        bool binary = b != n && b != open && (T[b].kind == kIdent || T[b].kind == kNumber || T[b].text == ")" || T[b].text == "]");
                        if (binary) last_add = k;
                    }
                } else if (d == 0 && comma != n && low_prec.count(w)) bad = true;
            }
            if (bad || commas != 1 || comma == n) continue;
            if (last_add != n && T[last_add].text != "+") continue;
            // what follows: `- H2` with H2 a multiplicative chain of primaries
            size_t minus = next_live(close);
            if (minus >= n || T[minus].text != "-") continue;
            size_t h2_last = parse_primary(next_live(minus));
            if (h2_last == n) continue;
            for (;;) {
                size_t q = next_live(h2_last);
                if (q < n && (T[q].text == "*" || T[q].text == "/")) {
                    size_t e = parse_primary(next_live(q));
                    if (e == n) { h2_last = n; break; }
                    h2_last = e;
                    continue;
                }
                break;
            }
            if (h2_last == n) continue;
            {   // the operand after H2 must not bind tighter than '-'
                size_t q = next_live(h2_last);
                if (q < n && (T[q].text == "%" || T[q].text == "." || T[q].text == "[" || T[q].text == "(")) continue;
            }
            // Bounded-floor sites.  In a carved scene (pass 1b: straight-line sdf body, parameter never written) a
            // repetition whose operand is the position parameter ITSELF and whose H1 and S are position-independent
            // becomes rm_rep_b / rm_rep0_b: the march kernels evaluate its floor() on the FP32 pipe without a range
            // guard, having checked once per evaluation that |position| <= rm_floor_plim() - the largest coordinate
            // for which every such site's floor argument stays within 2^22 (emitted below from the same H1 and S).
            bool bounded = false;
            if (carve.ok && m > carve.body_open && m < carve.body_close) {
                const size_t x_end = last_add != n ? last_add : comma;
                const size_t xf = next_live(open);
                auto range_clean = [&](size_t first, size_t end) {      // identifiers of [first, end)
                    char bt2; int bc2;
                    for (size_t k = first; k < end; k = next_live(k)) {
                        if (T[k].kind != kIdent) continue;
                        size_t pv2 = prev_live(k);
                        if (pv2 != n && T[pv2].text == ".") continue;
                        const std::string& w = T[k].text;
                        if (uniform_type_info(w, &bt2, &bc2)) continue;
                        size_t nx = next_live(k);
                        if (nx < n && T[nx].text == "(") { if (pure_builtins.count(w)) continue; return false; }
                        if (carve.clean.count(w) || uniform_names.count(w)) continue;
                        return false;
                    }
                    return true;
                };
                bounded = xf < x_end && T[xf].text == carve.param && next_live(xf) == x_end &&
                          (last_add == n || range_clean(next_live(last_add), comma)) && range_clean(next_live(comma), close);
            }
            if (bounded) carve.rep_sites.push_back(m);
            if (last_add != n) { T[m].text = bounded ? "rm_rep_b" : "rm_rep"; T[last_add].text = ","; }
            else T[m].text = bounded ? "rm_rep0_b" : "rm_rep0";
            T[close].text = ",";
            T[minus].drop = true;
            T[h2_last].text += ")";
        }
    }

    // ---- emit -------------------------------------------------------------------------------
    std::string out;
    out.reserve(glsl.size() + 256);
    for (const Token& t : T) {
        out += t.ws;
        if (t.drop) continue;
        // separate tokens that would otherwise paste after a dropped neighbour
        if (!out.empty() && is_ident_char(out.back()) && !t.text.empty() && is_ident_char(t.text[0]) && t.ws.empty()) out += ' ';
        out += t.text;
    }
    out += trailing;
    R.body = out;

    if (carve.ok) {
        // helper functions (members of the fragment struct, after the scene): token texts as they stand
        // after pass 2, so the domain-repetition rewrite applies to them exactly as it does to sdf()
        auto live = [&](size_t k) { return k < n && !T[k].drop && T[k].kind != kPP; };
        std::string outer, bound;
        for (size_t k = carve.ea_first; k <= carve.ea_last; k++) if (live(k)) { outer += ' '; outer += T[k].text; }
        std::set<size_t> lens(carve.len_tokens.begin(), carve.len_tokens.end());
        for (size_t k = carve.body_open + 1; k < carve.body_close; k++) {
            if (!live(k)) continue;
            bound += ' ';
            if (carve.boxes) {
                // pattern B: X starts below everything, every accepted sdBox(arg, B) becomes its lower bound rm_box0(B)
                if (k == carve.x_init_first) { bound += "-3.0e38f"; k = carve.x_init_last; continue; }
                auto site = carve.box_sites.find(k);
                if (site != carve.box_sites.end()) { bound += "rm_box0 ("; k = site->second; continue; }
                bound += T[k].text;
                continue;
            }
            if (k == carve.max_first) { bound += "(-" + carve.m_name + ")"; k = carve.max_close; continue; }
            bound += lens.count(k) ? std::string("rm_len0") : T[k].text;
        }
        R.carve_text = "\nfloat rm_carve_outer(vec3 " + carve.param + ") { return" + outer + "; }\n" +
                       "float rm_carve_bound() { vec3 " + carve.param + " = vec3(0.0f);" + bound + " }\n";
        if (!carve.rep_sites.empty()) {
            // rm_floor_plim(): sdf's body once more with every bounded site replaced by rm_plim_site(rm_plim, ..), which
            // lowers rm_plim to the site's coordinate limit (glsl_rt.h), and `return rm_plim` for the return statement
            std::set<size_t> sites(carve.rep_sites.begin(), carve.rep_sites.end());
            std::string plim;
            for (size_t k = carve.body_open + 1; k < carve.body_close; k++) {
                if (!live(k)) continue;
                plim += ' ';
                if (k == carve.ret_tok) { plim += "return rm_plim ;"; break; }
                if (sites.count(k)) {
                    plim += T[k].text == "rm_rep_b" ? "rm_plim_site" : "rm_plim_site0";
                    // the '(' that follows is kept; the accumulator becomes the first argument
                    size_t o = k + 1; while (o < n && !live(o)) o++;
                    plim += " ( rm_plim ,";
                    k = o;
                    continue;
                }
                plim += lens.count(k) ? std::string("rm_len0") : T[k].text;
            }
            R.carve_text += "float rm_floor_plim() { float rm_plim = 3.0e38f; vec3 " + carve.param + " = vec3(0.0f);" + plim + " }\n";
            R.floor_sites = (int)carve.rep_sites.size();
        }
    }
    R.ok = true;
    return R;
}

}  // namespace rmb
