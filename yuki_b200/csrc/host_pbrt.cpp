// pbrt-v3 scene loader for the host side of the B200 backend: the step before the hot path for config 1 ("Cornell-box
// pbrt-v3 scene"). Restates the subset yuki/src/scene/pbrt/{lexer,mod,param_set,cie}.rs accepts, with its defaults and
// quirks, and produces the same host scene description the programmatic scenes use (yk_host_scene_desc) plus the camera
// parameters and film resolution:
//   * lexer: pbrtlex rules of lexer.rs:66-361 (# comments, "strings" with \-escapes, [ ], keywords, f64 numbers);
//   * directives: ActiveTransform, AreaLightSource (ignored, mod.rs:502), AttributeBegin/End, Camera "perspective",
//     Film, Integrator / Sampler (ignored), Include, LightSource infinite|distant|point, LookAt, Material,
//     MakeNamedMaterial, NamedMaterial, Rotate, Scale, Translate, Shape sphere|trianglemesh|plymesh, Texture
//     "spectrum" "imagemap", TransformBegin/End (TransformEnd pops the *graphics state*, mod.rs:749-755), WorldBegin/End;
//     every other directive is the reference's UnimplementedToken error;
//   * parameter types: bool, float (float uv = pairs), integer, string, color/rgb, spectrum (inline pairs or file,
//     converted with the Wyman-Sloan-Shirley CIE fits, cie.rs), point, normal, blackbody (dropped), texture;
//   * materials glass / glossy / matte (sigma through to_radians twice, mod.rs:904-907) / metal (copper defaults);
//     unknown types fall back to grey matte; fov is vertical unless the film is taller than wide (mod.rs:827-835).
//   * Camera "perspective" also yields pbrt-v3's lensradius (default 0) and focaldistance (default 1e6), which the reference
//     ignores; a caller renders with them through YK_RENDER_THIN_LENS.
// Image textures are decoded here for PNG only (the reference uses the `image` crate, which is not vendored): 8/16-bit
// RGB / RGBA / palette, non-interlaced; other layouts are the reference's "Unsupported image format".
#include <zlib.h>

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <sstream>
#include <string>
#include <vector>

#include "host_loader.h"
#include "host_math.h"
#include "yuki_gpu.h"
#include "yk_guard.h"

int yk_set_error(int code, const std::string& msg);  // host_scene.cpp
extern "C" int yk_ply_load(const char* path, yk_ply** out);
extern "C" void yk_ply_view(const yk_ply*, yk_ply_data* out);
extern "C" void yk_ply_destroy(yk_ply*);

using namespace ykh;

namespace {

// ---- lexer (lexer.rs) ------------------------------------------------------------------------------------------------
enum class Tok {
    Number, String, LeftBracket, RightBracket, End,
    Accelerator, ActiveTransform, All, AreaLightSource, AttributeBegin, AttributeEnd, Camera, ConcatTransform, CoordinateSystem,
    CoordSysTransform, EndTime, Film, Identity, Include, LightSource, LookAt, MakeNamedMaterial, MakeNamedMedium, Material,
    MediumInterface, NamedMaterial, ObjectBegin, ObjectEnd, ObjectInstance, PixelFilter, ReverseOrientation, Rotate, Sampler, Scale,
    Shape, StartTime, Integrator, Texture, Transform, TransformBegin, TransformEnd, TransformTimes, Translate, WorldBegin, WorldEnd
};
const std::map<std::string, Tok>& keywords() {
    static const std::map<std::string, Tok> k = {
        {"Accelerator", Tok::Accelerator}, {"ActiveTransform", Tok::ActiveTransform}, {"All", Tok::All},
        {"AreaLightSource", Tok::AreaLightSource}, {"AttributeBegin", Tok::AttributeBegin}, {"AttributeEnd", Tok::AttributeEnd},
        {"Camera", Tok::Camera}, {"ConcatTransform", Tok::ConcatTransform}, {"CoordinateSystem", Tok::CoordinateSystem},
        {"CoordSysTransform", Tok::CoordSysTransform}, {"EndTime", Tok::EndTime}, {"Film", Tok::Film}, {"Identity", Tok::Identity},
        {"Include", Tok::Include}, {"Integrator", Tok::Integrator}, {"LightSource", Tok::LightSource}, {"LookAt", Tok::LookAt},
        {"MakeNamedMedium", Tok::MakeNamedMedium}, {"MakeNamedMaterial", Tok::MakeNamedMaterial}, {"Material", Tok::Material},
        {"MediumInterface", Tok::MediumInterface}, {"NamedMaterial", Tok::NamedMaterial}, {"ObjectBegin", Tok::ObjectBegin},
        {"ObjectEnd", Tok::ObjectEnd}, {"ObjectInstance", Tok::ObjectInstance}, {"PixelFilter", Tok::PixelFilter},
        {"ReverseOrientation", Tok::ReverseOrientation}, {"Rotate", Tok::Rotate}, {"Sampler", Tok::Sampler}, {"Scale", Tok::Scale},
        {"Shape", Tok::Shape}, {"StartTime", Tok::StartTime}, {"Texture", Tok::Texture}, {"TransformBegin", Tok::TransformBegin},
        {"TransformEnd", Tok::TransformEnd}, {"TransformTimes", Tok::TransformTimes}, {"Transform", Tok::Transform},
        {"Translate", Tok::Translate}, {"WorldBegin", Tok::WorldBegin}, {"WorldEnd", Tok::WorldEnd}};
    return k;
}
struct Token {
    Tok kind = Tok::End;
    double number = 0;
    std::string text;  // string contents, or the keyword / offending identifier
};
struct Lexer {
    std::string input, path, parent;
    size_t pos = 0;
    size_t line = 1;
    std::string error;

    bool next(Token* t) {  // false on error (message in `error`); Tok::End at end of input
        for (;;) {  // whitespace and comments
            if (pos >= input.size()) { t->kind = Tok::End; return true; }
            const char c = input[pos];
            if (c == ' ' || c == '\t' || c == '\r' || c == '\n') { line += c == '\n'; ++pos; continue; }
            if (c == '#') {
                while (pos < input.size() && input[pos] != '\n' && input[pos] != '\r') ++pos;
                if (pos >= input.size()) { t->kind = Tok::End; return true; }
                continue;
            }
            break;
        }
        const char c = input[pos];
        if (c == '"') {
            const size_t start = ++pos;
            for (;;) {
                if (pos >= input.size()) return fail("UnexpectedEndOfInput");
                const char s = input[pos++];
                if (s == '"') break;
                if (s == '\\') { if (pos >= input.size()) return fail("UnexpectedEndOfInput"); ++pos; }
                else if (s == '\n') return fail("UnterminatedString");
            }
            t->kind = Tok::String;
            t->text = input.substr(start, pos - 1 - start);
            return true;
        }
        if (c == '[') { ++pos; t->kind = Tok::LeftBracket; return true; }
        if (c == ']') { ++pos; t->kind = Tok::RightBracket; return true; }
        const size_t start = pos;
        while (pos < input.size()) {
            const char s = input[pos];
            if (s == ' ' || s == '\t' || s == '\r' || s == '\n' || s == ']') break;
            ++pos;
        }
        if (pos >= input.size()) { t->kind = Tok::End; return true; }  // lexer.rs:210-218: an identifier cut by EOF is dropped
        const std::string word = input.substr(start, pos - start);
        auto kw = keywords().find(word);
        if (kw != keywords().end()) { t->kind = kw->second; t->text = word; return true; }
        const char f = word[0];
        if (f == '-' || f == '.' || (f >= '0' && f <= '9')) {
            char* end = nullptr;
            const double v = std::strtod(word.c_str(), &end);
            if (end != word.c_str() + word.size()) return fail("InvalidNumber");
            t->kind = Tok::Number;
            t->number = v;
            return true;
        }
        return fail("UnknownIdentifier '" + word + "'");
    }
    bool fail(const std::string& what) {
        std::ostringstream o;
        o << path << ": line " << line << ": " << what;
        error = o.str();
        return false;
    }
};

// ---- ParamSet (param_set.rs) ------------------------------------------------------------------------------------------
template <class T>
struct Item { std::string name; std::vector<T> values; };
struct ParamSet {
    std::vector<Item<bool>> bools;
    std::vector<Item<float>> f32s;
    std::vector<Item<int32_t>> i32s;
    std::vector<Item<f3>> spectra, points, normals;
    std::vector<Item<std::pair<float, float>>> uvs;
    std::vector<Item<std::string>> strings;
    template <class T>
    static T one(const std::vector<Item<T>>& v, const std::string& n, T def) {  // single-value finders need exactly one value
        for (const auto& p : v) if (p.name == n && p.values.size() == 1) return p.values[0];
        return def;
    }
    template <class T>
    static const std::vector<T>* many(const std::vector<Item<T>>& v, const std::string& n) {
        for (const auto& p : v) if (p.name == n) return &p.values;
        return nullptr;
    }
};

// ---- spectra (mod.rs:979-1016, cie.rs) -----------------------------------------------------------------------------
float x_fit(float l) {
    const float t1 = (l - 442.0f) * (l < 442.0f ? 0.0624f : 0.0374f), t2 = (l - 599.8f) * (l < 599.8f ? 0.0264f : 0.0323f);
    const float t3 = (l - 501.1f) * (l < 501.1f ? 0.0490f : 0.0382f);
    return 0.362f * std::exp(-0.5f * t1 * t1) + 1.056f * std::exp(-0.5f * t2 * t2) - 0.065f * std::exp(-0.5f * t3 * t3);
}
float y_fit(float l) {
    const float t1 = (l - 568.8f) * (l < 568.8f ? 0.0213f : 0.0247f), t2 = (l - 530.9f) * (l < 530.9f ? 0.0613f : 0.0322f);
    return 0.821f * std::exp(-0.5f * t1 * t1) + 0.286f * std::exp(-0.5f * t2 * t2);
}
float z_fit(float l) {
    const float t1 = (l - 437.0f) * (l < 437.0f ? 0.0845f : 0.0278f), t2 = (l - 459.0f) * (l < 459.0f ? 0.0385f : 0.0725f);
    return 1.217f * std::exp(-0.5f * t1 * t1) + 0.681f * std::exp(-0.5f * t2 * t2);
}
// Riemann sum in the given order (the reference's "sort first" branch discards its result, mod.rs:984-998)
f3 spectrum_to_rgb(const std::vector<float>& lambda, const std::vector<float>& samples) {
    float x = 0, y = 0, z = 0;
    for (size_t i = 0; i < lambda.size(); ++i) {
        x += x_fit(lambda[i]) * samples[i];
        y += y_fit(lambda[i]) * samples[i];
        z += z_fit(lambda[i]) * samples[i];
    }
    const float scale = (lambda.back() - lambda.front()) / (float)lambda.size();
    x *= scale; y *= scale; z *= scale;
    return mk3(3.240479f * x - 1.537150f * y - 0.498535f * z, -0.969256f * x + 1.875991f * y + 0.041556f * z,
               0.055648f * x - 0.204043f * y + 1.057311f * z);
}
// Copper's measured n / k (pbrt-v3's defaults, mod.rs:1027-1105): wavelength, n, k
const float kCopper[56][3] = {
    {298.7570554f, 1.400313f, 1.662125f}, {302.4004341f, 1.38f, 1.687f}, {306.1337728f, 1.358438f, 1.703313f}, {309.960445f, 1.34f, 1.72f},
    {313.8839949f, 1.329063f, 1.744563f}, {317.9081487f, 1.325f, 1.77f}, {322.036826f, 1.3325f, 1.791625f}, {326.2741526f, 1.34f, 1.81f},
    {330.6244747f, 1.334375f, 1.822125f}, {335.092373f, 1.325f, 1.834f}, {339.6826795f, 1.317812f, 1.85175f}, {344.4004944f, 1.31f, 1.872f},
    {349.2512056f, 1.300313f, 1.89425f}, {354.2405086f, 1.29f, 1.916f}, {359.374429f, 1.281563f, 1.931688f}, {364.6593471f, 1.27f, 1.95f},
    {370.1020239f, 1.249062f, 1.972438f}, {375.7096303f, 1.225f, 2.015f}, {381.4897785f, 1.2f, 2.121562f}, {387.4505563f, 1.18f, 2.21f},
    {393.6005651f, 1.174375f, 2.177188f}, {399.9489613f, 1.175f, 2.13f}, {406.5055016f, 1.1775f, 2.160063f}, {413.2805933f, 1.18f, 2.21f},
    {420.2853492f, 1.178125f, 2.249938f}, {427.5316483f, 1.175f, 2.289f}, {435.0322035f, 1.172812f, 2.326f}, {442.8006357f, 1.17f, 2.362f},
    {450.8515564f, 1.165312f, 2.397625f}, {459.2006593f, 1.16f, 2.433f}, {467.8648226f, 1.155312f, 2.469187f}, {476.8622231f, 1.15f, 2.504f},
    {486.2124627f, 1.142812f, 2.535875f}, {495.936712f, 1.135f, 2.564f}, {506.0578694f, 1.131562f, 2.589625f}, {516.6007417f, 1.12f, 2.605f},
    {527.5922468f, 1.092437f, 2.595562f}, {539.0616435f, 1.04f, 2.583f}, {551.0407911f, 0.950375f, 2.5765f}, {563.5644455f, 0.826f, 2.599f},
    {576.6705953f, 0.645875f, 2.678062f}, {590.4008476f, 0.468f, 2.809f}, {604.8008683f, 0.35125f, 3.01075f}, {619.92089f, 0.272f, 3.24f},
    {635.8162974f, 0.230813f, 3.458187f}, {652.5483053f, 0.214f, 3.67f}, {670.1847459f, 0.20925f, 3.863125f}, {688.8009889f, 0.213f, 4.05f},
    {708.4810171f, 0.21625f, 4.239563f}, {729.3186941f, 0.223f, 4.43f}, {751.4192606f, 0.2365f, 4.619563f}, {774.9011125f, 0.25f, 4.817f},
    {799.8979226f, 0.254188f, 5.034125f}, {826.5611867f, 0.26f, 5.26f}, {855.0632966f, 0.28f, 5.485625f}, {885.6012714f, 0.3f, 5.717f}};
f3 copper_rgb(int column) {
    std::vector<float> l(56), s(56);
    for (int i = 0; i < 56; ++i) { l[i] = kCopper[i][0]; s[i] = kCopper[i][column]; }
    return spectrum_to_rgb(l, s);
}

// ---- PNG -> RGB f32 (stands in for image::io::Reader::decode + load_image_spectrum_f32, image_texture.rs:113-141) ----
bool decode_png(const std::string& path, uint32_t* w_out, uint32_t* h_out, std::vector<float>* rgb, std::string* why) {
    std::ifstream f(path, std::ios::binary);
    if (!f) { *why = "could not open image '" + path + "'"; return false; }
    std::vector<uint8_t> d((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
    if (d.size() < 8 || std::memcmp(d.data(), sig, 8) != 0) { *why = "Unsupported image format (only PNG is decoded)"; return false; }
    auto be32 = [&](size_t p) { return (uint32_t)d[p] << 24 | (uint32_t)d[p + 1] << 16 | (uint32_t)d[p + 2] << 8 | d[p + 3]; };
    uint32_t w = 0, h = 0, depth = 0, ctype = 0, interlace = 0;
    std::vector<uint8_t> idat, palette;
    for (size_t p = 8; p + 12 <= d.size();) {
        const uint32_t len = be32(p);
        const std::string type((const char*)&d[p + 4], 4);
        if (p + 12 + len > d.size()) { *why = "PNG: truncated chunk"; return false; }
        const uint8_t* body = &d[p + 8];
        if (type == "IHDR") { w = be32(p + 8); h = be32(p + 12); depth = body[8]; ctype = body[9]; interlace = body[12]; }
        else if (type == "PLTE") palette.assign(body, body + len);
        else if (type == "IDAT") idat.insert(idat.end(), body, body + len);
        else if (type == "IEND") break;
        p += 12 + len;
    }
    if (!w || !h || interlace) { *why = interlace ? "PNG: interlaced images are not decoded" : "PNG: missing IHDR"; return false; }
    int channels = 0;
    if (ctype == 2) channels = 3; else if (ctype == 6) channels = 4; else if (ctype == 3) channels = 1;
    if (!channels || (ctype != 3 && depth != 8 && depth != 16) || (ctype == 3 && depth != 8)) {
        *why = "Unsupported image format";  // grey / grey-alpha / sub-byte layouts: not RGB(A)8/16 after decode (image_texture.rs:132-136)
        return false;
    }
    const size_t bpp = (size_t)channels * depth / 8, stride = (size_t)w * bpp;
    std::vector<uint8_t> raw((stride + 1) * h);
    uLongf raw_len = (uLongf)raw.size();
    if (uncompress(raw.data(), &raw_len, idat.data(), (uLong)idat.size()) != Z_OK || raw_len != raw.size()) { *why = "PNG: inflate failed"; return false; }
    std::vector<uint8_t> img(stride * h);
    for (uint32_t y = 0; y < h; ++y) {  // undo the scanline filters
        const uint8_t ft = raw[(stride + 1) * y];
        const uint8_t* in = &raw[(stride + 1) * y + 1];
        uint8_t* out = &img[stride * y];
        const uint8_t* up = y ? &img[stride * (y - 1)] : nullptr;
        for (size_t x = 0; x < stride; ++x) {
            const int a = x >= bpp ? out[x - bpp] : 0, b = up ? up[x] : 0, c = (up && x >= bpp) ? up[x - bpp] : 0;
            int v = in[x];
            switch (ft) {
                case 0: break;
                case 1: v += a; break;
                case 2: v += b; break;
                case 3: v += (a + b) / 2; break;
                case 4: { const int pa = std::abs(b - c), pb = std::abs(a - c), pc = std::abs(a + b - 2 * c);
                          v += (pa <= pb && pa <= pc) ? a : (pb <= pc ? b : c); } break;
                default: *why = "PNG: bad filter"; return false;
            }
            out[x] = (uint8_t)v;
        }
    }
    rgb->resize((size_t)w * h * 3);
    for (size_t i = 0; i < (size_t)w * h; ++i) {
        for (int c = 0; c < 3; ++c) {
            float v;
            if (ctype == 3) {
                const size_t pi = (size_t)img[i] * 3 + c;
                if (pi >= palette.size()) { *why = "PNG: palette index out of range"; return false; }
                v = (float)palette[pi] / 255.0f;
            } else if (depth == 8) v = (float)img[i * bpp + c] / 255.0f;                                     // image_texture.rs:9-21
            else v = (float)((uint32_t)img[i * bpp + 2 * c] << 8 | img[i * bpp + 2 * c + 1]) / 65535.0f;       // :24-36
            (*rgb)[i * 3 + c] = v;
        }
    }
    *w_out = w; *h_out = h;
    return true;
}

// ---- parser state --------------------------------------------------------------------------------------------------
using MeshStore = YkMeshStore;

}  // namespace

namespace {

struct Parser {
    yk_pbrt_scene* out;
    std::vector<Lexer> scopes;
    Token pending;
    bool has_pending = false;
    std::string error;
    std::map<std::string, int32_t> named_materials, image_textures;
    int32_t default_material = -1;

    int32_t add_const_texture(f3 v) {
        yk_texture_desc t{};
        t.kind = YK_TEX_CONSTANT;
        t.value[0] = v.x; t.value[1] = v.y; t.value[2] = v.z;
        out->textures.push_back(t);
        return (int32_t)out->textures.size() - 1;
    }
    int32_t add_material(uint32_t kind, int32_t t0, int32_t t1, int32_t t2, float eta, bool remap) {
        yk_material_desc m{};
        m.kind = kind; m.tex[0] = t0; m.tex[1] = t1; m.tex[2] = t2; m.eta = eta; m.remap_roughness = remap ? 1u : 0u;
        out->materials.push_back(m);
        return (int32_t)out->materials.size() - 1;
    }
    bool fail(const std::string& m) { if (error.empty()) error = m; return false; }

    // token access; at end of an included file the parent scope resumes (mod.rs:131-136)
    bool next(Token* t) {
        if (has_pending) { *t = pending; has_pending = false; return true; }
        for (;;) {
            if (scopes.empty()) { t->kind = Tok::End; return true; }
            if (!scopes.back().next(t)) return fail(scopes.back().error);
            if (t->kind != Tok::End) return true;
            scopes.pop_back();
            // tokens needed in the middle of a directive do not cross file ends in the reference (EndOfInput leaves
            // 'top_parse); callers that need a value treat End as an error, top level simply continues
            t->kind = Tok::End;
            return true;
        }
    }
    void unget(const Token& t) { pending = t; has_pending = true; }
    bool unexpected(const Token& t) { return fail(where() + ": UnexpectedToken " + describe(t)); }
    std::string where() { return scopes.empty() ? std::string("<end>") : scopes.back().path + ": line " + std::to_string(scopes.back().line); }
    static std::string describe(const Token& t) {
        switch (t.kind) {
            case Tok::Number: return "Number(" + std::to_string(t.number) + ")";
            case Tok::String: return "String(\"" + t.text + "\")";
            case Tok::LeftBracket: return "LeftBracket";
            case Tok::RightBracket: return "RightBracket";
            case Tok::End: return "EndOfInput";
            default: return t.text;
        }
    }
    bool number(double* v) {
        Token t;
        if (!next(&t)) return false;
        if (t.kind != Tok::Number) return unexpected(t);
        *v = t.number;
        return true;
    }
    bool f32(float* v) { double d; if (!number(&d)) return false; *v = (float)d; return true; }
    bool string(std::string* s) {
        Token t;
        if (!next(&t)) return false;
        if (t.kind != Tok::String) return unexpected(t);
        *s = t.text;
        return true;
    }
    static int32_t as_i32(double v) {  // Rust `f64 as i32`: truncate, saturate, NaN -> 0
        if (v != v) return 0;
        if (v >= 2147483647.0) return INT32_MAX;
        if (v <= -2147483648.0) return INT32_MIN;
        return (int32_t)v;
    }
    bool numbers(std::vector<double>* v) {  // get_num_params!: one number or [ ... ]
        Token t;
        if (!next(&t)) return false;
        if (t.kind == Tok::Number) { v->push_back(t.number); return true; }
        if (t.kind != Tok::LeftBracket) return unexpected(t);
        for (;;) {
            if (!next(&t)) return false;
            if (t.kind == Tok::Number) v->push_back(t.number);
            else if (t.kind == Tok::RightBracket) return true;
            else return unexpected(t);
        }
    }
    bool strings(std::vector<std::string>* v) {
        Token t;
        if (!next(&t)) return false;
        if (t.kind == Tok::String) { v->push_back(t.text); return true; }
        if (t.kind != Tok::LeftBracket) return unexpected(t);
        for (;;) {
            if (!next(&t)) return false;
            if (t.kind == Tok::String) v->push_back(t.text);
            else if (t.kind == Tok::RightBracket) return true;
            else return unexpected(t);
        }
    }
    bool tuples(int n, std::vector<double>* v) {  // get_{two,three}_component_vector_params!: brackets required
        Token t;
        if (!next(&t)) return false;
        if (t.kind != Tok::LeftBracket) return unexpected(t);
        for (;;) {
            if (!next(&t)) return false;
            if (t.kind == Tok::RightBracket) return true;
            if (t.kind != Tok::Number) return unexpected(t);
            v->push_back(t.number);
            for (int k = 1; k < n; ++k) {
                if (!next(&t)) return false;
                if (t.kind != Tok::Number) return unexpected(t);
                v->push_back(t.number);
            }
        }
    }
    bool param_set(ParamSet* ps) {  // get_param_set!, mod.rs:382-474
        for (;;) {
            Token t;
            if (!next(&t)) return false;
            if (t.kind != Tok::String) { unget(t); return true; }
            std::istringstream def(t.text);
            std::string type, name, extra;
            if (!(def >> type >> name) || (def >> extra)) return fail(where() + ": UnexpectedToken " + t.text);
            if (type == "bool") {
                std::vector<std::string> s;
                if (!strings(&s)) return false;
                Item<bool> it{name, {}};
                for (const auto& b : s) {
                    if (b == "true") it.values.push_back(true);
                    else if (b == "false") it.values.push_back(false);
                    else return fail(where() + ": UnexpectedToken " + b);
                }
                ps->bools.push_back(it);
            } else if (type == "float" && name == "uv") {
                std::vector<double> v;
                if (!tuples(2, &v)) return false;
                Item<std::pair<float, float>> it{name, {}};
                for (size_t i = 0; i + 1 < v.size(); i += 2) it.values.push_back({(float)v[i], (float)v[i + 1]});
                ps->uvs.push_back(it);
            } else if (type == "float") {
                std::vector<double> v;
                if (!numbers(&v)) return false;
                Item<float> it{name, {}};
                for (double x : v) it.values.push_back((float)x);
                ps->f32s.push_back(it);
            } else if (type == "integer") {
                std::vector<double> v;
                if (!numbers(&v)) return false;
                Item<int32_t> it{name, {}};
                for (double x : v) it.values.push_back(as_i32(x));
                ps->i32s.push_back(it);
            } else if (type == "string" || type == "texture") {
                Item<std::string> it{name, {}};
                if (!strings(&it.values)) return false;
                ps->strings.push_back(it);
            } else if (type == "color" || type == "rgb" || type == "point" || type == "normal") {
                std::vector<double> v;
                if (!tuples(3, &v)) return false;
                Item<f3> it{name, {}};
                for (size_t i = 0; i + 2 < v.size(); i += 3) it.values.push_back(mk3((float)v[i], (float)v[i + 1], (float)v[i + 2]));
                (type == "point" ? ps->points : type == "normal" ? ps->normals : ps->spectra).push_back(it);
            } else if (type == "spectrum") {
                Token st;
                if (!next(&st)) return false;
                std::vector<float> vals;
                if (st.kind == Tok::String) {  // SPD file: "lambda value" pairs, # comments
                    std::ifstream f(scopes.back().parent + "/" + st.text);
                    if (!f) return fail("could not open spectrum file '" + st.text + "'");
                    std::string l;
                    while (std::getline(f, l)) {
                        std::istringstream ls(l.substr(0, l.find('#')));
                        float x;
                        while (ls >> x) vals.push_back(x);
                    }
                } else {
                    unget(st);
                    std::vector<double> v;
                    if (!numbers(&v)) return false;
                    for (double x : v) vals.push_back((float)x);
                }
                if (vals.size() < 2 || vals.size() % 2) return fail(where() + ": spectrum needs (wavelength, value) pairs");
                std::vector<float> lambda, samples;
                for (size_t i = 0; i + 1 < vals.size(); i += 2) { lambda.push_back(vals[i]); samples.push_back(vals[i + 1]); }
                ps->spectra.push_back({name, {spectrum_to_rgb(lambda, samples)}});
            } else if (type == "blackbody") {
                std::vector<double> v;  // 'blackbody' not supported, falling back to default (mod.rs:452-457)
                if (!numbers(&v)) return false;
            } else {
                return fail(where() + ": UnknownParamType " + type + " " + name);
            }
        }
    }

    // get_material, mod.rs:860-944
    bool material(const std::string& type, const ParamSet& ps, int32_t* out_index) {
        const f3 half = mk3(0.5f, 0.5f, 0.5f), ones = mk3(1, 1, 1);
        if (type == "glass") {
            const int32_t kr = add_const_texture(ParamSet::one(ps.spectra, "Kr", ones)), kt = add_const_texture(ParamSet::one(ps.spectra, "Kt", ones));
            *out_index = add_material(YK_MAT_GLASS, kr, kt, 0, ParamSet::one(ps.f32s, "eta", 1.5f), false);
        } else if (type == "glossy") {
            const int32_t rs = add_const_texture(ParamSet::one(ps.spectra, "Rs", half));
            const float r = ParamSet::one(ps.f32s, "roughness", 0.5f);
            *out_index = add_material(YK_MAT_GLOSSY, rs, add_const_texture(mk3(r, r, r)), 0, 0.0f, false);
        } else if (type == "matte") {
            int32_t kd;
            const std::string kd_tex = ParamSet::one(ps.strings, "Kd", std::string());
            if (kd_tex.empty()) kd = add_const_texture(ParamSet::one(ps.spectra, "Kd", half));
            else {
                auto it = image_textures.find(kd_tex);
                if (it == image_textures.end()) return fail("Texture '" + kd_tex + "' not found");
                kd = it->second;
            }
            const float rads_per_deg = 3.14159274101257324f / 180.0f;  // f32::to_radians
            const float sigma = (ParamSet::one(ps.f32s, "sigma", 0.0f) * rads_per_deg) * rads_per_deg;  // twice, mod.rs:904-907
            *out_index = add_material(YK_MAT_MATTE, kd, add_const_texture(mk3(sigma, sigma, sigma)), 0, 0.0f, false);
        } else if (type == "metal") {
            const int32_t eta = add_const_texture(ParamSet::one(ps.spectra, "eta", copper_rgb(1)));
            const int32_t k = add_const_texture(ParamSet::one(ps.spectra, "k", copper_rgb(2)));
            const float r = ParamSet::one(ps.f32s, "roughness", 0.01f);
            *out_index = add_material(YK_MAT_METAL, eta, k, add_const_texture(mk3(r, r, r)), 0.0f, ParamSet::one(ps.bools, "remaproughness", true));
        } else {  // Unsupported material type: default matte
            *out_index = add_material(YK_MAT_MATTE, add_const_texture(half), add_const_texture(mk3(0, 0, 0)), 0, 0.0f, false);
        }
        return true;
    }

    bool open_scope(const std::string& path) {
        std::ifstream f(path, std::ios::binary);
        if (!f) return fail("could not open '" + path + "'");
        Lexer lx;
        lx.input.assign((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
        lx.path = path;
        const size_t slash = path.find_last_of('/');
        lx.parent = slash == std::string::npos ? std::string(".") : path.substr(0, slash);
        scopes.push_back(std::move(lx));
        return true;
    }

    bool run(const std::string& path) {
        if (!open_scope(path)) return false;
        yk_camera_params& cam = out->result.camera;  // CameraParameters::default, camera.rs:33-42
        cam = yk_camera_params{{0, 0, 0}, {0, 0, 0}, {0, 1, 0}, YK_FOV_X, 0.0f};
        uint32_t res_x = 640, res_y = 480;  // FilmSettings::default, film.rs:25-38
        float fov = 0.0f;
        float lens_radius = 0.0f, focal_distance = 1e6f;  // pbrt-v3's PerspectiveCamera defaults
        struct Graphics { int32_t material; };
        ParamSet none;
        if (!material("matte", none, &default_material)) return false;
        Graphics gs{default_material};
        std::vector<Graphics> gs_stack;
        xform ctm = xf_id();
        std::vector<xform> ctm_stack;
        unsigned active_bits = 3;  // START | END
        std::vector<unsigned> bits_stack;
        float background[3] = {0, 0, 0};

        for (;;) {
            Token t;
            if (!next(&t)) return false;
            if (t.kind == Tok::End) {
                if (scopes.empty()) break;
                continue;
            }
            switch (t.kind) {
                case Tok::ActiveTransform: {
                    Token w;
                    if (!next(&w)) return false;
                    if (w.kind == Tok::All) active_bits = 3;
                    else if (w.kind == Tok::StartTime) active_bits = 1;
                    else if (w.kind == Tok::EndTime) active_bits = 2;
                    else return unexpected(w);
                } break;
                case Tok::AreaLightSource: case Tok::Integrator: case Tok::Sampler: {  // ignore_type_definition!
                    std::string name;
                    ParamSet ps;
                    if (!string(&name) || !param_set(&ps)) return false;
                } break;
                case Tok::AttributeBegin:
                    gs_stack.push_back(gs); ctm_stack.push_back(ctm); bits_stack.push_back(active_bits);
                    break;
                case Tok::AttributeEnd:
                    if (!gs_stack.empty()) {
                        gs = gs_stack.back(); gs_stack.pop_back();
                        // the three stacks move together in the reference; TransformBegin pushes only this one
                        ctm = ctm_stack.back(); ctm_stack.pop_back();
                        active_bits = bits_stack.back(); bits_stack.pop_back();
                    }
                    break;
                case Tok::Camera: {
                    std::string name;
                    ParamSet ps;
                    if (!string(&name)) return false;
                    if (name != "perspective") return fail("Only perspective camera is supported");
                    if (!param_set(&ps)) return false;
                    fov = ParamSet::one(ps.f32s, "fov", 45.0f);
                    lens_radius = ParamSet::one(ps.f32s, "lensradius", 0.0f);
                    focal_distance = ParamSet::one(ps.f32s, "focaldistance", 1e6f);
                } break;
                case Tok::Film: {
                    std::string name;
                    ParamSet ps;
                    if (!string(&name) || !param_set(&ps)) return false;
                    res_x = (uint16_t)ParamSet::one(ps.i32s, "xresolution", 640);
                    res_y = (uint16_t)ParamSet::one(ps.i32s, "yresolution", 480);
                } break;
                case Tok::Include: {
                    std::string file;
                    if (!string(&file)) return false;
                    if (!open_scope(scopes.back().parent + "/" + file)) return false;
                } break;
                case Tok::LightSource: {
                    std::string type;
                    ParamSet ps;
                    if (!string(&type) || !param_set(&ps)) return false;
                    const f3 ones = mk3(1, 1, 1);
                    if (type == "infinite") {
                        const f3 l = ParamSet::one(ps.spectra, "L", ones);
                        background[0] = l.x; background[1] = l.y; background[2] = l.z;
                    } else if (type == "distant") {
                        const f3 l = ParamSet::one(ps.spectra, "L", ones);
                        if (!(l.x == 0 && l.y == 0 && l.z == 0)) {
                            const f3 from = ParamSet::one(ps.points, "from", mk3(0, 0, 0)), to = ParamSet::one(ps.points, "to", mk3(0, 0, 1));
                            const f3 w = unit(sub(from, to));
                            yk_light_desc ld{};
                            ld.kind = YK_LIGHT_DISTANT;
                            const xform id = xf_id();
                            std::memcpy(ld.light_to_world.m, id.m.e, 64); std::memcpy(ld.light_to_world.m_inv, id.inv.e, 64);
                            ld.intensity[0] = l.x; ld.intensity[1] = l.y; ld.intensity[2] = l.z;
                            ld.direction[0] = w.x; ld.direction[1] = w.y; ld.direction[2] = w.z;
                            out->lights.push_back(ld);
                        }
                    } else if (type == "point") {
                        const f3 i = ParamSet::one(ps.spectra, "I", ones);
                        if (!(i.x == 0 && i.y == 0 && i.z == 0)) {
                            const f3 pos = ParamSet::one(ps.points, "from", mk3(0, 0, 0));
                            yk_light_desc ld{};
                            ld.kind = YK_LIGHT_POINT;
                            const xform tr = xf_translate(pos);
                            std::memcpy(ld.light_to_world.m, tr.m.e, 64); std::memcpy(ld.light_to_world.m_inv, tr.inv.e, 64);
                            ld.intensity[0] = i.x; ld.intensity[1] = i.y; ld.intensity[2] = i.z;
                            out->lights.push_back(ld);
                        }
                    }  // other light types: "not implemented", skipped
                } break;
                case Tok::LookAt:
                    if (active_bits & 1u) {  // only the start transform is tracked (mod.rs:589-596)
                        float v[9];
                        for (float& x : v) if (!f32(&x)) return false;
                        std::memcpy(cam.position, v, 12); std::memcpy(cam.target, v + 3, 12);
                        const f3 up = unit(mk3(v[6], v[7], v[8]));
                        cam.up[0] = up.x; cam.up[1] = up.y; cam.up[2] = up.z;
                    }
                    break;
                case Tok::NamedMaterial: {
                    std::string name;
                    if (!string(&name)) return false;
                    auto it = named_materials.find(name);
                    gs.material = it == named_materials.end() ? default_material : it->second;
                } break;
                case Tok::Material: {
                    std::string type;
                    ParamSet ps;
                    if (!string(&type) || !param_set(&ps)) return false;
                    if (!material(type, ps, &gs.material)) return false;
                } break;
                case Tok::MakeNamedMaterial: {
                    std::string name, key, type;
                    ParamSet ps;
                    if (!string(&name) || !string(&key)) return false;
                    if (key != "string type") return fail(where() + ": UnknownParamType MakeNamedMaterial");
                    if (!string(&type) || !param_set(&ps)) return false;
                    int32_t m;
                    if (!material(type, ps, &m)) return false;
                    named_materials[name] = m;
                } break;
                case Tok::Rotate: {
                    float a, x, y, z;
                    if (!f32(&a) || !f32(&x) || !f32(&y) || !f32(&z)) return false;
                    ctm = xf_compose(ctm, xf_rotate(a * (3.14159274101257324f / 180.0f), mk3(x, y, z)));
                } break;
                case Tok::Scale: {
                    float x, y, z;
                    if (!f32(&x) || !f32(&y) || !f32(&z)) return false;
                    ctm = xf_compose(ctm, xf_scaling(x, y, z));
                } break;
                case Tok::Translate: {
                    float x, y, z;
                    if (!f32(&x) || !f32(&y) || !f32(&z)) return false;
                    ctm = xf_compose(ctm, xf_translate(mk3(x, y, z)));
                } break;
                case Tok::Shape: {
                    std::string type;
                    ParamSet ps;
                    if (!string(&type) || !param_set(&ps)) return false;
                    if (type == "sphere") {
                        yk_sphere_desc sd{};
                        std::memcpy(sd.object_to_world.m, ctm.m.e, 64); std::memcpy(sd.object_to_world.m_inv, ctm.inv.e, 64);
                        sd.radius = ParamSet::one(ps.f32s, "radius", 1.0f);
                        sd.material = gs.material;
                        out->spheres.push_back(sd);
                        out->objects.push_back(-1 - (int32_t)(out->spheres.size() - 1));
                    } else if (type == "trianglemesh") {
                        const std::vector<int32_t>* idx = ParamSet::many(ps.i32s, "indices");
                        const size_t n = idx ? idx->size() : 0;
                        if (n < 3 || n % 3) break;  // "Invalid 'trianglemesh'": skipped
                        MeshStore m;
                        m.o2w = ctm;
                        m.material = gs.material;
                        for (int32_t i : *idx) m.indices.push_back((uint32_t)i);  // `i as usize`
                        if (const auto* p = ParamSet::many(ps.points, "P")) for (const f3& v : *p) { m.points.push_back(v.x); m.points.push_back(v.y); m.points.push_back(v.z); }
                        if (const auto* nn = ParamSet::many(ps.normals, "N")) for (const f3& v : *nn) { m.normals.push_back(v.x); m.normals.push_back(v.y); m.normals.push_back(v.z); }
                        if (const auto* uv = ParamSet::many(ps.uvs, "uv")) for (const auto& v : *uv) { m.uvs.push_back(v.first); m.uvs.push_back(v.second); }
                        out->meshes.push_back(std::move(m));
                        out->objects.push_back((int32_t)out->meshes.size() - 1);
                    } else if (type == "plymesh") {
                        const std::string file = ParamSet::one(ps.strings, "filename", std::string());
                        if (file.empty()) return fail("Empty PLY filename");
                        yk_ply* ply = nullptr;
                        if (yk_ply_load((scopes.back().parent + "/" + file).c_str(), &ply) != YK_OK) return fail(std::string("PLY: ") + yk_last_error());
                        yk_ply_data pd;
                        yk_ply_view(ply, &pd);
                        MeshStore m;
                        m.o2w = ctm;  // ply::load(path, material, Some(transform)): the file's own fit-to-unit is skipped
                        m.material = gs.material;
                        m.points.assign(pd.points, pd.points + (size_t)pd.n_points * 3);
                        if (pd.normals) m.normals.assign(pd.normals, pd.normals + (size_t)pd.n_points * 3);
                        if (pd.uvs) m.uvs.assign(pd.uvs, pd.uvs + (size_t)pd.n_points * 2);
                        m.indices.assign(pd.indices, pd.indices + pd.n_indices);
                        yk_ply_destroy(ply);
                        out->meshes.push_back(std::move(m));
                        out->objects.push_back((int32_t)out->meshes.size() - 1);
                    }  // other shape types: "Unsupported shape type", skipped
                } break;
                case Tok::Texture: {
                    std::string name, ttype, cls;
                    ParamSet ps;
                    if (!string(&name) || !string(&ttype) || !string(&cls) || !param_set(&ps)) return false;
                    if (ttype == "spectrum" && cls == "imagemap") {
                        const std::string file = ParamSet::one(ps.strings, "filename", std::string());
                        if (file.empty()) return fail("missing file for texture '" + name + "'");
                        uint32_t w = 0, h = 0;
                        std::string why;
                        out->texel_storage.emplace_back();
                        if (!decode_png(scopes.back().parent + "/" + file, &w, &h, &out->texel_storage.back(), &why)) return fail(why);
                        yk_texture_desc td{};
                        td.kind = YK_TEX_IMAGE;
                        td.width = w; td.height = h;
                        out->textures.push_back(td);  // texel pointer is patched after parsing (vector growth)
                        image_textures[name] = (int32_t)out->textures.size() - 1;
                        tex_of_storage.push_back((int32_t)out->textures.size() - 1);
                    }
                } break;
                case Tok::TransformBegin: ctm_stack.push_back(ctm); break;
                case Tok::TransformEnd:  // pops the graphics state, not the transform (mod.rs:749-755)
                    if (!gs_stack.empty()) { gs = gs_stack.back(); gs_stack.pop_back(); }
                    break;
                case Tok::WorldBegin: ctm = xf_id(); break;
                case Tok::WorldEnd: break;
                case Tok::Number: case Tok::String: case Tok::LeftBracket: case Tok::RightBracket:
                default:
                    return fail(where() + ": UnimplementedToken " + describe(t));
            }
        }
        // fov axis, mod.rs:827-835
        cam.fov_axis = res_y < res_x ? YK_FOV_Y : YK_FOV_X;
        cam.fov_deg = fov;
        out->result.res_x = res_x;
        out->result.res_y = res_y;
        out->result.lens_radius = lens_radius;
        out->result.focal_distance = focal_distance;
        std::memcpy(out->result.scene.background, background, 12);
        return true;
    }
    std::vector<int32_t> tex_of_storage;
};

}  // namespace

extern "C" {

int yk_pbrt_load(const char* path, uint32_t max_shapes_in_node, uint32_t split_method, yk_pbrt_scene** out) {
    return yk_guard("yk_pbrt_load", [&]() -> int {
    if (!path || !out) return yk_set_error(YK_ERR_INVALID, "yk_pbrt_load: null argument");
    auto sc = std::make_unique<yk_pbrt_scene>();
    Parser p;
    p.out = sc.get();
    if (!p.run(path)) return yk_set_error(YK_ERR_INVALID, "pbrt-v3: " + p.error);
    for (size_t i = 0; i < p.tex_of_storage.size(); ++i) sc->textures[p.tex_of_storage[i]].texels = sc->texel_storage[i].data();
    sc->finish(max_shapes_in_node, split_method);
    *out = sc.release();
    return YK_OK;
    });
}

const yk_pbrt_result* yk_pbrt_view(const yk_pbrt_scene* s) { return s ? &s->result : nullptr; }
void yk_pbrt_destroy(yk_pbrt_scene* s) { delete s; }

}  // extern "C"
