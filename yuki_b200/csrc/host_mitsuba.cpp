// Mitsuba 2.1.0 scene loader for the host side of the B200 backend (the second scene format of the step before the hot
// path). Accepts what yuki/src/scene/mitsuba/{mod,sensor,transform,emitter,material,shape,common}.rs accept, with the
// same defaults, axis conventions and error cases, and produces the host scene description the other front ends use:
//   * <scene version="2.1.0">; <default name="resx|resy">; <integrator> skipped with its subtree;
//   * <sensor>: fov / fov_axis / to_world transform; the camera is rebuilt from the decomposed matrix (Mike Day's Euler
//     extraction, math/matrix.rs:217-255) with Mitsuba's left-handed X mirrored (sensor.rs:71-106); after loading, the look-at
//     target moves to the middle of the visible scene bounds (mod.rs:185-197);
//   * <bsdf type="twosided|diffuse|dielectric"> -> Matte (sigma 0) / Glass (ext_ior must be air, material.rs:81-141);
//   * <emitter type="constant|point|spot"> (others are skipped with their subtree): background, PointLight with x
//     mirrored, SpotLight with cutoff_angle / beam_width (emitter.rs:23-162) — the only file format that yields spot lights;
//   * <shape type="ply"> with filename / ref bsdf / transform (rotate, translate, scale, matrix, each pre-multiplied,
//     transform.rs:26-77), loaded through the PLY loader with the file's own fit-to-unit skipped (shape.rs:84-93).
// The reference reads XML with the xml-rs pull parser; this file has its own small XML reader (elements, attributes with
// entity references, comments, the XML declaration) and walks the element tree with the reference's rules: a sub-parser
// sees every *descendant* start tag of its element unless a nested parser consumed it or it asked to skip the subtree
// (macros.rs:32-106), character data and CDATA outside tags are errors, unknown tags are errors.
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <sstream>
#include <string>
#include <utility>
#include <vector>

#include "host_loader.h"
#include "host_math.h"
#include "yuki_gpu.h"
#include "yk_guard.h"

int yk_set_error(int code, const std::string& msg);  // host_scene.cpp
extern "C" int yk_ply_load(const char* path, yk_ply** out);
extern "C" void yk_ply_view(const yk_ply*, yk_ply_data* out);
extern "C" void yk_ply_destroy(yk_ply*);
extern "C" const char* yk_last_error(void);

using namespace ykh;

namespace {

// ---- XML ---------------------------------------------------------------------------------------------------------------
struct Element {
    std::string name;
    std::vector<std::pair<std::string, std::string>> attrs;  // in file order
    std::vector<Element> children;
};

struct XmlReader {
    const std::string& in;
    size_t pos = 0;
    std::string error;

    explicit XmlReader(const std::string& s) : in(s) {}
    bool fail(const std::string& m) {
        if (error.empty()) error = m;
        return false;
    }
    bool starts(const char* lit) const { return in.compare(pos, std::strlen(lit), lit) == 0; }
    static bool is_space(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\n'; }
    static bool is_name_char(char c) {
        return (c >= 'a' && c <= 'z') || (c >= 'A' && c <= 'Z') || (c >= '0' && c <= '9') || c == '_' || c == '-' || c == '.' || c == ':' ||
               (unsigned char)c >= 0x80;
    }
    void skip_space() {
        while (pos < in.size() && is_space(in[pos])) ++pos;
    }
    bool name(std::string* out) {
        const size_t start = pos;
        while (pos < in.size() && is_name_char(in[pos])) ++pos;
        if (pos == start) return fail("XML error: expected a name");
        *out = in.substr(start, pos - start);
        return true;
    }
    bool decode(const std::string& raw, std::string* out) {  // entity and character references
        out->clear();
        for (size_t i = 0; i < raw.size(); ++i) {
            if (raw[i] != '&') {
                out->push_back(raw[i]);
                continue;
            }
            const size_t semi = raw.find(';', i);
            if (semi == std::string::npos) return fail("XML error: unterminated entity reference");
            const std::string ent = raw.substr(i + 1, semi - i - 1);
            if (ent == "amp") out->push_back('&');
            else if (ent == "lt") out->push_back('<');
            else if (ent == "gt") out->push_back('>');
            else if (ent == "quot") out->push_back('"');
            else if (ent == "apos") out->push_back('\'');
            else if (!ent.empty() && ent[0] == '#') {
                char* end = nullptr;
                const unsigned long cp = ent.size() > 1 && (ent[1] == 'x' || ent[1] == 'X') ? std::strtoul(ent.c_str() + 2, &end, 16)
                                                                                           : std::strtoul(ent.c_str() + 1, &end, 10);
                if (!end || *end != '\0' || cp == 0 || cp > 0x10ffff) return fail("XML error: bad character reference");
                if (cp < 0x80) out->push_back((char)cp);  // UTF-8
                else if (cp < 0x800) { out->push_back((char)(0xc0 | (cp >> 6))); out->push_back((char)(0x80 | (cp & 0x3f))); }
                else if (cp < 0x10000) {
                    out->push_back((char)(0xe0 | (cp >> 12))); out->push_back((char)(0x80 | ((cp >> 6) & 0x3f))); out->push_back((char)(0x80 | (cp & 0x3f)));
                } else {
                    out->push_back((char)(0xf0 | (cp >> 18))); out->push_back((char)(0x80 | ((cp >> 12) & 0x3f)));
                    out->push_back((char)(0x80 | ((cp >> 6) & 0x3f))); out->push_back((char)(0x80 | (cp & 0x3f)));
                }
            } else {
                return fail("XML error: unknown entity '" + ent + "'");
            }
            i = semi;
        }
        return true;
    }
    // Markup that is not an element. `top` = outside the root element.
    bool misc(bool* consumed) {
        *consumed = true;
        if (starts("<!--")) {
            const size_t end = in.find("-->", pos + 4);
            if (end == std::string::npos) return fail("XML error: unterminated comment");
            pos = end + 3;
            return true;
        }
        if (starts("<![CDATA[")) {  // mod.rs:165, macros.rs:86-88
            const size_t end = in.find("]]>", pos + 9);
            return fail("Unexpected CDATA: " + in.substr(pos + 9, end == std::string::npos ? std::string::npos : end - pos - 9));
        }
        if (starts("<?")) {
            const size_t end = in.find("?>", pos + 2);
            if (end == std::string::npos) return fail("XML error: unterminated processing instruction");
            std::string target;
            size_t p = pos + 2;
            while (p < end && is_name_char(in[p])) target.push_back(in[p++]);
            if (target != "xml") return fail("Unexpected processing instruction: " + target);  // mod.rs:162-164
            pos = end + 2;
            return true;
        }
        if (starts("<!DOCTYPE")) {
            int depth = 0;
            while (pos < in.size()) {
                const char c = in[pos++];
                if (c == '[') ++depth;
                else if (c == ']') --depth;
                else if (c == '>' && depth <= 0) return true;
            }
            return fail("XML error: unterminated DOCTYPE");
        }
        *consumed = false;
        return true;
    }
    bool text_until_markup() {  // character data: whitespace only (mod.rs:166-168)
        const size_t start = pos;
        while (pos < in.size() && in[pos] != '<') ++pos;
        for (size_t i = start; i < pos; ++i)
            if (!is_space(in[i])) {
                std::string chars;
                decode(in.substr(start, pos - start), &chars);
                return fail("Unexpected characters outside tags: " + chars);
            }
        return true;
    }
    bool element(Element* el) {  // pos at '<' of a start tag
        ++pos;
        if (!name(&el->name)) return false;
        for (;;) {
            skip_space();
            if (pos >= in.size()) return fail("XML error: unexpected end of input in a tag");
            if (in[pos] == '/') {
                if (!starts("/>")) return fail("XML error: malformed empty-element tag");
                pos += 2;
                return true;
            }
            if (in[pos] == '>') {
                ++pos;
                break;
            }
            std::string an;
            if (!name(&an)) return false;
            skip_space();
            if (pos >= in.size() || in[pos] != '=') return fail("XML error: attribute without a value");
            ++pos;
            skip_space();
            if (pos >= in.size() || (in[pos] != '"' && in[pos] != '\'')) return fail("XML error: attribute value must be quoted");
            const char q = in[pos++];
            const size_t end = in.find(q, pos);
            if (end == std::string::npos) return fail("XML error: unterminated attribute value");
            std::string value;
            if (!decode(in.substr(pos, end - pos), &value)) return false;
            pos = end + 1;
            el->attrs.emplace_back(an, value);
        }
        for (;;) {  // content
            if (!text_until_markup()) return false;
            if (pos >= in.size()) return fail("XML error: unexpected end of input inside <" + el->name + ">");
            if (starts("</")) {
                pos += 2;
                std::string closing;
                if (!name(&closing)) return false;
                if (closing != el->name) return fail("XML error: </" + closing + "> closes <" + el->name + ">");
                skip_space();
                if (pos >= in.size() || in[pos] != '>') return fail("XML error: malformed end tag");
                ++pos;
                return true;
            }
            bool consumed = false;
            if (!misc(&consumed)) return false;
            if (consumed) continue;
            el->children.emplace_back();
            if (!element(&el->children.back())) return false;
        }
    }
    bool document(Element* root) {
        if (in.compare(0, 3, "\xef\xbb\xbf") == 0) pos = 3;
        bool have_root = false;
        for (;;) {
            if (!text_until_markup()) return false;
            if (pos >= in.size()) break;
            bool consumed = false;
            if (!misc(&consumed)) return false;
            if (consumed) continue;
            if (starts("</")) return fail("XML error: unexpected end tag");
            if (have_root) return fail("XML error: more than one root element");
            if (!element(root)) return false;
            have_root = true;
        }
        return have_root || fail("XML error: no root element");
    }
};

// ---- value parsing (Rust's str::parse semantics: no surrounding white space, no hex) -----------------------------------
bool parse_f32(const std::string& s, float* out) {
    if (s.empty() || XmlReader::is_space(s.front()) || XmlReader::is_space(s.back())) return false;
    for (size_t i = 0; i + 1 < s.size(); ++i)
        if (s[i] == '0' && (s[i + 1] == 'x' || s[i + 1] == 'X')) return false;
    char* end = nullptr;
    const float v = std::strtof(s.c_str(), &end);
    if (end != s.c_str() + s.size()) return false;
    *out = v;
    return true;
}
bool parse_u16(const std::string& s, uint16_t* out) {
    if (s.empty()) return false;
    size_t i = s[0] == '+' ? 1 : 0;
    if (i >= s.size()) return false;
    uint32_t v = 0;
    for (; i < s.size(); ++i) {
        if (s[i] < '0' || s[i] > '9') return false;
        v = v * 10 + (uint32_t)(s[i] - '0');
        if (v > 0xffffu) return false;
    }
    *out = (uint16_t)v;
    return true;
}
std::vector<std::string> split_spaces(const std::string& s) {  // str::split(' '): empty pieces are kept
    std::vector<std::string> out;
    size_t start = 0;
    for (;;) {
        const size_t sp = s.find(' ', start);
        out.push_back(s.substr(start, sp == std::string::npos ? std::string::npos : sp - start));
        if (sp == std::string::npos) break;
        start = sp + 1;
    }
    return out;
}

// approx::relative_eq! with its f32 defaults (epsilon = max_relative = f32::EPSILON)
bool relative_eq(float a, float b) {
    if (a == b) return true;
    if (std::isinf(a) || std::isinf(b)) return false;
    const float diff = fabsf(a - b);
    if (diff <= 1.1920929e-7f) return true;
    return diff <= fmaxf(fabsf(a), fabsf(b)) * 1.1920929e-7f;
}

xform xf_rot_x(float t) {  // transforms.rs:45-61
    const float c = cosf(t), s = sinf(t);
    xform r = xf_id();
    r.m.at(1, 1) = c; r.m.at(1, 2) = -s; r.m.at(2, 1) = s; r.m.at(2, 2) = c;
    r.inv = mat_transpose(r.m);
    return r;
}
xform xf_rot_y(float t) {  // transforms.rs:63-79
    const float c = cosf(t), s = sinf(t);
    xform r = xf_id();
    r.m.at(0, 0) = c; r.m.at(0, 2) = s; r.m.at(2, 0) = -s; r.m.at(2, 2) = c;
    r.inv = mat_transpose(r.m);
    return r;
}
xform xf_rot_z(float t) {  // transforms.rs:81-97
    const float c = cosf(t), s = sinf(t);
    xform r = xf_id();
    r.m.at(0, 0) = c; r.m.at(0, 1) = -s; r.m.at(1, 0) = s; r.m.at(1, 1) = c;
    r.inv = mat_transpose(r.m);
    return r;
}

// ---- the loader --------------------------------------------------------------------------------------------------------
enum class Visit { Descend, Skip };  // what a sub-parser's body wants done with the element's own children

struct Loader {
    yk_pbrt_scene* out;
    std::string dir;
    std::string error;
    std::map<std::string, int32_t> materials;  // bsdf id -> material index
    bool have_shapes = false;

    bool fail(const std::string& m) {
        if (error.empty()) error = m;
        return false;
    }
    // find_attr! / try_find_attr! (macros.rs:1-23): the last attribute of that name
    static const std::string* try_attr(const Element& e, const char* name) {
        const std::string* v = nullptr;
        for (const auto& a : e.attrs)
            if (a.first == name) v = &a.second;
        return v;
    }
    bool attr(const Element& e, const char* name, const std::string** v) {
        *v = try_attr(e, name);
        return *v || fail(std::string("Could not find element attribute '") + name + "'");
    }
    int32_t const_texture(float r, float g, float b) {
        yk_texture_desc t{};
        t.kind = YK_TEX_CONSTANT;
        t.value[0] = r; t.value[1] = g; t.value[2] = b;
        out->textures.push_back(t);
        return (int32_t)out->textures.size() - 1;
    }
    int32_t add_material(uint32_t kind, int32_t t0, int32_t t1, float eta) {
        yk_material_desc m{};
        m.kind = kind; m.tex[0] = t0; m.tex[1] = t1; m.tex[2] = -1; m.eta = eta; m.remap_roughness = 0;
        out->materials.push_back(m);
        return (int32_t)out->materials.size() - 1;
    }
    int32_t matte(f3 kd) { return add_material(YK_MAT_MATTE, const_texture(kd.x, kd.y, kd.z), const_texture(0.0f, 0.0f, 0.0f), 1.5f); }

    // parse_element! (macros.rs:32-106): `body` sees every descendant start tag in document order.
    template <class Body>
    bool descendants(const Element& e, Body&& body) {
        for (const Element& ch : e.children) {
            Visit v = Visit::Descend;
            if (!body(ch, &v)) return false;
            if (v == Visit::Descend && !descendants(ch, body)) return false;
        }
        return true;
    }

    // common.rs:4-18. `soft` = the name mismatch is reported to the caller instead of failing the load.
    bool rgb(const Element& e, const char* expected, f3* v, bool* name_mismatch = nullptr) {
        float c[3] = {0.0f, 0.0f, 0.0f};
        const std::string *name, *value;
        if (!attr(e, "name", &name)) return false;
        if (*name != expected) {
            if (name_mismatch) { *name_mismatch = true; return true; }
            return fail(std::string("Expected rgb to be '") + expected + "', got '" + *name + "'");
        }
        if (!attr(e, "value", &value)) return false;
        const std::vector<std::string> parts = split_spaces(*value);
        for (size_t i = 0; i < parts.size(); ++i) {
            float f;
            if (!parse_f32(parts[i], &f)) return fail("rgb value '" + parts[i] + "' is not a float");
            if (i >= 3) return fail("rgb value has more than three components");
            c[i] = f;
        }
        *v = mk3(c[0], c[1], c[2]);
        return true;
    }

    // transform.rs:15-81: each entry is pre-multiplied onto the transform so far
    bool transform(const Element& e, xform* result) {
        xform t = xf_id();
        const bool ok = descendants(e, [&](const Element& ch, Visit*) -> bool {
            if (ch.name == "rotate") {
                float axis[3] = {0.0f, 0.0f, 0.0f};
                const char* names[3] = {"x", "y", "z"};
                for (int k = 0; k < 3; ++k)
                    if (const std::string* v = try_attr(ch, names[k]))
                        if (!parse_f32(*v, &axis[k])) return fail("rotate axis '" + *v + "' is not a float");
                const std::string* a;
                float deg;
                if (!attr(ch, "angle", &a)) return false;
                if (!parse_f32(*a, &deg)) return fail("rotate angle '" + *a + "' is not a float");
                t = xf_compose(xf_rotate(deg2rad(deg), unit(mk3(axis[0], axis[1], axis[2]))), t);
            } else if (ch.name == "translate") {
                const std::string* v;
                if (!attr(ch, "value", &v)) return false;
                std::vector<float> p;
                for (const std::string& s : split_spaces(*v)) {
                    float f;
                    if (!parse_f32(s, &f)) return fail("translate value '" + s + "' is not a float");
                    p.push_back(f);
                }
                if (p.size() < 3) return fail("translate needs three values");
                t = xf_compose(xf_translate(mk3(p[0], p[1], p[2])), t);
            } else if (ch.name == "scale") {
                const std::string* v;
                if (!attr(ch, "value", &v)) return false;
                const std::vector<std::string> parts = split_spaces(*v);
                if (parts.size() != 1 && parts.size() != 3) return fail("scale needs one or three values");
                float p[3];
                for (size_t i = 0; i < parts.size(); ++i)
                    if (!parse_f32(parts[i], &p[i])) return fail("scale value '" + parts[i] + "' is not a float");
                if (parts.size() == 1) p[1] = p[2] = p[0];
                t = xf_compose(xf_scaling(p[0], p[1], p[2]), t);
            } else if (ch.name == "matrix") {
                const std::string* v;
                if (!attr(ch, "value", &v)) return false;
                mat4 m;
                const std::vector<std::string> parts = split_spaces(*v);
                if (parts.size() != 16) return fail("matrix needs 16 values");
                for (int i = 0; i < 16; ++i)
                    if (!parse_f32(parts[i], &m.e[i])) return fail("matrix value '" + parts[i] + "' is not a float");
                xform mx;
                if (!xf_from_matrix(m, &mx)) return fail("Can't invert, singular matrix");
                t = xf_compose(mx, t);
            } else {
                return fail("Unknown transformation data type '" + ch.name + "'");
            }
            return true;
        });
        *result = t;
        return ok;
    }

    // sensor.rs:19-109
    bool sensor(const Element& e, yk_camera_params* cam) {
        std::string fov_axis;
        float fov_angle = 0.0f;
        xform to_world = xf_id();
        if (!descendants(e, [&](const Element& ch, Visit* v) -> bool {
                const std::string *n, *val;
                if (ch.name == "string") {
                    if (!attr(ch, "name", &n) || !attr(ch, "value", &val)) return false;
                    if (*n != "fov_axis") return fail("Unknown sensor string element '" + *n + "'");
                    fov_axis = *val;
                } else if (ch.name == "float") {
                    if (!attr(ch, "name", &n) || !attr(ch, "value", &val)) return false;
                    if (*n == "fov") {
                        if (!parse_f32(*val, &fov_angle)) return fail("fov '" + *val + "' is not a float");
                    } else if (*n != "near_clip" && *n != "far_clip" && !n->empty()) {
                        return fail("Unknown sensor string element '" + *n + "'");
                    }
                } else if (ch.name == "transform") {
                    *v = Visit::Skip;
                    return transform(ch, &to_world);
                } else if (ch.name == "sampler" || ch.name == "film") {
                    *v = Visit::Skip;
                } else {
                    return fail("Unknown sensor data type '" + ch.name + "'");
                }
                return true;
            }))
            return false;
        // Mitsuba's +X is to the left of +Z, ours to the right of it
        to_world = xf_compose(xf_scaling(-1.0f, 1.0f, 1.0f), to_world);
        // Matrix4x4::decompose (math/matrix.rs:217-255)
        const mat4& m = to_world.m;
        const f3 position = mk3(m.at(0, 3), m.at(1, 3), m.at(2, 3));
        const f3 sc = mk3(length(mk3(m.at(0, 0), m.at(1, 0), m.at(2, 0))), length(mk3(m.at(0, 1), m.at(1, 1), m.at(2, 1))),
                          length(mk3(m.at(0, 2), m.at(1, 2), m.at(2, 2))));
        if (sc.x == 0.0f || sc.y == 0.0f || sc.z == 0.0f)
            return fail("Cannot decompose camera to world matrix: Cannot decompose matrix with a zero scale component");
        float mr[3][3];
        for (int r = 0; r < 3; ++r) {
            mr[r][0] = m.at(r, 0) / sc.x; mr[r][1] = m.at(r, 1) / sc.y; mr[r][2] = m.at(r, 2) / sc.z;
        }
        const float theta_x = atan2f(mr[1][2], mr[2][2]);
        const float c2 = sqrtf(mr[0][0] * mr[0][0] + mr[0][1] * mr[0][1]);
        const float theta_y = atan2f(-mr[0][2], c2);
        const float s1 = sinf(theta_x), c1 = cosf(theta_x);
        const float theta_z = atan2f(s1 * mr[2][0] - c1 * mr[1][0], c1 * mr[1][1] - s1 * mr[2][1]);
        if (!(relative_eq(sc.x, 1.0f) && relative_eq(sc.y, 1.0f) && relative_eq(sc.z, 1.0f))) return fail("Camera to world has scaling");
        if (fov_axis == "x") cam->fov_axis = YK_FOV_X;
        else if (fov_axis == "y") cam->fov_axis = YK_FOV_Y;
        else return fail("Unknown fov axis '" + fov_axis + "'");
        cam->fov_deg = fov_angle;
        // We compensate for the flipped X axis in the rotation
        const xform c2w = xf_compose(xf_translate(position), xf_compose(xf_rot_x(-theta_x), xf_compose(xf_rot_y(-theta_y), xf_rot_z(theta_z))));
        store3(position, cam->position);
        store3(apply_point(c2w.m, mk3(0.0f, 0.0f, 1.0f)), cam->target);
        store3(apply_vec(c2w.m, mk3(0.0f, 1.0f, 0.0f)), cam->up);
        return true;
    }

    // material.rs:52-78
    bool diffuse(const Element& e, int32_t* material) {
        f3 kd = mk3(0.5f, 0.5f, 0.5f);
        if (!descendants(e, [&](const Element& ch, Visit*) -> bool {
                if (ch.name != "rgb") return fail("Unknown light data type '" + ch.name + "'");
                return rgb(ch, "reflectance", &kd);
            }))
            return false;
        *material = matte(kd);
        return true;
    }
    // material.rs:17-50 (the nested bsdf is read as a diffuse one whatever its type)
    bool twosided(const Element& e, int32_t* material) {
        int32_t m = -1;
        if (!descendants(e, [&](const Element& ch, Visit* v) -> bool {
                if (ch.name == "bsdf") {
                    *v = Visit::Skip;
                    return diffuse(ch, &m);
                }
                if (ch.name == "rgb") {
                    f3 kd;
                    if (!rgb(ch, "reflectance", &kd)) return false;
                    m = matte(kd);
                    return true;
                }
                return fail("Unknown material data type '" + ch.name + "'");
            }))
            return false;
        *material = m >= 0 ? m : matte(mk3(1.0f, 1.0f, 1.0f));
        return true;
    }
    // material.rs:80-142
    bool dielectric(const Element& e, int32_t* material) {
        float int_ior = 1.5046f, ext_ior = 1.000277f;  // BK7 glass, air
        f3 refl = mk3(1.0f, 1.0f, 1.0f), trans = mk3(1.0f, 1.0f, 1.0f);
        if (!descendants(e, [&](const Element& ch, Visit*) -> bool {
                if (ch.name == "rgb") {
                    bool other = false;
                    f3 v;
                    if (!rgb(ch, "specular_reflectance", &v, &other)) return false;
                    if (!other) { refl = v; return true; }
                    other = false;
                    if (!rgb(ch, "specular_transmittance", &v, &other)) return false;
                    if (!other) { trans = v; return true; }
                    const std::string* n;
                    if (!attr(ch, "name", &n)) return false;
                    return fail("Unknown dielectric rgb data '" + *n + "'");
                }
                if (ch.name == "float") {
                    const std::string *n, *val;
                    float f;
                    if (!attr(ch, "name", &n) || !attr(ch, "value", &val)) return false;
                    if (!parse_f32(*val, &f)) return fail("dielectric float '" + *val + "' is not a float");
                    if (*n == "int_ior") int_ior = f;
                    else if (*n == "ext_ior") ext_ior = f;
                    else return fail("Unknown dielectric float data '" + *n + "'");
                    return true;
                }
                return fail("Unknown dielectric data type '" + ch.name + "'");
            }))
            return false;
        if (!(fabsf(ext_ior - 1.000277f) <= 0.001f)) {
            char buf[64];
            std::snprintf(buf, sizeof buf, "%g", ext_ior);
            return fail(std::string("Only air supported for external IoR not supported but received '") + buf + "'");
        }
        *material = add_material(YK_MAT_GLASS, const_texture(refl.x, refl.y, refl.z), const_texture(trans.x, trans.y, trans.z), int_ior);
        return true;
    }

    void add_light(uint32_t kind, const xform& l2w, f3 intensity, float total_width = 0.0f, float falloff_start = 0.0f) {
        yk_light_desc l{};
        l.kind = kind;
        std::memcpy(l.light_to_world.m, l2w.m.e, 64);
        std::memcpy(l.light_to_world.m_inv, l2w.inv.e, 64);
        store3(intensity, l.intensity);
        l.total_width_deg = total_width;
        l.falloff_start_deg = falloff_start;
        out->lights.push_back(l);
    }
    // emitter.rs:70-121
    bool point_light(const Element& e) {
        f3 position = mk3(0.0f, 0.0f, 0.0f), intensity = mk3(0.0f, 0.0f, 0.0f);
        if (!descendants(e, [&](const Element& ch, Visit*) -> bool {
                if (ch.name == "point") {
                    const std::string* n;
                    if (!attr(ch, "name", &n)) return false;
                    if (*n != "position") return fail("Expected 'name': 'filename' as first mesh 'string' attribute");
                    for (size_t i = 1; i < ch.attrs.size(); ++i) {  // the first attribute is taken to be `name`
                        float* dst = ch.attrs[i].first == "x" ? &position.x : ch.attrs[i].first == "y" ? &position.y : ch.attrs[i].first == "z" ? &position.z : nullptr;
                        if (!dst) return fail("Invalid point axis '" + ch.attrs[i].first + "'");
                        if (!parse_f32(ch.attrs[i].second, dst)) return fail("point coordinate '" + ch.attrs[i].second + "' is not a float");
                    }
                    return true;
                }
                if (ch.name == "rgb") return rgb(ch, "intensity", &intensity);
                return fail("Unknown light data type '" + ch.name + "'");
            }))
            return false;
        position.x = -position.x;  // Mitsuba's +X is to the left of +Z, ours to the right of it
        add_light(YK_LIGHT_POINT, xf_translate(position), intensity);
        return true;
    }
    // emitter.rs:123-163
    bool spot_light(const Element& e) {
        xform l2w = xf_id();
        f3 intensity = mk3(0.0f, 0.0f, 0.0f);
        float total_width = 0.0f, falloff_start = 0.0f;
        if (!descendants(e, [&](const Element& ch, Visit* v) -> bool {
                if (ch.name == "float") {
                    const std::string *n, *val;
                    if (!attr(ch, "name", &n)) return false;
                    float* dst = *n == "cutoff_angle" ? &total_width : *n == "beam_width" ? &falloff_start : nullptr;
                    if (!dst) return fail("Unexpected spot light float 'name': '" + *n + "'");
                    if (!attr(ch, "value", &val)) return false;
                    if (!parse_f32(*val, dst)) return fail("spot light float '" + *val + "' is not a float");
                    return true;
                }
                if (ch.name == "transform") {
                    *v = Visit::Skip;
                    return transform(ch, &l2w);
                }
                if (ch.name == "rgb") return rgb(ch, "intensity", &intensity);
                return fail("Unknown spot light data type '" + ch.name + "'");
            }))
            return false;
        add_light(YK_LIGHT_SPOT, xf_compose(xf_scaling(-1.0f, 1.0f, 1.0f), l2w), intensity, total_width, falloff_start);
        return true;
    }
    // emitter.rs:44-68
    bool constant_emitter(const Element& e) {
        f3 radiance = mk3(0.0f, 0.0f, 0.0f);
        if (!descendants(e, [&](const Element& ch, Visit*) -> bool {
                if (ch.name != "rgb") return fail("Unknown constant emitter data type '" + ch.name + "'");
                return rgb(ch, "radiance", &radiance);
            }))
            return false;
        store3(radiance, out->result.scene.background);
        return true;
    }

    // shape.rs:18-94
    bool shape(const Element& e) {
        const std::string* type;
        if (!attr(e, "type", &type)) return false;
        if (*type != "ply") return fail("Unexpected shape type '" + *type + "'!");
        xform t = xf_id();
        std::string ply_path, material_id;
        bool have_path = false, have_material = false;
        if (!descendants(e, [&](const Element& ch, Visit* v) -> bool {
                const std::string *n, *val;
                if (ch.name == "string") {
                    if (!attr(ch, "name", &n)) return false;
                    if (*n != "filename") return fail("Expected 'name': 'filename' as mesh 'string' attribute");
                    if (!attr(ch, "value", &val)) return false;
                    std::string rel = *val;
                    for (char& c : rel)
                        if (c == '\\') c = '/';
                    const std::string joined = !rel.empty() && rel[0] == '/' ? rel : dir + "/" + rel;
                    char resolved[PATH_MAX];
                    if (!realpath(joined.c_str(), resolved)) return fail("Error canonicalizing absolute mesh path for '" + rel + "'");
                    ply_path = resolved;
                    have_path = true;
                    return true;
                }
                if (ch.name == "ref") {
                    if (!attr(ch, "name", &n)) return false;
                    if (*n != "bsdf") return fail("Expected mesh 'ref' to be 'bsdf', got '" + *n + "'");
                    if (!attr(ch, "id", &val)) return false;
                    material_id = *val;
                    have_material = true;
                    return true;
                }
                if (ch.name == "transform") {
                    *v = Visit::Skip;
                    return transform(ch, &t);
                }
                return fail("Unknown shape type '" + ch.name + "'");
            }))
            return false;
        t = xf_compose(xf_scaling(-1.0f, 1.0f, 1.0f), t);  // Mitsuba's +X is to the left of +Z, ours to the right of it
        if (!have_path) return fail("Mesh with no ply");
        if (!have_material) return fail("Mesh with no material");
        const auto mat = materials.find(material_id);
        if (mat == materials.end()) return fail("Unknown mesh material '" + material_id + "'");
        yk_ply* ply = nullptr;
        if (yk_ply_load(ply_path.c_str(), &ply) != YK_OK) return fail(std::string("PLY: ") + yk_last_error());
        yk_ply_data pd;
        yk_ply_view(ply, &pd);
        YkMeshStore m;
        m.o2w = t;  // ply::load(path, material, Some(transform)): the file's own fit-to-unit is skipped
        m.material = mat->second;
        m.points.assign(pd.points, pd.points + (size_t)pd.n_points * 3);
        if (pd.normals) m.normals.assign(pd.normals, pd.normals + (size_t)pd.n_points * 3);
        if (pd.uvs) m.uvs.assign(pd.uvs, pd.uvs + (size_t)pd.n_points * 2);
        m.indices.assign(pd.indices, pd.indices + pd.n_indices);
        yk_ply_destroy(ply);
        have_shapes = have_shapes || !m.indices.empty();
        out->meshes.push_back(std::move(m));
        out->objects.push_back((int32_t)out->meshes.size() - 1);
        return true;
    }

    // mod.rs:43-158: the document loop. Elements are dispatched by name at any depth.
    bool top(const Element& e) {
        yk_pbrt_result& r = out->result;
        const std::string *n, *v;
        if (e.name == "scene") {
            if (!attr(e, "version", &v)) return false;
            if (*v != "2.1.0") return fail("Scene file version is not 2.1.0");
        } else if (e.name == "default") {
            if (!attr(e, "name", &n) || !attr(e, "value", &v)) return false;
            uint16_t u;
            if (*n == "resx" || *n == "resy") {
                if (!parse_u16(*v, &u)) return fail("default " + *n + " '" + *v + "' is not a u16");
                (*n == "resx" ? r.res_x : r.res_y) = u;
            }
        } else if (e.name == "integrator") {
            return true;  // skipped with its subtree
        } else if (e.name == "sensor") {
            return sensor(e, &r.camera);
        } else if (e.name == "bsdf") {
            const std::string* type;
            if (!attr(e, "type", &type)) return false;
            int32_t m = -1;
            if (*type == "twosided") { if (!twosided(e, &m)) return false; }
            else if (*type == "diffuse") { if (!diffuse(e, &m)) return false; }
            else if (*type == "dielectric") { if (!dielectric(e, &m)) return false; }
            else return fail("Unknown bsdf type '" + *type + "'");
            const std::string* id;
            if (!attr(e, "id", &id)) return false;
            materials[*id] = m;
            return true;
        } else if (e.name == "emitter") {
            const std::string* type;
            if (!attr(e, "type", &type)) return false;
            if (*type == "constant") return constant_emitter(e);
            if (*type == "point") return point_light(e);
            if (*type == "spot") return spot_light(e);
            return true;  // other emitters are skipped with their subtree
        } else if (e.name == "shape") {
            return shape(e);
        } else {
            return fail("Unknown element: '" + e.name + "'");
        }
        for (const Element& ch : e.children)
            if (!top(ch)) return false;
        return true;
    }

    // mod.rs:185-197: the look-at target moves to the middle of the part of the scene bounds in front of the camera
    // (bvh.bounds() = the union of the world-space triangle bounds).
    void retarget_camera() {
        box3 bounds = empty_box();
        for (const YkMeshStore& m : out->meshes)
            for (uint32_t i : m.indices)
                if ((size_t)i * 3 + 2 < m.points.size()) bounds = grow(bounds, apply_point(m.o2w.m, load3(&m.points[(size_t)i * 3])));
        yk_camera_params& cam = out->result.camera;
        const f3 pos = load3(cam.position);
        const f3 fwd = unit(sub(load3(cam.target), pos));
        // Bounds3::intersections (math/bounds.rs:176-206) with t_max = inf
        const f3 inv = mk3(1.0f / fwd.x, 1.0f / fwd.y, 1.0f / fwd.z);
        const f3 t0 = mk3((bounds.lo.x - pos.x) * inv.x, (bounds.lo.y - pos.y) * inv.y, (bounds.lo.z - pos.z) * inv.z);
        const f3 t1 = mk3((bounds.hi.x - pos.x) * inv.x, (bounds.hi.y - pos.y) * inv.y, (bounds.hi.z - pos.z) * inv.z);
        const f3 lo = min3(t0, t1), hi = max3(t0, t1);
        const float p0 = fmaxf(fmaxf(lo.x, fmaxf(lo.y, lo.z)), 0.0f);
        const float p1 = fminf(fminf(hi.x, fminf(hi.y, hi.z)), INFINITY);
        if (p0 <= p1) {
            const f3 target = p0 > 0.0f ? add(pos, scale(fwd, (p0 + p1) / 2.0f)) : add(pos, scale(fwd, p1 / 2.0f));
            store3(target, cam.target);
        }
    }
};

}  // namespace

extern "C" int yk_mitsuba_load(const char* path, uint32_t max_shapes_in_node, uint32_t split_method, yk_pbrt_scene** out) {
    return yk_guard("yk_mitsuba_load", [&]() -> int {
    if (!path || !out) return yk_set_error(YK_ERR_INVALID, "yk_mitsuba_load: null argument");
    std::ifstream f(path, std::ios::binary);
    if (!f) return yk_set_error(YK_ERR_INVALID, std::string("mitsuba: cannot open '") + path + "'");
    std::stringstream ss;
    ss << f.rdbuf();
    const std::string text = ss.str();
    Element root;
    XmlReader xml(text);
    if (!xml.document(&root)) return yk_set_error(YK_ERR_INVALID, "mitsuba: " + xml.error);
    auto sc = std::make_unique<yk_pbrt_scene>();
    Loader ld;
    ld.out = sc.get();
    const std::string p(path);
    const size_t slash = p.find_last_of('/');
    ld.dir = slash == std::string::npos ? std::string(".") : (slash == 0 ? std::string("/") : p.substr(0, slash));
    // CameraParameters::default (camera.rs:32-41), FilmSettings::default (film.rs:25-38)
    yk_pbrt_result& r = sc->result;
    r.camera = yk_camera_params{};
    r.camera.up[1] = 1.0f;
    r.camera.fov_axis = YK_FOV_X;
    r.res_x = 640;
    r.res_y = 480;
    r.lens_radius = 0.0f;  // a pinhole: the thinlens sensor is not read
    r.focal_distance = 1e6f;
    if (!ld.top(root)) return yk_set_error(YK_ERR_INVALID, "mitsuba: " + ld.error);
    if (!ld.have_shapes) return yk_set_error(YK_ERR_INVALID, "mitsuba: the scene has no shapes (bvh.rs:68 needs at least one)");
    ld.retarget_camera();
    sc->finish(max_shapes_in_node, split_method);
    *out = sc.release();
    return YK_OK;
    });
}
