// rrtb_host.cpp -- host side of the drop-in: scene-file parser, camera derivation, tonemap, PNG.
//
// Restates, without copying, the behaviour of the reference's host code (file:line under
// /root/reference):
//   scene::scene               scene.h:212-452   line grammar + quirks (SURVEY Appendix A)
//   scene_obj_inst::transform  scene.h:110-181   translate / scale / Rodrigues rotate, applied in order
//   camera::camera             camera.h:8-29
//   convert_color              color.h:8-23
//   PNG output                 main.cpp:150-167  (stbi_write_png call site)
// The library never prints and never exits: the caller (rrt_b200/host/main.cpp) maps the returned
// reference exit code + message onto stderr/exit like the reference does.
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <zlib.h>

#include <fstream>
#include <map>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/rrtb.h"

namespace {

struct V3 {
    float x, y, z;
};
inline V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
inline V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline V3 operator*(float t, V3 a) { return {t * a.x, t * a.y, t * a.z}; }
inline V3 mul(V3 a, V3 b) { return {a.x * b.x, a.y * b.y, a.z * b.z}; }
inline float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline V3 cross(V3 u, V3 v) { return {u.y * v.z - u.z * v.y, u.z * v.x - u.x * v.z, u.x * v.y - u.y * v.x}; }
inline V3 unit(V3 v) { return (1.0f / sqrtf(dot(v, v))) * v; } // vec3.h: v / length == (1/len) * v
inline void put(float *o, V3 v)
{
    o[0] = v.x;
    o[1] = v.y;
    o[2] = v.z;
}

const float kPi = (float)3.1415926535897932385; // rtweekend.h:56

struct Xform { // scene.h:110-144
    char op;   // 't', 's', 'r'
    V3 v;
    double angle; // degrees, stored as double like xf_rotate::angle
};

V3 apply(const Xform &x, V3 v)
{
    if (x.op == 't') return v + x.v;
    if (x.op == 's') return mul(v, x.v);
    // Rodrigues about the axis AS GIVEN (not normalised), scene.h:136-143.  The reference calls the
    // double-precision ::cos/::sin on a float angle and narrows the results.
    float theta = (float)(x.angle * (double)(kPi / 180));
    float c = (float)cos((double)theta);
    float s = (float)sin((double)theta);
    V3 a = c * v;
    V3 b = s * cross(x.v, v);
    V3 k = (1.0f - c) * (dot(x.v, v) * x.v);
    return (a + b) + k;
}

struct Obj {
    int nv = 0, nt = 0;
    std::vector<V3> verts;
    std::vector<int> tris; // 3 per triangle
};

struct ObjInst {
    int obj, mat;
    std::vector<Xform> xf;
    bool moving = false; // `mobj` (SURVEY 8f4): translates by delta between time0 and time1
    float delta[3] = {0.f, 0.f, 0.f}, time0 = 0.f, time1 = 1.f;
    bool keyframed = false; // `kobj`: pose `xf` at time0, pose `xf_end` at time1, vertices move linearly in between
    std::vector<Xform> xf_end;
};

struct ParseError {
    int code;
    std::string msg;
};

std::vector<std::string> words_of(const std::string &line)
{
    // `while (iss) { iss >> s; push }` => every token plus ONE trailing empty word (scene.h:229-234)
    std::istringstream iss(line);
    std::vector<std::string> w;
    while (iss) {
        std::string s;
        iss >> s;
        w.push_back(s);
    }
    return w;
}

double to_d(const std::string &s)
{
    try {
        return std::stod(s);
    }
    catch (const std::exception &) {
        throw ParseError{1, "ERROR: bad number '" + s + "'"};
    }
}
int to_i(const std::string &s)
{
    try {
        return std::stoi(s);
    }
    catch (const std::exception &) {
        throw ParseError{1, "ERROR: bad integer '" + s + "'"};
    }
}
float to_f(const std::string &s) { return (float)to_d(s); }

} // namespace

struct rrtb_scene {
    rrtb_camera cam{};
    std::vector<rrtb_material> materials;
    std::vector<rrtb_sphere> spheres;
    std::vector<rrtb_msphere> mspheres;
    std::vector<rrtb_triangle> triangles;
    std::vector<rrtb_mtriangle> mtriangles; // of `mobj` instances
    int n_objs = 0, n_obj_insts = 0;
    bool has_background = false; // `background r g b` (grammar extension): replaces the sky
    float background[3] = {0.f, 0.f, 0.f};
};

extern "C" {

int rrtb_camera_derive(const float lookfrom[3], const float lookat[3], const float vup[3], float vfov,
                       float aspect_ratio, float aperture, float focus_dist, float time0, float time1,
                       rrtb_camera *out)
{
    if (!lookfrom || !lookat || !vup || !out) return RRTB_ERR_INVALID;
    // camera.h:12-15: theta is float; h, viewport_height and viewport_width are `auto` = double because
    // ::tan returns double; they are narrowed only when they scale a vec3.
    float theta = vfov * kPi / 180.0f;
    double h = tan((double)(theta / 2.0f));
    double viewport_height = (double)2.0f * h;
    double viewport_width = (double)aspect_ratio * viewport_height;
    V3 from{lookfrom[0], lookfrom[1], lookfrom[2]}, at{lookat[0], lookat[1], lookat[2]}, up{vup[0], vup[1], vup[2]};
    V3 w = unit(from - at);
    V3 u = unit(cross(up, w));
    V3 v = cross(w, u);
    V3 horizontal = (float)((double)focus_dist * viewport_width) * u;
    V3 vertical = (float)((double)focus_dist * viewport_height) * v;
    V3 llc = ((from - (1.0f / 2.0f) * horizontal) - (1.0f / 2.0f) * vertical) - focus_dist * w;
    put(out->origin, from);
    put(out->lower_left_corner, llc);
    put(out->horizontal, horizontal);
    put(out->vertical, vertical);
    put(out->u, u);
    put(out->v, v);
    put(out->w, w);
    out->lens_radius = aperture / 2.0f;
    out->time0 = time0;
    out->time1 = time1;
    return RRTB_OK;
}

int rrtb_scene_parse_file(const char *path, int image_width, int image_height, rrtb_scene **out, int *ref_exit_code,
                          char *err, int err_len)
{
    auto fail = [&](int status, int code, const std::string &msg) {
        if (out) *out = nullptr;
        if (ref_exit_code) *ref_exit_code = code;
        if (err && err_len > 0) {
            strncpy(err, msg.c_str(), (size_t)err_len - 1);
            err[err_len - 1] = 0;
        }
        return status;
    };
    if (!path || !out) return fail(RRTB_ERR_INVALID, 1, "null argument");
    std::ifstream fl(path);
    if (!fl.good()) return fail(RRTB_ERR_IO, 2, std::string("ERROR: problem with opening file: ") + path);

    rrtb_scene *sc = new rrtb_scene();
    std::map<std::string, int> mat_idx;
    std::vector<Obj> objs;
    std::vector<ObjInst> insts;
    bool got_camera = false, adding = false, open_obj = false;
    Obj cur;
    std::string line;
    try {
        while (std::getline(fl, line)) {
            if (line.find("camera") == 0) { // scene.h:226-257; the LAST camera line wins
                std::vector<std::string> w = words_of(line);
                if (w.size() < 14) throw ParseError{1, "ERROR: camera line needs 12 numbers"};
                float f[12];
                for (int k = 0; k < 9; ++k) f[k] = to_f(w[1 + k]);
                double vfov = to_d(w[10]), aperture = to_d(w[11]), focus = to_d(w[12]);
                double t0 = 0.0, t1 = 0.0;
                size_t idx = 13;
                if (idx < w.size() - 1) { // shutter times only when two more words follow
                    if (idx + 1 >= w.size()) throw ParseError{1, "ERROR: camera shutter needs two times"};
                    t0 = to_d(w[idx]);
                    t1 = to_d(w[idx + 1]);
                }
                double aspect = double(image_width) / image_height;
                rrtb_camera_derive(f, f + 3, f + 6, (float)vfov, (float)aspect, (float)aperture, (float)focus, (float)t0,
                                   (float)t1, &sc->cam);
                got_camera = true;
            }
            else if (line.find("material") == 0) { // scene.h:258-294
                std::istringstream iss(line);
                std::string kw, name, type;
                iss >> kw >> name >> type;
                rrtb_material m{};
                if (type == "lambertian") {
                    std::string r, g, b;
                    iss >> r >> g >> b;
                    m.type = RRTB_LAMBERTIAN;
                    m.albedo[0] = to_f(r);
                    m.albedo[1] = to_f(g);
                    m.albedo[2] = to_f(b);
                }
                else if (type == "metal") {
                    std::string r, g, b, f;
                    iss >> r >> g >> b >> f;
                    m.type = RRTB_METAL;
                    m.albedo[0] = to_f(r);
                    m.albedo[1] = to_f(g);
                    m.albedo[2] = to_f(b);
                    m.param = to_f(f); // clamped to <= 1 where it is used (material.h:48)
                }
                else if (type == "dielectric") {
                    std::string r;
                    iss >> r;
                    m.type = RRTB_DIELECTRIC;
                    m.param = to_f(r);
                }
                else if (type == "diffuse_light") { // grammar extension (include/rrtb.h): albedo = emitted radiance
                    std::string r, g, b;
                    iss >> r >> g >> b;
                    m.type = RRTB_DIFFUSE_LIGHT;
                    m.albedo[0] = to_f(r);
                    m.albedo[1] = to_f(g);
                    m.albedo[2] = to_f(b);
                }
                else {
                    throw ParseError{3, "ERROR: unknown material type: " + type};
                }
                int next = (int)sc->materials.size();
                sc->materials.push_back(m);
                mat_idx.insert(std::pair<std::string, int>(name, next)); // first definition of a name wins
            }
            else if (line.find("background") == 0) { // grammar extension (include/rrtb.h); the LAST background line wins
                std::istringstream iss(line);
                std::string kw, r, g, b;
                iss >> kw >> r >> g >> b;
                sc->background[0] = to_f(r);
                sc->background[1] = to_f(g);
                sc->background[2] = to_f(b);
                sc->has_background = true;
            }
            else if (line.find("sphere") == 0) { // scene.h:295-312
                std::istringstream iss(line);
                std::string kw, cx, cy, cz, r, mat;
                iss >> kw >> cx >> cy >> cz >> r >> mat;
                rrtb_sphere s{};
                s.center[0] = to_f(cx);
                s.center[1] = to_f(cy);
                s.center[2] = to_f(cz);
                s.radius = to_f(r);
                s.material = mat_idx[mat]; // unknown names silently become material 0 (scene.h:310)
                sc->spheres.push_back(s);
            }
            else if (line.find("msphere") == 0) { // scene.h:313-339
                std::istringstream iss(line);
                std::string kw, a0, a1, a2, b0, b1, b2, t0, t1, r, mat;
                iss >> kw >> a0 >> a1 >> a2 >> b0 >> b1 >> b2 >> t0 >> t1 >> r >> mat;
                rrtb_msphere m{};
                m.center0[0] = to_f(a0);
                m.center0[1] = to_f(a1);
                m.center0[2] = to_f(a2);
                m.center1[0] = to_f(b0);
                m.center1[1] = to_f(b1);
                m.center1[2] = to_f(b2);
                m.time0 = to_f(t0);
                m.time1 = to_f(t1);
                m.radius = to_f(r);
                m.material = mat_idx[mat];
                sc->mspheres.push_back(m);
            }
            else if (line.find("obj_beg") == 0) { // scene.h:340-352
                std::istringstream iss(line);
                std::string kw, nv, nt;
                iss >> kw >> nv >> nt;
                if (open_obj) throw ParseError{1, "ERROR: obj_beg called without prior obj_end."};
                cur = Obj();
                cur.nv = to_i(nv);
                cur.nt = to_i(nt);
                open_obj = true;
                adding = true;
            }
            else if (line.find("obj_vtx") == 0) { // scene.h:353-364
                if (!adding || !open_obj) throw ParseError{1, "ERROR: obj_vtx called without prior obj_beg"};
                std::istringstream iss(line);
                std::string kw, x, y, z;
                iss >> kw >> x >> y >> z;
                if ((int)cur.verts.size() == cur.nv)
                    throw ParseError{1, "ERROR: only expected " + std::to_string(cur.nv) + " vertices."};
                cur.verts.push_back(V3{to_f(x), to_f(y), to_f(z)});
            }
            else if (line.find("obj_tri") == 0) { // scene.h:365-376
                if (!adding || !open_obj) throw ParseError{1, "ERROR: obj_tri called without prior obj_beg."};
                std::istringstream iss(line);
                std::string kw, i, j, k;
                iss >> kw >> i >> j >> k;
                if ((int)cur.tris.size() == 3 * cur.nt)
                    throw ParseError{1, "ERROR: only expected " + std::to_string(cur.nt) + " triangles."};
                int idx[3] = {to_i(i), to_i(j), to_i(k)};
                for (int q = 0; q < 3; ++q) {
                    if (idx[q] < 0 || idx[q] >= cur.nv) throw ParseError{1, "ERROR: obj_tri vertex index out of range."};
                    cur.tris.push_back(idx[q]);
                }
            }
            else if (line.find("obj_end") == 0) { // scene.h:377-386
                if (!adding || !open_obj) throw ParseError{1, "ERROR: obj_end called without prior obj_beg."};
                if ((int)cur.verts.size() != cur.nv)
                    throw ParseError{1, "ERROR: expected " + std::to_string(cur.nv) + " vertices, got " +
                                            std::to_string(cur.verts.size()) + "."};
                if ((int)cur.tris.size() != 3 * cur.nt)
                    throw ParseError{1, "ERROR: expected " + std::to_string(cur.nt) + " triangles, got " +
                                            std::to_string(cur.tris.size() / 3) + "."};
                objs.push_back(cur);
                open_obj = false;
            }
            else if (line.find("obj") == 0 || line.find("mobj") == 0 || line.find("kobj") == 0) { // scene.h:387-427; mobj, kobj: include/rrtb.h
                const bool moving = line[0] == 'm', keyframed = line[0] == 'k';
                std::vector<std::string> w = words_of(line);
                if (w.size() < (moving ? 8u : (keyframed ? 5u : 3u)))
                    throw ParseError{1, "ERROR: obj called without enough args (count = " + std::to_string(w.size())};
                ObjInst inst;
                inst.obj = to_i(w[1]);
                inst.mat = mat_idx[w[2]];
                size_t idx = 3;
                if (moving) {
                    inst.moving = true;
                    for (int k = 0; k < 3; ++k) inst.delta[k] = to_f(w[3 + k]);
                    inst.time0 = to_f(w[6]);
                    inst.time1 = to_f(w[7]);
                    if (!(inst.time1 != inst.time0)) throw ParseError{1, "ERROR: mobj needs time0 != time1"};
                    idx = 8;
                }
                if (keyframed) {
                    inst.moving = inst.keyframed = true;
                    inst.time0 = to_f(w[3]);
                    inst.time1 = to_f(w[4]);
                    if (!(inst.time1 != inst.time0)) throw ParseError{1, "ERROR: kobj needs time0 != time1"};
                    idx = 5;
                }
                std::vector<Xform> *list = &inst.xf;
                while (idx < w.size() - 1) { // the words vector carries one trailing blank
                    char op = w[idx][0];
                    if (keyframed && w[idx] == "/") { // the pose at time1 follows
                        if (list == &inst.xf_end) throw ParseError{1, "ERROR: kobj has more than two poses"};
                        list = &inst.xf_end;
                        idx += 1;
                    }
                    else if (op == 't' || op == 's') {
                        if (idx + 3 >= w.size()) throw ParseError{1, "ERROR: obj transform needs 3 numbers"};
                        Xform x{op, V3{to_f(w[idx + 1]), to_f(w[idx + 2]), to_f(w[idx + 3])}, 0.0};
                        list->push_back(x);
                        idx += 4;
                    }
                    else if (op == 'r') {
                        if (idx + 4 >= w.size()) throw ParseError{1, "ERROR: obj rotate needs angle + axis"};
                        Xform x{'r', V3{to_f(w[idx + 2]), to_f(w[idx + 3]), to_f(w[idx + 4])}, (double)to_f(w[idx + 1])};
                        list->push_back(x);
                        idx += 5;
                    }
                    else {
                        // the reference would spin forever on an unknown op word (scene.h:400-420)
                        throw ParseError{1, "ERROR: unknown obj transform '" + w[idx] + "'"};
                    }
                }
                insts.push_back(inst);
            }
        }
        if (!got_camera) throw ParseError{4, "ERROR: Scene did not have a camera."};
        if (sc->materials.empty()) throw ParseError{4, "ERROR: Scene did not have any materials."};
        if (sc->spheres.size() + sc->mspheres.size() + insts.size() == 0)
            throw ParseError{4, "ERROR: Scene did not have any objects."};
        // flatten instances to world-space triangles (scene.h:157-170,467-472)
        for (const ObjInst &in : insts) {
            if (in.obj < 0 || in.obj >= (int)objs.size()) throw ParseError{1, "ERROR: obj instance of unknown obj index."};
            const Obj &o = objs[in.obj];
            for (int t = 0; t < o.nt; ++t) {
                rrtb_triangle tr{};
                float *dst[3] = {tr.v0, tr.v1, tr.v2};
                for (int q = 0; q < 3; ++q) {
                    V3 v = o.verts[o.tris[3 * t + q]];
                    for (const Xform &x : in.xf) v = apply(x, v);
                    put(dst[q], v);
                }
                tr.material = in.mat;
                if (!in.moving) {
                    sc->triangles.push_back(tr);
                    continue;
                }
                rrtb_mtriangle mt{};
                for (int k = 0; k < 3; ++k) {
                    mt.v0[k] = tr.v0[k];
                    mt.v1[k] = tr.v1[k];
                    mt.v2[k] = tr.v2[k];
                    mt.delta[k] = in.delta[k];
                }
                if (in.keyframed) { // the same triangle in the pose at time1: per-vertex displacements
                    float end[3][3];
                    for (int q = 0; q < 3; ++q) {
                        V3 v = o.verts[o.tris[3 * t + q]];
                        for (const Xform &x : in.xf_end) v = apply(x, v);
                        put(end[q], v);
                    }
                    for (int k = 0; k < 3; ++k) {
                        mt.delta[k] = end[0][k] - mt.v0[k];
                        mt.extra1[k] = (end[1][k] - mt.v1[k]) - mt.delta[k];
                        mt.extra2[k] = (end[2][k] - mt.v2[k]) - mt.delta[k];
                    }
                }
                mt.time0 = in.time0;
                mt.time1 = in.time1;
                mt.material = in.mat;
                sc->mtriangles.push_back(mt);
            }
        }
        // material indices produced by the name map are always valid except when the scene has a
        // sphere that names a material before any exists (index 0 of an empty list is caught above).
    }
    catch (const ParseError &e) {
        delete sc;
        return fail(RRTB_ERR_PARSE, e.code, e.msg);
    }
    sc->n_objs = (int)objs.size();
    sc->n_obj_insts = (int)insts.size();
    *out = sc;
    if (ref_exit_code) *ref_exit_code = 0;
    if (err && err_len > 0) err[0] = 0;
    return RRTB_OK;
}

void rrtb_scene_free(rrtb_scene *s) { delete s; }

int rrtb_scene_counts(const rrtb_scene *s, int32_t *c)
{
    if (!s || !c) return RRTB_ERR_INVALID;
    c[0] = (int32_t)s->materials.size();
    c[1] = (int32_t)s->spheres.size();
    c[2] = (int32_t)s->mspheres.size();
    c[3] = (int32_t)s->triangles.size();
    c[4] = s->n_objs;
    c[5] = s->n_obj_insts;
    return RRTB_OK;
}
const rrtb_camera *rrtb_scene_camera(const rrtb_scene *s) { return s ? &s->cam : nullptr; }
const rrtb_material *rrtb_scene_materials(const rrtb_scene *s) { return s ? s->materials.data() : nullptr; }
const rrtb_sphere *rrtb_scene_spheres(const rrtb_scene *s) { return s ? s->spheres.data() : nullptr; }
const rrtb_msphere *rrtb_scene_mspheres(const rrtb_scene *s) { return s ? s->mspheres.data() : nullptr; }
const rrtb_triangle *rrtb_scene_triangles(const rrtb_scene *s) { return s ? s->triangles.data() : nullptr; }
int rrtb_scene_mtriangle_count(const rrtb_scene *s) { return s ? (int)s->mtriangles.size() : 0; }
const rrtb_mtriangle *rrtb_scene_mtriangles(const rrtb_scene *s) { return s ? s->mtriangles.data() : nullptr; }
int rrtb_scene_background(const rrtb_scene *s, float *rgb3)
{
    if (!s || !s->has_background) return 0;
    if (rgb3)
        for (int k = 0; k < 3; ++k) rgb3[k] = s->background[k];
    return 1;
}

int rrtb_scene_upload(rrtb_ctx *ctx, const rrtb_scene *s, int use_bvh)
{
    if (!ctx || !s) return RRTB_ERR_INVALID;
    int rc = rrtb_scene_stage_moving_triangles(ctx, s->mtriangles.data(), (int)s->mtriangles.size());
    if (rc == RRTB_OK) rc = rrtb_scene_stage_background(ctx, s->has_background ? s->background : nullptr);
    if (rc != RRTB_OK) return rc;
    return rrtb_scene_set(ctx, &s->cam, s->materials.data(), (int)s->materials.size(), s->spheres.data(),
                          (int)s->spheres.size(), s->mspheres.data(), (int)s->mspheres.size(), s->triangles.data(),
                          (int)s->triangles.size(), use_bvh);
}

// color.h:8-23 (divide by spp, gamma 2, clamp to [0, 0.999], * 256) + the top-down flip of main.cpp:150-163
int rrtb_tonemap_rgb8(const float *rgb_sum, int width, int height, int spp, uint8_t *rgb8)
{
    if (!rgb_sum || !rgb8 || width <= 0 || height <= 0 || spp <= 0) return RRTB_ERR_INVALID;
    const float scale = 1.0f / (float)spp;
    for (int j = height - 1, k = 0; j >= 0; --j, ++k) {
        for (int i = 0; i < width; ++i) {
            const float *src = rgb_sum + 3 * ((size_t)j * width + i);
            uint8_t *dst = rgb8 + 3 * ((size_t)k * width + i);
            for (int c = 0; c < 3; ++c) {
                float x = sqrtf(scale * src[c]);
                // the reference's clamp() returns double (rtweekend.h:93-98); 256 * clamp is a double product
                double cl = x < 0.0f ? (double)0.0f : (x > 0.999f ? (double)0.999f : (double)x);
                dst[c] = (uint8_t)(int)(256 * cl);
            }
        }
    }
    return RRTB_OK;
}

// color.h:8-23 with FP_T = double (the rrtd build): sqrt in double, clamp to [0, 0.999], * 256
int rrtb_tonemap_rgb8_f64(const double *rgb_sum, int width, int height, int spp, uint8_t *rgb8)
{
    if (!rgb_sum || !rgb8 || width <= 0 || height <= 0 || spp <= 0) return RRTB_ERR_INVALID;
    const double scale = 1.0 / spp;
    for (int j = height - 1, k = 0; j >= 0; --j, ++k) {
        for (int i = 0; i < width; ++i) {
            const double *src = rgb_sum + 3 * ((size_t)j * width + i);
            uint8_t *dst = rgb8 + 3 * ((size_t)k * width + i);
            for (int c = 0; c < 3; ++c) {
                double x = sqrt(scale * src[c]);
                double cl = x < 0.0 ? 0.0 : (x > 0.999 ? 0.999 : x);
                dst[c] = (uint8_t)(int)(256 * cl);
            }
        }
    }
    return RRTB_OK;
}

// Minimal PNG (8-bit RGB, zlib deflate, filter 0) -- stands where the reference calls stbi_write_png.
static void png_chunk(FILE *f, const char *tag, const uint8_t *data, uint32_t len)
{
    uint8_t hdr[8] = {(uint8_t)(len >> 24), (uint8_t)(len >> 16), (uint8_t)(len >> 8), (uint8_t)len,
                      (uint8_t)tag[0],      (uint8_t)tag[1],      (uint8_t)tag[2],     (uint8_t)tag[3]};
    fwrite(hdr, 1, 8, f);
    if (len) fwrite(data, 1, len, f);
    uLong crc = crc32(0L, hdr + 4, 4);
    if (len) crc = crc32(crc, data, len);
    uint8_t c[4] = {(uint8_t)(crc >> 24), (uint8_t)(crc >> 16), (uint8_t)(crc >> 8), (uint8_t)crc};
    fwrite(c, 1, 4, f);
}

int rrtb_write_png(const char *path, int width, int height, const uint8_t *rgb8)
{
    if (!path || !rgb8 || width <= 0 || height <= 0) return RRTB_ERR_INVALID;
    const size_t row = (size_t)width * 3;
    std::vector<uint8_t> raw((row + 1) * (size_t)height);
    for (int y = 0; y < height; ++y) {
        raw[(row + 1) * y] = 0;
        memcpy(&raw[(row + 1) * y + 1], rgb8 + row * y, row);
    }
    uLongf clen = compressBound((uLong)raw.size());
    std::vector<uint8_t> comp(clen);
    if (compress2(comp.data(), &clen, raw.data(), (uLong)raw.size(), 6) != Z_OK) return RRTB_ERR_IO;
    FILE *f = fopen(path, "wb");
    if (!f) return RRTB_ERR_IO;
    static const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
    fwrite(sig, 1, 8, f);
    uint8_t ihdr[13] = {(uint8_t)(width >> 24),  (uint8_t)(width >> 16),  (uint8_t)(width >> 8),  (uint8_t)width,
                        (uint8_t)(height >> 24), (uint8_t)(height >> 16), (uint8_t)(height >> 8), (uint8_t)height,
                        8, 2, 0, 0, 0};
    png_chunk(f, "IHDR", ihdr, 13);
    png_chunk(f, "IDAT", comp.data(), (uint32_t)clen);
    png_chunk(f, "IEND", nullptr, 0);
    bool ok = fclose(f) == 0;
    return ok ? RRTB_OK : RRTB_ERR_IO;
}


// PFM (Portable Float Map): "PF" (3 channels) or "Pf" (1), width height, scale -1.0 (little endian), then the rows bottom
// to top, which is the framebuffer's own order.  The floats are written byte by byte, so the file is the same on any host.
int rrtb_write_pfm(const char *path, int width, int height, int channels, const float *data)
{
    if (!path || !data || width <= 0 || height <= 0 || (channels != 1 && channels != 3)) return RRTB_ERR_INVALID;
    const size_t n = (size_t)width * height * channels;
    std::vector<uint8_t> raw(4 * n);
    for (size_t k = 0; k < n; ++k) {
        uint32_t b;
        memcpy(&b, data + k, 4);
        for (int q = 0; q < 4; ++q) raw[4 * k + q] = (uint8_t)(b >> (8 * q));
    }
    FILE *f = fopen(path, "wb");
    if (!f) return RRTB_ERR_IO;
    bool ok = fprintf(f, "%s\n%d %d\n-1.0\n", channels == 3 ? "PF" : "Pf", width, height) > 0;
    ok = fwrite(raw.data(), 1, raw.size(), f) == raw.size() && ok;
    ok = fclose(f) == 0 && ok;
    return ok ? RRTB_OK : RRTB_ERR_IO;
}

} // extern "C"
