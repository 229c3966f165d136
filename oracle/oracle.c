/* oracle.c - plain-C restatement of the reference's per-pixel render path.
 *
 * TEST INFRASTRUCTURE ONLY - never on the product path (see oracle.h).
 *
 * Every function cites the reference lines (/root/reference/kernel.cu unless noted)
 * it restates.  The restatement keeps the reference's operation ORDER, its float /
 * double promotions (SURVEY.md appendix B) and its quirks (effective radius r^2,
 * negative-t hits, in-place normalise drift, non-Rodrigues rotate, pi = 3.1415).
 * Build with: gcc -O2 -ffp-contract=off (no -ffast-math, no FMA contraction).
 *
 * Parity pin: the reference ships no tests or golden vectors, so this file is pinned
 * against the reference's OWN code compiled as host C++ (oracle/_ref, built by
 * ref_build/make_ref.py in the build container) - tests/test_oracle_pin.py demands
 * bit-identical pixels / hit ids / t - and against fixtures that build generated
 * (tests/golden/, script tests/golden/make_golden.py).
 */
#include "oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

typedef struct { float x, y, z; } v3;

/* ---- vector helpers, kernel.cu:45-108 ---------------------------------------------- */
static inline v3 v_sub(v3 a, v3 b) { v3 r = {a.x - b.x, a.y - b.y, a.z - b.z}; return r; }      /* :46 */
static inline v3 v_add(v3 a, v3 b) { v3 r = {a.x + b.x, a.y + b.y, a.z + b.z}; return r; }      /* :61 */
static inline v3 v_scale(v3 a, float b) { v3 r = {a.x * b, a.y * b, a.z * b}; return r; }       /* :76 */
static inline v3 v_cross(v3 a, v3 b) {                                                          /* :81 */
    v3 r = {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
    return r;
}
static inline float v_dot(v3 a, v3 b) { return (a.x * b.x + a.y * b.y + a.z * b.z); }           /* :93 */
static inline float v_length(v3 a) { return sqrtf(v_dot(a, a)); }                               /* :98 */
/* :102-108 - divides by a DOUBLE length, writes the result back into its argument */
static inline v3 v_normalise(v3* v) {
    double l = v_length(*v);
    if (l != 0) {
        v->x /= l;
        v->y /= l;
        v->z /= l;
        return *v;
    }
    v3 zero = {0, 0, 0};
    return zero;
}

/* ---- sphere::intersect, kernel.cu:293-354 ------------------------------------------ */
static inline int sphere_intersect(v3 O, v3 D, v3 c, float radius, float* t_out) {
    float A = (D.x * (D.x) + D.y * (D.y) + D.z * (D.z));                                           /* :332 */
    float B = 2 * (D.x * (O.x - c.x) + D.y * (O.y - c.y) + D.z * (O.z - c.z));                     /* :333 */
    float C = (O.x - c.x) * (O.x - c.x) + (O.y - c.y) * (O.y - c.y) + (O.z - c.z) * (O.z - c.z)
              - radius * radius;                                                                   /* :334 */
    float t = (-B + sqrtf(B * B - 4 * A * C)) / (2 * A);                                           /* :336 */
    *t_out = t;
    if (t == 0.f) return 1;                                                                        /* :338 */
    if (t >= 0.0001) {                                                                             /* :342, double compare */
        float t2 = (-B - sqrtf(B * B - 4 * A * C)) / (2 * A);                                      /* :344 */
        if (t > t2) *t_out = t2;                                                                   /* :346-347 */
        return 1;
    }
    return 0;
}

/* ---- plane::intersect, kernel.cu:369-380 -------------------------------------------- */
static inline int plane_intersect(v3 O, v3 D, v3 pos, v3 normal, float* t_out) {
    float denom = v_dot(normal, D);
    if (denom < 0) {
        v3 pl0 = v_sub(pos, O);
        float t = v_dot(pl0, normal) / denom;
        *t_out = t;
        return t >= 0;
    }
    return 0;
}

/* ---- cube::intersect, kernel.cu:399-484 (live part :460-483); max/min are the reference's
 * ternary macros (kernel.cu:16-26), NaN behaviour included ------------------------------ */
#define REF_MAX(a, b) (((a) > (b)) ? (a) : (b))
#define REF_MIN(a, b) (((a) < (b)) ? (a) : (b))
static inline int cube_intersect(v3 O, v3 D, v3 b0, v3 b1, float* t_out) {
    float dirx = 1.f / D.x;
    float diry = 1.f / D.y;
    float dirz = 1.f / D.z;
    float t1 = (b0.x - O.x) * dirx;
    float t2 = (b1.x - O.x) * dirx;
    float t3 = (b0.y - O.y) * diry;
    float t4 = (b1.y - O.y) * diry;
    float t5 = (b0.z - O.z) * dirz;
    float t6 = (b1.z - O.z) * dirz;
    float tmin = REF_MAX(REF_MAX(REF_MIN(t1, t2), REF_MIN(t3, t4)), REF_MIN(t5, t6));
    float tmax = REF_MIN(REF_MIN(REF_MAX(t1, t2), REF_MAX(t3, t4)), REF_MAX(t5, t6));
    if (tmax < 0) {
        *t_out = tmax;
        return 0;
    }
    if (tmax < tmin) {
        *t_out = tmax;
        return 0;
    }
    *t_out = tmin;
    return 1;
}
static inline v3 cube_b0(const oracle_frame* f, int i) { const float* c = f->cubes + 6 * (size_t)i; v3 r = {c[0], c[1], c[2]}; return r; }
static inline v3 cube_b1(const oracle_frame* f, int i) { const float* c = f->cubes + 6 * (size_t)i; v3 r = {c[3], c[4], c[5]}; return r; }
/* cube ctor: orgin = divide(add(c1, c2), 2), kernel.cu:395 */
static inline v3 cube_origin(const oracle_frame* f, int i) {
    v3 a = cube_b0(f, i), b = cube_b1(f, i);
    v3 s = v_add(a, b);
    v3 r = {s.x / 2, s.y / 2, s.z / 2};
    return r;
}
static inline v3 plane_pos(const oracle_frame* f, int i) { const float* c = f->planes + 6 * (size_t)i; v3 r = {c[0], c[1], c[2]}; return r; }
static inline v3 plane_nrm(const oracle_frame* f, int i) { const float* c = f->planes + 6 * (size_t)i; v3 r = {c[3], c[4], c[5]}; return r; }

/* ---- mesh::rayIntersect (Moeller-Trumbore), kernel.cu:1024-1059 ------------------------ */
static inline int tri_intersect(v3 O, v3 D, const float* tri, float* t, float* u, float* v) {
    v3 p0 = {tri[0], tri[1], tri[2]}, p1 = {tri[3], tri[4], tri[5]}, p2 = {tri[6], tri[7], tri[8]};
    v3 edge1 = v_sub(p1, p0);
    v3 edge2 = v_sub(p2, p0);
    v3 h, s, q;
    float a, f;
    h = v_cross(D, edge2);
    a = v_dot(edge1, h);
    if (a > -0.0000001f && a < 0.0000001) return 0;   /* float literal, then DOUBLE literal */
    f = 1.f / a;
    s = v_sub(O, p0);
    *u = f * v_dot(s, h);
    if (*u < 0.f || *u > 1.f) return 0;
    q = v_cross(s, edge1);
    *v = f * v_dot(D, q);
    if (*v < 0.f || *u + *v > 1.f) return 0;
    *t = f * v_dot(edge2, q);
    if (*t > 0.0000001) return 1;                      /* double compare */
    return 0;
}
static inline v3 box_b0(const oracle_frame* f, int j) { const float* c = f->box_bounds + 6 * (size_t)j; v3 r = {c[0], c[1], c[2]}; return r; }
static inline v3 box_b1(const oracle_frame* f, int j) { const float* c = f->box_bounds + 6 * (size_t)j; v3 r = {c[3], c[4], c[5]}; return r; }

/* ---- camera::rotateDir, kernel.cu:248-258 ------------------------------------------- */
static inline v3 rotate_dir(v3 v, float yaw, float pitch) {
    float yawRad = yaw * (3.1415 / 180);
    float pitchRad = pitch * (3.1415 / 180);
    float y = v.y * cosf(pitchRad) - v.z * sinf(pitchRad);
    float z = v.y * sinf(pitchRad) + v.z * cosf(pitchRad);
    float x = v.x * cosf(yawRad) + z * sinf(yawRad);
    z = -v.x * sinf(yawRad) + z * cosf(yawRad);
    v3 r = {x, y, z};
    return r;
}

/* ---- rotate(), kernel.cu:1263-1280 (not a true Rodrigues matrix; kept as written) --- */
typedef struct { float m[3][3]; } m3;
static inline m3 rotate_m(float angle, v3 v) {
    m3 r;
    r.m[0][0] = cosf(angle) + v.x * v.x;
    r.m[0][1] = v.x * v.y * (1.f - cosf(angle)) - v.z * sinf(angle);
    r.m[0][2] = v.x * v.z * (1.f - cosf(angle)) - v.y * sinf(angle);
    r.m[1][0] = v.y * v.x * (1.f - cosf(angle)) + v.z * sinf(angle);
    r.m[1][1] = cosf(angle) + v.y * v.y * (1.f - cosf(angle));   /* `cos(angle)`: float overload */
    r.m[1][2] = v.y * v.z * (1.f - cosf(angle)) - v.x * sinf(angle);
    r.m[2][0] = v.z * v.x * (1.f - cosf(angle)) - v.y * sinf(angle);
    r.m[2][1] = v.z * v.y * (1.f - cosf(angle)) + v.x * sinf(angle);
    r.m[2][2] = cosf(angle) + v.z * v.z * (1.f - cosf(angle));
    return r;
}
/* multiply(matrix, vec3d), kernel.cu:120-128 : v^T * M */
static inline v3 m3_apply(m3 a, v3 v) {
    v3 r;
    r.x = v.x * a.m[0][0] + v.y * a.m[1][0] + v.z * a.m[2][0];
    r.y = v.x * a.m[0][1] + v.y * a.m[1][1] + v.z * a.m[2][1];
    r.z = v.x * a.m[0][2] + v.y * a.m[1][2] + v.z * a.m[2][2];
    return r;
}

/* ---- rgbToInt, kernel.cu:546-556 ---------------------------------------------------- */
uint32_t oracle_rgb_to_int(int r, int g, int b) {
    if (r > 255) r = 255;
    if (g > 255) g = 255;
    if (b > 255) b = 255;
    return (uint32_t)(((r & 0xff) << 16) + ((g & 0xff) << 8) + (b & 0xff));
}

int oracle_sphere_intersect(const float org[3], const float dir[3], const float centre[3],
                            float radius_member, float* t) {
    v3 O = {org[0], org[1], org[2]}, D = {dir[0], dir[1], dir[2]}, c = {centre[0], centre[1], centre[2]};
    float tt = 0.f;
    int hit = sphere_intersect(O, D, c, radius_member, &tt);
    if (t) *t = tt;
    return hit;
}

int oracle_cube_intersect(const float org[3], const float dir[3], const float c1[3], const float c2[3], float* t) {
    v3 O = {org[0], org[1], org[2]}, D = {dir[0], dir[1], dir[2]}, b0 = {c1[0], c1[1], c1[2]}, b1 = {c2[0], c2[1], c2[2]};
    float tt = 0.f;
    int hit = cube_intersect(O, D, b0, b1, &tt);
    if (t) *t = tt;
    return hit;
}

int oracle_plane_intersect(const float org[3], const float dir[3], const float pos[3], const float normal[3], float* t) {
    v3 O = {org[0], org[1], org[2]}, D = {dir[0], dir[1], dir[2]}, p = {pos[0], pos[1], pos[2]};
    v3 n = {normal[0], normal[1], normal[2]};
    float tt = 0.f;
    int hit = plane_intersect(O, D, p, n, &tt);
    if (t) *t = tt;
    return hit;
}

int oracle_tri_intersect(const float org[3], const float dir[3], const float tri[9], float* t, float* u, float* v) {
    v3 O = {org[0], org[1], org[2]}, D = {dir[0], dir[1], dir[2]};
    float tt = 0.f, uu = 0.f, vv = 0.f;
    int hit = tri_intersect(O, D, tri, &tt, &uu, &vv);
    if (t) *t = tt;
    if (u) *u = uu;
    if (v) *v = vv;
    return hit;
}

const char* oracle_kind(void) { return "port"; }

/* only the _ref library (the reference's own loader) can build a mesh from an OBJ file */
int oracle_ref_build_mesh(const char* obj_path, float* tris, int32_t cap_tris, int32_t* n_tris, int32_t* has_normals,
                          float* box_bounds, int32_t* box_offsets, int32_t cap_boxes, int32_t* n_boxes,
                          int32_t* box_indices, int32_t cap_indices) {
    (void)obj_path; (void)tris; (void)cap_tris; (void)n_tris; (void)has_normals; (void)box_bounds; (void)box_offsets;
    (void)cap_boxes; (void)n_boxes; (void)box_indices; (void)cap_indices;
    return 1;
}

/* texel index clamp: the reference reads up to width+1 floats past a plane at the poles
 * (undefined there); the harness defines those reads as the last texel (see
 * ref_build/sprite_raw.cpp, which pads the reference's buffers accordingly). */
static inline int clamp_index(int idx, int n) { return idx < 0 ? 0 : (idx >= n ? n - 1 : idx); }

/* ---- castLightRay, kernel.cu:1432-1544 (sphere scene: mesh/plane/cube loops run 0x) - */
static float cast_light_ray(const oracle_frame* f, v3 start, const float* l, v3 normal, uint64_t* n_tests) {
    float b = 0;
    const v3 lpos = {l[0], l[1], l[2]};
    const float lsize = l[3];
    v3 tmp = v_sub(lpos, start);
    v3 toL = v_normalise(&tmp);                                                          /* :1438 */
    const v3 up = {0, 1, 0}, fwd = {0, 0, 1};
    for (int j = 0; j < 10; j++) {
        v3 P = v_cross(toL, up);                                                         /* :1444 */
        v3 e = v_sub(v_add(lpos, v_scale(P, lsize)), start);
        v3 toEdge = v_normalise(&e);                                                     /* :1450 */
        float angle = cosf((v_dot(toL, toEdge)) * 2);                                    /* :1451 */
        float _z = (float)j / 10 * (1.0f - angle) + angle;                               /* :1453 */
        float phi = (float)j / 10 * 2.f * 3.1415f;                                       /* :1454 */
        float x = sqrtf(1.f - _z * _z) * cosf(phi);                                      /* :1462 */
        float y = sqrtf(1.f - _z * _z) * sinf(phi);                                      /* :1463 */
        v3 n1 = v_normalise(&toL);                 /* mutates toL */                     /* :1465 */
        v3 ax = v_cross(fwd, n1);
        v3 axis = v_normalise(&ax);
        v3 n2 = v_normalise(&toL);                 /* mutates toL again */               /* :1466 */
        float nAngle = acosf(v_dot(n2, fwd));
        v3 xyz = {x, y, _z};
        v3 nd = v_sub(lpos, m3_apply(rotate_m(nAngle, axis), xyz));
        v3 new_dir = v_normalise(&nd);                                                   /* :1468 */
        int shadow = 0;
        int i;
        for (int jb = 0; jb < f->n_boxes && !shadow; jb++) {                             /* :1475-1497 */
            float temp;
            if (cube_intersect(start, new_dir, box_b0(f, jb), box_b1(f, jb), &temp)) {
                for (int k = f->box_offsets[jb]; k < f->box_offsets[jb + 1]; k++) {
                    float t, u, v;
                    if (tri_intersect(start, new_dir, f->tris + 27 * (size_t)f->box_indices[k], &t, &u, &v)) {
                        shadow = 1;
                        break;
                    }
                }
            }
        }
        if (!shadow) {                                                                   /* :1499-1510 */
            for (i = 0; i < f->n_spheres; i++) {
                const float* s = f->spheres + 4 * (size_t)i;
                v3 c = {s[0], s[1], s[2]};
                float t;
                if (sphere_intersect(start, new_dir, c, s[3], &t)) {
                    shadow = 1;
                    break;
                }
            }
            /* sphere::intersect calls this ray made: up to and including its first blocker */
            *n_tests += (uint64_t)(shadow ? i + 1 : f->n_spheres);
        }
        if (!shadow)                                                                     /* planes, :1512-1523 */
            for (i = 0; i < f->n_planes; i++) {
                float t;
                if (plane_intersect(start, new_dir, plane_pos(f, i), plane_nrm(f, i), &t)) {
                    shadow = 1;
                    break;
                }
            }
        if (!shadow)                                                                     /* cubes, :1524-1536 */
            for (i = 0; i < f->n_cubes; i++) {
                float t;
                if (cube_intersect(start, new_dir, cube_b0(f, i), cube_b1(f, i), &t)) {
                    shadow = 1;
                    break;
                }
            }
        if (!shadow) b += 0.1;                     /* float += double */                 /* :1537-1539 */
    }
    float a = v_dot(normal, toL);                                                        /* :1541 */
    b *= a > 0 ? a : 0;
    return b;
}

/* ---- skybox::getFColor, kernel.cu:1146-1166 ----------------------------------------- */
static void sky_color(const oracle_frame* f, v3 O, v3 D, float* r, float* g, float* b) {
    const v3 c0 = {0, 0, 0};
    float t;
    sphere_intersect(O, D, c0, f->sky_size * f->sky_size, &t);      /* ctor squares, :287,1122 */
    v3 hp = v_add(O, v_scale(D, t));
    v3 n = v_sub(hp, c0);
    v_normalise(&n);
    int x = ((1.f + atan2f(n.z, n.x) / 3.1415f) * 0.5f * f->sky_w);
    int y = (acosf(n.y) / 3.1415f * f->sky_h);
    int index = clamp_index(y * f->sky_w + x, f->sky_w * f->sky_h);
    *r = f->sky_r[index];
    *g = f->sky_g[index];
    *b = f->sky_b[index];
}

/* ---- rayTrace, kernel.cu:1614-1690, one pixel ---------------------------------------- */
static uint32_t trace_pixel(const oracle_frame* f, int x, int y, int32_t* id_out, float* t_out, uint64_t* cnt) {
    const int width = f->width, height = f->height;
    const float aspect = f->aspect;
    float dx = aspect * (2 * (x + 0.5) / (float)width) - 1;                              /* :1624 */
    float dy = aspect * (2 * (y + 0.5) / (float)height) * ((float)height / width) - 1;   /* :1625 */
    v3 eyePos = {0, 0, (-1 / aspect)};                                                   /* :1629 */
    v3 dir = {dx, dy, 0};
    v3 camOrg = {f->cam_org[0], f->cam_org[1], f->cam_org[2]};
    v3 d0 = v_sub(dir, eyePos);
    v3 dn = v_normalise(&d0);
    v3 O = v_add(eyePos, camOrg);
    v3 D = rotate_dir(dn, f->cam_yaw, f->cam_pitch);                                     /* :1631 */

    float nt = INFINITY;
    int hit_index = -1;
    int hit_type = 1;
    float nu = 0.f, nv = 0.f;
    /* castRay triangle loop over the flat BVH, kernel.cu:1293-1328 */
    for (int jb = 0; jb < f->n_boxes; jb++) {
        float temp;
        if (cube_intersect(O, D, box_b0(f, jb), box_b1(f, jb), &temp)) {
            for (int k = f->box_offsets[jb]; k < f->box_offsets[jb + 1]; k++) {
                float t, u, v;
                if (tri_intersect(O, D, f->tris + 27 * (size_t)f->box_indices[k], &t, &u, &v)) {
                    if (t < nt) {
                        nt = t;
                        nv = v;
                        nu = u;
                        hit_index = f->box_indices[k];
                        hit_type = 0;
                    }
                }
            }
        }
    }
    /* castRay sphere loop, kernel.cu:1330-1342 */
    for (int i = 0; i < f->n_spheres; i++) {
        const float* s = f->spheres + 4 * (size_t)i;
        v3 c = {s[0], s[1], s[2]};
        float t;
        if (sphere_intersect(O, D, c, s[3], &t)) {
            if (t < nt) {
                nt = t;
                hit_index = i;
                hit_type = 1;
            }
        }
    }
    cnt[0] += (uint64_t)f->n_spheres;
    for (int i = 0; i < f->n_cubes; i++) {                                               /* :1344-1357 */
        float t;
        if (cube_intersect(O, D, cube_b0(f, i), cube_b1(f, i), &t)) {
            if (t < nt) {
                nt = t;
                hit_index = i;
                hit_type = 3;
            }
        }
    }
    for (int i = 0; i < f->n_planes; i++) {                                              /* :1359-1372 */
        float t;
        if (plane_intersect(O, D, plane_pos(f, i), plane_nrm(f, i), &t)) {
            if (t < nt) {
                nt = t;
                hit_index = i;
                hit_type = 2;
            }
        }
    }
    if (id_out) {
        int enc = hit_index;
        if (hit_type == 3) enc += f->n_spheres;
        if (hit_type == 2) enc += f->n_spheres + f->n_cubes;
        if (hit_type == 0) enc += f->n_spheres + f->n_cubes + f->n_planes;
        *id_out = (nt != INFINITY) ? enc : -1;
    }
    if (t_out) *t_out = nt;

    if (nt != INFINITY) {                                                                /* :1375 */
        cnt[3] += 1;
        /* hit attributes: sphere kernel.cu:1396-1405, plane :1407-1416, cube :1417-1425 */
        v3 new_org = v_add(O, v_scale(D, nt));
        v3 normal;
        float tx, ty;
        if (hit_type == 0) {                                                             /* :1380-1394 */
            const float* tr = f->tris + 27 * (size_t)hit_index;
            const v3 vn0 = {tr[12], tr[13], tr[14]}, vn1 = {tr[15], tr[16], tr[17]}, vn2 = {tr[18], tr[19], tr[20]};
            if (f->mesh_has_normals) {
                normal = v_add(v_add(v_scale(vn0, (1 - nu - nv)), v_scale(vn1, nu)), v_scale(vn2, nv));
                v_normalise(&normal);
            } else {
                normal.x = tr[9]; normal.y = tr[10]; normal.z = tr[11];
            }
            tx = ((1 - nu - nv) * tr[21]) + (nu * tr[23]) + (nv * tr[25]);
            ty = ((1 - nu - nv) * tr[22]) + (nu * tr[24]) + (nv * tr[26]);
            new_org = v_add(normal, v_add(O, v_scale(D, nt)));   /* the unit normal is ADDED to the hit point */
        } else if (hit_type == 2) {
            normal = plane_nrm(f, hit_index);
            tx = 0.5;
            ty = 0.5;
        } else {
            v3 c;
            if (hit_type == 1) {
                const float* s = f->spheres + 4 * (size_t)hit_index;
                c.x = s[0]; c.y = s[1]; c.z = s[2];
            } else {
                c = cube_origin(f, hit_index);
            }
            normal = v_sub(new_org, c);
            v_normalise(&normal);
            tx = (1 + atan2f(normal.z, normal.x) / 3.1415) * 0.5;
            ty = acosf(normal.y) / 3.1415;
        }

        int maxX = f->tex_w, maxY = f->tex_h;                                            /* :1643-1644 */
        v3 start_O = v_add(v_scale(normal, 0.00001), new_org);                           /* :1647 */
        int c_index = (int)(ty * maxY) * maxX + (int)(tx * maxX);                        /* :1653 */
        c_index = clamp_index(c_index, maxX * maxY);
        float r = f->tex_r[c_index], g = f->tex_g[c_index], b = f->tex_b[c_index];       /* :1655 */
        float fr = 0, fg = 0, fb = 0;
        for (int i = 0; i < f->n_lights; i++) {                                          /* :1665-1677 */
            const float* l = f->lights + 7 * (size_t)i;
            float brightness = cast_light_ray(f, start_O, l, normal, &cnt[1]);
            fr += brightness * l[4] * r;
            fg += brightness * l[5] * g;
            fb += brightness * l[6] * b;
        }
        return oracle_rgb_to_int(fr * 254, fg * 254, fb * 254);                          /* :1682 */
    }
    float r, g, b;
    cnt[2] += 1;
    sky_color(f, O, D, &r, &g, &b);                                                      /* :1686 */
    return oracle_rgb_to_int(r * 254, g * 254, b * 254);                                 /* :1688 */
}

int oracle_render(const oracle_frame* f, uint32_t* pixels, int32_t* hit_id, float* hit_t,
                  uint64_t* counts, int n_threads) {
    if (!f || f->width <= 0 || f->height <= 0 || f->y_step <= 0) return 1;
    const int W = f->width;
    const int n_rows = (f->y1 - f->y0 + f->y_step - 1) / f->y_step;
    uint64_t c0 = 0, c1 = 0, c2 = 0, c3 = 0;
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#endif
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : c0, c1, c2, c3)
    for (int k = 0; k < n_rows; k++) {
        const int y = f->y0 + k * f->y_step;
        uint64_t cnt[4] = {0, 0, 0, 0};
        for (int x = 0; x < W; x++) {
            size_t o = (size_t)k * W + x;
            uint32_t p = trace_pixel(f, x, y, hit_id ? &hit_id[o] : NULL, hit_t ? &hit_t[o] : NULL, cnt);
            if (pixels) pixels[o] = p;
        }
        c0 += cnt[0];
        c1 += cnt[1];
        c2 += cnt[2];
        c3 += cnt[3];
    }
    if (counts) {
        counts[0] = c0;
        counts[1] = c1;
        counts[2] = c2;
        counts[3] = c3;
    }
    return 0;
}
