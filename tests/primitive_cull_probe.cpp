// Test-only restatement, in plain g++ (std::fmaf, no -ffp-contract), of the conservative culls the kernels run on cubes
// and mesh leaves, next to the reference's own intersection tests (oracle_cube_intersect / oracle_tri_intersect, passed
// in as function pointers).  tests/test_primitive_cull_cpu.py checks that no cull ever rejects a hit the reference
// reports.  Two forms of each shadow cull: `old`, the predicate before the face-plane guard (a NaN cone test culled),
// and `new`, the kernels' current one (ore_kernels.cuh: zero_axes, on_face_plane, cone_misses_ball).
//
// rsqrt_approx is MUFU.RSQ, within 2^-22 of 1/sqrt: every cull is evaluated at both ends of that interval and counts as
// a cull when either end culls.  The stage-A axis (rsqrtf) gets the same treatment.
#include "ore_mesh_refit.h"   // mesh_box_ball, ORE_KAPPA_SHADOW

#include <cmath>
#include <cstdint>
#include <cstring>

typedef int (*cube_fn)(const float*, const float*, const float*, const float*, float*);
typedef int (*tri_fn)(const float*, const float*, const float*, float*, float*, float*);

namespace {

const double REL[2] = {1.0 - 0x1p-22, 1.0 + 0x1p-22};

float rsqrt_end(float x, int e) {   // MUFU.RSQ: +inf -> +0
    return (float)(1.0 / std::sqrt((double)x) * REL[e]);
}

// ore_set_cubes: centre = (c1 + c2) / 2 in float, radius = half diagonal + margins in double
void cube_ball(const float* c, float q[4]) {
    const double dx = (double)c[3] - c[0], dy = (double)c[4] - c[1], dz = (double)c[5] - c[2];
    const double rad = 0.5 * std::sqrt(dx * dx + dy * dy + dz * dz);
    const double mag = std::fabs((double)c[0]) + std::fabs((double)c[1]) + std::fabs((double)c[2]) + std::fabs((double)c[3]) +
                       std::fabs((double)c[4]) + std::fabs((double)c[5]);
    q[0] = (c[0] + c[3]) / 2;
    q[1] = (c[1] + c[4]) / 2;
    q[2] = (c[2] + c[5]) / 2;
    q[3] = (float)(rad * 1.001 + 1e-5 * mag + 1e-6);
}

void leaf_ball(const float* b, float q[4]) {
    const ore_host::Rec4 r = ore_host::mesh_box_ball(b, b + 3);
    q[0] = r.x;
    q[1] = r.y;
    q[2] = r.z;
    q[3] = r.w;
}

// cone_of10 and the stage-A cone (ore_sweep.cuh): false when the bundle is degenerate (every box is then a candidate)
bool light_cone(const float* d, int e, float A[3], float& ca, float& sa) {
    float sx = 0.f, sy = 0.f, sz = 0.f;
    for (int j = 0; j < 10; j++) {
        sx += d[3 * j];
        sy += d[3 * j + 1];
        sz += d[3 * j + 2];
    }
    const float inv = rsqrt_end(std::fmaf(sx, sx, std::fmaf(sy, sy, sz * sz)), e);
    bool ok = std::isfinite(inv);
    sx *= inv;
    sy *= inv;
    sz *= inv;
    float cmin = 1.f;
    for (int j = 0; j < 10; j++) {
        const float dd = std::fmaf(d[3 * j], d[3 * j], std::fmaf(d[3 * j + 1], d[3 * j + 1], d[3 * j + 2] * d[3 * j + 2]));
        ok = ok && std::fabs(dd - 1.f) < 4e-6f;
        cmin = std::fmin(cmin, std::fmaf(sx, d[3 * j], std::fmaf(sy, d[3 * j + 1], sz * d[3 * j + 2])));
    }
    if (!ok || !(cmin > 0.5f)) return false;
    const float cosa = cmin - 4e-6f;
    const float sina = std::sqrt(std::fmax(0.f, std::fmaf(-cosa, cosa, 1.f))) * 1.0001f + 1e-6f;
    A[0] = sx;
    A[1] = sy;
    A[2] = sz;
    ca = cosa - 0.00196f * sina;
    sa = 1.002f * sina;
    return true;
}

uint32_t zero_axes(const float* d) {
    uint32_t z = 0;
    for (int j = 0; j < 10; j++)
        for (int k = 0; k < 3; k++)
            if (!(std::fabs(d[3 * j + k]) >= 0x1p-126f)) z |= 1u << k;
    return z;
}

bool on_face_plane(uint32_t z, const float* O, const float* b) {
    for (int k = 0; k < 3; k++)
        if (((z >> k) & 1u) && (O[k] == b[k] || O[k] == b[3 + k])) return true;
    return false;
}

// the light-cone test of cubes_planes_block_light / mesh_blocks_light; `old`: a NaN result culls
bool cone_misses_ball(const float q[4], const float* O, const float A[3], float ca, float sa, int e, bool old) {
    const float lx = O[0] - q[0], ly = O[1] - q[1], lz = O[2] - q[2];
    const float LL = std::fmaf(lz, lz, std::fmaf(ly, ly, lx * lx));
    const float Cm = std::fmaf(LL, 1.0f - ORE_KAPPA_SHADOW, -(q[3] * q[3]));
    if (!(Cm > 1e-20f)) return false;
    const float sv = Cm * rsqrt_end(Cm, e);
    const float T = std::fmaf(ca, sv, -(sa * q[3]));
    const float x = std::fmaf(A[0], lx, std::fmaf(A[1], ly, std::fmaf(A[2], lz, T)));
    return old ? !(x < 0.f) : x >= 0.f;
}

// bit 0: the old predicate culls, bit 1: the new one does - for the 10 directions d as one light's bundle
uint32_t shadow_culls(const float q[4], const float* box, const float* O, const float* d) {
    uint32_t out = 0;
    const bool face = on_face_plane(zero_axes(d), O, box);
    for (int e1 = 0; e1 < 2; e1++) {
        float A[3], ca, sa;
        if (!light_cone(d, e1, A, ca, sa)) continue;
        for (int e2 = 0; e2 < 2; e2++) {
            if (cone_misses_ball(q, O, A, ca, sa, e2, true)) out |= 1u;
            if (!face && cone_misses_ball(q, O, A, ca, sa, e2, false)) out |= 2u;
        }
    }
    return out;
}

// nine more directions around D, normalised as the reference does (float divide by a double length): a bundle whose
// first ray is D exactly
void bundle(const float* D, uint64_t seed, float* d) {
    std::memcpy(d, D, 3 * sizeof(float));
    uint64_t s = seed * 6364136223846793005ull + 1442695040888963407ull;
    auto next = [&s]() {
        s = s * 6364136223846793005ull + 1442695040888963407ull;
        return (double)(s >> 11) * 0x1p-53;
    };
    const double spread = 1e-4 + 0.3 * next();
    for (int j = 1; j < 10; j++) {
        float v[3];
        for (int k = 0; k < 3; k++) v[k] = (float)(D[k] + spread * (2.0 * next() - 1.0));
        const double l = std::sqrt((double)v[0] * v[0] + (double)v[1] * v[1] + (double)v[2] * v[2]);
        for (int k = 0; k < 3; k++) d[3 * j + k] = (float)(v[k] / l);
    }
}

}  // namespace

extern "C" {

// Cubes, shadow pass.  Per case i (O, D: 3 floats, box: c1, c2): out[i] bit 0 = the reference reports a hit; bits 1, 2 =
// the old / new cull rejects it for D alone (a bundle of 10 copies); bits 3, 4 = the same for a bundle of D and nine
// directions around it.
void probe_shadow_cubes(cube_fn isect, int n, const float* O, const float* D, const float* box, uint8_t* out) {
    for (int i = 0; i < n; i++) {
        const float *o = O + 3 * (size_t)i, *dir = D + 3 * (size_t)i, *b = box + 6 * (size_t)i;
        float t, q[4], d[30];
        uint32_t r = isect(o, dir, b, b + 3, &t) ? 1u : 0u;
        cube_ball(b, q);
        for (int j = 0; j < 10; j++) std::memcpy(d + 3 * j, dir, 3 * sizeof(float));
        r |= shadow_culls(q, b, o, d) << 1;
        bundle(dir, (uint64_t)i, d);
        r |= shadow_culls(q, b, o, d) << 3;
        out[i] = (uint8_t)r;
    }
}

// Mesh leaves, shadow pass.  box: lo, hi; tri: 9 vertex floats.  Bit 0 = the reference reports a hit on this leaf (slab
// test, then the triangle); bits 1-4 as for cubes, with the leaf ball of mesh_box_ball.
void probe_shadow_leaves(cube_fn isect, tri_fn tri, int n, const float* O, const float* D, const float* box,
                         const float* tris9, uint8_t* out) {
    for (int i = 0; i < n; i++) {
        const float *o = O + 3 * (size_t)i, *dir = D + 3 * (size_t)i, *b = box + 6 * (size_t)i;
        float t, u, v, q[4], d[30];
        uint32_t r = (isect(o, dir, b, b + 3, &t) && tri(o, dir, tris9 + 9 * (size_t)i, &t, &u, &v)) ? 1u : 0u;
        leaf_ball(b, q);
        for (int j = 0; j < 10; j++) std::memcpy(d + 3 * j, dir, 3 * sizeof(float));
        r |= shadow_culls(q, b, o, d) << 1;
        bundle(dir, (uint64_t)i, d);
        r |= shadow_culls(q, b, o, d) << 3;
        out[i] = (uint8_t)r;
    }
}

// Mesh leaves, primary pass: ball_records (prep_frame_kernel) for an eye O with yaw = pitch = 0 (camera frame = world
// frame) and a tile of half-angle asin(1e-3) whose axis is D; cone_touches decides.  Bit 0 = reported hit, bit 1 = the
// cull without the eye-on-a-face-plane rule rejects it, bit 2 = with it.
void probe_primary_leaves(cube_fn isect, tri_fn tri, int n, const float* O, const float* D, const float* box,
                          const float* tris9, uint8_t* out) {
    const double a = std::asin(1e-3) * 1.001 + 1e-6;
    const float tile_ca = (float)(std::cos(a) * (1.0 - 1e-6) - 1e-6), tile_sa = (float)(std::sin(a) * (1.0 + 1e-6) + 1e-6);
    const double KP = 0x1p-17;   // ORE_KAPPA_PRIMARY (ore_kernels.cuh)
    for (int i = 0; i < n; i++) {
        const float *o = O + 3 * (size_t)i, *dir = D + 3 * (size_t)i, *b = box + 6 * (size_t)i;
        float t, u, v, q[4];
        uint32_t r = (isect(o, dir, b, b + 3, &t) && tri(o, dir, tris9 + 9 * (size_t)i, &t, &u, &v)) ? 1u : 0u;
        leaf_ball(b, q);
        const double Lx = (double)o[0] - q[0], Ly = (double)o[1] - q[1], Lz = (double)o[2] - q[2], r2 = (double)q[3] * q[3];
        const double LL = Lx * Lx + Ly * Ly + Lz * Lz;
        const double Cm = LL * (1.0 - KP) - r2 * (1.0 + KP);
        bool cand = true;
        if (Cm > 1e-9 * LL && Cm > 1e-30) {
            const double sv = std::sqrt(Cm), Rpp = std::sqrt(LL - Cm);
            const double Wd = (double)tile_ca * sv - (double)tile_sa * Rpp;
            const float rec[4] = {(float)Lx, (float)Ly, (float)Lz, (float)(Wd - 4e-6 * std::sqrt(LL) - 1e-30)};
            cand = std::fmaf(dir[0], rec[0], std::fmaf(dir[1], rec[1], std::fmaf(dir[2], rec[2], rec[3]))) <= 0.f;
        }
        if (!cand) r |= 2u;
        if (!cand && !on_face_plane(7u, o, b)) r |= 4u;
        out[i] = (uint8_t)r;
    }
}

}  // extern "C"
