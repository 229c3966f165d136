// ore_mesh_refit.h - the leaf boxes of the triangle mesh's flat BVH and their bounding spheres: the arithmetic shared by
// the device refit (ore_mesh_refit.cu) and the host functions below, which are the CPU reference the tests compare the
// device arrays with (tests/test_mesh_refit_cpu.py, tests/test_mesh_update_gpu.py).  No CUDA types outside the
// __CUDACC__ block; the rest is also compiled by plain g++.
//
// The topology (which triangles each leaf lists) comes from the reference's builder on the host and never changes here;
// only the boxes follow moved vertices.  With --fmad=false on the device and no FMA on the host, both sides give the
// same bits.
#ifndef ORE_MESH_REFIT_H
#define ORE_MESH_REFIT_H
#include "ore_clusters.h"   // ORE_HD, Rec4

namespace ore_host {

constexpr int TRI_FLOATS = 27;   // points[3], normal, vecNormal[3], vt[3]; the vertices are floats [0, 9)

// getMinMaxP's rule on one axis (kernel.cu:973-997; bounds_of in host/ore_mesh.cpp): a vertex coordinate replaces the
// running extreme only when it lies strictly beyond it.  So a NaN is never taken, a NaN extreme is never replaced, and
// of equal values (-0, +0) the one met first stays.
ORE_HD inline void grow_hi(float v, float& hi) {
    if (v > hi) hi = v;
}
ORE_HD inline void grow_lo(float v, float& lo) {
    if (v < lo) lo = v;
}

// The same rule as a reduction (the device refit and build): (v, p) <- (w, q) when w is beyond v, or equal to it and
// earlier in the list, or when (v, p) holds nothing yet (v NaN).  A NaN w never displaces a coordinate (both comparisons
// are false), and displacing "nothing" by a NaN still holds nothing.  "Larger value, or equal value and earlier position"
// is associative and commutative, so the order of reduction does not matter.
ORE_HD inline void take_hi(float& v, int& p, float w, int q) {
    if (w > v || (w == v && q < p) || isnan(v)) {
        v = w;
        p = q;
    }
}
ORE_HD inline void take_lo(float& v, int& p, float w, int q) {
    if (w < v || (w == v && q < p) || isnan(v)) {
        v = w;
        p = q;
    }
}

// The seed step: the seeds come first in the rule's order (lo from the first listed triangle's first vertex, hi from the
// last listed triangle's), and the reduced extremes (NaN: none taken) replace them only when strictly beyond.
ORE_HD inline void seed_and_grow(const float* first, const float* last, const float lo_ext[3], const float hi_ext[3], float lo[3],
                                 float hi[3]) {
    for (int k = 0; k < 3; k++) {
        lo[k] = first[k];
        hi[k] = last[k];
        grow_lo(lo_ext[k], lo[k]);
        grow_hi(hi_ext[k], hi[k]);
    }
}

// CPU reference of a leaf box: lo seeded with the first listed triangle's first vertex, hi with the last listed
// triangle's, then every vertex of every listed triangle grows them in list order.  m == 0: the box is left as it is.
inline void mesh_leaf_box(const float* tris27, const int32_t* idx, int m, float lo[3], float hi[3]) {
    if (m <= 0) return;
    for (int k = 0; k < 3; k++) {
        lo[k] = tris27[(size_t)idx[0] * TRI_FLOATS + k];
        hi[k] = tris27[(size_t)idx[m - 1] * TRI_FLOATS + k];
    }
    for (int i = 0; i < m; i++) {
        const float* t = tris27 + (size_t)idx[i] * TRI_FLOATS;
        for (int v = 0; v < 3; v++)
            for (int k = 0; k < 3; k++) {
                grow_hi(t[3 * v + k], hi[k]);
                grow_lo(t[3 * v + k], lo[k]);
            }
    }
}

// NaN bits of the ball below.  The formula used to run on the host only, where x86 arithmetic passes the first NaN
// operand through (quietened) and makes the "default NaN" (sign set) from numbers (inf - inf); a device returns its
// canonical NaN instead.  These helpers give the x86 bits on both sides, so the ball keeps the bytes it always had.
ORE_HD inline uint32_t f32_bits(float v) {
    uint32_t u;
    memcpy(&u, &v, sizeof u);
    return u;
}
ORE_HD inline float f32_of(uint32_t u) {
    float v;
    memcpy(&v, &u, sizeof v);
    return v;
}
ORE_HD inline float x86_quiet(float v) { return f32_of(f32_bits(v) | 0x00400000u); }
// fabs of a NaN with its payload kept.  Written as an integer AND, the device compiler recognises fabsf, and the device's
// fabsf returns its canonical NaN; the PTX `and` keeps the bits.
ORE_HD inline float x86_fabs_nan(float v) {
    uint32_t u = f32_bits(v);
#if defined(__CUDA_ARCH__)
    asm("and.b32 %0, %1, 0x7fffffff;" : "=r"(u) : "r"(u));
#else
    u &= 0x7fffffffu;
#endif
    return f32_of(u);
}
constexpr uint32_t X86_DEFAULT_NAN = 0xffc00000u;
// NaN of (double)a op b: a's if a is NaN, else b's, else the default NaN
ORE_HD inline float x86_nan2(float a, float b) {
    return isnan(a) ? x86_quiet(a) : isnan(b) ? x86_quiet(b) : f32_of(X86_DEFAULT_NAN);
}

// Bounding sphere of a leaf box for the conservative cone filters: centre, half diagonal + 0.1 % + a little absolute
// slack (the float slab test can accept a ray that misses the true box by rounding).  In double.
ORE_HD inline Rec4 mesh_box_ball(const float lo[3], const float hi[3]) {
    const double cx = 0.5 * ((double)lo[0] + hi[0]), cy = 0.5 * ((double)lo[1] + hi[1]), cz = 0.5 * ((double)lo[2] + hi[2]);
    const double dx = (double)hi[0] - lo[0], dy = (double)hi[1] - lo[1], dz = (double)hi[2] - lo[2];
    const double rad = 0.5 * sqrt(dx * dx + dy * dy + dz * dz);
    const double mag = fabs(cx) + fabs(cy) + fabs(cz) + rad;
    Rec4 b{(float)cx, (float)cy, (float)cz, (float)(rad * 1.001 + 1e-5 * mag + 1e-6)};
    // which results are NaN, decided from the inputs alone: lo + hi is NaN for a NaN or for infinities of opposite
    // signs, hi - lo for a NaN or for equal infinities; the radius (through mag, which holds rad) whenever any is
    bool cnan[3], dnan[3], any = false;
    for (int k = 0; k < 3; k++) {
        const bool n = isnan(lo[k]) || isnan(hi[k]), inf2 = isinf(lo[k]) && isinf(hi[k]);
        cnan[k] = n || (inf2 && lo[k] != hi[k]);
        dnan[k] = n || (inf2 && lo[k] == hi[k]);
        any = any || cnan[k] || dnan[k];
    }
    if (!any) return b;
    // the x86 NaNs: a centre coordinate's from lo + hi; the radius's from mag, the first NaN of |cx| + |cy| + |cz| + rad
    // - a centre's without its sign, or else rad's from the first NaN difference hi - lo
    float cn[3] = {b.x, b.y, b.z}, rn = b.w;
    for (int k = 0; k < 3; k++)
        if (cnan[k]) cn[k] = x86_nan2(lo[k], hi[k]);
    bool found = false;
    for (int k = 0; k < 3 && !found; k++)
        if (cnan[k]) {
            rn = x86_fabs_nan(cn[k]);
            found = true;
        }
    for (int k = 0; k < 3 && !found; k++)
        if (dnan[k]) {
            rn = x86_nan2(hi[k], lo[k]);
            found = true;
        }
    return Rec4{cn[0], cn[1], cn[2], rn};
}

}  // namespace ore_host

#if defined(__CUDACC__)
#include <cuda_runtime.h>
// Enqueued on `stream`; neither allocates nor blocks the host.
// Leaf boxes (2 float4 per leaf: lo, hi; .w = 0) of the n_boxes leaves from the triangles at tris27 and the leaf lists
// box_indices[box_offsets[j] .. box_offsets[j + 1]).  A leaf with no triangles keeps its box.
cudaError_t ore_mesh_refit(const float* tris27, const int* box_offsets, const int* box_indices, float4* boxes, int n_boxes,
                           cudaStream_t stream);
// box_sph[j] = mesh_box_ball of boxes[2j], boxes[2j + 1]
cudaError_t ore_mesh_balls(const float4* boxes, float4* box_sph, int n_boxes, cudaStream_t stream);
#endif
#endif
