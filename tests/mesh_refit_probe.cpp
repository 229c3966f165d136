// Test-only C wrapper: the host functions of csrc/ore_mesh_refit.h producing the mesh's leaf boxes and bounding spheres
// exactly as the device holds them after ore_set_mesh (refit = 0: the caller's boxes) or after
// ore_set_mesh_triangles_device (refit = 1: boxes recomputed from the triangles; a leaf listing no triangle keeps the box
// it had).  tests/test_mesh_update_gpu.py compares them byte for byte with ore_debug_mesh.
#include "ore_mesh_refit.h"

#include <cmath>

using ore_host::Rec4;

// boxes6: n_boxes x {lo.xyz, hi.xyz} before the call; boxes_out: 2 n_boxes float4 (lo, 0, hi, 0); box_sph: n_boxes float4
extern "C" void ore_probe_mesh(const float* tris27, const int* box_offsets, const int* box_indices, int n_boxes, const float* boxes6,
                               int refit, float* boxes_out, float* box_sph) {
    for (int j = 0; j < n_boxes; j++) {
        float lo[3] = {boxes6[6 * j], boxes6[6 * j + 1], boxes6[6 * j + 2]};
        float hi[3] = {boxes6[6 * j + 3], boxes6[6 * j + 4], boxes6[6 * j + 5]};
        if (refit) ore_host::mesh_leaf_box(tris27, box_indices + box_offsets[j], box_offsets[j + 1] - box_offsets[j], lo, hi);
        const float b[8] = {lo[0], lo[1], lo[2], 0.f, hi[0], hi[1], hi[2], 0.f};
        std::memcpy(boxes_out + 8 * (size_t)j, b, sizeof b);
        const Rec4 s = ore_host::mesh_box_ball(lo, hi);
        std::memcpy(box_sph + 4 * (size_t)j, &s, sizeof s);
    }
}

// The host loop ore_set_mesh ran before the ball moved to a kernel, verbatim: the bytes mesh_box_ball must keep.
extern "C" void ore_probe_host_ball_before(const float* b, float* out) {
    const double cx = 0.5 * ((double)b[0] + b[3]), cy = 0.5 * ((double)b[1] + b[4]), cz = 0.5 * ((double)b[2] + b[5]);
    const double dx = (double)b[3] - b[0], dy = (double)b[4] - b[1], dz = (double)b[5] - b[2];
    const double rad = 0.5 * sqrt(dx * dx + dy * dy + dz * dz);
    const double mag = fabs(cx) + fabs(cy) + fabs(cz) + rad;
    const float s[4] = {(float)cx, (float)cy, (float)cz, (float)(rad * 1.001 + 1e-5 * mag + 1e-6)};
    std::memcpy(out, s, sizeof s);
}

extern "C" void ore_probe_mesh_box_ball(const float* b, float* out) {
    const Rec4 s = ore_host::mesh_box_ball(b, b + 3);
    std::memcpy(out, &s, sizeof s);
}
