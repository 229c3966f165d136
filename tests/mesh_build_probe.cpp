// Test-only C wrapper: the host restatement of the reference's flat-BVH builder (ore_build_flat_bvh, compiled from
// host/ore_mesh.cpp) on raw triangle arrays.  tests/test_mesh_build_cpu.py pins it to the reference's own builder and
// to a transcription of the rule; tests/test_mesh_build_gpu.py compares ore_set_mesh_device's arrays with it.
#include <cstring>

#include "../ray-tracer-engine_b200/host/ore_mesh.h"

// Returns the leaf count (box_bounds6: 6 floats per leaf, box_offsets: leaves + 1, box_indices: box_offsets[leaves]),
// or -1 when the caller's arrays are too small.
extern "C" int ore_probe_build_flat_bvh(const float* tris27, int n_tris, float* box_bounds6, int* box_offsets, int* box_indices,
                                        int cap_boxes, int cap_indices) {
    OreMesh m;
    m.tris.assign(tris27, tris27 + (size_t)n_tris * 27);
    ore_build_flat_bvh(m, 10);
    if (m.n_boxes() > cap_boxes || (int)m.box_indices.size() > cap_indices) return -1;
    if (!m.box_bounds.empty()) std::memcpy(box_bounds6, m.box_bounds.data(), m.box_bounds.size() * sizeof(float));
    std::memcpy(box_offsets, m.box_offsets.data(), m.box_offsets.size() * sizeof(int));
    if (!m.box_indices.empty()) std::memcpy(box_indices, m.box_indices.data(), m.box_indices.size() * sizeof(int));
    return m.n_boxes();
}
