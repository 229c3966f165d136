// ore_mesh_build.h - the reference's flat BVH over the mesh's triangles (createBvhMesh, kernel.cu:782-936; its CPU
// restatement is ore_build_flat_bvh in host/ore_mesh.cpp) built on the device from device triangles, stream-ordered.
#ifndef ORE_MESH_BUILD_H
#define ORE_MESH_BUILD_H
#include <cuda_runtime.h>

#include <cstddef>

constexpr int ORE_MESH_LAYERS = 10;       // the reference's layer count
constexpr int ORE_MESH_MAX_LEAVES = 1024; // 2^10: every layer at most doubles the boxes

// leaf capacity of a device build of n_tris triangles: the leaf count is at most this, and is known on the device only
inline int ore_mesh_leaf_capacity(int n_tris) { return n_tris < ORE_MESH_MAX_LEAVES ? n_tris : ORE_MESH_MAX_LEAVES; }

// bytes of work space a build of up to cap_tris triangles needs (second index buffer, flags and their scan, the scan's
// temporary storage, the per-layer box arrays)
cudaError_t ore_mesh_build_bytes(int cap_tris, size_t* bytes);

// The buffers of one build.  Nothing here depends on the triangle count n: it is read on the device (written by
// ore_mesh_build_count), so the launch sequence of ore_mesh_build is the same for every n up to cap_tris and can be
// captured once per buffer set as a CUDA graph.
struct MeshBuildArgs {
    const float* tris;   // n x 27 floats (device)
    int cap_tris;        // capacity: every grid is sized from it; the work space was sized by ore_mesh_build_bytes(cap_tris)
    int* box_offsets;    // out: leaf j lists box_indices[box_offsets[j] .. box_offsets[j + 1]); = n past the live count
                         //      (ore_mesh_leaf_capacity(n) + 1 entries are written)
    int* box_indices;    // out: n entries (also the build's first index buffer)
    float4* boxes;       // out: lo, hi per leaf (.w = 0); zeros past the live count
    float4* box_sph;     // out: mesh_box_ball of each live leaf; zeros past the live count
    int* n_live;         // out: the leaf count (1 int)
    void* work;          // ore_mesh_build_bytes(cap_tris) bytes
    size_t work_bytes;
};

// Enqueued on `stream`: sets the triangle count (1 <= n <= cap_tris) the next ore_mesh_build on the same work space reads.
cudaError_t ore_mesh_build_count(const MeshBuildArgs& a, int n, cudaStream_t stream);
// Enqueued on `stream` (about 65 launches, all sized from cap_tris); neither allocates nor blocks the host.
cudaError_t ore_mesh_build(const MeshBuildArgs& a, cudaStream_t stream);

#endif
