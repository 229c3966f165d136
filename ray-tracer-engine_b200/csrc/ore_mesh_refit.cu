// ore_mesh_refit.cu - the mesh's leaf boxes and their bounding spheres on the device (sm_100a, --fmad=false).
//
//   mesh_refit_kernel  one warp per leaf: the lanes stride over the leaf's list, each keeps per axis the extreme of the
//                      vertices it read together with its position in list order, and a butterfly reduction over
//                      (value, position) pairs gives the coordinate getMinMaxP's sequential rule takes; one lane then
//                      applies the rule's seeds (grow_lo / grow_hi of ore_mesh_refit.h)
//   mesh_balls_kernel  one thread per leaf: mesh_box_ball, in double
//
// The sequential rule takes, per axis, the FIRST of the coordinates that compare as the maximum (strict `>`: of -0 and
// +0 the earlier stays), never a NaN, and keeps a NaN seed.  Reducing (value, position) with "larger value, or equal
// value and earlier position" is associative and commutative, so the lanes' order of reading does not matter and the
// result has the rule's bits (tests/test_mesh_update_gpu.py checks them byte for byte against the host functions).
#include "ore_mesh_refit.h"

namespace {

constexpr int REFIT_THREADS = 256;
constexpr unsigned FULL = 0xffffffffu;
constexpr int NO_POS = 0x7fffffff;   // with a NaN value: no coordinate taken yet

using ore_host::take_hi;
using ore_host::take_lo;

__global__ void __launch_bounds__(REFIT_THREADS) mesh_refit_kernel(const float* __restrict__ tris, const int* __restrict__ offs,
                                                                   const int* __restrict__ idx, float4* __restrict__ boxes,
                                                                   int n_boxes) {
    const int j = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);   // warp-uniform
    const int lane = threadIdx.x & 31;
    if (j >= n_boxes) return;
    const int o0 = offs[j], m = offs[j + 1] - o0;
    if (m <= 0) return;   // a leaf with no triangles keeps its box
    float lo[3], hi[3];
    int plo[3], phi[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        lo[k] = hi[k] = __int_as_float(0x7fffffff);
        plo[k] = phi[k] = NO_POS;
    }
    // position of vertex v of list entry i: 3 i + v (the rule's reading order); the lanes read in increasing position
    for (int i = lane; i < m; i += 32) {
        const float* t = tris + (size_t)idx[o0 + i] * ore_host::TRI_FLOATS;
#pragma unroll
        for (int v = 0; v < 3; v++)
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const float w = __ldg(t + 3 * v + k);
                take_hi(hi[k], phi[k], w, 3 * i + v);
                take_lo(lo[k], plo[k], w, 3 * i + v);
            }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1)
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const float wh = __shfl_xor_sync(FULL, hi[k], o), wl = __shfl_xor_sync(FULL, lo[k], o);
            const int qh = __shfl_xor_sync(FULL, phi[k], o), ql = __shfl_xor_sync(FULL, plo[k], o);
            take_hi(hi[k], phi[k], wh, qh);
            take_lo(lo[k], plo[k], wl, ql);
        }
    if (lane != 0) return;
    // the seeds come first in the rule's order: the reduced coordinate replaces one only when strictly beyond it
    float blo[3], bhi[3];
    ore_host::seed_and_grow(tris + (size_t)idx[o0] * ore_host::TRI_FLOATS, tris + (size_t)idx[o0 + m - 1] * ore_host::TRI_FLOATS,
                            lo, hi, blo, bhi);
    boxes[2 * j] = make_float4(blo[0], blo[1], blo[2], 0.f);
    boxes[2 * j + 1] = make_float4(bhi[0], bhi[1], bhi[2], 0.f);
}

__global__ void __launch_bounds__(REFIT_THREADS) mesh_balls_kernel(const float4* __restrict__ boxes, float4* __restrict__ box_sph,
                                                                   int n_boxes) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_boxes) return;
    const float4 a = boxes[2 * j], b = boxes[2 * j + 1];
    const float lo[3] = {a.x, a.y, a.z}, hi[3] = {b.x, b.y, b.z};
    const ore_host::Rec4 s = ore_host::mesh_box_ball(lo, hi);
    box_sph[j] = make_float4(s.x, s.y, s.z, s.w);
}

}  // namespace

cudaError_t ore_mesh_refit(const float* tris27, const int* box_offsets, const int* box_indices, float4* boxes, int n_boxes,
                           cudaStream_t stream) {
    if (n_boxes <= 0) return cudaSuccess;
    const int warps_per_block = REFIT_THREADS / 32;
    mesh_refit_kernel<<<(n_boxes + warps_per_block - 1) / warps_per_block, REFIT_THREADS, 0, stream>>>(tris27, box_offsets,
                                                                                                       box_indices, boxes, n_boxes);
    return cudaGetLastError();
}

cudaError_t ore_mesh_balls(const float4* boxes, float4* box_sph, int n_boxes, cudaStream_t stream) {
    if (n_boxes <= 0) return cudaSuccess;
    mesh_balls_kernel<<<(n_boxes + REFIT_THREADS - 1) / REFIT_THREADS, REFIT_THREADS, 0, stream>>>(boxes, box_sph, n_boxes);
    return cudaGetLastError();
}
