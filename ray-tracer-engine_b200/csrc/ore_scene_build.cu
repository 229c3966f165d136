// ore_scene_build.cu - the sphere hierarchy of ore_clusters.h built on the device (sm_100a, --fmad=false).
//
//   scene_bbox_kernel    per sphere: copy into sph_exact; per-axis min / max of the TAME centres (order-independent:
//                        atomics on order-preserving integer keys give the host loop's values)
//   scene_keys_kernel    30-bit Morton key of every centre with the host's double arithmetic (morton_key)
//   cub radix sort       stable sort of (key, original index) over bits [0, 30): std::stable_sort's permutation
//   scene_gather_kernel  sorted exact + shadow records (R' = shadow_radius), sort_index, padding to 32
//   scene_balls_kernel   leaf balls (one thread per leaf: bounding_ball itself) and super balls (one warp per super:
//                        box and max radius reduced across lanes, the mean summed by one lane in member order)
//   scene_hypers_kernel  large scenes only: hyper balls over the super balls (one thread per hyper: bounding_ball)
//
// Every value is computed by the ORE_HD helpers the host builder uses, with the same double expressions; only the
// order of min / max reductions differs, and min / max of finite values do not depend on it.  So the arrays are
// bit-identical to the host builder's (tests/test_scene_update_gpu.py checks them byte for byte).
#include <cub/device/device_radix_sort.cuh>

#include "ore_clusters.h"
#include "ore_scene_build.h"

using ore_host::Rec4;

namespace {

constexpr int BUILD_THREADS = 256;
constexpr unsigned FULL = 0xffffffffu;
constexpr uint32_t NO_KEY = 0xffffffffu;   // NaN's key: never the key of a tame value
constexpr int SUPER_SPHERES = ore_host::LEAF_SPHERES * ore_host::SUPER_LEAVES;

// float -> uint32 with the same order (-0 < +0); min over keys = min over values
__device__ __forceinline__ uint32_t ordered_key(float v) {
    const uint32_t u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ordered_value(uint32_t k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }
__device__ __forceinline__ Rec4 as_rec(float4 v) { return Rec4{v.x, v.y, v.z, v.w}; }
__device__ __forceinline__ float4 as_f4(const Rec4& r) { return make_float4(r.x, r.y, r.z, r.w); }

// bbox[k]: min key of the tame centres on axis k; bbox[3 + k]: min of ~key (= max).  NO_KEY: no tame centre on the axis.
__global__ void __launch_bounds__(BUILD_THREADS) scene_bbox_kernel(const float4* src, float4* sph_exact, int n, uint32_t* bbox) {
    uint32_t mn[6] = {NO_KEY, NO_KEY, NO_KEY, NO_KEY, NO_KEY, NO_KEY};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 v = src[i];
        if (src != sph_exact) sph_exact[i] = v;
        const float c[3] = {v.x, v.y, v.z};
#pragma unroll
        for (int k = 0; k < 3; k++)
            if (ore_host::tame_value(c[k])) {
                const uint32_t key = ordered_key(c[k]);
                mn[k] = min(mn[k], key);
                mn[3 + k] = min(mn[3 + k], ~key);
            }
    }
#pragma unroll
    for (int k = 0; k < 6; k++) mn[k] = __reduce_min_sync(FULL, mn[k]);
    if ((threadIdx.x & 31) == 0)
        for (int k = 0; k < 6; k++)
            if (mn[k] != NO_KEY) atomicMin(&bbox[k], mn[k]);
}

__global__ void __launch_bounds__(BUILD_THREADS) scene_keys_kernel(const float4* sph_exact, int n, const uint32_t* bbox,
                                                                   uint32_t* keys, int* vals) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    // the host loop's initial values (1e300, -1e300) where an axis has no tame centre: that axis contributes 0
    double lo[3], hi[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const bool any = bbox[k] != NO_KEY;
        lo[k] = any ? (double)ordered_value(bbox[k]) : 1e300;
        hi[k] = any ? (double)ordered_value(~bbox[3 + k]) : -1e300;
    }
    keys[i] = ore_host::morton_key(as_rec(sph_exact[i]), lo, hi);
    vals[i] = i;
}

__global__ void __launch_bounds__(BUILD_THREADS) scene_gather_kernel(float4* sph_exact, int n, const int* order, int n_sort,
                                                                     float4* xsort, float4* ssort, int* sort_index) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_sort) return;
    if (n == 0) {   // empty scene: one block of padding records (never read: every loop is bounded by n = 0)
        const float4 pad = make_float4(3e18f, -1e18f, 2e17f, 0.f);
        xsort[p] = pad;
        ssort[p] = pad;
        sort_index[p] = 0;
        if (p == 0) sph_exact[0] = make_float4(0.f, 0.f, 0.f, 0.f);
        return;
    }
    const int i = order[p < n ? p : n - 1];   // the tail repeats the last sorted sphere
    const float4 e = sph_exact[i];
    xsort[p] = e;
    ssort[p] = make_float4(e.x, e.y, e.z, ore_host::shadow_radius(e.w));
    sort_index[p] = i;
}

__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const double w = __shfl_xor_sync(FULL, v, o);
        v = w < v ? w : v;
    }
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const double w = __shfl_xor_sync(FULL, v, o);
        v = v < w ? w : v;
    }
    return v;
}

// bounding_ball of the m <= 256 sorted shadow records g[0, m) by one warp (same values: see the file comment); the
// members are staged in the warp's shared-memory slice s first, so that the one sequential sum reads shared memory
__device__ Rec4 warp_bounding_ball(const float4* g, int m, float4* s) {
    const int lane = threadIdx.x & 31;
    for (int p = lane; p < m; p += 32) s[p] = g[p];
    __syncwarp();
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    bool tame = true;
    for (int p = lane; p < m; p += 32) {
        const Rec4 r = as_rec(s[p]);
        tame = tame && ore_host::tame_record(r);
        const double c[3] = {r.x, r.y, r.z}, rr = fabs((double)r.w);
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const double a = c[k] - rr, b = c[k] + rr;
            lo[k] = a < lo[k] ? a : lo[k];
            hi[k] = hi[k] < b ? b : hi[k];
        }
    }
    if (!__all_sync(FULL, tame)) return Rec4{0.f, 0.f, 0.f, INFINITY};
    double mean[3] = {0, 0, 0};
    if (lane == 0)
#pragma unroll 8
        for (int p = 0; p < m; p++) {   // the one order-dependent sum: in member order, as the host does
            const float4 v = s[p];
            mean[0] += (double)v.x;
            mean[1] += (double)v.y;
            mean[2] += (double)v.z;
        }
#pragma unroll
    for (int k = 0; k < 3; k++) {
        mean[k] = __shfl_sync(FULL, mean[k], 0);
        lo[k] = warp_min(lo[k]);
        hi[k] = warp_max(hi[k]);
    }
    Rec4 best{0.f, 0.f, 0.f, INFINITY};
    for (int cand = 0; cand < 2; cand++) {
        float f[3];
        ore_host::ball_candidate(cand, mean, lo, hi, (double)m, f);
        double rad = 0;
        for (int p = lane; p < m; p += 32) {
            const double d = ore_host::member_reach(as_rec(s[p]), f);
            rad = rad < d ? d : rad;
        }
        rad = warp_max(rad);
        if (ore_host::boundable(rad)) {
            const float fr = ore_host::rounded_radius(rad);
            if (fr < best.w) best = Rec4{f[0], f[1], f[2], fr};
        }
    }
    return best;
}

// blocks [0, leaf_blocks): one thread per leaf (padding: radius -1); the rest: one warp per super-cluster
__global__ void __launch_bounds__(BUILD_THREADS) scene_balls_kernel(const float4* ssort, int n, float4* leaf_sph, int n_leaves,
                                                                    int n_leaves_pad, float4* super_sph, int n_supers,
                                                                    int n_supers_pad, int leaf_blocks) {
    const float4 pad = make_float4(0.f, 0.f, 0.f, -1.f);
    if ((int)blockIdx.x < leaf_blocks) {
        const int j = blockIdx.x * blockDim.x + threadIdx.x;
        if (j >= n_leaves_pad) return;
        if (j >= n_leaves) {
            leaf_sph[j] = pad;
            return;
        }
        const int p0 = j * ore_host::LEAF_SPHERES, m = min(ore_host::LEAF_SPHERES, n - p0);
        leaf_sph[j] = as_f4(ore_host::bounding_ball(reinterpret_cast<const Rec4*>(ssort + p0), (size_t)m));
        return;
    }
    __shared__ float4 s_members[BUILD_THREADS / 32][SUPER_SPHERES];   // (leaf blocks return above without touching it)
    const int k = (((int)blockIdx.x - leaf_blocks) * blockDim.x + threadIdx.x) >> 5;   // warp-uniform
    if (k >= n_supers_pad) return;
    if (k >= n_supers) {
        if ((threadIdx.x & 31) == 0) super_sph[k] = pad;
        return;
    }
    const int p0 = k * SUPER_SPHERES;
    const Rec4 b = warp_bounding_ball(ssort + p0, min(SUPER_SPHERES, n - p0), s_members[threadIdx.x >> 5]);
    if ((threadIdx.x & 31) == 0) super_sph[k] = as_f4(b);
}

// large scenes only: one thread per hyper-cluster, bounding_ball itself over its <= 32 super balls (padding: radius -1)
__global__ void __launch_bounds__(BUILD_THREADS) scene_hypers_kernel(const float4* super_sph, int n_supers, float4* hyper_sph,
                                                                     int n_hypers, int n_hypers_pad) {
    const int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= n_hypers_pad) return;
    if (h >= n_hypers) {
        hyper_sph[h] = make_float4(0.f, 0.f, 0.f, -1.f);
        return;
    }
    const int k0 = h * ore_host::HYPER_SUPERS, m = min(ore_host::HYPER_SUPERS, n_supers - k0);
    hyper_sph[h] = as_f4(ore_host::bounding_ball(reinterpret_cast<const Rec4*>(super_sph + k0), (size_t)m));
}

}  // namespace

cudaError_t ore_scene_sort_bytes(int n, size_t* bytes) {
    *bytes = 0;
    return cub::DeviceRadixSort::SortPairs(nullptr, *bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const int*)nullptr,
                                           (int*)nullptr, n > 0 ? n : 1, 0, 30);
}

cudaError_t ore_scene_build(const SceneBuildArgs& a, cudaStream_t stream) {
    static_assert(sizeof(Rec4) == sizeof(float4), "Rec4 must have float4's layout");
    const int n = a.n;
    cudaError_t e;
    if (n > 0) {
        if ((e = cudaMemsetAsync(a.bbox, 0xff, 6 * sizeof(uint32_t), stream)) != cudaSuccess) return e;
        const int blocks = (n + BUILD_THREADS - 1) / BUILD_THREADS;
        scene_bbox_kernel<<<blocks < 1024 ? blocks : 1024, BUILD_THREADS, 0, stream>>>(a.src, a.sph_exact, n, a.bbox);
        scene_keys_kernel<<<blocks, BUILD_THREADS, 0, stream>>>(a.sph_exact, n, a.bbox, a.keys_in, a.vals_in);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        size_t tmp = a.sort_tmp_bytes;
        if ((e = cub::DeviceRadixSort::SortPairs(a.sort_tmp, tmp, a.keys_in, a.keys_out, a.vals_in, a.vals_out, n, 0, 30, stream)) !=
            cudaSuccess)
            return e;
    }
    scene_gather_kernel<<<(a.n_sort + BUILD_THREADS - 1) / BUILD_THREADS, BUILD_THREADS, 0, stream>>>(
        a.sph_exact, n, a.vals_out, a.n_sort, a.sph_xsort, a.sph_sort, a.sort_index);
    if (a.n_leaves_pad > 0 || a.n_supers_pad > 0) {
        const int leaf_blocks = (a.n_leaves_pad + BUILD_THREADS - 1) / BUILD_THREADS;
        const int warps_per_block = BUILD_THREADS / 32;
        const int super_blocks = (a.n_supers_pad + warps_per_block - 1) / warps_per_block;
        scene_balls_kernel<<<leaf_blocks + super_blocks, BUILD_THREADS, 0, stream>>>(a.sph_sort, n, a.leaf_sph, a.n_leaves,
                                                                                      a.n_leaves_pad, a.super_sph, a.n_supers,
                                                                                      a.n_supers_pad, leaf_blocks);
    }
    if (a.n_hypers_pad > 0)
        scene_hypers_kernel<<<(a.n_hypers_pad + BUILD_THREADS - 1) / BUILD_THREADS, BUILD_THREADS, 0, stream>>>(
            a.super_sph, a.n_supers, a.hyper_sph, a.n_hypers, a.n_hypers_pad);
    return cudaGetLastError();
}
