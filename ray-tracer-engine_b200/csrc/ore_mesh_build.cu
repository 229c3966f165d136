// ore_mesh_build.cu - the reference's flat BVH (ore_build_flat_bvh in host/ore_mesh.cpp) on the device (sm_100a,
// --fmad=false).
//
// The rule: one root box lists 0 .. n-1.  Each of ten layers visits the boxes in order; a box of more than 5 triangles is
// split on axis split_dir (0 -> y, 1 -> x, 2 -> z; one counter that advances after every split box, across all layers)
// at split_p = (hi + lo) / 2, a triangle going to the lo side when its first vertex's coordinate is <= split_p; the
// non-empty sides are appended lo then hi, each keeping the parent's list order; a box of <= 5 triangles passes through.
// Every new box gets getMinMaxP's bounds of its own list.
//
// Every box owns a contiguous range of the index array, and a split is a stable partition of that range, so the
// children's ranges start where the parent's did.  Per layer:
//   mesh_plan_kernel      one block: the bounds of the layer's boxes (from the reduction below, or the parent's when a
//                         box passed through), the split flags, a block scan for the axes, split_p
//   mesh_classify_kernel  one thread per listed triangle: its box by binary search over the layer's offsets, its lo flag
//   cub::DeviceScan       exclusive scan of the flags: a box's lo count and a triangle's rank on its side
//   mesh_children_kernel  one block: the children's offsets, compacted in order; their reduction slots reset
//   mesh_scatter_kernel   the stable partition into the other index buffer
//   mesh_bounds_kernel    getMinMaxP of every split child, as a reduction of (value, list position) pairs split across
//                         blocks (below); pass-through boxes keep their bounds
// mesh_final_kernel writes the leaves (offsets, boxes, balls) and the live leaf count.
//
// The bounds reduction: the sequential rule takes, per axis, the first of the coordinates that compare as the extreme
// (strict comparisons: of -0 and +0 the earlier stays), never a NaN, and keeps a NaN seed (ore_mesh_refit.h, take_hi /
// take_lo).  Here a coordinate becomes a 64-bit key: its value in the high half (ordered as an unsigned integer, -0 as
// +0) and its list position in the low half (inverted for the maximum), so that 64-bit atomicMax / atomicMin pick the
// rule's coordinate; NaN coordinates are skipped.  The winner's bits are then read at its position (so -0 and +0 keep
// their sign) and the seeds applied by seed_and_grow - the same last step as the refit's.
#include "ore_mesh_build.h"
#include "ore_mesh_refit.h"

#include <cub/block/block_scan.cuh>
#include <cub/device/device_scan.cuh>
#include <cstdint>

namespace {

constexpr int LAYERS = ORE_MESH_LAYERS;
constexpr int MAXB = ORE_MESH_MAX_LEAVES;
constexpr int LEAF_MAX = 5;          // a box of more triangles is split
constexpr int THREADS = 256;         // grid kernels
constexpr int ITEMS = 8;             // list positions per thread of the grid kernels
constexpr int TILE = THREADS * ITEMS;
constexpr int SLOTS = 64;            // boxes a block of mesh_bounds_kernel pre-reduces in shared memory
constexpr unsigned FULL = 0xffffffffu;
constexpr unsigned long long HI_NONE = 0ull, LO_NONE = ~0ull;

// device work space, carved from one allocation
struct Work {
    int* idx2;        // the second index buffer (cap)
    int* flags;       // lo flag per list position (cap + 1; the last is 0)
    int* scan;        // exclusive scan of flags (cap + 1)
    void* cub_tmp;
    size_t cub_bytes;
    int* offs;        // (LAYERS + 1) x (MAXB + 1): box offsets of every layer
    int* src;         // (LAYERS + 1) x MAXB: the box a pass-through box copies (index in the layer before), -1 if split
    float4* bnd;      // (LAYERS + 1) x MAXB x 2: bounds lo, hi
    int* split;       // MAXB: the current layer's split coordinate per box (0 x, 1 y, 2 z), -1 when the box passes through
    float* split_p;   // MAXB
    unsigned long long* acc;   // MAXB x 6: reduction keys, hi x y z then lo x y z
    int* nbox;        // LAYERS + 1 box counts
    int* state;       // [0] split_dir counter, [1] boxes split in the current layer, [2] the triangle count n
};

size_t align_up(size_t v) { return (v + 255) & ~(size_t)255; }

cudaError_t carve(int cap, void* base, Work* w, size_t* total) {
    size_t cub_bytes = 0;
    cudaError_t e = cub::DeviceScan::ExclusiveSum(nullptr, cub_bytes, (const int*)nullptr, (int*)nullptr, cap + 1);
    if (e != cudaSuccess) return e;
    size_t off = 0;
    char* b = static_cast<char*>(base);
    auto take = [&](size_t bytes) -> void* {
        void* p = b ? b + off : nullptr;
        off += align_up(bytes);
        return p;
    };
    w->idx2 = (int*)take((size_t)cap * sizeof(int));
    w->flags = (int*)take((size_t)(cap + 1) * sizeof(int));
    w->scan = (int*)take((size_t)(cap + 1) * sizeof(int));
    w->cub_bytes = cub_bytes;
    w->cub_tmp = take(cub_bytes);
    w->offs = (int*)take((size_t)(LAYERS + 1) * (MAXB + 1) * sizeof(int));
    w->src = (int*)take((size_t)(LAYERS + 1) * MAXB * sizeof(int));
    w->bnd = (float4*)take((size_t)(LAYERS + 1) * MAXB * 2 * sizeof(float4));
    w->split = (int*)take(MAXB * sizeof(int));
    w->split_p = (float*)take(MAXB * sizeof(float));
    w->acc = (unsigned long long*)take((size_t)MAXB * 6 * sizeof(unsigned long long));
    w->nbox = (int*)take((LAYERS + 1) * sizeof(int));
    w->state = (int*)take(3 * sizeof(int));
    *total = off;
    return cudaSuccess;
}

// the box of list position i: offs[b] <= i < offs[b + 1] (boxes are never empty, so the offsets ascend strictly)
__device__ __forceinline__ int find_box(const int* o, int nb, int i) {
    int lo = 0, hi = nb;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (o[mid] <= i)
            lo = mid;
        else
            hi = mid;
    }
    return lo;
}

// a float's value as an unsigned integer of the same order, -0 as +0
__device__ __forceinline__ uint32_t ordered(float w) {
    uint32_t u = __float_as_uint(w);
    if (u == 0x80000000u) u = 0;
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
// the maximum key is the largest value, then the earliest position; the minimum key the smallest value, then the earliest
__device__ __forceinline__ unsigned long long key_hi(float w, uint32_t pos) {
    return ((unsigned long long)ordered(w) << 32) | (0xffffffffu - pos);
}
__device__ __forceinline__ unsigned long long key_lo(float w, uint32_t pos) { return ((unsigned long long)ordered(w) << 32) | pos; }

__device__ __forceinline__ void reset_keys(unsigned long long* a) {
#pragma unroll
    for (int k = 0; k < 3; k++) {
        a[k] = HI_NONE;
        a[3 + k] = LO_NONE;
    }
}

// getMinMaxP's bounds of box c of a layer whose keys were reduced into acc[6c ..]; idx: the layer's index buffer
__device__ void box_from_keys(const float* __restrict__ tris, const int* __restrict__ idx, int o0, int o1,
                              const unsigned long long* a, float lo[3], float hi[3]) {
    const float nan = __int_as_float(0x7fffffff);
    float lo_ext[3], hi_ext[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        hi_ext[k] = lo_ext[k] = nan;
        if (a[k] != HI_NONE) {
            const uint32_t p = 0xffffffffu - (uint32_t)a[k];
            hi_ext[k] = tris[(size_t)idx[o0 + p / 3] * ore_host::TRI_FLOATS + 3 * (p % 3) + k];
        }
        if (a[3 + k] != LO_NONE) {
            const uint32_t p = (uint32_t)a[3 + k];
            lo_ext[k] = tris[(size_t)idx[o0 + p / 3] * ore_host::TRI_FLOATS + 3 * (p % 3) + k];
        }
    }
    ore_host::seed_and_grow(tris + (size_t)idx[o0] * ore_host::TRI_FLOATS, tris + (size_t)idx[o1 - 1] * ore_host::TRI_FLOATS,
                            lo_ext, hi_ext, lo, hi);
}

// the bounds of box c of layer `layer`: its parent's when it passed through, else from the reduction
__device__ void final_bounds(const float* __restrict__ tris, const int* __restrict__ idx, const Work w, int layer, int c, float lo[3],
                             float hi[3]) {
    const int* offs = w.offs + (size_t)layer * (MAXB + 1);
    const int s = w.src[(size_t)layer * MAXB + c];
    if (s >= 0) {
        const float4 a = w.bnd[((size_t)(layer - 1) * MAXB + s) * 2], b = w.bnd[((size_t)(layer - 1) * MAXB + s) * 2 + 1];
        lo[0] = a.x, lo[1] = a.y, lo[2] = a.z;
        hi[0] = b.x, hi[1] = b.y, hi[2] = b.z;
    } else {
        box_from_keys(tris, idx, offs[c], offs[c + 1], w.acc + 6 * (size_t)c, lo, hi);
    }
}

__global__ void mesh_count_kernel(const Work w, int n) { w.state[2] = n; }

__global__ void __launch_bounds__(THREADS) mesh_init_kernel(int* __restrict__ idx, const Work w) {
    const int n = w.state[2];
    const int i = blockIdx.x * THREADS + threadIdx.x;
    if (i < n) idx[i] = i;
    if (i == 0) {
        w.offs[0] = 0;
        w.offs[1] = n;
        w.src[0] = -1;
        w.nbox[0] = 1;
        w.state[0] = 0;
        reset_keys(w.acc);
    }
}

__global__ void __launch_bounds__(MAXB) mesh_plan_kernel(const float* __restrict__ tris, const int* __restrict__ idx, const Work w,
                                                         int layer) {
    using Scan = cub::BlockScan<int, MAXB>;
    __shared__ typename Scan::TempStorage tmp;
    const int b = threadIdx.x;
    const int nb = w.nbox[layer];
    const int* offs = w.offs + (size_t)layer * (MAXB + 1);
    const int counter = w.state[0];
    float lo[3] = {0.f, 0.f, 0.f}, hi[3] = {0.f, 0.f, 0.f};
    int m = 0;
    if (b < nb) {
        final_bounds(tris, idx, w, layer, b, lo, hi);
        w.bnd[((size_t)layer * MAXB + b) * 2] = make_float4(lo[0], lo[1], lo[2], 0.f);
        w.bnd[((size_t)layer * MAXB + b) * 2 + 1] = make_float4(hi[0], hi[1], hi[2], 0.f);
        m = offs[b + 1] - offs[b];
    }
    const int split = m > LEAF_MAX ? 1 : 0;
    int rank, total;
    Scan(tmp).ExclusiveSum(split, rank, total);
    if (b < nb) {
        if (split) {
            const int dir = (counter + rank) % 3;   // 0 -> y, 1 -> x, 2 -> z
            const int k = dir == 0 ? 1 : (dir == 1 ? 0 : 2);
            w.split[b] = k;
            w.split_p[b] = (hi[k] + lo[k]) / 2;
        } else {
            w.split[b] = -1;
        }
    }
    __syncthreads();   // (every thread has read the counter)
    if (b == 0) {
        w.state[0] = (counter + total) % 3;
        w.state[1] = total;
    }
}

// loads the layer's offsets into shared memory; returns the box count
__device__ __forceinline__ int load_offsets(int* s_offs, const Work& w, int layer) {
    const int nb = w.nbox[layer];
    const int* offs = w.offs + (size_t)layer * (MAXB + 1);
    for (int j = threadIdx.x; j <= nb; j += blockDim.x) s_offs[j] = offs[j];
    __syncthreads();
    return nb;
}

// the lo flag of every list position; positions n .. cap (scanned too: the scan is sized from the capacity) get 0
__global__ void __launch_bounds__(THREADS) mesh_classify_kernel(const float* __restrict__ tris, const int* __restrict__ idx, int cap,
                                                                const Work w, int layer) {
    __shared__ int s_offs[MAXB + 1];
    const int n = w.state[2];
    const bool any_split = w.state[1] != 0;
    const int nb = load_offsets(s_offs, w, layer);
#pragma unroll 1
    for (int it = 0; it < ITEMS; it++) {
        const int i = blockIdx.x * TILE + it * THREADS + threadIdx.x;
        if (i > cap) break;
        int f = 0;
        if (i < n && any_split) {
            const int c = find_box(s_offs, nb, i);
            const int k = w.split[c];
            f = (k >= 0 && tris[(size_t)idx[i] * ore_host::TRI_FLOATS + k] <= w.split_p[c]) ? 1 : 0;
        }
        w.flags[i] = f;
    }
}

__global__ void __launch_bounds__(MAXB) mesh_children_kernel(const Work w, int layer) {
    using Scan = cub::BlockScan<int, MAXB>;
    __shared__ typename Scan::TempStorage tmp;
    const int n = w.state[2];
    const int b = threadIdx.x;
    const int nb = w.nbox[layer];
    const int* offs = w.offs + (size_t)layer * (MAXB + 1);
    int* offs_n = w.offs + (size_t)(layer + 1) * (MAXB + 1);
    int* src_n = w.src + (size_t)(layer + 1) * MAXB;
    int o0 = 0, o1 = 0, n_lo = 0, cnt = 0;
    bool split = false;
    if (b < nb) {
        o0 = offs[b];
        o1 = offs[b + 1];
        split = w.split[b] >= 0;
        if (split) {
            n_lo = w.scan[o1] - w.scan[o0];
            cnt = (n_lo > 0) + (o1 - o0 - n_lo > 0);
        } else {
            cnt = 1;
        }
    }
    int base, total;
    Scan(tmp).ExclusiveSum(cnt, base, total);
    if (b < nb) {
        if (split) {
            int c = base;
            if (n_lo > 0) {
                offs_n[c] = o0;
                src_n[c++] = -1;
            }
            if (o1 - o0 - n_lo > 0) {
                offs_n[c] = o0 + n_lo;
                src_n[c] = -1;
            }
        } else {
            offs_n[base] = o0;
            src_n[base] = b;
        }
        for (int c = base; c < base + cnt; c++) reset_keys(w.acc + 6 * (size_t)c);
    }
    if (b == 0) {
        offs_n[total] = n;
        w.nbox[layer + 1] = total;
    }
}

__global__ void __launch_bounds__(THREADS) mesh_scatter_kernel(const int* __restrict__ idx, int* __restrict__ idx_next, const Work w,
                                                               int layer) {
    __shared__ int s_offs[MAXB + 1];
    const int n = w.state[2];
    if (blockIdx.x * TILE >= n) return;   // (the grid covers the capacity)
    const int nb = load_offsets(s_offs, w, layer);
#pragma unroll 1
    for (int it = 0; it < ITEMS; it++) {
        const int i = blockIdx.x * TILE + it * THREADS + threadIdx.x;
        if (i >= n) break;
        const int c = find_box(s_offs, nb, i);
        int dest = i;
        if (w.split[c] >= 0) {
            const int o0 = s_offs[c], s0 = w.scan[o0];
            const int r = w.scan[i] - s0;                          // lo entries before i in the box
            const int n_lo = w.scan[s_offs[c + 1]] - s0;
            dest = w.flags[i] ? o0 + r : o0 + n_lo + (i - o0 - r);
        }
        idx_next[dest] = idx[i];
    }
}

__device__ __forceinline__ void push_keys(unsigned long long* a, const unsigned long long k[6]) {
#pragma unroll
    for (int j = 0; j < 3; j++) {
        if (k[j] != HI_NONE) atomicMax(&a[j], k[j]);
        if (k[3 + j] != LO_NONE) atomicMin(&a[3 + j], k[3 + j]);
    }
}

// the keys of the split boxes of layer `layer` over its index buffer idx: per block, pre-reduced over a warp when the
// warp's positions share a box and in shared memory for the first SLOTS boxes the block meets, then into w.acc
__global__ void __launch_bounds__(THREADS) mesh_bounds_kernel(const float* __restrict__ tris, const int* __restrict__ idx, const Work w,
                                                              int layer) {
    __shared__ int s_offs[MAXB + 1];
    __shared__ unsigned long long s_acc[SLOTS * 6];
    const int n = w.state[2];
    if (blockIdx.x * TILE >= n) return;          // (the grid covers the capacity)
    if (layer > 0 && w.state[1] == 0) return;   // nothing split: every box passed through
    for (int j = threadIdx.x; j < SLOTS; j += THREADS) reset_keys(s_acc + 6 * j);
    const int nb = load_offsets(s_offs, w, layer);
    const int* src = w.src + (size_t)layer * MAXB;
    const int lane = threadIdx.x & 31;
    const int c0 = find_box(s_offs, nb, min(blockIdx.x * TILE, n - 1));
#pragma unroll 1
    for (int it = 0; it < ITEMS; it++) {
        const int i = blockIdx.x * TILE + it * THREADS + threadIdx.x;
        int c = -1;
        unsigned long long k[6];
        reset_keys(k);
        if (i < n) {
            c = find_box(s_offs, nb, i);
            if (src[c] >= 0) {
                c = -1;
            } else {
                const float* t = tris + (size_t)idx[i] * ore_host::TRI_FLOATS;
                const uint32_t p0 = 3u * (uint32_t)(i - s_offs[c]);   // position of vertex v of list entry e: 3 e + v
#pragma unroll
                for (int v = 0; v < 3; v++)
#pragma unroll
                    for (int j = 0; j < 3; j++) {
                        const float x = __ldg(t + 3 * v + j);
                        if (isnan(x)) continue;
                        k[j] = max(k[j], key_hi(x, p0 + v));
                        k[3 + j] = min(k[3 + j], key_lo(x, p0 + v));
                    }
            }
        }
        const int c_first = __shfl_sync(FULL, c, 0);
        if (__all_sync(FULL, c == c_first)) {
            if (c_first < 0) continue;
#pragma unroll
            for (int o = 16; o; o >>= 1)
#pragma unroll
                for (int j = 0; j < 3; j++) {
                    k[j] = max(k[j], __shfl_xor_sync(FULL, k[j], o));
                    k[3 + j] = min(k[3 + j], __shfl_xor_sync(FULL, k[3 + j], o));
                }
            if (lane != 0) continue;
        }
        if (c < 0) continue;
        push_keys(c - c0 < SLOTS ? s_acc + 6 * (c - c0) : w.acc + 6 * (size_t)c, k);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < SLOTS * 6; j += THREADS) {
        const int c = c0 + j / 6;
        const unsigned long long v = s_acc[j];
        if (c >= nb || v == ((j % 6) < 3 ? HI_NONE : LO_NONE)) continue;
        if ((j % 6) < 3)
            atomicMax(&w.acc[6 * (size_t)c + j % 6], v);
        else
            atomicMin(&w.acc[6 * (size_t)c + j % 6], v);
    }
}

__global__ void __launch_bounds__(MAXB) mesh_final_kernel(const float* __restrict__ tris, const int* __restrict__ idx, const Work w,
                                                          int* __restrict__ box_offsets, float4* __restrict__ boxes,
                                                          float4* __restrict__ box_sph, int* __restrict__ n_live) {
    const int n = w.state[2];
    const int L = min(n, MAXB);   // ore_mesh_leaf_capacity(n): the leaves the context holds for this mesh
    const int j = threadIdx.x;
    const int nb = w.nbox[LAYERS];
    if (j < L) {
        if (j < nb) {
            float lo[3], hi[3];
            final_bounds(tris, idx, w, LAYERS, j, lo, hi);
            boxes[2 * j] = make_float4(lo[0], lo[1], lo[2], 0.f);
            boxes[2 * j + 1] = make_float4(hi[0], hi[1], hi[2], 0.f);
            const ore_host::Rec4 s = ore_host::mesh_box_ball(lo, hi);
            box_sph[j] = make_float4(s.x, s.y, s.z, s.w);
            box_offsets[j] = w.offs[(size_t)LAYERS * (MAXB + 1) + j];
        } else {   // past the live count: no triangles, defined bytes that no render kernel reads
            boxes[2 * j] = boxes[2 * j + 1] = box_sph[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            box_offsets[j] = n;
        }
    }
    if (j == 0) {
        box_offsets[L] = n;
        *n_live = nb;
    }
}

}  // namespace

cudaError_t ore_mesh_build_bytes(int cap_tris, size_t* bytes) {
    Work w;
    return carve(cap_tris > 1 ? cap_tris : 1, nullptr, &w, bytes);
}

static cudaError_t carve_args(const MeshBuildArgs& a, Work* w) {
    if (a.cap_tris < 1) return cudaErrorInvalidValue;
    size_t need = 0;
    const cudaError_t e = carve(a.cap_tris, a.work, w, &need);
    if (e != cudaSuccess) return e;
    return need > a.work_bytes ? cudaErrorInvalidValue : cudaSuccess;
}

cudaError_t ore_mesh_build_count(const MeshBuildArgs& a, int n, cudaStream_t stream) {
    Work w;
    cudaError_t e = carve_args(a, &w);
    if (e != cudaSuccess) return e;
    if (n < 1 || n > a.cap_tris) return cudaErrorInvalidValue;
    mesh_count_kernel<<<1, 1, 0, stream>>>(w, n);
    return cudaGetLastError();
}

cudaError_t ore_mesh_build(const MeshBuildArgs& a, cudaStream_t stream) {
    Work w;
    cudaError_t e = carve_args(a, &w);
    if (e != cudaSuccess) return e;
    // every grid and the scan's length from the capacity; the kernels read n (mesh_count_kernel) and stop there
    const int cap = a.cap_tris;
    const int grid_n = (cap + THREADS - 1) / THREADS, grid_t = (cap + TILE - 1) / TILE, grid_f = (cap + 1 + TILE - 1) / TILE;
    int* buf[2] = {a.box_indices, w.idx2};   // layer l's list is in buf[l & 1]; ten layers end where they began
    mesh_init_kernel<<<grid_n, THREADS, 0, stream>>>(buf[0], w);
    mesh_bounds_kernel<<<grid_t, THREADS, 0, stream>>>(a.tris, buf[0], w, 0);
    for (int l = 0; l < LAYERS; l++) {
        const int* cur = buf[l & 1];
        int* next = buf[(l + 1) & 1];
        mesh_plan_kernel<<<1, MAXB, 0, stream>>>(a.tris, cur, w, l);
        mesh_classify_kernel<<<grid_f, THREADS, 0, stream>>>(a.tris, cur, cap, w, l);
        size_t cb = w.cub_bytes;
        if ((e = cub::DeviceScan::ExclusiveSum(w.cub_tmp, cb, w.flags, w.scan, cap + 1, stream)) != cudaSuccess) return e;
        mesh_children_kernel<<<1, MAXB, 0, stream>>>(w, l);
        mesh_scatter_kernel<<<grid_t, THREADS, 0, stream>>>(cur, next, w, l);
        mesh_bounds_kernel<<<grid_t, THREADS, 0, stream>>>(a.tris, next, w, l + 1);
    }
    static_assert(LAYERS % 2 == 0, "the leaves' list must end in box_indices");
    mesh_final_kernel<<<1, MAXB, 0, stream>>>(a.tris, buf[0], w, a.box_offsets, a.boxes, a.box_sph, a.n_live);
    return cudaGetLastError();
}
