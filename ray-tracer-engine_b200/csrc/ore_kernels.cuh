// ore_kernels.cuh - kernels of the render hot path (sm_100a, --fmad=false).
//
//   prep_frame_kernel   (ore_primary.cuh) per-frame tables + camera-space filter records of spheres, leaves, super-clusters
//   primary_tile_kernel (ore_primary.cuh) nearest hit per 32 x 8 pixel tile, sky for the misses, compact hit records
//                                         (kernel.cu:1614-1640, 1288-1431, 1146-1166)
//   shade_setup_kernel  (here)            stage A of the shadow pass: shading set-up + the 10 shadow-ray directions and
//                                         their cone for every light of every hit pixel (kernel.cu:1396-1405,
//                                         1643-1655, 1438-1468) -> staging buffer
//   shadow_sweep_kernel (ore_sweep.cuh)   stage B: any-hit sweep per light, light accumulation, packed pixel
//                                         (kernel.cu:1470-1544, 1673-1684)
#pragma once
#include "ore_clusters.h"   // ORE_KAPPA_SHADOW (the margin R' is rounded up for)
#include "ore_device.cuh"

namespace ore {

constexpr int MAX_LIGHTS = 16;
constexpr int MAX_BATCH = 8;   // frames (cameras) rendered by one launch set
constexpr int CTA_THREADS = 256;
#ifndef ORE_STAGE_A_THREADS
#define ORE_STAGE_A_THREADS 64   // warp-independent persistent kernel: small CTAs hand an SM back almost warp by warp
#endif
constexpr int STAGE_A_THREADS = ORE_STAGE_A_THREADS;
// primary kernel: rows per 32-wide pixel tile
#ifndef ORE_TILE_P
#define ORE_TILE_P 8
#endif
constexpr int TILE_P = ORE_TILE_P;

// conservative filter margins (see DESIGN.md "Filter soundness")
#define ORE_KAPPA_PRIMARY 7.62939453125e-06  /* 2^-17 */
#define ORE_BIG 3.0e38f

enum CounterSlot {
    CNT_HITS = 0,          // hit-list length
    CNT_SHADOW_CURSOR = 1, // block cursor of the fused / catch-all sweep
    CNT_EXACT_PRIMARY = 2,
    CNT_EXACT_SHADOW = 3,
    CNT_SHADOW_TESTS_REF = 4,
    CNT_COUNT_CURSOR = 5,
    CNT_BEAM_L1 = 6,   // spheres passing the warp-level beam test (summed over warps, lights and groups)
    CNT_BEAM_L2 = 7,   // (pixel, sphere, light) triples passing the per-pixel cone test
    CNT_PRIMARY_CURSOR = 8,  // tile-batch cursor of the primary kernel
    CNT_PRIMARY_STEPS = 9,   // warp steps of the primary sweep (32 cone tests each)
    CNT_SWEEP_STEPS = 10,    // warp steps of the shadow sweep (32 beam tests each)
    CNT_SKY_EXACT = 11,      // miss pixels whose sky texel needed the exact sequence (the rest: sky_fast)
    CNT_STAGE_A0 = 12,                         // per-chunk block cursors of shade_setup_kernel
    CNT_STAGE_B0 = CNT_STAGE_A0 + 32,          // per-chunk block cursors of the staged shadow_sweep_kernel
    CNT_SLOTS = CNT_STAGE_B0 + 32
};
constexpr int MAX_STAGE_CHUNKS = 32;

// Staging buffer between shade_setup_kernel and the staged shadow_sweep_kernel: blocks of 32 hit-list items,
// value-major inside a block (value v of lane i at (block * nv + v) * 32 + i, so every access is one coalesced
// 128-byte line and a light's 30 direction components are one contiguous 3840-byte piece for a TMA bulk copy).
// Values: 0-2 start, 3-5 texel r,g,b, then 35 per light: cone axis (3), cone min-dot (-1: degenerate bundle),
// a = dot(normal, toL), 30 direction components.
constexpr int STAGE_HEADER = 6;
constexpr int STAGE_PER_LIGHT = 35;
constexpr int STAGE_DIRS_AT = 5;
struct StageArgs {
    float* buf;
    uint32_t first_block;  // hit-list block (32 items) held by stage block 0 of this chunk
    uint32_t cap_blocks;   // stage capacity in blocks
    int chunk;             // cursor slot
    int nv;                // values per item = STAGE_HEADER + STAGE_PER_LIGHT * n_lights
};

struct LightP {
    float px, py, pz, size, r, g, b;
};

// camera of one frame of the batch
struct CamP {
    float Ox, Oy, Oz;      // add(eyePos, cam.Org), kernel.cu:1631
    float cp, sp, cy, sy;  // cosf/sinf of pitchRad / yawRad (kernel.cu:249-255), host libm
};

// One launch set renders n_frames frames (1..MAX_BATCH cameras over the same scene, size and row band): every kernel
// sees n_frames times the work units, so launch latencies and the tail of each launch are paid once per batch - what
// matters when a rank of a multi-GPU job only holds an eighth of a frame.  Rendered-pixel indices in the hit list
// are frame * n_px_frame + k * W + x.
struct FrameParams {
    int W, H, y0, y_step, n_rows;
    int n_frames;
    uint32_t n_px_frame;   // n_rows * W
    int W_pad;       // W rounded up to a multiple of 32 (dx_tab entries)
    int y_block;     // rows come in blocks of y_block consecutive image rows, block starts y_step apart
    int pitch;       // output row pitch in pixels
    int out_global;  // 1: pixel rows are stored at their image position relative to y0, 0: packed
    int n_spheres, n_lights;
    uint32_t flags;
    float aspect, ez, fz;  // ez = -1/aspect (kernel.cu:1629), fz = 0 - ez
    CamP cam[MAX_BATCH];
    const float* dx_tab;
    const float* dy_tab;
    float tile_ca, tile_sa;   // cos/sin of the largest pixel-tile half-angle (+ margins), host-computed
    float px_delta;           // image-plane pixel pitch 2*aspect/width
    // scene records in the Morton order of the upload (ore_clusters.h): sorted position p holds original sphere
    // sort_index[p]; leaf j = spheres [8j, 8j+8), super-cluster k = leaves [32k, 32k+32)
    const float4* sph_exact;  // cx,cy,cz,radius member, ORIGINAL order (hit attributes by hit id)
    const float4* sph_xsort;  // the same records, sorted
    const float4* sph_sort;   // cx,cy,cz,R' (effective radius rounded up: R'^2 >= (1+k) radius^2), sorted (shadow filters)
    const int* sort_index;
    const float4* leaf_sph;   // bounding balls (centre, radius; radius +inf: always a candidate)
    const float4* super_sph;
    int n_sort, n_leaves, n_leaves_pad, n_supers, n_supers_pad;
    // camera-space records, one set per frame of the batch (frame f at base + f * {n_sort, n_leaves_pad, n_supers_pad})
    float4* prim_sorted;      // per-pixel primary filter coefficients a',b',c' (sorted order)
    float4* cone_sorted;      // tile-cone record Mx,My,Mz,W of every sphere (sorted order)
    float4* leaf_cone;        // tile-cone record of every leaf / super-cluster ball
    float4* super_cone;
    int cone_resident;        // the sphere-level cone records fit in the primary kernel's shared memory
    const float *tex_r, *tex_g, *tex_b;
    int tex_w, tex_h;
    const float *sky_r, *sky_g, *sky_b;
    int sky_w, sky_h;
    float sky_radius;  // skybox sphere member = size*size (kernel.cu:287,1122)
    // compact hit records, in hit-list order (nothing is stored for miss pixels)
    uint32_t* hit_list;   // rendered-pixel index frame * n_px_frame + k * W + x
    int32_t* hit_ids;     // nearest primitive
    float* hit_ts;        // nearest t
    unsigned long long* counters;
    uint32_t* pixels[MAX_BATCH];   // one framebuffer per frame of the batch (hit pixels: shadow pass)
    // Where the primary kernel stores its rows (sky pixels, 0 for hit pixels).  Normally the same place.  When the
    // framebuffers are ANOTHER GPU's memory (a rank of a multi-GPU job storing into the presenter's frame) the rows go
    // to a packed band buffer in local memory instead and a copy engine moves them over NVLink while the shadow pass
    // runs (ore_capi.cu: "band DMA"); only the hit pixels are then stored remotely by the sweep.
    uint32_t* sky_pixels[MAX_BATCH];
    int sky_pitch, sky_global;
    // "next" primitives (kernel.cu:360-509): cube i = 3 float4 {bounds[0], bounds[1], orgin}, plane i = 2 float4
    // {orgin, normal}; hit ids continue after the spheres: cube i -> n_spheres + i, plane i -> n_spheres + n_cubes + i
    const float4* cubes;
    const float4* planes;
    int n_cubes, n_planes;
    // triangle mesh + flat BVH as the reference's `mesh` holds it (kernel.cu:559-1017): triangle i = 27 floats;
    // leaf box j = 2 float4 {bounds[0], bounds[1]} with triangles box_indices[box_offsets[j] .. box_offsets[j+1]);
    // hit id of triangle i = n_spheres + n_cubes + n_planes + i
    const float* tris;
    const float4* boxes;
    const float4* box_sph;    // bounding sphere of each leaf box (centre, radius incl. margin) for the cone filters
    float4* box_cone;         // tile-cone record of each leaf box (camera frame; frame f at base + f * n_boxes)
    const int* box_offsets;
    const int* box_indices;
    int n_tris, n_boxes, mesh_has_normals;
    // 1: a light whose castLightRay factor a = normal.toL is not > 0 contributes exactly +0 to the pixel whatever its
    // shadow rays do (kernel.cu:1541-1542, 1673-1675: b *= a > 0 ? a : 0 with b finite, then b * colour * texel with
    // finite colours and texels), so its directions and its sweep are skipped.  0 (exhaustive mode, or a non-finite
    // light colour / texel somewhere): every light is evaluated in full.
    int skip_dark;
    // tools only (env ORE_DEBUG_BLOCK_CYCLES at ore_create): SM clocks spent on every hit-list block, [2][dbg_cap]
    // (0: shade_setup_kernel, 1: staged shadow_sweep_kernel); null on every product path
    uint32_t* dbg_cycles;
    uint32_t dbg_cap;
    LightP lights[MAX_LIGHTS];
};

// cosf/ORE_SINF((float)j/10*2.f*3.1415f), kernel.cu:1454,1462-1463 - ten frame-independent
// values, evaluated once on the host (same libm as the oracle) at context creation
__constant__ float c_cos_phi[10];
__constant__ float c_sin_phi[10];
// b after k unshadowed samples: `b += 0.1` is float += double (kernel.cu:1537-1539), so b depends only on
// how many of the 10 samples were unshadowed; the 11 values are produced on the host with that arithmetic
__constant__ float c_b_of_k[11];

// ------------------------------------------------------------------------------------
// primary ray of pixel (x, row k): kernel.cu:1624-1631 with dx/dy from the tables
// ------------------------------------------------------------------------------------
__device__ __forceinline__ v3 primary_dir(const CamP& c, float ez, float dx, float dy) {
    v3 v = mk(dx - 0.f, dy - 0.f, 0.f - ez);  // sub(dir, eyePos)
    v3 n = ref_normalise(v);
    // camera::rotateDir, kernel.cu:252-255
    float y = n.y * c.cp - n.z * c.sp;
    float z = n.y * c.sp + n.z * c.cp;
    float x = n.x * c.cy + z * c.sy;
    z = -n.x * c.sy + z * c.cy;
    return mk(x, y, z);
}
// frame and in-frame pixel of a hit-list entry
__device__ __forceinline__ void split_pixel(const FrameParams& prm, uint32_t o, int& frame, int& k, int& x) {
    frame = (int)(o / prm.n_px_frame);
    const uint32_t r = o - (uint32_t)frame * prm.n_px_frame;
    k = (int)(r / (uint32_t)prm.W);
    x = (int)(r - (uint32_t)k * (uint32_t)prm.W);
}

__device__ __forceinline__ int clamp_index(int idx, int n) { return idx < 0 ? 0 : (idx >= n ? n - 1 : idx); }

// image row (relative to y0) of rendered row k, and where its pixels go
__device__ __forceinline__ int image_row_rel(const FrameParams& prm, int k) {
    return (k / prm.y_block) * prm.y_step + (k % prm.y_block);
}
__device__ __forceinline__ size_t out_index(const FrameParams& prm, int k, int x) {
    return (size_t)(prm.out_global ? image_row_rel(prm, k) : k) * prm.pitch + x;
}
__device__ __forceinline__ size_t sky_out_index(const FrameParams& prm, int k, int x) {
    return (size_t)(prm.sky_global ? image_row_rel(prm, k) : k) * prm.sky_pitch + x;
}

// direction r of a bundle stored with `stride` floats between components (1: contiguous [10][3]; 32: a column of a
// shared-memory slot laid out [30][32])
__device__ __forceinline__ v3 dir_at(const float* __restrict__ d, int stride, int r) {
    return mk(d[(3 * r) * stride], d[(3 * r + 1) * stride], d[(3 * r + 2) * stride]);
}

// ---- out-of-line helpers: ONE copy of each cold or bulky sequence keeps the kernels' code small enough
// ---- for the instruction caches
struct DirArgs {
    float ez, cp, sp, cy, sy;
};
__device__ __noinline__ v3 primary_dir_call(const DirArgs a, float dx, float dy) {
    v3 v = mk(dx - 0.f, dy - 0.f, 0.f - a.ez);
    v3 n = ref_normalise(v);
    float y = n.y * a.cp - n.z * a.sp;
    float z = n.y * a.sp + n.z * a.cp;
    float x = n.x * a.cy + z * a.sy;
    z = -n.x * a.sy + z * a.cy;
    return mk(x, y, z);
}

// ---- cubes and planes (SURVEY.md 8f N1): small counts, exact tests, one out-of-line copy ----------------
// castRay's cube loop then plane loop (kernel.cu:1344-1372), continuing the strict '<' search after the spheres
__device__ __noinline__ void nearest_cube_plane(const float4* __restrict__ cubes, int nc, const float4* __restrict__ planes,
                                                int np, int id_base, float Ox, float Oy, float Oz, float Dx, float Dy,
                                                float Dz, float* best_t, int* best_id) {
    const v3 O = mk(Ox, Oy, Oz), D = mk(Dx, Dy, Dz);
    float nt = *best_t;
    int id = *best_id;
    for (int i = 0; i < nc; i++) {
        const float4 b0 = __ldg(&cubes[3 * i]), b1 = __ldg(&cubes[3 * i + 1]);
        float t;
        if (ref_cube_intersect(O, D, mk(b0.x, b0.y, b0.z), mk(b1.x, b1.y, b1.z), t)) {
            if (t < nt) {
                nt = t;
                id = id_base + i;
            }
        }
    }
    for (int i = 0; i < np; i++) {
        const float4 po = __ldg(&planes[2 * i]), no = __ldg(&planes[2 * i + 1]);
        float t;
        if (ref_plane_intersect(O, D, mk(po.x, po.y, po.z), mk(no.x, no.y, no.z), t)) {
            if (t < nt) {
                nt = t;
                id = id_base + nc + i;
            }
        }
    }
    *best_t = nt;
    *best_id = id;
}
// The light-cone culls below skip a box whose bounding sphere the cone cannot touch.  That is sound only for hits that
// lie in the box, and cube::intersect has one kind that does not (DESIGN.md 6b): a ray with D.k == +-0 that starts on a
// face plane of the box on axis k gets (b.k - O.k) * (1 / D.k) = 0 * inf = NaN for that slab, and the reference's max/min
// macros then drop that slab and every slab before it, so the test can report a hit far from the box.  zero_axes gives
// the axes (bits 0..2) on which some ray of `live` has a component whose reciprocal overflows (+-0, tiny, or NaN);
// the caller computes it once per light and passes it to both culls as `zaxes`.  on_face_plane says whether O lies on
// a face plane of box (b0, b1) on one of them.  Such a box is never culled.
__device__ __forceinline__ uint32_t zero_axes(const float* __restrict__ dirs, int dstride, uint32_t live) {
    uint32_t z = 0;
    while (live) {
        const int r = __ffs(live) - 1;
        live &= live - 1;
        const v3 D = dir_at(dirs, dstride, r);
        z |= (uint32_t)!(fabsf(D.x) >= 0x1p-126f) | (uint32_t)!(fabsf(D.y) >= 0x1p-126f) << 1 |
             (uint32_t)!(fabsf(D.z) >= 0x1p-126f) << 2;
    }
    return z;
}
__device__ __forceinline__ bool on_face_plane(uint32_t zaxes, float Ox, float Oy, float Oz, float4 b0, float4 b1) {
    return ((zaxes & 1u) && (Ox == b0.x || Ox == b1.x)) || ((zaxes & 2u) && (Oy == b0.y || Oy == b1.y)) ||
           ((zaxes & 4u) && (Oz == b0.z || Oz == b1.z));
}
// true when the light's cone (A, ca, sa) cannot touch the ball q (.xyz centre, .w radius incl. margin) seen from O.
// A NaN anywhere (a non-finite ball, or |O - q|^2 overflowing to inf) answers false: the box stays.
__device__ __forceinline__ bool cone_misses_ball(float4 q, float Ox, float Oy, float Oz, float Ax, float Ay, float Az, float ca,
                                                 float sa) {
    const float lx = Ox - q.x, ly = Oy - q.y, lz = Oz - q.z;
    const float LL = fmaf(lz, lz, fmaf(ly, ly, lx * lx));
    const float Cm = fmaf(LL, 1.0f - ORE_KAPPA_SHADOW, -(q.w * q.w));
    if (!(Cm > 1e-20f)) return false;   // O in or near the ball, or NaN
    const float sv = Cm * rsqrt_approx(Cm);
    const float T = fmaf(ca, sv, -(sa * q.w));
    return fmaf(Ax, lx, fmaf(Ay, ly, fmaf(Az, lz, T))) >= 0.f;
}
// castLightRay's plane loop then cube loop (kernel.cu:1512-1536) for the live rays `live` (bits 0..9) of ONE light (ray r =
// dir_at(dirs, dstride, r)):
// any hit blocks.  A cube whose bounding sphere (cubes[3*i+2].xyz = orgin, .w = radius incl. margin) the light's cone
// cannot touch is skipped, unless O lies on one of its face planes (above).  Returns the rays found blocked.
__device__ __noinline__ uint32_t cubes_planes_block_light(const float4* __restrict__ cubes, int nc,
                                                          const float4* __restrict__ planes, int np, float Ox, float Oy,
                                                          float Oz, float Ax, float Ay, float Az, float ca, float sa,
                                                          bool use_cone, uint32_t zaxes, const float* __restrict__ dirs, int dstride,
                                                          uint32_t live) {
    const v3 O = mk(Ox, Oy, Oz);
    uint32_t hit = 0;
    float t;
    for (int i = 0; i < np && live; i++) {
        const float4 po = __ldg(&planes[2 * i]), no = __ldg(&planes[2 * i + 1]);
        uint32_t todo = live;
        while (todo) {
            const int r = __ffs(todo) - 1;
            todo &= todo - 1;
            if (ref_plane_intersect(O, dir_at(dirs, dstride, r), mk(po.x, po.y, po.z),
                                    mk(no.x, no.y, no.z), t)) {
                hit |= 1u << r;
                live &= ~(1u << r);
            }
        }
    }
    for (int i = 0; i < nc && live; i++) {
        if (use_cone && cone_misses_ball(__ldg(&cubes[3 * i + 2]), Ox, Oy, Oz, Ax, Ay, Az, ca, sa) &&
            (!zaxes || !on_face_plane(zaxes, Ox, Oy, Oz, __ldg(&cubes[3 * i]), __ldg(&cubes[3 * i + 1]))))
            continue;
        const float4 b0 = __ldg(&cubes[3 * i]), b1 = __ldg(&cubes[3 * i + 1]);
        uint32_t todo = live;
        while (todo) {
            const int r = __ffs(todo) - 1;
            todo &= todo - 1;
            if (ref_cube_intersect(O, dir_at(dirs, dstride, r), mk(b0.x, b0.y, b0.z),
                                   mk(b1.x, b1.y, b1.z), t)) {
                hit |= 1u << r;
                live &= ~(1u << r);
            }
        }
    }
    return hit;
}

// ---- triangle mesh (SURVEY.md 8f N2): linear scan over the leaf boxes, exact tests, one out-of-line copy ----
struct MeshArgs {
    const float* tris;
    const float4* boxes;
    const int* offsets;
    const int* indices;
    int n_boxes;
};
// castRay's triangle loop (kernel.cu:1293-1328) for ONE leaf box: exact slab test, then exact triangle tests in leaf
// order, continuing the strict '<' search.  The caller visits the leaves in ascending order (all of them in the
// reference; here those whose bounding sphere the tile cone can touch - a leaf the ray misses contributes nothing).
__device__ __noinline__ void nearest_in_leaf(const MeshArgs m, int j, int id_base, float Ox, float Oy, float Oz, float Dx,
                                             float Dy, float Dz, float* best_t, int* best_id) {
    const v3 O = mk(Ox, Oy, Oz), D = mk(Dx, Dy, Dz);
    const float4 b0 = __ldg(&m.boxes[2 * j]), b1 = __ldg(&m.boxes[2 * j + 1]);
    float temp;
    if (!ref_cube_intersect(O, D, mk(b0.x, b0.y, b0.z), mk(b1.x, b1.y, b1.z), temp)) return;
    float nt = *best_t;
    int id = *best_id;
    const int k1 = __ldg(&m.offsets[j + 1]);
    for (int k = __ldg(&m.offsets[j]); k < k1; k++) {
        const int ti = __ldg(&m.indices[k]);
        float t, u, v;
        if (ref_tri_intersect(O, D, m.tris + 27 * (size_t)ti, t, u, v)) {
            if (t < nt) {
                nt = t;
                id = id_base + ti;
            }
        }
    }
    *best_t = nt;
    *best_id = id;
}
// castLightRay's triangle part (kernel.cu:1475-1497) for the live rays `live` (bits 0..9) of ONE light: a leaf is
// skipped when the light's cone (A, ca, sa; use_cone) cannot touch its bounding sphere and O lies on none of its face
// planes (above: the caller's boxes need not contain their triangles); otherwise every live ray runs the exact slab
// test and the exact triangle tests.  Returns the rays found blocked.
__device__ __noinline__ uint32_t mesh_blocks_light(const MeshArgs m, const float4* __restrict__ box_sph, float Ox, float Oy,
                                                   float Oz, float Ax, float Ay, float Az, float ca, float sa, bool use_cone,
                                                   uint32_t zaxes, const float* __restrict__ dirs, int dstride, uint32_t live) {
    const v3 O = mk(Ox, Oy, Oz);
    uint32_t hit = 0;
    for (int j = 0; j < m.n_boxes && live; j++) {
        if (use_cone && cone_misses_ball(__ldg(&box_sph[j]), Ox, Oy, Oz, Ax, Ay, Az, ca, sa) &&
            (!zaxes || !on_face_plane(zaxes, Ox, Oy, Oz, __ldg(&m.boxes[2 * j]), __ldg(&m.boxes[2 * j + 1]))))
            continue;
        const float4 b0 = __ldg(&m.boxes[2 * j]), b1 = __ldg(&m.boxes[2 * j + 1]);
        const int k0 = __ldg(&m.offsets[j]), k1 = __ldg(&m.offsets[j + 1]);
        uint32_t todo = live;
        while (todo) {
            const int r = __ffs(todo) - 1;
            todo &= todo - 1;
            const v3 D = dir_at(dirs, dstride, r);
            float temp;
            if (!ref_cube_intersect(O, D, mk(b0.x, b0.y, b0.z), mk(b1.x, b1.y, b1.z), temp)) continue;
            for (int k = k0; k < k1; k++) {
                float t, u, v;
                if (ref_tri_intersect(O, D, m.tris + 27 * (size_t)__ldg(&m.indices[k]), t, u, v)) {
                    hit |= 1u << r;
                    live &= ~(1u << r);
                    break;
                }
            }
        }
    }
    return hit;
}
// triangle hit attributes (kernel.cu:1380-1394): u,v come from re-running the winning test (deterministic)
__device__ __noinline__ void triangle_attributes(const float* __restrict__ tri, int has_normals, float Ox, float Oy, float Oz,
                                                 float Dx, float Dy, float Dz, float nt, v3* normal, v3* new_org, float* tx,
                                                 float* ty) {
    const v3 O = mk(Ox, Oy, Oz), D = mk(Dx, Dy, Dz);
    float t, nu = 0.f, nv = 0.f;
    ref_tri_intersect(O, D, tri, t, nu, nv);
    v3 n;
    if (has_normals) {
        const v3 vn0 = mk(tri[12], tri[13], tri[14]), vn1 = mk(tri[15], tri[16], tri[17]), vn2 = mk(tri[18], tri[19], tri[20]);
        n = ref_add(ref_add(ref_scale(vn0, (1 - nu - nv)), ref_scale(vn1, nu)), ref_scale(vn2, nv));
        ref_normalise(n);
    } else {
        n = mk(tri[9], tri[10], tri[11]);
    }
    *tx = ((1 - nu - nv) * tri[21]) + (nu * tri[23]) + (nv * tri[25]);
    *ty = ((1 - nu - nv) * tri[22]) + (nu * tri[24]) + (nv * tri[26]);
    *normal = n;
    *new_org = ref_add(n, ref_add(O, ref_scale(D, nt)));  // the unit normal is ADDED to the hit point (kernel.cu:1393)
}

// ------------------------------------------------------------------------------------
// light_facing: a = dot(normal, toL) exactly as castLightRay ends up computing it (kernel.cu:1541).  toL is
// normalise(l.pos - start) (:1438), re-normalised IN PLACE twice per sample (:1465-1466), i.e. 20 times per light;
// once two normalisations reproduce their input bit for bit the remaining ones do too, so the chain stops there.
// Costs a few normalisations - against ~2500 warp instructions for the ten directions of a light whose contribution
// is then multiplied by zero.
// ------------------------------------------------------------------------------------
__device__ __noinline__ float light_facing(float lpx, float lpy, float lpz, const v3 start, const v3 normal) {
    v3 tmp = ref_sub(mk(lpx, lpy, lpz), start);
    v3 toL = ref_normalise(tmp);
#pragma unroll 1
    for (int j = 0; j < 10; j++) {
        const v3 prev = toL;
        ref_normalise(toL);
        ref_normalise(toL);
        if (same_bits(toL, prev)) break;
    }
    return ref_dot(normal, toL);
}

// ------------------------------------------------------------------------------------
// light_directions_reuse: one light, one copy of the code (instruction-cache friendly), same exact reuse
// of angle / rotate() matrix while toL repeats bit for bit.  Returns a = dot(normal, toL_final).
// ------------------------------------------------------------------------------------
__device__ __noinline__ float light_directions_reuse(const LightP L, const v3 start, const v3 normal,
                                                     float* __restrict__ dir /* [10][3] */) {
    const v3 up = mk(0.f, 1.f, 0.f), fwd = mk(0.f, 0.f, 1.f);
    const v3 lpos = mk(L.px, L.py, L.pz);
    v3 tmp = ref_sub(lpos, start);
    v3 toL = ref_normalise(tmp);
    v3 prev = mk(__int_as_float(0x7fc00001), 0.f, 0.f);
    float angle = 0.f;
    RotM M = RotM{0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
    for (int j = 0; j < 10; j++) {
        if (!same_bits(toL, prev)) {
            prev = toL;
            v3 P = ref_cross(toL, up);
            v3 e = ref_sub(ref_add(lpos, ref_scale(P, L.size)), start);
            v3 toEdge = ref_normalise(e);
            angle = ORE_COSF((ref_dot(toL, toEdge)) * 2);
            v3 n1 = ref_normalise(toL);
            v3 ax = ref_cross(fwd, n1);
            v3 axis = ref_normalise(ax);
            v3 n2 = ref_normalise(toL);
            float nAngle = ORE_ACOSF(ref_dot(n2, fwd));
            M = ref_rotate_matrix(nAngle, axis);
        }
        const float _z = (float)j / 10 * (1.0f - angle) + angle;
        const float sq = sqrtf(1.f - _z * _z);
        const float x = sq * c_cos_phi[j];
        const float y = sq * c_sin_phi[j];
        v3 nd = ref_sub(lpos, ref_matrix_apply(M, mk(x, y, _z)));
        v3 nn = ref_normalise(nd);
        dir[j * 3 + 0] = nn.x;
        dir[j * 3 + 1] = nn.y;
        dir[j * 3 + 2] = nn.z;
    }
    return ref_dot(normal, toL);
}

// cone_of10: cone of one light's 10 sample directions (DESIGN.md 2.3): axis = normalised sum, w = min_j axis.D_j, from a
// 16-byte aligned bundle loaded once as vectors and reduced from registers; w = -1 for a degenerate bundle (zero-length
// or non-unit direction).  One out-of-line copy for all lights.
__device__ __noinline__ float4 cone_of10(const float* __restrict__ d /* 32 floats, 30 used */) {
    const float4* __restrict__ d4 = reinterpret_cast<const float4*>(d);
    float v[32];
#pragma unroll
    for (int q = 0; q < 8; q++) {
        const float4 w = d4[q];
        v[4 * q] = w.x;
        v[4 * q + 1] = w.y;
        v[4 * q + 2] = w.z;
        v[4 * q + 3] = w.w;
    }
    float sx = 0.f, sy = 0.f, sz = 0.f;
#pragma unroll
    for (int j = 0; j < 10; j++) {
        sx += v[3 * j];
        sy += v[3 * j + 1];
        sz += v[3 * j + 2];
    }
    const float inv = rsqrtf(fmaf(sx, sx, fmaf(sy, sy, sz * sz)));
    float cmin = 1.f;
    bool ok = isfinite(inv);
    sx *= inv;
    sy *= inv;
    sz *= inv;
#pragma unroll
    for (int j = 0; j < 10; j++) {
        const float dd = fmaf(v[3 * j], v[3 * j], fmaf(v[3 * j + 1], v[3 * j + 1], v[3 * j + 2] * v[3 * j + 2]));
        // the filters and the sure-hit shortcut assume |D| = 1: the reference's normalise() leaves | |D|^2 - 1 |
        // below 5e-7 unless it degenerated (zero or denormal input), which is what this check catches
        ok = ok && fabsf(dd - 1.f) < 4e-6f;
        cmin = fminf(cmin, fmaf(sx, v[3 * j], fmaf(sy, v[3 * j + 1], sz * v[3 * j + 2])));
    }
    return make_float4(sx, sy, sz, ok ? cmin : -1.f);
}

// ------------------------------------------------------------------------------------
// shade_point: the shading set-up of one hit pixel (kernel.cu:1380-1425, 1643-1655): hit point, normal, shadow-ray
// origin `start`, texel colour.  `item` indexes the hit list.
// ------------------------------------------------------------------------------------
__device__ __forceinline__ void shade_point(const FrameParams& prm, uint32_t item, uint32_t*& out_px, int& my_id,
                                            v3& start, v3& normal, float& tr, float& tg, float& tb) {
    const uint32_t o = prm.hit_list[item];
    int frame, k, x;
    split_pixel(prm, o, frame, k, x);
    out_px = prm.pixels[frame] + out_index(prm, k, x);
    const CamP cam = prm.cam[frame];
    const v3 O0 = mk(cam.Ox, cam.Oy, cam.Oz);
    const v3 D = primary_dir(cam, prm.ez, prm.dx_tab[x], prm.dy_tab[k]);
    const float nt = prm.hit_ts[item];
    my_id = prm.hit_ids[item];
    v3 new_org = ref_add(O0, ref_scale(D, nt));
    float txf, tyf;
    if (my_id >= prm.n_spheres + prm.n_cubes + prm.n_planes) {
        // triangle hit, kernel.cu:1380-1394
        triangle_attributes(prm.tris + 27 * (size_t)(my_id - prm.n_spheres - prm.n_cubes - prm.n_planes),
                            prm.mesh_has_normals, O0.x, O0.y, O0.z, D.x, D.y, D.z, nt, &normal, &new_org, &txf, &tyf);
    } else if (my_id >= prm.n_spheres + prm.n_cubes) {
        // plane hit, kernel.cu:1407-1416
        const float4 no = __ldg(&prm.planes[2 * (my_id - prm.n_spheres - prm.n_cubes) + 1]);
        normal = mk(no.x, no.y, no.z);
        txf = 0.5f;
        tyf = 0.5f;
    } else {
        // sphere hit kernel.cu:1396-1405 / cube hit :1417-1425: normal from the primitive's `orgin`
        const float4 sc = (my_id < prm.n_spheres) ? __ldg(&prm.sph_exact[my_id])
                                                  : __ldg(&prm.cubes[3 * (my_id - prm.n_spheres) + 2]);
        normal = ref_sub(new_org, mk(sc.x, sc.y, sc.z));
        ref_normalise(normal);
        txf = (float)((1 + (double)ORE_ATAN2F(normal.z, normal.x) / 3.1415) * 0.5);
        tyf = (float)((double)ORE_ACOSF(normal.y) / 3.1415);
    }
    const int maxX = prm.tex_w, maxY = prm.tex_h;
    start = ref_add(ref_scale(normal, 0.00001f), new_org);
    int c_index = (int)(tyf * (float)maxY) * maxX + (int)(txf * (float)maxX);
    c_index = clamp_index(c_index, maxX * maxY);
    tr = __ldg(&prm.tex_r[c_index]);
    tg = __ldg(&prm.tex_g[c_index]);
    tb = __ldg(&prm.tex_b[c_index]);
}

// ------------------------------------------------------------------------------------
// shade_setup_kernel (stage A of the default shadow pass)
//
// Per hit pixel: shading set-up + the 10 shadow-ray directions of every light and the cone around them, written to the
// staging buffer.  This is all the per-pixel transcendental code (atan2f/acosf/cosf/sinf, ~30 KB of instructions);
// keeping it out of the sweep kernel lets each kernel's hot loop stay resident in the SM instruction cache (DESIGN.md).
// Warps run independently: each fetches blocks of 32 consecutive hit-list items.
// ------------------------------------------------------------------------------------
#ifndef ORE_STAGE_A_MIN_CTAS
#define ORE_STAGE_A_MIN_CTAS (1024 / ORE_STAGE_A_THREADS)
#endif
__global__ void __launch_bounds__(STAGE_A_THREADS, ORE_STAGE_A_MIN_CTAS) shade_setup_kernel(const FrameParams prm, const StageArgs st) {
    const int lane = threadIdx.x & 31;
    const uint32_t n_items = (uint32_t)prm.counters[CNT_HITS];
    for (;;) {
        uint32_t wb = 0;
        if (lane == 0) wb = (uint32_t)atomicAdd(&prm.counters[CNT_STAGE_A0 + st.chunk], 1ull);
        wb = __shfl_sync(0xffffffffu, wb, 0);
        if (wb >= st.cap_blocks) break;
        const uint32_t blk = st.first_block + wb;
        if ((unsigned long long)blk * 32ull >= n_items) break;
        const uint32_t item = blk * 32u + lane;
        const bool valid = item < n_items;
        const long long dbg_t0 = prm.dbg_cycles ? clock64() : 0;
        uint32_t* out_px = nullptr;
        int my_id = -1;
        v3 start = mk(1e9f, 1e9f, 1e9f), normal = mk(0.f, 0.f, 0.f);
        float tr = 0.f, tg = 0.f, tb = 0.f;
        if (valid) shade_point(prm, item, out_px, my_id, start, normal, tr, tg, tb);
        float* __restrict__ sp = st.buf + ((size_t)wb * (size_t)st.nv) * 32u + lane;
        sp[0] = start.x;
        sp[32] = start.y;
        sp[64] = start.z;
        sp[96] = tr;
        sp[128] = tg;
        sp[160] = tb;
#pragma unroll 1
        for (int li = 0; li < prm.n_lights; li++) {
            __align__(16) float d[32];
            float a = 0.f;
            float4 cn = make_float4(0.f, 0.f, 0.f, -1.f);
            float* __restrict__ q = sp + (size_t)(STAGE_HEADER + STAGE_PER_LIGHT * li) * 32u;
            LightP L;
            {
                const LightP* __restrict__ src = &prm.lights[0];
                L.px = src[li].px; L.py = src[li].py; L.pz = src[li].pz; L.size = src[li].size;
                L.r = src[li].r; L.g = src[li].g; L.b = src[li].b;
            }
            if (prm.skip_dark) {
                // a light that faces none of the block's pixels (a > 0 nowhere) adds +0 to each of them: only `a` is
                // staged, the sweep skips the light as well
                if (valid) a = light_facing(L.px, L.py, L.pz, start, normal);
                if (!__any_sync(0xffffffffu, valid && a > 0.f)) {
                    q[128] = a;
                    continue;
                }
            }
            if (valid) {
                a = light_directions_reuse(L, start, normal, d);
                cn = cone_of10(d);
            }
            q[0] = cn.x;
            q[32] = cn.y;
            q[64] = cn.z;
            q[96] = cn.w;
            q[128] = a;
            if (valid) {
                const float4* __restrict__ d4 = reinterpret_cast<const float4*>(d);
                float* __restrict__ qd = q + STAGE_DIRS_AT * 32;
#pragma unroll
                for (int v = 0; v < 8; v++) {
                    const float4 w = d4[v];
                    qd[(4 * v) * 32] = w.x;
                    qd[(4 * v + 1) * 32] = w.y;
                    if (4 * v + 2 < 30) qd[(4 * v + 2) * 32] = w.z;
                    if (4 * v + 3 < 30) qd[(4 * v + 3) * 32] = w.w;
                }
            }
        }
        if (prm.dbg_cycles && lane == 0 && blk < prm.dbg_cap) prm.dbg_cycles[blk] = (uint32_t)(clock64() - dbg_t0);
    }
}

}  // namespace ore

#include "ore_primary.cuh"
#include "ore_sweep.cuh"

namespace ore {

// ------------------------------------------------------------------------------------
// count_reference_tests_kernel (ORE_FLAG_COUNT_REFERENCE_TESTS, never on the timed path)
// The reference's own any-hit loop, literally: one ray at a time, spheres in index order,
// exact sequence, break at the first hit (kernel.cu:1501-1510).  Sums the number of
// sphere::intersect calls that loop order makes - the "tests" of the algorithmic rate
// (SURVEY.md 8d).  One thread per (hit pixel, light).
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) count_reference_tests_kernel(const FrameParams prm) {
    const uint32_t n_items = (uint32_t)prm.counters[CNT_HITS];
    const unsigned long long total = (unsigned long long)n_items * (unsigned long long)prm.n_lights;
    unsigned long long mine = 0;
    for (unsigned long long w = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; w < total;
         w += (unsigned long long)gridDim.x * blockDim.x) {
        // consecutive threads = consecutive hit pixels of one light (coherent loops)
        const uint32_t light = (uint32_t)(w / n_items), item = (uint32_t)(w % n_items);
        const int id = prm.hit_ids[item];
        if (id >= prm.n_spheres) continue;   // the count is defined for sphere scenes (SURVEY.md 8d)
        const uint32_t o = prm.hit_list[item];
        int frame, k, x;
        split_pixel(prm, o, frame, k, x);
        const CamP cam = prm.cam[frame];
        const v3 O0 = mk(cam.Ox, cam.Oy, cam.Oz);
        const v3 D = primary_dir(cam, prm.ez, prm.dx_tab[x], prm.dy_tab[k]);
        const float nt = prm.hit_ts[item];
        const float4 sc = __ldg(&prm.sph_exact[id]);
        const v3 new_org = ref_add(O0, ref_scale(D, nt));
        v3 normal = ref_sub(new_org, mk(sc.x, sc.y, sc.z));
        ref_normalise(normal);
        const v3 start = ref_add(ref_scale(normal, 0.00001f), new_org);
        __align__(16) float dir[32];
        light_directions_reuse(prm.lights[light], start, normal, dir);
#pragma unroll 1
        for (int j = 0; j < 10; j++) {
            const v3 d = mk(dir[j * 3 + 0], dir[j * 3 + 1], dir[j * 3 + 2]);
            int i = 0;
            bool shadow = false;
            for (; i < prm.n_spheres; i++) {
                const float4 s = __ldg(&prm.sph_exact[i]);
                float t;
                if (ref_intersect(start, d, s.x, s.y, s.z, s.w, t)) {
                    shadow = true;
                    break;
                }
            }
            mine += (unsigned long long)(shadow ? i + 1 : prm.n_spheres);
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) mine += __shfl_down_sync(0xffffffffu, mine, d);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(&prm.counters[CNT_SHADOW_TESTS_REF], mine);
}

// ------------------------------------------------------------------------------------
// fp32_burn_kernel: dependent-chain-free FFMA burn used to MEASURE the FP32 roofline
// denominator on the box (MEASURED_PEAKS.json carries HBM and bf16 peaks only).
// 16 independent accumulators per thread, 2 FLOP per FFMA.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) fp32_burn_kernel(float* out, int iters, float a, float b) {
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; i++) acc[i] = (float)(threadIdx.x + i);
#pragma unroll 1
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
#pragma unroll
            for (int i = 0; i < 16; i++) acc[i] = fmaf(acc[i], a, b);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; i++) s += acc[i];
    if (s == 12345.678f) out[0] = s;  // never true; keeps the chain alive
}

// ------------------------------------------------------------------------------------
// libm_probe_kernel: evaluates the device libm used by the path on caller-supplied inputs (tests only)
// op: 0 cosf, 1 sinf, 2 acosf, 3 atan2f(y = a, x = b)
// ------------------------------------------------------------------------------------
__global__ void libm_probe_kernel(int op, int n, const float* a, const float* b, float* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float r;
    if (op == 0)
        r = ORE_COSF(a[i]);
    else if (op == 1)
        r = ORE_SINF(a[i]);
    else if (op == 2)
        r = ORE_ACOSF(a[i]);
    else if (op == 3)
        r = ORE_ATAN2F(a[i], b[i]);
    else {
        // ops 4-6: component (op - 4) of ref_normalise((a[i], b[i], a[(i + 1) % n]))
        v3 v = mk(a[i], b[i], a[(i + 1) % n]);
        ref_normalise(v);
        r = op == 4 ? v.x : (op == 5 ? v.y : v.z);
    }
    out[i] = r;
}

}  // namespace ore
