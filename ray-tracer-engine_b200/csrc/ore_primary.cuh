// ore_primary.cuh - prep_frame_kernel and primary_tile_kernel (round 2).
//
//   prep_frame_kernel   : per-frame tables (dx per column, dy per rendered row, in the reference's double arithmetic)
//                         and the camera-space filter records of every sphere (in the Morton order of the upload), of
//                         every LEAF (8 consecutive spheres), of every SUPER-cluster (32 leaves) and, in a large scene,
//                         of every HYPER-cluster (32 supers); same for the leaf boxes of a mesh.
//   primary_tile_kernel : nearest hit (castRay, kernel.cu:1288-1431) for tiles of 32 x 8 pixels, one warp per tile:
//                           1. the tile's bounding cone against the super-clusters, then the leaves, then - four
//                              surviving leaves per step - the spheres (records staged in shared memory by TMA bulk
//                              copies, shared by the CTA's warps);
//                           2. per surviving sphere the per-pixel filter (one FFMA per row) and, where it passes, the
//                              reference's exact sequence; candidates are adjudicated by (t, original index), which is
//                              what ascending order with the strict '<' of kernel.cu:1335 yields;
//                           3. hit records (pixel, id, t) appended to the hit list, grouped by hit primitive inside the
//                              tile - nothing is written for miss pixels;
//                           4. the sky (skybox::getFColor, kernel.cu:1146-1166) for the tile's miss pixels in a QUAD
//                              layout: every lane owns four consecutive pixels of a row and stores them with one 128-bit
//                              store (hit pixels of a quad are written as 0 and overwritten by the shadow pass).  The
//                              texel index is a piecewise constant function of the direction: a cheap approximate
//                              evaluation (sky_fast) decides it wherever the pixel lies clear of a texel boundary by
//                              more than its own error bound; the few pixels near a boundary (and those near the
//                              poles) are queued in shared memory and run the exact sequence 32 at a time.
//                         Warps fetch tiles dynamically (tile cost varies ~8x between sky and sphere tiles).
//                         Large scenes (LARGE) start the walk of step 1 one level higher, at the hyper-clusters.
#pragma once

namespace ore {

#ifndef ORE_PRIMARY_THREADS
#define ORE_PRIMARY_THREADS 128
#endif
#ifndef ORE_PRIMARY_MIN_CTAS
#define ORE_PRIMARY_MIN_CTAS 6
#endif
constexpr int PRIMARY_THREADS = ORE_PRIMARY_THREADS;
constexpr int PRIMARY_WARPS = PRIMARY_THREADS / 32;
constexpr int LEAF_SPHERES = 8;    // = ore_host::LEAF_SPHERES (ore_clusters.h)
constexpr int SUPER_LEAVES = 32;   // = ore_host::SUPER_LEAVES
constexpr int HYPER_SUPERS = 32;   // = ore_host::HYPER_SUPERS

// Tile-cone record of a ball (centre c, radius R) seen from the eye O (DESIGN.md 2.4): a pixel tile whose directions
// lie within `a` of its axis A can only contain a hit if  A.M + cos(a) sv - sin(a) sqrt(LL - sv^2) <= 0  with
// M = R^T (O - c), sv = sqrt(Cm).  r2 = R^2 (already including the caller's margin).
__device__ __forceinline__ void ball_records(const FrameParams& prm, const CamP& cam, double Lx, double Ly, double Lz, double r2,
                                             float4* prim, float4* cone) {
    const double LL = Lx * Lx + Ly * Ly + Lz * Lz;
    const double Cm = LL * (1.0 - ORE_KAPPA_PRIMARY) - r2 * (1.0 + ORE_KAPPA_PRIMARY);
    if (!(Cm > 1e-9 * LL) || !(Cm > 1e-30)) {
        // origin in / near the ball (or a non-finite record): always a candidate
        if (prim) *prim = make_float4(0.f, 0.f, -ORE_BIG, 0.f);
        *cone = make_float4(0.f, 0.f, 0.f, -ORE_BIG);
        return;
    }
    const double sv = sqrt(Cm);
    const double cp = cam.cp, sp = cam.sp, cy = cam.cy, sy = cam.sy;
    const double Mx = cy * Lx - sy * Lz;
    const double My = sp * sy * Lx + cp * Ly + sp * cy * Lz;
    const double Mz = cp * sy * Lx - sp * Ly + cp * cy * Lz;
    if (prim) *prim = make_float4((float)(Mx / sv), (float)(My / sv), (float)((double)prm.fz * Mz / sv), 0.f);
    const double Rpp = sqrt(LL - Cm);
    const double Wd = (double)prm.tile_ca * sv - (double)prm.tile_sa * Rpp;
    *cone = make_float4((float)Mx, (float)My, (float)Mz, (float)(Wd - 4e-6 * sqrt(LL) - 1e-30));
}

template <bool LARGE>
__global__ void prep_frame_kernel(const FrameParams prm) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < CNT_SLOTS) prm.counters[i] = 0ull;
    if (i < prm.W_pad) {
        // kernel.cu:1624  float dx = aspect * (2 * (x + 0.5) / (float)width) - 1;   (double)   [columns >= W: padding]
        double v = (double)prm.aspect * (2 * (i + 0.5) / (double)(float)prm.W) - 1;
        const_cast<float*>(prm.dx_tab)[i] = (float)v;
    }
    if (i < prm.n_rows) {
        // kernel.cu:1625  float dy = aspect * (2 * (y + 0.5) / (float)height)*((float)height/width) - 1;
        const int y = prm.y0 + image_row_rel(prm, i);
        float hw = (float)prm.H / (float)prm.W;
        double v = (double)prm.aspect * (2 * (y + 0.5) / (double)(float)prm.H) * (double)hw - 1;
        const_cast<float*>(prm.dy_tab)[i] = (float)v;
    }
    // camera-space records: one set per frame of the batch
    for (int f = 0; f < prm.n_frames; f++) {
        const CamP cam = prm.cam[f];
        if (i < prm.n_sort) {
            // sphere at sorted position i (positions >= n_spheres are padding: never a candidate)
            float4 out = make_float4(0.f, 0.f, ORE_BIG, 0.f);
            float4 cone = make_float4(0.f, 0.f, 0.f, ORE_BIG);
            if (i < prm.n_spheres) {
                const float4 s = prm.sph_xsort[i];
                // L exactly as the reference forms it (float), then the filter works in double
                ball_records(prm, cam, (double)(cam.Ox - s.x), (double)(cam.Oy - s.y), (double)(cam.Oz - s.z), (double)(s.w * s.w), &out, &cone);
            }
            prm.prim_sorted[(size_t)f * prm.n_sort + i] = out;
            prm.cone_sorted[(size_t)f * prm.n_sort + i] = cone;
        }
        if (i < prm.n_leaves_pad) {
            float4 cone = make_float4(0.f, 0.f, 0.f, ORE_BIG);
            if (i < prm.n_leaves) {
                const float4 q = prm.leaf_sph[i];
                ball_records(prm, cam, (double)cam.Ox - q.x, (double)cam.Oy - q.y, (double)cam.Oz - q.z, (double)q.w * q.w, nullptr, &cone);
            }
            prm.leaf_cone[(size_t)f * prm.n_leaves_pad + i] = cone;
        }
        if (i < prm.n_supers_pad) {
            float4 cone = make_float4(0.f, 0.f, 0.f, ORE_BIG);
            if (i < prm.n_supers) {
                const float4 q = prm.super_sph[i];
                ball_records(prm, cam, (double)cam.Ox - q.x, (double)cam.Oy - q.y, (double)cam.Oz - q.z, (double)q.w * q.w, nullptr, &cone);
            }
            prm.super_cone[(size_t)f * prm.n_supers_pad + i] = cone;
        }
        if (LARGE && i < prm.n_hypers_pad) {
            float4 cone = make_float4(0.f, 0.f, 0.f, ORE_BIG);
            if (i < prm.n_hypers) {
                const float4 q = prm.hyper_sph[i];
                ball_records(prm, cam, (double)cam.Ox - q.x, (double)cam.Oy - q.y, (double)cam.Oz - q.z, (double)q.w * q.w, nullptr, &cone);
            }
            prm.hyper_cone[(size_t)f * prm.n_hypers_pad + i] = cone;
        }
        if (i < prm.n_boxes && i < __ldg(prm.n_live_boxes)) {
            // tile-cone record of leaf box i of the mesh from its bounding sphere (same formula).  An eye on a face plane
            // of the box makes it always a candidate: a primary ray with a +-0 component on that axis can pass the slab
            // test through a NaN slab and then hit a triangle the box does not contain (ore_kernels.cuh, zero_axes)
            const float4 q = prm.box_sph[i];
            float4 rec;
            ball_records(prm, cam, (double)cam.Ox - q.x, (double)cam.Oy - q.y, (double)cam.Oz - q.z, (double)q.w * q.w, nullptr, &rec);
            if (on_face_plane(7u, cam.Ox, cam.Oy, cam.Oz, prm.boxes[2 * i], prm.boxes[2 * i + 1]))
                rec = make_float4(0.f, 0.f, 0.f, -ORE_BIG);
            prm.box_cone[(size_t)f * prm.n_boxes + i] = rec;
        }
    }
}

// skybox::getFColor + rgbToInt (kernel.cu:1146-1166, 1688) for the pixel with image-plane coordinates (dx, dy)
struct SkyArgs {
    const float *r, *g, *b;
    int w, h;
    float radius;
    float ez;
};
template <bool FAST_LIBM>
__device__ __noinline__ uint32_t sky_pixel(const SkyArgs sk, const CamP cam, float dx, float dy) {
    // primary ray, kernel.cu:1624-1631 + camera::rotateDir :252-255
    const v3 D = primary_dir(cam, sk.ez, dx, dy);
    const v3 O = mk(cam.Ox, cam.Oy, cam.Oz);
    float t;
    ref_intersect(O, D, 0.f, 0.f, 0.f, sk.radius, t);
    v3 hp = ref_add(O, ref_scale(D, t));
    v3 n = ref_sub(hp, mk(0.f, 0.f, 0.f));
    ref_normalise(n);
    int sx = (int)((1.f + libm_atan2f<FAST_LIBM>(n.z, n.x) / 3.1415f) * 0.5f * (float)sk.w);
    int sy = (int)(libm_acosf<FAST_LIBM>(n.y) / 3.1415f * (float)sk.h);
    int index = clamp_index(sy * sk.w + sx, sk.w * sk.h);
    float r = __ldg(&sk.r[index]), g = __ldg(&sk.g[index]), b = __ldg(&sk.b[index]);
    return ref_rgb_to_int((int)(r * 254.f), (int)(g * 254.f), (int)(b * 254.f));
}

// ------------------------------------------------------------------------------------
// sky_fast: conservative shortcut for skybox::getFColor.  The exact sequence (sky_pixel above) computes
//   n = normalise(O + D t), t = the NEAR root of the sky sphere (negative: kernel.cu:346-351 keeps the smaller root, so the
//   sky is looked up BEHIND the ray), sx = (int)((1 + atan2f(n.z, n.x) / 3.1415f) 0.5f w), sy = (int)(acosf(n.y) / 3.1415f h)
// and fetches texel sy * w + sx.  sky_fast evaluates u ~ (1 + phi/3.1415) w/2 and v ~ theta/3.1415 h with fused
// arithmetic, MUFU reciprocals / square roots and a degree-13 polynomial arctangent, and accepts its own (floor(u), floor(v))
// only when u and v lie further than Eu, Ev from the next integer:
//   direction error  |n~ - n| <= 8e-6 (budget: 1e-6 for D~ against the reference's float D, 0.7e-6 for t~ - relative
//                    error 1e-6 times |O|/R <= 0.5, guarded per frame - and 0.7e-6 for the roundings of both paths: 2.4e-6,
//                    x3), which moves phi and theta by at most 8e-6 / rho, rho = |(n.x, n.z)| (pixels with rho < 0.02, i.e.
//                    within 1.2 degrees of a pole, always take the exact path);
//   angle error      4e-6 rad for the polynomial (3.2e-7 evaluated in float, tests/test_sky_filter_cpu.py), the approximate
//                    reciprocal (1.2e-7), the quadrant fix-ups (2.4e-7) and the 1-ulp error of either libm's atan2f / acosf
//                    (2.4e-7; 2 ulp for CUDA's in the FAST_LIBM kernels) - under 1e-6 in total;
//   float roundings  of the u, v expressions on both sides: < 2.7e-7 (w or h) texels, budgeted 1e-6 (w or h) + 1e-4.
// NaNs fail every comparison and fall through to the exact path.
// ------------------------------------------------------------------------------------
struct SkyFast {
    float Ox, Oy, Oz, cp, sp, cy, sy, fz, fz2;
    float c;                  // O.O - R^2  (R^2 = sky_radius^2: the squared member, kernel.cu:334)
    float ku, hw, kv;         // u = phi * ku + hw, v = theta * kv
    float eu0, eu1, ev0, ev1; // Eu = eu0 + eu1 / rho, Ev = ev0 + ev1 / rho
    int ok;                   // 0: exact path for every pixel (exhaustive mode, camera not well inside the sky sphere)
};
__device__ __forceinline__ SkyFast make_sky_fast(const CamP& cam, float fz, int w, int h, float sky_radius, bool enabled) {
    SkyFast s;
    s.Ox = cam.Ox; s.Oy = cam.Oy; s.Oz = cam.Oz;
    s.cp = cam.cp; s.sp = cam.sp; s.cy = cam.cy; s.sy = cam.sy;
    s.fz = fz;
    s.fz2 = fz * fz;
    const float R2 = sky_radius * sky_radius;
    const float OO = fmaf(cam.Ox, cam.Ox, fmaf(cam.Oy, cam.Oy, cam.Oz * cam.Oz));
    s.c = OO - R2;
    s.ku = 0.5f * (float)w / 3.1415f;
    s.hw = 0.5f * (float)w;
    s.kv = (float)h / 3.1415f;
    s.eu1 = 8e-6f * s.ku;
    s.eu0 = fmaf(4e-6f, s.ku, fmaf(1e-6f, (float)w, 1e-4f));
    s.ev1 = 8e-6f * s.kv;
    s.ev0 = fmaf(4e-6f, s.kv, fmaf(1e-6f, (float)h, 1e-4f));
    // the camera well inside a sky sphere of sane size: the near root is the negative one and |O| / R <= 0.5
    s.ok = (enabled && R2 >= 1.f && R2 < 1e30f && OO <= 0.25f * R2 && fabsf(cam.cp) <= 1.f && fabsf(cam.sp) <= 1.f &&
            fabsf(cam.cy) <= 1.f && fabsf(cam.sy) <= 1.f && w > 0 && h > 0 && w <= 65536 && h <= 65536 &&
            (float)w * (float)h < 1.0e9f /* the texel index stays far inside int range */) ? 1 : 0;
    return s;
}
__device__ __forceinline__ float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// atan2(y, x) for (x, y) != (0, 0), absolute error < 1e-6: a / b = min / max of the magnitudes, odd polynomial on [0, 1]
__device__ __forceinline__ float atan2_approx(float y, float x) {
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    const float a = mn * rcp_approx(mx);
    const float q = a * a;
    float p = 0.006791701540350914f;
    p = fmaf(p, q, -0.03352927789092064f);
    p = fmaf(p, q, 0.07951410859823227f);
    p = fmaf(p, q, -0.132254496216774f);
    p = fmaf(p, q, 0.19804944097995758f);
    p = fmaf(p, q, -0.3331688940525055f);
    p = fmaf(p, q, 0.9999958276748657f);
    float r = p * a;
    if (ay > ax) r = 1.57079632679f - r;
    if (x < 0.f) r = 3.14159265359f - r;
    return y < 0.f ? -r : r;
}
// returns true and the pixel when the texel is decided without the exact sequence
__device__ __forceinline__ bool sky_fast(const SkyFast& s, const float* __restrict__ tr, const float* __restrict__ tg,
                                         const float* __restrict__ tb, int w, int h, float dx, float dy, uint32_t& px) {
    // primary direction (kernel.cu:1624-1631, 252-255), approximately
    const float inv = rsqrt_approx(fmaf(dx, dx, fmaf(dy, dy, s.fz2)));
    const float nx0 = dx * inv, ny0 = dy * inv, nz0 = s.fz * inv;
    const float Dy = fmaf(ny0, s.cp, -(nz0 * s.sp));
    const float z1 = fmaf(ny0, s.sp, nz0 * s.cp);
    const float Dx = fmaf(nx0, s.cy, z1 * s.sy);
    const float Dz = fmaf(-nx0, s.sy, z1 * s.cy);
    // near root of |O + D t| = R with A = |D|^2 ~ 1:  t = -(b + sqrt(b^2 - c)),  b = D.O,  c = O.O - R^2 < 0
    const float b = fmaf(Dx, s.Ox, fmaf(Dy, s.Oy, Dz * s.Oz));
    const float t = -(b + sqrt_approx(fmaf(b, b, -s.c)));
    const float hx = fmaf(Dx, t, s.Ox), hy = fmaf(Dy, t, s.Oy), hz = fmaf(Dz, t, s.Oz);
    const float hinv = rsqrt_approx(fmaf(hx, hx, fmaf(hy, hy, hz * hz)));
    const float nx = hx * hinv, ny = hy * hinv, nz = hz * hinv;
    const float rho2 = fmaf(nx, nx, nz * nz);
    if (!(rho2 > 4e-4f)) return false;                 // within 1.2 degrees of a pole (or NaN)
    const float irho = rsqrt_approx(rho2);
    const float rho = rho2 * irho;
    const float u = fmaf(atan2_approx(nz, nx), s.ku, s.hw);
    const float v = atan2_approx(rho, ny) * s.kv;      // theta = acos(n.y) = atan2(rho, n.y) for a unit n (|n|^2 - 1 <= 4e-7: inside the budget)
    const float fu = floorf(u), fv = floorf(v);
    const float Eu = fmaf(s.eu1, irho, s.eu0), Ev = fmaf(s.ev1, irho, s.ev0);
    const float du = u - fu, dv = v - fv;
    if (!(du >= Eu && du <= 1.f - Eu && dv >= Ev && dv <= 1.f - Ev && fu >= 0.f && fv >= 0.f)) return false;
    const int index = clamp_index((int)fv * w + (int)fu, w * h);
    const float r = __ldg(&tr[index]), g = __ldg(&tg[index]), bl = __ldg(&tb[index]);
    px = ref_rgb_to_int((int)(r * 254.f), (int)(g * 254.f), (int)(bl * 254.f));
    return true;
}

// tile cone against a staged record: candidate iff A.M + W <= 0
__device__ __forceinline__ bool cone_touches(float ax, float ay, float az, const float4 rec) {
    return fmaf(ax, rec.x, fmaf(ay, rec.y, fmaf(az, rec.z, rec.w))) <= 0.f;
}

// LARGE: the large-scene variant (FrameParams::hyper_cone).  Only the hyper-cluster records are staged in shared memory
// (<= 32 KB up to 2^24 spheres); the walk is hyper -> super -> leaf -> sphere, with the super, leaf and sphere records
// read through the read-only path (L2-resident: about 18 MB per frame at 1M spheres).  Everything past the leaf level
// is the same code as in the other instantiations.
template <int P, bool EXH, bool FAST_LIBM, bool LARGE>
__global__ void __launch_bounds__(PRIMARY_THREADS, ORE_PRIMARY_MIN_CTAS) primary_tile_kernel(const FrameParams prm) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t warp_tot[PRIMARY_WARPS];
    __shared__ uint32_t cta_base;
    __shared__ int s_batch;
    // sky phase: the tile's pixels (row p, column c at p * 32 + c) and the queue of pixels that need the exact sequence
    __shared__ __align__(16) uint32_t s_tile[PRIMARY_WARPS][32 * P];
    __shared__ uint8_t s_queue[PRIMARY_WARPS][32 * P];
    static_assert(32 * P <= 256, "queue entries are bytes");
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // ---- the cone records of ONE frame at a time are staged in shared memory: [supers][leaves][spheres, when they fit]
    //      - one TMA bulk copy each, shared by the CTA's warps for all their tiles of that frame.  Batches are fetched
    //      in ascending order, so a CTA restages at most once per frame of the batch. ----
    //      (LARGE: [hypers] only.) ----
    float4* const s_super = reinterpret_cast<float4*>(smem_raw);
    float4* const s_leaf = s_super + prm.n_supers_pad;
    float4* const s_sph = s_leaf + prm.n_leaves_pad;
    const float4* const s_hyper = reinterpret_cast<const float4*>(smem_raw);
    const float4* __restrict__ g_super = nullptr;   // LARGE: this frame's super and leaf records in global memory
    const float4* __restrict__ g_leaf = nullptr;
    if (tid == 0) {
        mbar_init(&bar, 1);
        mbar_fence_init();
        s_batch = (int)atomicAdd(&prm.counters[CNT_PRIMARY_CURSOR], 1ull);
    }
    __syncthreads();
    uint32_t bar_phase = 0;
    int staged_frame = -1;
    const float4* __restrict__ sph_cone = s_sph;

    const int tiles_x = (prm.W + 31) / 32;
    const int tiles_y = (prm.n_rows + P - 1) / P;
    const int total_tiles = tiles_x * tiles_y;
    const int batches_per_frame = (total_tiles + PRIMARY_WARPS - 1) / PRIMARY_WARPS;
    const int n_batches = batches_per_frame * prm.n_frames;
    const int n_sph = prm.n_spheres, n_leaf = prm.n_leaves, n_sup = prm.n_supers;
    const bool pitch_ok = (prm.sky_pitch & 3) == 0;
    const SkyArgs sk = {prm.sky_r, prm.sky_g, prm.sky_b, prm.sky_w, prm.sky_h, prm.sky_radius, prm.ez};
    unsigned long long n_exact = 0;
    unsigned int n_steps = 0, n_sky_exact = 0;

    // batches of PRIMARY_WARPS adjacent tiles of one frame, fetched dynamically (tile cost varies ~8x between sky and
    // sphere tiles); the CTA appends the hit records of a batch with ONE atomic, so neighbouring tiles stay neighbours in
    // the hit list
    for (;;) {
        const int batch = s_batch;
        if (batch >= n_batches) break;
        const int frame = batch / batches_per_frame;
        if (frame != staged_frame) {
            // (every warp is past its reads of the previous frame's records: it has gone through the barriers of the
            // previous batch since)
            __syncthreads();
            if constexpr (LARGE) {
                if (tid == 0) {
                    const uint32_t b_hyp = (uint32_t)prm.n_hypers_pad * 16u;
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    mbar_expect_tx(&bar, b_hyp);
                    if (b_hyp) tma_bulk_g2s(smem_raw, prm.hyper_cone + (size_t)frame * prm.n_hypers_pad, b_hyp, &bar);
                }
                g_super = prm.super_cone + (size_t)frame * prm.n_supers_pad;
                g_leaf = prm.leaf_cone + (size_t)frame * prm.n_leaves_pad;
                sph_cone = prm.cone_sorted + (size_t)frame * prm.n_sort;
            } else {
                if (tid == 0) {
                    const uint32_t b_sup = (uint32_t)prm.n_supers_pad * 16u, b_leaf = (uint32_t)prm.n_leaves_pad * 16u;
                    const uint32_t b_sph = prm.cone_resident ? (uint32_t)prm.n_sort * 16u : 0u;
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    mbar_expect_tx(&bar, b_sup + b_leaf + b_sph);
                    if (b_sup) tma_bulk_g2s(s_super, prm.super_cone + (size_t)frame * prm.n_supers_pad, b_sup, &bar);
                    if (b_leaf) tma_bulk_g2s(s_leaf, prm.leaf_cone + (size_t)frame * prm.n_leaves_pad, b_leaf, &bar);
                    if (b_sph) tma_bulk_g2s(s_sph, prm.cone_sorted + (size_t)frame * prm.n_sort, b_sph, &bar);
                }
            }
            mbar_wait(&bar, bar_phase);
            bar_phase ^= 1u;
            staged_frame = frame;
            if constexpr (!LARGE) sph_cone = prm.cone_resident ? s_sph : prm.cone_sorted + (size_t)frame * prm.n_sort;
        }
        const CamP cam = prm.cam[frame];
        const v3 O = mk(cam.Ox, cam.Oy, cam.Oz);
        const DirArgs da = {prm.ez, cam.cp, cam.sp, cam.cy, cam.sy};
        const float4* __restrict__ prim_rec = prm.prim_sorted + (size_t)frame * prm.n_sort;
        uint32_t* const frame_px = prm.sky_pixels[frame];
        const bool vec_ok = pitch_ok && ((reinterpret_cast<uintptr_t>(frame_px) & 15u) == 0);
        const int tile_id = (batch - frame * batches_per_frame) * PRIMARY_WARPS + warp;
        const bool tile_ok = tile_id < total_tiles;
        const int ty = tile_ok ? tile_id / tiles_x : 0;
        const int tx = tile_ok ? tile_id % tiles_x : 0;
        const int x = tx * 32 + lane;
        const bool x_ok = tile_ok && x < prm.W;
        const float dx = prm.dx_tab[x];   // dx_tab is padded to a multiple of 32 columns

        float dyp[P], negn[P], best_t[P];
        int best_id[P];
#pragma unroll
        for (int p = 0; p < P; p++) {
            const int k = ty * P + p;
            const bool ok = x_ok && k < prm.n_rows;
            dyp[p] = prm.dy_tab[min(k, prm.n_rows - 1)];
            const float nv = sqrtf(fmaf(dx, dx, fmaf(dyp[p], dyp[p], prm.fz * prm.fz)));
            // per-pixel filter threshold: candidate iff g' <= -|v| (shrunk a little: more candidates)
            negn[p] = ok ? (EXH ? INFINITY : -nv * 0.99999905f) : -INFINITY;
            best_t[p] = INFINITY;
            best_id[p] = -1;
        }
        // tile axis in the camera frame: nominal tile centre on the image plane (warp-uniform)
        float ax, ay, az;
        {
            const float cx = prm.dx_tab[tx * 32] + 15.5f * prm.px_delta;
            const float cy = 0.5f * (dyp[0] + dyp[P - 1]);
            const float inv = rsqrtf(fmaf(cx, cx, fmaf(cy, cy, prm.fz * prm.fz)));
            ax = cx * inv;
            ay = cy * inv;
            az = prm.fz * inv;
        }

        // ---- triangles first (kernel.cu:1293-1328): they seed the strict '<' search the spheres continue.
        //      Lane i tests leaf box s0+i (its bounding sphere) against the tile cone; surviving leaves, in
        //      ascending order, get the exact slab + triangle tests per pixel. ----
        if (prm.n_boxes) {
            const int n_live = __shfl_sync(0xffffffffu, lane == 0 ? __ldg(prm.n_live_boxes) : 0, 0);   // (one load per warp)
            const MeshArgs ma = {prm.tris, prm.boxes, prm.box_offsets, prm.box_indices, n_live};
            const int id_base = prm.n_spheres + prm.n_cubes + prm.n_planes;
#pragma unroll 1
            for (int s0 = 0; s0 < n_live; s0 += 32) {
                bool cand = false;
                if (s0 + lane < n_live) cand = EXH || cone_touches(ax, ay, az, __ldg(&prm.box_cone[(size_t)frame * prm.n_boxes + s0 + lane]));
                uint32_t mask = __ballot_sync(0xffffffffu, cand && tile_ok);
                while (mask) {
                    const int i = __ffs(mask) - 1;
                    mask &= mask - 1;
#pragma unroll
                    for (int p = 0; p < P; p++) {
                        if (x_ok && ty * P + p < prm.n_rows) {
                            const v3 D = primary_dir_call(da, dx, dyp[p]);
                            nearest_in_leaf(ma, s0 + i, id_base, O.x, O.y, O.z, D.x, D.y, D.z, &best_t[p], &best_id[p]);
                        }
                    }
                }
            }
        }

        // ---- spheres: (LARGE: hyper-clusters ->) super-clusters -> leaves -> (four leaves per step) spheres ->
        //      per-pixel filter -> exact.  open_super is everything below the super level. ----
        auto open_super = [&](const int sup) {
            const int leaf = sup * SUPER_LEAVES + lane;
            const int lc = min(leaf, n_leaf - 1);
            uint32_t cmask = __ballot_sync(0xffffffffu, leaf < n_leaf && (EXH || cone_touches(ax, ay, az, LARGE ? __ldg(&g_leaf[lc]) : s_leaf[lc])));
            n_steps++;
#pragma unroll 1
            while (cmask) {
                int mine = -1;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int c = cmask ? __ffs(cmask) - 1 : -1;
                    cmask &= cmask - 1;
                    if ((lane >> 3) == k) mine = c;
                }
                const int s_mine = mine >= 0 ? (sup * SUPER_LEAVES + mine) * LEAF_SPHERES + (lane & 7) : n_sph;
                const bool in = s_mine < n_sph;
                const int sc = in ? s_mine : 0;
                uint32_t wmask = __ballot_sync(0xffffffffu, in && (EXH || cone_touches(ax, ay, az, LARGE ? __ldg(&sph_cone[sc]) : sph_cone[sc])));
                n_steps++;
                while (wmask) {
                    const int i = __ffs(wmask) - 1;
                    wmask &= wmask - 1;
                    const int s = __shfl_sync(0xffffffffu, s_mine, i);
                    const float4 q = __ldg(&prim_rec[s]);
                    const float e = fmaf(dx, q.x, q.z);
                    uint32_t pass = 0;
#pragma unroll
                    for (int p = 0; p < P; p++) pass |= (fmaf(dyp[p], q.y, e) <= negn[p]) ? (1u << p) : 0u;
                    if (pass) {
                        const float4 ex = __ldg(&prm.sph_xsort[s]);
                        const int id = __ldg(&prm.sort_index[s]);
#pragma unroll
                        for (int p = 0; p < P; p++) {
                            if ((pass >> p) & 1u) {
                                const v3 D = primary_dir_call(da, dx, dyp[p]);
                                float t;
                                n_exact++;
                                if (ref_intersect(O, D, ex.x, ex.y, ex.z, ex.w, t)) {
                                    // kernel.cu:1335 visits the spheres in ascending index with a strict '<': the
                                    // winner is the smallest t and, among equal t, the lowest sphere index - but
                                    // never a sphere against a triangle found before it with the same t
                                    const bool better = t < best_t[p] ||
                                                        (t == best_t[p] && best_id[p] >= 0 && best_id[p] < n_sph && id < best_id[p]);
                                    if (better) {
                                        best_t[p] = t;
                                        best_id[p] = id;
                                    }
                                }
                            }
                        }
                    }
                }
            }
        };
        if constexpr (LARGE) {
            const int n_hyp = prm.n_hypers;
#pragma unroll 1
            for (int h0 = 0; h0 < n_hyp; h0 += 32) {
                uint32_t hmask = __ballot_sync(0xffffffffu, tile_ok && h0 + lane < n_hyp &&
                                                                (EXH || cone_touches(ax, ay, az, s_hyper[min(h0 + lane, n_hyp - 1)])));
                n_steps++;
#pragma unroll 1
                while (hmask) {
                    const int hyp = h0 + __ffs(hmask) - 1;
                    hmask &= hmask - 1;
                    const int sl = hyp * HYPER_SUPERS + lane;
                    uint32_t smask = __ballot_sync(0xffffffffu, sl < n_sup && (EXH || cone_touches(ax, ay, az, __ldg(&g_super[min(sl, n_sup - 1)]))));
                    n_steps++;
#pragma unroll 1
                    while (smask) {
                        const int sup = hyp * HYPER_SUPERS + __ffs(smask) - 1;
                        smask &= smask - 1;
                        open_super(sup);
                    }
                }
            }
        } else {
#pragma unroll 1
            for (int s0 = 0; s0 < n_sup; s0 += 32) {
                uint32_t smask = __ballot_sync(0xffffffffu, tile_ok && s0 + lane < n_sup &&
                                                                (EXH || cone_touches(ax, ay, az, s_super[min(s0 + lane, n_sup - 1)])));
                n_steps++;
#pragma unroll 1
                while (smask) {
                    const int sup = s0 + __ffs(smask) - 1;
                    smask &= smask - 1;
                    open_super(sup);
                }
            }
        }

        // ---- cubes, then planes (kernel.cu:1344-1372): exact tests continuing the same strict '<' search ----
        if (prm.n_cubes | prm.n_planes) {
#pragma unroll
            for (int p = 0; p < P; p++) {
                if (x_ok && ty * P + p < prm.n_rows) {
                    const v3 D = primary_dir_call(da, dx, dyp[p]);
                    nearest_cube_plane(prm.cubes, prm.n_cubes, prm.planes, prm.n_planes, prm.n_spheres, O.x, O.y, O.z, D.x, D.y,
                                       D.z, &best_t[p], &best_id[p]);
                }
            }
        }

        // ---- sky for the miss pixels, quad layout: lane L owns pixels x4 .. x4+3 of row 4h + L/8 and stores them
        //      with one 128-bit store (hit pixels of a quad are written as 0; the shadow pass overwrites them).
        //      Pass 1: sky_fast per pixel into the warp's tile buffer, undecided pixels into the queue; pass 2: the exact
        //      sequence for the queue, 32 entries at a time; pass 3: the stores. ----
        uint32_t hmask[P];
#pragma unroll
        for (int p = 0; p < P; p++) hmask[p] = __ballot_sync(0xffffffffu, best_id[p] >= 0);
        if (tile_ok) {
            uint32_t* const tp = s_tile[warp];
            uint8_t* const tq = s_queue[warp];
            const SkyFast sf = make_sky_fast(cam, prm.fz, prm.sky_w, prm.sky_h, prm.sky_radius, !EXH);
            const int x4 = tx * 32 + 4 * (lane & 7);
            uint32_t n_q = 0;
#pragma unroll 1
            for (int h = 0; h < P / 4; h++) {
                const int pr = 4 * h + (lane >> 3);
                uint32_t hm = 0;
                float dy = 0.f;
#pragma unroll
                for (int p = 0; p < P; p++)
                    if (p == pr) {
                        hm = hmask[p];
                        dy = dyp[p];
                    }
                const int k = ty * P + pr;
                const uint32_t hits4 = (hm >> (4 * (lane & 7))) & 0xFu;
                uint4 px = make_uint4(0u, 0u, 0u, 0u);
                uint32_t need = 0;
                if (k < prm.n_rows && x4 < prm.W) {
                    const float4 dx4 = *reinterpret_cast<const float4*>(&prm.dx_tab[x4]);
                    // (rolled, with selects instead of indexed registers: ONE copy of sky_fast in the instruction stream)
#pragma unroll 1
                    for (int j = 0; j < 4; j++) {
                        if (!((hits4 >> j) & 1u) && x4 + j < prm.W) {
                            const float dxj = j == 0 ? dx4.x : (j == 1 ? dx4.y : (j == 2 ? dx4.z : dx4.w));
                            uint32_t pj = 0u;
                            if (!sf.ok || !sky_fast(sf, sk.r, sk.g, sk.b, sk.w, sk.h, dxj, dy, pj)) need |= 1u << j;
                            px.x = j == 0 ? pj : px.x;
                            px.y = j == 1 ? pj : px.y;
                            px.z = j == 2 ? pj : px.z;
                            px.w = j == 3 ? pj : px.w;
                        }
                    }
                }
                *reinterpret_cast<uint4*>(&tp[pr * 32 + 4 * (lane & 7)]) = px;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const bool nd = (need >> j) & 1u;
                    const uint32_t bal = __ballot_sync(0xffffffffu, nd);
                    if (nd) tq[n_q + __popc(bal & ((1u << lane) - 1u))] = (uint8_t)(pr * 32 + 4 * (lane & 7) + j);
                    n_q += __popc(bal);
                }
            }
            __syncwarp();
#pragma unroll 1
            for (uint32_t q0 = 0; q0 < n_q; q0 += 32) {
                if (q0 + lane < n_q) {
                    const int e = tq[q0 + lane];
                    const int kq = min(ty * P + (e >> 5), prm.n_rows - 1);
                    tp[e] = sky_pixel<FAST_LIBM>(sk, cam, prm.dx_tab[tx * 32 + (e & 31)], prm.dy_tab[kq]);
                }
            }
            __syncwarp();
#pragma unroll 1
            for (int h = 0; h < P / 4; h++) {
                const int pr = 4 * h + (lane >> 3);
                const int k = ty * P + pr;
                if (k < prm.n_rows && x4 < prm.W) {
                    const uint4 v = *reinterpret_cast<const uint4*>(&tp[pr * 32 + 4 * (lane & 7)]);
                    uint32_t* dst = frame_px + sky_out_index(prm, k, x4);
                    if (vec_ok && x4 + 3 < prm.W) {
                        *reinterpret_cast<uint4*>(dst) = v;  // 128-bit RGBA store
                    } else {
                        const uint32_t pv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                        for (int j = 0; j < 4; j++)
                            if (x4 + j < prm.W) dst[j] = pv[j];
                    }
                }
            }
            n_sky_exact += n_q;
        }

        // ---- hit records, grouped by hit primitive (ascending id), row-major inside a group, so that the 32
        //      consecutive entries a shadow warp takes mostly lie on ONE sphere (tight beams) ----
        uint32_t warp_hits = 0;
        uint32_t my_off[P];
        {
            uint32_t rem = 0;
#pragma unroll
            for (int p = 0; p < P; p++) {
                my_off[p] = 0;
                if (best_id[p] >= 0) rem |= 1u << p;   // (only in-range pixels can have a hit)
            }
            while (__any_sync(0xffffffffu, rem != 0)) {
                int cur = 0x7fffffff;
#pragma unroll
                for (int p = 0; p < P; p++)
                    if ((rem >> p) & 1u) cur = min(cur, best_id[p]);
                cur = __reduce_min_sync(0xffffffffu, cur);
#pragma unroll
                for (int p = 0; p < P; p++) {
                    const bool m = ((rem >> p) & 1u) && best_id[p] == cur;
                    const uint32_t bal = __ballot_sync(0xffffffffu, m);
                    if (m) {
                        my_off[p] = warp_hits + __popc(bal & ((1u << lane) - 1u));
                        rem &= ~(1u << p);
                    }
                    warp_hits += __popc(bal);
                }
            }
        }
        if (lane == 0) warp_tot[warp] = warp_hits;
        __syncthreads();
        if (tid == 0) {
            uint32_t tot = 0;
            for (int w = 0; w < PRIMARY_WARPS; w++) {
                const uint32_t v = warp_tot[w];
                warp_tot[w] = tot;
                tot += v;
            }
            cta_base = tot ? (uint32_t)atomicAdd(&prm.counters[CNT_HITS], (unsigned long long)tot) : 0u;
            s_batch = (int)atomicAdd(&prm.counters[CNT_PRIMARY_CURSOR], 1ull);   // the CTA's next batch
        }
        __syncthreads();
        const uint32_t wbase = cta_base + warp_tot[warp];
#pragma unroll
        for (int p = 0; p < P; p++) {
            if (best_id[p] >= 0) {
                const uint32_t at = wbase + my_off[p];
                prm.hit_list[at] = (uint32_t)frame * prm.n_px_frame + (uint32_t)((ty * P + p) * prm.W + x);
                prm.hit_ids[at] = best_id[p];
                prm.hit_ts[at] = best_t[p];
            }
        }
        // (no third barrier: s_batch / cta_base / warp_tot are only rewritten after the NEXT batch's first barrier,
        // which every warp reaches after reading them here)
    }
    if (n_exact) atomicAdd(&prm.counters[CNT_EXACT_PRIMARY], n_exact);
    if (lane == 0 && n_steps) atomicAdd(&prm.counters[CNT_PRIMARY_STEPS], (unsigned long long)n_steps);
    if (lane == 0 && n_sky_exact) atomicAdd(&prm.counters[CNT_SKY_EXACT], (unsigned long long)n_sky_exact);
}

// ------------------------------------------------------------------------------------
// expand_hits_kernel (ore_get_hits only, never on the timed path): per-pixel id / t maps from the compact hit records
// ------------------------------------------------------------------------------------
__global__ void fill_hits_kernel(int32_t* __restrict__ hit_id, float* __restrict__ hit_t, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        hit_id[i] = -1;
        hit_t[i] = INFINITY;
    }
}
__global__ void expand_hits_kernel(const FrameParams prm, int32_t* __restrict__ hit_id, float* __restrict__ hit_t) {
    const uint32_t n_items = (uint32_t)prm.counters[CNT_HITS];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += gridDim.x * blockDim.x) {
        const uint32_t o = prm.hit_list[i];
        hit_id[o] = prm.hit_ids[i];
        hit_t[o] = prm.hit_ts[i];
    }
}

}  // namespace ore
