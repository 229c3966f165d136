// ore_sweep.cuh - shadow_sweep_kernel: stage B of the default shadow pass (round 2).
//
// castLightRay's any-hit search (kernel.cu:1470-1544) for blocks of 32 hit pixels, one warp per block, ONE LIGHT AT A
// TIME.  What changed against the round-1 beam kernel and why:
//
//  * The 30 direction components of a light (stage A's output, 3840 bytes per block and light) arrive in shared
//    memory by ONE TMA bulk copy per warp (cp.async.bulk + mbarrier), double-buffered: light l+1 - or the next
//    block's first light - is in flight while light l is swept.  No per-thread local-memory copy (round 1 spilled a
//    96-float array per thread through L1 into DRAM: 1.9 GB written per 8K frame) and no dependent global loads in
//    the sweep.  Lane i owns column i of the [30][32] slot: conflict-free reads, and any lane can read any pixel's ray.
//  * Lights are swept separately.  Their beams point in different directions, so a joint sweep opens the union of
//    three cluster sets and tests every opened sphere against all three beams; separate sweeps test each opened sphere
//    against one.  The per-light code also needs a third of the beam state (fewer registers, more warps).
//  * Three levels over the Morton order: super-clusters of 256 spheres -> leaves of 8 -> spheres, and the leaf level
//    is DENSE: the warp opens four surviving leaves per step (lane i tests sphere i%8 of leaf i/8).  With clusters of
//    32 a narrow beam through 1024 spheres opened a third of the clusters (24 sweep steps per pass); leaves of 8 are
//    tighter and packed (about 8).
//  * CTAs of 64 threads: the kernel is warp-independent and persistent, and an SM only hands a finished CTA's
//    registers and shared memory to the next kernel when the CTA's LAST warp has run dry.  Small CTAs release an SM
//    almost warp by warp at the tail of a launch - what decides throughput when a rank renders an eighth of a frame.
//    The sphere / cluster records are therefore read through L1 (34 KB hot at 1024 spheres) instead of a per-CTA
//    shared-memory copy.
//
//  * Lights that face none of a block's pixels are skipped altogether (FrameParams::skip_dark): castLightRay multiplies
//    its sample count by max(0, normal.toL) (kernel.cu:1541-1542), so such a light adds exactly +0 whatever its shadow
//    rays do.  Stage A stages only `a` for it, the sweep neither copies its directions nor walks the spheres; a lane whose
//    own a is not > 0 drops out of a light the rest of its block still needs.  About half of all (pixel, light) pairs of
//    the benchmark scenes.
//
// The filters are those of DESIGN.md 2.1-2.5 unchanged (beam -> per-pixel cone -> per-ray -> sure hit -> exact
// sequence); only their schedule differs, and the any-hit result does not depend on the order spheres are visited in.
#pragma once

namespace ore {

#ifndef ORE_SWEEP_THREADS
#define ORE_SWEEP_THREADS 64
#endif
#ifndef ORE_SWEEP_WARPS_PER_SM
#define ORE_SWEEP_WARPS_PER_SM 24
#endif
constexpr int SWEEP_THREADS = ORE_SWEEP_THREADS;
constexpr int SWEEP_WARPS = SWEEP_THREADS / 32;
constexpr int SWEEP_MIN_CTAS = ORE_SWEEP_WARPS_PER_SM / SWEEP_WARPS;
constexpr int SWEEP_SLOT_FLOATS = 30 * 32;                    // one light's directions of one block: [30][32]
constexpr int SWEEP_SLOT_BYTES = SWEEP_SLOT_FLOATS * 4;       // 3840
constexpr size_t SWEEP_SMEM_BYTES = (size_t)SWEEP_WARPS * 2 * SWEEP_SLOT_BYTES + (size_t)SWEEP_WARPS * 2 * 8;

// one light's warp beam (DESIGN.md 2.4) against the ball q = (centre, radius).  Radius >= 1e18 or NaN: always.
struct Beam {
    float bx, by, bz;   // centroid of the group's origins
    float ax, ay, az;   // axis
    float tan_a, k1, k2;  // tan of the half-angle, -a_min, rho_perp
};
__device__ __forceinline__ bool beam_touches(const Beam& b, const float4 q) {
    const float Lx = b.bx - q.x, Ly = b.by - q.y, Lz = b.bz - q.z;
    const float LL = fmaf(Lz, Lz, fmaf(Ly, Ly, Lx * Lx));
    const float Rq = fmaf(q.w, 1.0001f, fmaf(LL, 1e-12f, 1e-6f));  // radius + rounding slack
    const float slack = LL * 2e-6f;                                 // cancellation in LL - sc^2
    const float sc = -fmaf(b.ax, Lx, fmaf(b.ay, Ly, b.az * Lz));    // centre's axial coordinate
    const float u = sc + Rq + b.k1;                                 // >= 0 unless wholly behind the origins
    const float thr = fmaf(u, b.tan_a, Rq + b.k2);
    const float d2 = fmaf(-sc, sc, LL);
    return !(q.w < 1e18f) || (u >= 0.f && d2 <= fmaf(thr, thr, slack));
}

// LARGE: the large-scene variant, with a level-H pass over the hyper-cluster balls (FrameParams::hyper_sph) before the
// super level; everything from the super level down is the same code as in the other instantiations.
template <bool EXH, bool STAGED, bool FAST_LIBM, bool LARGE>
__global__ void __launch_bounds__(SWEEP_THREADS, SWEEP_MIN_CTAS) shadow_sweep_kernel(const FrameParams prm, const StageArgs st) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* const slots = reinterpret_cast<float*>(smem_raw) + (size_t)warp * 2 * SWEEP_SLOT_FLOATS;
    uint64_t* const bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)SWEEP_WARPS * 2 * SWEEP_SLOT_BYTES) + warp * 2;
    if (STAGED) {
        if (lane == 0) {
            mbar_init(&bars[0], 1);
            mbar_init(&bars[1], 1);
            mbar_fence_init();
        }
        __syncwarp();
    }
    const float4* __restrict__ spheres = prm.sph_sort;   // cx,cy,cz,R' in Morton order
    const float4* __restrict__ leaves = prm.leaf_sph;    // bounding ball of spheres [8j, 8j+8)
    const float4* __restrict__ supers = prm.super_sph;   // bounding ball of leaves [32k, 32k+32)
    const int n_sph = prm.n_spheres, n_leaf = prm.n_leaves, n_sup = prm.n_supers;
    const uint32_t n_items = (uint32_t)prm.counters[CNT_HITS];
    const int NLI = prm.n_lights;
    // the live leaf count of the mesh (the leaves past it list no triangles), loaded once
    const int n_live_boxes = prm.n_boxes ? __shfl_sync(0xffffffffu, lane == 0 ? __ldg(prm.n_live_boxes) : 0, 0) : 0;
    unsigned long long n_exact = 0;
    unsigned int n_l1 = 0, n_l2 = 0, n_steps = 0;

    // TMA sequence of this warp: copy number q goes to slot q & 1 and completes phase (q >> 1) & 1 of its barrier
    uint32_t seq_issued = 0, seq_waited = 0;
    auto issue_dirs = [&](uint32_t wblk, int light) {
        if (lane == 0) {
            const float* src = st.buf + ((size_t)wblk * (size_t)st.nv + (size_t)(STAGE_HEADER + STAGE_PER_LIGHT * light + STAGE_DIRS_AT)) * 32u;
            uint64_t* bar = &bars[seq_issued & 1u];
            // the slot was read through the generic proxy (by every lane, all done: __syncwarp at the end of the light
            // that used it) and is now written through the async proxy
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_expect_tx(bar, SWEEP_SLOT_BYTES);
            tma_bulk_g2s(slots + (seq_issued & 1u) * SWEEP_SLOT_FLOATS, src, SWEEP_SLOT_BYTES, bar);
        }
        seq_issued++;
    };

    // lights that face at least one pixel of stage block wblk (bit li); every light when nothing may be skipped
    const uint32_t all_lights = NLI >= 32 ? 0xffffffffu : ((1u << NLI) - 1u);
    const bool skip_dark = prm.skip_dark != 0 && !EXH;
    auto lit_lights = [&](uint32_t wblk) -> uint32_t {
        if (!STAGED || !skip_dark) return all_lights;
        const float* __restrict__ a_at = st.buf + ((size_t)wblk * (size_t)st.nv + (size_t)(STAGE_HEADER + 4)) * 32u + lane;
        uint32_t m = 0;
#pragma unroll 1
        for (int li = 0; li < NLI; li++)
            if (__any_sync(0xffffffffu, a_at[(size_t)(STAGE_PER_LIGHT * li) * 32u] > 0.f)) m |= 1u << li;   // (lanes past the list hold a = 0)
        return m;
    };

    unsigned long long* const cursor = &prm.counters[STAGED ? CNT_STAGE_B0 + st.chunk : CNT_SHADOW_CURSOR];
    uint32_t wb = 0;
    if (lane == 0) wb = (uint32_t)atomicAdd(cursor, 1ull);
    wb = __shfl_sync(0xffffffffu, wb, 0);
    bool have_first = false;   // lit_cur describes block wb already, and its first lit light (if any) is in flight
    uint32_t lit_cur = all_lights;
    for (;;) {
        if (STAGED && wb >= st.cap_blocks) break;
        const uint32_t blk = st.first_block + wb;  // fused: 0, or the first block past the staged chunks (catch-all)
        if ((unsigned long long)blk * 32ull >= n_items) break;
        const uint32_t item = blk * 32u + lane;
        const bool valid = item < n_items;
        const long long dbg_t0 = prm.dbg_cycles ? clock64() : 0;
        if (STAGED && !have_first) {
            lit_cur = lit_lights(wb);
            if (lit_cur) issue_dirs(wb, __ffs(lit_cur) - 1);
        }
        // the next block is reserved one ahead (its first light is then copied while this block's last light is swept),
        // except near the end of the list / chunk, where a reserved block would wait behind this one while other warps run dry
        const bool ahead = (unsigned long long)(blk + 8192u) * 32ull < n_items && (!STAGED || wb + 8192u < st.cap_blocks);
        uint32_t wb_next = 0;
        if (ahead) {
            if (lane == 0) wb_next = (uint32_t)atomicAdd(cursor, 1ull);
            wb_next = __shfl_sync(0xffffffffu, wb_next, 0);
        }

        // ---- shading set-up (kernel.cu:1396-1405, 1643-1655), or its staged result ----
        uint32_t* out_px = nullptr;
        int my_id = -1;
        v3 start = mk(1e9f, 1e9f, 1e9f), normal = mk(0.f, 0.f, 0.f);
        float tr = 0.f, tg = 0.f, tb = 0.f;
        const float* __restrict__ sp = STAGED ? st.buf + ((size_t)wb * (size_t)st.nv) * 32u + lane : nullptr;
        if (STAGED) {
            if (valid) {
                int frame, k, x;
                split_pixel(prm, prm.hit_list[item], frame, k, x);
                out_px = prm.pixels[frame] + out_index(prm, k, x);
                my_id = (int)__ldg(&prm.hit_ids[item]);
                start = mk(sp[0], sp[32], sp[64]);
                tr = sp[96];
                tg = sp[128];
                tb = sp[160];
            }
        } else if (valid) {
            shade_point<FAST_LIBM>(prm, item, out_px, my_id, start, normal, tr, tg, tb);
        }
        float fr = 0.f, fg = 0.f, fb = 0.f;

        // Lanes are processed in groups that hit the SAME primitive (the hit list is grouped that way, so a warp normally
        // is one group; a warp straddling a silhouette is two or three): origins on one sphere give a narrow beam.  There
        // is no cap on the number of groups: lumping the leftovers of a block that straddles two distant tiles into one
        // group makes a beam as wide as the scene, which opens every leaf (measured: blocks of 4.7 ms at 16384 spheres).
        const uint32_t valid_mask = __ballot_sync(0xffffffffu, valid);

        uint32_t lit_rem = STAGED ? lit_cur : all_lights;
        have_first = false;
#pragma unroll 1
        while (lit_rem) {
            const int li = __ffs(lit_rem) - 1;
            lit_rem &= lit_rem - 1;
            const float* __restrict__ dslot;   // this light's directions: component c of ray r at dslot[(3 r + c) * 32]
            float Ax = 0.f, Ay = 0.f, Az = 0.f, ca = 0.f, sa = 0.f, a_dot = 0.f, cmin = -1.f;
            bool force = false;   // the cone test cannot be used for this lane's bundle: every sphere is a candidate
            if (STAGED) {
                // keep the copies one ahead: the next lit light of this block, or the first lit light of the reserved block
                if (lit_rem) {
                    issue_dirs(wb, __ffs(lit_rem) - 1);
                } else if (ahead && wb_next < st.cap_blocks && (unsigned long long)(st.first_block + wb_next) * 32ull < n_items) {
                    lit_cur = lit_lights(wb_next);
                    if (lit_cur) issue_dirs(wb_next, __ffs(lit_cur) - 1);
                    have_first = true;
                }
                const float* __restrict__ q = sp + (size_t)(STAGE_HEADER + STAGE_PER_LIGHT * li) * 32u;
                if (valid) {
                    Ax = q[0];
                    Ay = q[32];
                    Az = q[64];
                    cmin = q[96];
                    a_dot = q[128];
                }
                mbar_wait(&bars[seq_waited & 1u], (seq_waited >> 1) & 1u);
                dslot = slots + (seq_waited & 1u) * SWEEP_SLOT_FLOATS + lane;
                seq_waited++;
            } else {
                // fused form (catch-all / no staging memory): the lane computes its own bundle into the slot
                float* ds = slots + lane;
                __align__(16) float d[32];
                LightP L;
                {
                    const LightP* __restrict__ src = &prm.lights[0];
                    L.px = src[li].px; L.py = src[li].py; L.pz = src[li].pz; L.size = src[li].size;
                    L.r = src[li].r; L.g = src[li].g; L.b = src[li].b;
                }
                if (skip_dark) {
                    if (valid) a_dot = light_facing(L.px, L.py, L.pz, start, normal);
                    if (!__any_sync(0xffffffffu, valid && a_dot > 0.f)) continue;   // adds +0 to every pixel of the block
                }
                if (valid) {
                    a_dot = light_directions_reuse<FAST_LIBM>(L, start, normal, d);
                    const float4 cn = cone_of10(d);
                    Ax = cn.x;
                    Ay = cn.y;
                    Az = cn.z;
                    cmin = cn.w;
#pragma unroll
                    for (int j = 0; j < 30; j++) ds[j * 32] = d[j];
                }
                __syncwarp();
                dslot = ds;
            }
            // a lane this light does not face (a <= 0 or NaN: its contribution is multiplied by zero) takes no part
            const bool takes_part = valid && !(skip_dark && !(a_dot > 0.f));
            uint32_t blocked = takes_part ? 0u : 0x3ffu;
            if (!takes_part) Ax = Ay = Az = 0.f;
            if (takes_part) {
                if (cmin > 0.5f && !EXH) {
                    const float cosa = cmin - 4e-6f;
                    const float sina = sqrtf(fmaxf(0.f, fmaf(-cosa, cosa, 1.f))) * 1.0001f + 1e-6f;
                    ca = cosa - 0.00196f * sina;
                    sa = 1.002f * sina;
                } else {
                    // degenerate bundle (zero direction, very wide cone) or exhaustive mode
                    force = true;
                    Ax = Ay = Az = 0.f;
                }
            }

            uint32_t pending = valid_mask;
#pragma unroll 1
            while (pending) {
                const int gid = __shfl_sync(0xffffffffu, my_id, __ffs(pending) - 1);
                const bool ing = ((pending >> lane) & 1u) && my_id == gid;
                const uint32_t gm = __ballot_sync(0xffffffffu, ing);
                pending &= ~gm;
                // ---- warp beam of this group and light: an axis line through the origins' centroid; the group's rays
                //      stay within rho_perp + (axial distance) * tan(a) of it (DESIGN.md 2.4) ----
                Beam bm;
                bool wforce = __any_sync(0xffffffffu, ing && force);
                {
                    const float nvalid = (float)__popc(gm);
                    float bx = ing ? start.x : 0.f, by = ing ? start.y : 0.f, bz = ing ? start.z : 0.f;
#pragma unroll
                    for (int d = 16; d > 0; d >>= 1) {
                        bx += __shfl_xor_sync(0xffffffffu, bx, d);
                        by += __shfl_xor_sync(0xffffffffu, by, d);
                        bz += __shfl_xor_sync(0xffffffffu, bz, d);
                    }
                    const float inv_n = 1.f / fmaxf(nvalid, 1.f);
                    bx *= inv_n;
                    by *= inv_n;
                    bz *= inv_n;
                    const float ex = ing ? start.x - bx : 0.f, ey = ing ? start.y - by : 0.f, ez = ing ? start.z - bz : 0.f;
                    const float escale = 1e-5f * (fabsf(bx) + fabsf(by) + fabsf(bz) + 1.f);  // rounding slack on offsets
                    const bool part = ing && ca > 0.f;  // lanes whose bundle takes part (lit, not degenerate, not fully blocked)
                    float sx = part ? Ax : 0.f, sy = part ? Ay : 0.f, sz = part ? Az : 0.f;
#pragma unroll
                    for (int d = 16; d > 0; d >>= 1) {
                        sx += __shfl_xor_sync(0xffffffffu, sx, d);
                        sy += __shfl_xor_sync(0xffffffffu, sy, d);
                        sz += __shfl_xor_sync(0xffffffffu, sz, d);
                    }
                    const float n2 = fmaf(sx, sx, fmaf(sy, sy, sz * sz));
                    const float inv = rsqrtf(fmaxf(n2, 1e-30f));
                    sx *= inv;
                    sy *= inv;
                    sz *= inv;
                    // widest angle between the group axis and any participating ray: theta_lane + a_lane
                    float cw = 1.f, amin = 3e38f, rp = 0.f;
                    if (part) {
                        const float sina = sa * (1.f / 1.002f);
                        const float cosa = ca + 0.00196f * sina;
                        const float c1 = fminf(1.f, fmaf(sx, Ax, fmaf(sy, Ay, sz * Az)));
                        const float s1 = sqrtf(fmaxf(0.f, fmaf(-c1, c1, 1.f))) + 1e-6f;
                        cw = fmaf(c1, cosa, -(s1 * sina)) - 2e-6f;
                        const float ai = fmaf(ex, sx, fmaf(ey, sy, ez * sz));  // axial offset of this origin
                        const float px = ex - ai * sx, py = ey - ai * sy, pz = ez - ai * sz;
                        amin = ai;
                        rp = sqrtf(fmaf(px, px, fmaf(py, py, pz * pz)));
                    }
#pragma unroll
                    for (int d = 16; d > 0; d >>= 1) {
                        cw = fminf(cw, __shfl_xor_sync(0xffffffffu, cw, d));
                        amin = fminf(amin, __shfl_xor_sync(0xffffffffu, amin, d));
                        rp = fmaxf(rp, __shfl_xor_sync(0xffffffffu, rp, d));
                    }
                    const bool any_part = __any_sync(0xffffffffu, part);
                    if (!any_part && !wforce) continue;   // nothing of this group is left to decide for this light
                    if (any_part && (!(n2 > 1e-12f) || !(cw > 0.3f))) wforce = true;  // bundle axes disagree wildly
                    const float sinw = sqrtf(fmaxf(0.f, fmaf(-cw, cw, 1.f))) * 1.0001f + 1e-6f;
                    bm.bx = bx;
                    bm.by = by;
                    bm.bz = bz;
                    bm.ax = sx;
                    bm.ay = sy;
                    bm.az = sz;
                    bm.tan_a = sinw / fmaxf(cw, 0.3f) * 1.0001f;
                    bm.k1 = -(amin - escale);   // u = sc + R' + k1 < 0: wholly behind every origin
                    bm.k2 = rp * 1.0001f + escale;
                }
                if (EXH) wforce = true;

                bool warp_done = false;
                // everything below the super level, for super-cluster `sup`
                auto open_super = [&](const int sup) {
                    // ---- level 0: lane i tests leaf sup * 32 + i (8 spheres) ----
                    const int leaf = sup * 32 + lane;
                    uint32_t cmask = __ballot_sync(0xffffffffu, leaf < n_leaf && (wforce || beam_touches(bm, __ldg(&leaves[min(leaf, n_leaf - 1)]))));
                    n_steps++;
#pragma unroll 1
                    while (cmask && !warp_done) {
                        // ---- level 1, dense: the four lowest surviving leaves, lane i tests sphere i % 8 of leaf i / 8 ----
                        int mine = -1;
#pragma unroll
                        for (int k = 0; k < 4; k++) {
                            const int c = cmask ? __ffs(cmask) - 1 : -1;
                            cmask &= cmask - 1;   // (0 & -1 = 0)
                            if ((lane >> 3) == k) mine = c;
                        }
                        const int s_mine = mine >= 0 ? (sup * 32 + mine) * 8 + (lane & 7) : n_sph;
                        const bool in = s_mine < n_sph;
                        uint32_t wmask = __ballot_sync(0xffffffffu, in && (wforce || beam_touches(bm, __ldg(&spheres[in ? s_mine : 0]))));
                        n_steps++;
                        n_l1 += __popc(wmask);
                        // ---- level 2: every lane of the group runs its own cone test on the surviving spheres ----
                        while (wmask) {
                            const int i = __ffs(wmask) - 1;
                            wmask &= wmask - 1;
                            const int s = __shfl_sync(0xffffffffu, s_mine, i);
                            const float4 q = __ldg(&spheres[s]);
                            const float lx = start.x - q.x, ly = start.y - q.y, lz = start.z - q.z;
                            const float LL = fmaf(lz, lz, fmaf(ly, ly, lx * lx));
                            const float Cm = fmaf(LL, 1.0f - ORE_KAPPA_SHADOW, -(q.w * q.w));
                            const float sq = Cm * rsqrt_approx(Cm);
                            const float svu = (EXH || !(Cm > 1e-20f)) ? -ORE_BIG : sq;
                            uint32_t live = ing ? (~blocked & 0x3ffu) : 0u;
                            if (!force) {
                                const float T = fmaf(ca, svu, -(sa * q.w));
                                if (!(fmaf(Ax, lx, fmaf(Ay, ly, fmaf(Az, lz, T))) < 0.f)) live = 0u;
                            }
                            if (live) {
                                n_l2++;
                                const float4 ex4 = __ldg(&prm.sph_xsort[s]);
                                // per-ray filter h = D.L + s' < 0 on the 10 rays (shared-memory directions), the "sure
                                // hit" shortcut (DESIGN.md 2.5), then the exact sequence on what lies in between
                                const float sure_thr = (EXH || force)
                                                           ? INFINITY
                                                           : fmaxf(fmaf(LL, 1e-6f, 1e-6f), fmaf(LL, 2e-5f, fmaf(-ex4.w, ex4.w, LL)));
                                uint32_t m = 0, sure = 0;
#pragma unroll
                                for (int j = 0; j < 10; j++) {
                                    const float b = fmaf(dslot[(3 * j) * 32], lx, fmaf(dslot[(3 * j + 1) * 32], ly, dslot[(3 * j + 2) * 32] * lz));
                                    if (b + svu < 0.f) m |= 1u << j;
                                    if (b < 0.f && b * b > sure_thr) sure |= 1u << j;
                                }
                                sure &= m & live;  // only rays the filter lets through, that are still unblocked
                                blocked |= sure;
                                uint32_t cand = m & live & ~sure;
                                while (cand) {
                                    const int j = __ffs(cand) - 1;
                                    cand &= cand - 1;
                                    float t;
                                    n_exact++;
                                    if (ref_intersect(start, dir_at(dslot, 32, j), ex4.x, ex4.y, ex4.z, ex4.w, t)) blocked |= 1u << j;
                                }
                                if (blocked == 0x3ffu) {   // all 10 rays of this light are blocked: the lane drops out
                                    Ax = Ay = Az = 0.f;
                                    ca = 0.f;
                                    sa = 0.f;
                                    force = false;
                                }
                            }
                        }
                        if (__all_sync(0xffffffffu, !ing || blocked == 0x3ffu)) warp_done = true;
                    }
                };
                if constexpr (LARGE) {
                    const float4* __restrict__ hypers = prm.hyper_sph;   // bounding ball of supers [32h, 32h+32)
                    const int n_hyp = prm.n_hypers;
#pragma unroll 1
                    for (int h0 = 0; h0 < n_hyp && !warp_done; h0 += 32) {
                        // ---- level H: lane i tests hyper-cluster h0 + i (8192 spheres) ----
                        uint32_t hmask = __ballot_sync(0xffffffffu, h0 + lane < n_hyp && (wforce || beam_touches(bm, __ldg(&hypers[min(h0 + lane, n_hyp - 1)]))));
                        n_steps++;
#pragma unroll 1
                        while (hmask && !warp_done) {
                            const int hyp = h0 + __ffs(hmask) - 1;
                            hmask &= hmask - 1;
                            // ---- level S: lane i tests super-cluster hyp * 32 + i ----
                            const int sl = hyp * 32 + lane;
                            uint32_t smask = __ballot_sync(0xffffffffu, sl < n_sup && (wforce || beam_touches(bm, __ldg(&supers[min(sl, n_sup - 1)]))));
                            n_steps++;
#pragma unroll 1
                            while (smask && !warp_done) {
                                const int sup = hyp * 32 + __ffs(smask) - 1;
                                smask &= smask - 1;
                                open_super(sup);
                            }
                        }
                    }
                } else {
#pragma unroll 1
                    for (int s0 = 0; s0 < n_sup && !warp_done; s0 += 32) {
                        // ---- level S: lane i tests super-cluster s0 + i (256 spheres) ----
                        uint32_t smask = __ballot_sync(0xffffffffu, s0 + lane < n_sup && (wforce || beam_touches(bm, __ldg(&supers[min(s0 + lane, n_sup - 1)]))));
                        n_steps++;
#pragma unroll 1
                        while (smask && !warp_done) {
                            const int sup = s0 + __ffs(smask) - 1;
                            smask &= smask - 1;
                            open_super(sup);
                        }
                    }
                }
            }

            // ---- triangles (kernel.cu:1475-1497; tested first in the reference - the result is an OR, order-free):
            //      leaves outside the light's cone are skipped ----
            const bool use_cone = !EXH && !force && ca > 0.f;
            // rays blocked later only shrink the live set: this mask covers every box test below
            const uint32_t zaxes = (use_cone && (prm.n_boxes | prm.n_cubes) && valid) ? zero_axes(dslot, 32, ~blocked & 0x3ffu) : 0u;
            if (prm.n_boxes && valid) {
                const uint32_t live = ~blocked & 0x3ffu;
                if (live) {
                    const MeshArgs ma = {prm.tris, prm.boxes, prm.box_offsets, prm.box_indices, n_live_boxes};
                    blocked |= mesh_blocks_light(ma, prm.box_sph, start.x, start.y, start.z, Ax, Ay, Az, ca, sa, use_cone, zaxes, dslot, 32, live);
                }
            }
            // ---- planes, then cubes (kernel.cu:1512-1536) for the rays nothing blocked yet ----
            if ((prm.n_cubes | prm.n_planes) && valid) {
                const uint32_t live = ~blocked & 0x3ffu;
                if (live)
                    blocked |= cubes_planes_block_light(prm.cubes, prm.n_cubes, prm.planes, prm.n_planes, start.x, start.y, start.z,
                                                        Ax, Ay, Az, ca, sa, use_cone, zaxes, dslot, 32, live);
            }
            // ---- light accumulation (kernel.cu:1537-1543, 1673-1675) ----
            if (valid) {
                float b = c_b_of_k[10 - __popc(blocked & 0x3ffu)];
                b *= a_dot > 0 ? a_dot : 0;
                const LightP* __restrict__ src = &prm.lights[0];
                fr += b * src[li].r * tr;
                fg += b * src[li].g * tg;
                fb += b * src[li].b * tb;
            }
            __syncwarp();   // every lane is done with this light's slot before a later copy may overwrite it
        }
        if (valid) *out_px = ref_rgb_to_int((int)(fr * 254.f), (int)(fg * 254.f), (int)(fb * 254.f));
        if (STAGED && prm.dbg_cycles && lane == 0 && blk < prm.dbg_cap)
            prm.dbg_cycles[prm.dbg_cap + blk] = (uint32_t)(clock64() - dbg_t0);
        if (!ahead) {
            if (lane == 0) wb_next = (uint32_t)atomicAdd(cursor, 1ull);
            wb_next = __shfl_sync(0xffffffffu, wb_next, 0);
        }
        wb = wb_next;
    }
    if (n_exact) atomicAdd(&prm.counters[CNT_EXACT_SHADOW], n_exact);
    if (lane == 0 && n_l1) atomicAdd(&prm.counters[CNT_BEAM_L1], (unsigned long long)n_l1);
    if (n_l2) atomicAdd(&prm.counters[CNT_BEAM_L2], (unsigned long long)n_l2);
    if (lane == 0 && n_steps) atomicAdd(&prm.counters[CNT_SWEEP_STEPS], (unsigned long long)n_steps);
}

}  // namespace ore
