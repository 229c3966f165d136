// ore_clusters.h - shadow-sweep clusters of the sphere set: the arithmetic shared by the device build
// (ore_scene_build.cu) and the host builder below, which is the CPU reference the tests compare the device build with
// (tests/test_clusters_cpu.py, tests/test_scene_update_gpu.py).  No CUDA types; also compiled by plain g++.
//
// The spheres in Morton order of their centres with two levels of bounding balls over them: LEAVES of 8 consecutive
// spheres and SUPER-clusters of 32 consecutive leaves (build_hierarchy below; build_clusters also returns round 1's
// 32-sphere cluster balls, which only the containment test still looks at).  Neither the any-hit result of a shadow ray
// nor - with candidates adjudicated by (t, original index) - the nearest hit depends on the order spheres are visited in,
// so the shadow sweep and the primary kernel test supers first, open the leaves of the survivors and only then single
// spheres (DESIGN.md 2.4).  Soundness rests on one property, which tests/test_clusters_cpu.py checks: every member ball
// (centre, R') lies inside the ball of its leaf AND inside the ball of its super-cluster, or that radius is +inf
// ("always open": a member with non-finite or >= 1e15 coordinates / radius).
//
// Every ORE_HD helper is compiled for both sides.  The library is built with --fmad=false and the host side with g++
// without FMA, so the same double / float expressions give the same bits on the host and on the device.
#ifndef ORE_CLUSTERS_H
#define ORE_CLUSTERS_H
#include <math.h>

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <utility>
#include <vector>

#if defined(__CUDACC__)
#define ORE_HD __host__ __device__
#else
#define ORE_HD
#endif

// shadow-ray margin of the sweep's sphere test; R' below is rounded up so that R'^2 >= (1 + kappa) r^4 in float
#define ORE_KAPPA_SHADOW 3.814697265625e-06f /* 2^-18 */

namespace ore_host {

struct Rec4 {  // layout of float4
    float x, y, z, w;
};

ORE_HD inline bool tame_value(float v) { return isfinite(v) && fabsf(v) < 1e15f; }
ORE_HD inline bool tame_record(const Rec4& s) { return tame_value(s.x) && tame_value(s.y) && tame_value(s.z) && tame_value(s.w); }

// R' of a sphere record's radius MEMBER: the test squares the stored member (kernel.cu:334), so the effective radius is
// sqrt(r4 (1 + kappa)) with r4 = member^2, rounded up so that R'^2 >= (1 + kappa) r4 in float
ORE_HD inline float shadow_radius(float member) {
    if (isnan(member)) {
        // the member's own NaN, quietened - what x86 arithmetic passes through the steps below (a device returns its
        // canonical NaN instead), so that both sides store the same bits
        uint32_t u;
        memcpy(&u, &member, sizeof u);
        u |= 0x00400000u;
        memcpy(&member, &u, sizeof u);
        return member;
    }
    const float r4 = member * member;
    float rp = (float)sqrt((double)r4 * (1.0 + (double)ORE_KAPPA_SHADOW));
    rp = nextafterf(rp, INFINITY);
    while (rp * rp < (float)((double)r4 * (1.0 + (double)ORE_KAPPA_SHADOW))) rp = nextafterf(rp, INFINITY);
    return rp;
}

// 10-bit Morton coordinate of one centre coordinate over [lo, hi], the range of the TAME centres on that axis
// (lo = 1e300, hi = -1e300 when there is none: every coordinate of that axis then maps to 0)
ORE_HD inline uint32_t morton_axis(float c, double lo, double hi) {
    double t = 0.0;
    if (tame_value(c) && hi > lo) t = ((double)c - lo) / (hi - lo);
    const double s = t * 1023.0;
    const double s0 = 0.0 < s ? s : 0.0;          // std::max(0.0, s)
    return (uint32_t)(s0 < 1023.0 ? s0 : 1023.0);  // std::min(1023.0, s0)
}
ORE_HD inline uint32_t morton_spread(uint32_t v) {
    v &= 1023u;
    v = (v | (v << 16)) & 0x030000FFu;
    v = (v | (v << 8)) & 0x0300F00Fu;
    v = (v | (v << 4)) & 0x030C30C3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}
ORE_HD inline uint32_t morton_key(const Rec4& s, const double lo[3], const double hi[3]) {
    return morton_spread(morton_axis(s.x, lo[0], hi[0])) | (morton_spread(morton_axis(s.y, lo[1], hi[1])) << 1) |
           (morton_spread(morton_axis(s.z, lo[2], hi[2])) << 2);
}

// |c_i - centre| + |R'_i| of one member ball, in double
ORE_HD inline double member_reach(const Rec4& s, const float f[3]) {
    const double dx = (double)s.x - f[0], dy = (double)s.y - f[1], dz = (double)s.z - f[2];
    return sqrt(dx * dx + dy * dy + dz * dz) + fabs((double)s.w);
}
// a radius the float tests can use: finite and below 1e15, rounded up to the next float
ORE_HD inline bool boundable(double rad) { return isfinite(rad) && rad < 1e15; }
ORE_HD inline float rounded_radius(double rad) { return nextafterf((float)(rad * (1.0 + 1e-6) + 1e-30), INFINITY); }

// ex / sh: n exact records (cx,cy,cz,radius member) and n shadow records (cx,cy,cz,R').  Outputs: sorted_shadow and
// sorted_exact with ceil(n/32)*32 entries (the tail repeats the last sphere; the kernels never read index >= n),
// bounds with ceil(n/32) rounded up to a multiple of 4 entries (centre, radius; padding = zeros) - the 32-sphere
// clusters of round 1, kept for the containment test - and, optionally, the permutation itself.
inline void build_clusters(const Rec4* ex, const Rec4* sh, int n, std::vector<Rec4>& sorted_shadow,
                           std::vector<Rec4>& sorted_exact, std::vector<Rec4>& bounds, std::vector<int>* sort_index = nullptr) {
    const int n_clu = (n + 31) / 32;
    const size_t n_sort = (size_t)n_clu * 32, n_clu_pad = ((size_t)n_clu + 3) & ~(size_t)3;
    sorted_shadow.assign(n_sort, Rec4{0.f, 0.f, 0.f, 0.f});
    sorted_exact.assign(n_sort, Rec4{0.f, 0.f, 0.f, 0.f});
    bounds.assign(n_clu_pad, Rec4{0.f, 0.f, 0.f, 0.f});
    if (sort_index) sort_index->assign(n_sort, 0);
    if (n <= 0) return;

    // Morton keys (10 bits per axis) over the bounding box of the tame centres
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    for (int i = 0; i < n; i++) {
        const float c[3] = {sh[i].x, sh[i].y, sh[i].z};
        for (int k = 0; k < 3; k++)
            if (tame_value(c[k])) {
                lo[k] = std::min(lo[k], (double)c[k]);
                hi[k] = std::max(hi[k], (double)c[k]);
            }
    }
    std::vector<std::pair<uint32_t, int>> order((size_t)n);
    for (int i = 0; i < n; i++) order[(size_t)i] = {morton_key(sh[i], lo, hi), i};
    std::stable_sort(order.begin(), order.end(), [](const std::pair<uint32_t, int>& a, const std::pair<uint32_t, int>& b) {
        return a.first < b.first;
    });

    for (size_t p = 0; p < n_sort; p++) {
        const int i = order[p < (size_t)n ? p : (size_t)n - 1].second;
        sorted_shadow[p] = sh[i];
        sorted_exact[p] = ex[i];
        if (sort_index) (*sort_index)[p] = i;   // original index of the sphere at sorted position p
    }
    for (size_t j = 0; j < (size_t)n_clu; j++) {
        const size_t p0 = j * 32, p1 = std::min(p0 + 32, (size_t)n);
        double cx = 0, cy = 0, cz = 0;
        bool tame = true;
        for (size_t p = p0; p < p1; p++) {
            const Rec4& s = sorted_shadow[p];
            tame = tame && tame_value(s.x) && tame_value(s.y) && tame_value(s.z) && tame_value(s.w);
            cx += s.x;
            cy += s.y;
            cz += s.z;
        }
        const double m = (double)(p1 - p0);
        const float fx = (float)(cx / m), fy = (float)(cy / m), fz = (float)(cz / m);
        double rad = 0;
        for (size_t p = p0; p < p1 && tame; p++) {
            const Rec4& s = sorted_shadow[p];
            const double dx = (double)s.x - fx, dy = (double)s.y - fy, dz = (double)s.z - fz;
            rad = std::max(rad, std::sqrt(dx * dx + dy * dy + dz * dz) + (double)s.w);
        }
        float fr = INFINITY;  // "always open": a member the float tests cannot bound
        if (tame && std::isfinite(rad) && rad < 1e15) fr = std::nextafter((float)(rad * (1.0 + 1e-6) + 1e-30), INFINITY);
        bounds[j] = Rec4{fx, fy, fz, fr};
    }
}

// Candidate centre of a tame member set: 0 = mean of the m centres (summed in member order), 1 = centre of the box
// around the member balls.
ORE_HD inline void ball_candidate(int cand, const double mean[3], const double lo[3], const double hi[3], double m, float f[3]) {
    for (int k = 0; k < 3; k++) f[k] = (float)(cand ? 0.5 * (lo[k] + hi[k]) : mean[k] / m);
}

// Bounding ball of the m member balls s[0, m): centre = the better of (mean of the centres, centre of the box around
// the member balls), radius = max |c_i - centre| + R'_i, rounded up.  +inf ("always open") when a member cannot be
// bounded by the float tests.  Only the mean depends on the order of the members; the box and the max do not.
ORE_HD inline Rec4 bounding_ball(const Rec4* s, size_t m) {
    if (m == 0) return Rec4{0.f, 0.f, 0.f, 0.f};
    double mean[3] = {0, 0, 0}, lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    bool tame = true;
    for (size_t p = 0; p < m; p++) {
        tame = tame && tame_record(s[p]);
        const double c[3] = {s[p].x, s[p].y, s[p].z}, r = fabs((double)s[p].w);
        for (int k = 0; k < 3; k++) {
            mean[k] += c[k];
            const double a = c[k] - r, b = c[k] + r;
            lo[k] = a < lo[k] ? a : lo[k];   // std::min(lo, a)
            hi[k] = hi[k] < b ? b : hi[k];   // std::max(hi, b)
        }
    }
    if (!tame) return Rec4{(float)0, (float)0, (float)0, INFINITY};
    Rec4 best{0.f, 0.f, 0.f, INFINITY};
    for (int cand = 0; cand < 2; cand++) {
        float f[3];
        ball_candidate(cand, mean, lo, hi, (double)m, f);
        double rad = 0;
        for (size_t p = 0; p < m; p++) {
            const double d = member_reach(s[p], f);
            rad = rad < d ? d : rad;         // std::max(rad, d)
        }
        if (boundable(rad)) {
            const float fr = rounded_radius(rad);
            if (fr < best.w) best = Rec4{f[0], f[1], f[2], fr};
        }
    }
    return best;
}
inline Rec4 bounding_ball(const std::vector<Rec4>& sorted, size_t p0, size_t p1) {
    return p1 <= p0 ? Rec4{0.f, 0.f, 0.f, 0.f} : bounding_ball(sorted.data() + p0, p1 - p0);
}

// Two more levels over the same Morton order (round 2, shadow_sweep_kernel): LEAVES of 8 consecutive spheres and
// SUPER-clusters of 32 consecutive leaves (256 spheres), one bounding ball each.  leaves: ceil(n/8) entries rounded up
// to a multiple of 32 (padding = radius -1: never touched); supers: ceil(n/256) entries rounded up to a multiple of 4.
constexpr int LEAF_SPHERES = 8;
constexpr int SUPER_LEAVES = 32;
inline void build_hierarchy(const std::vector<Rec4>& sorted_shadow, int n, std::vector<Rec4>& leaves, std::vector<Rec4>& supers) {
    const size_t n_leaf = ((size_t)std::max(n, 0) + LEAF_SPHERES - 1) / LEAF_SPHERES;
    const size_t n_sup = (n_leaf + SUPER_LEAVES - 1) / SUPER_LEAVES;
    leaves.assign((n_leaf + 31) & ~(size_t)31, Rec4{0.f, 0.f, 0.f, -1.f});
    supers.assign((n_sup + 3) & ~(size_t)3, Rec4{0.f, 0.f, 0.f, -1.f});
    for (size_t j = 0; j < n_leaf; j++)
        leaves[j] = bounding_ball(sorted_shadow, j * LEAF_SPHERES, std::min((j + 1) * LEAF_SPHERES, (size_t)n));
    const size_t per = (size_t)LEAF_SPHERES * SUPER_LEAVES;
    for (size_t k = 0; k < n_sup; k++) supers[k] = bounding_ball(sorted_shadow, k * per, std::min((k + 1) * per, (size_t)n));
}

}  // namespace ore_host
#endif
