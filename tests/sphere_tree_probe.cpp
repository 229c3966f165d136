// Test-only C wrapper: the host builder of csrc/ore_clusters.h producing the six arrays of the sphere hierarchy exactly
// as the device holds them after ore_set_spheres / ore_set_spheres_device (tests/test_scene_update_gpu.py compares them
// byte for byte with ore_debug_sphere_tree).
#include "ore_clusters.h"

#include <cstring>

using ore_host::Rec4;

// lengths: sph_exact, sorted arrays, leaves, supers (include/ore_render.h, ore_debug_sphere_tree); -1 on a mismatch
extern "C" int ore_probe_sphere_tree(const float* xyz_radius, int n, float* sph_exact, float* xsort, float* ssort, int* sort_index,
                                     float* leaves, float* supers, int n_exact, int n_sort, int n_leaves_pad, int n_supers_pad) {
    // (n = 0: one zero record in original order)
    std::vector<Rec4> ex((size_t)std::max(n, 1), Rec4{0.f, 0.f, 0.f, 0.f}), sh = ex;
    for (int i = 0; i < n; i++) {
        const float* s = xyz_radius + 4 * (size_t)i;
        ex[i] = Rec4{s[0], s[1], s[2], s[3]};
        sh[i] = Rec4{s[0], s[1], s[2], ore_host::shadow_radius(s[3])};
    }
    std::vector<Rec4> ss, xs, cl32, lv, sp;
    std::vector<int> order;
    ore_host::build_clusters(ex.data(), sh.data(), n, ss, xs, cl32, &order);
    ore_host::build_hierarchy(ss, n, lv, sp);
    if (ss.empty()) {   // empty scene: one block of padding records
        ss.assign(32, Rec4{3e18f, -1e18f, 2e17f, 0.f});
        xs = ss;
        order.assign(32, 0);
    }
    if ((int)ex.size() != n_exact || (int)ss.size() != n_sort || (int)lv.size() != n_leaves_pad || (int)sp.size() != n_supers_pad)
        return -1;
    std::memcpy(sph_exact, ex.data(), ex.size() * sizeof(Rec4));
    std::memcpy(xsort, xs.data(), xs.size() * sizeof(Rec4));
    std::memcpy(ssort, ss.data(), ss.size() * sizeof(Rec4));
    std::memcpy(sort_index, order.data(), order.size() * sizeof(int));
    if (!lv.empty()) std::memcpy(leaves, lv.data(), lv.size() * sizeof(Rec4));
    if (!sp.empty()) std::memcpy(supers, sp.data(), sp.size() * sizeof(Rec4));
    return 0;
}
