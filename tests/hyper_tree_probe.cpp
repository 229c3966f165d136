// Test-only C wrapper: the host builder of csrc/ore_clusters.h down to the hyper-cluster level of a large scene - the
// sorted shadow records, the super balls and the hyper balls exactly as the device holds them after ore_set_spheres /
// ore_set_spheres_device of a large scene (tests/test_hyper_clusters_cpu.py checks containment,
// tests/test_large_scenes_gpu.py compares the device's hyper balls byte for byte).
#include "ore_clusters.h"

#include <cstring>

using ore_host::Rec4;

// n >= 1 records; lengths n_sort, n_supers_pad, n_hypers_pad (include/ore_render.h, ore_debug_sphere_tree); -1 on a
// mismatch
extern "C" int ore_probe_hyper_tree(const float* xyz_radius, int n, float* ssort, float* supers, float* hypers, int n_sort,
                                    int n_supers_pad, int n_hypers_pad) {
    if (n < 1) return -1;
    std::vector<Rec4> ex((size_t)n), sh((size_t)n);
    for (int i = 0; i < n; i++) {
        const float* s = xyz_radius + 4 * (size_t)i;
        ex[i] = Rec4{s[0], s[1], s[2], s[3]};
        sh[i] = Rec4{s[0], s[1], s[2], ore_host::shadow_radius(s[3])};
    }
    std::vector<Rec4> ss, xs, cl32, lv, sp, hp;
    ore_host::build_clusters(ex.data(), sh.data(), n, ss, xs, cl32);
    ore_host::build_hierarchy(ss, n, lv, sp);
    const int n_sup = (int)(((size_t)n + 255) / 256);
    ore_host::build_hypers(sp, n_sup, hp);
    if ((int)ss.size() != n_sort || (int)sp.size() != n_supers_pad || (int)hp.size() != n_hypers_pad) return -1;
    std::memcpy(ssort, ss.data(), ss.size() * sizeof(Rec4));
    std::memcpy(supers, sp.data(), sp.size() * sizeof(Rec4));
    std::memcpy(hypers, hp.data(), hp.size() * sizeof(Rec4));
    return 0;
}
