// ore_scene_build.h - the sphere hierarchy built on the device (ore_scene_build.cu), enqueued on a stream.
//
// Input: n records (cx, cy, cz, radius member) in device memory.  Output: the scene arrays of ore_capi.cu - the
// records in original order, both sorted arrays, the permutation, the leaf / super-cluster balls and, for a large scene,
// the hyper-cluster balls - bit-identical to
// what the host builder of ore_clusters.h gives for the same values (DESIGN.md "Device build of the sphere hierarchy").
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

struct SceneBuildArgs {
    const float4* src;     // n input records; may be sph_exact itself (then it is not copied)
    int n;
    float4* sph_exact;     // max(n, 1) records, original order (n = 0: one zero record)
    float4* sph_xsort;     // n_sort exact records, sorted (padding repeats the last sorted sphere)
    float4* sph_sort;      // n_sort shadow records (cx, cy, cz, R'), sorted
    int* sort_index;       // n_sort: sorted position -> original index
    float4* leaf_sph;      // n_leaves_pad balls (padding: radius -1)
    float4* super_sph;     // n_supers_pad balls (padding: radius -1)
    int n_sort, n_leaves, n_leaves_pad, n_supers, n_supers_pad;
    float4* hyper_sph;     // n_hypers_pad balls over 32 supers each (padding: radius -1); n_hypers_pad = 0: not built
    int n_hypers, n_hypers_pad;
    // work space, all sized by the caller for at least n items
    uint32_t* keys_in;
    uint32_t* keys_out;
    int* vals_in;
    int* vals_out;
    uint32_t* bbox;        // 6 words
    void* sort_tmp;
    size_t sort_tmp_bytes;
};

// bytes of sort work space for n items (a host-side query; launches nothing)
cudaError_t ore_scene_sort_bytes(int n, size_t* bytes);
// enqueues the whole build on `stream`; never allocates and never blocks the host
cudaError_t ore_scene_build(const SceneBuildArgs& a, cudaStream_t stream);
