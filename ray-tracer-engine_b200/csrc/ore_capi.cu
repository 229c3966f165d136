// ore_capi.cu - C ABI (include/ore_render.h) over the sm_100a render kernels.
//
// Replaces the host half of the reference's kernel.cu for this path: the global scene
// set-up of onStart() (kernel.cu:1704-1714), object::sphereAllocMem (:1208-1212) and the
// per-frame body of update() (:1762-1792).  Where the reference allocates and frees
// managed memory every frame, the context keeps persistent SoA device buffers, a pinned
// host staging buffer for uploads / read-back and its own stream.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo --fmad=false -shared
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <algorithm>
#include <utility>
#include <vector>

#include "../../include/ore_render.h"
#include "ore_clusters.h"
#include "ore_kernels.cuh"
#include "ore_mesh_build.h"
#include "ore_mesh_refit.h"
#include "ore_scene_build.h"

using namespace ore;

namespace {   // (internal linkage: nothing here joins the library's exported symbols)

// Device memory (cudaMalloc) or pinned host memory (cudaMallocHost), as the allocator of a Buf.  slack: the capacity a
// growing buffer takes for n items, so that reallocations stay rare.
struct DeviceMem {
    static cudaError_t alloc(void** p, size_t bytes) { return cudaMalloc(p, bytes); }
    static cudaError_t free(void* p) { return cudaFree(p); }
    static size_t slack(size_t n) { return n + n / 8 + 64; }
};
struct PinnedMem {
    static cudaError_t alloc(void** p, size_t bytes) { return cudaMallocHost(p, bytes); }
    static cudaError_t free(void* p) { return cudaFreeHost(p); }
    static size_t slack(size_t n) { return n + n / 4 + 4096; }
};

// A buffer the context owns: the pointer and its capacity in items, freed with the buffer.  Growing never keeps the
// contents; the caller has waited for whatever may still use the old buffer.
template <typename T, typename Mem = DeviceMem>
class Buf {
public:
    Buf() = default;
    Buf(const Buf&) = delete;
    Buf& operator=(const Buf&) = delete;
    ~Buf() { release(); }
    operator T*() const { return p_; }
    size_t cap() const { return cap_; }
    bool fits(size_t n) const { return p_ && n <= cap_; }
    // exactly n items
    cudaError_t alloc(size_t n) {
        if (cudaError_t e = release()) return e;
        const cudaError_t e = Mem::alloc((void**)&p_, n * sizeof(T));
        if (e == cudaSuccess) cap_ = n;
        else p_ = nullptr;
        return e;
    }
    // at least n items: unchanged when they fit, else the allocator's slack
    cudaError_t reserve(size_t n) { return fits(n) ? cudaSuccess : alloc(Mem::slack(n)); }
    cudaError_t release() {
        const cudaError_t e = p_ ? Mem::free(p_) : cudaSuccess;
        p_ = nullptr;
        cap_ = 0;
        return e;
    }

private:
    T* p_ = nullptr;
    size_t cap_ = 0;
};
template <typename T>
using DevBuf = Buf<T, DeviceMem>;

// A stream, event or graph the context (or a scope) owns, destroyed with it.  A caller's stream is never owned.
template <typename H, cudaError_t (*Destroy)(H)>
class Handle {
public:
    Handle() = default;
    Handle(const Handle&) = delete;
    Handle& operator=(const Handle&) = delete;
    ~Handle() { reset(); }
    operator H() const { return h_; }
    cudaError_t reset() {
        const cudaError_t e = h_ ? Destroy(h_) : cudaSuccess;
        h_ = nullptr;
        return e;
    }
    // where a create call writes the new handle (the one held before is destroyed)
    H* put() {
        reset();
        return &h_;
    }

private:
    H h_ = nullptr;
};
using Stream = Handle<cudaStream_t, cudaStreamDestroy>;
using Event = Handle<cudaEvent_t, cudaEventDestroy>;
using Graph = Handle<cudaGraph_t, cudaGraphDestroy>;
using GraphExec = Handle<cudaGraphExec_t, cudaGraphExecDestroy>;

// The last X, if any: an event and whether it has been recorded.  Waiting for a marker never recorded (or forgotten)
// does nothing.
class Marker {
public:
    cudaEvent_t* put() { return ev_.put(); }
    cudaError_t record(cudaStream_t s) {
        const cudaError_t e = cudaEventRecord(ev_, s);
        if (e == cudaSuccess) recorded_ = true;
        return e;
    }
    cudaError_t stream_wait(cudaStream_t s) const { return recorded_ ? cudaStreamWaitEvent(s, ev_, 0) : cudaSuccess; }
    cudaError_t host_wait() const { return recorded_ ? cudaEventSynchronize(ev_) : cudaSuccess; }
    void forget() { recorded_ = false; }
    bool recorded() const { return recorded_; }
    cudaEvent_t event() const { return ev_; }

private:
    Event ev_;
    bool recorded_ = false;
};

}  // namespace

// Scenes from this many spheres on take the large-scene path: the primary kernel's shared-memory copy of the leaf and
// super-cluster records, (n_leaves_pad + n_supers_pad) x 16 bytes, would pass 200 KB at 99 073 spheres.
static constexpr int LARGE_SCENE_MIN_SPHERES = 99073;
// The largest scene a render accepts: the per-frame sphere records (prim_sorted, cone_sorted: MAX_BATCH frames of 16 bytes
// per sphere each) come to 4 GiB there, and the hyper-cluster records of a frame to 32 KB of shared memory.
static constexpr int MAX_RENDER_SPHERES = 1 << 24;

struct ore_context {
    // (frees every buffer, stream, event and graph below; not an export of the library)
    __attribute__((visibility("hidden"))) ~ore_context() = default;
    int device = 0;
    int sm_count = 0;
    Stream stream;
    Stream copy_stream;
    Event ev_rendered[2], ev_copied[2];
    // device framebuffers of the pipelined presentation: two sets (one being copied out while the other is rendered)
    // of `async_k` frames of `async_px` pixels each, one allocation
    DevBuf<uint32_t> async_pool;
    size_t async_px = 0;
    int async_k = 0;
    unsigned long long async_batches = 0;
    // kernel timing (ore_get_kernel_ms): ev[0..3] before each step of launch_frame, ev_end after the last (timed frames)
    Event ev[4];
    Marker ev_end;
    std::string err;

    // pinned staging (uploads and read-back)
    Buf<char, PinnedMem> pinned;

    // scene (structure of arrays on the device)
    int n_spheres = 0;
    DevBuf<float4> sph_exact;   // cx,cy,cz,radius member in ORIGINAL order (hit attributes by hit id)
    // the spheres in Morton order with two levels of bounding balls over them (ore_clusters.h)
    DevBuf<float4> sph_xsort;   // exact records, sorted
    DevBuf<float4> sph_sort;    // shadow records cx,cy,cz,R', sorted
    DevBuf<int> sort_index;     // sorted position -> original index
    DevBuf<float4> leaf_sph;    // ball of spheres [8j, 8j+8)
    DevBuf<float4> super_sph;   // ball of leaves [32k, 32k+32)
    // per-frame (camera-space) records of the primary kernel, one set per frame of a batch
    DevBuf<float4> prim_sorted;
    DevBuf<float4> cone_sorted;
    DevBuf<float4> leaf_cone;
    DevBuf<float4> super_cone;
    int n_sort = 0, n_leaves = 0, n_leaves_pad = 0, n_supers = 0, n_supers_pad = 0;
    // large scenes (n >= large_min) only: a fourth level of hyper-cluster balls over 32 supers each, and their per-frame
    // records; the render then runs the LARGE kernel instantiations.  n_hypers_pad = 0: the scene has no hyper level.
    DevBuf<float4> hyper_sph;
    DevBuf<float4> hyper_cone;
    int n_hypers = 0, n_hypers_pad = 0;
    int large_min = LARGE_SCENE_MIN_SPHERES;   // env ORE_LARGE_SCENE_MIN_SPHERES (tests: the large path on small scenes)
    // work space of the device build of the hierarchy (ore_scene_build.cu), sized with the scene buffers
    DevBuf<uint32_t> keys_in;
    DevBuf<uint32_t> keys_out;
    DevBuf<int> vals_in;
    DevBuf<int> vals_out;
    DevBuf<uint32_t> bbox;
    DevBuf<char> sort_tmp;
    int n_lights = 0;
    LightP lights[MAX_LIGHTS];
    DevBuf<float> tex[3];
    int tex_w = 0, tex_h = 0;
    bool tex_finite = false;   // every texel of the object texture is finite (checked at upload; FrameParams::skip_dark)
    DevBuf<float> sky[3];
    int sky_w = 0, sky_h = 0;
    float sky_radius = 0.f;
    DevBuf<float4> cubes;    // 3 float4 per cube: bounds[0], bounds[1], orgin
    DevBuf<float4> planes;   // 2 float4 per plane: orgin, normal
    int n_cubes = 0, n_planes = 0;
    // the mesh buffers, sized for the largest mesh uploaded by either setter since the mesh was last removed
    DevBuf<float> tris;         // 27 floats per triangle
    DevBuf<float4> boxes;       // 2 float4 per leaf box
    DevBuf<float4> box_sph;     // bounding sphere per leaf box (cone filters)
    DevBuf<float4> box_cone;    // per-frame tile-cone record per leaf box
    DevBuf<int> box_offsets;
    DevBuf<int> box_indices;
    // n_boxes: the leaf capacity (stride of box_cone, grid sizes); the live leaf count is *mesh_live on the device (the
    // render kernels' leaf loops end there; leaves past it list no triangles)
    int n_tris = 0, n_boxes = 0, mesh_has_normals = 0, mesh_n_idx = 0;
    DevBuf<int> mesh_live;
    DevBuf<char> mesh_work;   // the device build's work space
    // the device build's launch sequence (about 65 launches, all sized from the capacity; the triangle count is read on
    // the device) captured once per buffer set and replayed on the caller's stream: enqueuing it launch by launch costs
    // the host several hundred microseconds
    GraphExec mesh_graph;
    Stream mesh_capture;

    // per-frame buffers
    DevBuf<float> dx_tab;
    DevBuf<float> dy_tab;
    DevBuf<uint32_t> hit_list;  // compact hit records (pixel, id, t), one per hit pixel
    DevBuf<int32_t> hit_ids;
    DevBuf<float> hit_ts;
    DevBuf<uint32_t> pixels;    // the context's own framebuffer (ore_render)
    DevBuf<int32_t> hit_id_map;  // per-pixel id / t maps: only built by ore_get_hits
    DevBuf<float> hit_t_map;
    DevBuf<unsigned long long> counters;
    // band DMA (ORE_FLAG_BAND_DMA): packed local rows of the primary kernel + the stream / events of their copy
    DevBuf<uint32_t> band_buf;
    Stream band_stream;
    Event ev_band_go;
    Marker ev_band_done;
    DevBuf<float> stage;  // staging buffer between the two kernels of the default shadow pass (ore_stage_plan.h)
    size_t stage_blocks_override = 0;  // test hook (env ORE_STAGE_BLOCKS at ore_create): staging capacity in 32-item blocks
    size_t stage_max_items = (size_t)8 << 20;  // env ORE_STAGE_MAX_ITEMS: upper bound of the staging buffer in hit pixels
    bool no_memops = false;            // test hook (env ORE_NO_STREAM_MEMOPS=1): flags through the one-thread kernels
    std::string dbg_cycles_path;       // tools hook (env ORE_DEBUG_BLOCK_CYCLES=file): per-block SM clocks of the shadow pass
    DevBuf<uint32_t> dbg_cycles;       // [2][cap / 2]
    // hit count of this context's previous frame, copied to pinned memory at the end of every frame and read
    // WITHOUT synchronisation by the next one: only a hint for how many staged chunk pairs to launch - whatever
    // lies beyond them is swept by one catch-all fused launch, so any value (stale, zero, mid-copy) is safe
    Buf<unsigned long long, PinnedMem> hits_hint;
    bool hits_hint_set = false;
    FrameParams last_prm;              // the last frame's parameters (ore_get_hits expands its hit records)
    bool last_prm_valid = false;

    // occupancy-sized grids, computed once per (kernel, dynamic shared memory, block size)
    struct GridEntry {
        const void* fn;
        size_t smem;
        int threads, grid;
    };
    std::vector<GridEntry> grid_cache;
    // end of the last render on whichever stream it ran (scene setters wait for it before touching scene buffers)
    Marker ev_done;
    // end of the last stream-ordered scene update (ore_set_spheres_device, ore_set_mesh_device,
    // ore_set_mesh_triangles_device) on whichever
    // stream it ran: every render and every host setter enqueued later waits for it on the device
    Marker ev_scene;
    // ordered flag writes (ore_flag_write_after)
    Stream signal_stream;
    Event ev_signal[8];
    unsigned n_signals = 0;

    // last frame
    int last_frames = 1;
    size_t last_px = 0;
    int last_n_spheres = 0;
    uint64_t last_launches = 0;
};

#define ORE_CUDA(ctx, expr)                                                                         \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            char _b[512];                                                                           \
            snprintf(_b, sizeof _b, "CUDA error = %u at %s:%d '%s' (%s)", (unsigned)_e, __FILE__,   \
                     __LINE__, #expr, cudaGetErrorString(_e));                                      \
            (ctx)->err = _b;                                                                        \
            return ORE_ERR_CUDA;                                                                    \
        }                                                                                           \
    } while (0)

static int fail(ore_context* ctx, int code, const char* msg) {
    if (ctx) ctx->err = msg;
    return code;
}

// Replaces the device buffer by n items that fill(T* staging) writes into the pinned staging buffer, and waits for
// the copy.  n == 0 leaves no buffer and does not synchronise.  The caller has waited for the last render.
template <typename T, typename Fill>
static int replace_buffer(ore_context* ctx, DevBuf<T>& buf, size_t n, Fill fill) {
    ORE_CUDA(ctx, buf.release());
    if (n == 0) return ORE_OK;
    ORE_CUDA(ctx, ctx->pinned.reserve(n * sizeof(T)));
    fill((T*)(void*)ctx->pinned);
    ORE_CUDA(ctx, buf.alloc(n));
    ORE_CUDA(ctx, cudaMemcpyAsync(buf, ctx->pinned, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    ORE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ORE_OK;
}

// scene setters: the previous render may still be running on a caller-supplied stream, and a scene update on another
// stream may still be pending (what the setter enqueues next on the render stream follows it)
static int wait_last_render(ore_context* ctx) {
    ORE_CUDA(ctx, ctx->ev_done.host_wait());
    ORE_CUDA(ctx, ctx->ev_scene.stream_wait(ctx->stream));
    return ORE_OK;
}

// Before a buffer that a render may read or a pending stream-ordered update may write is freed or re-allocated: the host
// waits for the last render and the last update to complete.
static int scene_idle(ore_context* ctx) {
    if (int rc = wait_last_render(ctx)) return rc;
    ORE_CUDA(ctx, ctx->ev_scene.host_wait());
    ctx->ev_scene.forget();
    return ORE_OK;
}

// Growth of a buffer a frame reads or writes: an earlier frame may still be running on another stream, so the host waits
// for the last render before the buffer is re-allocated.
template <typename T>
static int frame_reserve(ore_context* ctx, DevBuf<T>& buf, size_t n) {
    if (buf.fits(n)) return ORE_OK;
    if (int rc = wait_last_render(ctx)) return rc;
    ORE_CUDA(ctx, buf.reserve(n));
    return ORE_OK;
}

// A stream-ordered update runs on `stream` (NULL: the render stream) after every render submitted so far and the
// previous update, on whatever streams they ran; the host never waits.  update_end marks its end for every render and
// setter submitted later.
static int update_begin(ore_context* ctx, void* stream, cudaStream_t* st) {
    *st = stream ? (cudaStream_t)stream : ctx->stream;
    ORE_CUDA(ctx, ctx->ev_done.stream_wait(*st));
    ORE_CUDA(ctx, ctx->ev_scene.stream_wait(*st));
    return ORE_OK;
}

static int update_end(ore_context* ctx, cudaStream_t st) {
    ORE_CUDA(ctx, ctx->ev_scene.record(st));
    return ORE_OK;
}

extern "C" int ore_abi_version(void) { return ORE_ABI_VERSION; }

extern "C" const char* ore_last_error(const ore_context* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

extern "C" int ore_create(ore_context** out, int device) {
    if (!out) return ORE_ERR_INVALID;
    *out = nullptr;
    ore_context* ctx = new (std::nothrow) ore_context();
    if (!ctx) return ORE_ERR_NOMEM;
    *out = ctx;  // returned even on failure so the caller can read ore_last_error
    ctx->device = device;
    ORE_CUDA(ctx, cudaSetDevice(device));
    cudaDeviceProp prop;
    ORE_CUDA(ctx, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        char b[160];
        snprintf(b, sizeof b, "device %d is sm_%d%d; this library only carries an sm_100a image (no fallback)", device,
                 prop.major, prop.minor);
        return fail(ctx, ORE_ERR_CUDA, b);
    }
    ctx->sm_count = prop.multiProcessorCount;
    ORE_CUDA(ctx, cudaStreamCreateWithFlags(ctx->stream.put(), cudaStreamNonBlocking));
    ORE_CUDA(ctx, cudaStreamCreateWithFlags(ctx->copy_stream.put(), cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
        ORE_CUDA(ctx, cudaEventCreateWithFlags(ctx->ev_rendered[i].put(), cudaEventDisableTiming));
        ORE_CUDA(ctx, cudaEventCreateWithFlags(ctx->ev_copied[i].put(), cudaEventDisableTiming));
    }
    for (Event& e : ctx->ev) ORE_CUDA(ctx, cudaEventCreate(e.put()));
    ORE_CUDA(ctx, cudaEventCreate(ctx->ev_end.put()));
    ORE_CUDA(ctx, cudaEventCreateWithFlags(ctx->ev_done.put(), cudaEventDisableTiming));
    ORE_CUDA(ctx, cudaEventCreateWithFlags(ctx->ev_scene.put(), cudaEventDisableTiming));
    ORE_CUDA(ctx, ctx->hits_hint.alloc(1));
    *ctx->hits_hint = 0;
    if (const char* e = getenv("ORE_NO_STREAM_MEMOPS")) ctx->no_memops = atoi(e) != 0;
    if (const char* e = getenv("ORE_STAGE_MAX_ITEMS")) {
        const long long v = atoll(e);
        if (v >= 32) ctx->stage_max_items = (size_t)v;
    }
    if (const char* e = getenv("ORE_DEBUG_BLOCK_CYCLES")) ctx->dbg_cycles_path = e;
    if (const char* e = getenv("ORE_STAGE_BLOCKS")) {
        const long v = atol(e);
        if (v > 0) ctx->stage_blocks_override = (size_t)v;
    }
    if (const char* e = getenv("ORE_LARGE_SCENE_MIN_SPHERES")) {   // (only ever lowers the threshold)
        const long v = atol(e);
        if (v >= 1 && v < LARGE_SCENE_MIN_SPHERES) ctx->large_min = (int)v;
    }
    ORE_CUDA(ctx, ctx->counters.alloc(CNT_SLOTS));
    ORE_CUDA(ctx, cudaMemset(ctx->counters, 0, CNT_SLOTS * sizeof(unsigned long long)));
    // kernel.cu:1454,1462-1463: phi = (float)j/10 * 2.f * 3.1415f; cosf(phi), sinf(phi)
    float cphi[10], sphi[10];
    for (int j = 0; j < 10; j++) {
        float phi = (float)j / 10 * 2.f * 3.1415f;
        cphi[j] = cosf(phi);
        sphi[j] = sinf(phi);
    }
    ORE_CUDA(ctx, cudaMemcpyToSymbol(c_cos_phi, cphi, sizeof cphi));
    ORE_CUDA(ctx, cudaMemcpyToSymbol(c_sin_phi, sphi, sizeof sphi));
    float bk[11];
    {
        float b = 0;
        bk[0] = b;
        for (int k = 1; k <= 10; k++) {
            b += 0.1;  // float += double, kernel.cu:1538
            bk[k] = b;
        }
    }
    ORE_CUDA(ctx, cudaMemcpyToSymbol(c_b_of_k, bk, sizeof bk));
    return ORE_OK;
}

extern "C" int ore_destroy(ore_context* ctx) {
    if (!ctx) return ORE_ERR_INVALID;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->dbg_cycles) {
        // tools hook: [2][cap] uint32 of the LAST frame, preceded by cap as one uint64
        cudaDeviceSynchronize();
        std::vector<uint32_t> h(ctx->dbg_cycles.cap());
        if (cudaMemcpy(h.data(), ctx->dbg_cycles, h.size() * 4, cudaMemcpyDeviceToHost) == cudaSuccess) {
            if (FILE* f = fopen(ctx->dbg_cycles_path.c_str(), "wb")) {
                const unsigned long long cap = h.size() / 2;
                fwrite(&cap, 8, 1, f);
                fwrite(h.data(), 4, h.size(), f);
                fclose(f);
            }
        }
    }
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (ctx->signal_stream) cudaStreamSynchronize(ctx->signal_stream);
    if (ctx->band_stream) cudaStreamSynchronize(ctx->band_stream);
    delete ctx;   // (and with it every buffer, stream, event and graph the context owns)
    return ORE_OK;
}

// ---- scene upload -----------------------------------------------------------------------

// Replaces object::sphereAllocMem: the n records go to the device twice - in their original order (hit attributes are
// looked up by hit id) and in the Morton order of their centres, with a bounding ball per leaf of 8 and per
// super-cluster of 32 leaves.  Both the primary kernel (tile cones) and the shadow sweep (beams) descend that
// hierarchy; neither result depends on the order spheres are visited in (nearest hit: candidates are adjudicated by
// (t, original index)).  The hierarchy is built on the device (ore_scene_build.cu) for both setters; the host builder
// of ore_clusters.h is its CPU reference (tests/test_clusters_cpu.py, tests/test_scene_update_gpu.py).

static void scene_sizes(int32_t n, size_t* n_sort, size_t* n_leaf_pad, size_t* n_sup_pad, size_t* n_hyp_pad) {
    const size_t n_clu = ((size_t)n + 31) / 32;
    *n_sort = n > 0 ? n_clu * 32 : 32;   // empty scene: one block of padding records
    const size_t n_leaf = ((size_t)n + ore_host::LEAF_SPHERES - 1) / ore_host::LEAF_SPHERES;
    const size_t n_sup = (n_leaf + ore_host::SUPER_LEAVES - 1) / ore_host::SUPER_LEAVES;
    const size_t n_hyp = (n_sup + ore_host::HYPER_SUPERS - 1) / ore_host::HYPER_SUPERS;
    *n_leaf_pad = (n_leaf + 31) & ~(size_t)31;
    *n_sup_pad = (n_sup + 3) & ~(size_t)3;
    *n_hyp_pad = (n_hyp + 3) & ~(size_t)3;
}

// the scene takes the large-scene path (hyper level, LARGE kernels); decided once per scene by the setters
static bool large_scene(const ore_context* ctx, int32_t n) { return n > 0 && n >= ctx->large_min; }

// Capacity of the scene buffers and of the build's work space for n spheres.  Only growth blocks the host: the old
// buffers may still be read by a render or written by an update on another stream, so both are waited for first.
static int scene_reserve(ore_context* ctx, int32_t n) {
    size_t n_sort, n_leaf_pad, n_sup_pad, n_hyp_pad;
    scene_sizes(n, &n_sort, &n_leaf_pad, &n_sup_pad, &n_hyp_pad);
    const bool large = large_scene(ctx, n);
    size_t tmp_bytes = 0;
    ORE_CUDA(ctx, ore_scene_sort_bytes(n, &tmp_bytes));
    const size_t n_ex = (size_t)std::max(n, 1), nb = MAX_BATCH;   // (camera-space records: one set per frame of a batch)
    // op(buffer, items it needs) over every buffer of the scene, until one returns false
    const auto each = [&](auto&& op) {
        return op(ctx->sph_exact, n_ex) && op(ctx->sph_xsort, n_sort) && op(ctx->sph_sort, n_sort) && op(ctx->sort_index, n_sort) &&
               op(ctx->prim_sorted, n_sort * nb) && op(ctx->cone_sorted, n_sort * nb) && op(ctx->leaf_sph, n_leaf_pad) &&
               op(ctx->leaf_cone, n_leaf_pad * nb) && op(ctx->super_sph, n_sup_pad) && op(ctx->super_cone, n_sup_pad * nb) &&
               op(ctx->keys_in, (size_t)n) && op(ctx->keys_out, (size_t)n) && op(ctx->vals_in, (size_t)n) &&
               op(ctx->vals_out, (size_t)n) && op(ctx->bbox, (size_t)6) &&
               (!large || (op(ctx->hyper_sph, n_hyp_pad) && op(ctx->hyper_cone, n_hyp_pad * nb)));
    };
    if (each([](auto& buf, size_t k) { return buf.fits(k); }) && ctx->sort_tmp.fits(tmp_bytes)) return ORE_OK;
    if (int rc = scene_idle(ctx)) return rc;
    cudaError_t e = cudaSuccess;
    each([&](auto& buf, size_t k) { return (e = buf.reserve(k)) == cudaSuccess; });
    ORE_CUDA(ctx, e);
    // sort work space for the whole key capacity, so that any n up to it needs no more
    ORE_CUDA(ctx, ore_scene_sort_bytes((int)std::min(ctx->keys_in.cap(), (size_t)INT32_MAX), &tmp_bytes));
    if (!ctx->sort_tmp.fits(tmp_bytes)) ORE_CUDA(ctx, ctx->sort_tmp.alloc(std::max(tmp_bytes, (size_t)256)));
    return ORE_OK;
}

// Enqueues the device build of the hierarchy over the n records at src (device memory; may be sph_exact itself) on
// `stream` and sets the scene's counts.  Capacity comes from scene_reserve.
static int scene_enqueue(ore_context* ctx, const float4* src, int32_t n, cudaStream_t stream) {
    size_t n_sort, n_leaf_pad, n_sup_pad, n_hyp_pad;
    scene_sizes(n, &n_sort, &n_leaf_pad, &n_sup_pad, &n_hyp_pad);
    const bool large = large_scene(ctx, n);
    SceneBuildArgs a;
    a.src = src;
    a.n = n;
    a.sph_exact = ctx->sph_exact;
    a.sph_xsort = ctx->sph_xsort;
    a.sph_sort = ctx->sph_sort;
    a.sort_index = ctx->sort_index;
    a.leaf_sph = ctx->leaf_sph;
    a.super_sph = ctx->super_sph;
    a.n_sort = (int)n_sort;
    a.n_leaves = (n + ore_host::LEAF_SPHERES - 1) / ore_host::LEAF_SPHERES;
    a.n_leaves_pad = (int)n_leaf_pad;
    a.n_supers = (a.n_leaves + ore_host::SUPER_LEAVES - 1) / ore_host::SUPER_LEAVES;
    a.n_supers_pad = (int)n_sup_pad;
    a.hyper_sph = large ? (float4*)ctx->hyper_sph : nullptr;
    a.n_hypers = large ? (a.n_supers + ore_host::HYPER_SUPERS - 1) / ore_host::HYPER_SUPERS : 0;
    a.n_hypers_pad = large ? (int)n_hyp_pad : 0;
    a.keys_in = ctx->keys_in;
    a.keys_out = ctx->keys_out;
    a.vals_in = ctx->vals_in;
    a.vals_out = ctx->vals_out;
    a.bbox = ctx->bbox;
    a.sort_tmp = ctx->sort_tmp;
    a.sort_tmp_bytes = ctx->sort_tmp.cap();
    ORE_CUDA(ctx, ore_scene_build(a, stream));
    ctx->n_spheres = n;
    ctx->n_sort = a.n_sort;
    ctx->n_leaves = a.n_leaves;
    ctx->n_leaves_pad = a.n_leaves_pad;
    ctx->n_supers = a.n_supers;
    ctx->n_supers_pad = a.n_supers_pad;
    ctx->n_hypers = a.n_hypers;
    ctx->n_hypers_pad = a.n_hypers_pad;
    return ORE_OK;
}

// The synchronous setters: the raw records through pinned staging into sph_exact, the device build behind them on the
// render stream, then a synchronisation.
static int upload_spheres(ore_context* ctx, const float* src, size_t stride_floats, size_t first, int32_t n) {
    if (!ctx || n < 0 || (n > 0 && !src)) return fail(ctx, ORE_ERR_INVALID, "ore_set_spheres: bad arguments");
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc;
    if ((rc = scene_idle(ctx))) return rc;
    if ((rc = scene_reserve(ctx, n))) return rc;
    if (n > 0) {
        ORE_CUDA(ctx, ctx->pinned.reserve((size_t)n * sizeof(float4)));
        float4* h = (float4*)(void*)ctx->pinned;
        for (int i = 0; i < n; i++) {
            const float* s = src + (size_t)i * stride_floats + first;
            h[i] = make_float4(s[0], s[1], s[2], s[3]);
        }
        ORE_CUDA(ctx, cudaMemcpyAsync(ctx->sph_exact, h, (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, ctx->stream));
    }
    if ((rc = scene_enqueue(ctx, ctx->sph_exact, n, ctx->stream))) return rc;
    ORE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ORE_OK;
}

extern "C" int ore_set_spheres(ore_context* ctx, const float* xyz_radius, int32_t n) {
    return upload_spheres(ctx, xyz_radius, 4, 0, n);
}

extern "C" int ore_set_spheres_aos32(ore_context* ctx, const void* records, int32_t n) {
    // reference record: vptr@0, orgin@8 (3 floats), reflective@20, radius@24, pad@28 (kernel.cu:265-358)
    // => floats 2,3,4 = centre; float 6 = radius.  Repack to x,y,z,radius through a temporary.
    if (!ctx || n < 0 || (n > 0 && !records)) return fail(ctx, ORE_ERR_INVALID, "ore_set_spheres_aos32: bad arguments");
    std::vector<float> tmp((size_t)n * 4);
    const float* f = (const float*)records;
    for (int i = 0; i < n; i++) {
        tmp[4 * (size_t)i + 0] = f[8 * (size_t)i + 2];
        tmp[4 * (size_t)i + 1] = f[8 * (size_t)i + 3];
        tmp[4 * (size_t)i + 2] = f[8 * (size_t)i + 4];
        tmp[4 * (size_t)i + 3] = f[8 * (size_t)i + 6];
    }
    return upload_spheres(ctx, tmp.data(), 4, 0, n);
}

// the records of a stream-ordered update: device (or managed) memory of the context's GPU - not host, pinned or another
// GPU's memory
static bool on_context_gpu(ore_context* ctx, const void* p) {
    cudaPointerAttributes at;
    const cudaError_t e = cudaPointerGetAttributes(&at, p);
    (void)cudaGetLastError();
    return e == cudaSuccess && (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) && at.device == ctx->device;
}

// The records of a stream-ordered update: on the context's GPU (above) and `align`-byte aligned.  `what` names the setter
// and its records for the message ("ore_set_spheres_device: the records").
static int device_records(ore_context* ctx, const void* p, unsigned align, const char* what) {
    char b[200];
    if (!p || ((uintptr_t)p & (align - 1))) {
        snprintf(b, sizeof b, "%s must be %u-byte aligned", what, align);
        return fail(ctx, ORE_ERR_INVALID, b);
    }
    if (!on_context_gpu(ctx, p)) {
        snprintf(b, sizeof b, "%s must be device memory of the context's GPU", what);
        return fail(ctx, ORE_ERR_INVALID, b);
    }
    return ORE_OK;
}

extern "C" int ore_set_spheres_device(ore_context* ctx, const float* xyz_radius_dev, int32_t n, void* stream) {
    if (!ctx) return ORE_ERR_INVALID;
    if (n < 0) return fail(ctx, ORE_ERR_INVALID, "ore_set_spheres_device: n < 0");
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc;
    if (n > 0 && (rc = device_records(ctx, xyz_radius_dev, 16, "ore_set_spheres_device: the records"))) return rc;
    if ((rc = scene_reserve(ctx, n))) return rc;   // blocks only when the scene buffers grow
    cudaStream_t st;
    if ((rc = update_begin(ctx, stream, &st))) return rc;
    if ((rc = scene_enqueue(ctx, (const float4*)xyz_radius_dev, n, st))) return rc;
    return update_end(ctx, st);
}

extern "C" int ore_set_cubes(ore_context* ctx, const float* c1_c2, int32_t n) {
    if (!ctx || n < 0 || (n > 0 && !c1_c2)) return fail(ctx, ORE_ERR_INVALID, "ore_set_cubes: bad arguments");
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    if (int rcw = wait_last_render(ctx)) return rcw;
    ctx->n_cubes = 0;
    int rc = replace_buffer(ctx, ctx->cubes, (size_t)n * 3, [&](float4* h) {
        for (int i = 0; i < n; i++) {
            const float* c = c1_c2 + 6 * (size_t)i;
            h[3 * i + 0] = make_float4(c[0], c[1], c[2], 0.f);  // bounds[0] = c1, kernel.cu:393
            h[3 * i + 1] = make_float4(c[3], c[4], c[5], 0.f);  // bounds[1] = c2
            // orgin = divide(add(c1, c2), 2), kernel.cu:395 (float add, float divide)
            // .w = radius of a bounding sphere about orgin (half diagonal + margins) for the light-cone filter
            const double dx = (double)c[3] - c[0], dy = (double)c[4] - c[1], dz = (double)c[5] - c[2];
            const double rad = 0.5 * sqrt(dx * dx + dy * dy + dz * dz);
            const double mag = fabs((double)c[0]) + fabs((double)c[1]) + fabs((double)c[2]) + fabs((double)c[3]) +
                               fabs((double)c[4]) + fabs((double)c[5]);
            h[3 * i + 2] = make_float4((c[0] + c[3]) / 2, (c[1] + c[4]) / 2, (c[2] + c[5]) / 2,
                                       (float)(rad * 1.001 + 1e-5 * mag + 1e-6));
        }
    });
    if (rc) return rc;
    ctx->n_cubes = n;
    return ORE_OK;
}

extern "C" int ore_set_planes(ore_context* ctx, const float* pos_normal, int32_t n) {
    if (!ctx || n < 0 || (n > 0 && !pos_normal)) return fail(ctx, ORE_ERR_INVALID, "ore_set_planes: bad arguments");
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    if (int rcw = wait_last_render(ctx)) return rcw;
    ctx->n_planes = 0;
    int rc = replace_buffer(ctx, ctx->planes, (size_t)n * 2, [&](float4* h) {
        for (int i = 0; i < n; i++) {
            const float* c = pos_normal + 6 * (size_t)i;
            h[2 * i + 0] = make_float4(c[0], c[1], c[2], 0.f);
            h[2 * i + 1] = make_float4(c[3], c[4], c[5], 0.f);
        }
    });
    if (rc) return rc;
    ctx->n_planes = n;
    return ORE_OK;
}

// Frees the mesh buffers and, unless tri_cap is 0, allocates them for tri_cap triangles, box_cap leaves and idx_cap
// (>= 1) listed indices, with the device build's work space for tri_cap triangles (tri_cap <= INT32_MAX / TRI_FLOATS: the
// setters check).  The caller has waited for every render and update that may use them.
static int mesh_alloc(ore_context* ctx, size_t tri_cap, size_t box_cap, size_t idx_cap) {
    ORE_CUDA(ctx, ctx->mesh_graph.reset());   // (it holds the old buffers' addresses)
    for (cudaError_t e : {ctx->tris.release(), ctx->boxes.release(), ctx->box_offsets.release(), ctx->box_indices.release(),
                          ctx->box_sph.release(), ctx->box_cone.release(), ctx->mesh_work.release()})
        ORE_CUDA(ctx, e);
    ctx->n_tris = ctx->n_boxes = ctx->mesh_has_normals = ctx->mesh_n_idx = 0;
    if (tri_cap == 0) return ORE_OK;
    size_t work = 0;
    ORE_CUDA(ctx, ore_mesh_build_bytes((int)tri_cap, &work));
    if (!ctx->mesh_live) ORE_CUDA(ctx, ctx->mesh_live.alloc(1));
    ORE_CUDA(ctx, ctx->tris.alloc(tri_cap * ore_host::TRI_FLOATS));
    ORE_CUDA(ctx, ctx->boxes.alloc(box_cap * 2));
    ORE_CUDA(ctx, ctx->box_offsets.alloc(box_cap + 1));
    ORE_CUDA(ctx, ctx->box_indices.alloc(idx_cap));
    ORE_CUDA(ctx, ctx->box_sph.alloc(box_cap));
    ORE_CUDA(ctx, ctx->box_cone.alloc(box_cap * MAX_BATCH));
    ORE_CUDA(ctx, ctx->mesh_work.alloc(work));
    return ORE_OK;
}

// the mesh buffers hold n_tris triangles, n_boxes leaves and n_idx listed indices
static bool mesh_fits(const ore_context* ctx, size_t n_tris, size_t n_boxes, size_t n_idx) {
    return ctx->tris.fits(n_tris * ore_host::TRI_FLOATS) && ctx->boxes.fits(n_boxes * 2) && ctx->box_offsets.fits(n_boxes + 1) &&
           ctx->box_indices.fits(n_idx) && ctx->box_sph.fits(n_boxes) && ctx->box_cone.fits(n_boxes * MAX_BATCH);
}

// capacity of the mesh buffers in triangles (0 without a mesh)
static size_t mesh_tri_cap(const ore_context* ctx) { return ctx->tris.cap() / ore_host::TRI_FLOATS; }

extern "C" int ore_set_mesh(ore_context* ctx, const float* tris27, int32_t n_tris, int32_t has_normals,
                            const float* box_bounds6, const int32_t* box_offsets, const int32_t* box_indices,
                            int32_t n_boxes) {
    if (!ctx || n_tris < 0 || n_boxes < 0) return fail(ctx, ORE_ERR_INVALID, "ore_set_mesh: bad arguments");
    const bool remove = n_tris == 0 || n_boxes == 0;
    int n_idx = 0;
    if (!remove) {
        if (!tris27 || !box_bounds6 || !box_offsets || !box_indices) return fail(ctx, ORE_ERR_INVALID, "ore_set_mesh: null array");
        if ((size_t)n_tris > (size_t)INT32_MAX / ore_host::TRI_FLOATS) return fail(ctx, ORE_ERR_INVALID, "ore_set_mesh: too many triangles");
        n_idx = box_offsets[n_boxes];
        if (box_offsets[0] != 0 || n_idx < 0) return fail(ctx, ORE_ERR_INVALID, "ore_set_mesh: bad offsets");
        for (int j = 0; j < n_boxes; j++)
            if (box_offsets[j + 1] < box_offsets[j]) return fail(ctx, ORE_ERR_INVALID, "ore_set_mesh: offsets must ascend");
        for (int k = 0; k < n_idx; k++)
            if (box_indices[k] < 0 || box_indices[k] >= n_tris) return fail(ctx, ORE_ERR_INVALID, "ore_set_mesh: triangle index out of range");
    }
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc;
    // a pending ore_set_mesh_device or ore_set_mesh_triangles_device still writes the mesh buffers and the build's
    // work space
    if ((rc = scene_idle(ctx))) return rc;
    if (remove) return mesh_alloc(ctx, 0, 0, 0);
    // the buffers are re-allocated at least at the capacity the device setters reached, so that they keep not blocking
    const size_t tri_cap = std::max(mesh_tri_cap(ctx), (size_t)n_tris);
    const size_t box_cap = std::max({ctx->box_sph.cap(), (size_t)n_boxes, (size_t)ore_mesh_leaf_capacity((int)tri_cap)});
    const size_t idx_cap = std::max({ctx->box_indices.cap(), (size_t)n_idx, tri_cap});
    if ((rc = mesh_alloc(ctx, tri_cap, box_cap, idx_cap))) return rc;
    const size_t tb = (size_t)n_tris * 27 * sizeof(float), bb = (size_t)n_boxes * 2 * sizeof(float4);
    const size_t ob = (size_t)(n_boxes + 1) * sizeof(int), ib = (size_t)(n_idx > 0 ? n_idx : 1) * sizeof(int);
    // pinned staging layout: the float4 section first (16-byte aligned: bb is a multiple of 16 and the pinned base is
    // page aligned), then the 4-byte-aligned sections, the live leaf count last
    const size_t off_b = 0, off_t = bb, off_o = off_t + tb, off_i = off_o + ob, off_l = off_i + ib;
    ORE_CUDA(ctx, ctx->pinned.reserve(off_l + sizeof(int)));
    char* h = ctx->pinned;
    float4* hb = (float4*)(h + off_b);
    memcpy(h + off_t, tris27, tb);
    for (int j = 0; j < n_boxes; j++) {
        const float* b = box_bounds6 + 6 * (size_t)j;
        hb[2 * j] = make_float4(b[0], b[1], b[2], 0.f);
        hb[2 * j + 1] = make_float4(b[3], b[4], b[5], 0.f);
    }
    memcpy(h + off_o, box_offsets, ob);
    memcpy(h + off_i, box_indices, (size_t)n_idx * sizeof(int));
    memcpy(h + off_l, &n_boxes, sizeof(int));
    ORE_CUDA(ctx, cudaMemcpyAsync(ctx->tris, h + off_t, tb, cudaMemcpyHostToDevice, ctx->stream));
    ORE_CUDA(ctx, cudaMemcpyAsync(ctx->boxes, hb, bb, cudaMemcpyHostToDevice, ctx->stream));
    ORE_CUDA(ctx, cudaMemcpyAsync(ctx->box_offsets, h + off_o, ob, cudaMemcpyHostToDevice, ctx->stream));
    ORE_CUDA(ctx, cudaMemcpyAsync(ctx->box_indices, h + off_i, ib, cudaMemcpyHostToDevice, ctx->stream));
    ORE_CUDA(ctx, cudaMemcpyAsync(ctx->mesh_live, h + off_l, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    // the leaf balls by the kernel the device update runs too (ore_mesh_refit.cu): one code path for box_sph
    ORE_CUDA(ctx, ore_mesh_balls(ctx->boxes, ctx->box_sph, n_boxes, ctx->stream));
    ORE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->n_tris = n_tris;
    ctx->n_boxes = n_boxes;
    ctx->mesh_n_idx = n_idx;
    ctx->mesh_has_normals = has_normals ? 1 : 0;
    return ORE_OK;
}

extern "C" int ore_set_mesh_device(ore_context* ctx, const float* tris27_dev, int32_t n_tris, int32_t has_normals, void* stream) {
    if (!ctx) return ORE_ERR_INVALID;
    if (n_tris < 1)
        return fail(ctx, ORE_ERR_INVALID, "ore_set_mesh_device: n_tris must be >= 1 (remove the mesh with ore_set_mesh(ctx, NULL, 0, ...))");
    if ((size_t)n_tris > (size_t)INT32_MAX / ore_host::TRI_FLOATS) return fail(ctx, ORE_ERR_INVALID, "ore_set_mesh_device: too many triangles");
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc;
    if ((rc = device_records(ctx, tris27_dev, 4, "ore_set_mesh_device: the triangles"))) return rc;
    const int L = ore_mesh_leaf_capacity(n_tris);
    if (!mesh_fits(ctx, n_tris, L, n_tris)) {
        // growth: the old buffers may still be read by a render or written by an update on another stream
        if ((rc = scene_idle(ctx))) return rc;
        const size_t tri_cap = std::max(mesh_tri_cap(ctx), (size_t)n_tris);
        if ((rc = mesh_alloc(ctx, tri_cap, std::max(ctx->box_sph.cap(), (size_t)L), std::max(ctx->box_indices.cap(), tri_cap)))) return rc;
    }
    cudaStream_t st;
    if ((rc = update_begin(ctx, stream, &st))) return rc;
    ORE_CUDA(ctx, cudaMemcpyAsync(ctx->tris, tris27_dev, (size_t)n_tris * ore_host::TRI_FLOATS * sizeof(float),
                                  cudaMemcpyDeviceToDevice, st));
    MeshBuildArgs a;
    a.tris = ctx->tris;
    a.cap_tris = (int)mesh_tri_cap(ctx);
    a.box_offsets = ctx->box_offsets;
    a.box_indices = ctx->box_indices;
    a.boxes = ctx->boxes;
    a.box_sph = ctx->box_sph;
    a.n_live = ctx->mesh_live;
    a.work = ctx->mesh_work;
    a.work_bytes = ctx->mesh_work.cap();
    if (!ctx->mesh_graph) {   // (mesh_alloc drops it with the buffers it holds)
        if (!ctx->mesh_capture) ORE_CUDA(ctx, cudaStreamCreateWithFlags(ctx->mesh_capture.put(), cudaStreamNonBlocking));
        Graph g;
        ORE_CUDA(ctx, cudaStreamBeginCapture(ctx->mesh_capture, cudaStreamCaptureModeThreadLocal));
        const cudaError_t eb = ore_mesh_build(a, ctx->mesh_capture);
        const cudaError_t ec = cudaStreamEndCapture(ctx->mesh_capture, g.put());
        ORE_CUDA(ctx, eb != cudaSuccess ? eb : ec);
        ORE_CUDA(ctx, cudaGraphInstantiate(ctx->mesh_graph.put(), g, 0));
    }
    ORE_CUDA(ctx, ore_mesh_build_count(a, n_tris, st));
    ORE_CUDA(ctx, cudaGraphLaunch(ctx->mesh_graph, st));
    if ((rc = update_end(ctx, st))) return rc;
    ctx->n_tris = n_tris;
    ctx->n_boxes = L;
    ctx->mesh_n_idx = n_tris;
    ctx->mesh_has_normals = has_normals != 0 ? 1 : 0;
    return ORE_OK;
}

extern "C" int ore_set_mesh_triangles_device(ore_context* ctx, const float* tris27_dev, int32_t n_tris, void* stream) {
    if (!ctx) return ORE_ERR_INVALID;
    if (ctx->n_tris == 0) return fail(ctx, ORE_ERR_INVALID, "ore_set_mesh_triangles_device: no mesh set (ore_set_mesh first)");
    if (n_tris != ctx->n_tris)
        return fail(ctx, ORE_ERR_INVALID, "ore_set_mesh_triangles_device: n_tris must equal the mesh's triangle count");
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc;
    if ((rc = device_records(ctx, tris27_dev, 4, "ore_set_mesh_triangles_device: the triangles"))) return rc;
    cudaStream_t st;
    if ((rc = update_begin(ctx, stream, &st))) return rc;
    ORE_CUDA(ctx, cudaMemcpyAsync(ctx->tris, tris27_dev, (size_t)n_tris * ore_host::TRI_FLOATS * sizeof(float),
                                  cudaMemcpyDeviceToDevice, st));
    ORE_CUDA(ctx, ore_mesh_refit(ctx->tris, ctx->box_offsets, ctx->box_indices, ctx->boxes, ctx->n_boxes, st));
    ORE_CUDA(ctx, ore_mesh_balls(ctx->boxes, ctx->box_sph, ctx->n_boxes, st));
    return update_end(ctx, st);
}

extern "C" int ore_set_lights(ore_context* ctx, const float* lights7, int32_t n) {
    if (!ctx || n < 0 || n > MAX_LIGHTS || (n > 0 && !lights7))
        return fail(ctx, ORE_ERR_INVALID, "ore_set_lights: 0..16 lights of 7 floats");
    // lights travel as kernel arguments: nothing on the device to wait for
    for (int i = 0; i < n; i++) {
        const float* l = lights7 + 7 * (size_t)i;
        ctx->lights[i] = LightP{l[0], l[1], l[2], l[3], l[4], l[5], l[6]};
    }
    ctx->n_lights = n;
    return ORE_OK;
}

static int upload_planes(ore_context* ctx, DevBuf<float>* dst, const float* r, const float* g, const float* b, int32_t w,
                         int32_t h) {
    if (!ctx || w <= 0 || h <= 0 || !r || !g || !b) return fail(ctx, ORE_ERR_INVALID, "sprite planes: bad arguments");
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    if (int rcw = wait_last_render(ctx)) return rcw;
    const size_t n = (size_t)w * h;
    const float* src[3] = {r, g, b};
    for (int c = 0; c < 3; c++)
        if (int rc = replace_buffer(ctx, dst[c], n, [&](float* p) { memcpy(p, src[c], n * sizeof(float)); })) return rc;
    return ORE_OK;
}

extern "C" int ore_set_texture(ore_context* ctx, const float* r, const float* g, const float* b, int32_t width,
                               int32_t height) {
    int rc = upload_planes(ctx, ctx ? ctx->tex : nullptr, r, g, b, width, height);
    if (rc) return rc;
    ctx->tex_w = width;
    ctx->tex_h = height;
    // (0 x texel must be 0 for lights that do not face a pixel to be skippable: see FrameParams::skip_dark)
    bool finite = true;
    const size_t n = (size_t)width * height;
    const float* planes[3] = {r, g, b};
    for (int c = 0; c < 3 && finite; c++)
        for (size_t i = 0; i < n; i++)
            if (!std::isfinite(planes[c][i])) {
                finite = false;
                break;
            }
    ctx->tex_finite = finite;
    return ORE_OK;
}

extern "C" int ore_set_sky(ore_context* ctx, const float* r, const float* g, const float* b, int32_t width,
                           int32_t height, float size) {
    int rc = upload_planes(ctx, ctx ? ctx->sky : nullptr, r, g, b, width, height);
    if (rc) return rc;
    ctx->sky_w = width;
    ctx->sky_h = height;
    ctx->sky_radius = size * size;  // sphere ctor stores r*r (kernel.cu:287)
    return ORE_OK;
}

// ---- render -------------------------------------------------------------------------------

static constexpr int TILE_ROWS = TILE_P;   // rows per tile of the primary kernel
// shared memory of the primary kernel: the leaf / super-cluster cone records always, the sphere-level records when
// everything stays within this budget (6 CTAs of 128 threads per SM)
static constexpr size_t PRIMARY_RESIDENT_BYTES = 30 * 1024;

// The opt-in dynamic shared-memory limit of a kernel (cudaFuncAttributeMaxDynamicSharedMemorySize) belongs to the kernel
// on a device, not to a context: every context of the process shares it.  It therefore only ever grows, per (device,
// kernel) and process-wide, so that a configuration any context has cached stays launchable whatever another context
// asks for later.
static cudaError_t raise_smem_limit(int device, const void* fn, size_t smem) {
    struct Limit {
        int device;
        const void* fn;
        size_t smem;
    };
    static std::mutex mu;
    static std::vector<Limit> limits;
    std::lock_guard<std::mutex> lock(mu);
    for (Limit& l : limits)
        if (l.device == device && l.fn == fn) {
            if (l.smem >= smem) return cudaSuccess;
            const cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e == cudaSuccess) l.smem = smem;
            return e;
        }
    const cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) limits.push_back({device, fn, smem});
    return e;
}

template <typename K>
static int grid_for(ore_context* ctx, K kernel, size_t smem, int* grid, int threads = CTA_THREADS) {
    const void* fn = reinterpret_cast<const void*>(kernel);
    for (const auto& e : ctx->grid_cache)
        if (e.fn == fn && e.smem == smem && e.threads == threads) {
            *grid = e.grid;
            return ORE_OK;
        }
    int occ = 0;
    ORE_CUDA(ctx, raise_smem_limit(ctx->device, fn, smem));
    ORE_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem));
    if (occ < 1) return fail(ctx, ORE_ERR_CUDA, "kernel does not fit on an SM");
    *grid = occ * ctx->sm_count;
    ctx->grid_cache.push_back({fn, smem, threads, *grid});
    return ORE_OK;
}

// rows y0 + m*y_step + j (j < y_block) below y1
static int frame_rows(const ore_frame* fr) {
    const int yb = fr->y_block > 0 ? fr->y_block : 1;
    const int span = fr->y1 - fr->y0;
    if (span <= 0 || fr->y_step <= 0) return 0;
    if (yb >= fr->y_step) return span;  // contiguous
    const int full = span / fr->y_step, rem = span % fr->y_step;
    return full * yb + (rem < yb ? rem : yb);
}

// the instantiation of each render kernel that a frame's scene and flags select, indexed [large scene][exhaustive]
// [staged][fast libm] (the indices the kernel has)
using PrimaryKernel = void (*)(FrameParams);
using StageKernel = void (*)(FrameParams, StageArgs);
static constexpr PrimaryKernel prep_kernels[2] = {prep_frame_kernel<false>, prep_frame_kernel<true>};
static constexpr PrimaryKernel primary_kernels[2][2][2] = {
    {{primary_tile_kernel<TILE_ROWS, false, false, false>, primary_tile_kernel<TILE_ROWS, false, true, false>},
     {primary_tile_kernel<TILE_ROWS, true, false, false>, primary_tile_kernel<TILE_ROWS, true, true, false>}},
    {{primary_tile_kernel<TILE_ROWS, false, false, true>, primary_tile_kernel<TILE_ROWS, false, true, true>},
     {primary_tile_kernel<TILE_ROWS, true, false, true>, primary_tile_kernel<TILE_ROWS, true, true, true>}}};
static constexpr StageKernel sweep_kernels[2][2][2][2] = {
    {{{shadow_sweep_kernel<false, false, false, false>, shadow_sweep_kernel<false, false, true, false>},
      {shadow_sweep_kernel<false, true, false, false>, shadow_sweep_kernel<false, true, true, false>}},
     {{shadow_sweep_kernel<true, false, false, false>, shadow_sweep_kernel<true, false, true, false>},
      {shadow_sweep_kernel<true, true, false, false>, shadow_sweep_kernel<true, true, true, false>}}},
    {{{shadow_sweep_kernel<false, false, false, true>, shadow_sweep_kernel<false, false, true, true>},
      {shadow_sweep_kernel<false, true, false, true>, shadow_sweep_kernel<false, true, true, true>}},
     {{shadow_sweep_kernel<true, false, false, true>, shadow_sweep_kernel<true, false, true, true>},
      {shadow_sweep_kernel<true, true, false, true>, shadow_sweep_kernel<true, true, true, true>}}}};
static constexpr StageKernel shade_setup_kernels[2] = {shade_setup_kernel<false>, shade_setup_kernel<true>};

// one launch of the sweep kernel (stage B / fused / catch-all)
static int launch_sweep(ore_context* ctx, const FrameParams& prm, const StageArgs& st, bool staged, bool exh, bool fast_libm,
                        cudaStream_t stream) {
    int rc, grid = 0;
    const StageKernel sweep = sweep_kernels[prm.n_hypers_pad > 0][exh][staged][fast_libm];
    if ((rc = grid_for(ctx, sweep, SWEEP_SMEM_BYTES, &grid, SWEEP_THREADS))) return rc;
    sweep<<<grid, SWEEP_THREADS, SWEEP_SMEM_BYTES, stream>>>(prm, st);
    ORE_CUDA(ctx, cudaGetLastError());
    return ORE_OK;
}

// Copies n_rows rows of W pixels that lie in blocks of B rows, S image rows apart, at dst, from src where they are packed:
// one strided copy of the full blocks, then one of the ragged tail.
static int copy_row_blocks(ore_context* ctx, uint32_t* dst, const uint32_t* src, size_t W, int n_rows, int B, int S,
                           cudaMemcpyKind kind, cudaStream_t stream) {
    const size_t full = (size_t)(n_rows / B), rem = (size_t)(n_rows % B), row_bytes = W * sizeof(uint32_t);
    if (full)
        ORE_CUDA(ctx, cudaMemcpy2DAsync(dst, (size_t)S * row_bytes, src, (size_t)B * row_bytes, (size_t)B * row_bytes, full, kind,
                                        stream));
    if (rem) ORE_CUDA(ctx, cudaMemcpyAsync(dst + full * S * W, src + full * B * W, rem * row_bytes, kind, stream));
    return ORE_OK;
}

struct TileCone {
    float px_delta, ca, sa;   // FrameParams::px_delta, tile_ca, tile_sa
};

// Largest half-angle of a 32 x TILE_ROWS pixel tile seen from the eye (tile cone of the primary kernel), for rendered rows
// in blocks of y_block, y_step image rows apart: |v_pixel - v_centre| <= halfdiag on the image plane and |v| >= fz, so
// sin(a) <= halfdiag/fz.
static TileCone tile_cone(float aspect, int W, int y_block, int y_step, float fz) {
    const double delta = 2.0 * (double)aspect / (double)W;
    // tallest image-row span of TILE_ROWS consecutive RENDERED rows
    int max_span = 0;
    for (int k0 = 0; k0 < y_block * TILE_ROWS; k0 += TILE_ROWS) {
        const int k1 = k0 + TILE_ROWS - 1;
        const int sp = ((k1 / y_block) * y_step + k1 % y_block) - ((k0 / y_block) * y_step + k0 % y_block);
        if (sp > max_span) max_span = sp;
    }
    const double hx = 16.0 * delta, hy = (0.5 * max_span + 0.5) * delta;
    const double xr = sqrt(hx * hx + hy * hy) / fabs((double)fz);
    if (!(xr < 0.9)) return {(float)delta, -1e20f, 0.f};   // tiles too wide for a cone: every sphere is a candidate
    const double a = asin(xr) * 1.001 + 1e-6;
    return {(float)delta, (float)(cos(a) * (1.0 - 1e-6) - 1e-6), (float)(sin(a) * (1.0 + 1e-6) + 1e-6)};
}

// The kernel parameters of a launch set: frame geometry and cameras, outputs (outs: the caller's framebuffers, null: the
// context's own), the context's scene, per-frame buffers (sized by the caller) and lights.  band_dma: the primary kernel
// writes its rows to band_buf.  *psmem: dynamic shared memory of the primary kernel.
static FrameParams frame_params(const ore_context* ctx, const ore_camera* cams, int n_frames, const ore_frame* fr,
                                uint32_t* const* outs, bool band_dma, size_t* psmem) {
    FrameParams prm;
    memset(&prm, 0, sizeof prm);
    const int W = fr->width;
    const int yb = fr->y_block > 0 ? fr->y_block : 1;
    prm.W = W;
    prm.W_pad = (W + 31) & ~31;
    prm.H = fr->height;
    prm.y0 = fr->y0;
    prm.y_step = (yb >= fr->y_step) ? 1 : fr->y_step;
    prm.n_rows = frame_rows(fr);
    prm.n_frames = n_frames;
    prm.n_px_frame = (uint32_t)((size_t)prm.n_rows * W);
    prm.y_block = (yb >= fr->y_step) ? 1 : yb;
    prm.out_global = (outs && fr->out_pitch > 0) ? 1 : 0;
    prm.pitch = prm.out_global ? fr->out_pitch : W;
    prm.n_spheres = ctx->n_spheres;
    prm.n_lights = ctx->n_lights;
    prm.flags = fr->flags;
    prm.aspect = fr->aspect;
    prm.ez = (-1 / fr->aspect);  // kernel.cu:1629
    prm.fz = 0.f - prm.ez;
    for (int f = 0; f < n_frames; f++) {
        const ore_camera* cam = &cams[f];
        CamP& c = prm.cam[f];
        c.Ox = 0.f + cam->org[0];  // add(eyePos, cam.Org), kernel.cu:1631
        c.Oy = 0.f + cam->org[1];
        c.Oz = prm.ez + cam->org[2];
        // camera::rotateDir, kernel.cu:249-255: frame-uniform, evaluated once on the host
        float yawRad = cam->yaw * (3.1415 / 180);
        float pitchRad = cam->pitch * (3.1415 / 180);
        c.cp = cosf(pitchRad);
        c.sp = sinf(pitchRad);
        c.cy = cosf(yawRad);
        c.sy = sinf(yawRad);
        prm.pixels[f] = outs ? outs[f] : (uint32_t*)ctx->pixels;
        prm.sky_pixels[f] = band_dma ? ctx->band_buf + (size_t)f * prm.n_px_frame : prm.pixels[f];
    }
    prm.sky_pitch = band_dma ? W : prm.pitch;
    prm.sky_global = band_dma ? 0 : prm.out_global;
    const TileCone tc = tile_cone(fr->aspect, W, prm.y_block, prm.y_step, prm.fz);
    prm.px_delta = tc.px_delta;
    prm.tile_ca = tc.ca;
    prm.tile_sa = tc.sa;
    prm.dx_tab = ctx->dx_tab;
    prm.dy_tab = ctx->dy_tab;
    prm.sph_exact = ctx->sph_exact;
    prm.sph_xsort = ctx->sph_xsort;
    prm.sph_sort = ctx->sph_sort;
    prm.sort_index = ctx->sort_index;
    prm.leaf_sph = ctx->leaf_sph;
    prm.super_sph = ctx->super_sph;
    prm.n_sort = ctx->n_sort;
    prm.n_leaves = ctx->n_leaves;
    prm.n_leaves_pad = ctx->n_leaves_pad;
    prm.n_supers = ctx->n_supers;
    prm.n_supers_pad = ctx->n_supers_pad;
    prm.prim_sorted = ctx->prim_sorted;
    prm.cone_sorted = ctx->cone_sorted;
    prm.leaf_cone = ctx->leaf_cone;
    prm.super_cone = ctx->super_cone;
    if (ctx->n_hypers_pad) {
        // large scene: only the hyper-cluster records are staged
        prm.hyper_sph = ctx->hyper_sph;
        prm.hyper_cone = ctx->hyper_cone;
        prm.n_hypers = ctx->n_hypers;
        prm.n_hypers_pad = ctx->n_hypers_pad;
        prm.cone_resident = 0;
        *psmem = (size_t)ctx->n_hypers_pad * sizeof(float4);
    } else {
        const size_t tree_bytes = ((size_t)ctx->n_supers_pad + (size_t)ctx->n_leaves_pad) * sizeof(float4);
        const size_t all_bytes = tree_bytes + (size_t)ctx->n_sort * sizeof(float4);
        prm.cone_resident = all_bytes <= PRIMARY_RESIDENT_BYTES ? 1 : 0;
        *psmem = prm.cone_resident ? all_bytes : tree_bytes;
    }
    prm.tex_r = ctx->tex[0];
    prm.tex_g = ctx->tex[1];
    prm.tex_b = ctx->tex[2];
    prm.tex_w = ctx->tex_w;
    prm.tex_h = ctx->tex_h;
    prm.sky_r = ctx->sky[0];
    prm.sky_g = ctx->sky[1];
    prm.sky_b = ctx->sky[2];
    prm.sky_w = ctx->sky_w;
    prm.sky_h = ctx->sky_h;
    prm.sky_radius = ctx->sky_radius;
    prm.cubes = ctx->cubes;
    prm.planes = ctx->planes;
    prm.n_cubes = ctx->n_cubes;
    prm.n_planes = ctx->n_planes;
    prm.tris = ctx->tris;
    prm.boxes = ctx->boxes;
    prm.box_offsets = ctx->box_offsets;
    prm.box_indices = ctx->box_indices;
    prm.box_sph = ctx->box_sph;
    prm.box_cone = ctx->box_cone;
    prm.n_tris = ctx->n_tris;
    prm.n_boxes = ctx->n_boxes;
    prm.n_live_boxes = ctx->mesh_live;
    prm.mesh_has_normals = ctx->mesh_has_normals;
    bool skip = ctx->tex_finite && !(fr->flags & ORE_FLAG_EXHAUSTIVE);
    for (int i = 0; i < ctx->n_lights && skip; i++)
        skip = std::isfinite(ctx->lights[i].r) && std::isfinite(ctx->lights[i].g) && std::isfinite(ctx->lights[i].b);
    prm.skip_dark = skip ? 1 : 0;
    prm.hit_list = ctx->hit_list;
    prm.hit_ids = ctx->hit_ids;
    prm.hit_ts = ctx->hit_ts;
    prm.counters = ctx->counters;
    for (int i = 0; i < ctx->n_lights; i++) prm.lights[i] = ctx->lights[i];
    return prm;
}

// Enqueues a launch set on `stream`, in this order: prep, primary, the band-DMA copy (on band_stream, joined before the
// first sweep), the shadow pass as ore_stage_plan.h plans it, the hint copy, the count kernel; timing events between them.
static int launch_frame(ore_context* ctx, const FrameParams& prm, size_t psmem, uint32_t* const* outs, bool band_dma,
                        cudaStream_t stream) {
    int rc;
    const size_t n_px = (size_t)prm.n_px_frame * (size_t)prm.n_frames;
    const bool timing = !(prm.flags & ORE_FLAG_NO_KERNEL_TIMING);
    const bool large = prm.n_hypers_pad > 0;
    if (timing) ORE_CUDA(ctx, cudaEventRecord(ctx->ev[0], stream));
    {
        // (n_hypers_pad <= n_supers_pad)
        int m = prm.W_pad > prm.n_rows ? prm.W_pad : prm.n_rows;
        m = std::max(m, std::max(ctx->n_sort, std::max(ctx->n_leaves_pad, ctx->n_supers_pad)));
        m = std::max(m, std::max(ctx->n_boxes, (int)CNT_SLOTS));
        prep_kernels[large]<<<(m + 255) / 256, 256, 0, stream>>>(prm);
        ORE_CUDA(ctx, cudaGetLastError());
        ctx->last_launches++;
    }
    if (timing) ORE_CUDA(ctx, cudaEventRecord(ctx->ev[1], stream));
    const bool exh = (prm.flags & ORE_FLAG_EXHAUSTIVE) != 0;
    const bool fast_libm = (prm.flags & ORE_FLAG_FAST_LIBM) != 0;
    {
        int grid = 0;
        const long long tiles = (long long)((prm.W + 31) / 32) * ((prm.n_rows + TILE_ROWS - 1) / TILE_ROWS);
        const long long n_batches = ((tiles + PRIMARY_WARPS - 1) / PRIMARY_WARPS) * prm.n_frames;
        const PrimaryKernel primary = primary_kernels[large][exh][fast_libm];
        if ((rc = grid_for(ctx, primary, psmem, &grid, PRIMARY_THREADS))) return rc;
        if (grid > n_batches) grid = (int)n_batches;
        primary<<<grid, PRIMARY_THREADS, psmem, stream>>>(prm);
        ORE_CUDA(ctx, cudaGetLastError());
        ctx->last_launches++;
    }
    if (timing) ORE_CUDA(ctx, cudaEventRecord(ctx->ev[2], stream));
    ctx->ev_band_done.forget();   // (recorded below when this frame copies its rows)
    if (band_dma) {
        // the rows the primary kernel has just written (sky pixels, 0 for hit pixels) travel to their place in the
        // destination frames on a copy engine, behind the primary kernel and concurrently with stage A of the shadow
        // pass; the sweep, which stores the hit pixels into the same rows, waits for them
        ORE_CUDA(ctx, cudaEventRecord(ctx->ev_band_go, stream));
        ORE_CUDA(ctx, cudaStreamWaitEvent(ctx->band_stream, ctx->ev_band_go, 0));
        for (int f = 0; f < prm.n_frames; f++)   // (y_block and y_step are 1 for a contiguous band)
            if ((rc = copy_row_blocks(ctx, outs[f], ctx->band_buf + (size_t)f * prm.n_px_frame, prm.W, prm.n_rows, prm.y_block,
                                      prm.y_step, cudaMemcpyDefault, ctx->band_stream)))
                return rc;
        ORE_CUDA(ctx, ctx->ev_band_done.record(ctx->band_stream));
    }
    auto join_band = [&]() -> int {   // (the first call waits for the copy, later ones do nothing)
        ORE_CUDA(ctx, ctx->ev_band_done.stream_wait(stream));
        ctx->ev_band_done.forget();
        return ORE_OK;
    };
    // Two-stage pass (default): shade_setup_kernel -> staging buffer -> staged shadow_sweep_kernel, in the chunk pairs of
    // plan_stage, from the previous frame's hit count (a hint read without synchronisation), and one catch-all launch
    // of the fused sweep for whatever lies beyond the staged chunks.  With no lights there is nothing to sweep: the
    // primary kernel has already written 0 to every hit pixel.
    const StagePlan plan = plan_stage(n_px, ctx->n_lights, (prm.flags & ORE_FLAG_FUSED_SHADOW) != 0, ctx->hits_hint_set,
                                      *(volatile unsigned long long*)ctx->hits_hint, ctx->stage.cap(), ctx->stage_blocks_override,
                                      ctx->stage_max_items);
    bool staged = plan.staged;
    if (staged && !ctx->stage.fits(plan.need_floats)) {
        // (an earlier frame of this context may still be reading the old buffer on another stream)
        if ((rc = wait_last_render(ctx))) return rc;
        ORE_CUDA(ctx, ctx->stage.release());
        if (ctx->stage.alloc(plan.need_floats) != cudaSuccess) {
            (void)cudaGetLastError();  // no room for the staging buffer: the fused sweep needs none
            staged = false;
        }
    }
    StageArgs st{};
    st.nv = STAGE_HEADER + STAGE_PER_LIGHT * ctx->n_lights;
    if (ctx->n_lights == 0) {
        // nothing to launch
    } else if (!staged) {
        if ((rc = join_band())) return rc;
        if ((rc = launch_sweep(ctx, prm, st, false, exh, fast_libm, stream))) return rc;
        ctx->last_launches++;
    } else {
        st.buf = ctx->stage;
        st.cap_blocks = (uint32_t)plan.cap_blocks;
        const StageKernel setup = shade_setup_kernels[fast_libm];
        int grid_a = 0;
        if ((rc = grid_for(ctx, setup, 0, &grid_a, STAGE_A_THREADS))) return rc;
        for (int c = 0; c < plan.n_chunks; c++) {
            st.chunk = c;
            st.first_block = (uint32_t)((size_t)c * plan.cap_blocks);
            setup<<<grid_a, STAGE_A_THREADS, 0, stream>>>(prm, st);
            ORE_CUDA(ctx, cudaGetLastError());
            if ((rc = join_band())) return rc;   // (band DMA: the first stage A ran beside the copy)
            if ((rc = launch_sweep(ctx, prm, st, true, exh, fast_libm, stream))) return rc;
            ctx->last_launches += 2;
        }
        if (plan.catch_all) {
            // catch-all: hit-list blocks beyond the staged chunks (normally none: exits at once), one fused launch
            StageArgs rest{};
            rest.first_block = (uint32_t)plan.catch_all_block;
            rest.nv = st.nv;
            if ((rc = launch_sweep(ctx, prm, rest, false, exh, fast_libm, stream))) return rc;
            ctx->last_launches++;
        }
    }
    if ((rc = join_band())) return rc;   // (no lights: nothing but the copy writes the frames)
    if (timing) ORE_CUDA(ctx, cudaEventRecord(ctx->ev[3], stream));
    // hint for the next frame of this context (see hits_hint): 8 bytes, no synchronisation
    ORE_CUDA(ctx, cudaMemcpyAsync(ctx->hits_hint, ctx->counters + CNT_HITS, sizeof(unsigned long long),
                                  cudaMemcpyDeviceToHost, stream));
    ctx->hits_hint_set = true;
    if (prm.flags & ORE_FLAG_COUNT_REFERENCE_TESTS) {
        count_reference_tests_kernel<<<ctx->sm_count * 8, CTA_THREADS, 0, stream>>>(prm);
        ORE_CUDA(ctx, cudaGetLastError());
        ctx->last_launches++;
    }
    if (timing) ORE_CUDA(ctx, ctx->ev_end.record(stream));
    ORE_CUDA(ctx, ctx->ev_done.record(stream));
    return ORE_OK;
}

// One launch set for a batch of n_frames cameras.  outs: n_frames device framebuffers, or null (n_frames == 1 only): the
// context's own framebuffer.
static int render_impl(ore_context* ctx, const ore_camera* cams, int n_frames, const ore_frame* fr, uint32_t* const* outs,
                       cudaStream_t stream) {
    if (!ctx) return ORE_ERR_INVALID;
    if (!cams || !fr) return fail(ctx, ORE_ERR_INVALID, "ore_render: null camera/frame");
    if (n_frames < 1 || n_frames > MAX_BATCH || (!outs && n_frames != 1))
        return fail(ctx, ORE_ERR_INVALID, "ore_render: a batch holds 1..8 frames");
    // a band may be empty (y0 >= y1: a rank with no rows of a short frame) but never reaches past the image
    if (fr->width <= 0 || fr->height <= 0 || fr->y_step <= 0 || fr->y0 < 0 || fr->y1 < 0 || fr->y1 > fr->height ||
        (fr->out_pitch != 0 && fr->out_pitch < fr->width))
        return fail(ctx, ORE_ERR_INVALID, "ore_render: bad frame geometry");
    // the eye sits 1/aspect behind the image plane (kernel.cu:1629): 0, +-inf, NaN and aspects whose reciprocal
    // overflows give no finite eye and are rejected before anything renders
    if (!std::isfinite(fr->aspect) || !std::isfinite(1.f / fr->aspect))
        return fail(ctx, ORE_ERR_INVALID, "ore_render: aspect must be finite and non-zero, with a finite 1/aspect");
    if (fr->flags & ~(uint32_t)(ORE_FLAG_EXHAUSTIVE | ORE_FLAG_COUNT_REFERENCE_TESTS | ORE_FLAG_FAST_LIBM | ORE_FLAG_FUSED_SHADOW |
                                ORE_FLAG_NO_KERNEL_TIMING | ORE_FLAG_BAND_DMA))
        return fail(ctx, ORE_ERR_INVALID, "ore_render: unknown flag");
    if (!ctx->tex[0] || !ctx->sky[0]) return fail(ctx, ORE_ERR_INVALID, "ore_render: texture and sky must be set first");
    if (ctx->n_spheres > MAX_RENDER_SPHERES)
        return fail(ctx, ORE_ERR_INVALID, "ore_render: a scene of more than 2^24 = 16 777 216 spheres is not supported");
    if (!ctx->sph_exact) {
        int rc = upload_spheres(ctx, nullptr, 4, 0, 0);
        if (rc) return rc;
    }
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    const int W = fr->width;
    const int yb = fr->y_block > 0 ? fr->y_block : 1;
    if (yb > fr->y_step && fr->y_step != 1) return fail(ctx, ORE_ERR_INVALID, "ore_render: y_block must not exceed y_step");
    const int n_rows = frame_rows(fr);
    const size_t n_px_frame = (size_t)n_rows * W;
    const size_t n_px = n_px_frame * (size_t)n_frames;   // pixels of the whole batch
    if (n_px_frame >= (size_t)1 << 31 || n_px >= ((size_t)1 << 32) - 64) return fail(ctx, ORE_ERR_INVALID, "ore_render: band / batch too large");
    ctx->last_px = n_px_frame;
    ctx->last_frames = n_frames;
    ctx->last_n_spheres = ctx->n_spheres;
    ctx->last_launches = 0;
    ctx->ev_end.forget();
    ctx->last_prm_valid = false;
    if (n_px == 0) return ORE_OK;
    for (int f = 0; outs && f < n_frames; f++)
        if (!outs[f]) return fail(ctx, ORE_ERR_INVALID, "ore_render: null framebuffer in the batch");
    // the scene of the last stream-ordered update, wherever it ran
    ORE_CUDA(ctx, ctx->ev_scene.stream_wait(stream));

    int rc;
    if ((rc = frame_reserve(ctx, ctx->dx_tab, (size_t)((W + 31) & ~31)))) return rc;
    if ((rc = frame_reserve(ctx, ctx->dy_tab, (size_t)n_rows))) return rc;
    if ((rc = frame_reserve(ctx, ctx->hit_list, n_px))) return rc;
    if ((rc = frame_reserve(ctx, ctx->hit_ids, n_px))) return rc;
    if ((rc = frame_reserve(ctx, ctx->hit_ts, n_px))) return rc;
    // the context's own framebuffer: only ore_render (one frame, host output) renders into it
    if (!outs && (rc = frame_reserve(ctx, ctx->pixels, n_px_frame))) return rc;
    // Band DMA (include/ore_render.h; opt-in): rows whose 8-row blocks are contiguous at the destination (pitch == width)
    const bool band_dma = outs && fr->out_pitch == W && (fr->flags & ORE_FLAG_BAND_DMA) != 0;
    if (band_dma) {
        if ((rc = frame_reserve(ctx, ctx->band_buf, n_px))) return rc;
        if (!ctx->band_stream) {   // (the stream last: it marks the group as made)
            ORE_CUDA(ctx, cudaEventCreateWithFlags(ctx->ev_band_go.put(), cudaEventDisableTiming));
            ORE_CUDA(ctx, cudaEventCreateWithFlags(ctx->ev_band_done.put(), cudaEventDisableTiming));
            ORE_CUDA(ctx, cudaStreamCreateWithFlags(ctx->band_stream.put(), cudaStreamNonBlocking));
        }
    }
    size_t psmem = 0;
    FrameParams prm = frame_params(ctx, cams, n_frames, fr, outs, band_dma, &psmem);
    if (!ctx->dbg_cycles_path.empty()) {
        const size_t nb = (n_px + 31) / 32;   // [2][nb]: stage A, stage B
        if (!ctx->dbg_cycles.fits(2 * nb)) ORE_CUDA(ctx, ctx->dbg_cycles.alloc(2 * nb));
        ORE_CUDA(ctx, cudaMemsetAsync(ctx->dbg_cycles, 0, ctx->dbg_cycles.cap() * sizeof(uint32_t), stream));
        prm.dbg_cycles = ctx->dbg_cycles;
        prm.dbg_cap = (uint32_t)(ctx->dbg_cycles.cap() / 2);
    }
    if ((rc = launch_frame(ctx, prm, psmem, outs, band_dma, stream))) return rc;
    ctx->last_prm = prm;
    ctx->last_prm_valid = true;
    return ORE_OK;
}

extern "C" int ore_render_device(ore_context* ctx, const ore_camera* cam, const ore_frame* frame,
                                 uint32_t* out_device, void* stream) {
    if (!ctx) return ORE_ERR_INVALID;
    if (!out_device) return fail(ctx, ORE_ERR_INVALID, "ore_render_device: null output");
    uint32_t* outs[1] = {out_device};
    return render_impl(ctx, cam, 1, frame, outs, stream ? (cudaStream_t)stream : ctx->stream);
}

extern "C" int ore_render_batch_device(ore_context* ctx, const ore_camera* cams, int32_t n_frames, const ore_frame* frame,
                                       uint32_t* const* out_device, void* stream) {
    if (!ctx) return ORE_ERR_INVALID;
    if (!out_device) return fail(ctx, ORE_ERR_INVALID, "ore_render_batch_device: null output");
    return render_impl(ctx, cams, n_frames, frame, out_device, stream ? (cudaStream_t)stream : ctx->stream);
}

extern "C" int ore_render(ore_context* ctx, const ore_camera* cam, const ore_frame* frame, uint32_t* out_host) {
    if (!ctx) return ORE_ERR_INVALID;
    if (!out_host) return fail(ctx, ORE_ERR_INVALID, "ore_render: null output");
    int rc = render_impl(ctx, cam, 1, frame, nullptr, ctx->stream);
    if (rc) return rc;
    if (ctx->last_px) {
        // device -> host of the band; CUDA stages pageable destinations through its own pinned pool
        ORE_CUDA(ctx, cudaMemcpyAsync(out_host, ctx->pixels, ctx->last_px * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                                      ctx->stream));
    }
    ORE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ORE_OK;
}

// ---- stream-ordered 32-bit flags (cuStreamWriteValue32 / cuStreamWaitValue32, no SM involved) ----------------
// The driver entry points are resolved at run time (the library links against cudart only).
typedef int (*ore_cu_memop32)(cudaStream_t, unsigned long long /*CUdeviceptr*/, unsigned int, unsigned int);
static ore_cu_memop32 driver_memop(const char* name) {   // null when the driver does not offer it
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    const bool ok = cudaGetDriverEntryPoint(name, &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess;
    (void)cudaGetLastError();
    return ok ? (ore_cu_memop32)f : nullptr;
}
struct MemOps {
    ore_cu_memop32 write32, wait32;
};
// resolved by the first flag call of the process (a function-local static: initialised once, thread-safely)
static const MemOps& memops() {
    static const MemOps m{driver_memop("cuStreamWriteValue32"), driver_memop("cuStreamWaitValue32")};
    return m;
}

// fallbacks on an SM: one thread.  The wait kernel is only ever used when the driver offers no stream wait; it
// polls a flag that ANOTHER GPU (or the host) writes, never another launch on this GPU.
__global__ void flag_write_kernel(uint32_t* flag, uint32_t value) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(value) : "memory");
}
__global__ void flag_wait_kernel(const uint32_t* flag, uint32_t value) {
    for (;;) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if ((int32_t)(v - value) >= 0) break;
        __nanosleep(200);
    }
}

static cudaStream_t pick_stream(ore_context* ctx, void* stream) { return stream ? (cudaStream_t)stream : ctx->stream; }

extern "C" void* ore_get_stream(ore_context* ctx, int which) {
    if (!ctx) return nullptr;
    if (which == 2) return (cudaStream_t)ctx->signal_stream;  // null until the first ore_flag_write_after
    return which == 1 ? (cudaStream_t)ctx->copy_stream : (cudaStream_t)ctx->stream;
}

extern "C" int ore_flag_write(ore_context* ctx, void* stream, uint32_t* flag, uint32_t value) {
    if (!ctx || !flag) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    const ore_cu_memop32 cu_write32 = memops().write32;
    cudaStream_t st = pick_stream(ctx, stream);
    // peer-mapped device memory (another GPU's flag, imported with ore_ipc_import) is written by a one-thread
    // kernel (st.release.sys over NVLink); local device memory and registered host memory by the stream itself
    cudaPointerAttributes at;
    bool local = false;
    if (cudaPointerGetAttributes(&at, flag) == cudaSuccess)
        local = (at.type == cudaMemoryTypeHost) || (at.type == cudaMemoryTypeDevice && at.device == ctx->device);
    (void)cudaGetLastError();
    if (local && cu_write32 && !ctx->no_memops) {
        void* dptr = flag;
        if (at.type == cudaMemoryTypeHost) ORE_CUDA(ctx, cudaHostGetDevicePointer(&dptr, flag, 0));
        if (cu_write32(st, (unsigned long long)(uintptr_t)dptr, value, 0) == 0) return ORE_OK;
    }
    flag_write_kernel<<<1, 1, 0, st>>>(flag, value);
    ORE_CUDA(ctx, cudaGetLastError());
    return ORE_OK;
}

// Ordered variant for frames rendered on SEVERAL streams (frames in flight): the flag is written on the context's
// signal stream once everything enqueued on `stream` so far has completed.  The signal stream is in-order, so flag
// values written through one context appear in call order even when the frames finish out of order.
extern "C" int ore_flag_write_after(ore_context* ctx, void* stream, uint32_t* flag, uint32_t value) {
    if (!ctx || !flag) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!ctx->signal_stream) {   // (the stream last: it marks the group as made)
        for (Event& e : ctx->ev_signal) ORE_CUDA(ctx, cudaEventCreateWithFlags(e.put(), cudaEventDisableTiming));
        ORE_CUDA(ctx, cudaStreamCreateWithFlags(ctx->signal_stream.put(), cudaStreamNonBlocking));
    }
    const Event& e = ctx->ev_signal[ctx->n_signals++ % 8];
    ORE_CUDA(ctx, cudaEventRecord(e, pick_stream(ctx, stream)));
    ORE_CUDA(ctx, cudaStreamWaitEvent(ctx->signal_stream, e, 0));
    return ore_flag_write(ctx, ctx->signal_stream, flag, value);
}

extern "C" int ore_flag_wait_geq(ore_context* ctx, void* stream, const uint32_t* flag, uint32_t value) {
    if (!ctx || !flag) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    const ore_cu_memop32 cu_wait32 = memops().wait32;
    cudaStream_t st = pick_stream(ctx, stream);
    cudaPointerAttributes at;
    void* dptr = (void*)flag;
    if (cudaPointerGetAttributes(&at, flag) == cudaSuccess && at.type == cudaMemoryTypeHost)
        ORE_CUDA(ctx, cudaHostGetDevicePointer(&dptr, (void*)flag, 0));
    (void)cudaGetLastError();
    if (cu_wait32 && !ctx->no_memops) {
        if (cu_wait32(st, (unsigned long long)(uintptr_t)dptr, value, 0 /* CU_STREAM_WAIT_VALUE_GEQ */) == 0) return ORE_OK;
    }
    flag_wait_kernel<<<1, 1, 0, st>>>((const uint32_t*)dptr, value);
    ORE_CUDA(ctx, cudaGetLastError());
    return ORE_OK;
}

extern "C" int ore_host_register(ore_context* ctx, void* host_ptr, size_t bytes) {
    if (!ctx || !host_ptr || bytes == 0) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaHostRegister(host_ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
    return ORE_OK;
}
extern "C" int ore_host_unregister(ore_context* ctx, void* host_ptr) {
    if (!ctx || !host_ptr) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaHostUnregister(host_ptr));
    return ORE_OK;
}

// Pipelined presentation.  A batch of frames is rendered into one of two sets of device framebuffers and copied to
// the host on the copy stream while the next batch renders.  frame->out_pitch == 0: rows packed at out_host[f].
// out_pitch == width: out_host[f] is image row y0 of a FULL host frame and every rendered row lands at its image
// position (a rank of a multi-GPU job copies its own row blocks into the shared host frame over its own PCIe link).
// done_flag (optional): first_value + f is stored there, in stream order, once frame f's copy has landed.
static int render_async_impl(ore_context* ctx, const ore_camera* cams, int n_frames, const ore_frame* frame,
                             uint32_t* const* out_host, uint32_t* done_flag, uint32_t first_value) {
    if (!ctx) return ORE_ERR_INVALID;
    if (!out_host || !frame || !cams) return fail(ctx, ORE_ERR_INVALID, "ore_render_async: null output/frame");
    if (n_frames < 1 || n_frames > MAX_BATCH) return fail(ctx, ORE_ERR_INVALID, "ore_render_async: a batch holds 1..8 frames");
    for (int f = 0; f < n_frames; f++)
        if (!out_host[f]) return fail(ctx, ORE_ERR_INVALID, "ore_render_async: null host frame in the batch");
    if (frame->out_pitch != 0 && frame->out_pitch != frame->width)
        return fail(ctx, ORE_ERR_INVALID, "ore_render_async: out_pitch must be 0 (packed) or the frame width (rows in place)");
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    const int n_rows = frame_rows(frame);
    const size_t W = (size_t)(frame->width > 0 ? frame->width : 0);
    const size_t n_px = (size_t)(n_rows > 0 ? n_rows : 0) * W;
    const int set = (int)(ctx->async_batches & 1ull);
    int rc;
    if (n_px != ctx->async_px || n_frames != ctx->async_k || !ctx->async_pool) {
        // new geometry: the two sets are laid out afresh, so nothing of the old layout may still be in flight
        ORE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ORE_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
        ORE_CUDA(ctx, ctx->async_pool.reserve(2 * (size_t)n_frames * (n_px ? n_px : 1)));
        ctx->async_px = n_px;
        ctx->async_k = n_frames;
    }
    uint32_t* targets[MAX_BATCH];
    for (int f = 0; f < n_frames; f++) targets[f] = ctx->async_pool + ((size_t)set * n_frames + f) * n_px;
    // do not overwrite framebuffers whose previous copy is still in flight
    ORE_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_copied[set], 0));
    ore_frame fr = *frame;
    fr.out_pitch = 0;
    if ((rc = render_impl(ctx, cams, n_frames, &fr, targets, ctx->stream))) return rc;
    ORE_CUDA(ctx, cudaEventRecord(ctx->ev_rendered[set], ctx->stream));
    ORE_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_rendered[set], 0));
    for (int f = 0; f < n_frames; f++) {
        if (n_px) {
            const int yb = frame->y_block > 0 ? frame->y_block : 1;
            if (frame->out_pitch == 0 || yb >= frame->y_step) {
                // packed, or a contiguous band: one linear copy
                ORE_CUDA(ctx, cudaMemcpyAsync(out_host[f], targets[f], n_px * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->copy_stream));
            } else {
                // block-interleaved rows: blocks of yb rows, y_step image rows apart
                if ((rc = copy_row_blocks(ctx, out_host[f], targets[f], W, n_rows, yb, frame->y_step, cudaMemcpyDeviceToHost,
                                          ctx->copy_stream)))
                    return rc;
            }
        }
        if (done_flag && (rc = ore_flag_write(ctx, ctx->copy_stream, done_flag, first_value + (uint32_t)f))) return rc;
    }
    ORE_CUDA(ctx, cudaEventRecord(ctx->ev_copied[set], ctx->copy_stream));
    ctx->async_batches++;
    return ORE_OK;
}

extern "C" int ore_render_async(ore_context* ctx, const ore_camera* cam, const ore_frame* frame, uint32_t* out_host) {
    uint32_t* outs[1] = {out_host};
    return render_async_impl(ctx, cam, 1, frame, outs, nullptr, 0);
}
extern "C" int ore_render_async_signal(ore_context* ctx, const ore_camera* cam, const ore_frame* frame, uint32_t* out_host,
                                       uint32_t* done_flag, uint32_t done_value) {
    if (!done_flag) return fail(ctx, ORE_ERR_INVALID, "ore_render_async_signal: null flag");
    uint32_t* outs[1] = {out_host};
    return render_async_impl(ctx, cam, 1, frame, outs, done_flag, done_value);
}
extern "C" int ore_render_batch_async(ore_context* ctx, const ore_camera* cams, int32_t n_frames, const ore_frame* frame,
                                      uint32_t* const* out_host, uint32_t* done_flag, uint32_t first_done_value) {
    return render_async_impl(ctx, cams, n_frames, frame, out_host, done_flag, first_done_value);
}

extern "C" int ore_wait(ore_context* ctx) {
    if (!ctx) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ORE_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
    return ORE_OK;
}

extern "C" int ore_host_alloc(ore_context* ctx, size_t bytes, void** host_ptr) {
    if (!ctx || !host_ptr || bytes == 0) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaMallocHost(host_ptr, bytes));
    return ORE_OK;
}
extern "C" int ore_host_free(ore_context* ctx, void* host_ptr) {
    if (!ctx) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaFreeHost(host_ptr));
    return ORE_OK;
}

extern "C" int ore_synchronize(ore_context* ctx) {
    if (!ctx) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ORE_CUDA(ctx, cudaDeviceSynchronize());
    return ORE_OK;
}

extern "C" int ore_dev_alloc(ore_context* ctx, size_t bytes, void** dev_ptr) {
    if (!ctx || !dev_ptr || bytes == 0) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaMalloc(dev_ptr, bytes));
    ORE_CUDA(ctx, cudaMemset(*dev_ptr, 0, bytes));
    return ORE_OK;
}
extern "C" int ore_dev_free(ore_context* ctx, void* dev_ptr) {
    if (!ctx) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaFree(dev_ptr));
    return ORE_OK;
}
extern "C" int ore_ipc_export(ore_context* ctx, void* dev_ptr, unsigned char handle[64]) {
    if (!ctx || !dev_ptr || !handle) return ORE_ERR_INVALID;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaIpcGetMemHandle(&h, dev_ptr));
    memcpy(handle, &h, 64);
    return ORE_OK;
}
extern "C" int ore_ipc_import(ore_context* ctx, const unsigned char handle[64], void** dev_ptr) {
    if (!ctx || !dev_ptr || !handle) return ORE_ERR_INVALID;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return ORE_OK;
}
extern "C" int ore_ipc_close(ore_context* ctx, void* dev_ptr) {
    if (!ctx) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaIpcCloseMemHandle(dev_ptr));
    return ORE_OK;
}
extern "C" int ore_copy_to_host(ore_context* ctx, void* host_dst, const void* dev_src, size_t bytes) {
    if (!ctx || !host_dst || !dev_src) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaMemcpyAsync(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ORE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ORE_OK;
}

extern "C" int ore_get_hits(ore_context* ctx, int32_t* hit_id_host, float* hit_t_host) {
    if (!ctx) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaDeviceSynchronize());
    if (ctx->last_px == 0) return ORE_OK;
    if (!ctx->last_prm_valid) return fail(ctx, ORE_ERR_INVALID, "ore_get_hits: no frame rendered");
    if (ctx->last_frames != 1) return fail(ctx, ORE_ERR_INVALID, "ore_get_hits: the last render was a batch (render the frame alone)");
    // the render path keeps compact hit records only; the per-pixel maps are built here, on demand
    ORE_CUDA(ctx, ctx->hit_id_map.reserve(ctx->last_px));
    ORE_CUDA(ctx, ctx->hit_t_map.reserve(ctx->last_px));
    fill_hits_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(ctx->hit_id_map, ctx->hit_t_map, ctx->last_px);
    expand_hits_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(ctx->last_prm, ctx->hit_id_map, ctx->hit_t_map);
    ORE_CUDA(ctx, cudaGetLastError());
    ORE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (hit_id_host)
        ORE_CUDA(ctx, cudaMemcpy(hit_id_host, ctx->hit_id_map, ctx->last_px * sizeof(int32_t), cudaMemcpyDeviceToHost));
    if (hit_t_host)
        ORE_CUDA(ctx, cudaMemcpy(hit_t_host, ctx->hit_t_map, ctx->last_px * sizeof(float), cudaMemcpyDeviceToHost));
    return ORE_OK;
}

extern "C" int ore_get_counters(ore_context* ctx, ore_counters* out) {
    if (!ctx || !out) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaDeviceSynchronize());
    unsigned long long c[CNT_SLOTS];
    ORE_CUDA(ctx, cudaMemcpy(c, ctx->counters, sizeof c, cudaMemcpyDeviceToHost));
    memset(out, 0, sizeof *out);
    const uint64_t batch_px = (uint64_t)ctx->last_px * (uint64_t)ctx->last_frames;
    out->pixels = batch_px;
    out->hit_pixels = batch_px ? c[CNT_HITS] : 0;
    out->primary_tests = batch_px * (uint64_t)ctx->last_n_spheres;
    out->shadow_tests_ref = c[CNT_SHADOW_TESTS_REF];
    out->sky_tests = batch_px ? batch_px - c[CNT_HITS] : 0;
    out->exact_primary = c[CNT_EXACT_PRIMARY];
    out->exact_shadow = c[CNT_EXACT_SHADOW];
    out->kernel_launches = ctx->last_launches;
    out->beam_l1 = c[CNT_BEAM_L1];
    out->beam_l2 = c[CNT_BEAM_L2];
    out->primary_steps = c[CNT_PRIMARY_STEPS];
    out->sweep_steps = c[CNT_SWEEP_STEPS];
    out->sky_exact = c[CNT_SKY_EXACT];
    return ORE_OK;
}

extern "C" int ore_get_kernel_ms(ore_context* ctx, float ms[4]) {
    if (!ctx || !ms) return ORE_ERR_INVALID;
    ms[0] = ms[1] = ms[2] = ms[3] = 0.f;
    if (!ctx->ev_end.recorded()) return ORE_OK;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, ctx->ev_end.host_wait());
    for (int i = 0; i < 4; i++)
        ORE_CUDA(ctx, cudaEventElapsedTime(&ms[i], ctx->ev[i], i < 3 ? (cudaEvent_t)ctx->ev[i + 1] : ctx->ev_end.event()));
    return ORE_OK;
}

extern "C" int ore_debug_libm(ore_context* ctx, int op, int n, const float* a_host, const float* b_host, float* out_host) {
    if (!ctx || n <= 0 || !a_host || !out_host || op < 0 || op > 6) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf<float> a, b, o;
    const size_t bytes = (size_t)n * sizeof(float);
    ORE_CUDA(ctx, a.alloc(n));
    ORE_CUDA(ctx, b.alloc(n));
    ORE_CUDA(ctx, o.alloc(n));
    // every copy on the kernel's stream: a plain cudaMemcpy from pageable memory may return before its DMA has landed,
    // and ctx->stream (non-blocking) does not wait for the legacy stream - the kernel could read part of the inputs
    // before they arrive
    ORE_CUDA(ctx, cudaMemcpyAsync(a, a_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    ORE_CUDA(ctx, cudaMemcpyAsync(b, b_host ? b_host : a_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    libm_probe_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(op, n, a, b, o);
    ORE_CUDA(ctx, cudaGetLastError());
    ORE_CUDA(ctx, cudaMemcpyAsync(out_host, o, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ORE_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ORE_OK;
}

extern "C" int ore_debug_sphere_tree(ore_context* ctx, int32_t which, void* host_out, int32_t n_items) {
    if (!ctx || which < 0 || which > 6 || n_items < 0 || (n_items > 0 && !host_out)) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaDeviceSynchronize());
    if (!ctx->sph_exact) return fail(ctx, ORE_ERR_INVALID, "ore_debug_sphere_tree: no spheres set");
    if (which == 6 && !ctx->n_hypers_pad) return fail(ctx, ORE_ERR_INVALID, "ore_debug_sphere_tree: the scene has no hyper level");
    const void* src[7] = {ctx->sph_exact, ctx->sph_xsort, ctx->sph_sort, ctx->sort_index, ctx->leaf_sph, ctx->super_sph, ctx->hyper_sph};
    const size_t count[7] = {(size_t)std::max(ctx->n_spheres, 1), (size_t)ctx->n_sort, (size_t)ctx->n_sort, (size_t)ctx->n_sort,
                             (size_t)ctx->n_leaves_pad, (size_t)ctx->n_supers_pad, (size_t)ctx->n_hypers_pad};
    if ((size_t)n_items != count[which]) return fail(ctx, ORE_ERR_INVALID, "ore_debug_sphere_tree: n_items must be the array's length");
    if (n_items > 0)
        ORE_CUDA(ctx, cudaMemcpy(host_out, src[which], (size_t)n_items * (which == 3 ? sizeof(int) : sizeof(float4)), cudaMemcpyDeviceToHost));
    return ORE_OK;
}

extern "C" int ore_debug_mesh(ore_context* ctx, int32_t which, void* host_out, int32_t n_items) {
    if (!ctx || which < 0 || which > 5 || n_items < 0 || (n_items > 0 && !host_out)) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    ORE_CUDA(ctx, cudaDeviceSynchronize());
    if (ctx->n_tris == 0) return fail(ctx, ORE_ERR_INVALID, "ore_debug_mesh: no mesh set");
    const void* src[6] = {ctx->tris, ctx->boxes, ctx->box_sph, ctx->box_offsets, ctx->box_indices, ctx->mesh_live};
    const size_t count[6] = {(size_t)ctx->n_tris * ore_host::TRI_FLOATS, 2 * (size_t)ctx->n_boxes, (size_t)ctx->n_boxes,
                             (size_t)ctx->n_boxes + 1, (size_t)ctx->mesh_n_idx, 1};
    const size_t item[6] = {sizeof(float), sizeof(float4), sizeof(float4), sizeof(int), sizeof(int), sizeof(int)};
    if ((size_t)n_items != count[which]) return fail(ctx, ORE_ERR_INVALID, "ore_debug_mesh: n_items must be the array's length");
    if (n_items > 0) ORE_CUDA(ctx, cudaMemcpy(host_out, src[which], (size_t)n_items * item[which], cudaMemcpyDeviceToHost));
    return ORE_OK;
}

extern "C" int ore_measure_fp32_peak(ore_context* ctx, double* tflops, double* sm_clock_mhz_nominal) {
    if (!ctx || !tflops) return ORE_ERR_INVALID;
    ORE_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf<float> d;
    ORE_CUDA(ctx, d.alloc(1));
    const int iters = 4096, grid = ctx->sm_count * 8;
    Event a, b;
    ORE_CUDA(ctx, cudaEventCreate(a.put()));
    ORE_CUDA(ctx, cudaEventCreate(b.put()));
    double best = 0.0;
    for (int rep = 0; rep < 6; rep++) {
        ORE_CUDA(ctx, cudaEventRecord(a, ctx->stream));
        fp32_burn_kernel<<<grid, CTA_THREADS, 0, ctx->stream>>>(d, iters, 1.0000001f, 1e-9f);
        ORE_CUDA(ctx, cudaGetLastError());
        ORE_CUDA(ctx, cudaEventRecord(b, ctx->stream));
        ORE_CUDA(ctx, cudaEventSynchronize(b));
        float ms = 0.f;
        ORE_CUDA(ctx, cudaEventElapsedTime(&ms, a, b));
        const double flop = 2.0 * 16 * 8 * (double)iters * CTA_THREADS * (double)grid;
        const double tf = flop / (ms * 1e-3) / 1e12;
        if (rep >= 1 && tf > best) best = tf;
    }
    *tflops = best;
    if (sm_clock_mhz_nominal) {
        int khz = 0;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
        *sm_clock_mhz_nominal = khz / 1000.0;
    }
    return ORE_OK;
}
