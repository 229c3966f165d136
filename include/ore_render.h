/* ore_render.h - C ABI of the B200-native render hot path (libore_b200.so).
 *
 * Drop-in boundary for ONE path of OpenRayAi (leonZtiger/Ray-Tracer-engine): the
 * per-pixel render kernel `rayTrace` and the host code that launches it.  Plain C
 * types only (pointers + sizes); no torch / C++ types cross this boundary.
 *
 * Each entry point names the reference interface it replaces (file:line in the
 * reference tree).  The C++ shims that keep the reference's own symbols
 * (`onStart()`, `update()`, `memManager`, `sprite`) on top of this ABI live in
 * ray-tracer-engine_b200/host/; INTEGRATION.md shows the binding a maintainer adds.
 *
 * Error convention: every call returns an int status (ORE_OK == 0).  The reference
 * prints and exit(99)s on any CUDA error (memManager.cpp:3-11); that behaviour is
 * kept in the C++ shim layer, not here.  There is NO CPU fallback: if no CUDA
 * device / kernel image is usable the calls fail with ORE_ERR_CUDA.
 */
#ifndef ORE_RENDER_H
#define ORE_RENDER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORE_ABI_VERSION 2

enum ore_status {
    ORE_OK = 0,
    ORE_ERR_INVALID = 1, /* bad argument / call order            */
    ORE_ERR_CUDA = 2,    /* CUDA runtime error (see ore_last_error) */
    ORE_ERR_NOMEM = 3
};

/* render flags */
enum ore_flags {
    ORE_FLAG_NONE = 0,
    /* Debug: evaluate the reference's exact intersection sequence for EVERY ray/sphere
     * pair instead of filter + exact re-adjudication.  Same results, much slower; used
     * by the parity tests to prove the filter never drops a hit. */
    ORE_FLAG_EXHAUSTIVE = 1,
    /* Also count, per frame, the sphere::intersect calls the REFERENCE's loop order
     * would make in castLightRay (first blocker index + 1, or N) - the "tests" of the
     * algorithmic rate (SURVEY.md 8d).  Costs one extra kernel; off on the timed path. */
    ORE_FLAG_COUNT_REFERENCE_TESTS = 2,
    /* Use CUDA's own cosf/sinf/acosf/atan2f instead of the glibc-bit-compatible device functions of the default
     * path (csrc/ore_libm.cuh).  ~10 % faster; ids and t unchanged; pixels within 1 LSB of the default on
     * >= 99.9 % (measured 99.999 %) instead of bit-identical to the host-compiled reference. */
    ORE_FLAG_FAST_LIBM = 16,
    /* Shadow pass as ONE kernel (shading set-up + light directions + sweep in one warp program) instead of the
     * two-stage pass through a staging buffer.  Same results; slower (its hot code does not fit the SM instruction
     * cache) but needs no staging memory.  Also what the catch-all launch runs and what a failed staging allocation
     * falls back to. */
    ORE_FLAG_FUSED_SHADOW = 32,
    /* Do not record the per-kernel CUDA events behind ore_get_kernel_ms for this call (five event records per
     * frame; throughput loops set this, ore_get_kernel_ms then reports zeros). */
    ORE_FLAG_NO_KERNEL_TIMING = 64,
    /* Band DMA (opt-in; ore_render_device / ore_render_batch_device with out_pitch == width).  The primary kernel writes
     * its rows into a packed local band buffer, a copy engine moves them to their place in the destination frames behind
     * the primary kernel and beside stage A of the shadow pass, and only the hit pixels are stored by the sweep.  Meant
     * for a rank whose frames live in ANOTHER GPU's memory.  Measured on 8 x B200 (profiles/r02_scaling.md) it is no
     * faster than storing every pixel from the kernels - the presenter's NVLink ingress is the limit either way - so
     * nothing selects it automatically. */
    ORE_FLAG_BAND_DMA = 128
};

typedef struct ore_context ore_context; /* opaque; owns device buffers, streams, pinned staging */

/* Layout-compatible with the reference's `camera` passed BY VALUE to rayTrace
 * (kernel.cu:237-262,1615): ray::Org @0, ray::Dir @12, aspect @24, Camyaw @28,
 * Campitch @32 - 36 bytes.  Dir and aspect are never read by the kernel. */
typedef struct ore_camera {
    float org[3];
    float dir[3];
    float aspect;
    float yaw;   /* degrees */
    float pitch; /* degrees */
} ore_camera;

/* One frame (or one row band of it).  Rows rendered: y0, y0+y_step, ... < y1 (see y_block), in
 * GLOBAL image coordinates (dy depends on the global row, kernel.cu:1625); output
 * row k is image row y0 + k*y_step, `width` pixels each, 0x00RRGGBB (rgbToInt,
 * kernel.cu:546-556), row 0 = bottom scanline on screen (window.cpp:43). */
typedef struct ore_frame {
    int32_t width, height;
    int32_t y0, y1, y_step; /* full frame: 0, height, 1 */
    float aspect;           /* the global `aspect` = tan(fov/2), kernel.cu:1701.  The eye sits at z = -1/aspect
                               (kernel.cu:1629) and the image plane spans dx in [-1, 2*aspect - 1],
                               dy in [-1, 2*aspect*height/width - 1].  0, +-inf, NaN and aspects whose
                               reciprocal is not finite return ORE_ERR_INVALID.  A negative aspect is
                               accepted (the view looks backwards, as the reference's would).  The tests
                               cover |aspect| from 1e-3 to 1e3 and aspect = -tan(45 deg). */
    uint32_t flags;         /* ore_flags */
    int32_t out_pitch;      /* ore_render_device only.  0: rendered rows are stored packed (row k of the
                               output = k-th rendered row).  > 0: pitch in pixels of ONE IMAGE ROW of the
                               destination; rendered rows are stored at their image position relative to
                               y0 (row y goes to out + (y - y0)*out_pitch).  A rank that renders its rows
                               straight into the presenter's frame passes out = frame + y0*width and
                               out_pitch = width. */
    int32_t y_block;        /* 0 or 1: single rows y0, y0+y_step, ...; B > 1: blocks of B consecutive rows
                               starting at y0, y0+y_step, ... (B <= y_step).  Block-interleaving keeps the
                               8-row pixel tiles of the primary kernel compact when rows are dealt to P GPUs:
                               rank r uses y0 = 8r, y_step = 8P, y_block = 8. */
} ore_frame;

/* counters of the last ore_render* call */
typedef struct ore_counters {
    uint64_t pixels;          /* pixels rendered                                          */
    uint64_t hit_pixels;      /* pixels whose primary ray hit a sphere                    */
    uint64_t primary_tests;   /* pixels * n_spheres (reference count, data independent)   */
    uint64_t shadow_tests_ref;/* reference-order shadow tests (only with COUNT flag)      */
    uint64_t sky_tests;       /* miss pixels (one sky-sphere test each)                   */
    uint64_t exact_primary;   /* exact re-adjudications executed, primary phase           */
    uint64_t exact_shadow;    /* exact re-adjudications executed, shadow phase            */
    uint64_t kernel_launches; /* kernels launched by the call                             */
    uint64_t beam_l1;         /* spheres passing the warp-level beam test (sum over warps, lights, groups) */
    uint64_t beam_l2;         /* (pixel, sphere, light) triples passing the per-pixel cone test */
    uint64_t primary_steps;   /* warp steps of the primary sweep: 32 tile-cone tests each (super / leaf / sphere) */
    uint64_t sweep_steps;     /* warp steps of the shadow sweep: 32 beam tests each                */
    uint64_t sky_exact;       /* miss pixels whose sky texel needed the exact sequence (near a texel boundary / a pole) */
} ore_counters;

/* ---- lifetime ---------------------------------------------------------------------
 * Replaces the static initialisers + onStart() that build the global scene
 * (kernel.cu:1692-1714) and the implicit default-stream context. `device` is the CUDA
 * ordinal.  One context per GPU; calls on one context must not overlap. */
int ore_create(ore_context** out, int device);
int ore_destroy(ore_context* ctx);
int ore_abi_version(void);
const char* ore_last_error(const ore_context* ctx); /* "" if none */

/* ---- scene upload (memManager / object side) --------------------------------------
 * All uploads copy from caller memory through the context's pinned staging buffer
 * into structure-of-arrays device buffers; the caller's memory is not retained. */

/* Replaces object::sphereAllocMem (kernel.cu:1208-1212): n records of cx,cy,cz and the
 * stored `radius` MEMBER (= ctor r*r, kernel.cu:287; squared again in the test :334). */
int ore_set_spheres(ore_context* ctx, const float* xyz_radius, int32_t n);
/* Same, from the reference's own 32-byte AoS records (vptr@0, orgin@8, reflective@20,
 * radius@24; `sizeof(float)*8` per sphere, kernel.cu:1218-1220). */
int ore_set_spheres_aos32(ore_context* ctx, const void* records, int32_t n);
/* Stream-ordered sphere update from DEVICE memory (an animated scene: a simulation or a torch model moving the spheres
 * on the GPU).  `xyz_radius_dev`: n records of cx, cy, cz, radius member - the meaning of ore_set_spheres - in device
 * memory of the context's GPU, 16-byte aligned (NULL allowed when n == 0).  Host memory, another GPU's memory, a
 * misaligned pointer or n < 0 return ORE_ERR_INVALID and change nothing.
 *   Ordering: the update is enqueued on `stream` (a cudaStream_t, NULL = the context's render stream).  It runs after
 *   every render already submitted through this context and after the previous update, on whatever streams they ran,
 *   and every render or scene setter submitted afterwards, on any stream, sees the new spheres.
 *   Host blocking: none, unless n needs more room than every earlier upload of this context: the scene buffers then
 *   grow, which first waits on the host for the last render and the last update.  A caller that sizes the buffers
 *   once with its largest n (one call with that n) never blocks afterwards.
 *   Caller's buffer: it must stay allocated and unchanged until the update has run on `stream` (the rules of
 *   cudaMemcpyAsync); the context does not keep it.
 *   Result: the device arrays are bit-identical to what ore_set_spheres builds for the same values, so every result
 *   guarantee of the render calls holds unchanged. */
int ore_set_spheres_device(ore_context* ctx, const float* xyz_radius_dev, int32_t n, void* stream);
/* "Next" primitives of castRay / castLightRay (SURVEY.md 8f N1).  The reference ships both counts at 0
 * (kernel.cu:1231).  Hit ids continue after the spheres: cube i -> n_spheres + i, plane i -> n_spheres +
 * n_cubes + i.  Exact tests, no filters: meant for the handful of objects the reference would hold.
 * Replaces object::cubeAllocMem (kernel.cu:1224-1228): n x {c1.xyz, c2.xyz} = the `cube(c1, c2)` ctor
 * arguments (kernel.cu:391-396; orgin = (c1+c2)/2 is derived here as the ctor does). */
int ore_set_cubes(ore_context* ctx, const float* c1_c2, int32_t n);
/* Replaces object::planeAllocMem (kernel.cu:1213-1217, which copies ONE plane; any count is accepted here):
 * n x {pos.xyz, normal.xyz} = the `plane(pos, normal)` ctor arguments (kernel.cu:364-367). */
int ore_set_planes(ore_context* ctx, const float* pos_normal, int32_t n);
/* Triangle mesh with its flat BVH (SURVEY.md 8f N2), exactly as the reference's `mesh` holds it once its OBJ
 * loader and createBvhMesh() have run on the host (kernel.cu:577-936) and mesh::allocMem / Bvhbox::AllocMem would
 * copy it (kernel.cu:999-1017, 528-535): the loader and the builder stay on the host, this call replaces the copy.
 *   tris27      : n_tris x 27 floats = `triangle` {points[3], normal, vecNormal[3], vt[3]} (kernel.cu:206-212)
 *   has_normals : mesh::has_normals
 *   box_bounds6 : n_boxes x {bounds[0].xyz, bounds[1].xyz} of each leaf's `bvhbox` cube.  A box need not contain
 *                 its triangles: the render then still equals the reference's (DESIGN.md 6c)
 *   box_offsets : n_boxes + 1; leaf j holds box_indices[box_offsets[j] .. box_offsets[j+1])  (Bvhbox::indexes/length)
 * Hit ids continue after spheres, cubes and planes: triangle i -> n_spheres + n_cubes + n_planes + i.
 * Exact tests, linear scan over the leaves per ray like the reference (kernel.cu:1293-1328,1475-1497).
 * n_tris == 0 or n_boxes == 0 removes the mesh.  Otherwise a NULL array, box_offsets[0] != 0, offsets that do not
 * ascend, a listed index outside [0, n_tris) or more than INT32_MAX / 27 triangles return ORE_ERR_INVALID and change
 * nothing: the previous mesh and the capacity the device setters reached stay. */
int ore_set_mesh(ore_context* ctx, const float* tris27, int32_t n_tris, int32_t has_normals, const float* box_bounds6,
                 const int32_t* box_offsets, const int32_t* box_indices, int32_t n_boxes);
/* Stream-ordered update of the mesh's triangles from DEVICE memory (a deforming mesh: skinning, cloth, a displaced
 * height field computed on the GPU).  `tris27_dev`: n_tris x 27 floats - the meaning of ore_set_mesh's tris27 - in
 * device memory of the context's GPU, 4-byte aligned.  The topology of the last ore_set_mesh stays: has_normals,
 * box_offsets and box_indices; n_tris must equal its triangle count.  No mesh set, a wrong n_tris, a NULL, misaligned
 * or host pointer, or another GPU's memory return ORE_ERR_INVALID and change nothing.
 *   Leaf boxes: recomputed on the GPU from the new triangles by the reference builder's rule (getMinMaxP,
 *   kernel.cu:973-997): lo seeded with the first listed triangle's first vertex, hi with the last listed triangle's
 *   first vertex, then every vertex of every listed triangle grows them in list order with strict > / <.  A leaf that
 *   lists no triangle keeps its box.  Their bounding spheres follow by the formula ore_set_mesh uses.
 *   Ordering and host blocking: as ore_set_spheres_device (the same events).  The update is enqueued on `stream`
 *   (NULL = the context's render stream) after every render already submitted and the previous update; renders
 *   submitted afterwards, on any stream, see the new triangles.  The host never blocks: nothing grows.
 *   Caller's buffer: it must stay allocated and unchanged until the update has run on `stream`. */
int ore_set_mesh_triangles_device(ore_context* ctx, const float* tris27_dev, int32_t n_tris, void* stream);
/* Stream-ordered replacement of the whole mesh from DEVICE memory, with the flat BVH built on the GPU (GPU-generated or
 * strongly deformed geometry, a changing triangle count).  `tris27_dev`: n_tris >= 1 records of ore_set_mesh's tris27
 * in device memory of the context's GPU, 4-byte aligned; has_normals is taken as != 0.  The leaves are exactly what the
 * reference's createBvhMesh (kernel.cu:782-936) - and ore_build_flat_bvh in host/ore_mesh.cpp - gives for these
 * triangles: the same leaf order, the same index order within each leaf and the same bits of every box, so every result
 * guarantee of ore_set_mesh carries over.  (Removing the mesh stays ore_set_mesh(ctx, NULL, 0, ...).)  n_tris < 1, a
 * NULL, misaligned or host pointer, or another GPU's memory return ORE_ERR_INVALID and change nothing.
 *   Leaf count: decided on the device.  The context holds min(1024, n_tris) leaves; those past the live count list no
 *   triangles and are never visited.  ore_set_mesh_triangles_device afterwards refits this topology.
 *   Ordering: as ore_set_spheres_device (the same events): enqueued on `stream` (NULL = the context's render stream)
 *   after every render already submitted and the previous update; renders and setters submitted afterwards, on any
 *   stream, see the new mesh.
 *   Host blocking: none while n_tris fits the mesh capacity - the largest mesh either setter uploaded since the mesh was
 *   last removed.  Growing it first waits on the host for the last render and the last update.
 *   Caller's buffer: it must stay allocated and unchanged until the update has run on `stream`. */
int ore_set_mesh_device(ore_context* ctx, const float* tris27_dev, int32_t n_tris, int32_t has_normals, void* stream);
/* Replaces cudaMalloc+cudaMemcpy of `lights` in update() (kernel.cu:1776-1778):
 * n x {pos.xyz, size, r, g, b} (kernel.cu:1246-1261). */
int ore_set_lights(ore_context* ctx, const float* lights7, int32_t n);
/* Replaces `objs->texture = new sprite(tex)` (kernel.cu:1201): sprite planes
 * (sprite.h:29-45; value = byte/255, row-major y*width+x, Sprite.cpp:41-46). */
int ore_set_texture(ore_context* ctx, const float* r, const float* g, const float* b,
                    int32_t width, int32_t height);
/* Replaces `new skybox(img, size)` (kernel.cu:1120-1123,1700). */
int ore_set_sky(ore_context* ctx, const float* r, const float* g, const float* b,
                int32_t width, int32_t height, float size);

/* ---- render ------------------------------------------------------------------------
 * Replaces the body of update(): rayTrace<<<...>>> + cudaDeviceSynchronize +
 * setPixelBuff (kernel.cu:1780-1788, window.cpp:130-132).
 *
 * ore_render        : `out_host` is HOST memory (pageable or pinned); synchronous; the
 *                     device->host copy of the band is part of the call.
 * ore_render_device : `out_device` is DEVICE memory on the context's GPU (or a peer-
 *                     mapped pointer); asynchronous on `stream` (a cudaStream_t, NULL =
 *                     the context's own stream); no host copies. */
int ore_render(ore_context* ctx, const ore_camera* cam, const ore_frame* frame, uint32_t* out_host);
int ore_render_device(ore_context* ctx, const ore_camera* cam, const ore_frame* frame,
                      uint32_t* out_device, void* stream);
int ore_synchronize(ore_context* ctx);
/* A BATCH of frames in one launch set: n_frames (1..8) cameras over the same scene, size and row band, frame f into
 * out_device[f].  Same pixels as n_frames single calls.  Every kernel of the pass then sees n_frames times the work
 * units, so launch latencies and the tail of each launch are paid once per batch - what decides throughput when one
 * rank of a multi-GPU job only holds an eighth of a frame (the reference renders one frame per update(); an orbit or
 * any scripted camera path can be submitted a few frames at a time).  ore_get_hits needs a single-frame render. */
int ore_render_batch_device(ore_context* ctx, const ore_camera* cams, int32_t n_frames, const ore_frame* frame,
                            uint32_t* const* out_device, void* stream);

/* Pipelined presentation (throughput mode of update()): frame f is copied to the host on a second stream
 * while frame f+1 renders into the other of two device framebuffers.  `out_host` should be pinned
 * (ore_host_alloc) for the copy to be asynchronous; it is valid after ore_wait() or after the second
 * following ore_render_async call.  Same pixels as ore_render. */
int ore_render_async(ore_context* ctx, const ore_camera* cam, const ore_frame* frame, uint32_t* out_host);
int ore_wait(ore_context* ctx);
/* Rows in place: with frame->out_pitch == frame->width, `out_host` is image row y0 of a FULL host frame and every
 * rendered row is copied to its image position (y_block / y_step honoured: one strided copy of the row blocks).
 * This is how the ranks of a multi-GPU job each send their own rows to ONE shared pinned host frame - the buffer
 * setPixelBuff reads (window.cpp:130-132) - over their own PCIe link.  out_pitch == 0 keeps the packed layout.
 * ore_render_async_signal additionally writes `done_value` to `*done_flag` (registered host memory or device
 * memory) in stream order AFTER the copy has landed, without blocking the caller. */
int ore_render_async_signal(ore_context* ctx, const ore_camera* cam, const ore_frame* frame, uint32_t* out_host,
                            uint32_t* done_flag, uint32_t done_value);
/* The batch form of ore_render_async(_signal): frame f is copied to out_host[f]; when done_flag is not NULL,
 * first_done_value + f is stored there once frame f's copy has landed (frames land in order). */
int ore_render_batch_async(ore_context* ctx, const ore_camera* cams, int32_t n_frames, const ore_frame* frame,
                           uint32_t* const* out_host, uint32_t* done_flag, uint32_t first_done_value);
/* Pin caller memory (e.g. a POSIX shared-memory frame mapped by every rank) for asynchronous copies and flags. */
int ore_host_register(ore_context* ctx, void* host_ptr, size_t bytes);
int ore_host_unregister(ore_context* ctx, void* host_ptr);
/* pinned host memory for framebuffers (the shim's `pixels` handed to setPixelBuff) */
int ore_host_alloc(ore_context* ctx, size_t bytes, void** host_ptr);
int ore_host_free(ore_context* ctx, void* host_ptr);

/* ---- device buffers for multi-GPU presentation --------------------------------------
 * The reference has one GPU and one managed `pixels` buffer per frame (kernel.cu:1775).
 * With row bands over several GPUs (one process each) the presenting GPU owns the frame;
 * it is exported with CUDA IPC so the other ranks' kernels store their rows into it
 * directly over NVLink (ore_render_device with out_pitch).  Plain cudaMalloc memory. */
int ore_dev_alloc(ore_context* ctx, size_t bytes, void** dev_ptr);
int ore_dev_free(ore_context* ctx, void* dev_ptr);
int ore_ipc_export(ore_context* ctx, void* dev_ptr, unsigned char handle[64]);
int ore_ipc_import(ore_context* ctx, const unsigned char handle[64], void** dev_ptr);
int ore_ipc_close(ore_context* ctx, void* dev_ptr);
/* Stream-ordered 32-bit flags: the completion / back-pressure signals of multi-GPU presentation, in place of a
 * collective.  ore_flag_write stores `value` to `*flag` after everything already enqueued on `stream` (NULL = the
 * context's render stream; ore_get_stream(ctx, 1) = its copy stream) has completed; ore_flag_wait_geq makes later
 * work on `stream` wait until (int32)(*flag - value) >= 0.  `flag` may be device memory of this GPU, registered
 * host memory, or - for writes - a peer GPU's memory imported with ore_ipc_import (stored over NVLink).  Neither
 * call blocks the host.  Implemented with cuStreamWriteValue32 / cuStreamWaitValue32 (no SM involved); a one-thread
 * kernel is the fallback for peer addresses and for drivers without stream memory operations. */
int ore_flag_write(ore_context* ctx, void* stream, uint32_t* flag, uint32_t value);
int ore_flag_wait_geq(ore_context* ctx, void* stream, const uint32_t* flag, uint32_t value);
/* Like ore_flag_write, but the store is issued from the context's in-order signal stream once the work enqueued on
 * `stream` so far is complete: flags written through one context appear in CALL order even when frames rendered on
 * different streams (several frames in flight) finish out of order. */
int ore_flag_write_after(ore_context* ctx, void* stream, uint32_t* flag, uint32_t value);
void* ore_get_stream(ore_context* ctx, int which); /* 0: render stream, 1: copy stream, 2: signal stream (cudaStream_t) */
/* device -> host copy on the context's stream, synchronous (the setPixelBuff copy) */
int ore_copy_to_host(ore_context* ctx, void* host_dst, const void* dev_src, size_t bytes);

/* ---- introspection of the LAST render (parity tests, roofline accounting) ---------
 * hit_id: nearest primitive or -1 (castRay, kernel.cu:1330-1372; spheres, then cubes, then planes); hit_t: nearest t,
 * +inf on miss.  Packed like the pixels.  Either pointer may be NULL.  The render path itself keeps one compact
 * (pixel, id, t) record per HIT pixel; the per-pixel maps are expanded from them inside this call. */
int ore_get_hits(ore_context* ctx, int32_t* hit_id_host, float* hit_t_host);
int ore_get_counters(ore_context* ctx, ore_counters* out);
/* average device time (ms) of each kernel of the last render, measured with CUDA events
 * on the launching stream: [0] frame prep, [1] primary, [2] shadow+shade, [3] count */
int ore_get_kernel_ms(ore_context* ctx, float ms[4]);
/* Measures the FP32 roofline denominator on this GPU with an FFMA burn (TFLOP/s, best of 5)
 * and returns the nominal SM clock; used by bench.py only. */
int ore_measure_fp32_peak(ore_context* ctx, double* tflops, double* sm_clock_mhz_nominal);
/* Tests only: evaluates the device libm the path uses on n host inputs.
 * op 0 cosf(a), 1 sinf(a), 2 acosf(a), 3 atan2f(a, b).  The path's versions return glibc's bits (ore_libm.cuh).
 * op 4, 5, 6: x, y, z of the path's normalise() applied to (a[i], b[i], a[(i + 1) % n]) - IEEE x / |v| bit for bit. */
int ore_debug_libm(ore_context* ctx, int op, int n, const float* a_host, const float* b_host, float* out_host);
/* Tests only: synchronises the device and copies one array of the sphere hierarchy to the host.  which: 0 records in
 * original order (max(n, 1) float4), 1 exact records sorted (n_sort float4), 2 shadow records cx,cy,cz,R' sorted
 * (n_sort float4), 3 sorted position -> original index (n_sort int32), 4 leaf balls (n_leaves_pad float4), 5 super-
 * cluster balls (n_supers_pad float4); n_sort = 32 ceil(n / 32) (32 when n = 0), n_leaves_pad = ceil(n / 8) rounded up
 * to a multiple of 32, n_supers_pad = ceil(n / 256) rounded up to a multiple of 4.  n_items must be that length. */
int ore_debug_sphere_tree(ore_context* ctx, int32_t which, void* host_out, int32_t n_items);
/* Tests only: synchronises the device and copies one array of the mesh to the host.  which: 0 triangles (n_tris * 27
 * floats), 1 leaf boxes lo, hi (2 * n_boxes float4, .w = 0), 2 leaf bounding spheres (n_boxes float4), 3 leaf offsets
 * (n_boxes + 1 int32), 4 leaf indices (n_idx int32: box_offsets[n_boxes] of ore_set_mesh, n_tris after
 * ore_set_mesh_device), 5 the live leaf count (1 int32).  n_boxes is ore_set_mesh's, or min(1024, n_tris) after
 * ore_set_mesh_device.  n_items must be that length. */
int ore_debug_mesh(ore_context* ctx, int32_t which, void* host_out, int32_t n_items);

#ifdef __cplusplus
}
#endif
#endif /* ORE_RENDER_H */
