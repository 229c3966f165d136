// ore_stage_plan.h - how one frame's shadow pass uses the staging buffer: fused or two-stage, how large the buffer must
// be, how many staged chunk pairs to launch and where the catch-all fused launch starts.  Host arithmetic only (no CUDA
// types): render_impl (ore_capi.cu) runs it every frame, tests/stage_plan_probe.cpp compiles it with plain g++, and the
// layout constants below are the kernels' own (ore_kernels.cuh includes this header).
#ifndef ORE_STAGE_PLAN_H
#define ORE_STAGE_PLAN_H
#include <cstddef>
#include <cstdint>

namespace ore {

constexpr int MAX_STAGE_CHUNKS = 32;   // per-chunk cursor slots of the staged kernels (CNT_STAGE_A0 / CNT_STAGE_B0)

// Staging buffer between shade_setup_kernel and the staged shadow_sweep_kernel: blocks of 32 hit-list items,
// value-major inside a block (value v of lane i at (block * nv + v) * 32 + i, so every access is one coalesced
// 128-byte line and a light's 30 direction components are one contiguous 3840-byte piece for a TMA bulk copy).
// Values: 0-2 start, 3-5 texel r,g,b, then 35 per light: cone axis (3), cone min-dot (-1: degenerate bundle),
// a = dot(normal, toL), 30 direction components.
constexpr int STAGE_HEADER = 6;
constexpr int STAGE_PER_LIGHT = 35;

struct StagePlan {
    bool staged = false;       // two-stage pass; false: one fused sweep (or, without lights, no sweep at all)
    size_t need_floats = 0;    // staging buffer the chunks need: a smaller buffer is re-allocated at this size
    size_t cap_blocks = 0;     // staged chunk capacity in 32-item blocks
    int n_chunks = 0;          // staged chunk pairs, chunk c starting at hit-list block c * cap_blocks
    bool catch_all = false;    // hit-list blocks from catch_all_block on are swept by one fused launch
    size_t catch_all_block = 0;
};

// n_px: pixels of the launch set (>= 1).  hint: hit count of the context's previous frame (any value is safe: a wrong
// guess only moves work between the staged chunks and the catch-all); hint_set false before the first frame.
// stage_floats: capacity of the current staging buffer (0: none).  blocks_override: ORE_STAGE_BLOCKS (0: unset).
// max_items: ORE_STAGE_MAX_ITEMS, the largest buffer the hint may ask for, in hit pixels.
//
// Normally ONE chunk pair per frame.  The buffer holds the expected hit list (hint + 12.5 % + 32 K items; half the
// pixels, at least 1 M, before the first frame has finished) with 25 % slack, never more than max_items unless
// MAX_STAGE_CHUNKS chunks would not cover the expected list; a longer list is split into equal chunks.
inline StagePlan plan_stage(size_t n_px, int n_lights, bool fused, bool hint_set, unsigned long long hint,
                            size_t stage_floats, size_t blocks_override, size_t max_items) {
    StagePlan p;
    p.staged = !fused && n_lights > 0;
    if (!p.staged) return p;
    const size_t nv = STAGE_HEADER + STAGE_PER_LIGHT * (size_t)n_lights;
    const size_t n_blocks_px = (n_px + 31) / 32;
    size_t est_items = hint_set ? (size_t)(hint + hint / 8 + 32768ull) : (n_px / 2 > ((size_t)1 << 20) ? n_px / 2 : ((size_t)1 << 20));
    if (est_items > n_px) est_items = n_px;
    const size_t est_blocks = (est_items + 31) / 32;
    const size_t max_blocks = (max_items + 31) / 32;
    const size_t have_blocks = stage_floats / (32 * nv);
    size_t cap_blocks = have_blocks;
    if (blocks_override) {
        cap_blocks = blocks_override;
        while ((n_blocks_px + cap_blocks - 1) / cap_blocks > (size_t)MAX_STAGE_CHUNKS) cap_blocks *= 2;
    } else if (est_blocks > have_blocks && have_blocks < max_blocks) {
        cap_blocks = est_blocks + est_blocks / 4;   // grow with some slack: reallocations stay rare
        if (cap_blocks > n_blocks_px) cap_blocks = n_blocks_px;
        if (cap_blocks > max_blocks) cap_blocks = max_blocks;
    }
    while ((est_blocks + cap_blocks - 1) / cap_blocks > (size_t)MAX_STAGE_CHUNKS) cap_blocks *= 2;
    p.need_floats = cap_blocks * 32 * nv;
    int n_chunks = (int)((est_blocks + cap_blocks - 1) / cap_blocks);
    if (n_chunks < 1) n_chunks = 1;
    // equal chunks: the expected hit list is split evenly instead of into full buffers plus a small remainder
    if (!blocks_override) cap_blocks = (est_blocks + n_chunks - 1) / n_chunks;
    const int n_chunks_max = (int)((n_blocks_px + cap_blocks - 1) / cap_blocks);
    if (n_chunks > n_chunks_max) n_chunks = n_chunks_max;
    p.cap_blocks = cap_blocks;
    p.n_chunks = n_chunks;
    p.catch_all = n_chunks < n_chunks_max;
    p.catch_all_block = (size_t)n_chunks * cap_blocks;
    return p;
}

}  // namespace ore

#endif
