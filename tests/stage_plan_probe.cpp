// Test-only C wrapper over csrc/ore_stage_plan.h (plain g++): plan_stage for a batch of inputs, and beside it the
// staging plan render_impl computed inline before it moved to that header, kept verbatim as the reference
// (tests/test_stage_plan_cpu.py compares the two).
#include "ore_stage_plan.h"

#include <cstddef>
#include <cstdint>

using namespace ore;

// Outputs per case, 6 x int64: staged, floats the chunks need, chunk capacity in blocks, chunk count, catch-all
// present, catch-all first block.  Only the first is meaningful when the pass is not staged (the rest are 0).
static void put(long long* o, bool staged, size_t need, size_t cap_blocks, int n_chunks, bool catch_all, size_t catch_all_block) {
    if (!staged) need = cap_blocks = n_chunks = 0, catch_all = false, catch_all_block = 0;
    o[0] = staged;
    o[1] = (long long)need;
    o[2] = (long long)cap_blocks;
    o[3] = n_chunks;
    o[4] = catch_all;
    o[5] = catch_all ? (long long)catch_all_block : 0;
}

// The block of render_impl (staging plan and launch loop) before the plan moved to ore_stage_plan.h, with the
// context's fields as arguments, the allocation taken as successful and the launches reduced to their arguments.
static void plan_before(size_t n_px, int n_lights, bool fused, bool hits_hint_set, unsigned long long hint, size_t stage_cap,
                        size_t stage_blocks_override, size_t stage_max_items, long long* out) {
    const bool have_stage = stage_cap > 0;
    const int st_nv = STAGE_HEADER + STAGE_PER_LIGHT * n_lights;
    const size_t n_blocks_px = (n_px + 31) / 32;
    bool staged = !fused;
    size_t cap_blocks = 0, est_blocks = n_blocks_px;
    size_t need = 0;
    if (n_lights == 0) {
        staged = false;
    } else if (staged) {
        size_t est_items;
        if (hits_hint_set) {
            // previous frame's hit count + 12.5 % + 32 K items; the catch-all below covers a wrong guess
            const unsigned long long h = hint;
            est_items = (size_t)(h + h / 8 + 32768ull);
        } else {
            // no frame of this context has finished yet: half the pixels (growing the buffer later costs a
            // device-wide synchronisation; the cap below bounds the memory)
            est_items = n_px / 2 > ((size_t)1 << 20) ? n_px / 2 : ((size_t)1 << 20);
        }
        if (est_items > n_px) est_items = n_px;
        est_blocks = (est_items + 31) / 32;
        // the staging buffer never grows past stage_max_items (448 bytes each with three lights: 3.6 GB); a longer hit
        // list - a batch of several 8K frames - is walked in chunk pairs of that size, each a full-size launch
        const size_t max_blocks = (stage_max_items + 31) / 32;
        const size_t have_blocks = have_stage ? stage_cap / (32 * (size_t)st_nv) : 0;
        cap_blocks = have_blocks;
        if (stage_blocks_override) {
            cap_blocks = stage_blocks_override;
            while ((n_blocks_px + cap_blocks - 1) / cap_blocks > (size_t)MAX_STAGE_CHUNKS) cap_blocks *= 2;
        } else if (est_blocks > have_blocks && have_blocks < max_blocks) {
            cap_blocks = est_blocks + est_blocks / 4;   // grow with some slack: reallocations stay rare
            if (cap_blocks > n_blocks_px) cap_blocks = n_blocks_px;
            if (cap_blocks > max_blocks) cap_blocks = max_blocks;
        }
        while ((est_blocks + cap_blocks - 1) / cap_blocks > (size_t)MAX_STAGE_CHUNKS) cap_blocks *= 2;
        need = cap_blocks * 32 * (size_t)st_nv;
    }
    if (n_lights == 0 || !staged) {
        put(out, false, 0, 0, 0, false, 0);
        return;
    }
    int n_chunks = (int)((est_blocks + cap_blocks - 1) / cap_blocks);
    if (n_chunks < 1) n_chunks = 1;
    // equal chunks: the expected hit list is split evenly instead of into full buffers plus a small remainder
    if (!stage_blocks_override) cap_blocks = (est_blocks + n_chunks - 1) / n_chunks;
    const uint32_t st_cap_blocks = (uint32_t)cap_blocks;
    const int n_chunks_max = (int)((n_blocks_px + cap_blocks - 1) / cap_blocks);
    if (n_chunks > n_chunks_max) n_chunks = n_chunks_max;
    const uint32_t rest_first_block = (uint32_t)((size_t)n_chunks * cap_blocks);
    put(out, true, need, st_cap_blocks, n_chunks, n_chunks < n_chunks_max, rest_first_block);
}

// in: n cases of 8 x uint64 (n_px, n_lights, fused, hint_set, hint, stage_floats, blocks_override, max_items);
// out / out_before: n cases of 6 x int64 (see put)
extern "C" void ore_probe_stage_plan(const unsigned long long* in, long long n, long long* out, long long* out_before) {
    for (long long i = 0; i < n; i++) {
        const unsigned long long* c = in + 8 * i;
        const StagePlan p = plan_stage(c[0], (int)c[1], c[2] != 0, c[3] != 0, c[4], c[5], c[6], c[7]);
        put(out + 6 * i, p.staged, p.need_floats, p.cap_blocks, p.n_chunks, p.catch_all, p.catch_all_block);
        plan_before(c[0], (int)c[1], c[2] != 0, c[3] != 0, c[4], c[5], c[6], c[7], out_before + 6 * i);
    }
}
