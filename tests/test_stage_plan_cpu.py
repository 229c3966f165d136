"""The staging plan of the shadow pass (csrc/ore_stage_plan.h through tests/stage_plan_probe.cpp, plain g++), no GPU: it
gives the same outputs as the block render_impl computed inline before (kept verbatim in the probe) over a grid of pixel
counts, lights, hints, existing buffers and settings, and it keeps the properties the staged kernels rely on."""
import ctypes as C
import itertools
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "ray-tracer-engine_b200", "csrc")
MAX_STAGE_CHUNKS = 32
DEFAULT_MAX_ITEMS = 8 << 20


@pytest.fixture(scope="module")
def plan_probe(tmp_path_factory):
    out = os.path.join(str(tmp_path_factory.mktemp("stage_plan")), "libstage_plan_probe.so")
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-Werror", "-shared", "-fPIC", "-I", CSRC,
                           os.path.join(ROOT, "tests", "stage_plan_probe.cpp"), "-o", out], env=env)
    lib = C.CDLL(out)
    lib.ore_probe_stage_plan.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]
    lib.ore_probe_stage_plan.restype = None

    def run(cases):
        cases = np.ascontiguousarray(cases, np.uint64)
        new = np.zeros((len(cases), 6), np.int64)
        before = np.zeros((len(cases), 6), np.int64)
        lib.ore_probe_stage_plan(cases.ctypes.data, len(cases), new.ctypes.data, before.ctypes.data)
        return new, before

    return run


def nv_of(lights):
    return 6 + 35 * lights


def grid():
    """(n_px, n_lights, fused, hint_set, hint, stage_floats, blocks_override, max_items) rows"""
    pixel_counts = [1, 31, 32, 33, 1000, 97 * 61, 200 * 150, 640 * 480, 1920 * 1080, 7680 * 4320, 8 * 7680 * 4320,
                    2**31 - 1, 2**32 - 65]   # (render_impl rejects a launch set of 2^32 - 64 pixels or more)
    rows = []
    for n_px in pixel_counts:
        nb = (n_px + 31) // 32
        hints = [(0, 0), (1, 0), (1, 17), (1, n_px), (1, 3 * n_px + 5), (1, 1 << 40), (1, 2**64 - 1)]   # unset .. stale
        capacities = [0, 32 * nv_of(3) * (nb // 7 + 1) + 5, 32 * nv_of(16) * (2 * nb + 100)]   # none, smaller, larger
        for lights, (hint_set, hint), cap, override, max_items, fused in itertools.product(
                [0, 1, 3, 16], hints, capacities, [0, 1, 40, 1 << 30], [32, DEFAULT_MAX_ITEMS, 1 << 40], [0, 1]):
            rows.append((n_px, lights, fused, hint_set, hint, cap, override, max_items))
    return np.array(rows, dtype=np.uint64)


def test_plan_equals_the_former_inline_block(plan_probe):
    cases = grid()
    new, before = plan_probe(cases)
    bad = np.nonzero(np.any(new != before, axis=1))[0]
    assert bad.size == 0, [(cases[i].tolist(), new[i].tolist(), before[i].tolist()) for i in bad[:5]]
    staged = new[:, 0] == 1
    assert np.array_equal(staged, (cases[:, 1] > 0) & (cases[:, 2] == 0))
    assert staged.sum() > 0 and new[staged, 4].any() and not new[staged, 4].all()   # with and without a catch-all


def test_plan_keeps_what_the_staged_kernels_rely_on(plan_probe):
    cases = grid()
    new, _ = plan_probe(cases)
    for c, p in zip(cases.tolist(), new.tolist()):
        n_px, lights, fused, _, _, stage_floats, override, max_items = c
        staged, need, cap, n_chunks, catch_all, catch_first = p
        if not staged:
            continue
        nv = nv_of(lights)
        nb = (n_px + 31) // 32
        assert 1 <= n_chunks <= MAX_STAGE_CHUNKS, (c, p)
        assert cap >= 1 and need % (32 * nv) == 0 and cap * 32 * nv <= need, (c, p)   # every chunk fits in the buffer
        assert (n_chunks - 1) * cap < nb, (c, p)                                      # no chunk starts past the hit list
        # the staged chunks and the catch-all cover every hit-list block, and the catch-all is there exactly when needed
        assert bool(catch_all) == (n_chunks * cap < nb), (c, p)
        if catch_all:
            assert catch_first == n_chunks * cap, (c, p)
        if not override:
            # no chunk above ORE_STAGE_MAX_ITEMS, unless the buffer already there was larger or a buffer half the size
            # would take more than MAX_STAGE_CHUNKS chunks for the pixel count
            max_blocks = (max_items + 31) // 32
            have_blocks = stage_floats // (32 * nv)
            buf_blocks = need // (32 * nv)
            assert cap <= max(max_blocks, have_blocks) or MAX_STAGE_CHUNKS * (buf_blocks // 2) < nb, (c, p)


def test_plan_follows_the_hint(plan_probe):
    """one chunk pair for the previous frame's hit count, the rest of an all-hit frame to the catch-all (the case
    test_parity_gpu.py::test_two_stage_shadow_pass_in_many_small_chunks renders)"""
    n_px = 640 * 480
    new, _ = plan_probe([(n_px, 3, 0, 1, 100, 0, 0, DEFAULT_MAX_ITEMS)])
    staged, need, cap, n_chunks, catch_all, catch_first = new[0].tolist()
    est_blocks = (100 + 100 // 8 + 32768 + 31) // 32
    assert (staged, n_chunks, cap, catch_all, catch_first) == (1, 1, est_blocks, 1, est_blocks)
    assert need == (est_blocks + est_blocks // 4) * 32 * nv_of(3)
