"""Light sets of 1-16 lights, the sweep's look-ahead, many staged chunks at 16 lights, the object texel lookup with a
texture whose every texel differs from its neighbours, and the device libm against a float64 reference.

Exact means, throughout: ids and t bit patterns equal the oracle's; the default shadow pass, FUSED_SHADOW and
EXHAUSTIVE give the same frame; and where the host libm is the one ore_libm.cuh reproduces (libm_matches), the pixels
equal the oracle's - otherwise they are within the 1-LSB bar."""
import math

import numpy as np
import pytest

from test_host_mesh import host_build, host_lib  # noqa: F401  (fixture re-export)
from test_lights_textures_cpu import light_scenes, lit_scene, texel_scene
from test_parity_gpu import assert_pixels_close, libm_matches  # noqa: F401  (fixture re-export)
from test_random_primitives_gpu import assert_oracle, mesh_probe, render_all  # noqa: F401  (fixture re-export)
from test_random_scenes_gpu import random_scene
from test_stage_plan_cpu import plan_probe  # noqa: F401  (fixture re-export)

pytestmark = pytest.mark.gpu
F32 = np.float32


# ---- A. light sets of 1-16 lights -------------------------------------------------------------------------------------

LIGHT_COUNTS = [1, 4, 5, 8, 15, 16]


@pytest.fixture(scope="module")
def scenes(pkg, host_lib, mesh_probe, tmp_path_factory):  # noqa: F811
    return {name: (sc, cam) for name, sc, cam in light_scenes(pkg, host_lib, mesh_probe, tmp_path_factory.mktemp("ls"))}


@pytest.mark.parametrize("n", LIGHT_COUNTS)
@pytest.mark.parametrize("which", ["reference", "overlap", "mixed"])
def test_light_sets_match_the_oracle(which, n, scenes, renderer, pkg, oracle_best, libm_matches):  # noqa: F811
    base, cam = scenes[which]
    sc = lit_scene(pkg, base, n, n)
    try:
        for W, H in ((97, 61), (200, 150)):
            px, ids, t = render_all(renderer, pkg, sc, cam, W, H)
            assert_oracle(px, ids, t, oracle_best.render(sc, cam, W, H), libm_matches)
            assert np.count_nonzero(px) > 0
    finally:
        renderer.set_mesh(None)


LOOK_AHEAD_ITEMS = 8192 * 32 + 32768   # a block reserves its successor only with 8192 blocks still ahead of it


@pytest.mark.parametrize("n", [3, 16])
def test_sweep_look_ahead_on_a_full_frame(n, renderer, pkg, oracle_best, libm_matches):  # noqa: F811
    """a 1280x720 frame where nearly every pixel hits: the staged sweep reserves the next block and prefetches its first
    lit light.  The frame is rendered once beforehand so that the hit-count hint gives one staged chunk holding the
    whole list (the prefetch runs only more than 8192 blocks before the end of a chunk).  A strided row sample is
    compared with the oracle - rows of the full GPU frame, since a band would be too small for the look-ahead"""
    sc, cam = random_scene(pkg, 29)
    if n != 3:
        sc = lit_scene(pkg, sc, n, 29)
    assert len(sc.lights) == n
    W, H = 1280, 720
    renderer.set_scene(sc)
    renderer.render(cam, W, H)
    px, ids, t = render_all(renderer, pkg, sc, cam, W, H)
    hits = renderer.counters()["hit_pixels"]
    print(f"{n} lights: hit_pixels {hits}")
    assert hits > LOOK_AHEAD_ITEMS, hits
    kw = dict(y0=3, y1=H, y_step=53)
    ref = oracle_best.render(sc, cam, W, H, **kw)
    rows = slice(3, H, 53)
    assert_oracle(px[rows], ids[rows], t[rows], ref, libm_matches)


def test_sixteen_lights_in_many_staged_chunks_and_the_catch_all(pkg, monkeypatch, plan_probe):  # noqa: F811
    """ORE_STAGE_MAX_ITEMS=2048 (read at ore_create) caps the staging buffer at 64 blocks of nv = 6 + 35*16 values: after
    a 16x16 frame, a 640x480 frame of 16 lights takes many staged chunk pairs and a catch-all fused launch, as
    plan_stage predicts, and equals the frame of a default context and the fused form"""
    sc, cam = random_scene(pkg, 29)
    sc = lit_scene(pkg, sc, 16, 7)
    monkeypatch.setenv("ORE_STAGE_MAX_ITEMS", "2048")
    small = pkg.Renderer(0)
    monkeypatch.delenv("ORE_STAGE_MAX_ITEMS")
    ref = pkg.Renderer(0)
    try:
        small.set_scene(sc)
        ref.set_scene(sc)
        small.render(cam, 16, 16)
        h = small.counters()["hit_pixels"]
        first = plan_probe([(16 * 16, 16, 0, 0, 0, 0, 0, 2048)])[0][0]
        a = small.render(cam, 640, 480)
        n_launch = small.counters()["kernel_launches"]
        plan = plan_probe([(640 * 480, 16, 0, 1, h, int(first[1]), 0, 2048)])[0][0]
        staged, need, cap, n_chunks, catch_all, _ = (int(v) for v in plan)
        assert staged and catch_all and n_chunks >= 4 and need >= cap * 32 * (6 + 35 * 16), plan
        print(f"16 lights, ORE_STAGE_MAX_ITEMS=2048: {n_chunks} staged chunk pairs of {cap} blocks + catch-all, "
              f"{n_launch} launches")
        assert n_launch == 2 + 2 * n_chunks + 1, (n_launch, plan.tolist(), h)   # prep, primary, chunk pairs, catch-all
        b = ref.render(cam, 640, 480)
        c = ref.render(cam, 640, 480, flags=pkg.capi.ORE_FLAG_FUSED_SHADOW)
        assert np.array_equal(a, b), int(np.count_nonzero(a != b))
        assert np.array_equal(b, c), int(np.count_nonzero(b != c))
    finally:
        small.close()
        ref.close()


def test_fast_libm_at_sixteen_lights(scenes, renderer, pkg, oracle_best):
    base, cam = scenes["reference"]
    sc = lit_scene(pkg, base, 16, 16)
    renderer.set_scene(sc)
    W, H = 200, 150
    px = renderer.render(cam, W, H, flags=pkg.capi.ORE_FLAG_FAST_LIBM)
    ids, t = renderer.hits(H, W)
    ref = oracle_best.render(sc, cam, W, H)
    assert np.array_equal(ids, ref["ids"])
    assert np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32))
    assert_pixels_close(px, ref["pixels"])


def test_sixteen_lights_after_none_equal_a_fresh_context(scenes, renderer, pkg):
    """16 rows are accepted, 17 are not; a context that rendered with one light, then none, then 16 (the staging
    buffer re-planned as nv grows from 41 to 566) gives the frame of a fresh context"""
    base, cam = scenes["reference"]
    sc = lit_scene(pkg, base, 16, 5)
    W, H = 200, 150
    renderer.set_lights(sc.lights)
    with pytest.raises(pkg.OreError):
        renderer.set_lights(np.zeros((17, 7), F32))
    fresh = pkg.Renderer(0)
    grown = pkg.Renderer(0)
    try:
        fresh.set_scene(sc)
        want = fresh.render(cam, W, H)
        grown.set_scene(sc, n_lights=1)
        one = grown.render(cam, W, H).copy()
        grown.set_lights(sc.lights[:0])
        dark = grown.render(cam, W, H).copy()
        grown.set_lights(sc.lights)
        got = grown.render(cam, W, H)
        assert np.array_equal(got, want), int(np.count_nonzero(got != want))
        assert not np.array_equal(one, want) and not np.array_equal(dark, want)
    finally:
        fresh.close()
        grown.close()


# ---- B. the object texel lookup ---------------------------------------------------------------------------------------

TEXTURE_SIZES = [(1, 1), (1, 7), (7, 1), (3, 5), (257, 129), (1024, 512), (4099, 4093)]   # (w, h); the last ~16.8 M
VT_SPECIAL = [(1.0, 1.0), (1.0, 0.0), (0.0, 1.0), (1.0, 0.5), (0.5, 1.0), (0.0, 0.0)]
VT_OUTSIDE = [(-0.3, 0.45), (1.3, 0.55), (-0.3, 0.55), (1.3, 0.45)]


def write_vt_grid_obj(path, n=9, outside=False):
    """a bumpy n x n grid (v / vt / vn / f a/b/c) inside the reference scene's cube: vt on the unit grid, exactly 0 and
    1 on its edges; every third cell takes one corner of VT_SPECIAL for all three vertices (tx, ty at 1.0: the index
    lands a row past the texture and clamp_index picks the last texel); with outside=True every fifth cell spans
    VT_OUTSIDE instead"""
    rng = np.random.default_rng(17)
    hgt = rng.uniform(0, 1.0, size=(n, n))
    vts = [(i / (n - 1), j / (n - 1)) for i in range(n) for j in range(n)]
    special0 = len(vts) + 1
    vts += VT_SPECIAL
    outside0 = len(vts) + 1
    vts += VT_OUTSIDE
    with open(path, "w") as fh:
        for i in range(n):
            for j in range(n):
                fh.write("v %.5f %.5f %.5f\n" % (1 + 0.9 * i, 4 + hgt[i, j], 1 + 0.9 * j))
        for u, v in vts:
            fh.write("vt %.5f %.5f\n" % (u, v))
        for i in range(n):
            for j in range(n):
                a = math.atan2(hgt[i, j] - 0.5, 1.0)
                fh.write("vn %.5f %.5f %.5f\n" % (math.sin(a) * 0.3, math.cos(a), math.sin(a) * 0.2))
        cell = 0
        for i in range(n - 1):
            for j in range(n - 1):
                q = [i * n + j + 1, (i + 1) * n + j + 1, (i + 1) * n + j + 2, i * n + j + 2]
                if outside and cell % 5 == 0:
                    t = [outside0 + k for k in range(4)]
                elif cell % 3 == 0:
                    t = [special0 + (cell // 3) % len(VT_SPECIAL)] * 4
                else:
                    t = q
                for f in ((0, 1, 2), (0, 2, 3)):
                    fh.write("f %s\n" % " ".join("%d/%d/%d" % (q[k], t[k], q[k]) for k in f))
                cell += 1


def vt_outside_stays_inside(w, h):
    """the reference indexes texel (int)(ty*h)*w + (int)(tx*w) with no clamp: vt outside [0, 1] is defined only where
    that index stays inside the texture for every (tx, ty) the VT_OUTSIDE cells interpolate (with a margin)"""
    us = np.linspace(-0.31, 1.31, 1001, dtype=F32)
    vs = np.linspace(0.44, 0.56, 101, dtype=F32)
    u, v = np.meshgrid(us, vs)
    idx = np.trunc(v * F32(h)).astype(np.int64) * w + np.trunc(u * F32(w)).astype(np.int64)
    return bool(idx.min() >= 0 and idx.max() < w * h)


def texel_cameras(pkg, sc):
    return [pkg.scene.Camera(org=(5.0, 14.0, 5.0), yaw=180.0, pitch=90.0),     # straight down: the upper poles
            pkg.scene.Camera(org=(5.0, -6.0, 5.0), yaw=0.0, pitch=-90.0),      # straight up: the lower poles
            pkg.scene.orbit_camera(sc, 30)]


@pytest.mark.parametrize("wh", TEXTURE_SIZES, ids=["%dx%d" % s for s in TEXTURE_SIZES])
def test_object_texels_match_the_oracle(wh, renderer, pkg, oracle_best, libm_matches, host_lib, tmp_path):  # noqa: F811
    w, h = wh
    sc = texel_scene(pkg, w, h)
    outside = vt_outside_stays_inside(w, h)
    obj = str(tmp_path / "grid.obj")
    write_vt_grid_obj(obj, outside=outside)
    sc.mesh = pkg.scene.Mesh.from_arrays(host_build(host_lib, obj))
    kinds = set()
    try:
        for cam in texel_cameras(pkg, sc):
            W, H = 128, 96
            px, ids, t = render_all(renderer, pkg, sc, cam, W, H)
            assert_oracle(px, ids, t, oracle_best.render(sc, cam, W, H), libm_matches)
            ns, nc, npl = len(sc.spheres), len(sc.cubes), len(sc.planes)
            kinds |= {("sphere", "cube", "plane", "mesh")[int(np.searchsorted([ns, ns + nc, ns + nc + npl], k, "right"))]
                      for k in np.unique(ids[ids >= 0])}
    finally:
        renderer.set_mesh(None)
    assert kinds == {"sphere", "cube", "plane", "mesh"}, kinds


# ---- C. device libm against a float64 reference ------------------------------------------------------------------------

def _ordered(x):
    i = np.ascontiguousarray(x, np.float32).view(np.int32).astype(np.int64)
    return np.where(i < 0, -(i & 0x7FFFFFFF), i)


def ulps(a, b):
    return np.abs(_ordered(a) - _ordered(b))


def test_device_libm_is_within_one_ulp_of_float64(renderer):
    """a few million inputs drawn on the device; numpy's float64 arccos / sin / cos / arctan2 of the float inputs,
    rounded to float, is the reference.  <= 1 ulp wherever ore_libm.cuh computes (|x| < 120 for sinf / cosf)"""
    import torch
    g = torch.Generator(device="cuda").manual_seed(2026)

    def draw(n, lo, hi):
        return (torch.rand(n, device="cuda", generator=g, dtype=torch.float64) * (hi - lo) + lo).float().cpu().numpy()

    n = 1 << 20
    a = np.concatenate([draw(n, -1, 1), (1 - draw(n // 4, 0, 1e-3)).astype(F32), (-1 + draw(n // 4, 0, 1e-3)).astype(F32)])
    d = ulps(renderer.debug_libm("acosf", a), np.arccos(a.astype(np.float64)).astype(F32))
    assert d.max() <= 1, ("acosf", a[np.argmax(d)], int(d.max()))
    x = np.concatenate([draw(n, -8, 8), draw(n, -120, 120)])
    x = x[np.abs(x) < 120]
    for op, f in (("sinf", np.sin), ("cosf", np.cos)):
        d = ulps(renderer.debug_libm(op, x), f(x.astype(np.float64)).astype(F32))
        assert d.max() <= 1, (op, x[np.argmax(d)], int(d.max()))
    # |x| >= 120 is CUDA's own sinf / cosf (the shading code never gets there): its documented 2-ulp bound, and no
    # glibc bits are promised there
    big = np.concatenate([draw(n // 4, 120, 1e4), -draw(n // 4, 120, 1e4)])
    for op, f in (("sinf", np.sin), ("cosf", np.cos)):
        d = ulps(renderer.debug_libm(op, big), f(big.astype(np.float64)).astype(F32))
        assert d.max() <= 2, (op, big[np.argmax(d)], int(d.max()))
    v = torch.randn(n, 3, device="cuda", generator=g)
    v = (v / v.norm(dim=1, keepdim=True)).cpu().numpy()
    scale = (10.0 ** draw(n, -3, 3)).astype(F32)
    for y, xx in ((v[:, 2].copy(), v[:, 0].copy()), ((v[:, 1] * scale).astype(F32), v[:, 2].copy())):
        d = ulps(renderer.debug_libm("atan2f", y, xx), np.arctan2(y.astype(np.float64), xx.astype(np.float64)).astype(F32))
        assert d.max() <= 1, ("atan2f", int(d.max()))
