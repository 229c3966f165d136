"""Large scenes (99 073 to 2^24 spheres): the hyper-cluster level built on the device against the host builder byte for
byte, the large-scene kernels against today's kernels (forced onto small scenes with ORE_LARGE_SCENE_MIN_SPHERES),
against the exhaustive mode and against the oracle, batches, bands and stream-ordered updates at 1M spheres, and the
limit of 2^24 spheres."""
import os

import numpy as np
import pytest

import cases
from test_hyper_clusters_cpu import load_probe, spheres
from test_random_scenes_gpu import random_scene

pytestmark = pytest.mark.gpu

LIMIT = 1 << 24
SENTINEL = np.uint32(0xDEADBEEF)


@pytest.fixture(scope="module")
def hyper_probe(tmp_path_factory):
    return load_probe(tmp_path_factory.mktemp("hyper_gpu"))


@pytest.fixture(scope="module")
def large_renderer(pkg):
    """a second context whose every non-empty scene takes the large-scene path"""
    pkg.build.build_library()
    old = os.environ.get("ORE_LARGE_SCENE_MIN_SPHERES")
    os.environ["ORE_LARGE_SCENE_MIN_SPHERES"] = "1"
    try:
        r = pkg.Renderer(0)
    finally:
        if old is None:
            del os.environ["ORE_LARGE_SCENE_MIN_SPHERES"]
        else:
            os.environ["ORE_LARGE_SCENE_MIN_SPHERES"] = old
    yield r
    r.close()


def big_scene(pkg, n, seed, weird=False):
    """n spheres at scaled_scene's density (numpy draws: the LCG loop of scaled_scene is slow at millions), with
    scaled_scene's lights, texture and sky, and an orbit camera"""
    sc = pkg.scene
    sp = spheres(n, seed, weird=weird)
    extent = 10.0 * (n / 64.0) ** (1.0 / 3.0)
    base = sc.scaled_scene(64, seed % 7 + 1)
    lights = base.lights.copy()
    lights[:, :4] *= np.float32(extent / 10.0)
    s = sc.Scene(spheres=sp, lights=lights, texture=base.texture, sky=base.sky, extent=extent, name=f"big{n}_{seed}")
    return s, sc.orbit_camera(s, 17 * seed % 240)


def frame_of(r, cam, W, H, **kw):
    px = r.render(cam, W, H, **kw).copy()
    rows = px.shape[0]
    ids, t = r.hits(rows, W)
    return px, ids, t


def assert_same_frame(a, b, what):
    assert np.array_equal(a[1], b[1]), (what, "ids", int(np.count_nonzero(a[1] != b[1])))
    assert np.array_equal(a[2].view(np.uint32), b[2].view(np.uint32)), (what, "t")
    assert np.array_equal(a[0], b[0]), (what, "pixels", int(np.count_nonzero(a[0] != b[0])))


def assert_oracle_close(px, ids, t, ref):
    assert np.array_equal(ids, ref["ids"])
    assert np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32))
    d = np.zeros(px.shape, dtype=np.int32)
    for sh in (0, 8, 16):
        d = np.maximum(d, np.abs(((px >> sh) & 255).astype(np.int32) - ((ref["pixels"] >> sh) & 255).astype(np.int32)))
    assert np.count_nonzero(d <= 1) >= 0.999 * d.size


# ---- 1. the hyper level on the device ----------------------------------------------------------------------------------

@pytest.mark.parametrize("n", [99073, 131072, 1000003, LIMIT])
def test_device_hyper_balls_equal_the_host_builder(n, renderer, hyper_probe, pkg):
    import torch
    sp = spheres(n, n, weird=True)
    _, want_sup, want_hyp = hyper_probe(sp)
    ln = pkg.capi.sphere_tree_lengths(n)
    renderer.set_spheres(sp)
    assert renderer.debug_sphere_tree("super_sph", n).tobytes() == want_sup.tobytes()
    assert renderer.debug_sphere_tree("hyper", n).tobytes() == want_hyp.tobytes(), ("host setter", n)
    assert ln["hyper"] == len(want_hyp)
    t = torch.from_numpy(sp).to("cuda:0")
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    renderer.set_spheres_device(t, st.cuda_stream)
    assert renderer.debug_sphere_tree("hyper", n).tobytes() == want_hyp.tobytes(), ("device setter", n)
    del t
    torch.cuda.empty_cache()


def test_small_scenes_have_no_hyper_level(renderer, large_renderer, pkg):
    sp = spheres(99072, 1)
    renderer.set_spheres(sp)
    with pytest.raises(pkg.capi.OreError):
        renderer.debug_sphere_tree("hyper", len(sp))
    large_renderer.set_spheres(sp[:300])
    assert large_renderer.debug_sphere_tree("hyper", 300).shape == (4, 4)


# ---- 2. the large-scene kernels forced onto small scenes: the same frames as today's kernels ---------------------------

MODES = [0, 32, 1]   # default, fused shadow pass, exhaustive (ORE_FLAG_FUSED_SHADOW = 32, ORE_FLAG_EXHAUSTIVE = 1)


@pytest.mark.parametrize("seed", list(range(24)))
def test_forced_large_path_equals_the_default_path_on_random_scenes(seed, renderer, large_renderer, pkg):
    sc, cam = random_scene(pkg, seed)
    renderer.set_scene(sc)
    large_renderer.set_scene(sc)
    for fast in (0, pkg.capi.ORE_FLAG_FAST_LIBM):
        for mode in MODES:
            a = frame_of(renderer, cam, 97, 61, flags=mode | fast)
            b = frame_of(large_renderer, cam, 97, 61, flags=mode | fast)
            assert_same_frame(a, b, (seed, mode | fast))


GOLDEN = ["S64_f0_161x91", "R1024_inside_96x54", "S1024_f100_band", "S16384_f0_64x36", "R1_one_sphere_64x48",
          "S64_cubes_plane_f0_160x90", "R16_cubes_plane_torus_128x96"]


@pytest.mark.parametrize("name", GOLDEN)
def test_forced_large_path_equals_the_default_path_on_golden_cases(name, renderer, large_renderer, pkg):
    _, make, W, H, kw = next(c for c in cases.SMALL if c[0] == name)
    sc, cam = make()
    renderer.set_scene(sc)
    large_renderer.set_scene(sc)
    for fast in (0, pkg.capi.ORE_FLAG_FAST_LIBM):
        for mode in MODES:
            a = frame_of(renderer, cam, W, H, flags=mode | fast, **kw)
            b = frame_of(large_renderer, cam, W, H, flags=mode | fast, **kw)
            assert_same_frame(a, b, (name, mode | fast))


# ---- 3. default == fused == exhaustive on large scenes -----------------------------------------------------------------

def _exhaustive_equality(renderer, sc, cam, W=64, H=40):
    renderer.set_scene(sc)
    a = frame_of(renderer, cam, W, H)
    assert np.count_nonzero(a[1] >= 0) > 0, "the frame must hit something"
    for mode in (32, 1):
        assert_same_frame(a, frame_of(renderer, cam, W, H, flags=mode), (sc.name, mode))


@pytest.mark.parametrize("weird", [False, True], ids=["tame", "untame"])
@pytest.mark.parametrize("n", [99073, 131072, 400000])
def test_default_equals_exhaustive_on_large_random_scenes(n, weird, renderer, pkg):
    sc, cam = big_scene(pkg, n, 3 + n % 11, weird=weird)
    _exhaustive_equality(renderer, sc, cam)


@pytest.mark.parametrize("n", [99073, 131072])
def test_default_equals_exhaustive_on_scaled_scenes(n, renderer, pkg):
    sc = pkg.scene.scaled_scene(n, 5)
    _exhaustive_equality(renderer, sc, pkg.scene.orbit_camera(sc, 40))


def test_default_equals_exhaustive_with_cubes_plane_and_torus(renderer, pkg):
    sc, cam = big_scene(pkg, 131072, 9)
    sc = pkg.scene.with_cubes_and_plane(sc, 12, 4)
    sc.mesh = cases.torus_mesh()
    _exhaustive_equality(renderer, sc, cam)
    renderer.set_mesh(None)


# ---- 4. the oracle on a row subset of a 1M-sphere scene ---------------------------------------------------------------

def test_one_million_spheres_match_the_oracle(renderer, oracle_best, pkg):
    sc, cam = big_scene(pkg, 1 << 20, 2)
    renderer.set_scene(sc)
    W, H, y0, y1, y_step = 48, 27, 3, 27, 12   # rows 3 and 15: 96 pixels
    px, ids, t = frame_of(renderer, cam, W, H, y0=y0, y1=y1, y_step=y_step)
    ref = oracle_best.render(sc, cam, W, H, y0=y0, y1=y1, y_step=y_step)
    assert np.count_nonzero(ids >= 0) > 0
    assert_oracle_close(px, ids, t, ref)


# ---- 5. batches, bands and stream-ordered updates at 1M spheres ---------------------------------------------------------

def test_batch_of_eight_equals_single_renders_at_one_million(renderer, pkg):
    import torch
    sc, _ = big_scene(pkg, 1 << 20, 4)
    renderer.set_scene(sc)
    cams = [pkg.scene.orbit_camera(sc, 30 * k) for k in range(8)]
    W, H = 96, 54
    frames = torch.full((8, H, W), int(SENTINEL.view(np.int32)), dtype=torch.int32, device="cuda:0")
    renderer.render_batch_device(cams, W, H, [frames[i].data_ptr() for i in range(8)])
    torch.cuda.synchronize()
    batch = frames.cpu().numpy().view(np.uint32)
    for k, c in enumerate(cams):
        assert np.array_equal(batch[k], renderer.render(c, W, H)), k


def test_band_equals_the_rows_of_the_full_frame_at_one_million(renderer, pkg):
    sc, cam = big_scene(pkg, 1 << 20, 6)
    renderer.set_scene(sc)
    W, H = 128, 256
    full = renderer.render(cam, W, H).copy()
    band = renderer.render(cam, W, H, y0=0, y1=H, y_step=64, y_block=8)
    rows = [y for y in range(H) if y % 64 < 8]
    assert np.array_equal(band, full[rows])


def test_device_updates_equal_the_host_setter_at_one_million(renderer, pkg):
    import torch
    sc, cam = big_scene(pkg, 1 << 20, 8)
    renderer.set_scene(sc)
    base = torch.from_numpy(sc.spheres).to("cuda:0")
    idx = torch.arange(base.shape[0], device="cuda:0", dtype=torch.float32)
    W, H = 64, 40
    for f in range(5):
        moved = base.clone()
        moved[:, 1] += 0.4 * torch.sin(0.7 * f + 0.013 * idx)
        renderer.set_spheres_device(moved, torch.cuda.current_stream().cuda_stream)
        a = frame_of(renderer, cam, W, H)
        host = moved.cpu().numpy()
        renderer.set_spheres(host)
        b = frame_of(renderer, cam, W, H)
        assert_same_frame(a, b, ("frame", f))


# ---- 6. the limit -------------------------------------------------------------------------------------------------------

def test_two_to_the_24_spheres_render_and_one_more_is_refused(renderer, pkg):
    sc, cam = big_scene(pkg, LIMIT, 5)
    renderer.set_scene(sc)
    W, H = 32, 16
    a = frame_of(renderer, cam, W, H)
    assert np.count_nonzero(a[1] >= 0) > 0
    assert_same_frame(a, frame_of(renderer, cam, W, H, flags=32), "fused at 2^24")
    one_more = np.concatenate([sc.spheres, sc.spheres[:1]])
    renderer.set_spheres(one_more)
    out = np.full((H, W), SENTINEL, dtype=np.uint32)
    with pytest.raises(pkg.capi.OreError, match="2\\^24"):
        renderer.render(cam, W, H, out=out)
    assert np.all(out == SENTINEL), "a refused render writes nothing"
    renderer.set_spheres(np.zeros((0, 4), np.float32))
