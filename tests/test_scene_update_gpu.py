"""Stream-ordered sphere updates from device memory (ore_set_spheres_device) and the hierarchy build on the GPU
(csrc/ore_scene_build.cu): the device arrays against the host builder of csrc/ore_clusters.h byte for byte, animated
frames against the oracle, ordering across streams, no host blocking, argument validation and buffer growth."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from streamlib import _held_stream, assert_rejected
from test_parity_gpu import assert_pixels_close, libm_matches  # noqa: F401  (fixture re-export)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "ray-tracer-engine_b200", "csrc")
ARRAYS = ("sph_exact", "sph_xsort", "sph_sort", "sort_index", "leaf_sph", "super_sph")
WEIRD = [(1e17, 0, 0, 1.0), (0, -3e19, 0, 1e10), (np.inf, 0, 0, 1.0), (-np.inf, np.inf, 0, 2.0), (np.nan, 1, 1, 0.5),
         (1, 1, 1, np.nan), (5e15, 5e15, 5e15, 1e3)]


@pytest.fixture(scope="module")
def tree_probe(tmp_path_factory, pkg):
    """host reference of the six hierarchy arrays (tests/sphere_tree_probe.cpp over ore_clusters.h, plain g++)"""
    out = str(tmp_path_factory.mktemp("tree") / "libsphere_tree_probe.so")
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC,
                           os.path.join(ROOT, "tests", "sphere_tree_probe.cpp"), "-o", out], env=env)
    lib = C.CDLL(out)
    vp, i = C.c_void_p, C.c_int
    lib.ore_probe_sphere_tree.argtypes = [vp, i, vp, vp, vp, vp, vp, vp, i, i, i, i]
    lib.ore_probe_sphere_tree.restype = i

    def build(spheres):
        sp = np.ascontiguousarray(spheres, dtype=np.float32).reshape(-1, 4)
        n = len(sp)
        ln = pkg.capi.sphere_tree_lengths(n)
        out = {k: (np.zeros(ln[k], np.int32) if k == "sort_index" else np.zeros((ln[k], 4), np.float32)) for k in ARRAYS}
        src = sp if n else np.zeros((1, 4), np.float32)
        rc = lib.ore_probe_sphere_tree(src.ctypes.data, n, *[out[k].ctypes.data for k in ARRAYS],
                                       ln["sph_exact"], ln["sph_xsort"], ln["leaf_sph"], ln["super_sph"])
        assert rc == 0
        return out

    return build


def read_tree(renderer, n):
    return {k: renderer.debug_sphere_tree(k, n) for k in ARRAYS}


def assert_same_tree(got, want, what):
    for k in ARRAYS:
        a, b = got[k], want[k]
        assert a.shape == b.shape, (what, k, a.shape, b.shape)
        assert a.tobytes() == b.tobytes(), (what, k, int(np.count_nonzero(a.view(np.uint32) != b.view(np.uint32))))


def random_spheres(n, seed, extent=40.0):
    rng = np.random.default_rng(seed)
    pos = rng.uniform(0, extent, size=(n, 3)).astype(np.float32)
    member = (rng.uniform(0.05, 1.0, size=n) ** 2).astype(np.float32)
    return np.ascontiguousarray(np.concatenate([pos, member[:, None]], axis=1), dtype=np.float32)


def sphere_set(pkg, name):
    if name.startswith("n"):
        return random_spheres(int(name[1:]), 17 + int(name[1:]))
    if name == "reference_1024":
        return pkg.scene.reference_scene(1024).spheres
    if name == "scaled_1024_3":
        return pkg.scene.scaled_scene(1024, 3).spheres
    if name == "scaled_16384_5":
        return pkg.scene.scaled_scene(16384, 5).spheres
    if name == "random_60000":
        return random_spheres(60000, 60000, extent=120.0)
    if name == "duplicates":      # equal keys everywhere: the order among them is the stable sort's
        base = random_spheres(37, 5)
        sp = base[np.random.default_rng(6).integers(0, 37, size=3000)].copy()
        sp[:, 3] = np.random.default_rng(7).uniform(0.1, 1.0, size=3000).astype(np.float32)
        return np.ascontiguousarray(sp)
    if name == "collapsed":       # every axis one value
        sp = np.tile(np.array([[2.5, -1.0, 7.0, 0.3]], np.float32), (1000, 1))
        sp[:, 3] = np.linspace(0.01, 1.0, 1000, dtype=np.float32)
        return sp
    if name == "untame":
        sp = random_spheres(700, 8)
        for k, w in enumerate(WEIRD):
            sp[(k * 97 + 3) % len(sp)] = np.array(w, dtype=np.float32)
        return sp
    if name == "untame_axis":     # no tame centre on the y axis: every y key is 0
        sp = random_spheres(900, 9)
        sp[:, 1] = np.where(np.arange(900) % 2 == 0, np.float32(np.inf), np.float32(3e16))
        return sp
    raise KeyError(name)


SETS = ["n0", "n1", "n7", "n8", "n9", "n255", "n256", "n257", "n4097", "reference_1024", "scaled_1024_3", "scaled_16384_5",
        "random_60000", "duplicates", "collapsed", "untame", "untame_axis"]


def test_tree_probe_builds_on_the_cpu(tree_probe):
    """the host reference itself (no GPU): sizes and the permutation of a small set"""
    sp = random_spheres(300, 1)
    t = tree_probe(sp)
    assert sorted(t["sort_index"][:300].tolist()) == list(range(300))
    assert np.array_equal(t["sph_xsort"][:300].view(np.uint32), sp[t["sort_index"][:300]].view(np.uint32))
    assert np.all(t["sort_index"][300:] == t["sort_index"][299])
    assert np.all(t["leaf_sph"][38:, 3] == -1) and np.all(t["super_sph"][2:, 3] == -1)


# ---- 1. bit-identity of the hierarchy ----------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", SETS)
def test_device_build_is_bit_identical_to_the_host_builder(name, renderer, tree_probe, pkg):
    import torch
    sp = sphere_set(pkg, name)
    n = len(sp)
    want = tree_probe(sp)
    t = torch.from_numpy(sp.copy()).to("cuda:0") if n else torch.zeros((0, 4), dtype=torch.float32, device="cuda:0")
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    renderer.set_spheres_device(t, st.cuda_stream)
    assert_same_tree(read_tree(renderer, n), want, (name, "device"))
    renderer.set_spheres(sp)
    assert_same_tree(read_tree(renderer, n), want, (name, "host setter"))
    renderer.set_spheres_device(t)    # the context's own stream
    assert_same_tree(read_tree(renderer, n), want, (name, "render stream"))


# ---- 2. an animated sequence against the oracle -----------------------------------------------------------------------

def _moved(base, f):
    """frame f of the animation: a torch op on the stream that is current when it is called"""
    import torch
    idx = torch.arange(base.shape[0], device=base.device, dtype=torch.float32)
    out = base.clone()
    out[:, 0] += 0.35 * torch.sin(0.9 * f + 0.37 * idx)
    out[:, 1] += 0.25 * torch.cos(0.6 * f + 0.11 * idx)
    out[:, 3] *= 1.0 + 0.05 * f
    return out


def _check_frame(px, ref, libm_ok):
    assert_pixels_close(px, ref)
    if libm_ok:
        assert np.array_equal(px, ref), f"{np.count_nonzero(px != ref)} pixels differ"


def _scene_with(sc, spheres, pkg, name, extent=None):
    return pkg.scene.Scene(spheres=np.ascontiguousarray(spheres, dtype=np.float32), lights=sc.lights, texture=sc.texture,
                           sky=sc.sky, extent=sc.extent if extent is None else extent, name=name)


@pytest.mark.gpu
def test_animated_frames_equal_the_oracle(renderer, oracle_best, pkg, libm_matches):
    import torch
    sc = pkg.scene.scaled_scene(1024, 3)
    renderer.set_scene(sc)
    base = torch.from_numpy(sc.spheres.copy()).to("cuda:0")
    W, H = 128, 72                      # a small whole frame ...
    W4, H4, band = 3840, 2160, dict(y0=11, y1=2160, y_step=541)   # ... and strided rows of a 4K frame
    rows4 = pkg.Renderer.rows(H4, **band)
    n_frames = 8
    small = torch.zeros((n_frames, H, W), dtype=torch.int32, device="cuda:0")
    big = torch.zeros((n_frames, rows4, W4), dtype=torch.int32, device="cuda:0")
    cams = [pkg.scene.orbit_camera(sc, 25 * f) for f in range(n_frames)]
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    inputs = []
    with torch.cuda.stream(st):
        for f in range(n_frames):
            cur = _moved(base, f)
            inputs.append(cur.clone())          # this frame's spheres, kept on the device
            renderer.set_spheres_device(cur, st.cuda_stream)
            renderer.render_device(cams[f], W, H, small[f].data_ptr(), stream=st.cuda_stream)
            renderer.render_device(cams[f], W4, H4, big[f].data_ptr(), stream=st.cuda_stream, **band)
    st.synchronize()                             # the first host synchronisation
    small_px, big_px = small.cpu().numpy().view(np.uint32), big.cpu().numpy().view(np.uint32)
    F = pkg.capi
    for f in range(n_frames):
        spheres = inputs[f].cpu().numpy()
        scf = _scene_with(sc, spheres, pkg, f"anim{f}")
        ref = oracle_best.render(scf, cams[f], W, H)
        _check_frame(small_px[f], ref["pixels"], libm_matches)
        ref4 = oracle_best.render(scf, cams[f], W4, H4, **band)
        _check_frame(big_px[f], ref4["pixels"], libm_matches)
        # ids and t bits of this frame's spheres through the device build
        renderer.set_spheres_device(inputs[f])
        px = renderer.render(cams[f], W, H)
        assert np.array_equal(px, small_px[f])
        ids, t = renderer.hits(H, W)
        assert np.array_equal(ids, ref["ids"]) and np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32)), f
        px4 = renderer.render(cams[f], W4, H4, **band)
        assert np.array_equal(px4, big_px[f])
        ids4, t4 = renderer.hits(rows4, W4)
        assert np.array_equal(ids4, ref4["ids"]) and np.array_equal(t4.view(np.uint32), ref4["t"].view(np.uint32)), f
        assert (ids >= 0).any()
        if f == 3:
            for flags in (F.ORE_FLAG_EXHAUSTIVE, F.ORE_FLAG_FUSED_SHADOW):
                assert np.array_equal(renderer.render(cams[f], W4, H4, flags=flags, **band), px4), flags
    renderer.set_scene(sc)


# ---- 3. ordering across streams ---------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_update_on_another_stream_is_ordered_between_renders(renderer, pkg):
    import torch
    sc = pkg.scene.scaled_scene(1024, 3)
    W, H = 7680, 4320
    cam = pkg.scene.orbit_camera(sc, 40)
    b_np = sc.spheres.copy()
    b_np[:, :3] = b_np[:, [2, 0, 1]]          # scene B: the same spheres, axes permuted
    b_np[:, 3] *= np.float32(1.3)
    renderer.set_scene(sc)
    want_a = renderer.render(cam, W, H).copy()
    renderer.set_spheres(b_np)
    want_b = renderer.render(cam, W, H).copy()
    assert np.count_nonzero(want_a != want_b) > 1000
    renderer.set_spheres(sc.spheres)
    scene_b = torch.from_numpy(b_np).to("cuda:0")
    T, S = torch.cuda.Stream(), torch.cuda.Stream()
    frames = torch.zeros((2, H, W), dtype=torch.int32, device="cuda:0")
    torch.cuda.synchronize()
    renderer.render_device(cam, W, H, frames[0].data_ptr(), stream=T.cuda_stream)
    renderer.set_spheres_device(scene_b, S.cuda_stream)
    renderer.render_device(cam, W, H, frames[1].data_ptr(), stream=T.cuda_stream)
    T.synchronize()
    got = frames.cpu().numpy().view(np.uint32)
    assert np.array_equal(got[0], want_a), int(np.count_nonzero(got[0] != want_a))
    assert np.array_equal(got[1], want_b), int(np.count_nonzero(got[1] != want_b))
    # a batch of 8 cameras after an update equals 8 single frames
    cams = [pkg.scene.orbit_camera(sc, 30 * f + 7) for f in range(8)]
    Wb, Hb = 480, 270
    renderer.set_spheres_device(scene_b, S.cuda_stream)
    batch = torch.zeros((8, Hb, Wb), dtype=torch.int32, device="cuda:0")
    T.wait_stream(torch.cuda.current_stream())
    renderer.render_batch_device(cams, Wb, Hb, [batch[i].data_ptr() for i in range(8)], stream=T.cuda_stream)
    T.synchronize()
    got = batch.cpu().numpy().view(np.uint32)
    for i, c in enumerate(cams):
        assert np.array_equal(got[i], renderer.render(c, Wb, Hb)), i
    renderer.set_scene(sc)


# ---- 4. no host blocking -----------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_update_with_capacity_does_not_block_the_host(renderer, tree_probe, pkg):
    import torch
    sp = pkg.scene.scaled_scene(4096, 2).spheres
    sp2 = sp.copy()
    sp2[:, 0] += np.float32(0.5)
    renderer.set_spheres(sp)                   # sizes the buffers for 4096 spheres
    t2 = torch.from_numpy(sp2).to("cuda:0")
    dt, pending = _held_stream(renderer, lambda s: renderer.set_spheres_device(t2, s))
    assert dt < 0.5, dt
    assert pending, "the update must still be waiting behind the held stream"
    assert_same_tree(read_tree(renderer, len(sp2)), tree_probe(sp2), "after release")


# ---- 5. validation ---------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_invalid_pointers_are_rejected_and_change_nothing(renderer, pkg):
    import torch
    sc = pkg.scene.reference_scene(64, 1)
    cam = pkg.scene.reference_camera()
    renderer.set_scene(sc)
    want = renderer.render(cam, 160, 120).copy()
    other = torch.from_numpy(pkg.scene.reference_scene(64, 2).spheres).to("cuda:0")
    lib, ctx = renderer.lib, renderer.ctx
    host = np.ascontiguousarray(pkg.scene.reference_scene(64, 2).spheres)
    pinned = renderer.host_alloc((64, 4), dtype=np.float32)
    pinned[:] = host
    raw = torch.zeros(64 * 4 + 4, dtype=torch.float32, device="cuda:0")
    try:
        bad = [(host.ctypes.data, 64), (pinned.ctypes.data, 64), (raw.data_ptr() + 4, 64), (other.data_ptr(), -1),
               (0, 64)]
        if torch.cuda.device_count() > 1:
            bad.append((torch.from_numpy(host).to("cuda:1").data_ptr(), 64))
        assert_rejected(lambda ptr, n: lib.ore_set_spheres_device(ctx, ptr or None, n, None), bad,
                        lambda: renderer.render(cam, 160, 120), want)
        # the Python binding checks before the call
        for t, err in ((other.double(), TypeError), (other[:, :3].contiguous(), ValueError), (other.cpu(), ValueError),
                       (other.t().contiguous().t(), ValueError), (host, TypeError)):
            with pytest.raises(err):
                renderer.set_spheres_device(t)
        assert np.array_equal(renderer.render(cam, 160, 120), want)
    finally:
        renderer.host_free(pinned)


# ---- 6. growth ---------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_growth_and_shrink_render_correctly(renderer, tree_probe, oracle_best, pkg, libm_matches):
    import torch
    sc = pkg.scene.scaled_scene(64, 2)
    renderer.set_scene(sc)
    F = pkg.capi
    for n in (64, 5000, 64, 70000):
        sp = random_spheres(n, n + 3, extent=10.0 * (n / 64.0) ** (1.0 / 3.0))
        t = torch.from_numpy(sp).to("cuda:0")
        torch.cuda.synchronize()
        renderer.set_spheres_device(t)
        assert_same_tree(read_tree(renderer, n), tree_probe(sp), n)
        scn = _scene_with(sc, sp, pkg, f"grow{n}", extent=10.0 * (n / 64.0) ** (1.0 / 3.0))
        cam = pkg.scene.orbit_camera(scn, 50)
        W, H = 96, 54
        px = renderer.render(cam, W, H)
        ids, tt = renderer.hits(H, W)
        assert (ids >= 0).any()
        assert np.array_equal(renderer.render(cam, W, H, flags=F.ORE_FLAG_EXHAUSTIVE), px), n
        if n <= 5000:
            ref = oracle_best.render(scn, cam, W, H)
            assert np.array_equal(ids, ref["ids"]) and np.array_equal(tt.view(np.uint32), ref["t"].view(np.uint32)), n
            _check_frame(px, ref["pixels"], libm_matches)
    renderer.set_scene(sc)
