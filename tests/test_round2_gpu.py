"""Round-2 GPU tests (through the C ABI): parity at the stated sizes of BASELINE.json's configs, the C ABI v2
additions (stream-ordered flags, rows-in-place asynchronous copies, registered host memory), the mesh upload with
unaligned section sizes, and the drop-in shim against the ORACLE."""
import json
import math
import os
import subprocess
import time

import numpy as np
import pytest

from test_parity_gpu import assert_pixels_close, libm_matches  # noqa: F401  (fixture re-export)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "ray-tracer-engine_b200", "host")


def _exact(px, ref, libm_ok):
    assert_pixels_close(px, ref)
    if libm_ok:
        assert np.array_equal(px, ref), f"{np.count_nonzero(px != ref)} pixels differ"


# ---- BASELINE.json configs at their stated sizes (VERDICT r01 "missing" 7) --------------------------------------

def test_config0_640x480_reference_scene_full_frame(renderer, oracle_best, pkg, libm_matches):
    """configs[0]: 640x480 single frame, R(64,1), the reference's camera - every pixel, id and t of the frame"""
    sc, cam = pkg.scene.reference_scene(64, 1), pkg.scene.reference_camera()
    renderer.set_scene(sc)
    px = renderer.render(cam, 640, 480)
    ids, t = renderer.hits(480, 640)
    ref = oracle_best.render(sc, cam, 640, 480)
    assert np.array_equal(ids, ref["ids"])
    assert np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32))
    _exact(px, ref["pixels"], libm_matches)


@pytest.mark.parametrize("scene_kind", ["S64_2", "R64_1"])
def test_config1_1920x1080_full_frame(scene_kind, renderer, oracle_best, pkg, libm_matches):
    """configs[1]: 1920x1080, 64 spheres - the whole frame against the oracle (S(64,2) orbit frame 0 and R(64,1))"""
    if scene_kind == "S64_2":
        sc = pkg.scene.scaled_scene(64, 2)
        cam = pkg.scene.orbit_camera(sc, 0)
    else:
        sc, cam = pkg.scene.reference_scene(64, 1), pkg.scene.reference_camera()
    renderer.set_scene(sc)
    px = renderer.render(cam, 1920, 1080)
    ids, t = renderer.hits(1080, 1920)
    ref = oracle_best.render(sc, cam, 1920, 1080)
    assert np.array_equal(ids, ref["ids"])
    assert np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32))
    _exact(px, ref["pixels"], libm_matches)


@pytest.mark.parametrize("frame", [0, 60, 120, 180])
def test_config2_4k_orbit_frames_row_subsets(frame, renderer, oracle_best, pkg, libm_matches):
    """configs[2] (SURVEY 8d config 3): 3840x2160, S(1024,3), orbit frames {0,60,120,180}, strided row subsets"""
    W, H = 3840, 2160
    sc = pkg.scene.scaled_scene(1024, 3)
    cam = pkg.scene.orbit_camera(sc, frame)
    renderer.set_scene(sc)
    kw = dict(y0=7 + frame % 11, y1=H, y_step=269)
    px = renderer.render(cam, W, H, **kw)
    ids, t = renderer.hits(px.shape[0], W)
    ref = oracle_best.render(sc, cam, W, H, **kw)
    assert np.array_equal(ids, ref["ids"])
    assert np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32))
    _exact(px, ref["pixels"], libm_matches)


def test_config3_8k_rows_ids_t_and_pixels(renderer, oracle_best, pkg, libm_matches):
    """configs[3] size (7680x4320): ids, t BITS and pixels of a strided row sample"""
    W, H = 7680, 4320
    sc = pkg.scene.scaled_scene(1024, 3)
    cam = pkg.scene.orbit_camera(sc, 77)
    renderer.set_scene(sc)
    kw = dict(y0=5, y1=H, y_step=617)
    px = renderer.render(cam, W, H, **kw)
    ids, t = renderer.hits(px.shape[0], W)
    ref = oracle_best.render(sc, cam, W, H, **kw)
    assert np.array_equal(ids, ref["ids"])
    assert np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32))
    _exact(px, ref["pixels"], libm_matches)


def test_config4_16384_spheres_more_rows(renderer, oracle_best, pkg, libm_matches):
    """configs[4] scene at 4K: six rows spread over the frame (two orbit frames) against the oracle"""
    W, H = 3840, 2160
    sc = pkg.scene.scaled_scene(16384, 5)
    renderer.set_scene(sc)
    for frame, kw in ((0, dict(y0=300, y1=H, y_step=700)), (130, dict(y0=650, y1=H, y_step=600))):
        cam = pkg.scene.orbit_camera(sc, frame)
        px = renderer.render(cam, W, H, **kw)
        ids, t = renderer.hits(px.shape[0], W)
        ref = oracle_best.render(sc, cam, W, H, **kw)
        assert np.array_equal(ids, ref["ids"])
        assert np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32))
        _exact(px, ref["pixels"], libm_matches)


# ---- mesh upload: section sizes that are not multiples of 16 bytes (ADVICE r01, high) ---------------------------

@pytest.mark.parametrize("n", [4, 5, 9])
def test_mesh_upload_with_unaligned_sections(n, renderer, oracle_best, pkg, tmp_path, libm_matches):
    """grid meshes whose triangle / box / index counts leave the staging sections 4-byte aligned only"""
    import ctypes as C
    from test_host_mesh import host_build, write_grid_obj

    subprocess.check_call(["make", "-s", "-C", HOST])
    lib = C.CDLL(os.path.join(HOST, "libore_host.so"), mode=os.RTLD_LAZY)
    obj = str(tmp_path / f"grid{n}.obj")
    write_grid_obj(obj, "vtn", n=n)
    d = host_build(lib, obj)
    mesh = pkg.scene.Mesh.from_arrays(d)
    assert mesh.n_tris == 2 * (n - 1) ** 2
    sc = pkg.scene.reference_scene(16, 3)
    sc.mesh = mesh
    cam = pkg.scene.reference_camera()
    try:
        renderer.set_scene(sc)
        px = renderer.render(cam, 160, 120)
        ids, t = renderer.hits(120, 160)
        ref = oracle_best.render(sc, cam, 160, 120)
        assert np.array_equal(ids, ref["ids"])
        assert np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32))
        _exact(px, ref["pixels"], libm_matches)
        assert (ids >= 16).any(), "the mesh must be visible in the frame"
    finally:
        renderer.set_mesh(None)


# ---- C ABI v2: flags, rows in place, registered host memory ----------------------------------------------------

def _read_u32(renderer, dev_ptr):
    out = np.zeros(1, dtype=np.uint32)
    renderer.copy_to_host(out, dev_ptr)
    return int(out[0])


def test_stream_flags_write_wait_and_order(renderer, pkg):
    import torch
    flag = renderer.dev_alloc(256)
    try:
        assert _read_u32(renderer, flag) == 0
        renderer.flag_write(flag, 5)
        renderer.synchronize()
        assert _read_u32(renderer, flag) == 5
        # a wait that is already satisfied does not block
        renderer.flag_wait_geq(flag, 3)
        renderer.flag_wait_geq(flag, 5)
        renderer.synchronize()
        # a stream blocked on a flag runs its work only after another stream has written it
        sc, cam = pkg.scene.reference_scene(16, 3), pkg.scene.reference_camera()
        renderer.set_scene(sc)
        want = renderer.render(cam, 96, 64)
        s1 = torch.cuda.Stream()
        frame = torch.zeros((64, 96), dtype=torch.int32, device="cuda:0")
        renderer.flag_wait_geq(flag, 7, s1.cuda_stream)
        renderer.render_device(cam, 96, 64, frame.data_ptr(), stream=s1.cuda_stream)
        time.sleep(0.05)
        assert not s1.query(), "the stream must still be waiting for the flag"
        renderer.flag_write(flag, 7)          # context's own stream
        s1.synchronize()
        assert np.array_equal(frame.cpu().numpy().view(np.uint32), want)
        # ordered writes from several streams: values appear in call order
        s2 = torch.cuda.Stream()
        for g, st in enumerate((s1, s2, s1, s2)):
            renderer.render_device(cam, 96, 64, frame.data_ptr(), stream=st.cuda_stream)
            renderer.flag_write_after(flag, 100 + g, st.cuda_stream)
        torch.cuda.synchronize()
        assert _read_u32(renderer, flag) == 103
    finally:
        renderer.synchronize()
        renderer.dev_free(flag)


def test_flag_write_kernel_fallback(pkg, monkeypatch):
    """ORE_NO_STREAM_MEMOPS=1: the one-thread st.release.sys kernel writes the flag (what peer addresses use)"""
    monkeypatch.setenv("ORE_NO_STREAM_MEMOPS", "1")
    r = pkg.Renderer(0)
    try:
        flag = r.dev_alloc(256)
        r.flag_write(flag, 42)
        r.synchronize()
        assert _read_u32(r, flag) == 42
        host = r.host_alloc((16,))
        host[:] = 0
        r.flag_write(host.ctypes.data, 9)
        r.synchronize()
        assert int(host[0]) == 9
        r.host_free(host)
        r.dev_free(flag)
    finally:
        r.close()


def test_rows_in_place_into_one_host_frame(renderer, pkg):
    """every "rank" copies its block-interleaved rows straight to their image position in ONE pinned host frame and
    stamps its completion counter behind the copy (all ranks on one GPU here)"""
    mg = pkg.multigpu
    sc = pkg.scene.scaled_scene(64, 2)
    cam = pkg.scene.orbit_camera(sc, 33)
    renderer.set_scene(sc)
    W, H, P = 333, 203, 3
    want = renderer.render(cam, W, H)
    frame = renderer.host_alloc((H, W))
    flags = renderer.host_alloc((64,))
    frame[:] = 0
    flags[:] = 0
    try:
        for rank in range(P):
            b = mg.block_band(rank, P, H)
            renderer.render_async(cam, W, H, out=frame.ctypes.data + 4 * W * b["y0"], in_place=True,
                                  done_flag=flags.ctypes.data + 64 * rank, done_value=rank + 11, **b)
        renderer.wait()
        assert np.array_equal(frame, want)
        assert [int(flags[16 * r]) for r in range(P)] == [11, 12, 13]
        # a contiguous band in place, and the packed layout still works
        frame[:] = 0
        renderer.render_async(cam, W, H, out=frame.ctypes.data + 4 * W * 50, in_place=True, y0=50, y1=120)
        renderer.wait()
        assert np.array_equal(frame[50:120], want[50:120]) and not frame[:50].any() and not frame[120:].any()
        with pytest.raises(pkg.OreError):   # rows in place need out_pitch == width
            f = renderer._frame(W, H, 0, H, 1, None, 0, W + 8, 1)
            c = renderer._cam(cam)
            import ctypes as C
            renderer._check(renderer.lib.ore_render_async(renderer.ctx, C.byref(c), C.byref(f), frame.ctypes.data), "ore_render_async")
    finally:
        renderer.wait()
        renderer.host_free(frame)
        renderer.host_free(flags)


def test_shared_host_frame_registered_and_written_by_the_gpu(renderer, pkg):
    """POSIX shared memory pinned with ore_host_register: the ring protocol of multigpu.SharedHostFrame with the GPU as
    the producer of every rank's rows (ranks emulated on one GPU, one after the other)"""
    mg = pkg.multigpu
    sc = pkg.scene.scaled_scene(64, 2)
    renderer.set_scene(sc)
    W, H, P, NB = 200, 90, 2, 2
    owner = mg.SharedHostFrame(W, H, 0, P, n_buffers=NB, register=renderer.host_register, unregister=renderer.host_unregister)
    other = mg.SharedHostFrame(W, H, 1, P, n_buffers=NB, name=owner.name)   # same mapping, second rank's view
    owner.touch_own_rows()      # several ranks: every rank touches its rows first, then the ring is pinned
    other.touch_own_rows()
    owner.pin()
    try:
        shown = []
        for g in range(5):
            cam = pkg.scene.orbit_camera(sc, g)
            for view in (owner, other):
                assert view.can_submit()
                gg, buf = view.next_slot()
                assert gg == g
                b = view.band()
                renderer.render_async(cam, W, H, out=owner.row_addr(buf, b["y0"]), in_place=True,
                                      done_flag=owner.done_addr(view.rank), done_value=g + 1, **b)
            t0 = time.time()
            while not owner.ready():
                assert time.time() - t0 < 20
            owner.present(lambda fr, f: shown.append(np.array_equal(fr, renderer.render(pkg.scene.orbit_camera(sc, f), W, H))))
            assert other.consumed == g + 1
        assert shown == [True] * 5
    finally:
        renderer.wait()
        other.close()
        owner.close()


def test_empty_band_of_a_short_frame_and_band_past_the_image(renderer, pkg):
    cam = pkg.scene.reference_camera()
    renderer.set_scene(pkg.scene.reference_scene(4, 1))
    b = pkg.multigpu.block_band(7, 8, 20)          # 8 ranks, 20 rows: rank 7 owns nothing
    assert renderer.render(cam, 64, 20, **b).shape == (0, 64)
    with pytest.raises(pkg.OreError):
        renderer.render(cam, 64, 20, y0=0, y1=21)   # past the image: rejected, not written


def test_sync_render_after_async_without_wait(renderer, pkg):
    """ore_render issued right behind ore_render_async (no ore_wait) must not clobber the frame still being copied"""
    sc = pkg.scene.scaled_scene(64, 2)
    renderer.set_scene(sc)
    W, H = 640, 360
    a_want = renderer.render(pkg.scene.orbit_camera(sc, 1), W, H).copy()
    b_want = renderer.render(pkg.scene.orbit_camera(sc, 2), W, H).copy()
    buf = renderer.host_alloc((H, W))
    try:
        for _ in range(3):
            renderer.render_async(pkg.scene.orbit_camera(sc, 1), W, H, out=buf)
            renderer.render_async(pkg.scene.orbit_camera(sc, 1), W, H, out=buf)   # back on device buffer 0 next
            got_b = renderer.render(pkg.scene.orbit_camera(sc, 2), W, H)
            renderer.wait()
            assert np.array_equal(got_b, b_want) and np.array_equal(buf, a_want)
    finally:
        renderer.host_free(buf)


# ---- the drop-in shim against the ORACLE (not against the binding) -----------------------------------------------

@pytest.mark.parametrize("pipelined", [0, 1])
def test_onstart_update_frame_equals_the_oracle(pipelined, oracle_best, pkg, tmp_path, libm_matches):
    subprocess.check_call(["make", "-s", "-C", HOST])
    out = tmp_path / "frame.ppm"
    W, H, frames = 320, 240, 3
    res = subprocess.run([os.path.join(HOST, "ore_headless"), str(W), str(H), str(frames), "64", str(out), "-", str(pipelined)],
                         capture_output=True, text=True, check=True)
    info = json.loads(res.stdout.strip().splitlines()[-1])
    assert info["pipelined"] == pipelined and info["frames"] == frames
    data = out.read_bytes()
    header = b"P6\n%d %d\n255\n" % (W, H)
    rgb = np.frombuffer(data[len(header):], dtype=np.uint8).reshape(H, W, 3)[::-1]
    got = (rgb[..., 0].astype(np.uint32) << 16) | (rgb[..., 1].astype(np.uint32) << 8) | rgb[..., 2]
    sc = pkg.scene.reference_scene(64, 1)
    f = frames - 1
    yaw, pitch = 180.0 + 360.0 * f / frames, 15.0
    yr, pr = yaw * math.pi / 180, pitch * math.pi / 180      # the harness's own expressions (headless_window.cpp)
    org = tuple(float(np.float32(v)) for v in (5 - 12 * math.cos(pr) * math.sin(yr), 5 + 12 * math.sin(pr),
                                               5 - 12 * math.cos(pr) * math.cos(yr)))
    cam = pkg.scene.Camera(org=org, yaw=float(np.float32(yaw)), pitch=float(np.float32(pitch)))
    ref = oracle_best.render(sc, cam, W, H)["pixels"]
    _exact(got, ref, libm_matches)
    assert info["checksum"] == int(got.astype(np.uint64).sum())


# ---- batches of frames: one launch set for several cameras ---------------------------------------------------------

def test_batch_of_frames_equals_single_frames(renderer, pkg):
    """ore_render_batch_device: K cameras in one launch set give exactly the K single-frame renders - full frames,
    block-interleaved bands stored in place, the fused form and the exhaustive mode"""
    import torch
    sc = pkg.scene.scaled_scene(64, 2)
    renderer.set_scene(sc)
    W, H = 333, 203
    cams = [pkg.scene.orbit_camera(sc, f) for f in (0, 31, 77, 140, 200)]
    want = [renderer.render(c, W, H).copy() for c in cams]
    F = pkg.capi
    for flags in (0, F.ORE_FLAG_FUSED_SHADOW, F.ORE_FLAG_EXHAUSTIVE, F.ORE_FLAG_FAST_LIBM):
        ref = want if flags != F.ORE_FLAG_FAST_LIBM else [renderer.render(c, W, H, flags=flags).copy() for c in cams]
        frames = torch.zeros((len(cams), H, W), dtype=torch.int32, device="cuda:0")
        renderer.render_batch_device(cams, W, H, [frames[i].data_ptr() for i in range(len(cams))], flags=flags)
        renderer.synchronize()
        got = frames.cpu().numpy().view(np.uint32)
        for i in range(len(cams)):
            assert np.array_equal(got[i], ref[i]), (flags, i, int(np.count_nonzero(got[i] != ref[i])))
    # three "ranks" rendering their row blocks of a batch of two frames straight into two shared frames
    frames = torch.zeros((2, H, W), dtype=torch.int32, device="cuda:0")
    for rank in range(3):
        b = pkg.multigpu.block_band(rank, 3, H)
        renderer.render_batch_device(cams[:2], W, H, [frames[i].data_ptr() + 4 * W * b["y0"] for i in range(2)], out_pitch=W, **b)
    renderer.synchronize()
    got = frames.cpu().numpy().view(np.uint32)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    c = renderer.counters()
    assert c["pixels"] == 2 * pkg.Renderer.rows(H, **pkg.multigpu.block_band(2, 3, H)) * W
    with pytest.raises(pkg.OreError):     # per-pixel maps need a single-frame render
        renderer.hits(H, W)
    with pytest.raises(pkg.OreError):     # at most 8 frames per launch set
        renderer.render_batch_device(cams + cams, W, H, [frames[0].data_ptr()] * 10)


def test_batch_async_lands_frames_in_order_with_flags(renderer, pkg):
    sc = pkg.scene.scaled_scene(64, 2)
    renderer.set_scene(sc)
    W, H, K = 320, 180, 3
    host = [renderer.host_alloc((H, W)) for _ in range(2 * K)]
    flag = renderer.host_alloc((16,))
    flag[:] = 0
    try:
        cams = [pkg.scene.orbit_camera(sc, 10 * f) for f in range(2 * K)]
        want = [renderer.render(c, W, H).copy() for c in cams]
        renderer.render_batch_async(cams[:K], W, H, host[:K], done_flag=flag.ctypes.data, first_done_value=1)
        renderer.render_batch_async(cams[K:], W, H, host[K:], done_flag=flag.ctypes.data, first_done_value=K + 1)
        t0 = time.time()
        while int(flag[0]) < 2 * K:
            assert time.time() - t0 < 20
        for a, b in zip(host, want):
            assert np.array_equal(a, b)
        # rows in place, two ranks, batch of two frames into two full host frames
        for h_ in host[:2]:
            h_[:] = 0
        for rank in range(2):
            b = pkg.multigpu.block_band(rank, 2, H)
            renderer.render_batch_async(cams[:2], W, H, [host[i].ctypes.data + 4 * W * b["y0"] for i in range(2)], in_place=True, **b)
        renderer.wait()
        assert np.array_equal(host[0], want[0]) and np.array_equal(host[1], want[1])
    finally:
        renderer.wait()
        for h_ in host:
            renderer.host_free(h_)
        renderer.host_free(flag)


# ---- lights that do not face a pixel (a = normal.toL <= 0) add exactly +0 and are skipped (FrameParams::skip_dark) ----
@pytest.mark.parametrize("case", ["below", "mixed", "one_of_three", "nan_colour"])
def test_lights_facing_away_are_skipped_without_changing_a_pixel(case, renderer, oracle_best, pkg, libm_matches):
    sc = pkg.scene.reference_scene(64, 1)
    lights = sc.lights.copy()
    if case == "below":
        lights = lights[:1].copy()
        lights[0, :3] = (5.0, -60.0, 5.0)        # under the scene: dark for every pixel seen from above -> whole blocks skipped
    elif case == "mixed":
        lights[0, :3] = (5.0, -60.0, 5.0)        # one light below, one level with the camera, one above
        lights[1, :3] = (4.0, 3.0, 30.0)
    elif case == "one_of_three":
        lights[2, :3] = (-40.0, 2.0, 4.0)        # grazing from the side: the terminator crosses many blocks
    elif case == "nan_colour":
        lights[1, 4] = np.float32("nan")         # 0 x NaN is not 0: nothing may be skipped for this scene
    sc2 = pkg.scene.Scene(spheres=sc.spheres, lights=np.ascontiguousarray(lights, dtype=np.float32), texture=sc.texture,
                          sky=sc.sky, extent=sc.extent, name=f"dark_{case}")
    cam = pkg.scene.reference_camera()
    W, H = 200, 150
    F = pkg.capi
    renderer.set_scene(sc2)
    a = renderer.render(cam, W, H)
    for flags in (F.ORE_FLAG_EXHAUSTIVE, F.ORE_FLAG_FUSED_SHADOW):
        b = renderer.render(cam, W, H, flags=flags)
        assert np.array_equal(a, b), (case, flags, int(np.count_nonzero(a != b)))
    if case != "nan_colour":      # (NaN -> int is implementation-defined on the host: out of the oracle's domain)
        ref = oracle_best.render(sc2, cam, W, H)
        if libm_matches:
            assert np.array_equal(a, ref["pixels"]), (case, int(np.count_nonzero(a != ref["pixels"])))
        else:
            d = np.zeros(a.shape, dtype=np.int32)
            for sh in (0, 8, 16):
                d = np.maximum(d, np.abs(((a >> sh) & 255).astype(np.int32) - ((ref["pixels"] >> sh) & 255).astype(np.int32)))
            assert np.count_nonzero(d <= 1) >= 0.999 * d.size
    renderer.set_scene(sc)


# ---- sky texel shortcut (sky_fast, csrc/ore_primary.cuh) against the oracle with an INDEX-ENCODING sky: every texel has
# ---- its own colour, so a pixel that picked a neighbouring texel differs from the reference's frame ----
def _index_sky(pkg, w, h):
    i = np.arange(w * h, dtype=np.int64)
    def chan(k):
        return ((k.astype(np.float64) + 0.5) / 254.0).astype(np.float32).reshape(h, w)
    return pkg.scene.Sprite(width=w, height=h, r=chan(i // 65025), g=chan((i // 255) % 255), b=chan(i % 255))


RA = float(np.float32(math.tan((90 * 0.5 * 3.1415) / 180)))   # scene.REFERENCE_ASPECT
SKY_CASES = [
    # (sky w, h, sky size, camera org, yaw, pitch, aspect); other fields of view: tests/test_view_geometry_gpu.py
    (1024, 512, 10000.0, (4.0, 3.0, 10.0), 180.0, -20.0, RA),       # the reference's camera
    (1024, 512, 10000.0, (4.0, 3.0, 10.0), 37.0, 88.5, RA),         # a pole in view
    (1024, 512, 10000.0, (4.0, 3.0, 10.0), 200.0, -89.0, RA),       # the other pole
    (300, 200, 10000.0, (-3.0, 12.0, 2.0), 301.0, 10.0, RA),        # odd texture size
    (4096, 2048, 10000.0, (4.0, 3.0, 10.0), 90.0, 0.0, RA),         # texels smaller than pixels
    (1024, 512, 10000.0, (3.0e7, 1.0e7, -2.0e7), 10.0, 5.0, RA),    # camera a third of the way to the sky sphere
    (1024, 512, 10000.0, (6.0e7, 0.0, 0.0), 10.0, 5.0, RA),         # |O| > R/2: the shortcut must stand down
    (512, 256, 3.0, (4.0, 3.0, 10.0), 180.0, -20.0, RA),            # tiny sky sphere: camera outside it (NaN roots)
    (512, 256, 0.5, (0.1, 0.0, 0.05), 45.0, 30.0, RA),              # R^2 < 1
]


@pytest.mark.parametrize("case", range(len(SKY_CASES)))
def test_sky_texel_shortcut_equals_the_oracle_with_an_index_encoding_sky(case, renderer, oracle_best, pkg, libm_matches):
    w, h, size, org, yaw, pitch, aspect = SKY_CASES[case]
    base = pkg.scene.reference_scene(64, 1)
    sc = pkg.scene.Scene(spheres=base.spheres, lights=base.lights, texture=base.texture, sky=_index_sky(pkg, w, h),
                         sky_size=size, aspect=np.float32(aspect), extent=base.extent, name=f"index_sky_{case}")
    cam = pkg.scene.Camera(org=org, yaw=yaw, pitch=pitch)
    W, H = 333, 187
    F = pkg.capi
    renderer.set_scene(sc)
    a = renderer.render(cam, W, H)
    c = renderer.counters()
    b = renderer.render(cam, W, H, flags=F.ORE_FLAG_EXHAUSTIVE)
    assert np.array_equal(a, b), (case, int(np.count_nonzero(a != b)))
    miss = c["pixels"] - c["hit_pixels"]
    if case in (0, 3):
        assert c["sky_exact"] < 0.25 * miss, (c["sky_exact"], miss)       # the shortcut decides most pixels
    if case in (6, 7, 8):
        assert c["sky_exact"] == miss, (c["sky_exact"], miss)             # ... and none where it must not be used
    if case not in (7, 8):   # (degenerate sky spheres: NaN roots, the reference indexes its texture out of bounds - no oracle)
        ref = oracle_best.render(sc, cam, W, H)
        if libm_matches:
            assert np.array_equal(a, ref["pixels"]), (case, int(np.count_nonzero(a != ref["pixels"])))
    renderer.set_scene(base)


# ---- band DMA: primary rows through a packed local buffer + a copy engine, hit pixels stored by the sweep ------------
@pytest.mark.parametrize("world,H", [(3, 203), (8, 270), (2, 64), (5, 37)])
def test_band_dma_rows_equal_direct_stores(world, H, renderer, pkg):
    """ORE_FLAG_BAND_DMA (what a rank uses automatically when the frame lives on another GPU) forced onto local memory:
    every rank's 8-row blocks, including a partial last block and ranks with no rows, land exactly where the direct
    stores put them - for batches, single frames, the fused form, and a frame with no lights (copy only)"""
    import torch
    sc = pkg.scene.scaled_scene(64, 2)
    renderer.set_scene(sc)
    W = 333
    cams = [pkg.scene.orbit_camera(sc, f) for f in (5, 90, 170)]
    want = [renderer.render(c, W, H).copy() for c in cams]
    F = pkg.capi
    for flags in (F.ORE_FLAG_BAND_DMA, F.ORE_FLAG_BAND_DMA | F.ORE_FLAG_FUSED_SHADOW, F.ORE_FLAG_BAND_DMA | F.ORE_FLAG_FAST_LIBM):
        ref = want if not (flags & F.ORE_FLAG_FAST_LIBM) else [renderer.render(c, W, H, flags=F.ORE_FLAG_FAST_LIBM).copy() for c in cams]
        frames = torch.full((len(cams), H, W), 0x5A5A5A5A, dtype=torch.int32, device="cuda:0")
        for rank in range(world):
            b = pkg.multigpu.block_band(rank, world, H)
            renderer.render_batch_device(cams, W, H, [frames[i].data_ptr() + 4 * W * b["y0"] for i in range(len(cams))],
                                         out_pitch=W, flags=flags, **b)
        renderer.synchronize()
        got = frames.cpu().numpy().view(np.uint32)
        for i in range(len(cams)):
            assert np.array_equal(got[i], ref[i]), (flags, i, int(np.count_nonzero(got[i] != ref[i])))
    # single frame per call, one rank at a time, rows of the other ranks must stay untouched
    frame = torch.full((H, W), 0x5A5A5A5A, dtype=torch.int32, device="cuda:0")
    b = pkg.multigpu.block_band(world - 1, world, H)
    renderer.render_device(cams[0], W, H, out_ptr=frame.data_ptr() + 4 * W * b["y0"], out_pitch=W, flags=F.ORE_FLAG_BAND_DMA, **b)
    renderer.synchronize()
    got = frame.cpu().numpy().view(np.uint32)
    mine = np.zeros(H, dtype=bool)
    mine[pkg.multigpu.block_rows(world - 1, world, H)] = True
    assert np.array_equal(got[mine], want[0][mine])
    assert np.all(got[~mine] == 0x5A5A5A5A)
    # no lights: the copy is the only writer of the frame
    renderer.set_lights(sc.lights[:0])
    dark = renderer.render(cams[1], W, H).copy()
    frame = torch.full((H, W), 0x5A5A5A5A, dtype=torch.int32, device="cuda:0")
    for rank in range(world):
        b = pkg.multigpu.block_band(rank, world, H)
        renderer.render_device(cams[1], W, H, out_ptr=frame.data_ptr() + 4 * W * b["y0"], out_pitch=W, flags=F.ORE_FLAG_BAND_DMA, **b)
    renderer.synchronize()
    assert np.array_equal(frame.cpu().numpy().view(np.uint32), dark)
    renderer.set_lights(sc.lights)
