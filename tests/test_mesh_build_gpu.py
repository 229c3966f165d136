"""Stream-ordered mesh uploads from device memory with the reference's flat BVH built on the GPU (ore_set_mesh_device,
csrc/ore_mesh_build.cu): the device arrays against the host builder (tests/mesh_build_probe.cpp) byte for byte, renders
equal to ore_set_mesh with the host-built arrays and to the oracle, an animated rebuilt mesh, ordering across streams,
host blocking only on growth, ore_set_mesh behind a pending build, refit of a device-built topology, batches, and
argument validation."""
import ctypes as C

import numpy as np
import pytest

from streamlib import _held_stream, assert_rejected
from test_host_mesh import host_build, host_lib, write_grid_obj  # noqa: F401  (fixture re-export)
from test_mesh_build_cpu import AWKWARD_CASES, build_probe, leaves_1024
from test_mesh_refit_cpu import boxes6, torus_arrays
from test_mesh_refit_cpu import build_probe as build_refit_probe
from test_mesh_update_gpu import deformed
from test_parity_gpu import assert_pixels_close, libm_matches  # noqa: F401  (fixture re-export)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def build_probe_lib(tmp_path_factory):
    return build_probe(tmp_path_factory.mktemp("mesh_build_probe"))


@pytest.fixture(scope="module")
def mesh_probe(tmp_path_factory):
    return build_refit_probe(tmp_path_factory.mktemp("mesh_probe"))


def host_mesh(pkg, build_probe_lib, tris, has_normals=True):
    """scene.Mesh with the host builder's leaves: what ore_set_mesh gets for these triangles"""
    tris = np.ascontiguousarray(tris, np.float32)
    bb, offs, idx = build_probe_lib.build(tris)
    return pkg.scene.Mesh(tris, has_normals, bb, offs, idx)


def assert_device_build(renderer, tris, build_probe_lib, mesh_probe, what):
    """every array of the device build against the probe; leaves past the live count list nothing and are zeros"""
    n = tris.shape[0]
    L = min(1024, n)
    bb, offs, idx = build_probe_lib.build(tris)
    nb = bb.shape[0]
    assert renderer.debug_mesh("n_live")[0] == nb, what
    got_offs = renderer.debug_mesh("box_offsets")
    assert got_offs.shape == (L + 1,), what
    assert np.array_equal(got_offs[:nb + 1], offs) and np.all(got_offs[nb + 1:] == n), what
    assert np.array_equal(renderer.debug_mesh("box_indices"), idx), what
    boxes, sph = mesh_probe.arrays(tris, bb, offs, idx, refit=False)
    got_b, got_s = renderer.debug_mesh("boxes"), renderer.debug_mesh("box_sph")
    assert got_b[:2 * nb].tobytes() == boxes.tobytes(), (what, int(np.count_nonzero(got_b[:2 * nb].view(np.uint32) != boxes.view(np.uint32))))
    assert got_s[:nb].tobytes() == sph.tobytes(), what
    assert not got_b[2 * nb:].view(np.uint32).any() and not got_s[nb:].view(np.uint32).any(), what
    assert np.array_equal(renderer.debug_mesh("tris").view(np.uint32), tris.view(np.uint32)), what


def grid_tris(host_lib, tmp_path, n):
    obj = str(tmp_path / f"grid{n}.obj")
    write_grid_obj(obj, "vtn", n=n)
    d = host_build(host_lib, obj, cap_tris=1 << 21)
    assert d["tris"].shape[0] == 2 * (n - 1) ** 2
    return d["tris"]


# ---- 1. the arrays against the host builder -----------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["torus", "grid4", "grid101", "grid200", "grid709", "leaves_1024"] + sorted(AWKWARD_CASES))
def test_device_build_equals_the_host_builder(name, renderer, build_probe_lib, mesh_probe, host_lib, tmp_path):
    import torch
    if name == "torus":
        tris = torus_arrays()[0]
    elif name.startswith("grid"):
        tris = grid_tris(host_lib, tmp_path, int(name[4:]))   # 18, 20 000, 79 202 and 1 002 528 triangles
    elif name == "leaves_1024":
        tris = leaves_1024()
    else:
        tris = AWKWARD_CASES[name]()
    tris = np.ascontiguousarray(tris, np.float32)
    t = torch.from_numpy(tris).to("cuda:0")
    try:
        st = torch.cuda.Stream()
        st.wait_stream(torch.cuda.current_stream())
        renderer.set_mesh_device(t, True, st.cuda_stream)
        assert_device_build(renderer, tris, build_probe_lib, mesh_probe, (name, "stream"))
        renderer.set_mesh(None)
        renderer.set_mesh_device(t, False)   # the context's own stream, from an empty context
        assert_device_build(renderer, tris, build_probe_lib, mesh_probe, (name, "render stream"))
        if name == "leaves_1024":
            assert renderer.debug_mesh("n_live")[0] == 1024
    finally:
        renderer.set_mesh(None)


# ---- 2. renders equal ore_set_mesh and the oracle ------------------------------------------------------------------------

def _scene(pkg, mesh):
    sc = pkg.scene.with_cubes_and_plane(pkg.scene.reference_scene(64, 1), 4, 5)
    sc.mesh = mesh
    return sc


def _frame(renderer, cam, W, H, flags=0):
    px = renderer.render(cam, W, H, flags=flags).copy()
    ids, t = renderer.hits(H, W)
    return px, ids, t


def _same_frame(a, b, what):
    assert np.array_equal(a[0], b[0]), (what, int(np.count_nonzero(a[0] != b[0])))
    assert np.array_equal(a[1], b[1]), (what, int(np.count_nonzero(a[1] != b[1])))
    assert np.array_equal(a[2].view(np.uint32), b[2].view(np.uint32)), what


def test_device_built_mesh_renders_like_set_mesh(renderer, build_probe_lib, oracle_best, pkg, libm_matches):
    import torch
    F = pkg.capi
    tris = torus_arrays()[0]
    sc = _scene(pkg, host_mesh(pkg, build_probe_lib, tris))
    W, H = 160, 120
    try:
        renderer.set_scene(sc)
        for k, angle in enumerate((15, 70, 160, 250)):
            cam = pkg.scene.orbit_camera(sc, angle)
            renderer.set_mesh(sc.mesh)
            want = _frame(renderer, cam, W, H)
            assert (want[1] >= 64 + 4 + 1).any(), "the mesh must be visible"
            renderer.set_mesh_device(torch.from_numpy(tris).to("cuda:0"), True)
            for flags in (0, F.ORE_FLAG_FUSED_SHADOW, F.ORE_FLAG_EXHAUSTIVE):
                _same_frame(_frame(renderer, cam, W, H, flags), want, (angle, flags))
            if k < 2:
                ref = oracle_best.render(sc, cam, W, H)
                assert np.array_equal(want[1], ref["ids"]) and np.array_equal(want[2].view(np.uint32), ref["t"].view(np.uint32))
                assert_pixels_close(want[0], ref["pixels"])
                if libm_matches:
                    assert np.array_equal(want[0], ref["pixels"])
    finally:
        renderer.set_mesh(None)


def strong_deformation(tris, f):
    """frame f: a large twist and a squash, so leaves built for frame 0 overlap badly"""
    out = deformed(tris, f)
    for v in range(3):
        x, z = out[:, 3 * v].copy(), out[:, 3 * v + 2].copy()
        a = 0.25 * f * (z - 5.0)
        out[:, 3 * v] = (x - 5.0) * np.cos(a) + 5.0
        out[:, 3 * v + 2] = z + 0.6 * np.sin(0.5 * f + x)
    return np.ascontiguousarray(out, np.float32)


def test_animated_rebuilt_mesh_equals_host_rebuild(renderer, build_probe_lib, oracle_best, pkg, libm_matches):
    import torch
    base = torus_arrays()[0]
    sc = _scene(pkg, host_mesh(pkg, build_probe_lib, base))
    W, H = 128, 96
    n_frames = 8
    frames_np = [strong_deformation(base, f) for f in range(n_frames)]
    inputs = [torch.from_numpy(x).to("cuda:0") for x in frames_np]
    cams = [pkg.scene.orbit_camera(sc, 20 + 25 * f) for f in range(n_frames)]
    out = torch.zeros((n_frames, H, W), dtype=torch.int32, device="cuda:0")
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    try:
        renderer.set_scene(sc)
        for f in range(n_frames):
            renderer.set_mesh_device(inputs[f], True, st.cuda_stream)
            renderer.render_device(cams[f], W, H, out[f].data_ptr(), stream=st.cuda_stream)
        st.synchronize()
        got = out.cpu().numpy().view(np.uint32)
        differs_from_refit = 0
        for f in range(n_frames):
            m = host_mesh(pkg, build_probe_lib, frames_np[f])
            renderer.set_mesh(m)
            want = _frame(renderer, cams[f], W, H)
            assert np.array_equal(got[f], want[0]), (f, int(np.count_nonzero(got[f] != want[0])))
            renderer.set_mesh_device(inputs[f], True)
            _same_frame(_frame(renderer, cams[f], W, H), want, f)
            if f % 3 == 0:
                ref = oracle_best.render(_scene(pkg, m), cams[f], W, H)
                assert np.array_equal(want[1], ref["ids"]) and np.array_equal(want[2].view(np.uint32), ref["t"].view(np.uint32)), f
                assert_pixels_close(want[0], ref["pixels"])
            # the refit of frame 0's leaves renders the same geometry; its leaves are not the reference's
            renderer.set_mesh(sc.mesh)
            renderer.set_mesh_triangles_device(inputs[f])
            differs_from_refit += int(not np.array_equal(renderer.debug_mesh("box_indices"), m.box_indices))
        assert differs_from_refit >= n_frames - 1
    finally:
        renderer.set_mesh(None)


# ---- 3. ordering, host blocking, lifecycle ------------------------------------------------------------------------------

def test_build_on_another_stream_is_ordered_between_renders(renderer, build_probe_lib, pkg):
    import torch
    base = torus_arrays()[0]
    a_np, b_np = base, strong_deformation(base, 5)
    sc = _scene(pkg, host_mesh(pkg, build_probe_lib, a_np))
    W, H = 1920, 1080
    cam = pkg.scene.orbit_camera(sc, 40)
    try:
        renderer.set_scene(sc)
        want_a = renderer.render(cam, W, H).copy()
        renderer.set_mesh(host_mesh(pkg, build_probe_lib, b_np))
        want_b = renderer.render(cam, W, H).copy()
        assert np.count_nonzero(want_a != want_b) > 1000
        renderer.set_mesh(sc.mesh)
        mesh_a, mesh_b = torch.from_numpy(a_np).to("cuda:0"), torch.from_numpy(b_np).to("cuda:0")
        T, S = torch.cuda.Stream(), torch.cuda.Stream()
        frames = torch.zeros((2, H, W), dtype=torch.int32, device="cuda:0")
        torch.cuda.synchronize()
        renderer.render_device(cam, W, H, frames[0].data_ptr(), stream=T.cuda_stream)
        renderer.set_mesh_device(mesh_b, True, S.cuda_stream)
        renderer.render_device(cam, W, H, frames[1].data_ptr(), stream=T.cuda_stream)
        T.synchronize()
        got = frames.cpu().numpy().view(np.uint32)
        assert np.array_equal(got[0], want_a), int(np.count_nonzero(got[0] != want_a))
        assert np.array_equal(got[1], want_b), int(np.count_nonzero(got[1] != want_b))
        # a batch of 4 cameras after a build equals 4 single frames
        cams = [pkg.scene.orbit_camera(sc, 45 * f + 7) for f in range(4)]
        Wb, Hb = 480, 270
        renderer.set_mesh_device(mesh_a, True, S.cuda_stream)
        batch = torch.zeros((4, Hb, Wb), dtype=torch.int32, device="cuda:0")
        T.wait_stream(torch.cuda.current_stream())
        renderer.render_batch_device(cams, Wb, Hb, [batch[i].data_ptr() for i in range(4)], stream=T.cuda_stream)
        T.synchronize()
        got = batch.cpu().numpy().view(np.uint32)
        for i, c in enumerate(cams):
            assert np.array_equal(got[i], renderer.render(c, Wb, Hb)), i
        renderer.set_mesh(sc.mesh)
        for i, c in enumerate(cams):
            assert np.array_equal(got[i], renderer.render(c, Wb, Hb)), i
    finally:
        renderer.set_mesh(None)


def test_build_blocks_the_host_only_on_growth(renderer, build_probe_lib, mesh_probe, host_lib, tmp_path, pkg):
    import torch
    torus = torus_arrays()[0]
    small = torch.from_numpy(strong_deformation(torus, 2)).to("cuda:0")
    big_np = np.ascontiguousarray(grid_tris(host_lib, tmp_path, 709))
    big = torch.from_numpy(big_np).to("cuda:0")
    try:
        renderer.set_mesh(None)
        renderer.set_mesh_device(torch.from_numpy(torus).to("cuda:0"), True)
        # capacity suffices: the call returns at once and the build still waits behind the held stream
        dt, pending = _held_stream(renderer, lambda s: renderer.set_mesh_device(small, True, s))
        assert dt < 0.5 and pending, dt
        assert_device_build(renderer, small.cpu().numpy(), build_probe_lib, mesh_probe, "held")
        # growth to 1 M triangles waits for the held stream's pending work first, then returns
        renderer.set_mesh_device(small, True)
        _held_stream(renderer, lambda s: renderer.set_mesh_device(big, True, s))
        assert_device_build(renderer, big_np, build_probe_lib, mesh_probe, "grown")
        # back to the torus and up to 1 M again: within capacity, no blocking
        for t, want in ((small, small.cpu().numpy()), (big, big_np)):
            dt, pending = _held_stream(renderer, lambda s, t=t: renderer.set_mesh_device(t, True, s))
            assert dt < 0.5 and pending, dt
            assert_device_build(renderer, want, build_probe_lib, mesh_probe, "within capacity")
        # a mesh set by ore_set_mesh keeps the capacity: a device build of the largest size afterwards does not block
        renderer.set_mesh(host_mesh(pkg, build_probe_lib, torus))
        dt, pending = _held_stream(renderer, lambda s: renderer.set_mesh_device(big, True, s))
        assert dt < 0.5 and pending, dt
    finally:
        renderer.set_mesh(None)


def test_set_mesh_waits_for_a_pending_build(renderer, build_probe_lib, oracle_best, pkg):
    import time

    import torch
    torus = torus_arrays()[0]
    sc = _scene(pkg, host_mesh(pkg, build_probe_lib, torus))
    other = host_mesh(pkg, build_probe_lib, strong_deformation(torus, 6))
    t = torch.from_numpy(strong_deformation(torus, 3)).to("cuda:0")
    cam = pkg.scene.orbit_camera(sc, 60)
    took = {}

    def host_setter():
        t0 = time.perf_counter()
        renderer.set_mesh(other)
        took["s"] = time.perf_counter() - t0

    try:
        renderer.set_scene(sc)
        dt, pending = _held_stream(renderer, lambda s: renderer.set_mesh_device(t, True, s), after=host_setter)
        assert pending and dt < 0.5, dt
        assert took["s"] > 1.0, f"ore_set_mesh returned after {took['s']:.3f} s, before the held build had run"
        assert np.array_equal(renderer.debug_mesh("tris"), other.tris)
        assert np.array_equal(renderer.debug_mesh("box_indices"), other.box_indices)
        assert renderer.debug_mesh("n_live")[0] == other.n_boxes
        px = renderer.render(cam, 128, 96)
        ref = oracle_best.render(_scene(pkg, other), cam, 128, 96)
        ids, tt = renderer.hits(96, 128)
        assert np.array_equal(ids, ref["ids"]) and np.array_equal(tt.view(np.uint32), ref["t"].view(np.uint32))
        assert_pixels_close(px, ref["pixels"])
    finally:
        renderer.set_mesh(None)


def test_refit_after_a_device_build_equals_the_probe(renderer, build_probe_lib, mesh_probe, pkg):
    import torch
    torus = torus_arrays()[0]
    built = strong_deformation(torus, 4)
    moved = strong_deformation(torus, 7)
    bb, offs, idx = build_probe_lib.build(built)
    nb = bb.shape[0]
    W, H = 160, 120
    sc = _scene(pkg, None)
    cam = pkg.scene.orbit_camera(sc, 100)
    try:
        renderer.set_scene(sc)
        renderer.set_mesh_device(torch.from_numpy(built).to("cuda:0"), True)
        renderer.set_mesh_triangles_device(torch.from_numpy(moved).to("cuda:0"))
        boxes, sph = mesh_probe.arrays(moved, bb, offs, idx, refit=True)
        got_b, got_s = renderer.debug_mesh("boxes"), renderer.debug_mesh("box_sph")
        assert got_b[:2 * nb].tobytes() == boxes.tobytes() and got_s[:nb].tobytes() == sph.tobytes()
        assert np.array_equal(renderer.debug_mesh("box_indices"), idx) and renderer.debug_mesh("n_live")[0] == nb
        got = _frame(renderer, cam, W, H)
        renderer.set_mesh(pkg.scene.Mesh(moved, True, np.ascontiguousarray(boxes6(boxes)), offs, idx))
        _same_frame(got, _frame(renderer, cam, W, H), "refit of the device topology")
    finally:
        renderer.set_mesh(None)


# ---- 4. validation ---------------------------------------------------------------------------------------------------

def test_invalid_arguments_are_rejected_and_change_nothing(renderer, build_probe_lib, pkg):
    import torch
    torus = torus_arrays()[0]
    sc = _scene(pkg, host_mesh(pkg, build_probe_lib, torus))
    cam = pkg.scene.orbit_camera(sc, 10)
    lib, ctx = renderer.lib, renderer.ctx
    n = torus.shape[0]
    moved = strong_deformation(torus, 5)
    good = torch.from_numpy(moved).to("cuda:0")
    pinned = renderer.host_alloc((n, 27), dtype=np.float32)
    pinned[:] = moved
    raw = torch.zeros(n * 27 + 4, dtype=torch.float32, device="cuda:0")
    try:
        renderer.set_scene(sc)
        want = renderer.render(cam, 160, 120).copy()
        bad = [(moved.ctypes.data, n), (pinned.ctypes.data, n), (raw.data_ptr() + 2, n), (0, n), (good.data_ptr(), 0),
               (good.data_ptr(), -1)]
        if torch.cuda.device_count() > 1:
            bad.append((torch.from_numpy(moved).to("cuda:1").data_ptr(), n))
        assert_rejected(lambda ptr, k: lib.ore_set_mesh_device(ctx, ptr or None, k, 1, None), bad,
                        lambda: renderer.render(cam, 160, 120), want)
        assert np.array_equal(renderer.debug_mesh("tris"), torus)
        assert np.array_equal(renderer.debug_mesh("box_indices"), sc.mesh.box_indices)
        for t, err in ((good.double(), TypeError), (good[:, :26].contiguous(), ValueError), (good[:0], ValueError),
                       (good.reshape(-1), ValueError), (good.cpu(), ValueError), (good.t().contiguous().t(), ValueError),
                       (moved, TypeError)):
            with pytest.raises(err):
                renderer.set_mesh_device(t, True)
        assert np.array_equal(renderer.render(cam, 160, 120), want)
        # 4-byte alignment only: an update at an offset inside an allocation is accepted
        raw[1:1 + n * 27] = good.reshape(-1)
        torch.cuda.synchronize()
        assert lib.ore_set_mesh_device(ctx, C.c_void_p(raw.data_ptr() + 4), n, 1, None) == 0
        assert np.array_equal(renderer.debug_mesh("tris"), moved)
    finally:
        renderer.host_free(pinned)
        renderer.set_mesh(None)


def test_rejected_set_mesh_keeps_the_mesh_and_its_capacity(renderer, build_probe_lib, host_lib, tmp_path, pkg):
    """ore_set_mesh checks its host arrays before it frees anything: a rejected call leaves the mesh, and the capacity a
    larger device build reached, so a device build of that size afterwards still does not block the host"""
    import torch
    torus = torus_arrays()[0]
    sc = _scene(pkg, host_mesh(pkg, build_probe_lib, torus))
    m = sc.mesh
    cam = pkg.scene.orbit_camera(sc, 10)
    big = torch.from_numpy(np.ascontiguousarray(grid_tris(host_lib, tmp_path, 101))).to("cuda:0")   # 20 000 triangles
    lib, ctx = renderer.lib, renderer.ctx
    ip = C.POINTER(C.c_int32)
    descending, shifted, out_of_range = m.box_offsets.copy(), m.box_offsets.copy(), m.box_indices.copy()
    descending[m.n_boxes // 2] = descending[m.n_boxes // 2 + 1] + 1
    shifted[0] = 1
    out_of_range[len(out_of_range) // 2] = m.n_tris

    def set_mesh(offsets, indices):
        return lib.ore_set_mesh(ctx, m.tris.ctypes.data_as(C.POINTER(C.c_float)), m.n_tris, 1,
                                m.box_bounds.ctypes.data_as(C.POINTER(C.c_float)), offsets.ctypes.data_as(ip),
                                indices.ctypes.data_as(ip), m.n_boxes)

    try:
        renderer.set_scene(sc)
        renderer.set_mesh_device(big, True)
        renderer.set_mesh(m)
        want = renderer.render(cam, 160, 120).copy()
        assert (renderer.hits(120, 160)[0] >= 64 + 4 + 1).any(), "the mesh must be visible"
        assert_rejected(set_mesh, [(descending, m.box_indices), (shifted, m.box_indices), (m.box_offsets, out_of_range)],
                        lambda: renderer.render(cam, 160, 120), want)
        assert np.array_equal(renderer.debug_mesh("tris"), m.tris)
        assert np.array_equal(renderer.debug_mesh("box_indices"), m.box_indices)
        assert renderer.debug_mesh("n_live")[0] == m.n_boxes
        dt, pending = _held_stream(renderer, lambda s: renderer.set_mesh_device(big, True, s))
        assert dt < 0.5 and pending, dt
    finally:
        renderer.set_mesh(None)


def test_rebuild_not_refit_matches_the_reference_on_tied_triangles(renderer, build_probe_lib, mesh_probe, oracle_best, pkg):
    """The torus plus 200 duplicates of its triangles with the vertices rotated: a duplicate ties with its original on
    some pixels and can sit in another leaf.  After a deformation the refit keeps the old leaf order and reports the
    other triangle of a tie on some pixel; the rebuild reports the reference's (the oracle given the rebuilt leaves,
    which is what the reference builds when it loads the deformed mesh)."""
    import torch
    base = torus_arrays()[0]
    pick = np.random.default_rng(0).permutation(base.shape[0])[:200]
    dup = base[pick].copy()
    dup[:, 0:9] = np.roll(dup[:, 0:9].reshape(-1, 3, 3), 1, axis=1).reshape(-1, 9)
    tris0 = np.ascontiguousarray(np.concatenate([base, dup]), np.float32)
    moved = strong_deformation(tris0, 2)
    sc = _scene(pkg, host_mesh(pkg, build_probe_lib, tris0))
    cam = pkg.scene.orbit_camera(sc, 20)
    W, H = 128, 96
    try:
        renderer.set_scene(sc)
        renderer.set_mesh_triangles_device(torch.from_numpy(moved).to("cuda:0"))
        refit = _frame(renderer, cam, W, H)
        renderer.set_mesh_device(torch.from_numpy(moved).to("cuda:0"), True)
        rebuilt = _frame(renderer, cam, W, H)
        assert np.count_nonzero(refit[1] != rebuilt[1]) >= 1
        ref = oracle_best.render(_scene(pkg, host_mesh(pkg, build_probe_lib, moved)), cam, W, H)
        assert np.array_equal(rebuilt[1], ref["ids"]) and np.array_equal(rebuilt[2].view(np.uint32), ref["t"].view(np.uint32))
        bb0, offs0, idx0 = build_probe_lib.build(tris0)
        boxes, _ = mesh_probe.arrays(moved, bb0, offs0, idx0, refit=True)
        ref_refit = oracle_best.render(_scene(pkg, pkg.scene.Mesh(moved, True, np.ascontiguousarray(boxes6(boxes)), offs0, idx0)),
                                       cam, W, H)
        assert np.array_equal(refit[1], ref_refit["ids"])
    finally:
        renderer.set_mesh(None)


def test_changing_triangle_counts_within_capacity(renderer, build_probe_lib, mesh_probe, host_lib, tmp_path):
    """generated geometry: every call a different count below the capacity the largest build set; each build equals the
    host builder, none blocks the host, and n <= 5 meshes keep one leaf"""
    import torch
    grid = np.ascontiguousarray(grid_tris(host_lib, tmp_path, 101))   # 20 000 triangles
    big = torch.from_numpy(grid).to("cuda:0")
    try:
        renderer.set_mesh(None)
        renderer.set_mesh_device(big, True)
        for n in (19999, 7, 3, 577, 1024, 1025, 12345, 6):
            view = big[:n]
            dt, pending = _held_stream(renderer, lambda s, v=view: renderer.set_mesh_device(v, True, s))
            assert dt < 0.5 and pending, (n, dt)
            assert_device_build(renderer, grid[:n], build_probe_lib, mesh_probe, ("count", n))
    finally:
        renderer.set_mesh(None)
