"""Stream-ordered triangle updates from device memory (ore_set_mesh_triangles_device) with the leaf boxes and their
spheres refit on the GPU (csrc/ore_mesh_refit.cu): the device arrays against the host functions of
csrc/ore_mesh_refit.h byte for byte, animated frames against the oracle, ordering across streams, no host blocking,
ore_set_mesh behind a pending update, and argument validation."""
import ctypes as C
import time

import numpy as np
import pytest

from streamlib import _held_stream, assert_rejected
from test_host_mesh import host_build, host_lib, write_grid_obj  # noqa: F401  (fixture re-export)
from test_mesh_refit_cpu import awkward_mesh, boxes6, build_probe, torus_arrays
from test_parity_gpu import assert_pixels_close, libm_matches  # noqa: F401  (fixture re-export)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mesh_probe(tmp_path_factory):
    return build_probe(tmp_path_factory.mktemp("mesh_probe"))


def deformed(tris, f):
    """frame f of a deformation of the vertices (numpy or torch, float32): a travelling wave plus a twist"""
    out = tris.clone() if hasattr(tris, "clone") else tris.copy()
    lib = __import__("torch") if hasattr(tris, "clone") else np
    for v in range(3):
        x, y, z = tris[:, 3 * v], tris[:, 3 * v + 1], tris[:, 3 * v + 2]
        out[:, 3 * v + 1] = y + 0.35 * lib.sin(1.3 * x + 0.7 * f)
        out[:, 3 * v] = x + 0.15 * lib.cos(0.9 * z + 0.4 * f)
    return out


def mesh_case(name, host_lib, tmp_path):
    """(topology + the boxes ore_set_mesh gets, the triangles of the device update)"""
    from rte_b200 import pkg
    if name.startswith("torus"):
        tris, bb, offs, idx = torus_arrays()
        new = tris.copy() if name == "torus" else deformed(tris, 3).astype(np.float32)
        d = dict(tris=tris, has_normals=True, box_bounds=bb, box_offsets=offs, box_indices=idx)
    elif name.startswith("grid"):
        n = int(name[4:])
        obj = str(tmp_path / f"{name}.obj")
        write_grid_obj(obj, "vtn", n=n)
        d = host_build(host_lib, obj, cap_tris=1 << 17)
        new = deformed(d["tris"], 1).astype(np.float32)
    else:   # awkward: NaN, +-inf, +-0 and 1e30 vertices; empty, single-triangle and repeating leaves
        tris, bb, offs, idx = awkward_mesh(11)
        new = awkward_mesh(12)[0]
        d = dict(tris=tris, has_normals=False, box_bounds=bb, box_offsets=offs, box_indices=idx)
    return pkg.scene.Mesh.from_arrays(d), np.ascontiguousarray(new, np.float32)


def assert_same_mesh(renderer, tris, boxes, sph, what):
    for k, want in (("tris", tris), ("boxes", boxes), ("box_sph", sph)):
        got = renderer.debug_mesh(k)
        assert got.shape == want.shape, (what, k, got.shape, want.shape)
        assert got.tobytes() == want.tobytes(), (what, k, int(np.count_nonzero(got.view(np.uint32) != want.view(np.uint32))))


# ---- 1. the arrays against the host functions ---------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["torus", "torus_deformed", "grid4", "grid23", "grid200", "awkward"])
def test_device_arrays_equal_the_probe(name, renderer, mesh_probe, host_lib, tmp_path):
    import torch
    mesh, new = mesh_case(name, host_lib, tmp_path)
    if name == "grid200":
        assert mesh.n_tris == 2 * 199 ** 2
    topo = (mesh.box_offsets, mesh.box_indices)
    try:
        renderer.set_mesh(mesh)
        boxes, sph = mesh_probe.arrays(mesh.tris, mesh.box_bounds, *topo, refit=False)
        assert_same_mesh(renderer, mesh.tris, boxes, sph, (name, "ore_set_mesh"))
        boxes, sph = mesh_probe.arrays(new, mesh.box_bounds, *topo, refit=True)
        t = torch.from_numpy(new).to("cuda:0")
        st = torch.cuda.Stream()
        st.wait_stream(torch.cuda.current_stream())
        renderer.set_mesh_triangles_device(t, st.cuda_stream)
        assert_same_mesh(renderer, new, boxes, sph, (name, "device"))
        renderer.set_mesh(mesh)
        renderer.set_mesh_triangles_device(t)   # the context's own stream
        assert_same_mesh(renderer, new, boxes, sph, (name, "render stream"))
        # leaves keep the topology's boxes only where empty: back to the original triangles gives the builder's boxes
        if name != "awkward":
            renderer.set_mesh_triangles_device(torch.from_numpy(mesh.tris).to("cuda:0"))
            got = renderer.debug_mesh("boxes")
            assert np.array_equal(boxes6(got).view(np.uint32), mesh.box_bounds.view(np.uint32)), name
    finally:
        renderer.set_mesh(None)


# ---- 2. an animated sequence against the oracle -------------------------------------------------------------------------

def _scene(pkg, mesh):
    from cases import torus_mesh
    sc = pkg.scene.with_cubes_and_plane(pkg.scene.reference_scene(64, 1), 4, 5)
    sc.mesh = mesh if mesh is not None else torus_mesh()
    return sc


def _non_finite(cur, f):
    """frames 5 and 6 carry NaN and infinite vertices"""
    if f == 5:
        cur[10:14, 0:9:4] = float("nan")
        cur[300, 4] = float("inf")
    if f == 6:
        cur[20:23, 1] = float("-inf")
        cur[400, 0:9] = float("nan")
    return cur


def test_animated_frames_equal_the_oracle(renderer, oracle_best, mesh_probe, pkg, libm_matches):
    import torch
    sc = _scene(pkg, None)
    m = sc.mesh
    renderer.set_scene(sc)
    base = torch.from_numpy(m.tris.copy()).to("cuda:0")
    W, H = 128, 96
    n_frames = 8
    frames = torch.zeros((n_frames, H, W), dtype=torch.int32, device="cuda:0")
    cams = [pkg.scene.orbit_camera(sc, 20 + 25 * f) for f in range(n_frames)]
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    inputs = []
    try:
        with torch.cuda.stream(st):
            for f in range(n_frames):
                cur = _non_finite(deformed(base, f), f)
                inputs.append(cur)
                renderer.set_mesh_triangles_device(cur, st.cuda_stream)
                renderer.render_device(cams[f], W, H, frames[f].data_ptr(), stream=st.cuda_stream)
        st.synchronize()
        got = frames.cpu().numpy().view(np.uint32)
        F = pkg.capi
        for f in range(n_frames):
            tris = inputs[f].cpu().numpy()
            boxes, _ = mesh_probe.arrays(tris, m.box_bounds, m.box_offsets, m.box_indices, refit=True)
            scf = _scene(pkg, pkg.scene.Mesh(tris, m.has_normals, np.ascontiguousarray(boxes6(boxes)), m.box_offsets,
                                              m.box_indices))
            ref = oracle_best.render(scf, cams[f], W, H)
            assert_pixels_close(got[f], ref["pixels"])
            if libm_matches:
                assert np.array_equal(got[f], ref["pixels"]), (f, int(np.count_nonzero(got[f] != ref["pixels"])))
            renderer.set_mesh_triangles_device(inputs[f])
            px = renderer.render(cams[f], W, H)
            assert np.array_equal(px, got[f]), f
            ids, t = renderer.hits(H, W)
            assert np.array_equal(ids, ref["ids"]) and np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32)), f
            assert (ids >= 64 + 4 + 1).any(), f"frame {f}: the mesh must be visible"
            assert np.array_equal(renderer.render(cams[f], W, H, flags=F.ORE_FLAG_EXHAUSTIVE), px), f
            ids_e, t_e = renderer.hits(H, W)
            assert np.array_equal(ids_e, ids) and np.array_equal(t_e.view(np.uint32), t.view(np.uint32)), f
    finally:
        renderer.set_mesh(None)


# ---- 3. ordering across streams ---------------------------------------------------------------------------------------

def test_update_on_another_stream_is_ordered_between_renders(renderer, pkg):
    import torch
    sc = _scene(pkg, None)
    m = sc.mesh
    W, H = 1920, 1080
    cam = pkg.scene.orbit_camera(sc, 40)
    b_np = deformed(m.tris, 2).astype(np.float32)
    try:
        renderer.set_scene(sc)
        want_a = renderer.render(cam, W, H).copy()
        renderer.set_mesh(pkg.scene.Mesh(b_np, m.has_normals, m.box_bounds, m.box_offsets, m.box_indices))
        renderer.set_mesh_triangles_device(torch.from_numpy(b_np).to("cuda:0"))   # (boxes of b from the refit)
        want_b = renderer.render(cam, W, H).copy()
        assert np.count_nonzero(want_a != want_b) > 1000
        renderer.set_mesh(m)
        mesh_b, mesh_a = torch.from_numpy(b_np).to("cuda:0"), torch.from_numpy(m.tris.copy()).to("cuda:0")
        T, S = torch.cuda.Stream(), torch.cuda.Stream()
        frames = torch.zeros((2, H, W), dtype=torch.int32, device="cuda:0")
        torch.cuda.synchronize()
        renderer.render_device(cam, W, H, frames[0].data_ptr(), stream=T.cuda_stream)
        renderer.set_mesh_triangles_device(mesh_b, S.cuda_stream)
        renderer.render_device(cam, W, H, frames[1].data_ptr(), stream=T.cuda_stream)
        T.synchronize()
        got = frames.cpu().numpy().view(np.uint32)
        assert np.array_equal(got[0], want_a), int(np.count_nonzero(got[0] != want_a))
        assert np.array_equal(got[1], want_b), int(np.count_nonzero(got[1] != want_b))
        # a batch of 8 cameras after an update equals 8 single frames
        cams = [pkg.scene.orbit_camera(sc, 30 * f + 7) for f in range(8)]
        Wb, Hb = 480, 270
        renderer.set_mesh_triangles_device(mesh_a, S.cuda_stream)
        batch = torch.zeros((8, Hb, Wb), dtype=torch.int32, device="cuda:0")
        T.wait_stream(torch.cuda.current_stream())
        renderer.render_batch_device(cams, Wb, Hb, [batch[i].data_ptr() for i in range(8)], stream=T.cuda_stream)
        T.synchronize()
        got = batch.cpu().numpy().view(np.uint32)
        for i, c in enumerate(cams):
            assert np.array_equal(got[i], renderer.render(c, Wb, Hb)), i
        # mesh and sphere updates on two streams interleave: each render sees the scene of the updates before it
        sp_b = sc.spheres.copy()
        sp_b[:, 1] += np.float32(0.75)
        renderer.set_spheres(sp_b)
        renderer.set_mesh_triangles_device(mesh_b)
        want_bb = renderer.render(cam, W, H).copy()
        renderer.set_spheres(sc.spheres)
        renderer.set_mesh_triangles_device(mesh_a)
        assert np.array_equal(renderer.render(cam, W, H), want_a)
        spheres_b = torch.from_numpy(sp_b).to("cuda:0")
        torch.cuda.synchronize()
        renderer.set_mesh_triangles_device(mesh_b, S.cuda_stream)
        renderer.set_spheres_device(spheres_b, T.cuda_stream)
        renderer.render_device(cam, W, H, frames[0].data_ptr(), stream=T.cuda_stream)
        renderer.set_mesh_triangles_device(mesh_a, S.cuda_stream)
        renderer.render_device(cam, W, H, frames[1].data_ptr(), stream=S.cuda_stream)
        torch.cuda.synchronize()
        got = frames.cpu().numpy().view(np.uint32)
        assert np.array_equal(got[0], want_bb), int(np.count_nonzero(got[0] != want_bb))
        renderer.set_mesh_triangles_device(mesh_a)
        renderer.set_spheres(sp_b)
        assert np.array_equal(got[1], renderer.render(cam, W, H))
    finally:
        renderer.set_mesh(None)
        renderer.set_spheres(sc.spheres)


# ---- 4. no host blocking; 5. ore_set_mesh behind a pending update ------------------------------------------------------

def test_update_does_not_block_the_host(renderer, mesh_probe, pkg):
    import torch
    m = _scene(pkg, None).mesh
    new = deformed(m.tris, 4).astype(np.float32)
    t = torch.from_numpy(new).to("cuda:0")
    try:
        renderer.set_mesh(m)
        dt, pending = _held_stream(renderer, lambda s: renderer.set_mesh_triangles_device(t, s))
        assert dt < 0.5, dt
        assert pending, "the update must still be waiting behind the held stream"
        boxes, sph = mesh_probe.arrays(new, m.box_bounds, m.box_offsets, m.box_indices, refit=True)
        assert_same_mesh(renderer, new, boxes, sph, "after release")
    finally:
        renderer.set_mesh(None)


def test_set_mesh_waits_for_a_pending_update(renderer, oracle_best, pkg):
    import torch
    sc = _scene(pkg, None)
    m = sc.mesh
    cam = pkg.scene.orbit_camera(sc, 60)
    other = pkg.scene.Mesh(deformed(m.tris, 6).astype(np.float32), m.has_normals, m.box_bounds, m.box_offsets, m.box_indices)
    t = torch.from_numpy(deformed(m.tris, 2).astype(np.float32)).to("cuda:0")
    took = {}

    def host_setter():
        t0 = time.perf_counter()
        renderer.set_mesh(other)    # issued while the device update is held
        took["s"] = time.perf_counter() - t0

    try:
        renderer.set_scene(sc)
        dt, pending = _held_stream(renderer, lambda s: renderer.set_mesh_triangles_device(t, s), after=host_setter)
        assert pending and dt < 0.5, dt
        assert took["s"] > 1.0, f"ore_set_mesh returned after {took['s']:.3f} s, before the held update had run"
        px = renderer.render(cam, 128, 96)
        assert np.array_equal(renderer.debug_mesh("tris"), other.tris)
        ref = oracle_best.render(_scene(pkg, other), cam, 128, 96)
        ids, tt = renderer.hits(96, 128)
        assert np.array_equal(ids, ref["ids"]) and np.array_equal(tt.view(np.uint32), ref["t"].view(np.uint32))
        assert_pixels_close(px, ref["pixels"])
    finally:
        renderer.set_mesh(None)


# ---- 6. validation ---------------------------------------------------------------------------------------------------

def test_invalid_arguments_are_rejected_and_change_nothing(renderer, pkg):
    import torch
    sc = _scene(pkg, None)
    m = sc.mesh
    cam = pkg.scene.orbit_camera(sc, 10)
    lib, ctx = renderer.lib, renderer.ctx
    n = m.n_tris
    moved = np.ascontiguousarray(deformed(m.tris, 5), np.float32)
    good = torch.from_numpy(moved).to("cuda:0")
    pinned = renderer.host_alloc((n, 27), dtype=np.float32)
    pinned[:] = moved
    raw = torch.zeros(n * 27 + 4, dtype=torch.float32, device="cuda:0")
    try:
        renderer.set_mesh(None)
        assert lib.ore_set_mesh_triangles_device(ctx, C.c_void_p(good.data_ptr()), n, None) == 1   # no mesh set
        renderer.set_scene(sc)
        want = renderer.render(cam, 160, 120).copy()
        bad = [(moved.ctypes.data, n), (pinned.ctypes.data, n), (raw.data_ptr() + 2, n), (0, n), (good.data_ptr(), n - 1),
               (good.data_ptr(), n + 1), (good.data_ptr(), -1), (good.data_ptr(), 0)]
        if torch.cuda.device_count() > 1:
            bad.append((torch.from_numpy(moved).to("cuda:1").data_ptr(), n))
        assert_rejected(lambda ptr, k: lib.ore_set_mesh_triangles_device(ctx, ptr or None, k, None), bad,
                        lambda: renderer.render(cam, 160, 120), want)
        assert np.array_equal(renderer.debug_mesh("tris"), m.tris)
        # the Python binding checks before the call
        for t, err in ((good.double(), TypeError), (good[:, :26].contiguous(), ValueError), (good[:-1], ValueError),
                       (good.cpu(), ValueError), (good.t().contiguous().t(), ValueError), (moved, TypeError)):
            with pytest.raises(err):
                renderer.set_mesh_triangles_device(t)
        assert np.array_equal(renderer.render(cam, 160, 120), want)
        # an aligned update at an offset inside an allocation is accepted (4-byte alignment only)
        raw[1:1 + n * 27] = good.reshape(-1)
        torch.cuda.synchronize()
        assert lib.ore_set_mesh_triangles_device(ctx, C.c_void_p(raw.data_ptr() + 4), n, None) == 0
        assert np.array_equal(renderer.debug_mesh("tris"), moved)
    finally:
        renderer.host_free(pinned)
        renderer.set_mesh(None)
