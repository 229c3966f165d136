"""Randomised and adversarial scenes of cubes, planes and triangle meshes: the default kernels (tile-cone cull of the
mesh leaves, light-cone culls of cubes and leaves) must give exactly the frame of FUSED_SHADOW and of the exhaustive
mode, and the oracle's ids, t and pixels.  The scenes put cameras and lights on face planes, look along the axes (exact
+-0 direction components), and mix both corner orders, flat, overlapping and coplanar cubes, non-unit and zero plane
normals, degenerate, NaN and duplicate triangles.  The reproducer scene is the one where cube::intersect reports a hit
through a NaN slab (DESIGN.md 6b, tests/test_primitive_cull_cpu.py); the tie scenes check the reference's order across
kinds; a 4-camera batch and 3-row bands must equal single full frames."""
import numpy as np
import pytest

from test_host_mesh import host_build, host_lib, write_grid_obj  # noqa: F401  (fixture re-export)
from test_mesh_refit_cpu import boxes6, build_probe
from test_parity_gpu import assert_pixels_close, libm_matches  # noqa: F401  (fixture re-export)

pytestmark = pytest.mark.gpu
F32 = np.float32


@pytest.fixture(scope="module")
def mesh_probe(tmp_path_factory):
    return build_probe(tmp_path_factory.mktemp("mesh_probe"))


def _base(pkg, spheres, lights):
    b = pkg.scene.reference_scene(0, 1)
    return pkg.scene.Scene(spheres=np.ascontiguousarray(spheres, F32), lights=np.ascontiguousarray(lights, F32),
                           texture=b.texture, sky=b.sky)


def reproducer_scene(pkg, with_cube=True, lift=0.0, around=None):
    """33 x 33, aspect 1, camera at (0, 0, -10) looking down +z: row 16 has D.y == 0 and hit points with y == 0.  One
    sphere, one point light at (-20, 0, -3).  The cube lies behind the camera, away from the light, its bottom face on
    y = lift.  around: extra planes and a mesh (a Scene whose planes / mesh are added)."""
    sc = _base(pkg, [[0, 0, 0, 4]], [[-20, 0, -3, 0, 1, 1, 1]])
    sc.aspect = F32(1.0)
    cubes = [[11, 1 + lift, -20, 10, lift, -30]] if with_cube else []
    sc.cubes = np.array(cubes, F32).reshape(-1, 6)
    if around is not None:
        sc.planes, sc.mesh = around.planes, around.mesh
    return sc, pkg.scene.Camera(org=(0.0, 0.0, -10.0), yaw=0.0, pitch=0.0), 33, 33


def render_all(renderer, pkg, sc, cam, W, H, **kw):
    """(pixels, ids, t) of the default mode, asserted equal to FUSED_SHADOW, EXHAUSTIVE and both"""
    F = pkg.capi
    renderer.set_scene(sc)
    a = renderer.render(cam, W, H, aspect=float(sc.aspect), **kw)
    ia, ta = renderer.hits(a.shape[0], W)
    for flags in (F.ORE_FLAG_FUSED_SHADOW, F.ORE_FLAG_EXHAUSTIVE, F.ORE_FLAG_FUSED_SHADOW | F.ORE_FLAG_EXHAUSTIVE):
        b = renderer.render(cam, W, H, aspect=float(sc.aspect), flags=flags, **kw)
        ib, tb = renderer.hits(b.shape[0], W)
        assert np.array_equal(ia, ib), (sc.name, flags, int(np.count_nonzero(ia != ib)))
        assert np.array_equal(ta.view(np.uint32), tb.view(np.uint32)), (sc.name, flags)
        assert np.array_equal(a, b), (sc.name, flags, int(np.count_nonzero(a != b)))
    return a, ia, ta


def assert_oracle(px, ids, t, ref, libm_matches):
    assert np.array_equal(ids, ref["ids"]), int(np.count_nonzero(ids != ref["ids"]))
    assert np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32))
    if libm_matches:
        assert np.array_equal(px, ref["pixels"]), int(np.count_nonzero(px != ref["pixels"]))
    else:
        assert_pixels_close(px, ref["pixels"])


# ---- random awkward scenes ------------------------------------------------------------------------------------------

ORACLE_SEEDS = [0, 4, 8, 12, 16, 20]   # at most one plane: the reference's own code takes one


def _mesh(pkg, rng, kind, host_lib, mesh_probe, tmp_path):
    """a grid or the torus, deformed, with awkward triangles, its boxes refit by the host functions of
    ore_mesh_refit.h"""
    from cases import torus_mesh
    if kind == "torus":
        m = torus_mesh()
    else:
        obj = str(tmp_path / "grid.obj")
        write_grid_obj(obj, "vtn", n=int(rng.integers(3, 12)), seed=int(rng.integers(0, 100)))
        m = pkg.scene.Mesh.from_arrays(host_build(host_lib, obj))
    tris = m.tris.copy()
    tris[:, :9] += rng.normal(0, 0.15, tris[:, :9].shape).astype(F32)
    n = tris.shape[0]
    pick = rng.permutation(n)
    tris[pick[0], 3:6] = tris[pick[0], 0:3]                                       # degenerate: two equal vertices
    tris[pick[1], 6:9] = 2 * tris[pick[1], 3:6] - tris[pick[1], 0:3]              # collinear
    tris[pick[2]] = tris[pick[3]]                                                 # duplicate
    if rng.random() < 0.5:
        tris[pick[4], int(rng.integers(0, 9))] = np.nan                           # a NaN vertex
    boxes, _ = mesh_probe.arrays(tris, m.box_bounds, m.box_offsets, m.box_indices, refit=True)
    return pkg.scene.Mesh(np.ascontiguousarray(tris, F32), m.has_normals, np.ascontiguousarray(boxes6(boxes)),
                          m.box_offsets, m.box_indices)


def random_primitive_scene(pkg, seed, host_lib, mesh_probe, tmp_path):
    rng = np.random.default_rng(7000 + seed)
    S = pkg.scene
    sph = S.reference_scene(int(rng.choice([0, 1, 8, 64])), 1 + seed % 3)
    lights = S.REFERENCE_LIGHTS.copy()
    lights[:, 3] = F32(rng.choice([0.0, 1.0, 20.0]))
    axis_view = seed % 3 == 0
    if axis_view:
        cam = S.Camera(org=tuple(float(F32(v)) for v in rng.uniform(0, 10, 3)), yaw=float(rng.choice([0, 90, 180, 270])),
                       pitch=0.0)
        W = H = int(rng.choice([31, 45, 61]))
        aspect = F32(1.0)
    else:
        cam = S.Camera(org=tuple(float(F32(v)) for v in rng.uniform(-5, 15, 3)), yaw=float(rng.uniform(0, 360)),
                       pitch=float(rng.uniform(-60, 60)))
        W, H = 97, 61
        aspect = S.REFERENCE_ASPECT
    O = np.array(cam.org, F32)
    # cubes: both corner orders, flat, overlapping, sharing face planes, faces on the camera's / a light's coordinates
    nc = int(rng.integers(1, 41))
    centre = rng.uniform(0, 10, (nc, 3))
    half = rng.uniform(0.05, 1.5, (nc, 3))
    half[rng.random(nc) < 0.2, int(rng.integers(0, 3))] = 0.0
    c1, c2 = (centre + half).astype(F32), (centre - half).astype(F32)
    for i in range(1, nc):
        r = rng.random()
        if r < 0.15:                                                             # overlapping copy
            c1[i], c2[i] = c1[i - 1] + F32(0.3), c2[i - 1] + F32(0.3)
        elif r < 0.3:                                                            # sharing a face plane
            k = int(rng.integers(0, 3))
            c2[i, k] = c1[i - 1, k]
        elif r < 0.45:                                                           # a face on the camera's coordinate
            k = int(rng.integers(0, 3))
            (c1 if rng.random() < 0.5 else c2)[i, k] = O[k]
        elif r < 0.55:                                                           # ... or a light's
            k = int(rng.integers(0, 3))
            (c1 if rng.random() < 0.5 else c2)[i, k] = lights[int(rng.integers(0, len(lights))), k]
    if rng.random() < 0.3:                                                       # the camera inside a cube
        c1[0], c2[0] = O + F32(0.7), O - F32(0.4)
    if rng.random() < 0.3:                                                       # a light inside a cube
        c1[-1], c2[-1] = lights[0, :3] + F32(0.5), lights[0, :3] - F32(0.5)
    swap = rng.random(nc) < 0.5
    c1[swap], c2[swap] = c2[swap].copy(), c1[swap].copy()
    cubes = np.concatenate([c1, c2], axis=1).astype(F32)
    # planes: non-unit and zero normals, one through the camera
    n_pl = int(rng.integers(0, 5)) if seed not in ORACLE_SEEDS else int(rng.integers(0, 2))
    planes = np.zeros((n_pl, 6), F32)
    for i in range(n_pl):
        planes[i, :3] = O if i == 0 and rng.random() < 0.4 else rng.uniform(-2, 8, 3)
        nrm = rng.normal(size=3) * rng.choice([0.1, 1.0, 10.0])
        if rng.random() < 0.15:
            nrm[:] = 0.0
        planes[i, 3:] = nrm
    kind = rng.choice(["none", "grid", "torus"])
    mesh = None if kind == "none" else _mesh(pkg, rng, kind, host_lib, mesh_probe, tmp_path)
    if mesh is not None and axis_view:                                          # the eye on a leaf box's face plane
        b = mesh.box_bounds[int(rng.integers(0, mesh.n_boxes))]
        org = list(cam.org)
        org[1] = float(b[1]) if np.isfinite(b[1]) else org[1]
        cam = S.Camera(org=tuple(org), yaw=cam.yaw, pitch=cam.pitch)
    sc = S.Scene(spheres=sph.spheres, lights=lights, texture=sph.texture, sky=sph.sky, aspect=aspect, cubes=cubes,
                 planes=planes, mesh=mesh, name=f"prims{seed}")
    return sc, cam, W, H


@pytest.mark.parametrize("seed", list(range(24)))
def test_default_equals_fused_and_exhaustive_on_random_primitive_scenes(seed, renderer, pkg, host_lib, mesh_probe,
                                                                         tmp_path, oracle_best, libm_matches):
    sc, cam, W, H = random_primitive_scene(pkg, seed, host_lib, mesh_probe, tmp_path)
    try:
        px, ids, t = render_all(renderer, pkg, sc, cam, W, H)
        if seed in ORACLE_SEEDS:
            assert_oracle(px, ids, t, oracle_best.render(sc, cam, W, H), libm_matches)
    finally:
        renderer.set_mesh(None)


# ---- the reproducer -------------------------------------------------------------------------------------------------

def test_nan_slab_reproducer_matches_exhaustive_and_the_oracle(renderer, pkg, oracle_best, libm_matches):
    sc, cam, W, H = reproducer_scene(pkg)
    px, ids, t = render_all(renderer, pkg, sc, cam, W, H)
    ref = oracle_best.render(sc, cam, W, H)
    assert_oracle(px, ids, t, ref, libm_matches)
    bare, _, _ = render_all(renderer, pkg, *reproducer_scene(pkg, with_cube=False))
    assert np.count_nonzero(bare != px) > 0, "the far cube must darken row 16"


def test_nan_slab_reproducer_among_planes_and_a_mesh(renderer, pkg, oracle_best, libm_matches, mesh_probe):
    from cases import torus_mesh
    m = torus_mesh()
    tris = m.tris.copy()
    tris[:, 0:9:3] -= F32(5.0)                                                     # the torus about (0, 5, 3)
    tris[:, 2:9:3] -= F32(2.0)
    boxes, _ = mesh_probe.arrays(tris, m.box_bounds, m.box_offsets, m.box_indices, refit=True)
    mesh = pkg.scene.Mesh(tris, m.has_normals, np.ascontiguousarray(boxes6(boxes)), m.box_offsets, m.box_indices)
    around = pkg.scene.Scene(spheres=np.zeros((0, 4), F32), lights=np.zeros((0, 7), F32), texture=None, sky=None,
                             planes=np.array([[0, -3, 0, 0, 2, 0]], F32), mesh=mesh)
    sc, cam, W, H = reproducer_scene(pkg, around=around)
    try:
        px, ids, t = render_all(renderer, pkg, sc, cam, W, H)
        assert_oracle(px, ids, t, oracle_best.render(sc, cam, W, H), libm_matches)
    finally:
        renderer.set_mesh(None)


# ---- caller boxes that do not contain their triangles -----------------------------------------------------------------

def _one_leaf(pkg, tri9, box6):
    tri = np.zeros((1, 27), F32)
    tri[0, :9] = tri9
    tri[0, 9:12] = [0, 0, -1]
    return pkg.scene.Mesh(tri, False, np.array([box6], F32), np.array([0, 1], np.int32), np.array([0], np.int32))


def test_leaf_boxes_that_do_not_contain_their_triangles(renderer, pkg, oracle_best, libm_matches):
    """ore_set_mesh takes the caller's boxes.  In the reproducer scene (eye and row 16's hit points on y = 0, row 16's
    primary rays and the first shadow ray with D.y == +-0), a leaf whose box has its bottom face on y = 0 lists a
    triangle far from the box.  The reference reaches that triangle only through the box's NaN slab: the oracle's frame
    changes with the mesh, and the same box lifted by 0.001 leaves the frame unchanged."""
    def check(tri9, box6, what):
        sc, cam, W, H = reproducer_scene(pkg, with_cube=False)
        bare = oracle_best.render(sc, cam, W, H)
        lifted = np.array(box6, F32) + np.array([0, 0.001, 0, 0, 0.001, 0], F32)
        sc.mesh = _one_leaf(pkg, tri9, lifted)
        assert np.array_equal(oracle_best.render(sc, cam, W, H)["pixels"], bare["pixels"]), what
        sc.mesh = _one_leaf(pkg, tri9, box6)
        ref = oracle_best.render(sc, cam, W, H)
        assert np.count_nonzero(ref["pixels"] != bare["pixels"]) > 0, what
        px, ids, t = render_all(renderer, pkg, sc, cam, W, H)
        assert_oracle(px, ids, t, ref, libm_matches)
        return ids, ref
    try:
        # shadow pass: the triangle lies between row 16's hit points and the light; the box lies behind the camera
        check([-30, -6, -9, -30, 6, -9, -30, 0, 6], [11, 1, -20, 10, 0, -30], "shadow")
        # primary pass: the triangle faces the eye at z = -5, the box lies far off to the side (x in [100, 101]), out
        # of every tile cone: without the eye-on-a-face-plane rule the tile cull would skip the leaf
        ids, ref = check([-3, -1, -5, 3, -1, -5, 0, 1, -5], [101, 1, -2, 100, 0, -8], "primary")
        seen = np.argwhere(ref["ids"] == 1)
        assert len(seen) > 0 and set(seen[:, 0]) == {16}, seen
    finally:
        renderer.set_mesh(None)


# ---- ties across kinds ----------------------------------------------------------------------------------------------

def _tie_scene(pkg, case):
    """several primitives hit at the same t; the reference's order decides: triangles, spheres, cubes, planes, each
    lowest index first"""
    sc = _base(pkg, np.zeros((0, 4), F32), [[3, 8, -6, 0, 1, 1, 1]])
    cube = [2, 2, 2, 0, 0, 0]
    quad = [[0, 2, 0, 2, 2, 0, 2, 2, 2], [0, 2, 0, 2, 2, 2, 0, 2, 2]]               # the cube's top face, y = 2
    def tris_of(rows):
        t = np.zeros((len(rows), 27), F32)
        t[:, :9] = rows
        t[:, 10] = 1.0
        return t
    if case == "plane_on_cube_face":
        sc.cubes = np.array([cube], F32)
        sc.planes = np.array([[0, 2, 0, 0, 1, 0]], F32)
    elif case == "identical_cubes":
        sc.cubes = np.array([cube, cube, [0, 0, 0, 2, 2, 2]], F32)
    elif case in ("triangle_on_cube_face", "duplicate_triangle_in_two_leaves"):
        sc.cubes = np.array([cube], F32)
        rows = quad if case == "triangle_on_cube_face" else quad + quad
        idx = [0, 1] if case == "triangle_on_cube_face" else [2, 0, 1, 3]
        offs = [0, 2] if case == "triangle_on_cube_face" else [0, 2, 4]
        bb = [[0, 2, 0, 2, 2, 2]] * (len(offs) - 1)
        sc.mesh = pkg.scene.Mesh(tris_of(rows), False, np.array(bb, F32), np.array(offs, np.int32), np.array(idx, np.int32))
    elif case == "sphere_tangent_to_cube_face":
        sc.spheres = np.array([[1, 3, 1, 1]], F32)                                  # radius 1 about (1, 3, 1): touches y = 2
        sc.cubes = np.array([cube], F32)
        sc.planes = np.array([[0, 2, 0, 0, 1, 0]], F32)
    return sc


TIE_CASES = ["plane_on_cube_face", "identical_cubes", "triangle_on_cube_face", "duplicate_triangle_in_two_leaves",
             "sphere_tangent_to_cube_face"]


@pytest.mark.parametrize("case", TIE_CASES)
def test_ties_across_kinds_follow_the_reference_order(case, renderer, pkg, oracle_best, libm_matches):
    sc = _tie_scene(pkg, case)
    cams = [pkg.scene.Camera(org=(1.0, 6.0, -3.0), yaw=0.0, pitch=45.0),
            pkg.scene.Camera(org=(1.0, 7.0, 1.0), yaw=0.0, pitch=90.0)]
    try:
        for cam in cams:
            px, ids, t = render_all(renderer, pkg, sc, cam, 45, 45)
            ref = oracle_best.render(sc, cam, 45, 45)
            assert_oracle(px, ids, t, ref, libm_matches)
            assert (ids >= 0).any()
    finally:
        renderer.set_mesh(None)


# ---- batches and bands ----------------------------------------------------------------------------------------------

def test_batch_and_bands_of_a_primitive_scene_equal_single_frames(renderer, pkg, host_lib, mesh_probe, tmp_path):
    import torch
    seed = next(s for s in range(3, 60, 3) if random_primitive_scene(pkg, s, host_lib, mesh_probe, tmp_path)[0].mesh
                is not None)
    sc, cam, W, H = random_primitive_scene(pkg, seed, host_lib, mesh_probe, tmp_path)
    try:
        renderer.set_scene(sc)
        asp = float(sc.aspect)
        cams = [cam] + [pkg.scene.Camera(org=tuple(float(F32(c + d)) for c in cam.org), yaw=cam.yaw + 30 * k,
                                         pitch=cam.pitch) for k, d in ((1, 0.5), (2, -1.0), (3, 2.0))]
        singles = [renderer.render(c, W, H, aspect=asp).copy() for c in cams]
        out = torch.zeros((4, H, W), dtype=torch.int32, device="cuda:0")
        st = torch.cuda.Stream()
        st.wait_stream(torch.cuda.current_stream())
        renderer.render_batch_device(cams, W, H, [out[i].data_ptr() for i in range(4)], stream=st.cuda_stream, aspect=asp)
        st.synchronize()
        got = out.cpu().numpy().view(np.uint32)
        for i in range(4):
            assert np.array_equal(got[i], singles[i]), (i, int(np.count_nonzero(got[i] != singles[i])))
        for y0 in range(3):
            band = renderer.render(cam, W, H, y0=y0, y_step=3, aspect=asp)
            assert np.array_equal(band, singles[0][y0::3]), y0
    finally:
        renderer.set_mesh(None)
