"""Soundness of the conservative culls on cubes and mesh leaves, no GPU: the light-cone cull of cubes_planes_block_light,
the leaf-ball cull of mesh_blocks_light and the primary tile-cone cull of mesh leaves (prep_frame_kernel + cone_touches),
restated in tests/primitive_cull_probe.cpp, must never reject a hit the reference's own tests report
(oracle_cube_intersect, oracle_tri_intersect).

The rays, origins and boxes are the awkward ones: directions with +-0 components, origins on face planes, edges and
corners, boxes in either corner order, flat, tiny, huge, far and non-finite.  cube::intersect reports hits outside its
box when a ray with D.k == +-0 starts on a face plane on axis k (a NaN slab, DESIGN.md 6b): the known-answer tests keep
that case, and the reproducer scene shows it changes a frame."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "ray-tracer-engine_b200", "csrc")
F32 = np.float32
N_CASES = 400_000   # per generator family below; three families (cubes, shadow leaves, primary leaves)


class CullProbe:
    def __init__(self, lib, oracle):
        self.lib = lib
        self.cube = C.cast(oracle.lib.oracle_cube_intersect, C.c_void_p)
        self.tri = C.cast(oracle.lib.oracle_tri_intersect, C.c_void_p)

    def _run(self, fn, O, D, box, tris=None):
        O, D, box = (np.ascontiguousarray(a, F32) for a in (O, D, box))
        out = np.zeros(O.shape[0], np.uint8)
        if tris is None:
            fn(self.cube, O.shape[0], O.ctypes.data, D.ctypes.data, box.ctypes.data, out.ctypes.data)
        else:
            tris = np.ascontiguousarray(tris, F32)
            fn(self.cube, self.tri, O.shape[0], O.ctypes.data, D.ctypes.data, box.ctypes.data, tris.ctypes.data,
               out.ctypes.data)
        return out

    def shadow_cubes(self, O, D, box):
        """bit 0 hit; bits 1 / 2: old / new cull rejects it for the ray alone; bits 3 / 4: in a 10-ray bundle"""
        return self._run(self.lib.probe_shadow_cubes, O, D, box)

    def shadow_leaves(self, O, D, box, tris):
        return self._run(self.lib.probe_shadow_leaves, O, D, box, tris)

    def primary_leaves(self, O, D, box, tris):
        """bit 0 hit; bits 1 / 2: cull without / with the eye-on-a-face-plane rule rejects it"""
        return self._run(self.lib.probe_primary_leaves, O, D, box, tris)


@pytest.fixture(scope="module")
def probe(tmp_path_factory, oracle_port):
    out = os.path.join(str(tmp_path_factory.mktemp("cull_probe")), "libprimitive_cull_probe.so")
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC,
                           os.path.join(ROOT, "tests", "primitive_cull_probe.cpp"), "-o", out], env=env)
    lib = C.CDLL(out)
    vp, i = C.c_void_p, C.c_int
    lib.probe_shadow_cubes.argtypes = [vp, i, vp, vp, vp, vp]
    lib.probe_shadow_leaves.argtypes = [vp, vp, i, vp, vp, vp, vp, vp]
    lib.probe_primary_leaves.argtypes = [vp, vp, i, vp, vp, vp, vp, vp]
    return CullProbe(lib, oracle_port)


# ---- generators -----------------------------------------------------------------------------------------------------

def random_boxes(rng, n):
    """(n, 6) c1, c2: either corner order, flat, tiny, huge (+-1e30), far (1e19..1e21 away, small), non-finite"""
    kind = rng.integers(0, 8, n)
    centre = rng.uniform(-20, 20, (n, 3))
    half = rng.uniform(0.05, 5, (n, 3))
    half[kind == 2, rng.integers(0, 3, n)[kind == 2]] = 0.0                     # flat
    half[kind == 3] *= 10.0 ** rng.uniform(-7, -3, (int((kind == 3).sum()), 1))  # tiny
    huge = kind == 4
    centre[huge] = rng.choice([-1e30, 1e30, 0.0], (int(huge.sum()), 3))
    half[huge] *= rng.choice([1.0, 1e29, 1e30], (int(huge.sum()), 1))
    far = kind == 5
    centre[far] = rng.uniform(-1, 1, (int(far.sum()), 3)) * 10.0 ** rng.uniform(19, 21, (int(far.sum()), 1))
    half[far] *= 10.0 ** rng.uniform(0, 14, (int(far.sum()), 1))
    c1, c2 = centre + half, centre - half
    swap = rng.random(n) < 0.5                                                   # the reference's order is c1 > c2
    c1[swap], c2[swap] = c2[swap].copy(), c1[swap].copy()
    box = np.concatenate([c1, c2], axis=1).astype(F32)
    bad = kind == 6
    pick = rng.integers(0, 6, n)
    box[bad, pick[bad]] = rng.choice(np.array([np.nan, np.inf, -np.inf], F32), int(bad.sum()))
    return box


def origins(rng, box):
    """inside the box or on 1, 2 or 3 of its face planes (a face, an edge, a corner); half of them then move away from
    the box along the other axes, so they stay on the face planes but leave the box and its ball (where a NaN slab can
    report a hit that the ball does not hold)"""
    n = box.shape[0]
    lo, hi = np.minimum(box[:, :3], box[:, 3:]), np.maximum(box[:, :3], box[:, 3:])
    with np.errstate(invalid="ignore", over="ignore"):
        O = (lo + (hi - lo) * rng.random((n, 3))).astype(F32)
        n_on = rng.integers(0, 4, n)
        on = np.zeros((n, 3), bool)
        for k in range(3):
            on[:, k] = rng.random(n) < n_on / 3.0
            which = rng.random(n) < 0.5
            O[on[:, k], k] = np.where(which[on[:, k]], box[on[:, k], k], box[on[:, k], 3 + k])
        away = (rng.random((n, 1)) < 0.5) & ~on
        O = np.where(away, O + rng.normal(0, 20, (n, 3)).astype(F32), O).astype(F32)
    bad = ~np.isfinite(O)
    O[bad] = rng.uniform(-20, 20, int(bad.sum())).astype(F32)
    return O


def directions(rng, O, box):
    """unit float directions: axis-aligned with +-0 components, one or two zero components, towards the box, random"""
    n = O.shape[0]
    with np.errstate(invalid="ignore", over="ignore"):
        target = (box[:, :3] + (box[:, 3:] - box[:, :3]) * rng.random((n, 3)).astype(F32)).astype(np.float64)
        D = target - O.astype(np.float64)
    D = np.where(np.isfinite(D), D, rng.normal(size=(n, 3)))
    D = np.where(rng.random((n, 1)) < 0.2, rng.normal(size=(n, 3)), D)
    n_zero = rng.integers(0, 3, n)
    for z in (1, 2):
        sel = n_zero >= z
        D[sel, rng.integers(0, 3, n)[sel]] = 0.0
    D[np.all(D == 0, axis=1), 0] = 1.0
    D = D / np.linalg.norm(D, axis=1, keepdims=True)
    D = D.astype(F32)
    D = np.where(D == 0, np.where(rng.random((n, 3)) < 0.5, F32(0.0), F32(-0.0)), D).astype(F32)   # signed zeros
    return np.ascontiguousarray(D)


def triangles_on_rays(rng, O, D, box, containing):
    """a triangle about a point of each ray (so many rays hit it), and with `containing` the leaf box of its vertices
    (the builder's boxes); otherwise the given box, which need not contain it"""
    n = O.shape[0]
    t0 = rng.uniform(0.01, 30, (n, 1))
    P = O.astype(np.float64) + D.astype(np.float64) * t0
    e = rng.normal(0, rng.uniform(0.01, 3, (n, 1, 1)), (n, 3, 3))
    e -= e.mean(axis=1, keepdims=True)
    flat = rng.random(n) < 0.3                                                   # triangles in an axis plane
    e[flat, :, rng.integers(0, 3, n)[flat]] = 0.0
    V = (P[:, None, :] + e).astype(F32)
    tris = np.ascontiguousarray(V.reshape(n, 9))
    if not containing:
        return tris, box
    lo, hi = V.min(axis=1), V.max(axis=1)
    return tris, np.ascontiguousarray(np.concatenate([lo, hi], axis=1), F32)


def cube_cases(seed, n=N_CASES):
    rng = np.random.default_rng(seed)
    box = random_boxes(rng, n)
    O = origins(rng, box)
    return O, directions(rng, O, box), box


# ---- known answers --------------------------------------------------------------------------------------------------

# the shadow ray of the reproducer scene below, reduced: it starts on the plane y = 0 with D.y = +0, the cube's bottom
# face is on y = 0, so its y slab is NaN and only the z slab decides - a hit at t ~ 350, nowhere near the cube
KAT_O = np.array([-2.0, 0.0, -0.5], F32)
KAT_D = (np.array([-1.0, 0.0, -0.05]) / np.linalg.norm([-1.0, 0.0, -0.05])).astype(F32)
KAT_CUBE = np.array([11, 1, -20, 10, 0, -30], F32)


def test_cube_intersect_reports_a_hit_outside_the_box_through_a_nan_slab(oracle_port):
    hit, t = oracle_port.cube_intersect(KAT_O, KAT_D, KAT_CUBE[:3], KAT_CUBE[3:])
    assert hit and t > 300, (hit, t)
    point = KAT_O + t * KAT_D
    assert point[0] < -300                                   # the cube spans x in [10, 11]
    # lower the cube by 0.5: the origin is inside the y slab, the test is the plain slab test and misses
    lowered = KAT_CUBE - np.array([0, 0.5, 0, 0, 0.5, 0], F32)
    assert not oracle_port.cube_intersect(KAT_O, KAT_D, lowered[:3], lowered[3:])[0]
    # a direction component of -0 does the same, a tiny nonzero one does not
    assert oracle_port.cube_intersect(KAT_O, KAT_D * np.array([1, -1, 1], F32), KAT_CUBE[:3], KAT_CUBE[3:])[0]
    nudged = KAT_D.copy()
    nudged[1] = F32(1e-30)
    assert not oracle_port.cube_intersect(KAT_O, nudged, KAT_CUBE[:3], KAT_CUBE[3:])[0]


def test_old_cube_cull_rejects_the_nan_slab_hit_and_the_guarded_one_keeps_it(probe):
    r = int(probe.shadow_cubes(KAT_O[None], KAT_D[None], KAT_CUBE[None])[0])
    assert r & 1, "the reference reports the hit"
    assert r & 2 and r & 8, "the predicate before the face-plane guard culls it (ray alone and in a bundle)"
    assert not (r & 4) and not (r & 16), "the guarded predicate keeps it"


def test_old_cube_cull_rejects_a_far_cube_through_an_overflowing_distance(probe):
    """|O - centre|^2 overflows to inf while the radius does not: sqrt(inf) * rsqrt(inf) = inf * 0 = NaN, which the
    old predicate took as a miss"""
    O = np.array([[0.0, 0.0, 0.0]], F32)
    D = np.array([[1.0, 0.0, 0.0]], F32)
    box = np.array([[3e19, 1.0, 1.0, 2e19, -1.0, -1.0]], F32)
    r = int(probe.shadow_cubes(O, D, box)[0])
    assert r & 1 and r & 2 and not (r & 4), r


# ---- the properties -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("seed", [0, 1, 2])
def test_cube_cone_cull_never_rejects_a_reported_hit(seed, probe):
    O, D, box = cube_cases(100 + seed)
    r = probe.shadow_cubes(O, D, box)
    hit = (r & 1) != 0
    assert hit.sum() > 0.2 * len(r), int(hit.sum())
    bad = hit & ((r & (4 | 16)) != 0)
    assert not bad.any(), (int(bad.sum()), O[bad][:3], D[bad][:3], box[bad][:3])
    # the generators reach the cases the guard is for: the old predicate loses hits here
    assert (hit & ((r & (2 | 8)) != 0)).sum() > 0


@pytest.mark.parametrize("containing", [True, False], ids=["builder_boxes", "caller_boxes"])
def test_leaf_cone_culls_never_reject_a_reported_triangle_hit(containing, probe):
    O, D, box = cube_cases(200 + containing)
    tris, box = triangles_on_rays(np.random.default_rng(300 + containing), O, D, box, containing)
    r = probe.shadow_leaves(O, D, box, tris)
    hit = (r & 1) != 0
    assert hit.sum() > 0.05 * len(r), int(hit.sum())
    bad = hit & ((r & (4 | 16)) != 0)
    assert not bad.any(), (int(bad.sum()), O[bad][:3], D[bad][:3], box[bad][:3], tris[bad][:3])
    if containing:
        # a triangle hit lies in a box that contains the triangle: even the unguarded cull keeps it (DESIGN.md 6c)
        assert not (hit & ((r & (2 | 8)) != 0)).any()
    # primary pass: eye O, the tile cone about D
    p = probe.primary_leaves(O, D, box, tris)
    phit = (p & 1) != 0
    bad = phit & ((p & 4) != 0)
    assert not bad.any(), (int(bad.sum()), O[bad][:3], D[bad][:3], box[bad][:3])
    if containing:
        assert not (phit & ((p & 2) != 0)).any()


def test_caller_boxes_need_the_face_plane_rule(probe, oracle_port):
    """a leaf whose box does not contain its triangle (ore_set_mesh takes the caller's boxes), an origin on the box's
    bottom face plane and D.y == 0: the reference reports the triangle hit through the NaN slab, the cone cull without
    the face-plane rule rejects it, in the shadow pass and in the primary pass"""
    box = KAT_CUBE                                                     # bottom face on y = 0 (hi first, as given)
    D = KAT_D
    O = KAT_O
    t_far = 200.0
    P = O + t_far * D                                                  # far from the box, on the ray
    tri = np.concatenate([P + [0, -1, -1], P + [0, 1, -1], P + [0, 0, 2]]).astype(F32)
    assert oracle_port.cube_intersect(O, D, box[:3], box[3:])[0] and oracle_port.tri_intersect(O, D, tri)[0]
    r = int(probe.shadow_leaves(O[None], D[None], box[None], tri[None])[0])
    assert r & 1 and r & 2 and not (r & 4) and not (r & 16), r
    p = int(probe.primary_leaves(O[None], D[None], box[None], tri[None])[0])
    assert p & 1 and p & 2 and not (p & 4), p


def test_the_reproducer_scene_changes_with_the_far_cube(oracle_best, pkg):
    """the scene the GPU tests render: a cube behind the camera, away from the light, with its bottom face on y = 0,
    changes pixels of row 16 (whose hit points have y == 0 and whose first shadow ray has D.y == +-0)"""
    from test_random_primitives_gpu import reproducer_scene
    sc, cam, W, H = reproducer_scene(pkg, with_cube=False)
    a = oracle_best.render(sc, cam, W, H)
    sc, cam, W, H = reproducer_scene(pkg, with_cube=True)
    b = oracle_best.render(sc, cam, W, H)
    diff = np.argwhere(a["pixels"] != b["pixels"])
    assert len(diff) > 0 and set(diff[:, 0]) == {16}, diff
    assert np.array_equal(a["ids"], b["ids"])
    sc, cam, W, H = reproducer_scene(pkg, with_cube=True, lift=-0.5)
    assert np.array_equal(oracle_best.render(sc, cam, W, H)["pixels"], a["pixels"])


# ---- the restatement against the reference's own code on these rays ---------------------------------------------------

def test_port_matches_the_reference_on_adversarial_rays(oracle_port, oracle_ref):
    """oracle.c's cube, plane and triangle tests, which the properties above call, bit for bit against the reference's
    own cube::intersect, plane::intersect and mesh::rayIntersect (the _ref build) on a sample of the same generators"""
    if not oracle_ref.has_primitive_tests:
        pytest.skip("this _ref build predates the single-primitive entry points")
    rng = np.random.default_rng(900)
    O, D, box = cube_cases(901, n=4000)
    tris, _ = triangles_on_rays(rng, O, D, box, containing=False)
    normals = rng.normal(size=(len(O), 3)).astype(F32) * rng.choice(np.array([0.0, 0.1, 1.0, 10.0], F32), (len(O), 1))
    bits = lambda r: tuple(np.float32(x).view(np.uint32) if i else bool(x) for i, x in enumerate(r))   # noqa: E731
    try:
        for i in range(len(O)):
            o, d, b = O[i], D[i], box[i]
            assert bits(oracle_port.cube_intersect(o, d, b[:3], b[3:])) == bits(oracle_ref.cube_intersect(o, d, b[:3], b[3:])), i
            assert bits(oracle_port.plane_intersect(o, d, b[:3], normals[i])) == \
                bits(oracle_ref.plane_intersect(o, d, b[:3], normals[i])), i
            assert bits(oracle_port.tri_intersect(o, d, tris[i])) == bits(oracle_ref.tri_intersect(o, d, tris[i])), i
    except NotImplementedError as e:
        pytest.skip(str(e))
