"""The host reference of the mesh refit (csrc/ore_mesh_refit.h through tests/mesh_refit_probe.cpp, plain g++), no GPU:
on unchanged triangles it gives the reference builder's own leaf boxes; on NaN, +-inf, +-0 and huge vertices, empty and
one-triangle leaves it agrees with a literal transcription of getMinMaxP's sequential rule; and the leaf-sphere formula
keeps the bytes of the host loop ore_set_mesh ran before, NaNs included."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_host_mesh import host_build, host_lib, write_grid_obj  # noqa: F401  (fixture re-export)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "ray-tracer-engine_b200", "csrc")
GOLDEN = os.path.join(ROOT, "tests", "golden")
AWKWARD = np.array([np.nan, -np.nan, np.inf, -np.inf, 0.0, -0.0, 1e30, -1e30, 1.0, -2.5], dtype=np.float32)


class MeshProbe:
    def __init__(self, lib):
        self.lib = lib

    def arrays(self, tris, box_bounds, box_offsets, box_indices, refit=True):
        """boxes (2 n_boxes, 4) and box_sph (n_boxes, 4) as the device holds them after ore_set_mesh (refit False) or
        after ore_set_mesh_triangles_device (refit True) with these triangles"""
        tris = np.ascontiguousarray(tris, np.float32)
        bb = np.ascontiguousarray(box_bounds, np.float32).reshape(-1, 6)
        offs = np.ascontiguousarray(box_offsets, np.int32)
        idx = np.ascontiguousarray(box_indices, np.int32)
        n_boxes = bb.shape[0]
        boxes = np.zeros((2 * n_boxes, 4), np.float32)
        sph = np.zeros((n_boxes, 4), np.float32)
        idx_ptr = idx.ctypes.data if idx.size else np.zeros(1, np.int32).ctypes.data
        self.lib.ore_probe_mesh(tris.ctypes.data, offs.ctypes.data, idx_ptr, n_boxes, bb.ctypes.data, int(refit),
                                boxes.ctypes.data, sph.ctypes.data)
        return boxes, sph

    def ball(self, b6, before=False):
        b = np.ascontiguousarray(b6, np.float32)
        out = np.zeros(4, np.float32)
        (self.lib.ore_probe_host_ball_before if before else self.lib.ore_probe_mesh_box_ball)(b.ctypes.data, out.ctypes.data)
        return out


def build_probe(out_dir) -> MeshProbe:
    out = os.path.join(str(out_dir), "libmesh_refit_probe.so")
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC,
                           os.path.join(ROOT, "tests", "mesh_refit_probe.cpp"), "-o", out], env=env)
    lib = C.CDLL(out)
    vp, i = C.c_void_p, C.c_int
    lib.ore_probe_mesh.argtypes = [vp, vp, vp, i, vp, i, vp, vp]
    lib.ore_probe_mesh.restype = None
    lib.ore_probe_host_ball_before.argtypes = [vp, vp]
    lib.ore_probe_mesh_box_ball.argtypes = [vp, vp]
    return MeshProbe(lib)


@pytest.fixture(scope="module")
def mesh_probe(tmp_path_factory):
    return build_probe(tmp_path_factory.mktemp("mesh_probe"))


def torus_arrays():
    d = dict(np.load(os.path.join(GOLDEN, "mesh_torus.npz")))
    return d["tris"], d["box_bounds"], d["box_offsets"], d["box_indices"]


def boxes6(boxes):
    """(2 b, 4) lo / hi float4 -> (b, 6), the layout of box_bounds"""
    return np.concatenate([boxes[0::2, :3], boxes[1::2, :3]], axis=1)


def sequential_rule(tris, offs, idx, bounds):
    """getMinMaxP (kernel.cu:973-997) as bounds_of in host/ore_mesh.cpp applies it, literally, in float32"""
    out = bounds.copy()
    for j in range(len(offs) - 1):
        lst = idx[offs[j]:offs[j + 1]]
        if len(lst) == 0:
            continue
        lo = [np.float32(tris[lst[0], k]) for k in range(3)]
        hi = [np.float32(tris[lst[-1], k]) for k in range(3)]
        for i in lst:
            for v in range(3):
                for k in range(3):
                    x = np.float32(tris[i, 3 * v + k])
                    if x > hi[k]:
                        hi[k] = x
                    if x < lo[k]:
                        lo[k] = x
        out[j] = lo + hi
    return out


def awkward_mesh(seed=11):
    """60 triangles with NaN, +-inf, +-0 and +-1e30 among their vertices (the other 18 floats random too), leaves of
    0, 1, 2, 5 and 40 entries listed in shuffled order, repeats included"""
    rng = np.random.default_rng(seed)
    n = 60
    tris = rng.uniform(-3, 3, size=(n, 27)).astype(np.float32)
    pick = rng.integers(0, len(AWKWARD), size=(n, 9))
    mask = rng.uniform(size=(n, 9)) < 0.45
    tris[:, :9] = np.where(mask, AWKWARD[pick], tris[:, :9])
    tris[7, :9] = 0.0                       # every vertex +0 ...
    tris[8, :9] = -0.0                      # ... every vertex -0: which one a leaf keeps is the rule's order
    tris[9, :9] = np.nan
    lists = [[], [9], [7, 8], [8, 7, 8, 7, 8], list(rng.permutation(n)[:40]), [], [8], [3, 9, 3], list(rng.permutation(n)[:12])]
    offs = np.concatenate([[0], np.cumsum([len(x) for x in lists])]).astype(np.int32)
    idx = np.array([i for x in lists for i in x], dtype=np.int32)
    bounds = rng.uniform(-1, 1, size=(len(lists), 6)).astype(np.float32)
    return tris, bounds, offs, idx


def test_probe_reproduces_the_reference_builders_boxes_on_the_torus(mesh_probe):
    """tests/golden/mesh_torus.npz was built by the reference's own loader and builder"""
    tris, bb, offs, idx = torus_arrays()
    boxes, sph = mesh_probe.arrays(tris, np.zeros_like(bb), offs, idx, refit=True)
    assert np.array_equal(boxes6(boxes).view(np.uint32), bb.view(np.uint32))
    assert np.all(boxes[:, 3] == 0)
    _, sph_set = mesh_probe.arrays(tris, bb, offs, idx, refit=False)
    assert np.array_equal(sph.view(np.uint32), sph_set.view(np.uint32))


@pytest.mark.parametrize("n", [4, 23, 200])
def test_probe_reproduces_the_host_builders_boxes_on_grids(n, mesh_probe, host_lib, tmp_path):
    obj = str(tmp_path / f"grid{n}.obj")
    write_grid_obj(obj, "vtn", n=n)
    d = host_build(host_lib, obj, cap_tris=1 << 17)
    assert d["tris"].shape[0] == 2 * (n - 1) ** 2
    boxes, _ = mesh_probe.arrays(d["tris"], np.zeros_like(d["box_bounds"]), d["box_offsets"], d["box_indices"], refit=True)
    assert np.array_equal(boxes6(boxes).view(np.uint32), d["box_bounds"].view(np.uint32))


@pytest.mark.parametrize("seed", [11, 12, 13])
def test_probe_follows_the_sequential_rule_on_awkward_values(seed, mesh_probe):
    tris, bounds, offs, idx = awkward_mesh(seed)
    boxes, _ = mesh_probe.arrays(tris, bounds, offs, idx, refit=True)
    want = sequential_rule(tris, offs, idx, bounds)
    assert np.array_equal(boxes6(boxes).view(np.uint32), want.view(np.uint32))
    # the cases the rule decides by its order: empty leaves keep their box, a NaN seed stays, -0 / +0 keep the first met
    got = boxes6(boxes)
    assert np.array_equal(got[0].view(np.uint32), bounds[0].view(np.uint32))
    assert np.all(np.isnan(got[1]))
    assert np.all(np.signbit(got[2][:3]) == False) and np.all(np.signbit(got[2][3:]))   # noqa: E712  lo from tri 7, hi from tri 8
    assert np.all(np.signbit(got[3][:3])) and np.all(np.signbit(got[3][3:]))


def test_leaf_sphere_keeps_the_bytes_of_the_former_host_loop(mesh_probe):
    """finite, infinite, NaN (both signs, other payloads, signalling) and +-0 box coordinates in every combination the
    ball can meet"""
    rng = np.random.default_rng(5)
    payloads = np.array([0x7fc12345, 0xffd00001, 0x7f800001], np.uint32).view(np.float32)
    values = np.concatenate([AWKWARD, payloads])
    cases = [rng.uniform(-50, 50, size=6).astype(np.float32) for _ in range(200)]
    for _ in range(5000):
        b = rng.uniform(-5, 5, size=6).astype(np.float32)
        m = rng.uniform(size=6) < 0.45
        b[m] = values[rng.integers(0, len(values), size=int(m.sum()))]
        cases.append(b)
    for b in cases:
        want = mesh_probe.ball(b, before=True)
        got = mesh_probe.ball(b)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (b, got.view(np.uint32), want.view(np.uint32))
