"""The host restatement of the reference's flat-BVH builder (ore_build_flat_bvh in host/ore_mesh.cpp, through
tests/mesh_build_probe.cpp, plain g++), no GPU: it reproduces the reference's own builder on the torus and the shim's
OBJ path on grids, and agrees with a literal Python transcription of the rule ore_set_mesh_device builds on the GPU
on awkward inputs: NaN, +-inf, +-0 and +-1e30 vertices, NaN first vertices, all split keys equal, 1 to 7 triangles,
duplicate triangles and a mesh that reaches 1024 leaves.  tests/test_mesh_build_gpu.py compares the device arrays with
the same probe."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_host_mesh import host_build, host_lib, write_grid_obj  # noqa: F401  (fixture re-export)
from test_mesh_refit_cpu import AWKWARD, torus_arrays

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "ray-tracer-engine_b200", "host")


class BuildProbe:
    def __init__(self, lib):
        self.lib = lib

    def build(self, tris):
        """(box_bounds (b, 6) float32, box_offsets (b + 1,) int32, box_indices int32) of ore_build_flat_bvh(mesh, 10)"""
        tris = np.ascontiguousarray(tris, np.float32).reshape(-1, 27)
        n = tris.shape[0]
        cap = max(n, 1)
        bb = np.zeros((min(cap, 1024), 6), np.float32)
        offs = np.zeros(min(cap, 1024) + 1, np.int32)
        idx = np.zeros(cap, np.int32)
        nb = self.lib.ore_probe_build_flat_bvh(tris.ctypes.data, n, bb.ctypes.data, offs.ctypes.data, idx.ctypes.data,
                                               bb.shape[0], idx.size)
        assert nb >= 0
        return bb[:nb].copy(), offs[:nb + 1].copy(), idx[:offs[nb]].copy()


def build_probe(out_dir) -> BuildProbe:
    out = os.path.join(str(out_dir), "libmesh_build_probe.so")
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC",
                           os.path.join(ROOT, "tests", "mesh_build_probe.cpp"), os.path.join(HOST, "ore_mesh.cpp"),
                           "-o", out], env=env)
    lib = C.CDLL(out)
    vp, i = C.c_void_p, C.c_int
    lib.ore_probe_build_flat_bvh.argtypes = [vp, i, vp, vp, vp, i, i]
    lib.ore_probe_build_flat_bvh.restype = i
    return BuildProbe(lib)


@pytest.fixture(scope="module")
def build_probe_lib(tmp_path_factory):
    return build_probe(tmp_path_factory.mktemp("mesh_build_probe"))


def flat_bvh_rule(tris, layers=10):
    """The builder's rule, literally (ore_build_flat_bvh; createBvhMesh, kernel.cu:782-936): one root box, ten layers,
    a box of more than 5 triangles split on axis split_dir (0 -> y, 1 -> x, 2 -> z; advanced after every split box) at
    (hi + lo) / 2 in float32 by the first vertex's coordinate (<= goes low), non-empty sides appended lo then hi, bounds
    by getMinMaxP.  Returns the arrays of BuildProbe.build."""
    t32 = np.ascontiguousarray(tris, np.float32).reshape(-1, 27)
    T = t32.astype(np.float64).tolist()   # float32 values exactly; the rule only compares them

    def bounds_of(lst):
        lo = [T[lst[0]][k] for k in range(3)]
        hi = [T[lst[-1]][k] for k in range(3)]
        for i in lst:
            row = T[i]
            for v in range(3):
                for k in range(3):
                    x = row[3 * v + k]
                    if x > hi[k]:
                        hi[k] = x
                    if x < lo[k]:
                        lo[k] = x
        return lo + hi

    n = len(T)
    if n == 0:
        return np.zeros((0, 6), np.float32), np.zeros(1, np.int32), np.zeros(0, np.int32)
    prev = [(list(range(n)), bounds_of(list(range(n))))]
    split_dir = 0
    with np.errstate(all="ignore"):
        for _ in range(layers):
            nxt = []
            for lst, b in prev:
                if len(lst) > 5:
                    k = (1, 0, 2)[split_dir]
                    p = float((np.float32(b[3 + k]) + np.float32(b[k])) / np.float32(2))
                    lo_side = [i for i in lst if T[i][k] <= p]
                    hi_side = [i for i in lst if not T[i][k] <= p]
                    for side in (lo_side, hi_side):
                        if side:
                            nxt.append((side, bounds_of(side)))
                    split_dir = (split_dir + 1) % 3
                else:
                    nxt.append((lst, b))
            prev = nxt
    bb = np.array([b for _, b in prev], np.float64).astype(np.float32).reshape(-1, 6)
    offs = np.concatenate([[0], np.cumsum([len(lst) for lst, _ in prev])]).astype(np.int32)
    idx = np.array([i for lst, _ in prev for i in lst], np.int32)
    return bb, offs, idx


# ---- the awkward meshes (shared with tests/test_mesh_build_gpu.py) -------------------------------------------------------

def random_tris(n, seed, scale=3.0):
    rng = np.random.default_rng(seed)
    return rng.uniform(-scale, scale, size=(n, 27)).astype(np.float32)


def awkward_values(n=300, seed=21):
    """NaN, +-inf, +-0 and +-1e30 among the vertices"""
    rng = np.random.default_rng(seed)
    tris = random_tris(n, seed)
    pick = rng.integers(0, len(AWKWARD), size=(n, 9))
    mask = rng.uniform(size=(n, 9)) < 0.3
    tris[:, :9] = np.where(mask, AWKWARD[pick], tris[:, :9])
    return tris


def nan_first_vertices(n=200, seed=22):
    """a third of the first vertices NaN on one or all axes: NaN keys go to the hi side, NaN seeds stay"""
    rng = np.random.default_rng(seed)
    tris = random_tris(n, seed)
    rows = rng.permutation(n)[: n // 3]
    tris[rows[: len(rows) // 2], 0:3] = np.nan
    tris[rows[len(rows) // 2:], rng.integers(0, 3)] = np.nan
    tris[0, 0:3] = np.nan         # the root's lo seed
    tris[n - 1, 1] = np.nan       # the root's hi seed on y
    return tris


def equal_keys(n=50, seed=23):
    """every first vertex the same point: each split leaves the hi side empty, and split_dir still advances"""
    tris = random_tris(n, seed)
    tris[:, 0:3] = np.float32([0.5, -1.25, 2.0])
    return tris


def duplicates(n=240, seed=24):
    """triangles repeated (same records) at scattered places"""
    rng = np.random.default_rng(seed)
    base = random_tris(n // 4, seed)
    return np.ascontiguousarray(base[rng.integers(0, base.shape[0], size=n)])


def mixed_signed_zeros(n=120, seed=25):
    """only -0 / +0 and a few ones: which zero a box keeps is the rule's order"""
    rng = np.random.default_rng(seed)
    vals = np.array([0.0, -0.0, 1.0, -1.0], np.float32)
    return np.ascontiguousarray(vals[rng.integers(0, 4, size=(n, 27))])


def leaves_1024(n=24000, seed=26):
    """uniform triangles: every box splits into two non-empty halves down to the 1024 leaves of layer 10"""
    rng = np.random.default_rng(seed)
    c = rng.uniform(-50, 50, size=(n, 1, 3))
    v = c + rng.uniform(-0.05, 0.05, size=(n, 3, 3))
    tris = np.zeros((n, 27), np.float32)
    tris[:, :9] = v.reshape(n, 9)
    tris[:, 9:] = rng.uniform(-1, 1, size=(n, 18))
    return tris


AWKWARD_CASES = {
    "awkward_values": awkward_values,
    "nan_first_vertices": nan_first_vertices,
    "equal_keys": equal_keys,
    "duplicates": duplicates,
    "signed_zeros": mixed_signed_zeros,
    **{f"n{k}": (lambda k=k: random_tris(k, 30 + k)) for k in range(1, 8)},
}


def assert_same_build(got, want, what):
    for name, g, w in zip(("box_bounds", "box_offsets", "box_indices"), got, want):
        assert g.shape == w.shape, (what, name, g.shape, w.shape)
        assert g.tobytes() == w.tobytes(), (what, name, int(np.count_nonzero(g.view(np.uint32) != w.view(np.uint32))))


# ---- tests ------------------------------------------------------------------------------------------------------------

def test_probe_reproduces_the_reference_builder_on_the_torus(build_probe_lib):
    """tests/golden/mesh_torus.npz was built by the reference's own loader and builder"""
    tris, bb, offs, idx = torus_arrays()
    assert_same_build(build_probe_lib.build(tris), (bb, offs, idx), "torus")
    assert_same_build(flat_bvh_rule(tris), (bb, offs, idx), "torus rule")


@pytest.mark.parametrize("n", [4, 23, 200])
def test_probe_equals_the_obj_path_on_grids(n, build_probe_lib, host_lib, tmp_path):
    obj = str(tmp_path / f"grid{n}.obj")
    write_grid_obj(obj, "vtn", n=n)
    d = host_build(host_lib, obj, cap_tris=1 << 17)
    assert_same_build(build_probe_lib.build(d["tris"]), (d["box_bounds"], d["box_offsets"], d["box_indices"]), n)


@pytest.mark.parametrize("name", sorted(AWKWARD_CASES))
def test_probe_follows_the_rule_on_awkward_inputs(name, build_probe_lib):
    tris = AWKWARD_CASES[name]()
    got = build_probe_lib.build(tris)
    assert_same_build(got, flat_bvh_rule(tris), name)
    bb, offs, idx = got
    assert offs[-1] == tris.shape[0] and np.array_equal(np.sort(idx), np.arange(tris.shape[0]))
    if name == "equal_keys":
        # every split keeps all triangles on the lo side: one box, never divided, whose list is the input order
        assert bb.shape[0] == 1 and np.array_equal(idx, np.arange(tris.shape[0]))
    if name.startswith("n") and name[1:].isdigit() and tris.shape[0] <= 5:
        assert bb.shape[0] == 1 and np.array_equal(idx, np.arange(tris.shape[0]))   # a small root passes through


def test_split_dir_advances_across_boxes_and_layers(build_probe_lib):
    """12 triangles whose split on y would leave one side empty: the rule then splits the next box on x, not y"""
    n = 12
    tris = random_tris(n, 40)
    tris[:, 1] = 7.0                                       # all keys equal on y: layer 1's split is one-sided
    tris[:, 0] = np.arange(n, dtype=np.float32)           # distinct on x
    got = build_probe_lib.build(tris)
    assert_same_build(got, flat_bvh_rule(tris), "split_dir")
    bb, offs, idx = got
    # layer 1 (y): one-sided; layer 2 (x): 0..5 | 6..11 -> two boxes of 6, split again on z and y
    assert bb.shape[0] >= 2
    assert set(idx[offs[0]:offs[1]]) <= set(range(6))


def test_probe_reaches_1024_leaves(build_probe_lib):
    tris = leaves_1024()
    got = build_probe_lib.build(tris)
    assert got[0].shape[0] == 1024
    assert_same_build(got, flat_bvh_rule(tris), "1024 leaves")
