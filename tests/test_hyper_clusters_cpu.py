"""Hyper-clusters of large scenes (csrc/ore_clusters.h, build_hypers), built by the host builder with g++ and checked on
the CPU.  The large-scene kernels cull 8192 spheres at a time by one hyper ball, so the property everything rests on is
containment: every sphere ball (centre, R') lies inside its hyper ball - or that ball is 'always open' (+inf)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "ray-tracer-engine_b200", "csrc")
HYPER_SPHERES = 8192
# members the float tests cannot bound (the awkward members of test_clusters_cpu.py, and larger coordinates)
WEIRD = [(1e17, 0, 0, 1.0), (0, -3e19, 0, 1e10), (np.inf, 0, 0, 1.0), (-np.inf, np.inf, 0, 2.0), (np.nan, 1, 1, 0.5),
         (1, 1, 1, np.nan), (5e15, 5e15, 5e15, 1e3), (3, 3, 3, 2e15), (1e30, -1e30, 1e30, 1.0), (0, 0, 1e25, 1e20)]


def tree_lengths(n):
    n_sup = (n + 255) // 256
    n_hyp = (n_sup + 31) // 32
    return (n + 31) // 32 * 32, (n_sup + 3) // 4 * 4, (n_hyp + 3) // 4 * 4


def load_probe(out_dir):
    """host reference of the sorted shadow records, super balls and hyper balls (tests/hyper_tree_probe.cpp)"""
    out = os.path.join(str(out_dir), "libhyper_tree_probe.so")
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC,
                           os.path.join(ROOT, "tests", "hyper_tree_probe.cpp"), "-o", out], env=env)
    lib = C.CDLL(out)
    vp, i = C.c_void_p, C.c_int
    lib.ore_probe_hyper_tree.argtypes = [vp, i, vp, vp, vp, i, i, i]
    lib.ore_probe_hyper_tree.restype = i

    def build(spheres):
        sp = np.ascontiguousarray(spheres, dtype=np.float32).reshape(-1, 4)
        n_sort, n_sup_pad, n_hyp_pad = tree_lengths(len(sp))
        ss = np.zeros((n_sort, 4), np.float32)
        su = np.zeros((n_sup_pad, 4), np.float32)
        hy = np.zeros((n_hyp_pad, 4), np.float32)
        rc = lib.ore_probe_hyper_tree(sp.ctypes.data, len(sp), ss.ctypes.data, su.ctypes.data, hy.ctypes.data, n_sort,
                                      n_sup_pad, n_hyp_pad)
        assert rc == 0
        return ss, su, hy

    return build


@pytest.fixture(scope="module")
def hyper_probe(tmp_path_factory):
    return load_probe(tmp_path_factory.mktemp("hyper"))


def spheres(n, seed, extent=None, weird=False):
    """n random spheres at about the density of scene.scaled_scene; weird: WEIRD members spread over the set"""
    rng = np.random.default_rng(seed)
    extent = extent or 10.0 * (n / 64.0) ** (1.0 / 3.0)
    pos = rng.uniform(0, extent, size=(n, 3)).astype(np.float32)
    member = (rng.integers(0, 100, size=n) / 100.0).astype(np.float32) ** 2
    sp = np.concatenate([pos, member[:, None]], axis=1).astype(np.float32)
    if weird:
        for k, w in enumerate(WEIRD):
            sp[(k * 7919 + seed) % n] = np.array(w, dtype=np.float32)
    return np.ascontiguousarray(sp)


def assert_contained(ss, balls, n, per):
    """every tame member ball of ss[:n] lies inside ball p // per; a group with an untame member has radius +inf"""
    mem = ss[:n].astype(np.float64)
    idx = np.arange(n) // per
    tame_rec = np.all(np.isfinite(mem) & (np.abs(mem) < 1e15), axis=1)
    group_tame = np.ones(len(balls), dtype=bool)
    np.logical_and.at(group_tame, idx, tame_rec)
    r = balls[idx, 3].astype(np.float64)
    assert np.all(r[~group_tame[idx]] == np.inf), "a group with an untame member must be always open"
    ok = group_tame[idx]
    c = balls[idx, :3].astype(np.float64)
    d = np.sqrt(((mem[:, :3] - c) ** 2).sum(axis=1)) + np.abs(mem[:, 3])
    assert np.all(np.isfinite(r[ok])), "tame groups stay bounded"
    bad = ok & ~(d <= r)
    assert not np.any(bad), (int(np.count_nonzero(bad)), np.flatnonzero(bad)[:5])


@pytest.mark.parametrize("weird", [False, True], ids=["random", "untame"])
@pytest.mark.parametrize("n", [8191, 8192, 8193, 99073, 300001])
def test_every_sphere_ball_lies_inside_its_hyper_ball(hyper_probe, n, weird):
    ss, su, hy = hyper_probe(spheres(n, n, weird=weird))
    n_sup = (n + 255) // 256
    n_hyp = (n_sup + 31) // 32
    assert_contained(ss, hy, n, HYPER_SPHERES)
    # the level below too, and the hyper over its super balls as member balls
    assert_contained(ss, su, n, 256)
    for h in range(n_hyp):
        sup = su[32 * h:min(32 * h + 32, n_sup)].astype(np.float64)
        if np.isinf(hy[h, 3]):
            continue
        d = np.sqrt(((sup[:, :3] - hy[h, :3].astype(np.float64)) ** 2).sum(axis=1)) + sup[:, 3]
        assert np.all(d <= hy[h, 3]), h
    assert np.all(hy[n_hyp:, 3] == -1) and np.all(su[n_sup:, 3] == -1)   # padding: never touched
    if weird:
        assert np.count_nonzero(np.isinf(hy[:n_hyp, 3])) >= 1
    else:
        assert np.all(np.isfinite(hy[:n_hyp, 3]))


def test_hyper_balls_are_compact(hyper_probe):
    """Morton order: at 300 001 spheres (edge about 167) the mean hyper radius stays far below the scene's extent"""
    n = 300001
    extent = 10.0 * (n / 64.0) ** (1.0 / 3.0)
    _, _, hy = hyper_probe(spheres(n, 3))
    n_hyp = ((n + 255) // 256 + 31) // 32
    assert np.mean(hy[:n_hyp, 3]) < 0.45 * extent
