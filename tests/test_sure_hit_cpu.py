"""Soundness of the shadow sweep's "sure hit" shortcut (csrc/ore_kernels.cuh, DESIGN.md 2.5) on the CPU.

The kernel marks a shadow ray blocked WITHOUT running the reference's exact sequence when
    b = D.L < 0   and   b^2 > max(1e-6 |L|^2 + 1e-6, |L|^2 - r^2 + 2e-5 |L|^2),   L = start - centre,
for directions with | |D|^2 - 1 | < 5e-6 (cone_of10 admits nothing else; the reference's normalise() gives 5e-7).
Every such ray must make sphere::intersect (kernel.cu:293-354) return true.  Checked here against a float32
numpy restatement of that function (itself checked against the C oracle on a subsample), on random rays and on
adversarial families: grazing rays, origins on / just off the surface, tiny and huge spheres, far origins,
directions whose squared length is off by up to 5e-6 (the kernel's admission limit).
"""
import os

import numpy as np
import pytest

f32 = np.float32


def ref_hit(O, D, Cn, rad):
    """boolean of sphere::intersect, float32 operation by operation (no contraction)"""
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        l = [(O[:, k] - Cn[:, k]).astype(f32) for k in range(3)]
        A = ((D[:, 0] * D[:, 0]).astype(f32) + (D[:, 1] * D[:, 1]).astype(f32)).astype(f32)
        A = (A + (D[:, 2] * D[:, 2]).astype(f32)).astype(f32)
        Bq = ((D[:, 0] * l[0]).astype(f32) + (D[:, 1] * l[1]).astype(f32)).astype(f32)
        Bq = (f32(2) * (Bq + (D[:, 2] * l[2]).astype(f32)).astype(f32)).astype(f32)
        Cq = ((l[0] * l[0]).astype(f32) + (l[1] * l[1]).astype(f32)).astype(f32)
        Cq = (Cq + (l[2] * l[2]).astype(f32)).astype(f32)
        Cq = (Cq - (rad * rad).astype(f32)).astype(f32)
        disc = ((Bq * Bq).astype(f32) - ((f32(4) * A).astype(f32) * Cq).astype(f32)).astype(f32)
        sq = np.sqrt(disc).astype(f32)
        t = ((-Bq + sq).astype(f32) / (f32(2) * A).astype(f32)).astype(f32)
        return (t == 0) | (t.astype(np.float64) >= 0.0001)


def sure_hit(O, D, Cn, rad):
    """the kernel's criterion, float32 (the kernel uses fused multiply-adds: 1e-7 relative, the margin is 2e-5)"""
    l = (O - Cn).astype(f32)
    LL = (l * l).sum(axis=1, dtype=f32)
    b = (D * l).sum(axis=1, dtype=f32)
    thr = np.maximum(LL * f32(1e-6) + f32(1e-6), LL * f32(2e-5) + (LL - rad * rad).astype(f32)).astype(f32)
    return (b < 0) & ((b * b).astype(f32) > thr)


def unit(v):
    v = v.astype(np.float64)
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(f32)


def families(rng, n):
    """(name, O, D, centre, radius member) float32 arrays"""
    out = []
    # 1. generic
    O = rng.uniform(-50, 50, (n, 3)).astype(f32)
    Cn = rng.uniform(-50, 50, (n, 3)).astype(f32)
    rad = rng.uniform(0.05, 8, n).astype(f32)
    aim = Cn + rng.normal(0, 1, (n, 3)).astype(f32) * rad[:, None] * f32(0.8)
    out.append(("aimed", O, unit(aim - O), Cn, rad))
    # 2. grazing: aim at a point at distance r*(1 +- eps) from the centre, perpendicular to the view line
    eps = (10.0 ** rng.uniform(-7, -1, n)) * rng.choice([-1, 1], n)
    view = unit(Cn - O).astype(np.float64)
    perp = np.cross(view, rng.normal(0, 1, (n, 3)))
    perp /= np.linalg.norm(perp, axis=1, keepdims=True)
    tgt = Cn.astype(np.float64) + perp * (rad.astype(np.float64) * (1 + eps))[:, None]
    out.append(("grazing", O, unit((tgt - O).astype(f32)), Cn, rad))
    # 3. origin on / just off the surface (the shadow ray's own sphere and touching neighbours)
    nrm = unit(rng.normal(0, 1, (n, 3)))
    off = (10.0 ** rng.uniform(-7, -2, n)) * rng.choice([-1, 1], n)
    O3 = (Cn.astype(np.float64) + nrm * (rad * (1 + off))[:, None]).astype(f32)
    out.append(("surface", O3, unit(rng.normal(0, 1, (n, 3))), Cn, rad))
    # 4. tiny spheres close by, huge spheres, far origins
    rad4 = (10.0 ** rng.uniform(-4, 3.5, n)).astype(f32)
    O4 = (Cn.astype(np.float64) + unit(rng.normal(0, 1, (n, 3))) * (rad4 * 10.0 ** rng.uniform(0, 3, n))[:, None]).astype(f32)
    aim4 = Cn + rng.normal(0, 1, (n, 3)).astype(f32) * rad4[:, None]
    out.append(("scales", O4, unit(aim4 - O4), Cn, rad4))
    # 5. squared direction length off by up to 5e-6
    s = (1 + rng.uniform(-2.5e-6, 2.5e-6, n)).astype(f32)
    out.append(("non-unit", O, (unit(aim - O) * s[:, None]).astype(f32), Cn, rad))
    out.append(("grazing non-unit", O, (unit((tgt - O).astype(f32)) * s[:, None]).astype(f32), Cn, rad))
    return out


def test_numpy_restatement_matches_the_c_oracle(oracle_port):
    rng = np.random.default_rng(5)
    for name, O, D, Cn, rad in families(rng, 400):
        want = np.array([oracle_port.sphere_intersect(O[i], D[i], Cn[i], rad[i])[0] for i in range(len(rad))])
        assert np.array_equal(ref_hit(O, D, Cn, rad), want), name


def test_numpy_restatement_matches_the_references_own_code(oracle_ref):
    """same check against sphere::intersect of the reference itself (kernel.cu compiled for the host, oracle/_ref)"""
    rng = np.random.default_rng(6)
    for name, O, D, Cn, rad in families(rng, 400):
        want = np.array([oracle_ref.sphere_intersect(O[i], D[i], Cn[i], rad[i])[0] for i in range(len(rad))])
        assert np.array_equal(ref_hit(O, D, Cn, rad), want), name


def test_numpy_restatement_and_sure_hits_agree_with_the_stored_reference_answers():
    """ref_hit and sure_hit against the answers the reference's own sphere::intersect gave for the 4096 rays of
    tests/golden/intersect_kat.npz (stored, so this runs without the reference's source).  Those rays are generic, not
    the adversarial families: on the families sure_hit is checked against ref_hit, and ref_hit against the C oracle."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "intersect_kat.npz"))
    O, D, Cn, rad, hit = g["org"], g["dir"], g["centre"], g["radius"], g["hit"].astype(bool)
    assert np.array_equal(ref_hit(O, D, Cn, rad), hit)
    sure = sure_hit(O, D, Cn, rad)
    assert np.count_nonzero(sure) > 500
    assert not np.any(sure & ~hit)


def test_every_sure_hit_sample_is_a_hit_of_the_references_own_code(oracle_ref):
    rng = np.random.default_rng(7)
    checked = 0
    for name, O, D, Cn, rad in families(rng, 20_000):
        idx = np.flatnonzero(sure_hit(O, D, Cn, rad))[:1500]
        for i in idx:
            assert oracle_ref.sphere_intersect(O[i], D[i], Cn[i], rad[i])[0], (name, int(i))
        checked += len(idx)
    assert checked > 3000


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_every_sure_hit_is_a_hit_of_the_reference_sequence(seed):
    rng = np.random.default_rng(100 + seed)
    for name, O, D, Cn, rad in families(rng, 400_000):
        sure = sure_hit(O, D, Cn, rad)
        hit = ref_hit(O, D, Cn, rad)
        assert not np.any(sure & ~hit), (name, int(np.count_nonzero(sure & ~hit)))
        if name == "aimed":
            # and it is worth having: most real hits are sure hits
            assert np.count_nonzero(sure) > 0.9 * np.count_nonzero(hit & ((D * (O - Cn)).sum(axis=1) < 0)), name
