"""Soundness of sky_fast (csrc/ore_primary.cuh) restated in numpy float32: whenever the shortcut accepts a pixel, its
texel index equals the one the reference's exact float sequence (skybox::getFColor, kernel.cu:1146-1166, after
sphere::intersect :292-354 and normalise :101-108) produces.  Also pins the error of the polynomial arctangent the
error budget in the kernel's comment relies on.  CPU only; the GPU suite checks the real kernels against the oracle with
an index-encoding sky texture (tests/test_round2_gpu.py)."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = open(os.path.join(ROOT, "ray-tracer-engine_b200", "csrc", "ore_primary.cuh")).read()
f32 = np.float32


def _coefficients():
    body = SRC[SRC.index("float atan2_approx"):]
    body = body[:body.index("float r = p * a;")]
    c = [float(m) for m in re.findall(r"(-?\d\.\d+)f", body)]
    assert len(c) == 7, c
    return [f32(v) for v in c]   # highest degree first


def fma(a, b, c):
    return (a.astype(np.float64) * np.asarray(b, dtype=np.float64) + np.asarray(c, dtype=np.float64)).astype(f32)


def atan2_approx(y, x):
    c = _coefficients()
    ax, ay = np.abs(x), np.abs(y)
    mx, mn = np.maximum(ax, ay), np.minimum(ax, ay)
    a = (mn * (f32(1) / mx)).astype(f32)
    q = (a * a).astype(f32)
    p = np.full_like(a, c[0])
    for ci in c[1:]:
        p = fma(p, q, ci)
    r = (p * a).astype(f32)
    r = np.where(ay > ax, f32(1.57079632679) - r, r).astype(f32)
    r = np.where(x < 0, f32(3.14159265359) - r, r).astype(f32)
    return np.where(y < 0, -r, r).astype(f32)


def test_polynomial_arctangent_error_is_inside_the_budget():
    rng = np.random.default_rng(1)
    ang = rng.uniform(-np.pi, np.pi, 2_000_000)
    rad = 10.0 ** rng.uniform(-3, 3, ang.size)
    x, y = (rad * np.cos(ang)).astype(f32), (rad * np.sin(ang)).astype(f32)
    err = np.abs(atan2_approx(y, x).astype(np.float64) - np.arctan2(y.astype(np.float64), x.astype(np.float64)))
    assert err.max() < 1e-6, err.max()     # the kernel's comment budgets 4e-6 for this + both libms


# ---- exact float32 restatement of the reference's sky lookup --------------------------------------------------
def normalise(v):
    l = np.sqrt((v[0] * v[0] + v[1] * v[1] + v[2] * v[2]).astype(f32)).astype(f32)
    return [(c / l).astype(f32) for c in v]


def primary_dir(dx, dy, fz, cp, sp, cy, sy):
    n = normalise([dx, dy, np.full_like(dx, fz)])
    y = (n[1] * cp - n[2] * sp).astype(f32)
    z = (n[1] * sp + n[2] * cp).astype(f32)
    x = (n[0] * cy + z * sy).astype(f32)
    z = (-n[0] * sy + z * cy).astype(f32)
    return [x, y, z]


def exact_index(dx, dy, fz, cam, O, radius_member, w, h):
    D = primary_dir(dx, dy, fz, *cam)
    A = (D[0] * D[0] + D[1] * D[1] + D[2] * D[2]).astype(f32)
    B = (f32(2) * (D[0] * O[0] + D[1] * O[1] + D[2] * O[2]).astype(f32)).astype(f32)
    C = ((O[0] * O[0] + O[1] * O[1] + O[2] * O[2]).astype(f32) - f32(radius_member) * f32(radius_member)).astype(f32)
    sq = np.sqrt((B * B - (f32(4) * A * C).astype(f32)).astype(f32)).astype(f32)
    t = ((-B + sq) / (f32(2) * A)).astype(f32)
    t2 = ((-B - sq) / (f32(2) * A)).astype(f32)
    t = np.where(t >= f32(1.00000005e-4), np.minimum(t, t2), t).astype(f32)
    hp = [(O[i] + (D[i] * t).astype(f32)).astype(f32) for i in range(3)]
    n = normalise(hp)
    sx = ((f32(1) + np.arctan2(n[2], n[0]).astype(f32) / f32(3.1415)).astype(f32) * f32(0.5) * f32(w)).astype(f32)
    sy = (np.arccos(n[1]).astype(f32) / f32(3.1415) * f32(h)).astype(f32)
    return sy.astype(np.int64) * w + sx.astype(np.int64)


def sky_fast(dx, dy, fz, cam, O, radius_member, w, h):
    """numpy float32 mirror of the kernel function; returns (accepted, index)"""
    cp, sp, cy, sy = cam
    R2 = f32(radius_member) * f32(radius_member)
    OO = f32(O[0] * O[0] + O[1] * O[1] + O[2] * O[2])
    c = f32(OO - R2)
    ku = f32(f32(0.5) * f32(w) / f32(3.1415)); hw = f32(0.5) * f32(w); kv = f32(f32(h) / f32(3.1415))
    eu1 = f32(8e-6) * ku; eu0 = f32(4e-6 * ku + 1e-6 * w + 1e-4)
    ev1 = f32(8e-6) * kv; ev0 = f32(4e-6 * kv + 1e-6 * h + 1e-4)
    if not (R2 >= 1 and R2 < 1e30 and OO <= 0.25 * R2):
        return np.zeros(dx.shape, dtype=bool), np.zeros(dx.shape, dtype=np.int64)
    inv = (f32(1) / np.sqrt(fma(dx, dx, fma(dy, dy, f32(fz) * f32(fz))))).astype(f32)
    nx0, ny0, nz0 = (dx * inv).astype(f32), (dy * inv).astype(f32), (f32(fz) * inv).astype(f32)
    Dy = fma(ny0, cp, -(nz0 * sp).astype(f32))
    z1 = fma(ny0, sp, (nz0 * cp).astype(f32))
    Dx = fma(nx0, cy, (z1 * sy).astype(f32))
    Dz = fma(-nx0, sy, (z1 * cy).astype(f32))
    b = fma(Dx, O[0], fma(Dy, O[1], (Dz * O[2]).astype(f32)))
    t = -(b + np.sqrt(fma(b, b, -c)).astype(f32)).astype(f32)
    hx, hy, hz = fma(Dx, t, O[0]), fma(Dy, t, O[1]), fma(Dz, t, O[2])
    hinv = (f32(1) / np.sqrt(fma(hx, hx, fma(hy, hy, (hz * hz).astype(f32))))).astype(f32)
    nx, ny, nz = (hx * hinv).astype(f32), (hy * hinv).astype(f32), (hz * hinv).astype(f32)
    rho2 = fma(nx, nx, (nz * nz).astype(f32))
    ok = rho2 > f32(4e-4)
    rho2s = np.where(ok, rho2, f32(1))
    irho = (f32(1) / np.sqrt(rho2s)).astype(f32)
    rho = (rho2s * irho).astype(f32)
    u = fma(atan2_approx(nz, nx), ku, hw)
    v = (atan2_approx(rho, ny) * kv).astype(f32)
    fu, fv = np.floor(u), np.floor(v)
    Eu, Ev = fma(irho, eu1, eu0), fma(irho, ev1, ev0)
    du, dv = (u - fu).astype(f32), (v - fv).astype(f32)
    ok &= (du >= Eu) & (du <= f32(1) - Eu) & (dv >= Ev) & (dv <= f32(1) - Ev) & (fu >= 0) & (fv >= 0)
    return ok, fv.astype(np.int64) * w + fu.astype(np.int64)


def _camera(rng, extent):
    yaw, pitch = rng.uniform(0, 360), rng.uniform(-89.9, 89.9)
    yr, pr = f32(yaw * (3.1415 / 180)), f32(pitch * (3.1415 / 180))
    cam = (f32(np.cos(pr)), f32(np.sin(pr)), f32(np.cos(yr)), f32(np.sin(yr)))
    O = [f32(v) for v in rng.uniform(-extent, extent, 3)]
    return cam, O


def test_sky_fast_never_accepts_a_wrong_texel():
    rng = np.random.default_rng(5)
    aspect = f32(np.tan(90 * 0.5 * 3.1415 / 180))
    fz = f32(0) - (f32(-1) / aspect)
    total = accepted = 0
    for it in range(60):
        w, h = [(1024, 512), (2048, 1024), (300, 200), (4096, 2048), (64, 32)][it % 5]
        size = [10000.0, 10000.0, 30.0, 1e3][it % 4]                 # sphere ctor stores size^2, intersect squares again
        extent = [30.0, 2000.0, 5.0, 100.0][it % 4]
        cam, O = _camera(rng, extent)
        n = 40000
        dx = (aspect * rng.uniform(-1, 1, n)).astype(f32)
        dy = (aspect * rng.uniform(-1, 1, n) * 0.5625).astype(f32)
        ok, idx = sky_fast(dx, dy, fz, cam, O, size * size, w, h)
        ref = exact_index(dx, dy, fz, cam, O, size * size, w, h)
        bad = ok & (idx != ref)
        assert not bad.any(), (it, int(bad.sum()), w, h, size, O)
        total += n
        accepted += int(ok.sum())
    assert accepted > 0.5 * total, (accepted, total)     # and it is useful: most pixels are decided by the shortcut


REF_ASPECT = float(f32(np.tan(90 * 0.5 * 3.1415 / 180)))
ASPECTS = [1e-3, 0.02, 0.35, REF_ASPECT, 1.7, 4.0, 25.0, 1e3, -REF_ASPECT]


@pytest.mark.parametrize("aspect", ASPECTS, ids=[f"{a:g}" for a in ASPECTS])
def test_sky_fast_never_accepts_a_wrong_texel_at_other_fields_of_view(aspect):
    """the image-plane coordinates the reference really produces at this field of view (kernel.cu:1624-1625):
    dx in [-1, 2 aspect - 1], dy in [-1, 2 aspect H/W - 1], fz = 1/aspect (negative: the view looks backwards)"""
    rng = np.random.default_rng(int(1000 + 7 * ASPECTS.index(aspect)))
    a = f32(aspect)
    fz = f32(0) - (f32(-1) / a)
    hw = 0.5625                                                    # a 16:9 frame
    total = accepted = 0
    for it in range(24):
        w, h = [(1024, 512), (300, 200), (4096, 2048)][it % 3]
        size = [10000.0, 10000.0, 30.0, 1e3][it % 4]
        extent = [30.0, 2000.0, 5.0, 100.0][it % 4]
        cam, O = _camera(rng, extent)
        n = 20000
        dx = (np.float64(a) * rng.uniform(0, 2, n) - 1).astype(f32)
        dy = (np.float64(a) * rng.uniform(0, 2, n) * hw - 1).astype(f32)
        ok, idx = sky_fast(dx, dy, fz, cam, O, size * size, w, h)
        ref = exact_index(dx, dy, fz, cam, O, size * size, w, h)
        bad = ok & (idx != ref)
        assert not bad.any(), (aspect, it, int(bad.sum()), w, h, size, O)
        total += n
        accepted += int(ok.sum())
    assert accepted > 0.5 * total, (accepted, total)
