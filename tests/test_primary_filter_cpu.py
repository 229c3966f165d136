"""Monte-Carlo soundness of the primary-ray filters restated in numpy from csrc (DESIGN.md 2.2, 2.4): the per-pixel
one-FFMA filter on the per-frame sphere records of prep_frame_kernel, and the 32x8 tile cone.

Truth is float64 geometry on the reference's own ray directions (kernel.cu:1624-1631, camera::rotateDir :252-255):
positive discriminant and far root >= 0.  A real hit must pass the pixel filter, and a tile containing one must pass
the tile cone.
"""
import math

import numpy as np
import pytest

f32 = np.float32
KP = 7.62939453125e-06          # ORE_KAPPA_PRIMARY = 2^-17
P = 8                           # tile rows


def frame_tables(W, H, aspect):
    x = np.arange(W)
    y = np.arange(H)
    dx = (np.float64(aspect) * (2 * (x + 0.5) / np.float64(f32(W))) - 1).astype(f32)
    hw = f32(f32(H) / f32(W))
    dy = (np.float64(aspect) * (2 * (y + 0.5) / np.float64(f32(H))) * np.float64(hw) - 1).astype(f32)
    return dx, dy


def directions(dx, dy, fz, cp, sp, cy, sy):
    vx, vy = np.meshgrid(dx, dy)                                  # [H,W]
    vz = np.full_like(vx, fz)
    ln = np.sqrt((vx * vx + vy * vy + vz * vz).astype(f32)).astype(f32)
    nx, ny, nz = (vx / ln).astype(f32), (vy / ln).astype(f32), (vz / ln).astype(f32)
    y = (ny * cp - nz * sp).astype(f32)
    z = (ny * sp + nz * cp).astype(f32)
    x = (nx * cy + z * sy).astype(f32)
    z2 = (-nx * sy + z * cy).astype(f32)
    return np.stack([x, y, z2], axis=-1)


REF_ASPECT = float(f32(math.tan(90 * 0.5 * 3.1415 / 180)))
ASPECTS = [1e-3, 0.02, 0.35, REF_ASPECT, 1.7, 4.0, 25.0, 1e3, -REF_ASPECT]
BLOCKS = [(2, 3), (2, 7), (2, 24), (3, 7), (3, 24), (8, 24), (8, 8)]


def image_row(k, y_block, y_step):
    """image row (from y0 = 0) of rendered row k: blocks of y_block rows, y_step apart (ore_kernels.cuh image_row_rel)"""
    return (k // y_block) * y_step + k % y_block


def tile_half_angle_ratio(aspect, W, y_block, y_step, fz):
    """xr = sin(a) bound of tile_cone (csrc/ore_capi.cu): tallest image-row span of TILE_ROWS consecutive rendered rows"""
    delta = 2.0 * aspect / W
    span = max(image_row(k0 + P - 1, y_block, y_step) - image_row(k0, y_block, y_step) for k0 in range(0, y_block * P, P))
    hx, hy = 16.0 * delta, (0.5 * span + 0.5) * delta
    return math.sqrt(hx * hx + hy * hy) / abs(float(fz)), delta


def check_filters(rng, aspect=REF_ASPECT, pitch_span=80.0, y_block=1, y_step=1, frame_scaled=False):
    """the filters of one frame geometry on 6 random cameras and 60 spheres each; returns (spheres hit, tile-sphere
    pairs, pairs culled, xr).  frame_scaled: sphere sizes follow the frame's angular size instead of a fixed range"""
    W, n_rows = 256, 128
    aspect = f32(aspect)
    if y_block >= y_step:                                         # frame_params: a contiguous band
        y_block, y_step = 1, 1
    rows = np.array([image_row(k, y_block, y_step) for k in range(n_rows)])
    H = int(rows[-1]) + 1
    ez = f32(-1.0) / aspect
    fz = f32(0.0) - ez
    dx, dy_all = frame_tables(W, H, aspect)
    dy = dy_all[rows]                                             # dy_tab: one entry per rendered row
    xr, delta = tile_half_angle_ratio(float(aspect), W, y_block, y_step, fz)
    if xr < 0.9:
        a = math.asin(xr) * 1.001 + 1e-6
        tile_ca, tile_sa = f32(math.cos(a) * (1 - 1e-6) - 1e-6), f32(math.sin(a) * (1 + 1e-6) + 1e-6)
    else:                                                         # tiles too wide for a cone: every sphere a candidate
        tile_ca, tile_sa = f32(-1e20), f32(0.0)
    frame_angle = math.atan2(abs(2.0 * float(aspect)), abs(float(fz)))
    n_hit = n_tiles_culled = n_tiles = 0
    for _ in range(6):
        yaw, pitch = rng.uniform(0, 360), rng.uniform(-pitch_span, pitch_span)
        cp, sp = f32(math.cos(math.radians(pitch))), f32(math.sin(math.radians(pitch)))
        cy, sy = f32(math.cos(math.radians(yaw))), f32(math.sin(math.radians(yaw)))
        O = rng.uniform(-10, 10, 3).astype(f32)
        D = directions(dx, dy, fz, cp, sp, cy, sy).astype(np.float64)            # [rows,W,3]
        n = 60
        # spheres: most of them in front of the camera along some pixel's ray
        py, px = rng.integers(0, n_rows, n), rng.integers(0, W, n)
        t = 10.0 ** rng.uniform(-0.5, 2.5, n)
        if frame_scaled:
            member = (t * frame_angle * 10.0 ** rng.uniform(-2.0, -0.3, n)).astype(f32)
        else:
            member = (10.0 ** rng.uniform(-1.5, 0.7, n)).astype(f32)             # effective radius
        c = O.astype(np.float64) + D[py, px] * t[:, None] + rng.normal(0, 1, (n, 3)) * member[:, None] * 1.5
        c[n - 10:] = O + rng.normal(0, 1, (10, 3)) * 30                           # anywhere, incl. behind
        c = c.astype(f32)
        # per-frame records (prep_frame_kernel, double precision)
        L = (O[None, :] - c).astype(f32).astype(np.float64)                       # reference forms L in float
        LL = (L * L).sum(axis=1)
        r4 = (member * member).astype(f32).astype(np.float64)
        Cm = LL * (1 - KP) - r4 * (1 + KP)
        always = ~((Cm > 1e-9 * LL) & (Cm > 1e-30))
        sv = np.sqrt(np.where(always, 1.0, Cm))
        cpd, spd, cyd, syd = float(cp), float(sp), float(cy), float(sy)
        Mx = cyd * L[:, 0] - syd * L[:, 2]
        My = spd * syd * L[:, 0] + cpd * L[:, 1] + spd * cyd * L[:, 2]
        Mz = cpd * syd * L[:, 0] - spd * L[:, 1] + cpd * cyd * L[:, 2]
        ra, rb, rc = (Mx / sv).astype(f32), (My / sv).astype(f32), (float(fz) * Mz / sv).astype(f32)
        Rpp = np.sqrt(np.maximum(LL - Cm, 0))
        Wd = (float(tile_ca) * sv - float(tile_sa) * Rpp - 4e-6 * np.sqrt(LL) - 1e-30).astype(f32)
        # truth per pixel and sphere
        b = np.einsum("hwk,nk->hwn", D, L)
        disc = b * b - (LL - r4)[None, None, :]
        hit = (disc >= 0) & ((-b + np.sqrt(np.maximum(disc, 0))) >= 0)            # [rows,W,n]
        # per-pixel filter: fma(dy, b', fma(dx, a', c')) <= -|v| (1 - 2^-20)
        nv = np.sqrt((dx[None, :] ** 2 + dy[:, None] ** 2 + fz * fz).astype(f32)).astype(f32)
        lhs = (dy[:, None, None] * rb[None, None, :] + (dx[None, :, None] * ra[None, None, :] + rc[None, None, :])).astype(f32)
        passed = (lhs <= (-nv * f32(0.99999905))[:, :, None]) | always[None, None, :]
        assert not np.any(hit & ~passed), "pixel filter rejected a hit"
        # tile cone: axis through the nominal tile centre (primary_tile_kernel)
        for ty in range(n_rows // P):
            cyt = f32(0.5) * (dy[ty * P] + dy[ty * P + P - 1])
            for tx in range(W // 32):
                cxt = dx[tx * 32] + f32(15.5) * f32(delta)
                inv = f32(1) / np.sqrt(f32(cxt * cxt + cyt * cyt + fz * fz))
                axv = np.array([cxt * inv, cyt * inv, fz * inv], dtype=f32)
                hA = (axv[0] * Mx.astype(f32) + (axv[1] * My.astype(f32) + (axv[2] * Mz.astype(f32) + Wd))).astype(f32)
                cone_ok = (hA <= 0) | always
                th = hit[ty * P:(ty + 1) * P, tx * 32:(tx + 1) * 32].any(axis=(0, 1))
                assert not np.any(th & ~cone_ok), "tile cone rejected a tile with a hit"
                n_tiles += n
                n_tiles_culled += int((~cone_ok).sum())
        n_hit += int(hit.any(axis=(0, 1)).sum())
    return n_hit, n_tiles, n_tiles_culled, xr


@pytest.mark.parametrize("seed", range(5))
def test_primary_filters_never_reject_a_hit(seed):
    n_hit, n_tiles, n_tiles_culled, _ = check_filters(np.random.default_rng(900 + seed))
    assert n_hit > 100
    assert n_tiles_culled > 0.5 * n_tiles, "the tile cone must cull most (tile, sphere) pairs"


# tile_cone lowers cos(a) by about 2e-6 (its absolute margins), which widens every cone to a half-angle of at least
# sqrt(4e-6) = 2e-3 rad.  Telephoto tiles (aspect 0.02: 1e-4 rad; 1e-3: 2.5e-7 rad) are far narrower, so there the cone
# keeps every sphere near the frame and culling is only asked of tiles wider than 10x that floor.
CONE_FLOOR = 2e-3


def _assert_culls_where_it_can(n_tiles, n_tiles_culled, xr, aspect, fz_abs):
    tile_angle = 32 * 2.0 * abs(aspect) / 256 / fz_abs
    if xr < 0.9 and tile_angle > 10 * CONE_FLOOR:
        assert n_tiles_culled > 0.5 * n_tiles, ("the tile cone must cull most (tile, sphere) pairs", xr, n_tiles_culled, n_tiles)


@pytest.mark.parametrize("aspect", ASPECTS, ids=[f"{a:g}" for a in ASPECTS])
def test_primary_filters_never_reject_a_hit_at_other_fields_of_view(aspect):
    """aspect 1e-3 .. 1e3 and a negative one (fz < 0: the view looks backwards); sphere sizes follow the field"""
    n_hit, n_tiles, n_tiles_culled, xr = check_filters(np.random.default_rng(950 + ASPECTS.index(aspect)), aspect=aspect,
                                                       frame_scaled=True)
    assert n_hit > 100
    _assert_culls_where_it_can(n_tiles, n_tiles_culled, xr, aspect, abs(1.0 / aspect))


@pytest.mark.parametrize("seed", range(3))
def test_primary_filters_never_reject_a_hit_at_unclamped_pitch(seed):
    """pitch drawn from +-720 degrees: the reference's checkKey never clamps it (kernel.cu:1716-1759)"""
    n_hit, n_tiles, n_tiles_culled, xr = check_filters(np.random.default_rng(970 + seed), pitch_span=720.0)
    assert n_hit > 100
    assert n_tiles_culled > 0.5 * n_tiles, "the tile cone must cull most (tile, sphere) pairs"


@pytest.mark.parametrize("y_block,y_step", BLOCKS, ids=[f"b{b}s{s}" for b, s in BLOCKS])
def test_primary_filters_never_reject_a_hit_in_block_interleaved_bands(y_block, y_step):
    """a tile's 8 rendered rows span up to several blocks of image rows; the cone's half-angle follows tile_cone"""
    n_hit, n_tiles, n_tiles_culled, xr = check_filters(np.random.default_rng(990 + y_block * 31 + y_step), y_block=y_block,
                                                       y_step=y_step)
    assert n_hit > 100
    _assert_culls_where_it_can(n_tiles, n_tiles_culled, xr, REF_ASPECT, 1.0 / REF_ASPECT)
