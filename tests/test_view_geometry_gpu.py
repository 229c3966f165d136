"""View geometry outside the reference's own: fields of view from aspect 1e-3 to 1e3 (and a negative one), unclamped
yaw and pitch, cameras far away / inside a sphere / on a sphere's surface / on face planes, tiny and ragged frames,
block-interleaved bands, strided and misaligned device outputs, and batches whose frames need different per-frame
decisions.  The primary kernel's conservative filters (tile cone, per-pixel threshold, sky texel shortcut) and its sky
store layout all depend on this geometry (DESIGN.md 2.2, 2.4, 2.7).

Each frame is held three ways: ids and t bits equal the oracle's, pixels equal the oracle's where the host libm is
the one ore_libm.cuh reproduces (else 99.9 % within 1 LSB), and the default, fused and exhaustive forms give the same
frame; ORE_FLAG_FAST_LIBM stays within 1 LSB of the default."""
import dataclasses
import math

import numpy as np
import pytest

import cases
from test_parity_gpu import assert_pixels_close, libm_matches  # noqa: F401  (fixture re-export)
from test_round2_gpu import _index_sky

pytestmark = pytest.mark.gpu
SENTINEL = 0x5A5A5A5A
RA = float(cases.scene.REFERENCE_ASPECT)
ASPECTS = [1e-3, 0.02, 0.35, RA, 1.7, 4.0, 25.0, 1e3, -RA]


# ---- scenes and cameras ---------------------------------------------------------------------------------------------
def _aspect(sc, a):
    return dataclasses.replace(sc, aspect=np.float32(a), name=f"{sc.name}@{a:g}")


def _prim_scene(n, seed):
    sc = cases.scene.with_cubes_and_plane(cases.scene.scaled_scene(n, seed), 12, 5)
    sc.mesh = cases.torus_mesh()
    return sc


def _rotate(v, yaw, pitch):
    """camera::rotateDir (kernel.cu:252-255) in float64: camera space -> world"""
    yr, pr = yaw * (3.1415 / 180), pitch * (3.1415 / 180)
    cp, sp, cy, sy = math.cos(pr), math.sin(pr), math.cos(yr), math.sin(yr)
    y = v[1] * cp - v[2] * sp
    z = v[1] * sp + v[2] * cp
    return np.array([v[0] * cy + z * sy, y, -v[0] * sy + z * cy])


def _cam_dir(a, dx, dy):
    v = np.array([dx, dy, 1.0 / a])
    return v / np.linalg.norm(v)


def _half_diagonal(a, W, H):
    """angle between the image centre's ray and a corner's: dx in [-1, 2a - 1], dy in [-1, 2a H/W - 1] (kernel.cu:1624-1625)"""
    c = _cam_dir(a, a - 1, a * H / W - 1)
    return math.acos(min(1.0, float(c @ _cam_dir(a, -1, -1))))


def _eye_to_org(eye, a):
    """camera org that puts the eye (org + (0, 0, -1/aspect), kernel.cu:1629-1631) at `eye`"""
    return tuple(float(np.float32(v)) for v in (eye[0], eye[1], eye[2] + 1.0 / a))


def _aim(a, W, H, target, dist, yaw, pitch):
    """camera whose image centre looks at `target` from `dist` away"""
    d = _rotate(_cam_dir(a, a - 1, a * H / W - 1), yaw, pitch)
    eye = np.asarray(target, dtype=np.float64) - dist * d
    return cases.scene.Camera(org=_eye_to_org(eye, a), yaw=yaw, pitch=pitch)


def _silhouette_camera(sc, a, W, H, yaw):
    """the image centre grazes the top of the scene's topmost sphere (the centre row splits it from the sky above):
    telephoto fields from 10^3 units back (|L| >> the sphere's size), wide ones from close by"""
    s = sc.spheres[np.argmax(sc.spheres[:, 1] + sc.spheres[:, 3])].astype(np.float64)
    R = s[3]                                           # effective radius: intersect squares the radius member
    th = _half_diagonal(a, W, H)
    dist = 1e3 if th < 0.01 else max(R / (0.5 * th), 1.5 * R)
    # pitch the off-axis image centre 3 degrees above the horizon, so that rays past the sphere's top reach the sky
    # (the scene's plane catches every descending ray)
    cc = _cam_dir(a, a - 1, a * H / W - 1)
    pitch = math.degrees(math.atan2(cc[1], cc[2])) - 3.0
    c = _rotate(_cam_dir(a, a - 1, a * H / W - 1), yaw, pitch)
    up = _rotate(_cam_dir(a, a - 1, a * H / W - 1 + 1e-3 * abs(a)), yaw, pitch) - c
    up -= c * (up @ c)
    up /= np.linalg.norm(up)
    return _aim(a, W, H, s[:3] + R * up, dist, yaw, pitch)


# ---- checks ---------------------------------------------------------------------------------------------------------
def _use(renderer, sc):
    renderer.set_scene(sc)   # (every time: other tests change the context's lights and scene behind renderer.scene)


def check_three_ways(renderer, oracle, pkg, sc, cam, W, H, libm_ok, **kw):
    """oracle (ids, t bits, pixels), default == fused == exhaustive (pixels, ids, t), fast libm within 1 LSB; returns
    (pixels, ids, counters) of the default render"""
    F = pkg.capi
    _use(renderer, sc)
    px = renderer.render(cam, W, H, **kw).copy()
    ids, t = renderer.hits(px.shape[0], W)
    c = renderer.counters()
    ref = oracle.render(sc, cam, W, H, **kw)
    assert np.array_equal(ids, ref["ids"]), f"{np.count_nonzero(ids != ref['ids'])} ids differ from the oracle"
    assert np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32)), "t bits differ from the oracle"
    assert_pixels_close(px, ref["pixels"])
    if libm_ok:
        assert np.array_equal(px, ref["pixels"]), f"{np.count_nonzero(px != ref['pixels'])} pixels differ from the oracle"
    for flags in (F.ORE_FLAG_FUSED_SHADOW, F.ORE_FLAG_EXHAUSTIVE):
        q = renderer.render(cam, W, H, flags=flags, **kw)
        qi, qt = renderer.hits(q.shape[0], W)
        assert np.array_equal(qi, ids) and np.array_equal(qt.view(np.uint32), t.view(np.uint32)), flags
        assert np.array_equal(q, px), (flags, int(np.count_nonzero(q != px)))
    assert_pixels_close(renderer.render(cam, W, H, flags=F.ORE_FLAG_FAST_LIBM, **kw), px)
    return px, ids, c


# ---- fields of view -------------------------------------------------------------------------------------------------
FOV_SCENES = {
    "R64_1": lambda: cases.scene.reference_scene(64, 1),
    "S1024_3": lambda: cases.scene.scaled_scene(1024, 3),
    "S64_2_prims": lambda: _prim_scene(64, 2),
}
_fov_cache = {}


@pytest.mark.parametrize("size", [(161, 91), (200, 150)], ids=["161x91", "200x150"])
@pytest.mark.parametrize("scene_kind", list(FOV_SCENES))
@pytest.mark.parametrize("a", ASPECTS, ids=[f"{a:g}" for a in ASPECTS])
def test_fields_of_view_equal_the_oracle(a, scene_kind, size, renderer, oracle_best, pkg, libm_matches):
    W, H = size
    if scene_kind not in _fov_cache:
        _fov_cache[scene_kind] = FOV_SCENES[scene_kind]()
    base = _fov_cache[scene_kind]
    key = (scene_kind, a)
    if key not in _fov_cache:
        _fov_cache[key] = _aspect(base, a)
    sc = _fov_cache[key]
    cam = _silhouette_camera(base, a, W, H, yaw=30.0 + 37.0 * ASPECTS.index(a))
    px, ids, _ = check_three_ways(renderer, oracle_best, pkg, sc, cam, W, H, libm_matches)
    assert (ids >= 0).any() and (ids < 0).any(), "the frame must hold both hits and sky"


# ---- the sky texel shortcut at other fields of view (index-encoding sky: a neighbouring texel changes the pixel) ------
VIEW_SKY_CASES = [
    # (aspect, camera org, yaw, pitch).  A pole projects to the image column dx = 0 (rotateDir has no roll), which lies
    # in the frame only for aspect >= 1/2: the two pole cases are at aspect 4, each with a pixel inside the 1.2 degree cap
    # that always takes the exact path.
    (0.02, (4.0, 3.0, 10.0), 180.0, -20.0),
    (0.35, (4.0, 3.0, 10.0), 71.0, 12.0),
    (4.0, (4.0, 3.0, 10.0), 180.0, -60.0),      # the pole above in view
    (4.0, (4.0, 3.0, 10.0), 30.0, 43.09),       # the pole below in view
    (-1.0, (4.0, 3.0, 10.0), 200.0, 75.0),      # looking backwards (fz < 0)
]


@pytest.mark.parametrize("case", range(len(VIEW_SKY_CASES)))
def test_sky_texel_shortcut_at_other_fields_of_view(case, renderer, oracle_best, pkg, libm_matches):
    a, org, yaw, pitch = VIEW_SKY_CASES[case]
    base = pkg.scene.reference_scene(64, 1)
    sc = dataclasses.replace(base, sky=_index_sky(pkg, 1024, 512), aspect=np.float32(a), name=f"index_sky_fov{case}")
    cam = pkg.scene.Camera(org=org, yaw=yaw, pitch=pitch)
    W, H = 333, 187
    px, ids, c = check_three_ways(renderer, oracle_best, pkg, sc, cam, W, H, libm_matches)
    miss = c["pixels"] - c["hit_pixels"]
    assert miss > 0.2 * c["pixels"]
    if a > 0:
        assert c["sky_exact"] < 0.25 * miss, (c["sky_exact"], miss)   # the shortcut decides the frame's sky


# ---- unclamped camera angles (checkKey steps +-1 degree with no clamp, kernel.cu:1716-1759) --------------------------
ANGLES = [("pitch", p) for p in (90.0, -90.0, 90.5, 135.0, 180.0, -200.0, 271.0, 735.0)] + \
         [("yaw", y) for y in (-3590.0, 359.999, 100000.25)]


@pytest.mark.parametrize("scene_kind", ["R64_1", "prims"])
@pytest.mark.parametrize("which,angle", ANGLES, ids=[f"{w}{v:g}" for w, v in ANGLES])
def test_unclamped_camera_angles(which, angle, scene_kind, renderer, oracle_best, pkg, libm_matches):
    if scene_kind == "R64_1":
        if "R64_1" not in _fov_cache:
            _fov_cache["R64_1"] = FOV_SCENES["R64_1"]()
        sc, cam = _fov_cache["R64_1"], pkg.scene.reference_camera()
    else:
        if "S64_2_prims" not in _fov_cache:
            _fov_cache["S64_2_prims"] = FOV_SCENES["S64_2_prims"]()
        sc = _fov_cache["S64_2_prims"]
        cam = pkg.scene.orbit_camera(sc, 40)
    cam = dataclasses.replace(cam, **{which: angle})
    check_three_ways(renderer, oracle_best, pkg, sc, cam, 96, 64, libm_matches)


# ---- camera positions -----------------------------------------------------------------------------------------------
def test_camera_far_from_the_scene(renderer, oracle_best, pkg, libm_matches):
    """10^3 units back (telephoto, a sphere's silhouette in view), and 10^5 units away outside a small sky sphere
    (R = size^2 = 4e4): the sky shortcut must stand down for every miss pixel"""
    W, H = 161, 91
    base = pkg.scene.reference_scene(64, 1)
    sc = _aspect(base, 0.02)
    cam = _silhouette_camera(base, 0.02, W, H, yaw=250.0)
    _, ids, c = check_three_ways(renderer, oracle_best, pkg, sc, cam, W, H, libm_matches)
    assert (ids >= 0).any() and (ids < 0).any()
    small_sky = dataclasses.replace(sc, sky_size=200.0, name="far_small_sky")
    cam = _aim(0.02, W, H, (5.0, 5.0, 5.0), 1e5, yaw=123.0, pitch=-7.0)
    _, ids, c = check_three_ways(renderer, oracle_best, pkg, small_sky, cam, W, H, libm_matches)
    assert (ids >= 0).any() and (ids < 0).any()
    assert c["sky_exact"] == c["pixels"] - c["hit_pixels"], c


def _last_hit_first_miss(oracle, eye_yz, centre, member):
    """floats x below / at which the reference's float sphere test of an outward ray (+x) from (x, y, z) still hits
    (inside or on the sphere) and the first one above at which it misses (outside, looking away)"""
    def hit(x):
        return oracle.sphere_intersect((float(x), *eye_yz), (1.0, 0.0, 0.0), centre, member)[0]
    lo = np.float32(centre[0])
    hi = np.float32(centre[0] + 2.0 * member + 1.0)
    assert hit(lo) and not hit(hi)
    lo_b, hi_b = int(lo.view(np.int32)), int(hi.view(np.int32))   # positive floats: bits are monotonic
    while hi_b - lo_b > 1:
        mid = (lo_b + hi_b) // 2
        if hit(np.int32(mid).view(np.float32)):
            lo_b = mid
        else:
            hi_b = mid
    return np.int32(lo_b).view(np.float32), np.int32(hi_b).view(np.float32)


def test_camera_inside_and_on_the_surface_of_a_sphere(renderer, oracle_best, pkg, libm_matches):
    """the eye at a sphere's centre, and on its surface as the reference's float C sees it: the last float of one
    coordinate inside, the first outside (where the result flips) and the float nearest the real surface"""
    sc = pkg.scene.reference_scene(64, 1)
    a = float(sc.aspect)
    ez = np.float32(-1.0 / a)
    i = int(np.argmax(sc.spheres[:, 3]))
    cx, cy, cz, member = (float(v) for v in sc.spheres[i])
    W, H = 96, 64
    for yaw, pitch in ((180.0, -20.0), (0.0, 0.0), (77.0, 45.0)):
        org_z = np.float32(np.float32(cz) - ez)
        eye_z = float(np.float32(ez + org_z))                    # c.Oz = ez + org.z (float)
        cam = pkg.scene.Camera(org=(cx, cy, float(org_z)), yaw=yaw, pitch=pitch)
        _, ids, _ = check_three_ways(renderer, oracle_best, pkg, sc, cam, W, H, libm_matches)
        assert (ids == i).any(), "inside the sphere: its far wall is seen"
        x_in, x_out = _last_hit_first_miss(oracle_best, (cy, eye_z), (cx, cy, cz), member)
        x_geo = np.float32(cx + math.sqrt(max(0.0, member * member - (eye_z - cz) ** 2)))
        for x in (x_in, x_out, x_geo):
            cam = pkg.scene.Camera(org=(float(x), cy, float(org_z)), yaw=yaw, pitch=pitch)
            check_three_ways(renderer, oracle_best, pkg, sc, cam, W, H, libm_matches)


def test_camera_on_a_cube_face_plane(renderer, oracle_best, pkg, libm_matches):
    sc = _prim_scene(64, 2)
    a = float(sc.aspect)
    cube = sc.cubes[3]
    lo, hi = np.minimum(cube[:3], cube[3:]), np.maximum(cube[:3], cube[3:])
    mid = 0.5 * (lo + hi)
    for eye, yaw, pitch in (((hi[0], mid[1], mid[2] + 3.0), 90.0, 10.0), ((lo[0], mid[1], mid[2]), 270.0, -5.0),
                            ((mid[0], hi[1], mid[2]), 180.0, 60.0)):
        cam = pkg.scene.Camera(org=_eye_to_org(eye, a), yaw=yaw, pitch=pitch)
        check_three_ways(renderer, oracle_best, pkg, sc, cam, 96, 64, libm_matches)


# ---- frame shapes and bands -----------------------------------------------------------------------------------------
SHAPES = [(1, 1), (1, 97), (97, 1), (2, 3), (3, 5), (31, 8), (32, 8), (33, 9), (63, 17), (4099, 2)]


@pytest.mark.parametrize("W,H", SHAPES, ids=[f"{w}x{h}" for w, h in SHAPES])
def test_tiny_and_ragged_frames(W, H, renderer, oracle_best, pkg, libm_matches):
    """ragged tiles, dx_tab padding and the sky's quad stores (x4 + 3 < W) on their other branches"""
    if "R64_1" not in _fov_cache:
        _fov_cache["R64_1"] = FOV_SCENES["R64_1"]()
    sc = _fov_cache["R64_1"]
    # a camera that sees spheres and sky in every one of these frames' few pixels is not guaranteed; two views
    for cam in (pkg.scene.reference_camera(), pkg.scene.Camera(org=(5.0, 5.0, -4.0), yaw=0.0, pitch=0.0)):
        check_three_ways(renderer, oracle_best, pkg, sc, cam, W, H, libm_matches)


def test_4k_band_whose_row_span_makes_the_tile_cone_fall_back(renderer, oracle_best, pkg, libm_matches):
    sc = pkg.scene.scaled_scene(1024, 3)
    cam = pkg.scene.orbit_camera(sc, 60)
    _, ids, _ = check_three_ways(renderer, oracle_best, pkg, sc, cam, 3840, 2160, libm_matches, y0=20, y1=2160, y_step=2100)
    assert ids.shape == (2, 3840) and (ids >= 0).any()


BLOCKS = [(2, 3), (2, 7), (2, 24), (3, 3), (3, 7), (3, 24), (8, 24), (8, 8), (7, 7)]


def _band_rows(H, y0, y_step, y_block):
    return [y for y in range(y0, H) if (y - y0) % y_step < y_block]


@pytest.mark.parametrize("y_block,y_step", BLOCKS, ids=[f"b{b}s{s}" for b, s in BLOCKS])
def test_block_interleaved_bands_equal_the_oracle_rows(y_block, y_step, renderer, oracle_best, pkg, libm_matches):
    """the oracle has no y_block: the band's rows are compared with its full frame"""
    if "S64_2_prims" not in _fov_cache:
        _fov_cache["S64_2_prims"] = FOV_SCENES["S64_2_prims"]()
    sc = _fov_cache["S64_2_prims"]
    cam = pkg.scene.orbit_camera(sc, 17)
    W, H, y0 = 161, 91, 5
    F = pkg.capi
    key = ("full", W, H)
    if key not in _fov_cache:
        _fov_cache[key] = oracle_best.render(sc, cam, W, H)
    ref = _fov_cache[key]
    rows = _band_rows(H, y0, y_step, y_block)
    kw = dict(y0=y0, y_step=y_step, y_block=y_block)
    _use(renderer, sc)
    px = renderer.render(cam, W, H, **kw).copy()
    ids, t = renderer.hits(px.shape[0], W)
    assert px.shape[0] == len(rows)
    assert np.array_equal(ids, ref["ids"][rows])
    assert np.array_equal(t.view(np.uint32), ref["t"][rows].view(np.uint32))
    assert_pixels_close(px, ref["pixels"][rows])
    if libm_matches:
        assert np.array_equal(px, ref["pixels"][rows])
    for flags in (F.ORE_FLAG_FUSED_SHADOW, F.ORE_FLAG_EXHAUSTIVE):
        assert np.array_equal(renderer.render(cam, W, H, flags=flags, **kw), px), flags
    assert_pixels_close(renderer.render(cam, W, H, flags=F.ORE_FLAG_FAST_LIBM, **kw), px)


# ---- strided and misaligned device outputs --------------------------------------------------------------------------
# Which sky stores run: the primary kernel stores a quad of 4 sky pixels with one 128-bit store when the output base is
# 16-byte aligned (offset 0 here: torch allocations and the guard are 16-byte multiples), the row pitch is a multiple
# of 4 pixels (out_pitch 0 means a pitch of W) and the quad lies inside the row (x4 + 3 < W).  Every other quad - an
# offset of 4, 8 or 12 bytes, a pitch of W + 1 or W + 3 for W = 161, any pitch of an odd W, the last partial quad of
# W = 33 or 161, and W = 1 or 3 - is stored pixel by pixel.  _vector_stores() says which, and the test asserts both occur.
GUARD = 64   # words before and after the output (a multiple of 4: the offset alone decides the alignment)


def _vector_stores(offset_bytes, pitch, W):
    return offset_bytes % 16 == 0 and pitch % 4 == 0 and W >= 4


def _sentinel_buffer(n_words):
    import torch
    return torch.full((n_words,), SENTINEL, dtype=torch.int32, device="cuda:0")


def _host(buf):
    return buf.cpu().numpy().view(np.uint32)


def _expect(n_words, base, frame, row_of, pitch, rows):
    """a sentinel buffer with `rows` of `frame` stored at base + row_of(k) * pitch"""
    want = np.full(n_words, SENTINEL, dtype=np.uint32)
    W = frame.shape[1]
    for k in rows:
        want[base + row_of(k) * pitch: base + row_of(k) * pitch + W] = frame[k]
    return want


def test_strided_and_misaligned_device_outputs(renderer, pkg):
    sc = pkg.scene.scaled_scene(64, 2)
    cam = pkg.scene.orbit_camera(sc, 21)
    renderer.set_scene(sc)
    H = 19
    seen = set()
    for W in (1, 3, 33, 161):
        want = renderer.render(cam, W, H).copy()
        for off in (0, 4, 8, 12):
            for out_pitch in (0, W, W + 1, W + 3, W + 4):
                pitch = out_pitch or W
                n = 2 * GUARD + off // 4 + H * pitch
                buf = _sentinel_buffer(n)
                base = GUARD + off // 4
                renderer.render_device(cam, W, H, out_ptr=buf.data_ptr() + 4 * base, out_pitch=out_pitch)
                renderer.synchronize()
                got = _host(buf)
                exp = _expect(n, base, want, lambda k: k, pitch, range(H))
                assert np.array_equal(got, exp), (W, off, out_pitch, int(np.count_nonzero(got != exp)))
                seen.add(_vector_stores(off, pitch, W))
    assert seen == {True, False}


def test_strided_outputs_of_batches_and_bands(renderer, pkg):
    """a batch of 3 frames at different offsets, 3-rank block_band bands into shared frames with a padded pitch, and
    the band-DMA copy: every rendered pixel right, every other word (guards, pitch padding, other ranks' rows) intact"""
    sc = pkg.scene.scaled_scene(64, 2)
    renderer.set_scene(sc)
    F = pkg.capi
    W, H = 161, 37
    cams = [pkg.scene.orbit_camera(sc, f) for f in (3, 100, 190)]
    want = [renderer.render(c, W, H).copy() for c in cams]
    for out_pitch in (0, W, W + 3, W + 4):
        pitch = out_pitch or W
        offs = (0, 4, 12)
        bufs = [_sentinel_buffer(2 * GUARD + 3 + H * pitch) for _ in cams]
        renderer.render_batch_device(cams, W, H, [b.data_ptr() + 4 * (GUARD + o // 4) for b, o in zip(bufs, offs)],
                                     out_pitch=out_pitch)
        renderer.synchronize()
        for i, (b, o) in enumerate(zip(bufs, offs)):
            exp = _expect(b.numel(), GUARD + o // 4, want[i], lambda k: k, pitch, range(H))
            assert np.array_equal(_host(b), exp), (out_pitch, i)
    # ranks of a block-interleaved frame: rank r writes image rows at their place; the others' rows stay sentinel
    for pitch, flags in ((W, 0), (W + 4, 0), (W + 1, 0), (W, F.ORE_FLAG_BAND_DMA), (W, F.ORE_FLAG_BAND_DMA | F.ORE_FLAG_FUSED_SHADOW)):
        for off in (0, 8):
            bufs = [_sentinel_buffer(2 * GUARD + 3 + H * pitch) for _ in cams]
            for rank in (0, 2):             # rank 1 renders nothing: its rows must keep the sentinel
                b = pkg.multigpu.block_band(rank, 3, H)
                base = GUARD + off // 4 + b["y0"] * pitch
                renderer.render_batch_device(cams, W, H, [x.data_ptr() + 4 * base for x in bufs], out_pitch=pitch,
                                             flags=flags, **b)
            renderer.synchronize()
            mine = pkg.multigpu.block_rows(0, 3, H) + pkg.multigpu.block_rows(2, 3, H)
            for i, x in enumerate(bufs):
                exp = _expect(x.numel(), GUARD + off // 4, want[i], lambda k: k, pitch, mine)
                got = _host(x)
                assert np.array_equal(got, exp), (pitch, flags, off, i, int(np.count_nonzero(got != exp)))


# ---- mixed batches --------------------------------------------------------------------------------------------------
def _mixed_cameras(sc):
    """8 frames in different regimes of one scene with cubes, a plane and the torus"""
    Cam = cases.scene.Camera
    a = float(sc.aspect)
    e = sc.extent
    s0 = sc.spheres[int(np.argmax(sc.spheres[:, 3]))]
    box = sc.mesh.box_bounds[0]
    blo = np.minimum(box[:3], box[3:])
    bmid = 0.5 * (box[:3] + box[3:])
    cube = sc.cubes[0]
    chi = np.maximum(cube[:3], cube[3:])
    cmid = 0.5 * (cube[:3] + cube[3:])
    R_sky = float(sc.sky_size) ** 2
    return [
        cases.scene.reference_camera(),
        Cam(org=_eye_to_org(s0[:3], a), yaw=33.0, pitch=10.0),                                  # inside a sphere
        _aim(a, 128, 72, (e / 2, e / 2, e / 2), 1e3, yaw=210.0, pitch=5.0),                     # far away
        Cam(org=(e / 2, e / 2, -e), yaw=-3590.0, pitch=135.0),                                  # upside down
        Cam(org=(e / 2, 2 * e, e / 2), yaw=0.0, pitch=90.0),                                    # straight down
        Cam(org=_eye_to_org((blo[0], bmid[1], bmid[2]), a), yaw=90.0, pitch=5.0),               # torus leaf face plane
        Cam(org=_eye_to_org((chi[0], cmid[1], cmid[2]), a), yaw=270.0, pitch=0.0),              # cube face plane
        _aim(a, 128, 72, (0.0, 0.0, 0.0), 1.05 * R_sky, yaw=180.0, pitch=0.0),                  # outside the sky sphere
    ]


PRIMARY_COUNTERS = ("hit_pixels", "sky_exact", "exact_primary", "primary_steps")


@pytest.mark.parametrize("n,seed", [(64, 2), (16384, 5)], ids=["S64_2_prims", "S16384_5_prims"])
def test_mixed_batch_equals_single_frames_and_the_oracle(n, seed, renderer, oracle_best, pkg, libm_matches):
    import torch
    sc = _prim_scene(n, seed)
    lens = pkg.capi.sphere_tree_lengths(n)
    resident = 16 * (lens["sph_sort"] + lens["leaf_sph"] + lens["super_sph"]) <= 30 * 1024   # frame_params' check
    assert resident == (n == 64)
    cams = _mixed_cameras(sc)
    W, H = 128, 72
    renderer.set_scene(sc)
    F = pkg.capi
    for flags in (0, F.ORE_FLAG_EXHAUSTIVE):
        singles, sums = [], dict.fromkeys(PRIMARY_COUNTERS, 0)
        for c in cams:
            singles.append(renderer.render(c, W, H, flags=flags).copy())
            cn = renderer.counters()
            for k in PRIMARY_COUNTERS:
                sums[k] += cn[k]
        frames = torch.full((len(cams), H, W), SENTINEL, dtype=torch.int32, device="cuda:0")
        renderer.render_batch_device(cams, W, H, [frames[i].data_ptr() for i in range(len(cams))], flags=flags)
        renderer.synchronize()
        cb = renderer.counters()
        got = frames.cpu().numpy().view(np.uint32)
        for i in range(len(cams)):
            assert np.array_equal(got[i], singles[i]), (flags, i, int(np.count_nonzero(got[i] != singles[i])))
        assert {k: cb[k] for k in PRIMARY_COUNTERS} == sums, flags
        if flags == 0:
            kw = dict(y0=3, y1=H, y_step=11)
            for i, c in enumerate(cams):
                ref = oracle_best.render(sc, c, W, H, **kw)
                rows = slice(3, H, 11)
                if libm_matches:
                    assert np.array_equal(got[i][rows], ref["pixels"]), (i, int(np.count_nonzero(got[i][rows] != ref["pixels"])))
                else:
                    assert_pixels_close(got[i][rows], ref["pixels"])
                px = renderer.render(c, W, H, **kw)
                ids, t = renderer.hits(px.shape[0], W)
                assert np.array_equal(ids, ref["ids"]) and np.array_equal(t.view(np.uint32), ref["t"].view(np.uint32)), i


# ---- rejected aspects -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("a", [0.0, float("inf"), float("-inf"), float("nan"), 1e-40])
def test_aspects_without_a_finite_eye_are_rejected(a, renderer, pkg):
    """0, +-inf, NaN and an aspect whose reciprocal overflows return ORE_ERR_INVALID from every render entry point and
    leave the output untouched"""
    import ctypes as C
    sc = pkg.scene.reference_scene(16, 3)
    renderer.set_scene(sc)
    cam = pkg.scene.reference_camera()
    W, H = 40, 24
    lib, ctx = renderer.lib, renderer.ctx
    f = renderer._frame(W, H, 0, H, 1, a, 0)
    cs = renderer._cams([cam, cam])
    host = np.full((H, W), SENTINEL, dtype=np.uint32)
    assert lib.ore_render(ctx, C.byref(cs[0]), C.byref(f), host.ctypes.data) == 1
    assert "aspect" in lib.ore_last_error(ctx).decode()
    assert np.all(host == SENTINEL)
    dev = _sentinel_buffer(2 * H * W)
    assert lib.ore_render_device(ctx, C.byref(cs[0]), C.byref(f), C.c_void_p(dev.data_ptr()), None) == 1
    ptrs = (C.c_void_p * 2)(dev.data_ptr(), dev.data_ptr() + 4 * H * W)
    assert lib.ore_render_batch_device(ctx, cs, 2, C.byref(f), ptrs, None) == 1
    pinned = renderer.host_alloc((H, W))
    try:
        pinned[:] = SENTINEL
        assert lib.ore_render_async(ctx, C.byref(cs[0]), C.byref(f), pinned.ctypes.data) == 1
        renderer.wait()
        assert np.all(pinned == SENTINEL)
    finally:
        renderer.host_free(pinned)
    renderer.synchronize()
    assert np.all(_host(dev) == SENTINEL)
    assert np.array_equal(renderer.render(cam, W, H), renderer.render(cam, W, H, aspect=float(sc.aspect)))
