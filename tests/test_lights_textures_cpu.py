"""CPU side of tests/test_lights_textures_gpu.py (oracle and host libm only, no GPU): the light sets of 1-16 lights give
32-pixel blocks with every kind of lit-light mask, the texel-hash texture makes a one-texel error visible in nearly
every lit pixel (object texture and sky), and the stored libm table equals this host's libm where it is glibc 2.39 with
FMA."""
import math
import platform

import numpy as np
import pytest

import libmkat
from test_host_mesh import host_lib  # noqa: F401  (fixture re-export)
from test_random_primitives_gpu import mesh_probe  # noqa: F401  (fixture re-export)

F32 = np.float32
# rows of every light set: 0 is the all-zero colour when there are at least four lights
LIGHT_SIZES = (0.0, 1.0, 20.0, 400.0)
LIGHT_KINDS = ("above", "side", "above", "grazing", "below", "above", "back", "inside")


# ---- shared with the GPU file -----------------------------------------------------------------------------------------

def hash_texture(pkg, w, h, seed=1):
    """every texel its own pseudo-random 24-bit colour (a seeded hash of its index): a neighbouring texel differs by
    tens of levels per channel almost everywhere, so a pixel that read the wrong texel shows it"""
    i = np.arange(w * h, dtype=np.uint64)
    x = i + np.uint64((seed * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF)
    for sh, mul in ((30, 0xBF58476D1CE4E5B9), (27, 0x94D049BB133111EB)):   # splitmix64
        x = ((x ^ (x >> np.uint64(sh))) * np.uint64(mul)) & np.uint64(0xFFFFFFFFFFFFFFFF)
    x ^= x >> np.uint64(31)
    rgb = np.stack([(x >> np.uint64(s)) & np.uint64(0xFF) for s in (0, 8, 16)], axis=-1).astype(np.uint8)
    return pkg.scene.Sprite.from_bytes(rgb.reshape(h, w, 3))


def light_set(n, seed, spheres, centre, extent):
    """n lights (7 floats each) about a scene of the given centre and extent, from a few directions only, so that many
    surfaces face none or one of them: above it, beside it, level with it (the terminator crosses many blocks), below
    it and behind it, all to its +x side, and inside its largest sphere (facing, but every shadow ray blocked); sizes
    0, 1, 20 and 400; colours small enough that 16 of them rarely saturate a pixel, one all zero"""
    rng = np.random.default_rng(1000 + seed)
    c = np.asarray(centre, np.float64)
    E = float(extent)
    big = None
    if len(spheres):
        big = np.asarray(spheres[int(np.argmax(spheres[:, 3]))], np.float64)
    # every direction leans to +x: surfaces that face -x see none of them
    where = {"above": (1.5, 3, 0), "side": (4, 1.5, 0), "grazing": (4, 0, 0), "below": (1.5, -3, 0), "back": (1.5, 0.5, -3)}
    out = np.zeros((n, 7), F32)
    for i in range(n):
        kind = LIGHT_KINDS[(i + seed) % len(LIGHT_KINDS)]
        j = rng.uniform(-0.3, 0.3, 3)
        if kind == "inside" and big is not None:
            p = big[:3] + 0.01
        else:
            p = c + (np.array(where.get(kind, (0, 3, 0)), np.float64) + j) * E
        out[i, :3] = p
        out[i, 3] = LIGHT_SIZES[i % 4]
        out[i, 4:] = rng.uniform(0.01, 0.13, 3)
    if n >= 4:
        out[0, 4:] = 0.0
    return out


def with_lights(pkg, sc, lights):
    return pkg.scene.Scene(spheres=sc.spheres, lights=np.ascontiguousarray(lights, F32), texture=sc.texture, sky=sc.sky,
                           aspect=sc.aspect, sky_size=sc.sky_size, extent=sc.extent, name=sc.name, cubes=sc.cubes,
                           planes=sc.planes, mesh=sc.mesh)


def light_scenes(pkg, host_lib, mesh_probe, tmp_path):
    """(name, scene, camera) of the light-set tests: the reference scene, overlapping spheres, every primitive kind"""
    from test_random_primitives_gpu import random_primitive_scene
    from test_random_scenes_gpu import random_scene
    ref = pkg.scene.reference_scene(64, 1)
    ov, ov_cam = random_scene(pkg, 13)                   # style 1: radii up to 1.8, heavy overlap, 301 spheres
    mixed, _, _, _ = random_primitive_scene(pkg, 12, host_lib, mesh_probe, tmp_path)   # spheres, cubes, plane, torus
    mixed_cam = pkg.scene.orbit_camera(mixed, 30)                 # (the scene's own camera looks along an axis at little)
    return [("reference", ref, pkg.scene.reference_camera()), ("overlap", ov, ov_cam), ("mixed", mixed, mixed_cam)]


def lit_scene(pkg, sc, n, seed):
    e = sc.extent
    return with_lights(pkg, sc, light_set(n, seed, sc.spheres, (e / 2, e / 2, e / 2), e))


# ---- the light sets vary the lit mask from block to block ---------------------------------------------------------------

def _rays(cam, W, H, aspect):
    """primary rays of the reference's camera (kernel.cu:1624-1631), float64: enough to tell which side of a surface a
    light is on"""
    y, x = np.meshgrid(np.arange(H, dtype=np.float64), np.arange(W, dtype=np.float64), indexing="ij")
    a = float(aspect)
    dx = a * (2 * (x + 0.5) / W) - 1
    dy = a * (2 * (y + 0.5) / H) * (H / W) - 1
    d = np.stack([dx, dy, np.full_like(dx, 1 / a)], axis=-1)
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    yaw, pitch = cam.yaw * (3.1415 / 180), cam.pitch * (3.1415 / 180)
    yy = d[..., 1] * math.cos(pitch) - d[..., 2] * math.sin(pitch)
    z = d[..., 1] * math.sin(pitch) + d[..., 2] * math.cos(pitch)
    xx = d[..., 0] * math.cos(yaw) + z * math.sin(yaw)
    zz = -d[..., 0] * math.sin(yaw) + z * math.cos(yaw)
    O = np.array([0, 0, -1 / a]) + np.asarray(cam.org, np.float64)
    return O, np.stack([xx, yy, zz], axis=-1)


def facing_masks(sc, cam, W, H, ids, t):
    """bit li of each hit pixel (row order): normal . (light - hit point) > 0; face normals for triangles"""
    O, D = _rays(cam, W, H, sc.aspect)
    hit = ids >= 0
    P = O + D[hit] * t[hit].astype(np.float64)[:, None]
    k = ids[hit]
    ns, nc, npl = len(sc.spheres), len(sc.cubes), len(sc.planes)
    nrm = np.zeros_like(P)
    s = k < ns
    nrm[s] = P[s] - sc.spheres[k[s], :3]
    c = (k >= ns) & (k < ns + nc)
    nrm[c] = P[c] - (sc.cubes[k[c] - ns, :3].astype(np.float64) + sc.cubes[k[c] - ns, 3:]) / 2
    p = (k >= ns + nc) & (k < ns + nc + npl)
    nrm[p] = sc.planes[k[p] - ns - nc, 3:]
    m = k >= ns + nc + npl
    if m.any():
        nrm[m] = sc.mesh.tris[k[m] - ns - nc - npl, 9:12]
    mask = np.zeros(len(k), np.int64)
    for li, L in enumerate(sc.lights):
        a = np.einsum("ij,ij->i", nrm, L[:3].astype(np.float64) - P)
        mask |= (a > 0).astype(np.int64) << li
    return mask


LIGHT_COUNTS = [1, 4, 5, 8, 15, 16]   # the light sets of test_lights_textures_gpu.py: n lights, seed n


def test_light_sets_give_blocks_with_none_one_and_many_lit_lights(pkg, oracle_best, host_lib, mesh_probe, tmp_path):  # noqa: F811
    """over the light sets and scenes the GPU tests render (200x150), runs of 32 hit pixels - the shadow pass's blocks;
    the hit list keeps a warp's tile together, row order is the stand-in here - face 0, 1 and many lights, odd and even
    counts, lights past bit 8 included"""
    per_n = {}
    masks = 0
    scenes = light_scenes(pkg, host_lib, mesh_probe, tmp_path)
    for n in LIGHT_COUNTS:
        counts = []
        for name, base, cam in scenes:
            sc = lit_scene(pkg, base, n, n)
            W, H = 200, 150
            ref = oracle_best.render(sc, cam, W, H)
            mask = facing_masks(sc, cam, W, H, ref["ids"], ref["t"])
            assert mask.size > 2000, (name, mask.size)
            for b in range(0, mask.size - 31, 32):
                m = int(np.bitwise_or.reduce(mask[b:b + 32]))
                counts.append(bin(m).count("1"))
                masks |= m
        per_n[n] = np.bincount(counts, minlength=n + 1)
        print(n, "lights: blocks by lit-light count", per_n[n].tolist())
    several = np.concatenate([per_n[n][:5] for n in LIGHT_COUNTS if n >= 4]).reshape(-1, 5).sum(axis=0)
    assert several[0] > 0 and several[1] > 0, several          # with 4 or more lights: blocks that face none, one
    for n in (8, 15, 16):
        c = per_n[n]
        assert c[8:].sum() > 0, (n, c)                          # ... and many
        assert c[3::2].sum() > 0 and c[2::2].sum() > 0, (n, c)   # odd and even counts above one
        assert np.count_nonzero(c) >= 5, (n, c)
    assert masks >> 8, "lights 8..15 must face some block"


# ---- a one-texel error is visible ---------------------------------------------------------------------------------------

def _roll(pkg, sprite, dx, dy):
    def r(p):
        return np.ascontiguousarray(np.roll(p.reshape(sprite.height, sprite.width), (dy, dx), axis=(0, 1)).reshape(-1))
    return pkg.scene.Sprite(sprite.width, sprite.height, r(sprite.r), r(sprite.g), r(sprite.b))


def texel_scene(pkg, w, h):
    """spheres, cubes and the plane under the reference's lights, textured with the texel hash"""
    base = pkg.scene.reference_scene(64, 1, texture=hash_texture(pkg, w, h), sky=hash_texture(pkg, 1024, 512, 2))
    return pkg.scene.with_cubes_and_plane(base, 12, 5)


def test_the_hash_texture_differs_from_its_neighbours(pkg):
    s = hash_texture(pkg, 257, 129)
    r = np.rint(s.r.reshape(129, 257) * 255)
    for d in (np.abs(np.diff(r, axis=0)), np.abs(np.diff(r, axis=1))):
        assert np.count_nonzero(d >= 8) >= 0.9 * d.size and d.mean() > 60


@pytest.mark.parametrize("wh", [(257, 129), (1024, 512)])
def test_a_neighbouring_object_texel_changes_nearly_every_lit_pixel(wh, pkg, oracle_best):
    sc = texel_scene(pkg, *wh)
    cam = pkg.scene.orbit_camera(sc, 30)
    W, H = 160, 120
    ref = oracle_best.render(sc, cam, W, H)
    lit = (ref["ids"] >= 0) & (ref["pixels"] != 0)
    assert lit.sum() > 0.2 * W * H
    for dx, dy in ((1, 0), (0, 1)):
        sc.texture = _roll(pkg, texel_scene(pkg, *wh).texture, dx, dy)
        px = oracle_best.render(sc, cam, W, H)["pixels"]
        frac = np.count_nonzero(px[lit] != ref["pixels"][lit]) / lit.sum()
        print(f"texture {wh} rolled by ({dx}, {dy}): {frac:.4f} of {int(lit.sum())} lit hit pixels change")
        assert frac >= 0.9, (dx, dy, frac)


def test_a_neighbouring_sky_texel_changes_nearly_every_sky_pixel(pkg, oracle_best):
    sc = texel_scene(pkg, 257, 129)
    cam = pkg.scene.Camera(org=(4.0, 3.0, 10.0), yaw=150.0, pitch=-45.0)   # (negative pitch looks up)
    W, H = 160, 120
    ref = oracle_best.render(sc, cam, W, H)
    sky = ref["ids"] < 0
    assert sky.sum() > 0.2 * W * H
    for dx, dy in ((1, 0), (0, 1)):
        sc.sky = _roll(pkg, texel_scene(pkg, 257, 129).sky, dx, dy)
        px = oracle_best.render(sc, cam, W, H)["pixels"]
        frac = np.count_nonzero(px[sky] != ref["pixels"][sky]) / sky.sum()
        print(f"sky rolled by ({dx}, {dy}): {frac:.4f} of {int(sky.sum())} sky pixels change")
        assert frac >= 0.9, (dx, dy, frac)


# ---- mesh vt outside [0, 1] ---------------------------------------------------------------------------------------------

def test_the_obj_loader_keeps_vt_outside_the_unit_square(host_lib, tmp_path):
    """the reference's loader reads vt with operator>> (kernel.cu:594-700, host/ore_mesh.cpp): values outside [0, 1]
    reach the texel lookup unchanged; tests/test_lights_textures_gpu.py uses them only where the reference's index
    stays inside the texture"""
    from test_host_mesh import host_build
    from test_lights_textures_gpu import VT_OUTSIDE, write_vt_grid_obj
    obj = str(tmp_path / "vt.obj")
    write_vt_grid_obj(obj, outside=True)
    m = host_build(host_lib, obj)
    vt = m["tris"][:, 21:27].reshape(-1, 2)
    for u, v in VT_OUTSIDE:
        assert np.any(np.all(vt == np.array([u, v], F32), axis=1)), (u, v)
    assert vt.min() < 0 and vt.max() > 1


# ---- the stored libm table ----------------------------------------------------------------------------------------------

def test_the_stored_libm_table_is_this_hosts_libm():
    """tests/golden/libm_kat.npz re-checked against the host libm, where the host is the variant it came from"""
    if not (libmkat.glibc_version() == "2.39" and platform.machine() == "x86_64" and libmkat.cpu_has_fma()):
        pytest.skip(f"the table holds glibc 2.39 / x86-64 / FMA answers; this host has {libmkat.host_description()}")
    table, host = libmkat.load()
    assert host == libmkat.host_description(), host
    lm = libmkat.host_libm()
    problems = []
    for op, t in table.items():
        problems += libmkat.check(op, t, lambda a, b, op=op: libmkat.host_eval(lm, op, a, b))
        assert t["ra"].size == libmkat.RANDOM_N and t["rbits_head"].size == libmkat.RANDOM_STORED, op
    assert not problems, problems
    sizes = {op: t["a"].size for op, t in table.items()}
    assert sizes["acosf"] > 50 and min(sizes["sinf"], sizes["cosf"], sizes["atan2f"]) > 1000, sizes


PINNED_ACOSF_INPUTS = [0x3F444150, 0x3E08516F, 0x3E3AC1AF]   # the first random acosf inputs of tests/libmkat.py


def test_the_random_libm_inputs_do_not_depend_on_the_host():
    """the random inputs behind the stored digests come from integer hashing and IEEE float operations only; pinned
    here by a few values and their range"""
    a, _ = libmkat.random_inputs("acosf")
    x, _ = libmkat.random_inputs("sinf")
    y, xx = libmkat.random_inputs("atan2f")
    assert a.size == x.size == y.size == libmkat.RANDOM_N
    assert np.all(np.abs(a) <= 1) and np.all(np.abs(x) < 120)
    n2 = y.astype(np.float64) ** 2 + xx.astype(np.float64) ** 2
    assert np.all(n2 <= 1 + 1e-6)
    assert a[:3].view(np.uint32).tolist() == PINNED_ACOSF_INPUTS, [hex(v) for v in a[:3].view(np.uint32)]
