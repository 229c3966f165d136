"""ctypes front-end for the CPU checkers in oracle/ (TEST INFRASTRUCTURE ONLY).

`load("port")`  -> oracle/liboracle.so        (C restatement, oracle/oracle.c)
`load("ref")`   -> oracle/_ref/libref_oracle.so (the reference's own code as host C++;
                   only present when the build container produced it)
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
PORT_SO = os.path.join(ORACLE_DIR, "liboracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libref_oracle.so")

_fp = C.POINTER(C.c_float)


class OracleFrame(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32),
        ("y0", C.c_int32), ("y1", C.c_int32), ("y_step", C.c_int32),
        ("cam_org", C.c_float * 3), ("cam_yaw", C.c_float), ("cam_pitch", C.c_float),
        ("aspect", C.c_float),
        ("n_spheres", C.c_int32), ("spheres", _fp),
        ("n_lights", C.c_int32), ("lights", _fp),
        ("tex_w", C.c_int32), ("tex_h", C.c_int32), ("tex_r", _fp), ("tex_g", _fp), ("tex_b", _fp),
        ("sky_w", C.c_int32), ("sky_h", C.c_int32), ("sky_r", _fp), ("sky_g", _fp), ("sky_b", _fp),
        ("sky_size", C.c_float),
        ("n_cubes", C.c_int32), ("cubes", _fp), ("n_planes", C.c_int32), ("planes", _fp),
        ("n_tris", C.c_int32), ("tris", _fp), ("mesh_has_normals", C.c_int32), ("n_boxes", C.c_int32),
        ("box_bounds", _fp), ("box_offsets", C.POINTER(C.c_int32)), ("box_indices", C.POINTER(C.c_int32)),
    ]


def _ptr(a: np.ndarray):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_fp)


def _vec(v, n=3):
    a = np.ascontiguousarray(v, dtype=np.float32).reshape(-1)
    assert a.size == n
    return (C.c_float * n).from_buffer_copy(a.tobytes())


def _supported(hit):
    if hit < 0:   # _ref: the reference revision has none of the call forms ref_driver.cpp knows for this test
        raise NotImplementedError("this reference build does not provide the single-primitive test")


def build_port():
    if not os.path.isfile(PORT_SO) or os.path.getmtime(PORT_SO) < os.path.getmtime(os.path.join(ORACLE_DIR, "oracle.c")):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "port"], stdout=subprocess.DEVNULL)
    return PORT_SO


def have_ref() -> bool:
    return os.path.isfile(REF_SO)


class Oracle:
    def __init__(self, path: str):
        self.path = path
        self.lib = C.CDLL(path)
        self.lib.oracle_render.restype = C.c_int
        self.lib.oracle_render.argtypes = [C.POINTER(OracleFrame), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        self.lib.oracle_sphere_intersect.restype = C.c_int
        self.lib.oracle_sphere_intersect.argtypes = [_fp, _fp, _fp, C.c_float, _fp]
        # single-primitive tests: liboracle always has them; a _ref library built before they existed does not
        self.has_primitive_tests = all(hasattr(self.lib, n) for n in
                                       ("oracle_cube_intersect", "oracle_plane_intersect", "oracle_tri_intersect"))
        if self.has_primitive_tests:
            for name in ("oracle_cube_intersect", "oracle_plane_intersect"):
                getattr(self.lib, name).restype = C.c_int
                getattr(self.lib, name).argtypes = [_fp, _fp, _fp, _fp, _fp]
            self.lib.oracle_tri_intersect.restype = C.c_int
            self.lib.oracle_tri_intersect.argtypes = [_fp, _fp, _fp, _fp, _fp, _fp]
        self.lib.oracle_rgb_to_int.restype = C.c_uint32
        self.lib.oracle_rgb_to_int.argtypes = [C.c_int, C.c_int, C.c_int]
        self.lib.oracle_kind.restype = C.c_char_p
        self.kind = self.lib.oracle_kind().decode()

    def render(self, scene, camera, width, height, y0=0, y1=None, y_step=1, n_threads=0,
               want_ids=True, want_t=True, n_lights=None):
        """Returns dict(pixels[u32 rows,W], ids[i32], t[f32], counts[u64 x4])."""
        y1 = height if y1 is None else y1
        rows = (y1 - y0 + y_step - 1) // y_step
        f = OracleFrame()
        f.width, f.height, f.y0, f.y1, f.y_step = width, height, y0, y1, y_step
        f.cam_org = (C.c_float * 3)(*[float(v) for v in camera.org])
        f.cam_yaw, f.cam_pitch = float(camera.yaw), float(camera.pitch)
        f.aspect = float(scene.aspect)
        sph = np.ascontiguousarray(scene.spheres, dtype=np.float32)
        lig = np.ascontiguousarray(scene.lights, dtype=np.float32)
        f.n_spheres, f.spheres = sph.shape[0], _ptr(sph.reshape(-1)) if sph.size else None
        nl = lig.shape[0] if n_lights is None else n_lights
        f.n_lights, f.lights = nl, _ptr(lig.reshape(-1))
        t, s = scene.texture, scene.sky
        f.tex_w, f.tex_h, f.tex_r, f.tex_g, f.tex_b = t.width, t.height, _ptr(t.r), _ptr(t.g), _ptr(t.b)
        f.sky_w, f.sky_h, f.sky_r, f.sky_g, f.sky_b = s.width, s.height, _ptr(s.r), _ptr(s.g), _ptr(s.b)
        f.sky_size = float(scene.sky_size)
        cubes = np.ascontiguousarray(getattr(scene, "cubes", np.zeros((0, 6), np.float32)), dtype=np.float32)
        planes = np.ascontiguousarray(getattr(scene, "planes", np.zeros((0, 6), np.float32)), dtype=np.float32)
        f.n_cubes, f.cubes = cubes.shape[0], (_ptr(cubes.reshape(-1)) if cubes.size else None)
        f.n_planes, f.planes = planes.shape[0], (_ptr(planes.reshape(-1)) if planes.size else None)
        mesh = getattr(scene, "mesh", None)
        if mesh is not None and mesh.n_tris > 0:
            _ip = C.POINTER(C.c_int32)
            f.n_tris, f.tris, f.mesh_has_normals = mesh.n_tris, _ptr(mesh.tris.reshape(-1)), int(mesh.has_normals)
            f.n_boxes, f.box_bounds = mesh.n_boxes, _ptr(mesh.box_bounds.reshape(-1))
            f.box_offsets = mesh.box_offsets.ctypes.data_as(_ip)
            f.box_indices = mesh.box_indices.ctypes.data_as(_ip)
        pixels = np.zeros((rows, width), dtype=np.uint32)
        ids = np.zeros((rows, width), dtype=np.int32) if want_ids else None
        tt = np.zeros((rows, width), dtype=np.float32) if want_t else None
        counts = np.zeros(4, dtype=np.uint64)
        rc = self.lib.oracle_render(
            C.byref(f), pixels.ctypes.data,
            ids.ctypes.data if want_ids else None, tt.ctypes.data if want_t else None,
            counts.ctypes.data, int(n_threads))
        if rc != 0:
            raise RuntimeError(f"oracle_render failed rc={rc}")
        return {"pixels": pixels, "ids": ids, "t": tt, "counts": counts}

    def build_mesh(self, obj_path: str, cap_tris=1 << 20, cap_boxes=4096):
        """_ref only: the reference's own OBJ loader + BVH builder; returns dict of flat arrays"""
        tris = np.zeros((cap_tris, 27), dtype=np.float32)
        bounds = np.zeros((cap_boxes, 6), dtype=np.float32)
        offs = np.zeros(cap_boxes + 1, dtype=np.int32)
        idx = np.zeros(cap_tris * 2, dtype=np.int32)
        nt, hn, nb = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        _ip = C.POINTER(C.c_int32)
        self.lib.oracle_ref_build_mesh.restype = C.c_int
        self.lib.oracle_ref_build_mesh.argtypes = [C.c_char_p, _fp, C.c_int32, _ip, _ip, _fp, _ip, C.c_int32, _ip, _ip, C.c_int32]
        rc = self.lib.oracle_ref_build_mesh(obj_path.encode(), _ptr(tris.reshape(-1)), cap_tris, C.byref(nt), C.byref(hn),
                                            _ptr(bounds.reshape(-1)), offs.ctypes.data_as(_ip), cap_boxes, C.byref(nb),
                                            idx.ctypes.data_as(_ip), idx.size)
        if rc != 0:
            raise RuntimeError(f"oracle_ref_build_mesh rc={rc}")
        n, b = nt.value, nb.value
        return dict(tris=tris[:n].copy(), has_normals=bool(hn.value), box_bounds=bounds[:b].copy(),
                    box_offsets=offs[: b + 1].copy(), box_indices=idx[: offs[b]].copy())

    def sphere_intersect(self, org, direction, centre, radius_member):
        o = (C.c_float * 3)(*org)
        d = (C.c_float * 3)(*direction)
        c = (C.c_float * 3)(*centre)
        t = C.c_float(0)
        hit = self.lib.oracle_sphere_intersect(o, d, c, C.c_float(radius_member), C.byref(t))
        return bool(hit), np.float32(t.value)

    def cube_intersect(self, org, direction, c1, c2):
        """cube::intersect: (hit, t) - t is tmin on a hit, tmax otherwise"""
        t = C.c_float(0)
        hit = self.lib.oracle_cube_intersect(_vec(org), _vec(direction), _vec(c1), _vec(c2), C.byref(t))
        _supported(hit)
        return bool(hit), np.float32(t.value)

    def plane_intersect(self, org, direction, pos, normal):
        t = C.c_float(0)
        hit = self.lib.oracle_plane_intersect(_vec(org), _vec(direction), _vec(pos), _vec(normal), C.byref(t))
        _supported(hit)
        return bool(hit), np.float32(t.value)

    def tri_intersect(self, org, direction, tri9):
        """mesh::rayIntersect on the 9 vertex floats: (hit, t, u, v)"""
        t, u, v = C.c_float(0), C.c_float(0), C.c_float(0)
        hit = self.lib.oracle_tri_intersect(_vec(org), _vec(direction), _vec(tri9, 9), C.byref(t), C.byref(u), C.byref(v))
        _supported(hit)
        return bool(hit), np.float32(t.value), np.float32(u.value), np.float32(v.value)

    def rgb_to_int(self, r, g, b) -> int:
        return int(self.lib.oracle_rgb_to_int(int(r), int(g), int(b)))


REF_GPU_SO = os.path.join(ORACLE_DIR, "_ref", "libref_sm100.so")
REF_GPU_FAST_SO = os.path.join(ORACLE_DIR, "_ref", "libref_sm100_fast.so")


class RefGpu:
    """The reference's OWN rayTrace kernel + update() built for sm_100 (oracle/ref_build/make_ref_gpu.py).
    Measurement infrastructure: "reference kernel on B200"."""

    def __init__(self, fast: bool = False):
        path = REF_GPU_FAST_SO if fast else REF_GPU_SO
        if not os.path.isfile(path):
            raise FileNotFoundError(path)
        self.lib = C.CDLL(path)
        self.lib.refgpu_render.restype = C.c_int
        self.lib.refgpu_render.argtypes = [C.POINTER(OracleFrame), _fp, C.c_int, C.c_void_p, _fp, _fp]
        self.fast = fast

    def render(self, scene, cameras, width, height):
        """cameras: list of Camera; returns (last frame u32[H,W], ms per update(), ms per bare kernel)"""
        f = OracleFrame()
        f.width, f.height, f.y0, f.y1, f.y_step = width, height, 0, height, 1
        f.aspect = float(scene.aspect)
        sph = np.ascontiguousarray(scene.spheres, dtype=np.float32)
        lig = np.ascontiguousarray(scene.lights, dtype=np.float32)
        f.n_spheres, f.spheres = sph.shape[0], _ptr(sph.reshape(-1))
        f.n_lights, f.lights = lig.shape[0], _ptr(lig.reshape(-1))
        t, s = scene.texture, scene.sky
        f.tex_w, f.tex_h, f.tex_r, f.tex_g, f.tex_b = t.width, t.height, _ptr(t.r), _ptr(t.g), _ptr(t.b)
        f.sky_w, f.sky_h, f.sky_r, f.sky_g, f.sky_b = s.width, s.height, _ptr(s.r), _ptr(s.g), _ptr(s.b)
        f.sky_size = float(scene.sky_size)
        cams = np.array([[*c.org, c.yaw, c.pitch] for c in cameras], dtype=np.float32)
        px = np.zeros((height, width), dtype=np.uint32)
        a, b = C.c_float(0), C.c_float(0)
        rc = self.lib.refgpu_render(C.byref(f), _ptr(cams.reshape(-1)), len(cameras), px.ctypes.data, C.byref(a), C.byref(b))
        if rc != 0:
            raise RuntimeError(f"refgpu_render rc={rc}")
        return px, float(a.value), float(b.value)


def have_ref_gpu(fast: bool = False) -> bool:
    return os.path.isfile(REF_GPU_FAST_SO if fast else REF_GPU_SO)


def load(which: str = "port") -> Oracle:
    if which == "port":
        return Oracle(build_port())
    if which == "ref":
        if not have_ref():
            raise FileNotFoundError(REF_SO)
        return Oracle(REF_SO)
    if which == "best":
        return load("ref") if have_ref() else load("port")
    raise ValueError(which)
