"""ctypes binding of the C ABI in include/ore_render.h (libore_b200.so).

This is the only way Python reaches the render path: plain pointers and sizes, exactly the
calls a C/C++ host makes.  There is no CPU fallback - if the library is missing or no
sm_100 device is usable, construction fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

ORE_FLAG_EXHAUSTIVE = 1
ORE_FLAG_COUNT_REFERENCE_TESTS = 2
ORE_FLAG_FAST_LIBM = 16
ORE_FLAG_FUSED_SHADOW = 32
ORE_FLAG_NO_KERNEL_TIMING = 64
ORE_FLAG_BAND_DMA = 128

EXPORTS = [
    "ore_create", "ore_destroy", "ore_abi_version", "ore_last_error",
    "ore_set_spheres", "ore_set_spheres_aos32", "ore_set_cubes", "ore_set_planes", "ore_set_mesh", "ore_set_lights", "ore_set_texture", "ore_set_sky",
    "ore_render", "ore_render_device", "ore_synchronize",
    "ore_get_hits", "ore_get_counters", "ore_get_kernel_ms", "ore_measure_fp32_peak", "ore_debug_libm",
    "ore_render_async", "ore_wait", "ore_host_alloc", "ore_host_free",
    "ore_dev_alloc", "ore_dev_free", "ore_ipc_export", "ore_ipc_import", "ore_ipc_close", "ore_copy_to_host",
    "ore_render_async_signal", "ore_host_register", "ore_host_unregister", "ore_flag_write", "ore_flag_wait_geq",
    "ore_flag_write_after", "ore_get_stream", "ore_render_batch_device", "ore_render_batch_async",
    "ore_set_spheres_device", "ore_debug_sphere_tree", "ore_set_mesh_triangles_device", "ore_debug_mesh",
    "ore_set_mesh_device",
]

# ore_debug_sphere_tree: which array of the sphere hierarchy, and its element type
SPHERE_TREE_ARRAYS = {"sph_exact": 0, "sph_xsort": 1, "sph_sort": 2, "sort_index": 3, "leaf_sph": 4, "super_sph": 5}


# ore_debug_mesh: which array of the mesh
MESH_ARRAYS = {"tris": 0, "boxes": 1, "box_sph": 2, "box_offsets": 3, "box_indices": 4, "n_live": 5}

# leaves of a mesh built on the device (ore_set_mesh_device) hold this many at most
MESH_MAX_LEAVES = 1024


def sphere_tree_lengths(n: int) -> dict:
    """item counts of the six hierarchy arrays for n spheres (include/ore_render.h, ore_debug_sphere_tree)"""
    n_sort = max(1, (n + 31) // 32) * 32
    n_leaf = (n + 7) // 8
    n_sup = (n_leaf + 31) // 32
    return {"sph_exact": max(n, 1), "sph_xsort": n_sort, "sph_sort": n_sort, "sort_index": n_sort,
            "leaf_sph": (n_leaf + 31) // 32 * 32, "super_sph": (n_sup + 3) // 4 * 4}


class OreCamera(C.Structure):
    _fields_ = [("org", C.c_float * 3), ("dir", C.c_float * 3), ("aspect", C.c_float),
                ("yaw", C.c_float), ("pitch", C.c_float)]


class OreFrame(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("y0", C.c_int32), ("y1", C.c_int32),
                ("y_step", C.c_int32), ("aspect", C.c_float), ("flags", C.c_uint32), ("out_pitch", C.c_int32), ("y_block", C.c_int32)]


class OreCounters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "pixels", "hit_pixels", "primary_tests", "shadow_tests_ref", "sky_tests",
        "exact_primary", "exact_shadow", "kernel_launches", "beam_l1", "beam_l2", "primary_steps", "sweep_steps", "sky_exact")]


class OreError(RuntimeError):
    pass


_lib = None


def load_library(path: str | None = None) -> C.CDLL:
    """Load libore_b200.so; raise if it is absent (never falls back to anything else)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or os.environ.get("ORE_LIB") or _build.LIB_PATH
    if not os.path.isfile(path):
        raise OreError(f"{path} not built - run `python -c 'import __graft_entry__ as g; g.build()'`")
    lib = C.CDLL(path)
    vp, fp, i32 = C.c_void_p, C.POINTER(C.c_float), C.c_int32
    lib.ore_create.argtypes = [C.POINTER(vp), C.c_int]
    lib.ore_destroy.argtypes = [vp]
    lib.ore_abi_version.argtypes = []
    lib.ore_last_error.argtypes = [vp]
    lib.ore_last_error.restype = C.c_char_p
    lib.ore_set_spheres.argtypes = [vp, fp, i32]
    lib.ore_set_spheres_aos32.argtypes = [vp, vp, i32]
    lib.ore_set_spheres_device.argtypes = [vp, vp, i32, vp]
    lib.ore_debug_sphere_tree.argtypes = [vp, i32, vp, i32]
    lib.ore_set_lights.argtypes = [vp, fp, i32]
    lib.ore_set_cubes.argtypes = [vp, fp, i32]
    lib.ore_set_planes.argtypes = [vp, fp, i32]
    ip = C.POINTER(C.c_int32)
    lib.ore_set_mesh.argtypes = [vp, fp, i32, i32, fp, ip, ip, i32]
    lib.ore_set_mesh_triangles_device.argtypes = [vp, vp, i32, vp]
    lib.ore_set_mesh_device.argtypes = [vp, vp, i32, i32, vp]
    lib.ore_debug_mesh.argtypes = [vp, i32, vp, i32]
    lib.ore_set_texture.argtypes = [vp, fp, fp, fp, i32, i32]
    lib.ore_set_sky.argtypes = [vp, fp, fp, fp, i32, i32, C.c_float]
    lib.ore_render.argtypes = [vp, C.POINTER(OreCamera), C.POINTER(OreFrame), vp]
    lib.ore_render_device.argtypes = [vp, C.POINTER(OreCamera), C.POINTER(OreFrame), vp, vp]
    lib.ore_synchronize.argtypes = [vp]
    lib.ore_render_async.argtypes = [vp, C.POINTER(OreCamera), C.POINTER(OreFrame), vp]
    lib.ore_wait.argtypes = [vp]
    lib.ore_host_alloc.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
    lib.ore_host_free.argtypes = [vp, vp]
    lib.ore_get_hits.argtypes = [vp, vp, vp]
    lib.ore_get_counters.argtypes = [vp, C.POINTER(OreCounters)]
    lib.ore_get_kernel_ms.argtypes = [vp, C.POINTER(C.c_float * 4)]
    lib.ore_measure_fp32_peak.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.ore_debug_libm.argtypes = [vp, C.c_int, C.c_int, fp, fp, fp]
    lib.ore_dev_alloc.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
    lib.ore_dev_free.argtypes = [vp, vp]
    lib.ore_ipc_export.argtypes = [vp, vp, C.POINTER(C.c_ubyte * 64)]
    lib.ore_ipc_import.argtypes = [vp, C.POINTER(C.c_ubyte * 64), C.POINTER(vp)]
    lib.ore_ipc_close.argtypes = [vp, vp]
    lib.ore_copy_to_host.argtypes = [vp, vp, vp, C.c_size_t]
    lib.ore_render_async_signal.argtypes = [vp, C.POINTER(OreCamera), C.POINTER(OreFrame), vp, vp, C.c_uint32]
    lib.ore_host_register.argtypes = [vp, vp, C.c_size_t]
    lib.ore_host_unregister.argtypes = [vp, vp]
    lib.ore_flag_write.argtypes = [vp, vp, vp, C.c_uint32]
    lib.ore_flag_wait_geq.argtypes = [vp, vp, vp, C.c_uint32]
    lib.ore_flag_write_after.argtypes = [vp, vp, vp, C.c_uint32]
    lib.ore_render_batch_device.argtypes = [vp, C.POINTER(OreCamera), i32, C.POINTER(OreFrame), C.POINTER(vp), vp]
    lib.ore_render_batch_async.argtypes = [vp, C.POINTER(OreCamera), i32, C.POINTER(OreFrame), C.POINTER(vp), vp, C.c_uint32]
    lib.ore_get_stream.argtypes = [vp, C.c_int]
    lib.ore_get_stream.restype = vp
    for name in EXPORTS:
        if name not in ("ore_last_error", "ore_get_stream"):
            getattr(lib, name).restype = C.c_int
    if path == _build.LIB_PATH:
        _lib = lib
    return lib


def _fptr(a: np.ndarray):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _stream(stream: int):
    """a raw cudaStream_t for the ABI; 0 = the context's render stream"""
    return C.c_void_p(stream) if stream else None


class Renderer:
    """One render context on one GPU (mirrors the reference's global scene + update())."""

    def __init__(self, device: int = 0, lib: C.CDLL | None = None):
        self.lib = lib or load_library()
        self.ctx = C.c_void_p()
        rc = self.lib.ore_create(C.byref(self.ctx), int(device))
        if rc != 0:
            msg = self.lib.ore_last_error(self.ctx).decode() if self.ctx else "allocation failed"
            if self.ctx:
                self.lib.ore_destroy(self.ctx)
                self.ctx = C.c_void_p()
            raise OreError(f"ore_create(device={device}) failed rc={rc}: {msg}")
        self.device = device
        self.scene = None

    def _check(self, rc, what):
        if rc != 0:
            raise OreError(f"{what} failed rc={rc}: {self.lib.ore_last_error(self.ctx).decode()}")

    def _device_tensor(self, t, what: str, cols: int, rows: int | None = None, min_rows: int = 0) -> int:
        """the argument checks of a stream-ordered setter: a contiguous torch float32 tensor of shape (n, cols) on this
        context's GPU with n == rows (or n >= min_rows); returns n"""
        import torch
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"{what}: expected a torch.Tensor, got {type(t).__name__}")
        if t.dtype != torch.float32:
            raise TypeError(f"{what}: expected dtype torch.float32, got {t.dtype}")
        if t.dim() != 2 or t.shape[1] != cols or (t.shape[0] != rows if rows is not None else t.shape[0] < min_rows):
            want = f"({rows}, {cols})" if rows is not None else f"(n, {cols})" + (f" with n >= {min_rows}" if min_rows else "")
            raise ValueError(f"{what}: expected shape {want}, got {tuple(t.shape)}")
        if t.device.type != "cuda" or t.device.index != self.device:
            raise ValueError(f"{what}: the tensor must live on cuda:{self.device}, not {t.device}")
        if not t.is_contiguous():
            raise ValueError(f"{what}: the tensor must be contiguous")
        return int(t.shape[0])

    def close(self):
        if self.ctx:
            self.lib.ore_destroy(self.ctx)
            self.ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- scene ----
    def set_spheres(self, xyz_radius: np.ndarray):
        a = np.ascontiguousarray(xyz_radius, dtype=np.float32).reshape(-1, 4)
        self._check(self.lib.ore_set_spheres(self.ctx, _fptr(a.reshape(-1)) if a.size else None, a.shape[0]), "ore_set_spheres")

    def set_spheres_aos32(self, records: np.ndarray):
        a = np.ascontiguousarray(records)
        assert a.nbytes % 32 == 0
        self._check(self.lib.ore_set_spheres_aos32(self.ctx, a.ctypes.data, a.nbytes // 32), "ore_set_spheres_aos32")

    def set_spheres_device(self, t, stream: int = 0):
        """Stream-ordered sphere update from a torch CUDA float32 tensor of shape (n, 4) (cx, cy, cz, radius member) on
        this context's GPU.  `stream`: a raw cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream; 0 = the
        context's render stream).  Keep `t` alive and unchanged until the update has run on that stream."""
        n = self._device_tensor(t, "set_spheres_device", 4)
        self._check(self.lib.ore_set_spheres_device(self.ctx, C.c_void_p(t.data_ptr()) if n else None, n, _stream(stream)),
                    "ore_set_spheres_device")

    def debug_sphere_tree(self, which: str, n: int) -> np.ndarray:
        """one array of the sphere hierarchy of the current n-sphere scene, read back after a device synchronise
        (tests): float32 (len, 4), or int32 (len,) for sort_index"""
        length = sphere_tree_lengths(n)[which]
        out = np.zeros(length, np.int32) if which == "sort_index" else np.zeros((length, 4), np.float32)
        self._check(self.lib.ore_debug_sphere_tree(self.ctx, SPHERE_TREE_ARRAYS[which], out.ctypes.data if length else None,
                                                   length), "ore_debug_sphere_tree")
        return out

    def set_cubes(self, c1_c2: np.ndarray):
        a = np.ascontiguousarray(c1_c2, dtype=np.float32).reshape(-1, 6)
        self._check(self.lib.ore_set_cubes(self.ctx, _fptr(a.reshape(-1)) if a.size else None, a.shape[0]), "ore_set_cubes")

    def set_planes(self, pos_normal: np.ndarray):
        a = np.ascontiguousarray(pos_normal, dtype=np.float32).reshape(-1, 6)
        self._check(self.lib.ore_set_planes(self.ctx, _fptr(a.reshape(-1)) if a.size else None, a.shape[0]), "ore_set_planes")

    def set_mesh(self, mesh):
        """mesh: scene.Mesh (triangles + flat BVH as the reference holds them) or None"""
        ip = C.POINTER(C.c_int32)
        if mesh is None or mesh.n_tris == 0:
            self._check(self.lib.ore_set_mesh(self.ctx, None, 0, 0, None, None, None, 0), "ore_set_mesh")
            self._mesh_counts = (0, 0)
            self._mesh_n_idx = 0
            return
        self._check(self.lib.ore_set_mesh(self.ctx, _fptr(mesh.tris.reshape(-1)), mesh.n_tris, int(mesh.has_normals),
                                          _fptr(mesh.box_bounds.reshape(-1)), mesh.box_offsets.ctypes.data_as(ip),
                                          mesh.box_indices.ctypes.data_as(ip), mesh.n_boxes), "ore_set_mesh")
        self._mesh_counts = (mesh.n_tris, mesh.n_boxes) if mesh.n_boxes else (0, 0)   # (no leaves: no mesh)
        self._mesh_n_idx = int(mesh.box_offsets[mesh.n_boxes]) if mesh.n_boxes else 0

    def set_mesh_device(self, t, has_normals: bool, stream: int = 0):
        """Stream-ordered replacement of the whole mesh from a torch CUDA float32 tensor of shape (n_tris, 27), n_tris >= 1
        (the records of set_mesh) on this context's GPU, with the reference's flat BVH built on the GPU: the leaves
        equal the host builder's bit for bit.  `stream`: a raw cudaStream_t (0 = the context's render stream).  Keep `t`
        alive and unchanged until the update has run on that stream."""
        n = self._device_tensor(t, "set_mesh_device", 27, min_rows=1)
        self._check(self.lib.ore_set_mesh_device(self.ctx, C.c_void_p(t.data_ptr()), n, int(bool(has_normals)), _stream(stream)),
                    "ore_set_mesh_device")
        self._mesh_counts = (n, min(MESH_MAX_LEAVES, n))   # (leaf capacity: the live count is on the device)
        self._mesh_n_idx = n

    def set_mesh_triangles_device(self, t, stream: int = 0):
        """Stream-ordered update of the mesh's triangles from a torch CUDA float32 tensor of shape (n_tris, 27) (the
        records of set_mesh) on this context's GPU; the leaf boxes and their spheres are recomputed on the GPU and the
        topology of the last set_mesh stays.  `stream`: a raw cudaStream_t (0 = the context's render stream).  Keep `t`
        alive and unchanged until the update has run on that stream."""
        n_tris = self._device_tensor(t, "set_mesh_triangles_device", 27, rows=getattr(self, "_mesh_counts", (0, 0))[0])
        self._check(self.lib.ore_set_mesh_triangles_device(self.ctx, C.c_void_p(t.data_ptr()), n_tris, _stream(stream)),
                    "ore_set_mesh_triangles_device")

    def debug_mesh(self, which: str) -> np.ndarray:
        """one array of the current mesh, read back after a device synchronise (tests): tris float32 (n_tris, 27), boxes
        float32 (2 * n_boxes, 4) (lo, hi per leaf), box_sph float32 (n_boxes, 4), box_offsets int32 (n_boxes + 1,),
        box_indices int32 (n_idx,), n_live int32 (1,) (the live leaf count); n_boxes is the leaf capacity after
        set_mesh_device"""
        n_tris, n_boxes = getattr(self, "_mesh_counts", (0, 0))
        n_idx = getattr(self, "_mesh_n_idx", 0)
        out = {"tris": lambda: np.zeros((n_tris, 27), np.float32), "boxes": lambda: np.zeros((2 * n_boxes, 4), np.float32),
               "box_sph": lambda: np.zeros((n_boxes, 4), np.float32), "box_offsets": lambda: np.zeros(n_boxes + 1, np.int32),
               "box_indices": lambda: np.zeros(n_idx, np.int32), "n_live": lambda: np.zeros(1, np.int32)}[which]()
        self._check(self.lib.ore_debug_mesh(self.ctx, MESH_ARRAYS[which], out.ctypes.data if out.size else None,
                                            out.size if which == "tris" else out.shape[0]), "ore_debug_mesh")
        return out

    def set_lights(self, lights7: np.ndarray):
        a = np.ascontiguousarray(lights7, dtype=np.float32).reshape(-1, 7)
        self._check(self.lib.ore_set_lights(self.ctx, _fptr(a.reshape(-1)) if a.size else None, a.shape[0]), "ore_set_lights")

    def set_texture(self, sprite):
        self._check(self.lib.ore_set_texture(self.ctx, _fptr(sprite.r), _fptr(sprite.g), _fptr(sprite.b),
                                             sprite.width, sprite.height), "ore_set_texture")

    def set_sky(self, sprite, size: float):
        self._check(self.lib.ore_set_sky(self.ctx, _fptr(sprite.r), _fptr(sprite.g), _fptr(sprite.b),
                                         sprite.width, sprite.height, float(size)), "ore_set_sky")

    def set_scene(self, scene, n_lights: int | None = None):
        self.set_spheres(scene.spheres)
        lights = scene.lights if n_lights is None else scene.lights[:n_lights]
        self.set_lights(lights)
        self.set_texture(scene.texture)
        self.set_sky(scene.sky, scene.sky_size)
        self.set_cubes(getattr(scene, "cubes", np.zeros((0, 6), np.float32)))
        self.set_planes(getattr(scene, "planes", np.zeros((0, 6), np.float32)))
        self.set_mesh(getattr(scene, "mesh", None))
        self.scene = scene

    # ---- render ----
    @staticmethod
    def _cam(camera) -> OreCamera:
        c = OreCamera()
        c.org = (C.c_float * 3)(*[float(v) for v in camera.org])
        c.dir = (C.c_float * 3)(0.0, 0.0, 1.0)
        c.aspect = 0.0
        c.yaw, c.pitch = float(camera.yaw), float(camera.pitch)
        return c

    def _frame(self, width, height, y0, y1, y_step, aspect, flags, out_pitch=0, y_block=1) -> OreFrame:
        f = OreFrame()
        f.out_pitch = int(out_pitch)
        f.y_block = int(y_block)
        f.width, f.height = int(width), int(height)
        f.y0, f.y1, f.y_step = int(y0), int(height if y1 is None else y1), int(y_step)
        f.aspect = float(self.scene.aspect if aspect is None else aspect)
        f.flags = int(flags)
        return f

    @staticmethod
    def rows(height, y0=0, y1=None, y_step=1, y_block=1) -> int:
        y1 = height if y1 is None else y1
        span = y1 - y0
        if span <= 0:
            return 0
        if y_block >= y_step:
            return span
        return (span // y_step) * y_block + min(span % y_step, y_block)

    def render(self, camera, width, height, y0=0, y1=None, y_step=1, aspect=None, flags=0, out=None, y_block=1) -> np.ndarray:
        """Render into HOST memory (device->host copy inside the call). Returns uint32 [rows, W]."""
        f = self._frame(width, height, y0, y1, y_step, aspect, flags, 0, y_block)
        rows = self.rows(height, y0, y1, y_step, y_block)
        if out is None:
            out = np.empty((rows, max(0, width)), dtype=np.uint32)
        assert out.dtype == np.uint32 and out.size == rows * width and out.flags["C_CONTIGUOUS"]
        cam = self._cam(camera)
        dummy = C.c_uint32(0)  # an empty band still goes through the ABI's argument checks
        ptr = out.ctypes.data if out.size else C.addressof(dummy)
        self._check(self.lib.ore_render(self.ctx, C.byref(cam), C.byref(f), ptr), "ore_render")
        return out

    def render_device(self, camera, width, height, out_ptr: int, stream: int = 0, y0=0, y1=None, y_step=1,
                      aspect=None, flags=0, out_pitch=0, y_block=1):
        """Render into DEVICE memory at `out_ptr` (asynchronous on `stream`)."""
        f = self._frame(width, height, y0, y1, y_step, aspect, flags, out_pitch, y_block)
        cam = self._cam(camera)
        self._check(self.lib.ore_render_device(self.ctx, C.byref(cam), C.byref(f), C.c_void_p(out_ptr), _stream(stream)),
                    "ore_render_device")

    # ---- batches of frames (one launch set for several cameras) ----
    def _cams(self, cameras):
        arr = (OreCamera * len(cameras))()
        for i, c in enumerate(cameras):
            arr[i] = self._cam(c)
        return arr

    def render_batch_device(self, cameras, width, height, out_ptrs, stream: int = 0, y0=0, y1=None, y_step=1, aspect=None,
                            flags=0, out_pitch=0, y_block=1):
        """frames of `cameras` into the device framebuffers `out_ptrs` (same band arguments for all), one launch set"""
        assert len(cameras) == len(out_ptrs)
        f = self._frame(width, height, y0, y1, y_step, aspect, flags, out_pitch, y_block)
        ptrs = (C.c_void_p * len(out_ptrs))(*[int(p) for p in out_ptrs])
        self._check(self.lib.ore_render_batch_device(self.ctx, self._cams(cameras), len(cameras), C.byref(f), ptrs,
                                                     _stream(stream)), "ore_render_batch_device")

    def render_batch_async(self, cameras, width, height, outs, y0=0, y1=None, y_step=1, aspect=None, flags=0, y_block=1,
                           in_place=False, done_flag: int = 0, first_done_value: int = 0):
        """pipelined render + device->host copy of a batch; outs: host addresses (int) or numpy arrays, one per frame"""
        assert len(cameras) == len(outs)
        f = self._frame(width, height, y0, y1, y_step, aspect, flags, width if in_place else 0, y_block)
        ptrs = (C.c_void_p * len(outs))(*[(o if isinstance(o, int) else o.ctypes.data) for o in outs])
        self._check(self.lib.ore_render_batch_async(self.ctx, self._cams(cameras), len(cameras), C.byref(f), ptrs,
                                                    C.c_void_p(done_flag) if done_flag else None, int(first_done_value)),
                    "ore_render_batch_async")

    # ---- device buffers / IPC (multi-GPU presentation) ----
    def dev_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self._check(self.lib.ore_dev_alloc(self.ctx, nbytes, C.byref(p)), "ore_dev_alloc")
        return int(p.value)

    def dev_free(self, ptr: int):
        self._check(self.lib.ore_dev_free(self.ctx, C.c_void_p(ptr)), "ore_dev_free")

    def ipc_export(self, ptr: int) -> bytes:
        h = (C.c_ubyte * 64)()
        self._check(self.lib.ore_ipc_export(self.ctx, C.c_void_p(ptr), C.byref(h)), "ore_ipc_export")
        return bytes(h)

    def ipc_import(self, handle: bytes) -> int:
        h = (C.c_ubyte * 64)(*handle)
        p = C.c_void_p()
        self._check(self.lib.ore_ipc_import(self.ctx, C.byref(h), C.byref(p)), "ore_ipc_import")
        return int(p.value)

    def ipc_close(self, ptr: int):
        self._check(self.lib.ore_ipc_close(self.ctx, C.c_void_p(ptr)), "ore_ipc_close")

    def copy_to_host(self, host: np.ndarray, dev_ptr: int):
        assert host.flags["C_CONTIGUOUS"]
        self._check(self.lib.ore_copy_to_host(self.ctx, host.ctypes.data, C.c_void_p(dev_ptr), host.nbytes), "ore_copy_to_host")

    # ---- pipelined presentation ----
    def host_alloc(self, shape, dtype=np.uint32) -> np.ndarray:
        """numpy view of pinned host memory allocated through the ABI (freed with host_free)."""
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        self._check(self.lib.ore_host_alloc(self.ctx, n, C.byref(p)), "ore_host_alloc")
        buf = (C.c_ubyte * n).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype).reshape(shape)
        self._pinned = getattr(self, "_pinned", {})
        self._pinned[arr.ctypes.data] = p.value
        return arr

    def host_free(self, arr: np.ndarray):
        p = getattr(self, "_pinned", {}).pop(arr.ctypes.data, None)
        if p is not None:
            self._check(self.lib.ore_host_free(self.ctx, C.c_void_p(p)), "ore_host_free")

    def render_async(self, camera, width, height, out, y0=0, y1=None, y_step=1, aspect=None, flags=0, y_block=1,
                     in_place=False, done_flag: int = 0, done_value: int = 0):
        """Pipelined render + device->host copy.  `out`: numpy array (packed band) or, with in_place=True, the address
        (int) / array of image row y0 inside a FULL host frame.  done_flag: address of a 32-bit flag written with
        done_value once the copy has landed (0 = none)."""
        f = self._frame(width, height, y0, y1, y_step, aspect, flags, width if in_place else 0, y_block)
        cam = self._cam(camera)
        ptr = out if isinstance(out, int) else out.ctypes.data
        if done_flag:
            self._check(self.lib.ore_render_async_signal(self.ctx, C.byref(cam), C.byref(f), C.c_void_p(ptr),
                                                         C.c_void_p(done_flag), int(done_value)), "ore_render_async_signal")
        else:
            self._check(self.lib.ore_render_async(self.ctx, C.byref(cam), C.byref(f), C.c_void_p(ptr)), "ore_render_async")

    # ---- stream-ordered flags / registered host memory (multi-GPU presentation) ----
    def host_register(self, ptr: int, nbytes: int):
        self._check(self.lib.ore_host_register(self.ctx, C.c_void_p(ptr), nbytes), "ore_host_register")

    def host_unregister(self, ptr: int):
        self._check(self.lib.ore_host_unregister(self.ctx, C.c_void_p(ptr)), "ore_host_unregister")

    def stream_handle(self, which: int = 0) -> int:
        return int(self.lib.ore_get_stream(self.ctx, which) or 0)

    def flag_write(self, flag_ptr: int, value: int, stream: int = 0):
        self._check(self.lib.ore_flag_write(self.ctx, _stream(stream), C.c_void_p(flag_ptr), int(value) & 0xffffffff),
                    "ore_flag_write")

    def flag_write_after(self, flag_ptr: int, value: int, stream: int = 0):
        """ordered variant: issued from this context's signal stream once `stream`'s work so far is complete"""
        self._check(self.lib.ore_flag_write_after(self.ctx, _stream(stream), C.c_void_p(flag_ptr),
                                                  int(value) & 0xffffffff), "ore_flag_write_after")

    def flag_wait_geq(self, flag_ptr: int, value: int, stream: int = 0):
        self._check(self.lib.ore_flag_wait_geq(self.ctx, _stream(stream), C.c_void_p(flag_ptr), int(value) & 0xffffffff),
                    "ore_flag_wait_geq")

    def wait(self):
        self._check(self.lib.ore_wait(self.ctx), "ore_wait")

    def synchronize(self):
        self._check(self.lib.ore_synchronize(self.ctx), "ore_synchronize")

    def hits(self, rows, width):
        ids = np.empty((rows, width), dtype=np.int32)
        t = np.empty((rows, width), dtype=np.float32)
        self._check(self.lib.ore_get_hits(self.ctx, ids.ctypes.data, t.ctypes.data), "ore_get_hits")
        return ids, t

    def counters(self) -> dict:
        c = OreCounters()
        self._check(self.lib.ore_get_counters(self.ctx, C.byref(c)), "ore_get_counters")
        return {n: int(getattr(c, n)) for n, _ in OreCounters._fields_}

    def measure_fp32_peak(self):
        """FFMA-burn FP32 peak of this GPU in TFLOP/s and the nominal SM clock in MHz."""
        tf, mhz = C.c_double(0), C.c_double(0)
        self._check(self.lib.ore_measure_fp32_peak(self.ctx, C.byref(tf), C.byref(mhz)), "ore_measure_fp32_peak")
        return tf.value, mhz.value

    def debug_libm(self, op: str, a: np.ndarray, b: np.ndarray | None = None) -> np.ndarray:
        """device libm of the path on host inputs (tests): op in cosf, sinf, acosf, atan2f(a=y, b=x)"""
        code = {"cosf": 0, "sinf": 1, "acosf": 2, "atan2f": 3, "normalise_x": 4, "normalise_y": 5, "normalise_z": 6}[op]
        a = np.ascontiguousarray(a, dtype=np.float32)
        b = np.ascontiguousarray(a if b is None else b, dtype=np.float32)
        out = np.empty_like(a)
        self._check(self.lib.ore_debug_libm(self.ctx, code, a.size, _fptr(a), _fptr(b), _fptr(out)), "ore_debug_libm")
        return out

    def kernel_ms(self):
        ms = (C.c_float * 4)()
        self._check(self.lib.ore_get_kernel_ms(self.ctx, C.byref(ms)), "ore_get_kernel_ms")
        return [float(v) for v in ms]
