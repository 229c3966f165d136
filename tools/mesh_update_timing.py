"""Cost of a stream-ordered triangle update (ore_set_mesh_triangles_device) and what it does to an animated 4K loop.

Prints one JSON line (and writes it to --out when given):
  update:   CUDA-event time per ore_set_mesh_triangles_device call on a stream, over back-to-back updates after warm-up,
            and host time to enqueue one call, for the torus of the tests (576 triangles) and height-field grids of
            about 20 000 and 80 000 triangles (leaf topology from the reference builder's transcription in host/)
  animated: 4K frames of R(64, 1) plus the torus on an orbit, one frame per iteration on one stream with no host
            synchronisation inside the timed window - (fixed) the mesh never changes, (device) a torch op deforms the
            triangles then ore_set_mesh_triangles_device, (host) the same torch op, the triangles copied to the host and
            ore_set_mesh with the topology's boxes (the host path without recomputing any box: a lower bound of its
            cost); Mrays/s (primary rays) of each
The GPU's name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rte_b200  # noqa: E402
from scene_update_timing import gpu_info  # noqa: E402

HOST = os.path.join(ROOT, "ray-tracer-engine_b200", "host")


def grid_mesh(pkg, n):
    """(n-1)^2 * 2 triangles of a bumpy height field, loaded and split into leaves by host/ore_mesh.cpp"""
    import numpy as np
    subprocess.check_call(["make", "-s", "-C", HOST, "libore_host.so"])
    lib = C.CDLL(os.path.join(HOST, "libore_host.so"), mode=os.RTLD_LAZY)
    hgt = np.random.default_rng(3).uniform(0, 1.5, size=(n, n))
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "grid.obj")
        with open(path, "w") as fh:
            for i in range(n):
                for j in range(n):
                    fh.write("v %.5f %.5f %.5f\n" % (1 + 8.0 * i / n, 2 + hgt[i, j], 1 + 8.0 * j / n))
            for i in range(n - 1):
                for j in range(n - 1):
                    a, b, c, d = i * n + j + 1, (i + 1) * n + j + 1, (i + 1) * n + j + 2, i * n + j + 2
                    fh.write("f %d %d %d\nf %d %d %d\n" % (a, b, c, a, c, d))
        cap = 2 * n * n
        tris = np.zeros((cap, 27), np.float32)
        bounds = np.zeros((4096, 6), np.float32)
        offs = np.zeros(4097, np.int32)
        idx = np.zeros(2 * cap, np.int32)
        nt, hn, nb = C.c_int(0), C.c_int(0), C.c_int(0)
        fp, ip = C.POINTER(C.c_float), C.POINTER(C.c_int)
        lib.ore_host_build_mesh.argtypes = [C.c_char_p, fp, C.c_int, ip, ip, fp, ip, C.c_int, ip, ip, C.c_int]
        rc = lib.ore_host_build_mesh(path.encode(), tris.ctypes.data_as(fp), cap, C.byref(nt), C.byref(hn),
                                     bounds.ctypes.data_as(fp), offs.ctypes.data_as(ip), 4096, C.byref(nb),
                                     idx.ctypes.data_as(ip), idx.size)
    if rc:
        raise SystemExit(f"mesh_update_timing: ore_host_build_mesh failed for a {n} x {n} grid")
    t, b = nt.value, nb.value
    return pkg.scene.Mesh.from_arrays(dict(tris=tris[:t], has_normals=hn.value, box_bounds=bounds[:b],
                                           box_offsets=offs[:b + 1], box_indices=idx[:offs[b]]))


def torus_mesh(pkg):
    import numpy as np
    return pkg.scene.Mesh.from_arrays(np.load(os.path.join(ROOT, "tests", "golden", "mesh_torus.npz")))


def deformed(base, f):
    out = base.clone()
    for v in range(3):
        out[:, 3 * v + 1] += 0.35 * (1.3 * base[:, 3 * v] + 0.05 * f).sin()
    return out


def update_cost(pkg, name, mesh, reps, warmup):
    import torch
    r = pkg.Renderer(0)
    r.set_mesh(mesh)
    t = torch.from_numpy(mesh.tris.copy()).to("cuda:0")
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    for _ in range(warmup):
        r.set_mesh_triangles_device(t, st.cuda_stream)
    st.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    h0 = time.perf_counter()
    for _ in range(reps):
        r.set_mesh_triangles_device(t, st.cuda_stream)
    h1 = time.perf_counter()
    b.record(st)
    b.synchronize()
    dev_us = a.elapsed_time(b) * 1e3 / reps
    host_ms = []
    for k in range(warmup + 20):
        t0 = time.perf_counter()
        r.set_mesh(mesh)
        if k >= warmup:
            host_ms.append((time.perf_counter() - t0) * 1e3)
    r.close()
    host_ms.sort()
    return {"mesh": name, "n_tris": mesh.n_tris, "n_boxes": mesh.n_boxes, "device_update_us": dev_us,
            "enqueue_us_per_call": (h1 - h0) * 1e6 / reps, "set_mesh_ms_median": host_ms[len(host_ms) // 2],
            "updates_timed": reps}


def animated(pkg, mode, frames, warmup):
    import torch
    W, H = 3840, 2160
    sc = pkg.scene.reference_scene(64, 1)
    sc.mesh = torus_mesh(pkg)
    m = sc.mesh
    r = pkg.Renderer(0)
    r.set_scene(sc)
    F = pkg.capi
    base = torch.from_numpy(m.tris.copy()).to("cuda:0")
    out = torch.zeros((2, H, W), dtype=torch.int32, device="cuda:0")
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    keep = []

    def frame(f):
        if mode == "device":
            cur = deformed(base, f)
            r.set_mesh_triangles_device(cur, st.cuda_stream)
            keep.append(cur)
            del keep[:-4]
        elif mode == "host":
            cur = deformed(base, f).cpu().numpy()   # (.cpu() waits for the torch op; the setter synchronises)
            r.set_mesh(pkg.scene.Mesh(cur, m.has_normals, m.box_bounds, m.box_offsets, m.box_indices))
        r.render_device(pkg.scene.orbit_camera(sc, f), W, H, out[f & 1].data_ptr(), stream=st.cuda_stream,
                        flags=F.ORE_FLAG_NO_KERNEL_TIMING)

    with torch.cuda.stream(st):
        for f in range(warmup):
            frame(f)
        st.synchronize()
        h0 = time.perf_counter()
        a.record(st)
        for f in range(warmup, warmup + frames):
            frame(f)
        b.record(st)
        b.synchronize()
        wall = time.perf_counter() - h0
    ms = a.elapsed_time(b)
    r.close()
    return {"mode": mode, "frames": frames, "ms_per_frame_events": ms / frames, "ms_per_frame_wall": wall * 1e3 / frames,
            "mrays_per_s": W * H * frames / (wall * 1e3) / 1e3, "workload": "3840x2160 R(64,1) + torus (576 triangles)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--frames", type=int, default=120)
    ap.add_argument("--rounds", type=int, default=2, help="the three animated modes, alternated, this many times")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mesh_update_timing: no CUDA device (nothing here runs without one)")
    pkg = rte_b200.pkg
    pkg.build.build_library()
    meshes = [("torus", torus_mesh(pkg)), ("grid_101", grid_mesh(pkg, 101)), ("grid_201", grid_mesh(pkg, 201))]
    res = {"gpu": gpu_info(), "update": [update_cost(pkg, name, m, args.reps, args.warmup) for name, m in meshes],
           "animated": []}
    for _ in range(args.rounds):
        for mode in ("fixed", "device", "host"):
            res["animated"].append(animated(pkg, mode, args.frames, 10))
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
