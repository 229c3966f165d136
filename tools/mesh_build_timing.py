"""Cost of a stream-ordered mesh upload with the flat BVH built on the GPU (ore_set_mesh_device), what it does to an
animated 4K loop, and what refit leaves cost against rebuilt ones after a large deformation.

Prints one JSON line (and writes it to --out when given):
  build:    CUDA-event time per ore_set_mesh_device call on a stream, over back-to-back builds after warm-up, and host
            time to enqueue one call, for the torus of the tests (576 triangles) and height-field grids of about
            20 000, 80 000 and 1 000 000 triangles; beside it the same for ore_set_mesh_triangles_device (the refit of
            the host builder's topology) on the same meshes
  varying:  the same for builds whose triangle count changes on every call (prefixes of a height field, from 1 000 to
            80 000 triangles), with the capacity sized once by the largest: the case of generated geometry
  animated: 4K frames of R(64, 1) plus the torus on an orbit, one frame per iteration on one stream, no host
            synchronisation inside the timed window: (fixed) the mesh never changes, (refit) a torch op deforms the
            triangles, then ore_set_mesh_triangles_device, (rebuild) the same op, then ore_set_mesh_device, (host) the
            same op, the triangles copied to the host, the host builder (ore_build_flat_bvh) and ore_set_mesh
  leaves:   after a large deformation of the torus, the render time (primary + shadow kernels, 4K, 4 orbit cameras) of
            the refit of the undeformed mesh's leaves against the leaves rebuilt for the deformed triangles
The GPU's name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import rte_b200  # noqa: E402
from mesh_update_timing import grid_mesh, torus_mesh  # noqa: E402
from scene_update_timing import gpu_info  # noqa: E402


def host_builder(out_dir):
    """ore_build_flat_bvh of host/ore_mesh.cpp on raw triangles (tests/mesh_build_probe.cpp, built with g++)"""
    import numpy as np
    so = os.path.join(out_dir, "libmesh_build_probe.so")
    env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC",
                           os.path.join(ROOT, "tests", "mesh_build_probe.cpp"),
                           os.path.join(ROOT, "ray-tracer-engine_b200", "host", "ore_mesh.cpp"), "-o", so], env=env)
    lib = C.CDLL(so)
    lib.ore_probe_build_flat_bvh.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int]

    def build(tris):
        n = tris.shape[0]
        bb, offs, idx = np.zeros((1024, 6), np.float32), np.zeros(1025, np.int32), np.zeros(n, np.int32)
        nb = lib.ore_probe_build_flat_bvh(tris.ctypes.data, n, bb.ctypes.data, offs.ctypes.data, idx.ctypes.data, 1024, n)
        return bb[:nb], offs[:nb + 1], idx
    return build


def deformed(base, f, amp=0.35):
    out = base.clone()
    for v in range(3):
        out[:, 3 * v + 1] += amp * (1.3 * base[:, 3 * v] + 0.05 * f).sin()
        out[:, 3 * v] += 0.5 * amp * (0.9 * base[:, 3 * v + 2] + 0.04 * f).cos()
    return out


def event_cost(r, call, reps, warmup, st):
    import torch
    torch.cuda.synchronize()
    for _ in range(warmup):
        call()
    st.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    h0 = time.perf_counter()
    for _ in range(reps):
        call()
    h1 = time.perf_counter()
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / reps, (h1 - h0) * 1e6 / reps


def build_cost(pkg, name, mesh, reps, warmup):
    import torch
    r = pkg.Renderer(0)
    t = torch.from_numpy(mesh.tris.copy()).to("cuda:0")
    st = torch.cuda.Stream()
    r.set_mesh_device(t, True, st.cuda_stream)
    dev_b, host_b = event_cost(r, lambda: r.set_mesh_device(t, True, st.cuda_stream), reps, warmup, st)
    r.set_mesh(mesh)
    dev_r, host_r = event_cost(r, lambda: r.set_mesh_triangles_device(t, st.cuda_stream), reps, warmup, st)
    r.close()
    return {"mesh": name, "n_tris": mesh.n_tris, "n_leaves": mesh.n_boxes, "build_device_us": dev_b,
            "build_enqueue_us_per_call": host_b, "refit_device_us": dev_r, "refit_enqueue_us_per_call": host_r,
            "calls_timed": reps}


def varying_cost(pkg, mesh, reps, warmup):
    """builds of a different triangle count on every call, within the capacity the first (largest) build set"""
    import torch
    r = pkg.Renderer(0)
    t = torch.from_numpy(mesh.tris.copy()).to("cuda:0")
    st = torch.cuda.Stream()
    r.set_mesh_device(t, True, st.cuda_stream)   # sizes the capacity
    counts = [1000 + (79 * k * k + 997 * k) % (mesh.n_tris - 1000) for k in range(reps)]
    views = [t[:c] for c in counts]
    it = iter(range(1 << 30))

    def call():
        r.set_mesh_device(views[next(it) % len(views)], True, st.cuda_stream)
    dev, host = event_cost(r, call, reps, warmup, st)
    r.close()
    return {"capacity_tris": mesh.n_tris, "n_tris_min": min(counts), "n_tris_max": max(counts),
            "distinct_counts": len(set(counts)), "build_device_us": dev, "build_enqueue_us_per_call": host,
            "calls_timed": reps}


def animated(pkg, mode, frames, warmup, build):
    import numpy as np
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
        if mode in ("refit", "rebuild"):
            cur = deformed(base, f)
            if mode == "refit":
                r.set_mesh_triangles_device(cur, st.cuda_stream)
            else:
                r.set_mesh_device(cur, True, st.cuda_stream)
            keep.append(cur)
            del keep[:-4]
        elif mode == "host":
            cur = np.ascontiguousarray(deformed(base, f).cpu().numpy())   # (.cpu() waits for the torch op)
            bb, offs, idx = build(cur)
            r.set_mesh(pkg.scene.Mesh(cur, True, bb, offs, idx))
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


def leaf_quality(pkg, build, amps=(1.0, 3.0)):
    """4K render time of refit leaves (topology of the undeformed torus) against leaves rebuilt for the same triangles"""
    import torch
    W, H = 3840, 2160
    sc = pkg.scene.reference_scene(64, 1)
    sc.mesh = torus_mesh(pkg)
    r = pkg.Renderer(0)
    r.set_scene(sc)
    base = torch.from_numpy(sc.mesh.tris.copy()).to("cuda:0")
    res = []
    for amp in amps:
        cur = deformed(base, 7, amp).contiguous()
        row = {"amplitude": amp}
        for mode in ("refit", "rebuild"):
            if mode == "refit":
                r.set_mesh(sc.mesh)
                r.set_mesh_triangles_device(cur)
            else:
                r.set_mesh_device(cur, True)
            ms = []
            for rep in range(3):
                for k in range(4):
                    r.render(pkg.scene.orbit_camera(sc, 90 * k + 10), W, H)
                    if rep:
                        ms.append(r.kernel_ms()[:3])
            row[mode + "_primary_ms"] = statistics.median(x[1] for x in ms)
            row[mode + "_shadow_ms"] = statistics.median(x[2] for x in ms)
            row[mode + "_total_ms"] = statistics.median(sum(x) for x in ms)
        row["rebuilt_leaves"] = int(r.debug_mesh("n_live")[0])
        res.append(row)
    r.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--frames", type=int, default=120)
    ap.add_argument("--rounds", type=int, default=2, help="the four animated modes, alternated, this many times")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("mesh_build_timing: no CUDA device (nothing here runs without one)")
    pkg = rte_b200.pkg
    pkg.build.build_library()
    with tempfile.TemporaryDirectory() as td:
        build = host_builder(td)
        meshes = [("torus", torus_mesh(pkg)), ("grid_101", grid_mesh(pkg, 101)), ("grid_201", grid_mesh(pkg, 201)),
                  ("grid_708", grid_mesh(pkg, 708))]
        res = {"gpu": gpu_info(), "build": [build_cost(pkg, name, m, args.reps if m.n_tris < 500000 else args.reps // 4,
                                                       args.warmup) for name, m in meshes],
               "varying": varying_cost(pkg, meshes[2][1], args.reps, args.warmup), "animated": []}
        for _ in range(args.rounds):
            for mode in ("fixed", "refit", "rebuild", "host"):
                res["animated"].append(animated(pkg, mode, args.frames, 10, build))
        res["leaves"] = leaf_quality(pkg, build)
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
