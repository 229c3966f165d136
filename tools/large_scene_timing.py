"""Cost of large sphere scenes: 4K frames at scene.scaled_scene's density from 65 536 spheres (the three-level path)
through 131 072, 1M and 4M to 2^24 = 16 777 216 spheres (the large-scene path, hyper-clusters of 8192 spheres).

Prints one JSON line (and writes it to --out when given), per sphere count:
  mrays_per_s       primary rays per second over --frames orbit frames on one stream (host wall time, ending in a
                    synchronise), after --warmup frames
  kernel_ms         ore_get_kernel_ms of the last frame: [prep, primary, shadow pass, tail], CUDA events
  update_device_ms  CUDA-event time per ore_set_spheres_device call (the device build of the hierarchy), over --reps
                    calls after one warm-up call
The spheres are drawn with numpy (scaled_scene's LCG loop is slow at millions): centres uniform in the cube of edge
E = 10 (n / 64)^(1/3), radius members (k / 100)^2 for k uniform in 0..99, scaled_scene's lights, texture and sky.
The GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rte_b200  # noqa: E402

SIZES = [65536, 131072, 1 << 20, 1 << 22, 1 << 24]


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in out.split(",")][:2]
    except Exception as e:   # (the numbers below are still device-event times; say where the limit is missing)
        info["power_limit"] = f"unavailable: {e}"
    return info


def scene_of(pkg, n, seed=3):
    rng = np.random.default_rng(seed)
    extent = 10.0 * (n / 64.0) ** (1.0 / 3.0)
    pos = rng.uniform(0, extent, size=(n, 3)).astype(np.float32)
    member = (rng.integers(0, 100, size=n) / 100.0).astype(np.float32) ** 2
    base = pkg.scene.scaled_scene(64, seed)
    lights = base.lights.copy()
    lights[:, :4] *= np.float32(extent / 10.0)
    sp = np.ascontiguousarray(np.concatenate([pos, member[:, None]], axis=1), dtype=np.float32)
    return pkg.scene.Scene(spheres=sp, lights=lights, texture=base.texture, sky=base.sky, extent=extent, name=f"N({n})")


def measure(pkg, n, W, H, frames, warmup, reps):
    import torch
    sc = scene_of(pkg, n)
    r = pkg.Renderer(0)
    r.set_scene(sc)
    out = torch.zeros((2, H, W), dtype=torch.int32, device="cuda:0")
    st = torch.cuda.Stream()
    cams = [pkg.scene.orbit_camera(sc, f) for f in range(warmup + frames)]
    for f in range(warmup):
        r.render_device(cams[f], W, H, out[f & 1].data_ptr(), stream=st.cuda_stream)
    st.synchronize()
    t0 = time.perf_counter()
    for f in range(warmup, warmup + frames):
        r.render_device(cams[f], W, H, out[f & 1].data_ptr(), stream=st.cuda_stream)
    st.synchronize()
    wall = time.perf_counter() - t0
    kernel_ms = r.kernel_ms()
    large = True
    try:
        r.debug_sphere_tree("hyper", n)
    except pkg.capi.OreError:
        large = False
    t = torch.from_numpy(sc.spheres).to("cuda:0")
    r.set_spheres_device(t, st.cuda_stream)
    st.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(reps):
        r.set_spheres_device(t, st.cuda_stream)
    b.record(st)
    b.synchronize()
    update_ms = a.elapsed_time(b) / reps
    r.close()
    del t, out
    torch.cuda.empty_cache()
    return {"n": n, "large_path": large, "width": W, "height": H, "frames": frames,
            "mrays_per_s": W * H * frames / wall / 1e6, "ms_per_frame_wall": wall * 1e3 / frames,
            "kernel_ms": {"prep": kernel_ms[0], "primary": kernel_ms[1], "shadow": kernel_ms[2], "tail": kernel_ms[3]},
            "update_device_ms": update_ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sizes", default=",".join(map(str, SIZES)))
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("large_scene_timing: no CUDA device (nothing here runs without one)")
    pkg = rte_b200.pkg
    pkg.build.build_library()
    res = {"gpu": gpu_info(), "points": []}
    for n in (int(v) for v in args.sizes.split(",")):
        res["points"].append(measure(pkg, n, args.width, args.height, args.frames, args.warmup, args.reps))
        print(json.dumps(res["points"][-1]), file=sys.stderr, flush=True)
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
