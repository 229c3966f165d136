"""Cost of a stream-ordered sphere update (ore_set_spheres_device) and what it does to an animated 8K loop.

Prints one JSON line (and writes it to --out when given):
  update:   CUDA-event time per ore_set_spheres_device call on a stream, over back-to-back updates after warm-up, at
            n in {1024, 16384, 65536}; host time to enqueue one call; host wall time of one synchronous ore_set_spheres
  animated: the 8K / S(1024,3) orbit loop of bench.py, one frame per iteration on one stream with no host
            synchronisation inside the timed window - (fixed) scene never changes, (device) a torch op moves the
            spheres then ore_set_spheres_device, (host) the same torch op, the spheres copied to the host and
            ore_set_spheres; Mrays/s (primary rays) of each
The GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import rte_b200  # noqa: E402


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


def moved(base, idx, f):
    import torch
    out = base.clone()
    out[:, 0] += 0.35 * torch.sin(0.05 * f + 0.37 * idx)
    out[:, 1] += 0.25 * torch.cos(0.03 * f + 0.11 * idx)
    return out


def update_cost(pkg, n, reps, warmup):
    import torch
    sc = pkg.scene.scaled_scene(n, 3)
    r = pkg.Renderer(0)
    r.set_scene(sc)
    t = torch.from_numpy(sc.spheres.copy()).to("cuda:0")
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    for _ in range(warmup):
        r.set_spheres_device(t, st.cuda_stream)
    st.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    h0 = time.perf_counter()
    for _ in range(reps):
        r.set_spheres_device(t, st.cuda_stream)
    h1 = time.perf_counter()
    b.record(st)
    b.synchronize()
    dev_us = a.elapsed_time(b) * 1e3 / reps
    host_ms = []
    for k in range(warmup + 20):
        t0 = time.perf_counter()
        r.set_spheres(sc.spheres)
        if k >= warmup:
            host_ms.append((time.perf_counter() - t0) * 1e3)
    r.close()
    host_ms.sort()
    return {"n": n, "device_update_us": dev_us, "enqueue_us_per_call": (h1 - h0) * 1e6 / reps,
            "host_setter_ms_median": host_ms[len(host_ms) // 2], "host_setter_ms_min": host_ms[0], "updates_timed": reps}


def animated(pkg, mode, frames, warmup):
    import torch
    W, H, sc, camera, desc = bench.make_workload(pkg, "8k1024")
    r = pkg.Renderer(0)
    r.set_scene(sc)
    F = pkg.capi
    base = torch.from_numpy(sc.spheres.copy()).to("cuda:0")
    idx = torch.arange(base.shape[0], device="cuda:0", dtype=torch.float32)
    out = torch.zeros((2, H, W), dtype=torch.int32, device="cuda:0")
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    keep = []

    def frame(f):
        if mode == "device":
            cur = moved(base, idx, f)
            r.set_spheres_device(cur, st.cuda_stream)
            keep.append(cur)
            del keep[:-4]
        elif mode == "host":
            cur = moved(base, idx, f)
            r.set_spheres(cur.cpu().numpy())   # (.cpu() waits for the torch op; the setter synchronises)
        r.render_device(camera(f), W, H, out[f & 1].data_ptr(), stream=st.cuda_stream, flags=F.ORE_FLAG_NO_KERNEL_TIMING)

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
            "mrays_per_s": W * H * frames / (wall * 1e3) / 1e3, "workload": desc}


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
        raise SystemExit("scene_update_timing: no CUDA device (nothing here runs without one)")
    pkg = rte_b200.pkg
    pkg.build.build_library()
    res = {"gpu": gpu_info(), "update": [update_cost(pkg, n, args.reps, args.warmup) for n in (1024, 16384, 65536)],
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
