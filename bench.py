#!/usr/bin/env python3
"""bench.py - Mrays/s of the render hot path on N B200s (one process per GPU).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's own CPU code on the host cores

A "step" is one frame: one pass of the hot path (frame prep -> primary nearest hit -> shadow +
shade -> packed framebuffer) over one camera of the orbit.  Default workload = BASELINE.json
configs[3] (7680x4320, 1024 spheres): the configuration the 1/2/4/8-GPU metric is quoted on; it fits
one GPU, so the SAME workload and the SAME code path run at every N (strong scaling).  With N > 1 the
frame is split into block-interleaved row bands.

value : every rank's kernels store their rows straight into the presenting GPU's frame ring over NVLink
        (peer-mapped); completion and ring-buffer reuse are signalled with stream-ordered flags
        (ore_flag_write / ore_flag_wait_geq), not with a collective.  Device-resident, CUDA events, max over ranks.
e2e   : every rank copies its own rows into ONE shared pinned HOST frame ring (POSIX shared memory registered with
        CUDA) over its own PCIe link, asynchronously behind its kernels; the presenter (rank 0's host thread) sees
        the per-rank completion counters in the same shared memory.  The device->host copies are inside the timed
        region.  Same code at N = 1.

Prints ONE JSON line on rank 0 (contract in the task statement).  `config` is the same object in both arms
(--impl ours / reference); run details live under `run`.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (W, H, n_spheres, seed, kind, description)
    "vga64": (640, 480, 64, 1, "reference", "configs[0]: 640x480, reference-formula scene R(64,1), reference camera"),
    "1080p64": (1920, 1080, 64, 2, "scaled", "configs[1]: 1920x1080, 64 random spheres S(64,2), orbit"),
    "4k1024": (3840, 2160, 1024, 3, "scaled", "configs[2]: 3840x2160, 1024 random spheres S(1024,3), 240-frame camera orbit"),
    "8k1024": (7680, 4320, 1024, 3, "scaled", "configs[3]: 7680x4320, 1024 spheres S(1024,3), row bands"),
    "4k16384": (3840, 2160, 16384, 5, "scaled", "configs[4]: 3840x2160, 16384 spheres S(16384,5)"),
}
FLOP_PER_TEST = 18  # SURVEY.md section 8(d): the reference formula after CSE, per ray-sphere test
NOMINAL_FP32_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12


def make_workload(pkg, name):
    W, H, n, seed, kind, desc = WORKLOADS[name]
    sc = pkg.scene.reference_scene(n, seed) if kind == "reference" else pkg.scene.scaled_scene(n, seed)

    def camera(frame):
        return pkg.scene.reference_camera() if kind == "reference" else pkg.scene.orbit_camera(sc, frame % 240)

    return W, H, sc, camera, desc


def base_config(desc, W, H, sc):
    """the SAME object in both arms (the driver compares it)"""
    return {"workload": desc, "width": W, "height": H, "n_spheres": sc.n_spheres, "n_lights": int(sc.lights.shape[0]),
            "rays_per_pixel": 1, "scene": sc.name}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (profiling recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t_begin=None, t_end=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = self.rows
        if t_begin is not None:
            inside = [r for r in rows if t_begin - 0.06 <= r[0] <= t_end + 0.12]
            rows = inside or rows
        for _, r in rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for i, n in enumerate(names):
                if f[5 + i].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def executed_table(workload):
    """Executed FP32 work per unit of each kernel: committed ncu op counts (fadd + fmul + 2 ffma, thread level,
    predicated on) divided by the units the profiled launch processed (profiles/r02_executed_flops.json, written by
    tools/executed_flops.py from an `ncu --metrics smsp__sass_thread_inst_executed_op_*` capture).  bench.py multiplies
    them by the LIVE unit counts of the timed frames and divides by the LIVE kernel times."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r02_executed_flops.json"))).get(workload)
    except Exception:
        return None


def dump_outputs(out_dir, frame, max_pixels=1 << 21):
    """Writes the frame the last timed step rendered so that two builds can be compared output for output:
    frame_rgb.npy (float32 [n, 3], the 0..255 R, G, B of each pixel) and frame_pixel_index.npy (float64 [n], y * W + x).
    n is every pixel up to max_pixels, else a fixed seeded sample of that many (40 MiB in all at most)."""
    os.makedirs(out_dir, exist_ok=True)
    flat = frame.reshape(-1)
    if flat.size <= max_pixels:
        idx = np.arange(flat.size)
    else:
        idx = np.sort(np.random.default_rng(0).choice(flat.size, max_pixels, replace=False))
    px = flat[idx]
    rgb = np.stack([(px >> 16) & 255, (px >> 8) & 255, px & 255], axis=1).astype(np.float32)
    np.save(os.path.join(out_dir, "frame_rgb.npy"), rgb)
    np.save(os.path.join(out_dir, "frame_pixel_index.npy"), idx.astype(np.float64))


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return rank, local, world


def host_threads():
    """threads the CPU arm can really use: the affinity mask, not OMP_NUM_THREADS (torchrun sets that to 1)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU code (oracle/_ref) or its C restatement
# ---------------------------------------------------------------------------------------------
def cpu_sample_plan(orc, sc, cam, W, H, budget_s, n_threads):
    """pick a row stride so that one sample costs about `budget_s` seconds on the host cores"""
    probe_step = max(1, H // 8)
    t0 = time.perf_counter()
    orc.render(sc, cam, W, H, y0=probe_step // 2, y_step=probe_step, want_ids=False, want_t=False, n_threads=n_threads)
    dt = time.perf_counter() - t0
    rows_probe = (H - probe_step // 2 + probe_step - 1) // probe_step
    per_row = dt / max(1, rows_probe)
    rows = int(max(1, min(H, budget_s / max(per_row, 1e-9))))
    return max(1, H // rows)


def run_cpu(args, pkg, what):
    """times the CPU checker on a bounded sample; returns (mrays, info, seconds per step)"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oraclelib  # the one place bench.py executes oracle/ (cpu_baseline + --impl reference)

    orc = oraclelib.load("best")
    W, H, sc, camera, desc = make_workload(pkg, args.workload)
    n_thr = host_threads()          # passed explicitly: omp_set_num_threads(n) inside the checker
    n_steps = args.steps if what == "reference" else 1
    n_warm = args.warmup if what == "reference" else 0
    budget = min(10.0, 150.0 / max(1, n_steps + n_warm)) if what == "reference" else 12.0
    step = cpu_sample_plan(orc, sc, camera(0), W, H, budget, n_thr)
    y0 = step // 2
    rows = (H - y0 + step - 1) // step
    times = []
    for i in range(n_warm + n_steps):
        cam = camera(i if what == "reference" else 0)
        t0 = time.perf_counter()
        orc.render(sc, cam, W, H, y0=y0, y_step=step, want_ids=False, want_t=False, n_threads=n_thr)
        dt = time.perf_counter() - t0
        if i >= n_warm:
            times.append(dt)
    total = sum(times)
    mrays = rows * W * len(times) / total / 1e6
    info = {"value": mrays, "unit": "Mrays/s", "cores": n_thr, "kind": orc.kind,
            "sample": f"rows {y0}::{step} of each {W}x{H} frame ({rows} rows, {rows * W} primary rays per step, "
                      f"{len(times)} step(s), {total:.1f} s), {n_thr} OpenMP threads requested explicitly "
                      f"(OMP_NUM_THREADS in the environment: {os.environ.get('OMP_NUM_THREADS', 'unset')})"}
    return mrays, info, total / len(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="8k1024", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the N = 1 side measurements (4K, primary-only, fast libm, reference kernel)")
    ap.add_argument("--batch", type=int, default=8, help="frames (cameras) per launch set of the device-resident path: ore_render_batch_device")
    ap.add_argument("--e2e-batch", type=int, default=4,
                    help="frames per launch set of the host-resident path (ore_render_batch_async): smaller, because a batch's "
                         "device->host copies only start when its kernels are done and the run is 20 steps long")
    ap.add_argument("--in-flight", type=int, default=2, help="batches in flight per GPU (contexts/streams used round-robin)")
    ap.add_argument("--host-buffers", type=int, default=3, help="frames in the shared host ring of the e2e path")
    ap.add_argument("--ring", type=int, default=0, help="frames in the presenter's ring (default: batch x (in-flight + 1))")
    ap.add_argument("--emulate-world", type=int, default=0,
                    help="tool, single process only: render just the rows rank --emulate-rank of this many ranks would "
                         "render (isolates per-rank effects of short frames from NVLink effects); the line says so")
    ap.add_argument("--emulate-rank", type=int, default=0)
    ap.add_argument("--band-dma", action="store_true",
                    help="N > 1: move the primary kernel's rows to the presenter with a copy engine (ORE_FLAG_BAND_DMA) instead "
                         "of storing every pixel from the kernels - the A/B switch of that design choice (default: off)")
    ap.add_argument("--diag-local-frames", action="store_true",
                    help="diagnostic, N > 1: every rank stores its rows into its own memory instead of the presenter's frame "
                         "(no NVLink stores; the frame is never assembled and the line says so)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--impl ours: after the timed steps, write the frame the last of them rendered to DIR/*.npy "
                         "(see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and (args.emulate_world > 1 or args.diag_local_frames):
        ap.error("--dump-outputs writes whole frames; --emulate-world and --diag-local-frames never assemble one")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank, local, world = dist_env()

    import rte_b200
    pkg = rte_b200.pkg
    W, H, sc, camera, desc = make_workload(pkg, args.workload)
    config = base_config(desc, W, H, sc)

    if args.impl == "reference":
        if rank != 0:
            return 0
        mrays, info, sec = run_cpu(args, pkg, "reference")
        line = {"impl": "reference", "metric": "Mrays/s (primary rays)", "value": mrays, "unit": "Mrays/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "cpu_baseline": info,
                "e2e": {"value": mrays, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ---------------- our arm ----------------
    # rank 0's stdout is ONE JSON line: anything libraries print while the job runs (NCCL's version banner, ...) goes to
    # stderr; the saved descriptor is restored for the line itself
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the render path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # NCCL prints its version banner on stdout; rank 0's stdout is ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
    emulate = args.emulate_world if (world == 1 and args.emulate_world > 1) else 0
    mg = pkg.multigpu
    F = pkg.capi
    pkg.build.build_library()
    NF = max(1, args.in_flight)
    KB = max(1, min(8, args.batch))
    ctxs = []
    for _ in range(NF):
        rx = pkg.Renderer(local)
        rx.set_scene(sc)
        ctxs.append((rx, torch.cuda.Stream(device=local)))
    r, stream = ctxs[0]
    present_stream = torch.cuda.Stream(device=local)
    # frame ring on the presenter + completion / ack flags
    NRING = args.ring if args.ring >= NF * KB else KB * (NF + 1)   # one batch of slack: a rank may run ahead of the slowest
    peer = mg.PeerFrame(r, W, H, n_buffers=NRING, band_of=(args.emulate_rank, emulate) if emulate else None,
                        local_frames=args.diag_local_frames and world > 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n_batches_done = [0]

    XF = F.ORE_FLAG_BAND_DMA if (args.band_dma and world > 1) else 0

    def render_steps(f0, n, flags=F.ORE_FLAG_NO_KERNEL_TIMING):
        """device-resident steps f0 .. f0+n-1: this rank's rows of those frames into the presenter's ring, KB frames per
        launch set, each batch announced by a flag"""
        for b0 in range(0, n, KB):
            kk = min(KB, n - b0)
            rr, st = ctxs[n_batches_done[0] % NF]
            n_batches_done[0] += 1
            peer.submit_batch([camera(f0 + b0 + i) for i in range(kk)], stream=st.cuda_stream, flags=flags | XF, renderer=rr)
            if rank == 0:
                # presenter: on the present stream, wait for every rank's rows of the batch, then acknowledge it to all
                peer.present_batch(present_stream.cuda_stream, kk)

    def join_streams(ev_list=None):
        """make `stream` wait for everything enqueued on the other streams of this rank"""
        sig = r.stream_handle(2)
        others = [st for _, st in ctxs[1:]] + [present_stream] + ([torch.cuda.ExternalStream(sig, device=dev)] if sig else [])
        for st in others:
            ev = torch.cuda.Event()
            ev.record(st)
            stream.wait_event(ev)

    frame_bytes = W * H * 4
    n_rows_mine = pkg.Renderer.rows(H, **mg.block_band(peer.band_rank, peer.band_world, H))

    # warm-up: at least three launch sets per context (the staging buffer of a context is sized from the hit count of
    # its previous frames and has settled by then)
    render_steps(0, max(args.warmup, 3 * KB * NF))
    barrier()
    # hit pixels of this rank's band (for the working-set note and the roofline units)
    warm_hits = r.counters()["hit_pixels"]

    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.15)
    ev_start = torch.cuda.Event(enable_timing=True)
    ev_end = torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin = time.perf_counter()
    ev_start.record(stream)
    for _, st in ctxs[1:]:
        st.wait_event(ev_start)
    present_stream.wait_event(ev_start)
    t_host0 = time.perf_counter()
    render_steps(args.warmup, args.steps)   # no host sync, no collective inside the timed region
    t_host1 = time.perf_counter()
    join_streams()
    ev_end.record(stream)
    barrier()
    t_end = time.perf_counter()
    clocks = sampler.stop(t_begin, t_end)
    last_frame = None
    if args.dump_outputs and rank == 0:
        # the presenter's ring slot of the last timed frame: every rank's rows have landed (barrier above) and no
        # later frame has been submitted yet
        last_frame = np.empty((H, W), dtype=np.uint32)
        r.copy_to_host(last_frame, peer.ptrs[(peer.submitted - 1) % peer.n_buffers])
    my_ms = ev_start.elapsed_time(ev_end)
    per_rank_ms = [my_ms]
    total_ms = torch.tensor([my_ms], dtype=torch.float64, device=dev)
    if world > 1:
        gathered = [torch.zeros_like(total_ms) for _ in range(world)]
        dist.all_gather(gathered, total_ms)
        per_rank_ms = [float(g.item()) for g in gathered]
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    value = W * H * args.steps / (total_ms * 1e-3) / 1e6
    host_issue_ms = (t_host1 - t_host0) * 1e3 / args.steps

    # ---- per-kernel device times (CUDA events inside the library, on the launching stream): separate untimed
    # ---- pass, one frame at a time
    kernel_ms = []
    launches_per_batch = 0
    for i in range(min(args.steps, 8)):
        render_steps(args.warmup + i, 1, flags=0)      # single frames: per-FRAME kernel times
        torch.cuda.synchronize()
        rr = ctxs[(n_batches_done[0] - 1) % NF][0]
        kernel_ms.append(rr.kernel_ms())
    render_steps(args.warmup, KB, flags=0)
    torch.cuda.synchronize()
    launches_per_batch = int(ctxs[(n_batches_done[0] - 1) % NF][0].counters()["kernel_launches"])
    launches_per_frame = launches_per_batch / KB
    barrier()

    # ---- e2e: ONE shared pinned host frame ring, every rank copies its own rows over its own PCIe link ----------
    KE = max(1, min(KB, args.e2e_batch))
    NHB = max(2 * KE, args.host_buffers)
    name = [None]
    shared = None
    if rank == 0:
        shared = mg.SharedHostFrame(W, H, peer.band_rank, peer.band_world, n_buffers=NHB,
                                    register=r.host_register, unregister=r.host_unregister)
        name = [shared.name]
    numa_note = "single process"
    if world == 1:
        shared.pin()     # (also when only one rank's rows of a larger job are rendered: --emulate-world)
    if world > 1:
        dist.broadcast_object_list(name, src=0)
        if rank != 0:
            shared = mg.SharedHostFrame(W, H, rank, world, n_buffers=NHB, name=name[0], register=r.host_register,
                                        unregister=r.host_unregister)
        # NUMA: every rank first-touches ITS rows from a CPU next to its GPU, then everybody pins the ring
        try:
            bus = torch.cuda.get_device_properties(local).pci_bus_id
            dom = getattr(torch.cuda.get_device_properties(local), "pci_domain_id", 0)
            devn = getattr(torch.cuda.get_device_properties(local), "pci_device_id", 0)
            pci = f"{dom:08x}:{bus:02x}:{devn:02x}.0"
        except Exception:
            pci = None
        cpus = mg.gpu_local_cpus(pci) if pci else None
        numa_note = (f"rows first-touched from the {len(cpus)} CPUs NVML reports local to each rank's GPU" if cpus
                     else "GPU-local CPUs unknown: rows first-touched where the rank happens to run")
        shared.touch_own_rows(pci)
        dist.barrier()
        shared.pin()
        dist.barrier()
    band = shared.band()
    e2e_ranks = [shared.rank] if emulate else list(range(world))

    def e2e_ready():
        f = shared.presented
        return all(shared.done(q) >= f + 1 for q in e2e_ranks)

    def e2e_drain(upto, block):
        while rank == 0 and shared.presented < upto:
            if e2e_ready():
                shared.present()
            elif not block:
                return
    e2e_events = []

    def e2e_run(n_frames, first_cam, timed):
        """n_frames through ore_render_async_signal into the shared host ring"""
        copy_stream = torch.cuda.ExternalStream(r.stream_handle(1), device=dev)
        render_stream = torch.cuda.ExternalStream(r.stream_handle(0), device=dev)
        target = shared.submitted + n_frames
        if timed:
            e0 = torch.cuda.Event(enable_timing=True)
            e0.record(render_stream)
        for b0 in range(0, n_frames, KE):
            kk = min(KE, n_frames - b0)
            while not shared.can_submit_batch(kk):   # ring full: wait for the presenter (rank 0 keeps presenting meanwhile)
                e2e_drain(target, False)
            slots = [shared.next_slot() for _ in range(kk)]
            r.render_batch_async([camera(first_cam + b0 + i) for i in range(kk)], W, H,
                                 [shared.row_addr(buf, band["y0"]) for _, buf in slots], in_place=True,
                                 done_flag=shared.done_addr(shared.rank), first_done_value=slots[0][0] + 1,
                                 flags=F.ORE_FLAG_NO_KERNEL_TIMING, **band)
            e2e_drain(target, False)
        if timed:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record(copy_stream)               # behind the last frame's copy and its completion flag
            e2e_events.append((e0, e1))
        e2e_drain(target, True)                  # presenter: every rank's rows of every frame have landed
        r.wait()

    e2e_run(2 * KE, 0, False)
    barrier()
    t0 = time.perf_counter()
    e2e_run(args.steps, args.warmup, True)
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - t0
    e0, e1 = e2e_events[-1]
    tt = torch.tensor([e0.elapsed_time(e1), wall * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e_ms, e2e_wall_ms = [float(v) for v in tt.tolist()]
    e2e_value = W * H * args.steps / (e2e_ms * 1e-3) / 1e6
    e2e_wall_value = W * H * args.steps / (e2e_wall_ms * 1e-3) / 1e6
    frame_check = None
    if rank == 0:
        last_g = shared.submitted - 1
        got = shared.frames[last_g % NHB]
        alone = r.render(camera(args.warmup + args.steps - 1), W, H)
        if emulate:
            rows = mg.block_rows(peer.band_rank, peer.band_world, H)
            frame_check = "identical" if np.array_equal(alone[rows], got[rows]) else "MISMATCH"
        else:
            frame_check = "identical" if np.array_equal(alone, got) else "MISMATCH"
    # ---- what the platform allows: all ranks copy device -> host at the same time, no rendering (the bound of e2e) ----
    d2h_probe = None
    try:
        slice_bytes = min(64 << 20, (NHB * frame_bytes // max(1, world)) & ~0xFFF)
        src = torch.empty(slice_bytes, dtype=torch.uint8, device=dev)
        pinned = torch.empty(slice_bytes, dtype=torch.uint8).pin_memory()
        reps = 6
        res = {}
        for label in ("cudaHostAlloc", "registered_shared_ring"):
            barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                if label == "cudaHostAlloc":
                    pinned.copy_(src, non_blocking=True)
                    torch.cuda.current_stream().synchronize()
                else:
                    r.copy_to_host(np.frombuffer(shared.shm.buf, dtype=np.uint8, count=slice_bytes,
                                                 offset=shared.HEADER + (rank if not emulate else 0) * slice_bytes), src.data_ptr())
            barrier()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            res[label] = world * reps * slice_bytes / float(dt.item()) / 1e9
        d2h_probe = {"aggregate_gbs": res, "bytes_per_copy": slice_bytes, "copies": reps,
                     "what": "every rank copies device -> pinned host memory at the same time, nothing else running; "
                             "Mrays/s bound of ANY host-resident frame = aggregate GB/s / 4 bytes per pixel"}
        d2h_probe["e2e_bound_mrays"] = res["registered_shared_ring"] / 4 * 1e3
    except Exception as e:   # a measurement extra only
        d2h_probe = {"unavailable": str(e)[:200]}
    # synchronous update() semantics at N = 1, for reference: launch + sync + copy per call
    e2e_sync_value = None
    if world == 1 and not emulate:
        hostbuf = r.host_alloc((H, W))
        for f in range(2):
            r.render(camera(f), W, H, out=hostbuf)
        t0 = time.perf_counter()
        for i in range(args.steps):
            r.render(camera(args.warmup + i), W, H, out=hostbuf, flags=F.ORE_FLAG_NO_KERNEL_TIMING)
        e2e_sync_value = W * H * args.steps / (time.perf_counter() - t0) / 1e6
        r.host_free(hostbuf)
    barrier()

    # ---- accounting (untimed): live unit counts of the timed frames + reference-order test counts ----
    own = {"primary": 0.0, "shadow": 0.0, "sky": 0.0, "hits": 0.0, "pixels": 0.0, "exact_p": 0.0, "exact_s": 0.0,
           "l1": 0.0, "l2": 0.0}
    band_kw = peer.band_args(0)
    for i in range(args.steps):
        r.render_device(camera(args.warmup + i), W, H, flags=F.ORE_FLAG_COUNT_REFERENCE_TESTS, **band_kw)
        c = r.counters()
        own["primary"] += c["primary_tests"]
        own["shadow"] += c["shadow_tests_ref"]
        own["sky"] += c["sky_tests"]
        own["hits"] += c["hit_pixels"]
        own["pixels"] += c["pixels"]
        own["exact_p"] += c["exact_primary"]
        own["exact_s"] += c["exact_shadow"]
        own["l1"] += c["beam_l1"]
        own["l2"] += c["beam_l2"]
    keys = list(own)
    counts = torch.tensor([own[k] for k in keys], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(counts)
    tot = dict(zip(keys, [float(v) for v in counts.tolist()]))
    peak_tf, nominal_mhz = r.measure_fp32_peak()
    k_shadow_ms = statistics.mean(m[2] for m in kernel_ms)
    k_primary_ms = statistics.mean(m[1] for m in kernel_ms)
    k_prep_ms = statistics.mean(m[0] for m in kernel_ms)
    # (1) algorithmic rate: what a literal implementation of the reference's loops would have to execute
    alg_tf_shadow = FLOP_PER_TEST * own["shadow"] / args.steps / (k_shadow_ms * 1e-3) / 1e12
    alg_tf_step = FLOP_PER_TEST * (tot["primary"] + tot["shadow"] + tot["sky"]) / args.steps / (total_ms / args.steps * 1e-3) / 1e12
    # (2) executed rate: FP32 operations the kernels really execute = committed ncu op counts per unit x LIVE units
    ex = executed_table(args.workload)
    executed = None
    frac = None
    achieved_tf = None
    if ex:
        hits_f, px_f = own["hits"] / args.steps, own["pixels"] / args.steps
        fl_shadow = ex["shadow_pass"]["flop_per_hit_pixel"] * hits_f
        fl_primary = ex["primary"]["flop_per_pixel"] * px_f
        achieved_tf = fl_shadow / (k_shadow_ms * 1e-3) / 1e12
        frac = achieved_tf / peak_tf if peak_tf else None
        executed = {
            "source": ex.get("source"),
            "shadow_pass": {"flop_per_hit_pixel": ex["shadow_pass"]["flop_per_hit_pixel"], "hit_pixels_per_launch": hits_f,
                            "flop_per_launch": fl_shadow, "kernel_ms": k_shadow_ms, "achieved_tflops": achieved_tf,
                            "frac_of_measured_peak": frac},
            "primary": {"flop_per_pixel": ex["primary"]["flop_per_pixel"], "pixels_per_launch": px_f,
                        "flop_per_launch": fl_primary, "kernel_ms": k_primary_ms,
                        "achieved_tflops": fl_primary / (k_primary_ms * 1e-3) / 1e12,
                        "frac_of_measured_peak": (fl_primary / (k_primary_ms * 1e-3) / 1e12 / peak_tf) if peak_tf else None},
            "issue_slot_utilisation": ex.get("issue_slot_utilisation"),
            "live_cross_check": {
                "what": "device counters of the timed frames against the profiled frame's (same units => same work)",
                "exact_shadow_tests_per_hit_pixel": own["exact_s"] / max(1.0, own["hits"]),
                "profiled_exact_shadow_tests_per_hit_pixel": ex.get("exact_shadow_per_hit_pixel"),
                "cone_tests_per_hit_pixel": own["l2"] / max(1.0, own["hits"]),
                "profiled_cone_tests_per_hit_pixel": ex.get("cone_tests_per_hit_pixel")},
        }
    hbm_peak, hbm_src = measured_hbm_peak()
    traffic = (ex or {}).get("shadow_pass", {}).get("dram_bytes_per_hit_pixel")
    traffic_launch = traffic * own["hits"] / args.steps if traffic else None

    # ---- N = 1 side measurements ----------------------------------------------------------------
    extras = {}
    count_out = peer.ptrs[0]
    if world == 1 and not emulate and not args.no_extras:
        def timed_frames(n, w, h, flags=0, cam0=args.warmup):
            """ms per frame over n frames, KB frames per launch set like the main measurement (one context, one stream)"""
            outs = peer.ptrs[:KB]
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

            def run(first, count):
                for b0 in range(0, count, KB):
                    kk = min(KB, count - b0)
                    r.render_batch_device([camera(first + b0 + i) for i in range(kk)], w, h, outs[:kk], stream=stream.cuda_stream,
                                          flags=flags | F.ORE_FLAG_NO_KERNEL_TIMING)
            run(0, KB)
            stream.synchronize()
            ev0.record(stream)
            run(cam0, n)
            ev1.record(stream)
            ev1.synchronize()
            return ev0.elapsed_time(ev1) / n

        if args.workload == "8k1024":
            ms4 = timed_frames(12, 3840, 2160)
            kms4 = []
            for i in range(4):
                r.render_device(camera(args.warmup + i), 3840, 2160, out_ptr=count_out, stream=stream.cuda_stream)
                stream.synchronize()
                kms4.append(r.kernel_ms())
            extras["also_configs2_4k1024"] = {
                "workload": WORKLOADS["4k1024"][5], "value": 3840 * 2160 / ms4 / 1e3, "unit": "Mrays/s", "ms_per_step": ms4,
                "steps": 12, "kernel_ms": {"prep": statistics.mean(m[0] for m in kms4), "primary": statistics.mean(m[1] for m in kms4),
                                           "shadow": statistics.mean(m[2] for m in kms4)}}
        r.set_lights(sc.lights[:0])
        po_ms = timed_frames(12, W, H)
        r.set_lights(sc.lights)
        po_tf = FLOP_PER_TEST * W * H * sc.n_spheres / (po_ms * 1e-3) / 1e12
        extras["primary_only"] = {"what": "n_lights = 0: primary nearest hit + sky only; reference tests = W*H*N", "ms_per_step": po_ms,
                                  "value": W * H / po_ms / 1e3, "unit": "Mrays/s",
                                  "algorithmic_tflops": po_tf, "algorithmic_speedup_vs_literal": po_tf / peak_tf if peak_tf else None}
        fl_ms = timed_frames(12, W, H, flags=F.ORE_FLAG_FAST_LIBM)
        extras["fast_libm"] = {"flag": "ORE_FLAG_FAST_LIBM", "value": W * H / fl_ms / 1e3, "unit": "Mrays/s", "ms_per_step": fl_ms, "steps": 12,
                               "note": "CUDA's cosf/sinf/acosf/atan2f instead of the glibc-bit-compatible device functions; ids/t "
                                       "unchanged, pixels within 1 LSB on >= 99.9 % instead of bit-identical"}
        if not args.no_cpu_baseline:
            try:
                sys.path.insert(0, os.path.join(ROOT, "tests"))
                import oraclelib
                ref_gpu = {}
                cams = [camera(args.warmup + i) for i in range(3)]
                for fast in (False, True):
                    if oraclelib.have_ref_gpu(fast):
                        _, ms_up, ms_k = oraclelib.RefGpu(fast=fast).render(sc, cams, W, H)
                        ref_gpu["use_fast_math" if fast else "default_flags"] = {
                            "ms_per_update": ms_up, "ms_per_kernel": ms_k,
                            "mrays_per_s_update": W * H / ms_up / 1e3, "mrays_per_s_kernel": W * H / ms_k / 1e3}
                ref_gpu["what"] = ("the reference's rayTrace kernel / update() compiled unmodified in arithmetic for sm_100 "
                                   "(oracle/ref_build/make_ref_gpu.py), run headless on this GPU in this run")
                extras["reference_kernel_on_b200"] = ref_gpu
            except Exception as e:  # measurement extra only
                extras["reference_kernel_on_b200"] = {"unavailable": str(e)[:200]}
    mem_used = None
    try:
        free_b, total_b = torch.cuda.mem_get_info(local)
        mem_used = (total_b - free_b) / 1e9
    except Exception:
        pass

    if rank == 0:
        cpu = None
        if world == 1 and not emulate and not args.no_cpu_baseline:
            _, cpu, _ = run_cpu(args, pkg, "cpu_baseline")
        hits_rank = own["hits"] / args.steps
        ws_mb = (n_rows_mine * W * 4 * 3 + hits_rank * (4 + 4 * (6 + 31 * int(sc.lights.shape[0])))) / 1e6
        line = {
            "metric": "Mrays/s (primary rays)", "value": value, "unit": "Mrays/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config,
            "run": {
                "l2": (f"not flushed at any N (one policy): the inputs a step reads are the 64 KB of scene records the kernels keep "
                       f"in shared memory by design; what it WRITES and re-reads is larger than L2 - per rank and step "
                       f"{ws_mb:.0f} MB of framebuffer rows, hit records and shadow staging, x {NF * KB} frames in flight, L2 126 MB"),
                "frame_overlap": (f"{KB} frames (cameras) per launch set (ore_render_batch_device / ore_render_batch_async), {NF} launch sets "
                                  f"in flight per GPU (contexts/streams used round-robin), ring of {NRING} presenter frames; the same at every N"),
                "parallelism": (f"row-bands x{world} (8-row blocks dealt round-robin), presenter = rank 0; rows land in the presenter's "
                                f"ring over NVLink - " + ("the primary kernel's rows by copy engine behind the shadow pass, hit pixels stored by the sweep (--band-dma)"
                                                        if args.band_dma else "every pixel stored by the render kernels") +
                                f"; completion = per-rank flags (no collective in the timed region)"
                                if world > 1 else "1 GPU (same code path: frame ring + flags)"),
                "emulated": (f"rows of rank {peer.band_rank} of {emulate} only, on ONE GPU: value counts the WHOLE frame's pixels, i.e. it is "
                             f"the rate {emulate} such ranks would reach together if NVLink cost nothing - a tool output, not a bench line"
                             if emulate else None),
                "diagnostic": ("--diag-local-frames: rows stored into each rank's own memory, frame never assembled - not a bench line"
                               if (args.diag_local_frames and world > 1) else None),
                "hit_pixel_fraction": tot["hits"] / max(1.0, tot["pixels"]),
                "host_issue_ms_per_step": host_issue_ms,
                "timed_region_ms_per_rank": per_rank_ms,
                "device_memory_used_gb": mem_used,
                "tests_per_pixel": {"primary": tot["primary"] / max(1.0, tot["pixels"]),
                                    "shadow_reference_order": tot["shadow"] / max(1.0, tot["pixels"])},
            },
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": 36 + 36,
                    "d2h_bytes_per_step": W * H * 4 + 4 * world,
                    "mode": (f"ore_render_batch_async, {KE} frames per launch set: every rank copies its own row blocks into ONE shared pinned host frame ring "
                             f"({NHB} frames, POSIX shm registered with CUDA) over its own PCIe link, copy of frame f behind the kernels "
                             f"of f+1; per-rank completion counters in the same shared memory; the presenter's host thread consumes "
                             f"frames in order. Timed with CUDA events (first render -> last copy + flag landed), max over ranks"),
                    "wall_clock_value": e2e_wall_value,
                    "synchronous_value": e2e_sync_value,
                    "note": "inputs per step are the 36-byte camera and the 36-byte frame descriptor (kernel arguments); output per "
                            "step is the whole framebuffer in pinned host memory plus a 4-byte counter per rank; "
                            "synchronous_value = ore_render (launch + sync + copy per call, the reference update() semantics, N = 1)",
                    "host_pages": numa_note,
                    "platform_d2h_probe": d2h_probe,
                    "sharded_frame_check": frame_check},
            "gpu_launches": int(round(launches_per_frame * args.steps)),
            "gpu_launches_per_frame": {"count": launches_per_frame, "per_launch_set": launches_per_batch, "frames_per_launch_set": KB,
                                       "kernels": "prep_frame, primary_tile, catch-all sweep (normally empty), shade_setup, shadow_sweep"},
            "roofline": {
                "bound": "fp32",
                "kernel": "shadow pass (soft-shadow any-hit + shading; the dominant kernels of the step)",
                "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": frac,
                "traffic": traffic_launch,
                "peak_source": "measured: FFMA burn on this GPU in this run (MEASURED_PEAKS.json carries HBM and bf16 only); "
                               f"nominal 148 SM x 128 lanes x 2 x 1.965 GHz = {NOMINAL_FP32_TFLOPS:.2f}",
                "definition": "achieved = EXECUTED FP32 FLOP of the launch (fadd + fmul + 2 ffma, thread level: committed ncu op "
                              "counts per hit pixel x the hit pixels of the timed frames, counted on the device) / CUDA-event "
                              "kernel time; frac = achieved / measured FFMA peak. The kernels are bound by instruction issue, "
                              "not by the FP32 pipe (see `executed`); the algorithmic rate of SURVEY.md 8(d) is reported "
                              "separately as algorithmic_speedup_vs_literal.",
                "executed": executed,
                "algorithmic": {
                    "flop_per_test": FLOP_PER_TEST, "reference_order_shadow_tests_per_launch": own["shadow"] / args.steps,
                    "shadow_pass_tflops": alg_tf_shadow, "whole_step_tflops": alg_tf_step,
                    "algorithmic_speedup_vs_literal": alg_tf_shadow / peak_tf if peak_tf else None,
                    "whole_step_speedup_vs_literal": alg_tf_step / peak_tf if peak_tf else None,
                    "definition": "18 FLOP x sphere tests the REFERENCE's loop order makes (counted exactly on the device by "
                                  "the literal loop, untimed) / time / FFMA peak: how many times faster than a perfect literal "
                                  "implementation of kernel.cu:332-336 the pass runs. Not a hardware utilisation."},
                "kernel_ms_all": {"prep": k_prep_ms, "primary": k_primary_ms, "shadow": k_shadow_ms},
                "dram_write_gbs_framebuffer": n_rows_mine * W * 4 / ((k_primary_ms + k_shadow_ms) * 1e-3) / 1e9,
                "hbm": {"peak_gbs": hbm_peak, "peak_source": hbm_src,
                        "achieved_gbs": (traffic_launch / (k_shadow_ms * 1e-3) / 1e9) if traffic_launch else None,
                        "frac": (traffic_launch / (k_shadow_ms * 1e-3) / 1e9 / hbm_peak) if traffic_launch else None},
            },
            "cpu_baseline": cpu,
        }
        line.update(extras)
        if last_frame is not None:
            dump_outputs(args.dump_outputs, last_frame)
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line))
        sys.stdout.flush()
        os.dup2(2, 1)
    shared.close()
    peer.close()
    for rx, _ in ctxs[1:]:
        rx.close()
    r.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
