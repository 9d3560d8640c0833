#!/usr/bin/env python3
"""bench.py — headline benchmark of the B200-native path-tracing hot path.

Metric (BASELINE.json): Mrays/s and time-to-image at 1080p / 1024 spp on 1/2/4/8 B200, next to the
reference's CPU renderer on the box's host cores.

  workload   scenes/cornell-box-scene.json, 1920x1080, 1024 spp, max depth 50 (BASELINE config C3, the one
             the metric is quoted on at 1/2/4/8 GPUs); camera/geometry from the scene file.
  step       one full render of that image (one pass of Camera::render over all pixels x samples).
  value      ray segments (closest-hit queries, camera.rs:280) per second, whole job, scene resident in HBM,
             framebuffer left on the device of rank 0 (N>1: includes the NCCL gather of the owned rows).
  e2e        the same metric through the public API call a user makes (Scene.render, mirror of the
             reference's Scene::render): host scene description in, host f32 image out — scene flatten +
             H2D upload and the framebuffer D2H are inside the timed region.
  scaling    "strong": the same image is tile-partitioned over N GPUs (time-to-image is the point).

`--impl reference` times the reference's CPU algorithm (the C++ restatement in oracle/, because the Rust
crate cannot be built here) with all host threads on a bounded sample (same scene / resolution / depth,
reduced spp: cost is exactly linear in spp, camera.rs:325-329).
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
CALLER_CWD = os.getcwd()  # where a relative --dump-outputs DIR is meant to be
os.chdir(ROOT)  # scene files reference textures / sub-scenes relative to the CWD, like the reference CLI

SCENE = "scenes/cornell-box-scene.json"
WIDTH, HEIGHT, SPP, DEPTH = 1920, 1080, 1024, 50
METRIC, UNIT = "path_tracing_throughput_1080p_1024spp", "Mrays/s"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples nvidia-smi during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons, power = [], None, set(), []
        for ts, line in self.lines:
            if ts < t0 or ts > t1 + 0.3:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power) if power else None}


# ----------------------------------------------------------------------------- reference arm / cpu baseline
def host_threads() -> int:
    """All host cores this process may use (torchrun exports OMP_NUM_THREADS=1; the reference arm ignores that)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def oracle_sample(spp_sample: int, n_threads: int = 0, repeats: int = 1):
    """Times the oracle on the bench workload at reduced spp.  Returns (Mrays/s, seconds, segments, threads, image)."""
    if n_threads <= 0:
        n_threads = host_threads()
    from nr_ray_tracer_b200.scene_config import CameraConfig, load_scene
    from oracle import oracle as O
    g = load_scene(SCENE, camera_override=CameraConfig(width=WIDTH, height=HEIGHT, samples_per_pixel=spp_sample,
                                                       ray_max_bounces=DEPTH))
    sc = O.OracleScene(g)
    cam = O.camera_build(g.camera.to_builder_config())
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        img, cnt = sc.render(cam, seed=0, n_threads=n_threads)
        dt = time.perf_counter() - t0
        if best is None or dt < best[1]:
            best = (cnt["segments"] / dt / 1e6, dt, cnt["segments"])
    return best + (n_threads, img)


DUMP_BYTES = 64 * 1024 * 1024


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy, at most DUMP_BYTES in all.  An array larger than its even share of what
    the smaller ones leave is replaced by a fixed, seeded sample of its pixels (last axis kept; the same pixels for the
    same shape), so that two builds run with the same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES - 4096 * len(arrays)  # room for each .npy header
    for k, (name, a) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].nbytes)):
        share = left // (len(arrays) - k)
        if a.nbytes > share:
            px = a.reshape(-1, a.shape[-1])
            keep = np.random.default_rng(0).choice(len(px), share // px[0].nbytes, replace=False)
            a = px[np.sort(keep)]
        left -= a.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    spp_sample = args.ref_spp
    sample = f"{SCENE} {WIDTH}x{HEIGHT}, depth {DEPTH}, {spp_sample} spp per step (of {SPP}; cost is linear in spp)"
    for _ in range(args.warmup):
        oracle_sample(spp_sample)
    times, segs, threads = [], 0, 1
    for _ in range(args.steps):
        _m, dt, s, threads, img = oracle_sample(spp_sample)
        times.append(dt)
        segs += s
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"image": img, "segments": np.array([s], dtype=np.float64)})
    total = sum(times)
    value = segs / total / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / max(args.steps, 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{SCENE} {WIDTH}x{HEIGHT} {SPP}spp depth{DEPTH}", "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "time_to_image_s_extrapolated": (total / max(args.steps, 1)) * SPP / spp_sample,
        "note": "C++ restatement of the reference algorithm (oracle/oracle.cpp), OpenMP over pixels; "
                "the Rust crate cannot be built in this image (no cargo/rustc)",
    }
    print(json.dumps(line))
    return 0


# ----------------------------------------------------------------------------- B200 arm
def scene_h2d_bytes(desc) -> int:
    d = desc
    b = d.n_wnodes * 128 + d.n_wnodes * 8 * 48 + (d.n_nodes * (64 + 96) if d.n_nodes < 64 else 0)
    b += d.n_spheres * (32 + 3 * 4) + d.n_planes * (128 + 3 * 4)
    b += d.n_instances * (64 + 4) + d.n_xforms * 200 + d.n_materials * 16 + d.n_textures * 72
    for i in range(d.n_images):
        b += d.images[i].width * d.images[i].height * 4
    return int(b)


def primary_rays(cam, min_rays=2_000_000):
    """Coherent camera rays of `cam` (pixel centres, no lens), supersampled on a regular sub-pixel grid until there
    are at least min_rays of them: the input of the traversal-only microbenchmark."""
    W, H = cam.width, cam.height
    k = 1
    while W * H * k * k < min_rays:
        k += 1
    sub = (np.arange(k, dtype=np.float64) + 0.5) / k - 0.5
    xs = (np.arange(W, dtype=np.float64)[:, None] + sub[None, :]).reshape(-1)
    ys = (np.arange(H, dtype=np.float64)[:, None] + sub[None, :]).reshape(-1)
    gx, gy = np.meshgrid(xs, ys)
    tl, du, dv = (np.array(list(v)) for v in (cam.viewport_top_left, cam.pixel_delta_u, cam.pixel_delta_v))
    org = np.array(list(cam.look_from))
    pts = tl + gx[..., None] * du + gy[..., None] * dv
    return np.ascontiguousarray(np.concatenate([np.broadcast_to(org, pts.shape), pts - org], axis=-1).reshape(-1, 6))


def run_b200(args):
    import torch
    import torch.distributed as dist
    from nr_ray_tracer_b200 import _abi as A, api, distributed as D
    from nr_ray_tracer_b200.scene_config import CameraConfig, load_scene

    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local_rank = env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 arm has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    mode = {"auto": A.MODE_AUTO, "pool": A.MODE_POOL, "fused": A.MODE_FUSED, "wavefront": A.MODE_WAVEFRONT,
            "megakernel": A.MODE_MEGAKERNEL}[args.mode]
    KERNEL = {A.MODE_POOL: "k_render_pool", A.MODE_FUSED: "k_render_fused", A.MODE_WAVEFRONT: "k_wf_extend",
              A.MODE_MEGAKERNEL: "k_render_mega"}
    R = D.rows_per_block_for(world)

    graph = load_scene(SCENE, camera_override=CameraConfig(width=args.width, height=args.height,
                                                           samples_per_pixel=args.spp, ray_max_bounces=DEPTH))
    cam = api.camera_build(graph.camera.to_builder_config())
    ctx = api.Context(local_rank)
    ctx.set_stream(torch.cuda.current_stream().cuda_stream)
    host = api.HostScene(graph, bvh=args.bvh)
    ctx.upload(host)
    W, H = cam.width, cam.height
    G = D.FramebufferGather(H, W, rank, world, R, dev)      # persistent buffers of the multi-GPU exchange
    pinned = torch.zeros((H, W, 3), dtype=torch.float32).pin_memory() if rank == 0 else None
    pageable = np.zeros((H, W, 3), dtype=np.float32) if rank == 0 else None
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def step_device():
        """value: scene resident, result left on the device (rank 0 holds the assembled image)."""
        last["image"], st, _ = D.render_distributed(ctx, cam, rank, world, seed=0, mode=mode, gather=G)
        return st

    def step_e2e(out_np=None):
        """e2e: the call a user makes — Scene(...).render(): host scene description in (BVH build + flatten on the
        host, H2D upload of the flat scene), host f32 image out (D2H inside nrrt_render).  N > 1: the same per rank
        through distributed.render_distributed (render -> NCCL gather -> D2H on rank 0)."""
        scene = api.Scene(graph, ctx=ctx, bvh=args.bvh)
        if world == 1:
            scene.render(out=out_np, seed=0, mode=mode)
            return scene.last_stats
        _, st, _ = D.render_distributed(ctx, scene.camera, rank, world, seed=0, mode=mode, gather=G, host_out=pinned)
        return st

    def timed(fn, k):
        """Runs fn k times; each step bracketed by barrier+sync, timed with CUDA events on the launch stream,
        max over ranks; L2 flushed (untimed) between steps."""
        per_step, stats = [], []
        for _ in range(k):
            flush.fill_(1.0)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            st = fn()
            e1.record()
            barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            per_step.append(float(ms.item()))
            stats.append(st)
        return per_step, stats

    def total(stats, key):
        t = torch.tensor([float(sum(s[key] for s in stats))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- untimed: the N-GPU image must be the 1-GPU image, bit for bit (low spp, once)
    identical = None
    if world > 1:
        ccam = api.camera_build(graph.camera.to_builder_config())
        ccam.samples_per_pixel = min(4, cam.samples_per_pixel)
        full, _, _ = D.render_distributed(ctx, ccam, rank, world, seed=0, mode=mode, gather=G)
        if rank == 0:
            one = torch.zeros((H, W, 3), dtype=torch.float32, device=dev)
            ctx.render(ccam, seed=0, mode=mode, out_device_ptr=one.data_ptr())
            torch.cuda.synchronize()
            identical = bool(torch.equal(full, one))
            del one
        barrier()

    # ---- warm-up
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()

    # ---- timed: device-resident
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    t_wall0 = time.time()
    ms_steps, stats = timed(step_device, args.steps)
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    segs = total(stats, "segments")
    paths = total(stats, "paths")
    launches = total(stats, "launches")
    sum_ms = sum(ms_steps)
    value = segs / (sum_ms * 1e-3) / 1e6
    ext_ms = sum(s["extend_ms"] for s in stats)
    ext_launches = sum(s["extend_launches"] for s in stats)
    my_segs = sum(s["segments"] for s in stats)
    mode_used = stats[0]["mode"]
    kernel_name = KERNEL.get(mode_used, "?")
    # ---- untimed: what the last timed step of each path handed its caller (the gather buffers are reused below)
    outputs = {}
    if args.dump_outputs:
        outputs["segments"] = np.array([total(stats[-1:], "segments")], dtype=np.float64)
        if rank == 0:
            outputs["image"] = last["image"].cpu().numpy()

    # ---- timed: end to end through the public API (host buffers)
    pinned_np = pinned.numpy() if rank == 0 else None
    step_e2e(pinned_np)
    ms_e2e, stats_e2e = timed(lambda: step_e2e(pinned_np), args.steps)
    if args.dump_outputs and rank == 0:
        outputs["e2e_image"] = pinned_np.copy()
    segs_e2e = total(stats_e2e, "segments")
    e2e_value = segs_e2e / (sum(ms_e2e) * 1e-3) / 1e6
    e2e_pageable = None
    if world == 1:
        ms_pg, stats_pg = timed(lambda: step_e2e(pageable), args.steps)
        e2e_pageable = total(stats_pg, "segments") / (sum(ms_pg) * 1e-3) / 1e6

    line = None
    if rank == 0:
        # ---- per-segment traversal counts from an instrumented low-spp pass over the same scene/camera (untimed)
        ccam = api.camera_build(graph.camera.to_builder_config())
        ccam.samples_per_pixel = 2
        ctx.upload(host)
        fb = torch.zeros((H, W, 3), dtype=torch.float32, device=dev)
        _, cst = ctx.render(ccam, seed=0, count=True, out_device_ptr=fb.data_ptr())
        del fb
        nodes_seg = cst["node_visits"] / cst["segments"]
        prims_seg = cst["prim_tests"] / cst["segments"]
        exact_seg = cst["box_exact"] / cst["segments"]
        d = host.desc
        b_prim = 128 if d.n_planes >= d.n_spheres else 32   # bytes one exact primitive test reads (one record)
        b_state = 48 + 24 + 4 if mode_used == A.MODE_WAVEFRONT else 0  # extend kernel: ray in, hit out, queue index
        bytes_seg = nodes_seg * 128 + exact_seg * 48 + prims_seg * b_prim + b_state   # four-slot nodes: 128 B each
        # ---- the traversal ceiling, measured here: coherent primary rays of the same camera (>= 2 M of them) through
        # the closest-hit entry point of the same library — same BVH, same box filter and exact primitive tests, no
        # shading, no path state, 16 bytes out per ray
        prim_rays = torch.from_numpy(primary_rays(cam)).to(dev)
        n_rays = prim_rays.shape[0]
        prim_hits = torch.zeros((n_rays, 16), dtype=torch.uint8, device=dev)
        trav_best = 0.0
        for _ in range(6):
            ts = ctx.trace_rays_device(prim_rays.data_ptr(), n_rays, prim_hits.data_ptr(), compact=True)
            trav_best = max(trav_best, n_rays / ts["kernel_ms"] / 1e3)
        del prim_rays, prim_hits
        kernel_rate = (my_segs / (ext_ms * 1e-3) / 1e6) if ext_ms > 0 else None
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except (OSError, ValueError):
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        hbm_achieved = (my_segs * bytes_seg) / (ext_ms * 1e-3) / 1e9 if ext_ms > 0 else None
        # ---- ncu figures of the same kernel from ONE --set full capture of this build on this workload
        # (profiles/ncu_traffic.json names the capture; tools/ncu_traffic.py regenerates it)
        traffic = issue_pct = lanes = capture = None
        try:
            nt = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            k = nt[kernel_name]
            # DRAM traffic of this kernel is the per-item partial sums: it scales with the image, not with spp / segments
            iw, ih = k.get("image", [1920, 1080])
            traffic = k["dram_bytes"] * (W * H) / float(iw * ih) / world
            issue_pct, lanes = k.get("issue_slot_utilisation_pct"), k.get("active_threads_per_instruction")
            capture = k.get("source")
        except (OSError, ValueError, KeyError):
            pass
        roofline = {
            "bound": "issue", "kernel": kernel_name, "kernel_design": A.MODE_NAMES.get(mode_used),
            "achieved": kernel_rate, "peak": trav_best, "unit": "Mrays/s",
            "frac": (kernel_rate / trav_best) if kernel_rate and trav_best else None,
            "peak_source": f"traversal-only microbenchmark measured in this run: {n_rays} coherent primary rays of the same "
                           "camera through nrrt_trace_rays (NRRT_TRACE_COMPACT: closest hit only, 16 B out per ray), best of 6",
            "traffic": traffic,
            "traffic_source": f"profiles/ncu_traffic.json <- {capture}: dram__bytes_read.sum + dram__bytes_write.sum of one launch of "
                              "the same kernel on the same scene and image size (the traffic is the per-item partial sums: it "
                              "scales with the image, not with spp), per rank",
            "ncu_issue_slot_utilisation_pct": issue_pct, "ncu_active_threads_per_instruction": lanes,
            "ncu_useful_lane_slot_frac": (issue_pct / 100.0 * lanes / 32.0) if issue_pct and lanes else None,
            "why_issue": "the scene (KB-MB) lives in L1/L2 and path state in shared memory; DRAM sees only the per-item partial "
                         "sums, so the binding limit is warp-instruction issue x lanes active per instruction, not HBM",
            "hbm": {"algorithmic_gbs": hbm_achieved, "peak_gbs": hbm_peak,
                    "frac": (hbm_achieved / hbm_peak) if hbm_achieved else None,
                    "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650",
                    "note": "algorithmic node/primitive bytes are served by L1/L2, not HBM; reported for scale only"},
            "algorithmic_bytes_per_launch": bytes_seg * (my_segs / max(ext_launches, 1)),
            "bytes_per_segment": bytes_seg, "nodes_per_segment": nodes_seg, "prims_per_segment": prims_seg,
            "exact_box_tests_per_segment": exact_seg, "segments_per_launch": my_segs / max(ext_launches, 1),
            "avg_launch_ms": ext_ms / max(ext_launches, 1), "launches": ext_launches,
            "kernel_share_of_step": ext_ms / sum_ms,
        }
        # ---- CPU baseline on a bounded sample (rank 0, N=1 only)
        cpu = None
        if world == 1 and not args.no_cpu:
            m, dt, s, threads, _ = oracle_sample(args.cpu_spp)
            cpu = {"value": m, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": f"{SCENE} {args.width}x{args.height} depth {DEPTH} at {args.cpu_spp} spp "
                             f"({s} segments in {dt:.1f} s; C++ restatement of the reference algorithm, OpenMP)"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": sum_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{SCENE} {args.width}x{args.height} {args.spp}spp depth{DEPTH}",
                       "kernel_design": A.MODE_NAMES.get(mode_used), "requested_mode": args.mode, "bvh": args.bvh,
                       "partition": f"row-blocks of {R}, round-robin over {world} GPU(s)",
                       "l2": "flushed between timed steps (256 MB write); the scene (KB-MB) is cache-resident by design, path "
                             "state lives in shared memory",
                       "rng": "Philox4x32-10, seed 0"},
            "time_to_image_s": sum_ms / args.steps / 1e3,
            "segments_per_step": segs / args.steps, "paths_per_step": paths / args.steps,
            "segments_per_path": segs / max(paths, 1),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": scene_h2d_bytes(host.desc),
                    "d2h_bytes_per_step": W * H * 3 * 4, "ms_per_step": sum(ms_e2e) / args.steps,
                    "call": "api.Scene(graph).render(out=<pinned host buffer>) — host BVH build + flatten, H2D scene upload, "
                            "nrrt_render with a host out_rgb (D2H inside)" if world == 1 else
                            "api.Scene(graph) per rank + distributed.render_distributed(..., host_out=<pinned>) — render, "
                            "NCCL gather to rank 0, D2H",
                    "pageable_host_buffer_value": e2e_pageable},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu,
        }
        if identical is not None:
            line["multi_gpu_image_identical_to_single_gpu"] = identical
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line))
        if identical is False:
            return 3
    return 0


def main():
    global SCENE, WIDTH, HEIGHT, SPP, DEPTH
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="auto", choices=["auto", "pool", "fused", "wavefront", "megakernel"],
                    help="auto = the product path: pooled kernel on deep trees, fused kernel otherwise")
    ap.add_argument("--bvh", default="reference", choices=["reference", "sah"],
                    help="reference = the reference's tree (parity contract, default); sah = opt-in SAH inner nodes")
    ap.add_argument("--scene", default=SCENE, help="scene file (default: the benchmark workload)")
    ap.add_argument("--depth", type=int, default=DEPTH)
    ap.add_argument("--width", type=int, default=WIDTH)
    ap.add_argument("--height", type=int, default=HEIGHT)
    ap.add_argument("--spp", type=int, default=SPP)
    ap.add_argument("--cpu-spp", type=int, default=128, help="spp of the bounded cpu_baseline sample")
    ap.add_argument("--ref-spp", type=int, default=32, help="spp per step of the --impl reference arm")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (f32 image, f64 "
                         "segment count; at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        args.dump_outputs = os.path.join(CALLER_CWD, args.dump_outputs)
    SCENE, WIDTH, HEIGHT, SPP, DEPTH = args.scene, args.width, args.height, args.spp, args.depth
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
