#!/usr/bin/env python
"""Benchmark of the path-tracing hot path (BASELINE.json metric: Mrays/s and path samples/s at
1080p, depth 8).

    python bench.py --gpus N --steps K --warmup W            # our CUDA core
    python bench.py --impl reference --gpus N --steps K ...   # CPU oracle on the host cores

One STEP = one render of ONE FRAME of the workload (configs[1]: the ABeautifulGame-class chess scene,
1920x1080, `--spp` samples per pixel, depth 8) through `pt_render_samples`, plus — for N > 1 —
the sum-reduce of the float4 accumulation buffer onto rank 0.  At N > 1 the SAME frame is partitioned over
the ranks (strong scaling: image tiles, or sample slices for the street workload — BASELINE configs 4 / 5);
a `weak` block alongside times the round-1 arrangement (every rank adds its own `--spp` samples).

  value  : Mrays/s (closest-hit + occlusion queries of all ranks) over the device time of the
           step: CUDA events recorded by the library on its launching stream around the
           wavefront loop, plus torch CUDA events around the NCCL reduce; max over ranks.
  e2e    : the same metric over wall time of the public call sequence with HOST buffers:
           pt_render_samples (parameters cross host->device) + reduce + pt_readback of the
           accumulation image into pinned host memory.
  roofline: both candidate bounds of SURVEY §8(d) for the dominant kernel — the algorithmic-HBM proxy (bytes
           of the §8d formula with the measured N_box / N_tri / N_texel of this very run / its CUDA-event
           duration / measured HBM peak) and FP32 lane-issue (lane-instructions per ray from the committed ncu
           counters, profiles/r2_kernel_counters.json, x the rays of this run / the same duration / SMs x 128 x
           clock); `bound` names the larger fraction, `traffic` is the kernel's DRAM bytes per launch (ncu).
  parity : the same frame at the CPU baseline's sample count rendered on the GPU and compared with the
           oracle's image (relMSE, LDR-FLIP, fraction of pixels within 1e-3 / 1e-4, first-hit id mismatches).
  cpu_baseline: the CPU oracle (port of the reference's shaders, pinned bit for bit to the reference's compiled
           GLSL: tests/test_oracle_vs_glsl.py) on a bounded sample of the same workload, all host threads.
"""
from __future__ import annotations

import argparse
import contextlib
import ctypes
import importlib
import io
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

POOLS = int(os.environ.get("PT_POOLS", "2"))  # the library's default (core_internal.h: Context::poolCount)
METRIC = "Mrays/s (closest-hit + occlusion rays; path samples/s alongside), 1080p, depth 8"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="chess", choices=["chess", "dragon", "atrium", "street"],
                    help="chess = BASELINE.json configs[1] (the default and the headline); dragon / atrium / street = "
                         "configs[2..4] stand-ins (extra lines, not the headline)")
    ap.add_argument("--spp", type=int, default=None, help="samples per pixel of one step (default: the config's, chess 256)")
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--bounces", type=int, default=None)
    ap.add_argument("--partition", default="auto", choices=["auto", "tiles", "samples"],
                    help="how ONE frame of --spp samples is split over N > 1 GPUs (strong scaling): tiles = 8-row blocks "
                         "dealt round robin (bit-identical to one GPU); samples = sample slices of the whole frame; "
                         "auto = tiles, samples for the street workload (BASELINE configs 4 / 5)")
    ap.add_argument("--scaling", default="both", choices=["strong", "weak", "both"],
                    help="N > 1: which arrangement is timed; the headline is strong unless --scaling weak")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--small", action="store_true", help="reduced tessellation (debugging only; reported in config)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned to its caller as DIR/<name>.npy "
                         "(the float32 accumulation image), so that two builds can be compared output for output")
    args = ap.parse_args()
    scenes = importlib.import_module("path-tracing_b200.scenes")
    _, _, w, h, spp, depth = scenes.WORKLOADS[args.workload]
    args.width, args.height = args.width or w, args.height or h
    args.spp, args.bounces = args.spp or spp, args.bounces or depth
    if args.partition == "auto":
        args.partition = "samples" if args.workload == "street" else "tiles"
    return args


WORKLOAD_LABEL = {
    "chess": "ABeautifulGame-class procedural stand-in",
    "dragon": "DragonAttenuation-class procedural stand-in (transmission + volume attenuation)",
    "atrium": "Sponza-scale procedural stand-in (alpha-tested foliage)",
    "street": "Bistro-scale procedural stand-in (emissive lamps, 64 point lights)",
}


def build_scene(args):
    scenes = importlib.import_module("path-tracing_b200.scenes")
    if args.small:
        assert args.workload == "chess"
        return (scenes.chess_scene(args.width, args.height, segments=48, rings=40, board_tess=32, texture_size=256),
                "chess_scene(small): " + WORKLOAD_LABEL["chess"])
    builder = scenes.WORKLOADS[args.workload][0]
    return builder(args.width, args.height), f"{builder.__name__}: {WORKLOAD_LABEL[args.workload]}"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.proc = None
        self.lines = []
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={device_index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
                power.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": statistics.median(sm) if sm else None,
            "sm_max_mhz": max(smax) if smax else None,
            "power_w_max": max(power) if power else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


DUMP_BYTES = 64 << 20


def dump_outputs(directory: str, arrays: dict):
    """Writes each (H, W, C) array as directory/<name>.npy in float32.  Arrays of more than DUMP_BYTES in all are each
    replaced by a fixed, seeded sample of their pixels, the same on every run (rows of the (H*W, C) view, in pixel order)."""
    os.makedirs(directory, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        a = np.asarray(a, np.float32)
        if total > DUMP_BYTES:
            flat = a.reshape(a.shape[0] * a.shape[1], -1)
            keep = int(len(flat) * DUMP_BYTES / total)
            a = flat[np.sort(np.random.default_rng(0).choice(len(flat), keep, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


class CudaArray:
    """Zero-copy view of a device pointer for torch.as_tensor (__cuda_array_interface__)."""

    def __init__(self, ptr: int, shape, typestr="<f4"):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (ptr, False), "version": 3}


def algorithmic_bytes(st: dict, kernel: str) -> float:
    """SURVEY §8(d) constants, split per kernel class; counters come from a stats run of the same
    (deterministic) workload."""
    rc, rs, hits, samples = st["rays_closest"], st["rays_shadow"], st["hits"], st["samples"]
    if kernel == "extend":  # ray in (32 B) + hit out (16 B) + 32 B per box test + 36 B per triangle test
        return 48.0 * rc + 32.0 * st["box_tests_closest"] + 36.0 * st["tri_tests_closest"] + 184.0 * st["alpha_tests_closest"]
    if kernel == "shade":  # per hit 384 B geometry/material + 4 B per texel; 288 B path state per bounce
        return 384.0 * hits + 4.0 * st["texel_fetches"] + 288.0 * rc
    if kernel == "shadow":
        return 36.0 * rs + 32.0 * st["box_tests_shadow"] + 36.0 * st["tri_tests_shadow"] + 184.0 * st["alpha_tests_shadow"]
    if kernel == "finish":  # accumulation read + write per sample
        return 32.0 * samples
    raise KeyError(kernel)


def load_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def load_kernel_counters(workload: str) -> dict:
    """ncu instruction / DRAM counters per kernel and ray of the workload (profiles/r2_kernel_counters.json,
    collected by tools/ncu_all.sh with the production kernels; see its `note`)."""
    path = os.path.join(ROOT, "profiles", "r2_kernel_counters.json")
    try:
        return json.load(open(path)).get(workload, {}).get("kernels", {})
    except Exception:
        return {}


def probe_lavapipe() -> str:
    """BASELINE.md §4 step 1: is the reference's own CPU path (Vulkan on Mesa lavapipe) runnable on this box?"""
    import ctypes.util
    import glob

    loader = ctypes.util.find_library("vulkan") or next(iter(glob.glob("/usr/lib/*/libvulkan.so.1")), None)
    icds = glob.glob("/usr/share/vulkan/icd.d/lvp_icd*.json") + glob.glob("/etc/vulkan/icd.d/lvp_icd*.json")
    shaderc = ctypes.util.find_library("shaderc_shared") or ctypes.util.find_library("shaderc")
    sdk = os.environ.get("VULKAN_SDK")
    found = [n for n, v in (("libvulkan", loader), ("lvp_icd", icds), ("shaderc", shaderc), ("VULKAN_SDK", sdk)) if v]
    if loader and icds and shaderc:
        return "lavapipe present (" + ", ".join(found) + ") but the reference needs a headless patch to run: not attempted"
    return "lavapipe unavailable (probed at bench time: " + ("found only " + ", ".join(found) if found else "no libvulkan.so.1, lvp_icd*.json, shaderc or VULKAN_SDK") + ")"


def cpu_baseline(scene, params, args, threads=None, tile=(0, 0, 1 << 30, 1 << 30), spp=12):
    """Times the CPU oracle on a bounded sample of the same workload (default: the whole frame at
    `spp` samples per pixel instead of --spp, full depth; 10-30 s of CPU work on a 16-core host)."""
    from oracle import oracle

    threads = threads or os.cpu_count() or 1
    t0 = time.perf_counter()
    o = oracle.OracleScene(scene)
    build_s = time.perf_counter() - t0
    x0, y0, x1, y1 = (min(tile[0], args.width), min(tile[1], args.height), min(tile[2], args.width), min(tile[3], args.height))
    spp = max(1, min(int(round(spp * (1920 * 1080) / (args.width * args.height))), args.spp))
    tiles = np.array([(x0, y0, x1, y1)], importlib.import_module("path-tracing_b200.scene").TILE)
    t0 = time.perf_counter()
    image, cnt = o.render(params, args.width, args.height, 0, spp, tiles=tiles, threads=threads)
    dt = time.perf_counter() - t0
    rays = cnt["rays_closest"] + cnt["rays_shadow"]
    lavapipe = probe_lavapipe()
    return {
        "value": rays / dt / 1e6,
        "unit": "Mrays/s",
        "samples_per_s": cnt["samples"] / dt,
        "cores": threads,
        "kind": "port",
        "sample": f"CPU restatement of the reference shaders ({lavapipe}): pixels [{x0},{x1})x[{y0},{y1}) of the "
                  f"{args.width}x{args.height} frame, {spp} spp, depth {args.bounces}; {rays} rays in {dt:.2f} s "
                  f"(+ {build_s:.1f} s CPU SAH BVH build, not counted)",
        "oracle": o,
        "image": image,
        "spp": spp,
        "full_frame": (x0, y0, x1, y1) == (0, 0, args.width, args.height),
    }


def parity_block(r, oracle_scene, oracle_image, params, W, H, spp):
    """The GPU against the oracle on the benchmarked workload itself: the same `spp` samples of the frame through
    pt_render_samples, and the pixel-centre first hits of the whole frame."""
    metrics = importlib.import_module("path-tracing_b200.metrics")
    r.on_resize(W, H)
    r.render(spp, params=params, first_sample=0)
    img = r.read_accumulation()
    a, b = img[..., :3] / spp, oracle_image[..., :3] / spp
    # LDR-FLIP on (at most) the central 1920 x 1080 pixels: the filters are evaluated in numpy
    y0, x0 = max(0, (H - 1080) // 2), max(0, (W - 1920) // 2)
    crop = (slice(y0, y0 + min(H, 1080)), slice(x0, x0 + min(W, 1920)))
    t0 = time.perf_counter()
    gpu_hits = r.first_hit_aov(params, W, H)
    ora_hits = oracle_scene.first_hit_aov(params, W, H)
    ids_differ = (gpu_hits["instance"] != ora_hits["instance"]) | (gpu_hits["geometry"] != ora_hits["geometry"]) | \
                 (gpu_hits["primitive"] != ora_hits["primitive"])
    hit = ora_hits["instance"] != 0xFFFFFFFF
    same = hit & ~ids_differ
    t_rel = np.abs(gpu_hits["t"][same] - ora_hits["t"][same]) / np.maximum(np.abs(ora_hits["t"][same]), 1e-20)
    return {
        "spp": int(spp),
        "relMSE": metrics.rel_mse(a, b),
        "flip": metrics.flip(a[crop], b[crop]),
        "flip_region": f"LDR-FLIP (Andersson et al. 2020, 67 ppd) of the tone-mapped images, central {min(W, 1920)}x{min(H, 1080)} pixels",
        "mean_radiance_rel_diff": float(abs(a.mean() - b.mean()) / max(b.mean(), 1e-20)),
        "note": "relMSE <= 1e-3 is the bar for converged images at matched spp; at the few samples the CPU leg can afford, the paths "
                "that took another route (1 - close_fraction: a lobe / visibility decision flipped by the last bit) are independent "
                "samples of the same integrand and dominate a squared-error metric where emitters are small and bright",
        "close_fraction_1e-3": metrics.close_fraction(img, oracle_image, 1e-3),
        "close_fraction_1e-4": metrics.close_fraction(img, oracle_image, 1e-4),
        "first_hit_pixels": int(ids_differ.size),
        "first_hit_mismatch": int(ids_differ.sum()),
        "first_hit_t_max_rel_err": float(t_rel.max()) if t_rel.size else 0.0,
        "seconds": time.perf_counter() - t0,
    }


def run_reference(args):
    """--impl reference: the reference semantics on the host CPU (oracle port; the reference's own
    Vulkan path cannot run: no Vulkan loader / lavapipe / shaderc on the box)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    scene, scene_name = build_scene(args)
    params = scene.default_params(args.bounces)
    threads = os.cpu_count() or 1
    step_spp = 2
    base = cpu_baseline(scene, params, args, threads=threads, spp=step_spp)  # also warms the caches
    o = base.pop("oracle")
    base.pop("image")
    tiles = None
    for _ in range(max(0, args.warmup - 1)):
        o.render(params, args.width, args.height, 0, step_spp, tiles=tiles, threads=threads)
    rays = samples = 0
    t0 = time.perf_counter()
    for k in range(args.steps):
        image, cnt = o.render(params, args.width, args.height, k * step_spp, step_spp, tiles=tiles, threads=threads)
        rays += cnt["rays_closest"] + cnt["rays_shadow"]
        samples += cnt["samples"]
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"accumulation": image})
    value = rays / dt / 1e6
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": value,
        "unit": "Mrays/s",
        "samples_per_s": samples / dt,
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"{scene_name}, {args.width}x{args.height}, depth {args.bounces}; "
                               f"each step = {step_spp} spp of the whole frame on the host CPU (bounded sample of the {args.spp}-spp step)",
                   "triangles": scene.instanced_triangle_count()},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": threads, "kind": "port",
                         "sample": f"CPU restatement of the reference shaders ({probe_lavapipe()}): {args.steps} steps x {step_spp} spp of the "
                                   f"whole {args.width}x{args.height} frame, depth {args.bounces}; {rays} rays in {dt:.2f} s on {threads} threads"},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_ours(args):
    import torch
    import torch.distributed as dist

    core = importlib.import_module("path-tracing_b200.core")
    partition = importlib.import_module("path-tracing_b200.partition")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    scene, scene_name = build_scene(args)
    params = scene.default_params(args.bounces)
    W, H, spp = args.width, args.height, args.spp

    r = core.Renderer(local_rank)  # raises if the CUDA library / device is missing: no fallback
    r.update_scene_data(scene)
    r.on_resize(W, H)
    build_stats = r.stats()

    ptr, pitch, _ = r.accum_device_ptr()
    accum_t = torch.as_tensor(CudaArray(ptr, (H, W, 4)), device=torch.device("cuda", local_rank)) if world > 1 else None
    host_img = torch.empty((H, W, 4), dtype=torch.float32).pin_memory()
    host_ptr, host_bytes = host_img.data_ptr(), host_img.numel() * 4

    # ---- the two arrangements of an N-GPU step --------------------------------------------------------
    #   strong: ONE frame of `spp` samples split over the ranks (tiles: disjoint pixels; samples: sample slices)
    #   weak  : every rank renders its own `spp` samples of the whole frame (N * spp per frame)
    def arrangement(kind):
        if world == 1:
            return None, 0, spp
        if kind == "weak":
            return (None,) + partition.sample_slice(0, spp * world, rank, world)
        if args.partition == "tiles":
            return partition.row_block_tiles(W, H, rank, world, block_rows=8), 0, spp
        return (None,) + partition.sample_slice(0, spp, rank, world)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(kind):
        tiles, first, count = arrangement(kind)

        def one_step():
            """Returns (device_ms, e2e_wall_ms, stats) of this rank."""
            t0 = time.perf_counter()
            r.on_resize(W, H)  # accumulation reset (a new render)
            if count > 0:
                r.render(count, tiles=tiles, params=params, first_sample=first)
            st = r.stats()
            dev_ms = st["last_render_ms"] if count > 0 else 0.0
            if world > 1:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                partition.reduce_accumulation(accum_t, dst=0)
                e1.record()
                e1.synchronize()
                dev_ms += e0.elapsed_time(e1)
            r.readback_into(host_ptr, host_bytes)  # D2H of the (reduced) float4 image into pinned memory
            return dev_ms, (time.perf_counter() - t0) * 1e3, st

        for _ in range(args.warmup):
            one_step()
        sampler = ClockSampler(local_rank) if rank == 0 else None
        sync_all()
        wall0 = time.perf_counter()
        m = {"dev_ms": 0.0, "e2e_ms": 0.0, "launches": 0, "rays_c": 0, "rays_s": 0, "samples": 0}
        for _ in range(args.steps):
            dev_ms, e2e_ms, st = one_step()
            m["dev_ms"] += dev_ms
            m["e2e_ms"] += e2e_ms
            m["launches"] += st["kernel_launches"]
            m["rays_c"], m["rays_s"], m["samples"] = m["rays_c"] + st["rays_closest"], m["rays_s"] + st["rays_shadow"], m["samples"] + st["samples"]
        sync_all()
        m["wall_ms"] = (time.perf_counter() - wall0) * 1e3
        m["clocks"] = sampler.stop() if sampler else None
        # aggregate over ranks: times -> max, work -> sum
        if world > 1:
            t = torch.tensor([m["dev_ms"], m["e2e_ms"], m["wall_ms"]], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            m["dev_ms"], m["e2e_ms"], m["wall_ms"] = t.tolist()
            w = torch.tensor([m["rays_c"], m["rays_s"], m["samples"], m["launches"]], dtype=torch.float64, device="cuda")
            dist.all_reduce(w, op=dist.ReduceOp.SUM)
            m["rays_c"], m["rays_s"], m["samples"], m["launches"] = (int(x) for x in w.tolist())
        m["rays"] = m["rays_c"] + m["rays_s"]
        m["value"] = m["rays"] / (m["dev_ms"] * 1e-3) / 1e6
        m["tiles"], m["first"], m["count"] = tiles, first, count
        return m

    head_kind = "weak" if (args.scaling == "weak" and world > 1) else "strong"
    head = measure(head_kind)
    if args.dump_outputs and rank == 0:
        # the last timed step's (reduced) image, written before the weak arrangement reads back into host_img
        dump_outputs(args.dump_outputs, {"accumulation": host_img.numpy()})
    other = None
    if world > 1 and args.scaling == "both":
        other = measure("weak")

    # ---- roofline inputs: one stats run + one kernel-timing run of the headline arrangement (rank 0's share).
    # The timing run uses ONE wavefront pool: with several pools the kernels of different streams
    # overlap and a CUDA-event pair around one launch would also time its neighbours.
    tiles, first, count = head["tiles"], head["first"], head["count"]
    r.set_traversal_stats(True)
    r.on_resize(W, H)
    r.render(count, tiles=tiles, params=params, first_sample=first)
    cst = r.stats()
    r.set_traversal_stats(False)
    r.set_tuning("pools", 1)
    r.set_kernel_timing(True)
    r.on_resize(W, H)
    r.render(count, tiles=tiles, params=params, first_sample=first)
    tst = r.stats()
    r.set_kernel_timing(False)
    r.set_tuning("pools", POOLS)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    peak, peak_src = load_peak()
    counters = load_kernel_counters(args.workload if not args.small else "")
    clk_mhz = (head["clocks"] or {}).get("sm_mhz") or 1965.0
    sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
    issue_peak = sm_count * 128 * clk_mhz * 1e6  # FP32 lanes x clock = lane-instructions / s
    units = {"extend": cst["rays_closest"], "shade": cst["hits"], "shadow": cst["rays_shadow"]}
    kernels = {}
    trace_classes = ("extend", "shade", "shadow")
    total_kernel_ms = sum(tst["kernel_ms"][k] for k in core.KERNEL_CLASSES) or 1.0
    for name in trace_classes:
        ms, n = tst["kernel_ms"][name], max(1, tst["kernel_launch_count"][name])
        nbytes = algorithmic_bytes(cst, name)
        k = {
            "ms_total": ms,
            "launches": n,
            "avg_launch_us": ms / n * 1e3,
            "share": ms / total_kernel_ms,
            "algorithmic_bytes_per_launch": nbytes / n,
            "achieved_gbs": nbytes / (ms * 1e-3) / 1e9 if ms > 0 else None,
            "hbm_frac": nbytes / (ms * 1e-3) / 1e9 / peak if ms > 0 else None,
        }
        c = counters.get("k_" + name)
        if c and ms > 0:
            lane_rate = c["lane_inst_per_unit"] * units[name] / (ms * 1e-3)
            k["issue"] = {
                "lane_instr_per_unit": c["lane_inst_per_unit"],
                "unit": c["unit"],
                "active_lanes_per_inst": c["active_lanes_per_inst"],
                "achieved_Tlane_s": lane_rate / 1e12,
                "peak_Tlane_s": issue_peak / 1e12,
                "frac": lane_rate / issue_peak,
            }
            k["dram_traffic_bytes_per_launch"] = c["dram_bytes_per_unit"] * units[name] / n
            k["dram_frac"] = c["dram_bytes_per_unit"] * units[name] / (ms * 1e-3) / 1e9 / peak
        kernels[name] = k
    # k_resolve (once per round, ~1 ms) reads a sample buffer that is still L2-resident: time share only
    kernels["resolve"] = {"ms_total": tst["kernel_ms"]["finish"], "launches": tst["kernel_launch_count"]["finish"],
                          "share": tst["kernel_ms"]["finish"] / total_kernel_ms}
    dominant = max(trace_classes, key=lambda k: kernels[k]["ms_total"])
    dom = kernels[dominant]
    issue = dom.get("issue")
    # the BINDING roof: real DRAM utilisation (ncu traffic / time / peak) against FP32 lane-issue utilisation; the
    # algorithmic-bytes proxy (`frac`) is kept beside it as SURVEY 8(d) defines it, but it overstates HBM pressure
    # whenever the BVH is served by L1 / L2 (it can exceed 1)
    bound = "issue" if issue and issue["frac"] > (dom.get("dram_frac") or dom["hbm_frac"] or 0.0) else "hbm"
    rays_total = head["rays"]
    samples = head["samples"]
    per_ray = {
        "n_box_closest": cst["box_tests_closest"] / max(1, cst["rays_closest"]),
        "n_tri_closest": cst["tri_tests_closest"] / max(1, cst["rays_closest"]),
        "n_box_shadow": cst["box_tests_shadow"] / max(1, cst["rays_shadow"]),
        "n_tri_shadow": cst["tri_tests_shadow"] / max(1, cst["rays_shadow"]),
        "hit_rate": cst["hits"] / max(1, cst["rays_closest"]),
        "n_texel_per_hit": cst["texel_fetches"] / max(1, cst["hits"]),
        "alpha_tests_per_ray": (cst["alpha_tests_closest"] + cst["alpha_tests_shadow"]) / max(1, cst["rays_closest"] + cst["rays_shadow"]),
        "rays_per_sample": rays_total / max(1, samples),
    }
    all_bytes = sum(algorithmic_bytes(cst, k) for k in trace_classes)

    def workload_text(kind):
        if world == 1:
            return f"{spp} spp per step"
        if kind == "weak":
            return f"{spp} spp per GPU per step ({spp * world} spp per frame: every rank adds its own samples)"
        how = "8-row blocks of the image dealt round robin" if args.partition == "tiles" else "sample slices of the whole frame"
        return f"ONE frame of {spp} spp per step split over {world} GPUs ({how})"

    line = {
        "metric": METRIC,
        "value": head["value"],
        "unit": "Mrays/s",
        "samples_per_s": samples / (head["dev_ms"] * 1e-3),
        "rays_closest": head["rays_c"],
        "rays_shadow": head["rays_s"],
        "samples": samples,
        "n_gpus": world,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": head["dev_ms"] / args.steps,
        "wall_ms_per_step": head["wall_ms"] / args.steps,
        "higher_is_better": True,
        "scaling": head_kind,
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {
            "workload": f"{scene_name}, {W}x{H}, {workload_text(head_kind)}, depth {args.bounces}",
            "triangles": int(build_stats["triangle_count"]),
            "bvh_nodes": int(build_stats["bvh_node_count"]),
            "bvh_bytes": int(build_stats["bvh_bytes"]),
            "materials": int(len(scene.mr_materials)),
            "textures": len(scene.textures),
            "partition": "none" if world == 1 else ("samples (weak)" if head_kind == "weak" else args.partition),
            "l2": f"working set (path state of 8 M paths in flight 2 GB + sample buffer up to 8 GB + triangles/BVH "
                  f"{build_stats['bvh_bytes'] / 1e9:.2f} GB + textures) exceeds the 126 MB L2 many times over; no explicit flush",
            "scheduling": f"8 M path slots in {POOLS} wavefront pools on {POOLS} CUDA streams, paths regenerated inside k_extend, "
                          "hits shaded in triangle order",
            "bvh_build_ms": build_stats["bvh_build_ms"],
            "scene_upload_ms": build_stats["scene_upload_ms"],
        },
        "per_ray": per_ray,
        "roofline": {
            "bound": bound,
            "kernel": f"k_{dominant}",
            "timing": "CUDA events on the launching stream around every launch of a separate, identical render with ONE "
                      f"wavefront pool (kernels of different pools overlap otherwise); value/ms_per_step come from the {POOLS}-pool runs",
            "achieved": dom["achieved_gbs"],
            "peak": peak,
            "unit": "GB/s",
            "frac": dom["hbm_frac"],
            "peak_source": peak_src,
            "note": "achieved / peak / frac are the ALGORITHMIC-bytes proxy of SURVEY 8(d) (what HBM would have to stream if nothing "
                    "were cached); the BVH and triangles are served by L1 / L2, so DRAM traffic is `traffic` (dram_frac of the peak) "
                    "and the kernel is bound by issue and load latency under divergence: see `issue` (FP32 lane-instructions / s "
                    "against SMs x 128 x clock) and active_lanes_per_inst",
            "traffic": dom.get("dram_traffic_bytes_per_launch"),
            "issue": issue,
            "all_kernels_achieved_gbs": all_bytes / (total_kernel_ms * 1e-3) / 1e9,
            "kernels": kernels,
            "counters_source": "profiles/r2_kernel_counters.json (tools/ncu_all.sh: ncu smsp__inst_executed / smsp__thread_inst_executed / "
                               "dram__bytes per kernel of a one-pool render of this workload, divided by its rays)" if counters else None,
        },
        "e2e": {
            "value": rays_total / (head["e2e_ms"] * 1e-3) / 1e6,
            "unit": "Mrays/s",
            "ms_per_step": head["e2e_ms"] / args.steps,
            "h2d_bytes_per_step": int(params.nbytes()),
            "d2h_bytes_per_step": int(host_bytes),
        },
        "gpu_launches": int(head["launches"]),
        "clocks": head["clocks"],
    }
    if other is not None:
        line["weak"] = {
            "scaling": "weak",
            "value": other["value"],
            "unit": "Mrays/s",
            "ms_per_step": other["dev_ms"] / args.steps,
            "e2e_value": other["rays"] / (other["e2e_ms"] * 1e-3) / 1e6,
            "samples": other["samples"],
            "workload": workload_text("weak"),
            "clocks": other["clocks"],
        }
    if not args.no_cpu_baseline and world == 1:  # the CPU baseline is a rank-0, N = 1 leg
        base = cpu_baseline(scene, params, args)
        o, image, base_spp, full = base.pop("oracle"), base.pop("image"), base.pop("spp"), base.pop("full_frame")
        line["cpu_baseline"] = base
        if not args.no_parity and full:
            line["parity"] = parity_block(r, o, image, params, W, H, base_spp)
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to fd 1 when
    # the box sets NCCL_DEBUG): while the bench runs, fd 1 is stderr; the line goes to the saved descriptor.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        buf = io.StringIO()
        with contextlib.redirect_stdout(buf):
            if args.impl == "reference":
                run_reference(args)
            else:
                run_ours(args)
        sys.stdout.flush()
    finally:
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    sys.stdout.write(buf.getvalue())
    sys.stdout.flush()


if __name__ == "__main__":
    main()
