"""Cost and benefit of adaptive sampling (pt_render_adaptive, DESIGN.md §3i) on chess and street at 1920x1080.

For each scene and threshold, in one process on one GPU: the time of one adaptive call (min 16, max 1024, batch 16 spp,
the default min_pass_items) on a fresh target, its passes and its mean and maximum samples per pixel; relMSE and FLIP of
its mean image against a 1024-spp render of independent samples, beside uniform renders at equal samples and at equal
time; and, in a separate profiled call, the device time of the new kernels (k_adaptive_*, the scan, k_resolve<true>) as
a share of that profiled call's wall time.  Street renders in the emissive-MIS light-sampling mode.  Prints one JSON line
per scene and threshold and writes them to --out."""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

scenes = importlib.import_module("path-tracing_b200.scenes")
core = importlib.import_module("path-tracing_b200.core")
metrics = importlib.import_module("path-tracing_b200.metrics")

REF_FIRST = 1 << 20  # the reference's samples start here: independent of the samples 0.. the compared images use


def card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unavailable"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def quality(img, ref):
    return {"relmse": round(float(metrics.rel_mse(img, ref)), 5), "flip": round(float(metrics.flip(img, ref)), 5)}


def uniform(r, p, w, h, spp, ref):
    r.on_resize(w, h)
    r.render(spp, params=p)
    out = {"spp": spp, "call_ms": round(r.stats()["last_render_ms"], 2)}
    out.update(quality(r.read_accumulation()[..., :3] / np.float32(spp), ref))
    return out


def kernel_share(r, p, w, h, kw):
    """Device time of the new kernels in one adaptive call, from torch.profiler, over the wall time of that profiled call."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    r.on_resize(w, h)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        t0 = time.perf_counter()
        r.render_adaptive(params=p, **kw)
        wall = (time.perf_counter() - t0) * 1e3
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        # the pass's scan is CUB's DeviceScan (the hit sort uses DeviceRadixSort kernels, which do not match)
        for k in ("k_adaptive_blocks", "k_adaptive_select", "DeviceScan", "k_adaptive_scatter", "k_adaptive_mean", "k_resolve<true>"):
            if k in e.key:
                t = getattr(e, "device_time_total", None) or e.cuda_time_total
                kernels[k] = kernels.get(k, 0.0) + t / 1e3
    return {"profiled_call_ms": round(wall, 2), "kernel_ms": {k: round(v, 3) for k, v in kernels.items()},
            "new_kernels_share": round(sum(kernels.values()) / wall, 5)}


def run(name, w, h, mode, thresholds, ref_spp):
    builder, _, _, _, _, depth = scenes.WORKLOADS[name]
    s = builder(w, h)
    p = s.default_params(depth)
    r = core.Renderer(0)
    out = []
    try:
        r.update_scene_data(s)
        r.set_light_sampling(mode)
        r.on_resize(w, h)
        r.render(2, params=p, first_sample=0)  # warm-up
        r.on_resize(w, h)
        r.render(16, params=p, first_sample=0)
        sample_ms = r.stats()["last_render_ms"] / 16
        r.on_resize(w, h)
        r.render(ref_spp, params=p, first_sample=REF_FIRST)
        ref = r.read_accumulation()[..., :3] / np.float32(ref_spp)
        for t in thresholds:
            kw = dict(min_samples=16, max_samples=1024, batch=16, threshold=t)
            r.on_resize(w, h)
            r.render_adaptive(params=p, min_samples=2, max_samples=2, batch=1, threshold=t)  # warm-up of the new kernels
            r.on_resize(w, h)
            t0 = time.perf_counter()
            info = r.render_adaptive(params=p, **kw)
            call_ms = (time.perf_counter() - t0) * 1e3  # the call ends in a stream synchronise
            counts = r.sample_counts()
            img = r.read_accumulation()[..., :3] / counts[..., None].astype(np.float32)
            res = {"scene": name, "extent": [w, h], "light_sampling": mode, "threshold": t, "params": kw, "info": info,
                   "call_ms": round(call_ms, 2), "stats_ms": round(r.stats()["last_render_ms"], 2),
                   "mean_spp": round(float(counts.mean()), 3), "max_spp": int(counts.max()),
                   "sample_ms": round(sample_ms, 4)}
            res.update(quality(img, ref))
            res["uniform_equal_samples"] = uniform(r, p, w, h, max(1, int(round(info["samples"] / (w * h)))), ref)
            res["uniform_equal_time"] = uniform(r, p, w, h, max(1, int(round(call_ms / sample_ms))), ref)
            res.update(kernel_share(r, p, w, h, kw))
            out.append(res)
        return out
    finally:
        r.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--ref-spp", type=int, default=1024)
    ap.add_argument("--thresholds", default="0.05,0.02")
    ap.add_argument("--scenes", default="chess,street")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    a = ap.parse_args()
    info = card()
    lines = []
    for name in a.scenes.split(","):
        mode = "emissive_mis" if name == "street" else "reference"
        for res in run(name, a.width, a.height, mode, [float(t) for t in a.thresholds.split(",")], a.ref_spp):
            res["card"] = info
            lines.append(json.dumps(res))
            print(lines[-1], flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
