"""Cost and benefit of the temporal denoiser (pt_denoise_temporal, DESIGN.md §3j) on chess and street at 1920x1080.

For each scene, in one process on one GPU: the time of one pt_denoise_temporal call (K = 5, suggested sigmas, alpha 0.2)
from the host clock around the synchronising call with no host copy, alternating between two cameras one pixel apart so
that every timed call reprojects; the kernel split from torch.profiler in a separate run; the history's bytes; and over a
16-frame pan of about one pixel per frame at 1 spp per frame, relMSE and FLIP of the noisy frame, pt_denoise of it and
the temporal result at frames 1, 4 and 16 against 1024-spp renders at those frames' cameras (the frames use samples the
references did not).  Street renders in the emissive-MIS light-sampling mode.  Prints one JSON line per scene and writes
them to --out."""
import argparse
import ctypes as C
import dataclasses
import importlib
import json
import math
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

FRAMES = 16
CHECKPOINTS = (1, 4, 16)


def card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unavailable"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def panned(p, yaw_deg):
    """p with the camera turned by yaw_deg about its own up axis."""
    m = np.asarray(p.view_inverse, np.float64).reshape(4, 4).T
    c, s = math.cos(math.radians(yaw_deg)), math.sin(math.radians(yaw_deg))
    rot = np.eye(4)
    rot[0, 0], rot[0, 2], rot[2, 0], rot[2, 2] = c, s, -s, c
    return dataclasses.replace(p, view_inverse=(m @ rot).T.astype(np.float32).reshape(-1))


def pixel_yaw(p, w):
    """The yaw that moves the image centre by about one pixel: proj_inverse[0] is tan of half the horizontal field."""
    return math.degrees(math.atan(2.0 * float(np.asarray(p.proj_inverse)[0]) / w))


def temporal_device(r, params, d, t, spp):
    """pt_denoise_temporal without the host copy of the result (out_rgba = NULL)."""
    p = params.to_c()
    r._check(r._L.pt_denoise_temporal(r._h, C.addressof(p), C.addressof(d), C.addressof(t), spp, None, 0))


def time_temporal(r, cams, spp, calls):
    import torch
    from torch.profiler import ProfilerActivity, profile

    d = core.DenoiseParams(5, 4.0, 128.0, 1.0)
    t = core.TemporalParams(0.2, 0.2, 0)
    for k in range(3):
        temporal_device(r, cams[k % 2], d, t, spp)
    t0 = time.perf_counter()
    for k in range(calls):
        temporal_device(r, cams[k % 2], d, t, spp)  # ends in a stream synchronise
    wall_ms = (time.perf_counter() - t0) * 1e3 / calls
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for k in range(calls):
            temporal_device(r, cams[k % 2], d, t, spp)
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        if "denoise" in e.key or "atrous" in e.key or "temporal" in e.key or "Memcpy DtoD" in e.key:
            if "Memcpy" in e.key:
                name = "copy of the (N, t) taps"
            elif "guides" in e.key:
                name = "k_denoise_guides"
            else:
                name = "k_" + e.key.split("k_")[-1].split("(")[0].split("E")[0]
            dt = getattr(e, "device_time_total", None) or e.cuda_time_total
            kernels[name] = kernels.get(name, 0.0) + dt / 1e3 / calls
    return {"call_ms": wall_ms, "kernel_ms": {k: round(v, 4) for k, v in kernels.items()}}


def run(name, w, h, mode, calls, ref_spp):
    builder, _, _, _, _, depth = scenes.WORKLOADS[name]
    s = builder(w, h)
    p = s.default_params(depth)
    step = pixel_yaw(p, w)
    cams = [panned(p, step * k) for k in range(FRAMES)]
    r = core.Renderer(0)
    try:
        r.update_scene_data(s)
        r.set_light_sampling(mode)
        r.on_resize(w, h)
        r.render(2, params=p, first_sample=0)  # warm-up
        r.on_resize(w, h)
        r.render(16, params=p, first_sample=0)
        sample_ms = r.stats()["last_render_ms"] / 16
        out = {"scene": name, "extent": [w, h], "light_sampling": mode, "sample_ms": sample_ms, "pan_deg_per_frame": step,
               "history_bytes": w * h * (3 * 16 + 2 * 8)}
        r.on_resize(w, h)
        r.render(1, params=cams[0], first_sample=0)
        out.update(time_temporal(r, cams[:2], 1, calls))
        out["temporal_over_1_sample"] = out["call_ms"] / sample_ms
        refs = {}
        for k in CHECKPOINTS:
            r.on_resize(w, h)
            r.render(ref_spp, params=cams[k - 1], first_sample=0)
            refs[k] = r.read_accumulation()[..., :3] / ref_spp
        for k, cam in enumerate(cams, 1):
            r.on_resize(w, h)
            r.render(1, params=cam, first_sample=ref_spp + k)
            temporal = r.denoise_temporal(cam, total_samples=1, reset=(k == 1))[..., :3]
            if k not in CHECKPOINTS:
                continue
            noisy = r.read_accumulation()[..., :3]
            spatial = r.denoise(cam, total_samples=1)[..., :3]
            ref = refs[k]
            q = {}
            for label, img in (("noisy", noisy), ("spatial", spatial), ("temporal", temporal)):
                q[f"{label}_relmse"] = metrics.rel_mse(img, ref)
                q[f"{label}_flip"] = metrics.flip(img, ref)
            q["temporal_over_spatial_relmse"] = q["temporal_relmse"] / q["spatial_relmse"]
            out[f"frame{k}"] = {kk: round(float(v), 5) for kk, v in q.items()}
        return out
    finally:
        r.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--ref-spp", type=int, default=1024)
    ap.add_argument("--scenes", default="chess,street")
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    a = ap.parse_args()
    info = card()
    lines = []
    for name in a.scenes.split(","):
        res = run(name, a.width, a.height, "emissive_mis" if name == "street" else "reference", a.calls, a.ref_spp)
        res["card"] = info
        lines.append(json.dumps(res))
        print(lines[-1], flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
