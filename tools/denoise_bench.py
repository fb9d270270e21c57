"""Cost and benefit of the denoiser (pt_denoise, DESIGN.md §3h) on chess and street at 1920x1080.

For each scene, in one process on one GPU: the time of pt_denoise (K = 5, suggested sigmas) over repeated calls after
warm-up, split into the guide pass and the filter by torch.profiler's device times; the time of one rendered sample at
the same extent; relMSE and FLIP of noisy and denoised images at 1, 4 and 16 spp against a 1024-spp render (the noisy
images use samples the reference did not).  Street renders in the emissive-MIS light-sampling mode.  Prints one JSON
line per scene and writes them to --out."""
import argparse
import ctypes as C
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


def card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unavailable"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def denoise_device(r, params, d, spp):
    """pt_denoise without the host copy of the result (out_rgba = NULL)."""
    p = params.to_c()
    r._check(r._L.pt_denoise(r._h, C.addressof(p), C.addressof(d), spp, None, 0))


def time_denoise(r, params, spp, calls):
    import torch
    from torch.profiler import ProfilerActivity, profile

    d = core.DenoiseParams(5, 4.0, 128.0, 1.0)
    for _ in range(3):
        denoise_device(r, params, d, spp)
    t0 = time.perf_counter()
    for _ in range(calls):
        denoise_device(r, params, d, spp)  # ends in a stream synchronise
    wall_ms = (time.perf_counter() - t0) * 1e3 / calls
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            denoise_device(r, params, d, spp)
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        if "denoise" in e.key or "atrous" in e.key:
            name = "k_denoise_guides" if "guides" in e.key else e.key.split("k_")[-1].split("(")[0].split("E")[0]
            t = getattr(e, "device_time_total", None) or e.cuda_time_total
            kernels[name] = kernels.get(name, 0.0) + t / 1e3 / calls
    guides = kernels.get("k_denoise_guides", 0.0)
    return {"call_ms": wall_ms, "guides_ms": guides, "filter_ms": sum(kernels.values()) - guides,
            "kernel_ms": {k: round(v, 4) for k, v in kernels.items()}}


def run(name, w, h, mode, calls, ref_spp):
    builder, _, _, _, _, depth = scenes.WORKLOADS[name]
    s = builder(w, h)
    p = s.default_params(depth)
    r = core.Renderer(0)
    try:
        r.update_scene_data(s)
        r.set_light_sampling(mode)
        r.on_resize(w, h)
        r.render(2, params=p, first_sample=0)  # warm-up
        r.on_resize(w, h)
        r.render(16, params=p, first_sample=0)
        sample_ms = r.stats()["last_render_ms"] / 16
        out = {"scene": name, "extent": [w, h], "light_sampling": mode, "sample_ms": sample_ms}
        out.update(time_denoise(r, p, 16, calls))
        out["denoise_over_4_samples"] = out["call_ms"] / (4 * sample_ms)
        r.on_resize(w, h)
        r.render(ref_spp, params=p, first_sample=0)
        ref = r.read_accumulation()[..., :3] / ref_spp
        for spp in (1, 4, 16):
            r.on_resize(w, h)
            r.render(spp, params=p, first_sample=ref_spp)
            noisy = r.read_accumulation()[..., :3] / spp
            den = r.denoise(p, total_samples=spp)[..., :3]
            q = {"noisy_relmse": metrics.rel_mse(noisy, ref), "denoised_relmse": metrics.rel_mse(den, ref),
                 "noisy_flip": metrics.flip(noisy, ref), "denoised_flip": metrics.flip(den, ref)}
            q["relmse_gain"] = q["noisy_relmse"] / q["denoised_relmse"]
            out[f"spp{spp}"] = {k: round(float(v), 5) for k, v in q.items()}
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
