#!/usr/bin/env python
"""Cost and benefit of the emissive-MIS light sampling (pt_set_light_sampling, DESIGN.md §3g) on one GPU:
    python tools/emissive_nee_bench.py [--width 1920 --height 1080] [--ref-spp 4096] [--out DIR]
Street workload (its builder's default geometry) at the given size, in both modes:
  * Mrays/s (library CUDA-event time of the wavefront loop) and k_shade time (per-kernel CUDA events, separate render);
  * relMSE at 16 and 64 spp against the same mode's --ref-spp image, and the equal-time efficiency 1 / (relMSE x time);
  * the mean-radiance difference between the two modes' --ref-spp images;
  * the emitter-table build time after the upload and after a pt_scene_update.
Chess, dragon and atrium (no emitters: the mode renders them with the reference kernel): Mrays/s in both modes.
Prints one JSON object, with the card's name and power limit read in the same run; --out also writes it there."""
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
MODES = ("reference", "emissive_mis")


def card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unavailable"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def render(r, params, w, h, spp, timing=False):
    r.set_kernel_timing(timing)
    r.on_resize(w, h)
    r.render(spp, params=params, first_sample=0)
    st = r.stats()
    r.set_kernel_timing(False)
    return r.read_accumulation()[..., :3] / spp, st


def mrays(st):
    return (st["rays_closest"] + st["rays_shadow"]) / (st["last_render_ms"] * 1e3)


def street(a):
    w, h = a.width, a.height
    scene = scenes.street_scene(w, h)
    depth = scenes.WORKLOADS["street"][5]
    params = scene.default_params(depth)
    r = core.Renderer(0)
    out = {"workload": f"street_scene(default geometry), {w}x{h}, depth {depth}"}
    try:
        r.update_scene_data(scene)
        t0 = time.perf_counter()
        table = r.emitter_table()
        out["emitters"] = int(len(table["flat_ids"]))
        out["table_build_ms_after_upload"] = (time.perf_counter() - t0) * 1e3
        r.update_scene(instance_transforms=scene.instances["transform"])
        t0 = time.perf_counter()
        r.emitter_table()
        out["table_build_ms_after_scene_update"] = (time.perf_counter() - t0) * 1e3
        for mode in MODES:
            r.set_light_sampling(mode)
            render(r, params, w, h, 2)  # warm-up (and, in the new mode, the table build)
            m = {}
            _, st = render(r, params, w, h, 16)
            m["mrays_per_s"] = mrays(st)
            _, st = render(r, params, w, h, 16, timing=True)
            m["k_shade_ms_per_spp"] = st["kernel_ms"]["shade"] / 16
            ref, st = render(r, params, w, h, a.ref_spp)
            m["ref_spp"], m["ref_render_s"], m["ref_mean_radiance"] = a.ref_spp, st["last_render_ms"] / 1e3, float(ref.mean())
            for spp in (16, 64):
                img, st = render(r, params, w, h, spp)
                e = float(metrics.rel_mse(img, ref))
                m[f"relmse_{spp}spp"] = e
                m[f"render_s_{spp}spp"] = st["last_render_ms"] / 1e3
                m[f"efficiency_{spp}spp"] = 1.0 / (e * st["last_render_ms"] / 1e3)
            out[mode] = m
        ref_mean, mis_mean = out["reference"]["ref_mean_radiance"], out["emissive_mis"]["ref_mean_radiance"]
        out["mean_radiance_rel_difference"] = (mis_mean - ref_mean) / ref_mean
        for spp in (16, 64):
            out[f"efficiency_gain_{spp}spp"] = out["emissive_mis"][f"efficiency_{spp}spp"] / out["reference"][f"efficiency_{spp}spp"]
    finally:
        r.close()
    return out


def others(spp):
    out = {}
    for name in ("chess", "dragon", "atrium"):
        builder, _, w, h, _, depth = scenes.WORKLOADS[name]
        scene = builder(w, h)
        params = scene.default_params(depth)
        r = core.Renderer(0)
        try:
            r.update_scene_data(scene)
            res = {}
            for rep in range(2):  # alternate the modes, two rounds
                for mode in MODES:
                    r.set_light_sampling(mode)
                    render(r, params, w, h, 2)
                    _, st = render(r, params, w, h, spp)
                    res.setdefault(mode, []).append(mrays(st))
            out[name] = {"size": f"{w}x{h}, {spp} spp, depth {depth}", **{m: max(v) for m, v in res.items()}}
        finally:
            r.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--ref-spp", type=int, default=4096)
    ap.add_argument("--other-spp", type=int, default=16)
    ap.add_argument("--out", default=None, help="directory for emissive_nee_bench.json")
    a = ap.parse_args()
    result = {"card": card(), "street": street(a), "mode_cost_without_emitters": others(a.other_spp)}
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "emissive_nee_bench.json"), "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
