"""The cases the oracle is compared on with the reference's compiled shaders (oracle/_ref/libglsl_ref.so):
shared by tests/test_oracle_vs_glsl.py (live comparison, where the library exists) and
tests/golden/make_glsl_vectors.py (golden vectors that travel to machines without the reference), and the recorded
digests that let the live comparisons of test_oracle_vs_glsl.py and test_oracle_vs_glsl_compute.py run without it."""
import hashlib
import importlib
import json
import os

import numpy as np

import unit_inputs as ui

pkg = importlib.import_module("path-tracing_b200")
scenes = importlib.import_module("path-tracing_b200.scenes")
sc = importlib.import_module("path-tracing_b200.scene")

GOLDEN_RECORDS = 256  # per mode in the golden file


def stage_scenes(default_scene):
    """name -> (scene, params, width, height, first_sample, frames, samples_per_frame)"""
    out = {}
    out["default"] = (default_scene, default_scene.default_params(bounce_count=8), 48, 48, 0, 3, 1)
    out["default_spp3"] = (default_scene, default_scene.default_params(bounce_count=8), 32, 32, 5, 2, 3)
    fs = scenes.feature_scene(width=40, height=30)
    p = fs.default_params(bounce_count=8)
    out["feature"] = (fs, p, 40, 30, 0, 2, 1)
    pl = fs.default_params(bounce_count=5)
    pl.lens_radius, pl.focal_distance, pl.hit_flags = 0.05, 5.0, sc.HIT_FLAGS_DX_NORMAL_TEXTURES
    out["feature_lens_dx_spp2"] = (fs, pl, 40, 30, 2, 2, 2)
    return out


def closest_hit_inputs(oracle_scene, oracle_mod, params, width, height, frame=0):
    """Pixel-centre primary rays of a width x height frame that hit something: (hits, rays6, payload_in)
    with the payload raygen.rgen:56-67 hands to the first traceRayEXT."""
    aov = oracle_scene.first_hit_aov(params, width, height).reshape(-1)
    ys, xs = np.divmod(np.arange(width * height, dtype=np.uint32), np.uint32(width))
    rec = np.zeros((width * height, 42), np.float32)
    rec[:, 0], rec[:, 1] = xs.view(np.float32), ys.view(np.float32)
    rec[:, 2] = np.full(width * height, width, np.uint32).view(np.float32)
    rec[:, 3] = np.full(width * height, height, np.uint32).view(np.float32)
    rec[:, 4:6] = 0.5
    rec[:, 10:26] = np.asarray(params.view_inverse, np.float32).reshape(-1)
    rec[:, 26:42] = np.asarray(params.proj_inverse, np.float32).reshape(-1)
    rays = oracle_mod.test_shading(12, rec)  # ray o,d; rx o,d; ry o,d
    rng = oracle_mod.test_shading(11, np.column_stack([rec[:, 0], rec[:, 1], rec[:, 2], np.full(len(rec), frame, np.uint32).view(np.float32)]))
    payload = np.zeros((width * height, 36), np.float32)
    payload[:, 15] = rng[:, 0]  # RngState (bits)
    payload[:, 19] = -1.0  # DirectLightPdf
    payload[:, 24:27], payload[:, 27] = rays[:, 6:9], rays[:, 9]  # RayDifferentials0 = (rx.Origin, rx.Direction.x)
    payload[:, 28:30], payload[:, 30:32] = rays[:, 10:12], rays[:, 12:14]
    payload[:, 32], payload[:, 33:36] = rays[:, 14], rays[:, 15:18]
    hit = aov["instance"] != 0xFFFFFFFF
    return aov[hit], rays[hit, :6], payload[hit]


# ---- the debug pipeline (Debug/debug*.r*): (render mode, raygen flags, hit-group flags) ------------------------------
DEBUG_MODES = ("color", "world_position", "normal", "texture_coords", "mips", "geometry", "primitive", "instance")
DEBUG_FLAG_SETS = ((0, 0), (1, 0), (2, 0), (3, 0x1F), (0, 0x04), (0, 0x08), (0, 0x01 | 0x02), (0, 0x10))
# the combinations whose images travel as golden vectors
DEBUG_GOLDEN = (("default", "color", 0, 0), ("feature", "color", 0, 0), ("feature", "color", 2, 0x10), ("feature", "normal", 1, 0x02),
                ("feature", "mips", 0, 0), ("feature", "instance", 0, 0), ("feature", "primitive", 3, 0x1F))


def debug_key(scene, mode, raygen_flags, hit_flags):
    return f"dbg_{scene}_{mode}_{raygen_flags}_{hit_flags}"


# ---- recorded outputs of the compiled shaders (tests/golden/glsl_digests.json, make_glsl_digests.py) --------------------
DIGESTS_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "glsl_digests.json")
RECORD = os.environ.get("PT_RECORD_GLSL_DIGESTS") == "1"


def digest(a) -> str:
    """SHA-256 of a float32 array's shape and bits, every NaN written as one NaN (the comparisons let any NaN equal any NaN)."""
    a = np.array(a, np.float32)
    a[np.isnan(a)] = np.nan
    return hashlib.sha256(repr(a.shape).encode() + a.tobytes()).hexdigest()


def check_recorded(key, got, want, compare, what):
    """`got` (the oracle's) against the compiled shaders' output on the same input.  Where the library is built, `want` is
    that output: compare(got, want, what), and the digest recorded under `key` must still be want's.  Without the library
    `want` is None and got's digest must be the recorded one."""
    if want is not None:
        compare(got, want, what)
    value = digest(got if want is None else want)
    recorded = json.load(open(DIGESTS_PATH)) if os.path.exists(DIGESTS_PATH) else {}
    if RECORD:
        recorded[key] = value
        with open(DIGESTS_PATH, "w") as f:
            json.dump(recorded, f, indent=1, sort_keys=True)
            f.write("\n")
        return
    assert value == recorded[key], (f"{what}: not the compiled shaders' output recorded in tests/golden/glsl_digests.json "
                                    f"under '{key}'" + (" (the record is stale: tests/golden/make_glsl_digests.py)" if want is not None else ""))
