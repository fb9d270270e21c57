"""The temporal denoiser (pt_denoise_temporal, DESIGN.md §3j) in the CUDA core: each call against the numpy reference
(tests/temporal_ref.py) stepped from the library's own previous state, the static-camera closed form, disocclusion, the
history's lifetime, image quality against 1024-spp renders, the contract with the rest of the API, and the kernels' spills."""
import ctypes as C
import dataclasses
import importlib
import math
import re

import numpy as np
import pytest

import conftest
import denoise_ref as dr
import emissive_scenes as es
import metrics
import temporal_ref as tr
import test_kernel_budgets

pytestmark = pytest.mark.gpu
core = conftest.core
scenes = importlib.import_module("path-tracing_b200.scenes")
W, H = 160, 120
F = np.float32


def moved(p, yaw_deg=0.0, right=0.0):
    """p with the camera turned by yaw_deg about its own up axis after moving `right` along its own x axis."""
    m = np.asarray(p.view_inverse, np.float64).reshape(4, 4).T
    c, s = math.cos(math.radians(yaw_deg)), math.sin(math.radians(yaw_deg))
    rot = np.eye(4)
    rot[0, 0], rot[0, 2], rot[2, 0], rot[2, 2] = c, s, -s, c
    shift = np.eye(4)
    shift[0, 3] = right
    return dataclasses.replace(p, view_inverse=(m @ shift @ rot).T.astype(F).reshape(-1))


def open_renderer(s, w=W, h=H):
    r = core.Renderer(0)
    r.update_scene_data(s)
    r.on_resize(w, h)
    return r


def frame(r, p, first, spp=2, **kw):
    """One preview frame: restart the accumulation, render spp samples from `first`, denoise temporally."""
    r.on_resize(r.width, r.height)
    r.render(spp, params=p, first_sample=first)
    return r.denoise_temporal(p, total_samples=spp, **kw)


def guide_arrays(g):
    albedo_t = np.concatenate([g["albedo"], g["t"][..., None]], -1)
    normal = np.concatenate([g["normal"], np.zeros(g["t"].shape + (1,), F)], -1)
    return albedo_t, normal


def device_state(r, p, prepared):
    """The library's state after a call, in temporal_ref's form."""
    hist = r.temporal_history()
    return {"view": np.asarray(p.view_inverse, F), "proj": np.asarray(p.proj_inverse, F), "t": prepared["t"], "n": prepared["n"],
            "irr": np.concatenate([hist["irradiance"], hist["length"][..., None]], -1), "moments": hist["moments"]}


def close(got, want):
    return np.abs(got - want) <= 1e-4 * np.maximum(1.0, np.abs(want))


def feature_path(p, t_scale):
    """Six cameras: a pan, then sideways moves large enough to disocclude."""
    return [p, moved(p, 1.5), moved(p, 3.0), moved(p, 4.5), moved(p, 4.5, 0.04 * t_scale), moved(p, 4.5, 0.08 * t_scale)]


@pytest.fixture(scope="module")
def feature():
    s = scenes.feature_scene()
    p = s.default_params(8)
    r = open_renderer(s)
    r.render(1, params=p)
    r.denoise(p, 0, total_samples=1)
    t = r.denoise_guides()["t"]
    yield s, r, p, float(np.median(t[t >= 0]))
    r.close()


def test_each_call_matches_the_reference(feature):
    s, r, p, depth = feature
    prev = None
    for k, cam in enumerate(feature_path(p, depth)):
        out = frame(r, cam, 2 * k, reset=(k == 0))
        g = r.denoise_guides()
        albedo_t, normal = guide_arrays(g)
        prepared = dr.prepare(r.read_accumulation(), 2, albedo_t, normal)
        want = tr.step(prepared, cam.view_inverse, cam.proj_inverse, prev)
        got = device_state(r, cam, prepared)
        ok = ~want["mark"]
        n_got, n_want = got["irr"][..., 3], want["irr"][..., 3]
        print(f"call {k}: {want['mark'].sum()} marked pixels, mean n {n_got[prepared['valid']].mean():.3f}, "
              f"n = 1 on {(n_got == 1).sum()} pixels")
        assert want["mark"].mean() < 1e-3, k
        assert np.array_equal(n_got[ok], n_want[ok]), (k, np.abs(n_got - n_want)[ok].max())
        assert close(got["irr"][..., :3], want["irr"][..., :3])[ok].all(), k
        assert close(got["moments"], want["moments"])[ok].all(), k
        # the filter on the library's own state (a marked pixel would spread through the a-trous taps otherwise)
        ref_out = tr.filter_state(prepared, albedo_t, got)
        assert np.array_equal(np.isnan(out), np.isnan(ref_out)), k
        fin = ~np.isnan(ref_out)
        assert close(out[fin], ref_out[fin]).all(), (k, (np.abs(out - ref_out)[fin] / np.maximum(1.0, np.abs(ref_out[fin]))).max())
        if k >= 1:
            assert (n_got[prepared["valid"]] > 1).mean() > 0.5, k  # the history is used
        prev = got


def test_static_camera_is_the_running_mean(feature):
    s, r, p, _ = feature
    means = []
    for k in range(8):
        out = frame(r, p, 2 * k, iterations=0, alpha=0.0, alpha_moments=0.0, reset=(k == 0))
        means.append(r.read_accumulation()[..., :3] / F(2))
    want = np.mean(np.stack(means).astype(np.float64), 0)
    n = r.temporal_history()["length"]
    hit = r.denoise_guides()["t"] >= 0
    assert hit.any() and (~hit).any()
    assert (n[hit] == 8).all() and (n[~hit] == 0).all()
    assert np.allclose(out[hit][:, :3], want[hit], rtol=1e-5, atol=1e-7)
    assert np.array_equal(out[~hit][:, :3], means[-1][~hit])


def test_disocclusion_rejects_the_history(feature):
    s, r, p, depth = feature
    # a sideways pan: what enters the image at one side has no history
    p1 = moved(p, 3.0)
    frame(r, p, 0, reset=True)
    frame(r, p1, 2)
    g = r.denoise_guides()
    n = r.temporal_history()["length"]
    rp = tr.reproject(p1.view_inverse, p1.proj_inverse, p.view_inverse, p.proj_inverse, g["t"], W, H)
    hit = g["t"] >= 0
    outside = hit & ~rp["mark"] & ((rp["x"] < -1) | (rp["x"] >= W))
    print(f"pan: {outside.sum()} pixels reproject outside the image")
    assert outside.sum() >= H and (n[outside] == 1).all()
    # a sideways move: pixels whose first-hit instance differs from the one at every history tap around their previous
    # position (the 2x2 bilinear taps inside the image) lose their history
    p2 = moved(p, 0.0, 0.08 * depth)
    frame(r, p, 4, reset=True)
    frame(r, p2, 6)
    g = r.denoise_guides()
    n = r.temporal_history()["length"]
    rp = tr.reproject(p2.view_inverse, p2.proj_inverse, p.view_inverse, p.proj_inverse, g["t"], W, H)
    before = r.first_hit_aov(p, W, H)["instance"]
    now = r.first_hit_aov(p2, W, H)["instance"]
    inside = (g["t"] >= 0) & rp["front"] & (rp["x"] >= 0) & (rp["x"] <= W - 1) & (rp["y"] >= 0) & (rp["y"] <= H - 1) & ~rp["mark"]
    x0 = np.floor(np.where(inside, rp["x"], 0)).astype(np.int64)
    y0 = np.floor(np.where(inside, rp["y"], 0)).astype(np.int64)
    other = inside.copy()
    for k in range(4):
        qx, qy = np.clip(x0 + (k & 1), 0, W - 1), np.clip(y0 + (k >> 1), 0, H - 1)
        other &= now != before[qy, qx]
    rejected = (n[other] == 1).mean()
    print(f"move: {other.sum()} pixels see another instance than at all their history taps, {rejected:.4f} of them rejected")
    assert other.sum() >= 50 and rejected >= 0.95


def test_history_lifetime(feature):
    s, r, p, _ = feature
    L, h = r._L, r._h

    def length():
        return r.temporal_history()["length"]

    def two_frames():
        frame(r, p, 0, reset=True)
        frame(r, p, 2)
        assert length().max() == 2

    two_frames()
    frame(r, p, 4, reset=True)
    assert length().max() == 1
    # the same extent keeps the history, and pt_denoise in between does not touch it
    two_frames()
    r.on_resize(W, H)
    r.render(2, params=p, first_sample=4)
    r.denoise(p, 5, total_samples=2)
    r.denoise(moved(p, 10.0), 3, total_samples=2)
    r.denoise_temporal(p, total_samples=2)
    assert length().max() == 3
    # an extent change, a scene update and a texture upload discard it
    irr = np.zeros((H, W, 4), F)
    for name, event in (("extent", lambda: (r.on_resize(W + 8, H), r.on_resize(W, H))),
                        ("scene update", lambda: r.update_scene(instance_transforms=s.instances["transform"])),
                        ("texture upload", lambda: r.upload_texture(0, s.textures[0]))):
        two_frames()
        event()
        assert L.pt_denoise_temporal_history(h, irr.ctypes.data, None, W * H) == -1, name
        assert "no history" in L.pt_last_error(h).decode(), name
        frame(r, p, 4)
        assert length().max() == 1, name
    # so does a new scene
    two_frames()
    r.update_scene_data(s)
    frame(r, p, 4)
    assert length().max() == 1


def quality(s, mode, p, frames=16, step_deg=0.36):
    """relMSE of the last of `frames` 1-spp frames against 1024 spp at its camera: noisy, pt_denoise and temporal."""
    r = open_renderer(s)
    try:
        r.set_light_sampling(mode)
        cams = [moved(p, step_deg * k) for k in range(frames)]
        r.render(1024, params=cams[-1], first_sample=0)
        ref = r.read_accumulation()[..., :3] / 1024
        for k, cam in enumerate(cams):
            temporal = frame(r, cam, 1024 + k, spp=1, reset=(k == 0))[..., :3]
        noisy = r.read_accumulation()[..., :3]
        spatial = r.denoise(cams[-1], total_samples=1)[..., :3]
    finally:
        r.close()
    return metrics.rel_mse(noisy, ref), metrics.rel_mse(spatial, ref), metrics.rel_mse(temporal, ref)


# temporal relMSE / spatial relMSE of the last frame must stay below these bounds (measured on the B200: DESIGN §3j)
QUALITY_BOUND = {"feature/pan": 0.4, "feature/static": 0.45, "room/reference/pan": 0.15, "room/emissive_mis/pan": 0.2}


@pytest.mark.parametrize("case", sorted(QUALITY_BOUND))
def test_temporal_beats_spatial_on_a_slow_pan(case):
    parts = case.split("/")
    if parts[0] == "feature":
        s, mode = scenes.feature_scene(), "reference"
        p = s.default_params(8)
    else:
        s, mode = es.room(W, H), parts[1]
        p = s.default_params(6)
    noisy, spatial, temporal = quality(s, mode, p, step_deg=0.0 if parts[-1] == "static" else 0.36)
    ratio = temporal / spatial
    print(f"{case}: relMSE noisy {noisy:.5f} spatial {spatial:.5f} temporal {temporal:.5f} temporal/spatial {ratio:.3f}")
    assert ratio <= QUALITY_BOUND[case], (case, noisy, spatial, temporal)


def test_contract(feature, tmp_path):
    s, r, p, depth = feature
    cams = feature_path(p, depth)[:4]

    def sequence(tiles=None):
        outs = []
        for k, cam in enumerate(cams):
            r.on_resize(W, H)
            r.render(2, params=cam, first_sample=2 * k, tiles=tiles)
            before = r.read_accumulation().copy()
            outs.append(r.denoise_temporal(cam, total_samples=2, reset=(k == 0)))
            assert np.array_equal(r.read_accumulation().view(np.uint32), before.view(np.uint32))
        hist = r.temporal_history()
        return np.stack(outs), np.concatenate([hist["irradiance"], hist["length"][..., None], hist["moments"]], -1)

    a, ha = sequence()
    assert r.stats()["kernel_launches"] == 3 + 2 + 5
    b, hb = sequence()
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(ha.view(np.uint32), hb.view(np.uint32))
    tiles = np.array([(0, 0, W, 50), (0, 50, 70, H), (70, 50, W, H)], conftest.pkg.scene.TILE)
    c, hc = sequence(tiles)
    assert np.array_equal(a.view(np.uint32), c.view(np.uint32)) and np.array_equal(ha.view(np.uint32), hc.view(np.uint32))
    # the post-process chain and the writers run on the result: with K = 0 and alpha = 1 it is the frame itself
    pp = r.postprocess(denoised=True)
    assert pp.shape == (H, W, 4) and pp.dtype == np.uint8
    r.save_png(str(tmp_path / "temporal.png"), denoised=True)
    assert (tmp_path / "temporal.png").stat().st_size > 0
    out = r.denoise_temporal(cams[-1], 0, alpha=1.0, alpha_moments=1.0, total_samples=2)
    assert r.stats()["kernel_launches"] == 3
    assert np.allclose(out[..., :3], r.read_accumulation()[..., :3] / 2, rtol=1e-6, atol=1e-7)


def test_errors(feature):
    s, r, p, _ = feature
    L, h = r._L, r._h
    out = np.zeros((H, W, 4), F)
    cp = p.to_c()
    d = core.DenoiseParams(5, 4.0, 128.0, 1.0)

    def call(alpha=0.2, alpha_m=0.2, n=2, nbytes=out.nbytes, params=cp, dn=d, temporal=True, ctx=None):
        t = core.TemporalParams(alpha, alpha_m, 0)
        return (ctx or r)._L.pt_denoise_temporal((ctx or r)._h, C.addressof(params) if params is not None else None,
                                                 C.addressof(dn) if dn is not None else None, C.addressof(t) if temporal else None,
                                                 n, out.ctypes.data, nbytes)

    r.on_resize(W, H)
    r.render(2, params=p)
    assert call() == 0
    assert call(params=None) == -1 and call(dn=None) == -1 and call(temporal=False) == -1
    for bad in (-0.1, 1.1, float("nan"), float("inf")):
        assert call(alpha=bad) == -1 and call(alpha_m=bad) == -1, bad
    assert call(alpha=0.0, alpha_m=1.0) == 0
    assert call(n=0) == -1
    assert call(nbytes=out.nbytes - 1) == -1
    assert L.pt_denoise_temporal_history(h, out.ctypes.data, None, W * H - 1) == -1
    lens = p.to_c()
    lens.lens_radius = 0.1
    assert call(params=lens) == -7
    r.on_resize(W, H)
    r.render_adaptive(min_samples=2, max_samples=4, batch=2, params=p)
    assert call() == -1 and "adaptive" in L.pt_last_error(h).decode()
    r.on_resize(W, H)
    r2 = core.Renderer(0)
    try:
        assert call(ctx=r2) == -5  # no scene
        r2.update_scene_data(s)
        assert call(ctx=r2) == -6  # no target
        assert r2._L.pt_denoise_temporal_history(r2._h, out.ctypes.data, None, W * H) == -6
    finally:
        r2.close()


def test_temporal_kernels_do_not_spill():
    test_kernel_budgets.kernel_stats()  # builds the library if the log is missing
    text = open(test_kernel_budgets.LOG.replace("wavefront.ptxas.log", "temporal.ptxas.log")).read()
    found = 0
    for m in re.finditer(r"Function properties for (\S*(k_temporal_\w+?)E\S*)\n\s+(\d+) bytes stack frame, "
                         r"(\d+) bytes spill stores, (\d+) bytes spill loads\nptxas info\s+: Used (\d+) registers", text):
        found += 1
        print(f"{m[2]}: {m[6]} registers, stack {m[3]} bytes, spills {m[4]} / {m[5]} bytes (stores / loads)")
        assert int(m[3]) == 0 and int(m[4]) == 0 and int(m[5]) == 0, m[0]
    assert found == 2
