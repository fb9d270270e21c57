"""The numpy reference of the temporal denoiser (tests/temporal_ref.py) on closed forms; runs without a GPU."""
import importlib
import math

import numpy as np

import denoise_ref as dr
import temporal_ref as tr

F = np.float32
H, W = 40, 56
FOV = 45.0
scenes = importlib.import_module("path-tracing_b200.scenes")


def plane_frame(view, proj, depth, radiance, normal=(0.0, 0.0, -1.0)):
    """prepare() of a fronto-parallel plane z = depth seen by the camera (view, proj), albedo 1, constant normal."""
    origin, d = tr.camera_rays(view, proj, W, H)
    albedo_t = np.ones((H, W, 4), F)
    albedo_t[..., 3] = (F(depth) - origin[2]) / d[..., 2]
    nrm = np.zeros((H, W, 4), F)
    nrm[..., :3] = normal
    acc = np.ones((H, W, 4), F)
    acc[..., :3] = radiance
    return dr.prepare(acc, 1, albedo_t, nrm), albedo_t


def camera(position=(0.0, 0.0, 0.0)):
    return scenes.camera_matrices(position, (0.0, 0.0, 1.0), W, H, FOV)


def test_equal_cameras_reproject_every_pixel_onto_itself():
    view, proj = camera((0.3, -0.2, 0.1))
    g, _ = plane_frame(view, proj, 5.0, 1.0)
    rp = tr.reproject(view, proj, view.copy(), proj.copy(), g["t"], W, H)
    assert rp["identity"] and not rp["mark"].any()
    assert (rp["x"] == np.arange(W)[None, :]).all() and (rp["y"] == np.arange(H)[:, None]).all()
    rng = np.random.default_rng(1)
    prev = tr.step(g, view, proj, None)
    prev["irr"][..., :3] = rng.uniform(0, 5, (H, W, 3)).astype(F)
    prev["irr"][..., 3] = 7
    state = tr.step(g, view, proj, prev, alpha=0.0, alpha_moments=0.0)
    assert (state["irr"][..., 3] == 8).all()
    want = prev["irr"][..., :3] + F(0.125) * (g["irr"] - prev["irr"][..., :3])
    assert np.array_equal(state["irr"][..., :3], want)


def test_sideways_translation_shifts_a_fronto_parallel_plane_by_f_delta_over_d():
    depth, delta = 6.0, 0.05
    v0, p0 = camera()
    v1, p1 = camera((delta, 0.0, 0.0))
    g, _ = plane_frame(v1, p1, depth, 1.0)
    rp = tr.reproject(v1, p1, v0, p0, g["t"], W, H)
    f = (H / 2) / math.tan(math.radians(FOV) / 2)
    shift = f * delta / depth
    dx = rp["x"] - np.arange(W)[None, :]
    assert np.allclose(np.abs(dx), shift, rtol=0, atol=2e-4), (dx.min(), dx.max(), shift)
    assert np.allclose(rp["y"], np.arange(H)[:, None], rtol=0, atol=2e-4)
    assert rp["front"].all()
    o1, d1 = tr.camera_rays(v1, p1, W, H)
    X = o1.astype(np.float64) + g["t"][..., None].astype(np.float64) * d1
    assert np.allclose(rp["dist"], np.linalg.norm(X - np.asarray(v0[12:15], np.float64), axis=-1), rtol=1e-6)
    # the history follows the plane: a horizontal ramp in the previous frame is read back shifted by the same amount
    prev = tr.step(plane_frame(v0, p0, depth, 1.0)[0], v0, p0, None)
    prev["irr"][..., 0] = np.arange(W, dtype=F)[None, :]
    state = tr.step(g, v1, p1, prev, alpha=0.0, alpha_moments=0.0)
    inner = (rp["x"] >= 0) & (rp["x"] <= W - 1)
    assert inner.mean() > 0.9
    assert np.allclose(2 * state["irr"][..., 0][inner] - g["irr"][..., 0][inner], rp["x"][inner], atol=1e-4)
    assert np.allclose(state["irr"][..., 3][inner], 2, rtol=1e-6)


def test_alpha_zero_is_the_running_mean():
    view, proj = camera()
    rng = np.random.default_rng(3)
    state, frames = None, []
    for k in range(8):
        c = rng.uniform(0, 4, (H, W, 3)).astype(F)
        frames.append(c)
        g, albedo_t = plane_frame(view, proj, 4.0, c)
        state = tr.step(g, view, proj, state, alpha=0.0, alpha_moments=0.0)
        mean = np.mean(np.stack(frames).astype(np.float64), 0)
        assert np.allclose(state["irr"][..., :3], mean, rtol=1e-5, atol=0)
        l = dr.luminance(np.stack(frames)).astype(np.float64)
        assert np.allclose(state["moments"][..., 0], l.mean(0), rtol=1e-5)
        assert np.allclose(state["moments"][..., 1], (l * l).mean(0), rtol=1e-5)
        assert (state["irr"][..., 3] == k + 1).all()
    out = tr.filter_state(g, albedo_t, state, iterations=0)
    assert np.allclose(out[..., :3], mean, rtol=1e-5)


def test_alpha_sets_the_weight_of_a_long_history():
    view, proj = camera()
    g0, _ = plane_frame(view, proj, 4.0, 1.0)
    state = tr.step(g0, view, proj, None)
    for _ in range(9):
        state = tr.step(g0, view, proj, state, alpha=0.2)
    g1, _ = plane_frame(view, proj, 4.0, 2.0)
    state = tr.step(g1, view, proj, state, alpha=0.2)  # n = 11: a = max(0.2, 1/11) = 0.2
    assert np.allclose(state["irr"][..., :3], 1.2, rtol=1e-6)


def test_rejected_history_restarts_at_length_one():
    view, proj = camera()
    g, _ = plane_frame(view, proj, 4.0, 3.0)
    prev = tr.step(g, view, proj, None)
    prev["irr"][..., 3] = 5
    v1, p1 = camera((0.0, 0.0, 1e-3))  # not bit-identical: the taps are tested
    # another depth (a disocclusion), a turned normal, a miss and no history: each restarts the pixel
    for name, edit in (("depth", lambda p: p["t"].__imul__(F(1.05))), ("normal", lambda p: p["n"].__imul__(F(-1))),
                       ("miss", lambda p: p["t"].fill(F(-1)))):
        p = {k: v.copy() for k, v in prev.items()}
        edit(p)
        g1, _ = plane_frame(v1, p1, 4.0, 3.0)
        state = tr.step(g1, v1, p1, p)
        assert (state["irr"][..., 3] == 1).all(), name
        assert np.array_equal(state["irr"][..., :3], g1["irr"]), name
    # unedited, the same pixels keep their history (n is the taps' weighted mean, exact up to rounding)
    state = tr.step(g1, v1, p1, prev)
    inner = np.abs(state["irr"][..., 3] - 6) <= 6e-6
    assert inner.mean() > 0.9
    # a reset (no previous state) is n = 1
    assert (tr.step(g1, v1, p1, None)["irr"][..., 3] == 1).all()


def test_invalid_pixels_keep_c_and_a_zero_history():
    view, proj = camera()
    g, albedo_t = plane_frame(view, proj, 4.0, 2.0)
    g["valid"][3, 4] = False
    g["t"][3, 4] = -1
    g["c"][3, 4] = np.nan
    state = tr.step(g, view, proj, None)
    assert (state["irr"][3, 4] == 0).all() and (state["moments"][3, 4] == 0).all()
    out = tr.filter_state(g, albedo_t, state, iterations=2)
    assert np.isnan(out[3, 4, :3]).all() and np.isfinite(np.delete(out.reshape(-1, 4), 3 * W + 4, 0)).all()
