"""The numpy reference of the denoiser (tests/denoise_ref.py) on closed forms; runs without a GPU."""
import numpy as np

import denoise_ref as dr

F = np.float32
H, W = 40, 56


def guides(seed=0, normal=None):
    """Arbitrary guides: random albedo, a slanted depth with noise, random unit normals (unless given)."""
    rng = np.random.default_rng(seed)
    albedo_t = np.empty((H, W, 4), F)
    albedo_t[..., :3] = rng.uniform(0.0, 1.0, (H, W, 3))
    ys, xs = np.mgrid[0:H, 0:W]
    albedo_t[..., 3] = 3.0 + 0.02 * xs + 0.01 * ys + rng.uniform(0, 0.05, (H, W))
    if normal is None:
        normal = rng.normal(size=(H, W, 3)).astype(F)
        normal /= np.linalg.norm(normal, axis=-1, keepdims=True)
    nrm = np.zeros((H, W, 4), F)
    nrm[..., :3] = normal
    return albedo_t, nrm


def accumulate(mean_radiance, samples):
    acc = np.ones((H, W, 4), F)
    acc[..., :3] = mean_radiance * F(samples)
    return acc


def test_zero_iterations_is_the_identity():
    rng = np.random.default_rng(1)
    acc = rng.uniform(0, 40, (H, W, 4)).astype(F)
    acc[3, 4, 0] = np.nan
    at, n = guides()
    out = dr.denoise(acc, 7, at, n, iterations=0)
    want = acc[..., :3] / F(7)
    assert np.array_equal(out[..., :3], want, equal_nan=True) and (out[..., 3] == 1).all()


def test_a_constant_irradiance_field_stays_constant():
    """Irradiance constant, radiance = irradiance * max(albedo, 1e-3) with arbitrary albedo, normals and depth: every
    level returns the constant, so the output is the input radiance to 1e-6."""
    at, n = guides(2)
    at[0, :5, :3] = 0  # below the albedo floor
    radiance = F(0.7) * np.fmax(at[..., :3], dr.ALBEDO_FLOOR)
    for k, sigmas in ((1, (4.0, 128.0, 1.0)), (5, (4.0, 128.0, 1.0)), (8, (0.5, 16.0, 0.2))):
        out = dr.denoise(accumulate(radiance, 4), 4, at, n, k, *sigmas)
        assert np.allclose(out[..., :3], radiance, rtol=1e-6, atol=1e-7), k


def test_the_weights_of_every_pixel_are_normalised():
    rng = np.random.default_rng(3)
    at, n = guides(3)
    at[5:9, 10:20, 3] = -1  # some misses
    acc = accumulate(rng.uniform(0, 2, (H, W, 3)).astype(F), 2)
    g = dr.prepare(acc, 2, at, n)
    var = dr.variance(g, 128.0, 1.0)
    for step in (1, 4, 16):
        _, w = dr.atrous_level(g, g["irr"], var, step, 4.0, 128.0, 1.0, return_weights=True)
        v = g["valid"]
        assert (w[v] >= 0).all()
        assert np.allclose(w[v].sum(-1), 1.0, atol=1e-6), step
        assert (w[v][:, 12] > 0).all()  # the centre tap always counts


def test_a_normal_edge_of_90_degrees_survives():
    """Two half-planes whose normals are 90° apart never exchange weight (w_n = 0): after 5 levels each side keeps its
    value beyond one pixel from the edge, on a noisy image too."""
    normal = np.zeros((H, W, 3), F)
    normal[:, : W // 2] = (0, 0, 1)
    normal[:, W // 2 :] = (1, 0, 0)
    at, n = guides(4, normal)
    at[..., :3] = 0.5
    at[..., 3] = 5.0
    radiance = np.where(np.arange(W)[None, :, None] < W // 2, F(0.2), F(3.0)).astype(F) * np.ones((H, W, 3), F)
    out = dr.denoise(accumulate(radiance, 8), 8, at, n, 5)
    far = np.abs(np.arange(W) + 0.5 - W / 2) > 1.5
    assert np.allclose(out[:, far, :3], radiance[:, far], rtol=1e-6)
    rng = np.random.default_rng(5)
    noisy = (radiance * rng.uniform(0.5, 1.5, (H, W, 1))).astype(F)
    out = dr.denoise(accumulate(noisy, 8), 8, at, n, 5)
    left, right = out[:, : W // 2 - 1, :3], out[:, W // 2 + 1 :, :3]
    assert left.max() <= noisy[:, : W // 2].max() + 1e-6 and right.min() >= noisy[:, W // 2 :].min() - 1e-6


def test_miss_and_nan_pixels_pass_through():
    rng = np.random.default_rng(6)
    at, n = guides(6)
    acc = accumulate(rng.uniform(0, 2, (H, W, 3)).astype(F), 4)
    at[10:14, 20:30, 3] = -1  # misses
    acc[2, 3, 1] = np.nan
    acc[30, 40, 2] = np.inf
    out = dr.denoise(acc, 4, at, n, 5)
    c = acc[..., :3] / F(4)
    passthrough = (at[..., 3] < 0) | ~np.isfinite(c).all(-1)
    assert passthrough.sum() == 42
    assert np.array_equal(out[passthrough][:, :3], c[passthrough], equal_nan=True)
    assert np.isfinite(out[~passthrough]).all() and (out[..., 3] == 1).all()
