"""The denoiser (pt_denoise, DESIGN.md §3h) in the CUDA core: its guides against the debug view, its filter against the
numpy reference (tests/denoise_ref.py), closed forms written into the accumulation, image quality against a 1024-spp
render, the contract with the rest of the API, and the kernels' spills."""
import importlib
import re

import numpy as np
import pytest

import conftest
import denoise_ref as dr
import emissive_scenes as es
import metrics
import test_kernel_budgets

pytestmark = pytest.mark.gpu
core = conftest.core
scenes = importlib.import_module("path-tracing_b200.scenes")
W, H = 160, 120
SIGMAS = ((4.0, 128.0, 1.0), (1.0, 32.0, 0.25))


class _CudaArray:
    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f4", "data": (ptr, False), "version": 3}


def set_accumulation(r, image):
    """Writes a host image into the accumulation buffer through a torch view of pt_accum_device_ptr."""
    import torch

    ptr, pitch, _ = r.accum_device_ptr()
    assert pitch == r.width * 16
    dev = torch.as_tensor(_CudaArray(ptr, (r.height, r.width, 4)), device="cuda:0")
    r.synchronize()
    dev.copy_(torch.from_numpy(np.ascontiguousarray(image, np.float32)))
    torch.cuda.synchronize()


def extent(s):
    return tuple(s.camera_extent) if s.camera_extent[0] else (W, H)


def open_renderer(s, w, h):
    r = core.Renderer(0)
    r.update_scene_data(s)
    r.on_resize(w, h)
    return r


def guides_of(r, p):
    r.denoise(p, iterations=0, total_samples=1)
    return r.denoise_guides()


def albedo_t(g):
    return np.concatenate([g["albedo"], g["t"][..., None]], -1)


@pytest.fixture(scope="module")
def feature():
    s = scenes.feature_scene()
    p = s.default_params(8)
    r = open_renderer(s, W, H)
    r.render(4, params=p)
    yield s, r, p
    r.close()


@pytest.mark.parametrize("name", ["default", "feature"])
def test_guides_are_the_debug_views(name, default_scene):
    s = default_scene if name == "default" else scenes.feature_scene()
    w, h = extent(s)
    p = s.default_params()
    r = open_renderer(s, w, h)
    try:
        g = guides_of(r, p)
        normal = r.debug_render(p, w, h, "normal")
        pos = r.debug_render(p, w, h, "world_position")
        hit = r.first_hit_aov(p, w, h)["instance"] != 0xFFFFFFFF
    finally:
        r.close()
    assert hit.any() and (~hit).any(), name
    assert np.array_equal(g["normal"][hit].view(np.uint32), normal[hit][:, :3].view(np.uint32)), name
    eye = np.asarray(s.view_inverse, np.float64).reshape(4, 4).T[:3, 3]
    dist = np.linalg.norm(pos[hit][:, :3].astype(np.float64) - eye, axis=-1)
    assert np.allclose(g["t"][hit], dist, rtol=1e-4, atol=0), name
    assert (g["t"][~hit] == -1).all() and (g["t"][hit] > 0).all(), name


def test_guide_albedo_is_the_unlit_debug_colour():
    """Without lights and emission the debug colour view is base colour x 0.1 (the ambient term)."""
    s = scenes.feature_scene()
    s.point_lights = s.point_lights[:0]
    s.directional_light = s.directional_light.copy()
    s.directional_light["color"] = 0
    for m in (s.mr_materials, s.sg_materials, s.phong_materials):
        m["emissive_color"] = 0
        m["emissive_intensity"] = 0
    p = s.default_params()
    r = open_renderer(s, W, H)
    try:
        g = guides_of(r, p)
        color = r.debug_render(p, W, H, "color")
    finally:
        r.close()
    hit = g["t"] >= 0
    assert np.allclose(g["albedo"][hit], color[hit][:, :3] / np.float32(0.1), rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("iterations", [1, 3, 5])
@pytest.mark.parametrize("sigmas", SIGMAS)
def test_filter_matches_the_reference(feature, iterations, sigmas):
    s, r, p = feature
    got = r.denoise(p, iterations, *sigmas, total_samples=4)
    g = r.denoise_guides()
    acc = r.read_accumulation()
    want = dr.denoise(acc, 4, albedo_t(g), np.concatenate([g["normal"], np.zeros((H, W, 1), np.float32)], -1), iterations, *sigmas)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    fin = ~np.isnan(want)
    err = np.abs(got[fin] - want[fin]) / np.maximum(1.0, np.abs(want[fin]))
    assert err.max() <= 1e-4, err.max()
    assert not np.array_equal(got[..., :3], acc[..., :3] / 4)  # it did filter


def test_closed_forms_on_the_device(feature):
    s, r, p = feature
    hits = r.first_hit_aov(p, W, H)
    hit = hits["instance"] != 0xFFFFFFFF
    # a constant field comes back constant.  The filter works on irradiance (radiance / max(albedo, 1e-3)), so the
    # constant field is a constant irradiance: a constant radiance over a textured surface is not one
    g = guides_of(r, p)
    mean = np.float32(2.5) * np.fmax(g["albedo"], dr.ALBEDO_FLOOR)
    const = np.ones((H, W, 4), np.float32)
    const[..., :3] = mean * np.float32(3)
    set_accumulation(r, const)
    out = r.denoise(p, 5, total_samples=3)
    assert np.allclose(out[..., :3], mean, rtol=2e-6) and (out[..., 3] == 1).all()
    # iterations = 0 is accumulation / total_samples, bit for bit
    rng = np.random.default_rng(9)
    noisy = rng.uniform(0, 30, (H, W, 4)).astype(np.float32)
    set_accumulation(r, noisy)
    out = r.denoise(p, 0, total_samples=7)
    assert np.array_equal(out[..., :3].view(np.uint32), (noisy[..., :3] / np.float32(7)).view(np.uint32))
    # a step in irradiance at a first-hit instance boundary keeps its edge: the instance with the most pixels against the rest
    ids, counts = np.unique(hits["instance"][hit], return_counts=True)
    inst = hits["instance"] == ids[np.argmax(counts)]
    level = np.where(inst, np.float32(0.25), np.float32(4.0))
    want = level[..., None] * np.fmax(g["albedo"], dr.ALBEDO_FLOOR)
    step = np.ones((H, W, 4), np.float32)
    step[..., :3] = want
    set_accumulation(r, step)
    out = r.denoise(p, 5, total_samples=1)
    ratio = out[..., :3] / want
    # nearly every pixel keeps its value; a leak needs a neighbour across the edge with similar normal and depth
    for mask, v in ((inst & hit, 0.25), (~inst & hit, 4.0)):
        close = np.isclose(ratio[mask], 1.0, rtol=1e-2).all(-1)
        print(f"step edge at {v}: {close.mean():.4f} of the pixels within 1 %")
        assert close.mean() >= 0.95 and np.median(ratio[mask]) == pytest.approx(1.0, rel=1e-5), (v, close.mean())
    # non-finite pixels pass through and keep their markers in the post-process chain
    img = rng.uniform(0, 4, (H, W, 4)).astype(np.float32)
    ys, xs = np.nonzero(hit)
    img[ys[10], xs[10], 0] = np.nan
    img[ys[500], xs[500], 1] = np.inf
    set_accumulation(r, img)
    out = r.denoise(p, 5, total_samples=2)
    assert np.isnan(out[ys[10], xs[10], 0]) and np.isinf(out[ys[500], xs[500], 1])
    finite = np.isfinite(img[..., :3]).all(-1)
    assert np.isfinite(out[finite]).all()
    hdr = r.postprocess(hdr=True, denoised=True, bloom_intensity=0.0)
    assert tuple(hdr[ys[10], xs[10], :3]) == (5000.0, 0.0, 0.0)
    assert tuple(hdr[ys[500], xs[500], :3]) == (0.0, 5000.0, 0.0)


def rel_mse_pair(r, p, w, h, spp=16, ref_spp=1024):
    r.on_resize(w, h)
    r.render(ref_spp, params=p, first_sample=0)
    ref = r.read_accumulation()[..., :3] / ref_spp
    r.on_resize(w, h)
    r.render(spp, params=p, first_sample=ref_spp)  # samples independent of the reference's
    noisy = r.read_accumulation()[..., :3] / spp
    den = r.denoise(p, total_samples=spp)[..., :3]
    return metrics.rel_mse(noisy, ref), metrics.rel_mse(den, ref)


@pytest.mark.parametrize("case", ["feature", "room/reference", "room/emissive_mis", "default"])
def test_denoising_halves_the_relmse_at_16_spp(case, default_scene):
    if case == "default":
        s, w, h, mode = default_scene, *extent(default_scene), "reference"
    elif case == "feature":
        s, w, h, mode = scenes.feature_scene(), W, H, "reference"
    else:
        s, w, h, mode = es.room(W, H), W, H, case.split("/")[1]
    r = core.Renderer(0)
    try:
        r.update_scene_data(s)
        r.set_light_sampling(mode)
        noisy, den = rel_mse_pair(r, s.default_params(6 if case.startswith("room") else 8), w, h)
    finally:
        r.close()
    print(f"{case}: relMSE noisy {noisy:.5f} denoised {den:.5f} ratio {den / noisy:.3f}")
    if case != "default":  # mirror and glass: first-hit guides blur what they show; reported only
        assert den <= 0.5 * noisy, (case, noisy, den)


def test_contract(feature):
    s, r, p = feature
    r.on_resize(W, H)
    r.render(4, params=p)
    before = r.read_accumulation().copy()
    pp_before = r.postprocess()
    a = r.denoise(p, 5)
    b = r.denoise(p, 5)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert np.array_equal(r.read_accumulation().view(np.uint32), before.view(np.uint32))
    assert np.array_equal(r.postprocess(), pp_before)
    assert r.stats()["kernel_launches"] > 0
    r.denoise(p, 0)
    assert r.stats()["kernel_launches"] == 2
    assert np.array_equal(r.postprocess(denoised=True), pp_before)
    assert np.array_equal(r.postprocess(denoised=True, hdr=True), r.postprocess(hdr=True))
    r.denoise(p, 5)
    assert r.stats()["kernel_launches"] == 8


def test_tiled_render_denoises_like_the_full_frame(feature):
    s, r, p = feature
    r.on_resize(W, H)
    r.render(4, params=p, first_sample=0)
    full = r.denoise(p, 5, total_samples=4)
    tiles = np.array([(0, 0, W, 50), (0, 50, 70, H), (70, 50, W, H)], conftest.pkg.scene.TILE)
    r.on_resize(W, H)
    r.render(4, params=p, first_sample=0, tiles=tiles)
    assert np.array_equal(r.denoise(p, 5, total_samples=4).view(np.uint32), full.view(np.uint32))


def test_errors(feature):
    s, r, p = feature
    L, h = r._L, r._h
    import ctypes as C

    out = np.zeros((H, W, 4), np.float32)
    cp = p.to_c()

    def call(k=5, sl=4.0, sn=128.0, sd=1.0, n=4, nbytes=out.nbytes, params=cp):
        d = core.DenoiseParams(k, sl, sn, sd)
        return L.pt_denoise(h, C.addressof(params) if params is not None else None, C.addressof(d), n, out.ctypes.data, nbytes)

    assert call() == 0
    assert call(n=0) == -1
    assert call(k=9) == -1
    for bad in (-1.0, float("nan"), float("inf")):
        assert call(sl=bad) == -1 and call(sn=bad) == -1 and call(sd=bad) == -1
    assert call(nbytes=out.nbytes - 1) == -1
    assert call(params=None) == -1
    lens = p.to_c()
    lens.lens_radius = 0.1
    assert call(params=lens) == -7
    r.on_resize(W, H)  # no pt_denoise since pt_render_begin
    pp = core.PostProcessParams(1.0, 1.0, 0.1, core.TONE_MAPPING_SDR)
    img = np.zeros((H, W, 4), np.uint8)
    assert L.pt_postprocess_denoised(h, C.addressof(pp), core.OUTPUT_RGBA8_SRGB, img.ctypes.data, img.nbytes) == -1
    assert "no pt_denoise" in L.pt_last_error(h).decode()
    assert L.pt_denoise_guides(h, out.ctypes.data, out.ctypes.data, out.nbytes) == -1
    assert "no pt_denoise" in L.pt_last_error(h).decode()
    assert call() == 0
    assert L.pt_denoise_guides(h, out.ctypes.data, None, out.nbytes - 1) == -1
    r2 = core.Renderer(0)
    try:
        d = core.DenoiseParams(5, 4.0, 128.0, 1.0)
        assert r2._L.pt_denoise(r2._h, C.addressof(cp), C.addressof(d), 4, out.ctypes.data, out.nbytes) == -5  # no scene
        r2.update_scene_data(s)
        assert r2._L.pt_denoise(r2._h, C.addressof(cp), C.addressof(d), 4, out.ctypes.data, out.nbytes) == -6  # no target
        assert r2._L.pt_denoise_guides(r2._h, out.ctypes.data, None, out.nbytes) == -6
    finally:
        r2.close()


def test_denoise_kernels_do_not_spill():
    test_kernel_budgets.kernel_stats()  # builds the library if the log is missing
    log = test_kernel_budgets.LOG.replace("wavefront.ptxas.log", "denoise.ptxas.log")
    found = 0
    for path in (log, test_kernel_budgets.LOG):
        text = open(path).read()
        for m in re.finditer(r"Function properties for (\S*(k_atrous|k_denoise_\w+?)E\S*)\n\s+(\d+) bytes stack frame, "
                             r"(\d+) bytes spill stores, (\d+) bytes spill loads\nptxas info\s+: Used (\d+) registers", text):
            found += 1
            print(f"{m[2]}: {m[6]} registers, stack {m[3]} bytes, spills {m[4]} / {m[5]} bytes (stores / loads)")
            assert int(m[4]) == 0, m[0]
    assert found == 5
