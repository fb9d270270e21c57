"""Adaptive sampling (pt_render_adaptive, DESIGN.md §3i) in the CUDA core: a pixel with n samples holds exactly the
accumulation of a uniform n-sample render, the statistics and the pass schedule equal the numpy reference's replay
(tests/adaptive_ref.py) bit for bit, the limits, continuation, scheduling independence, the output paths, the contract
with the rest of the API, the benefit at equal samples, and the new kernels' spills."""
import ctypes as C
import importlib
import re

import numpy as np
import pytest

import adaptive_ref as ar
import conftest
import emissive_scenes as es
import metrics
import test_kernel_budgets

pytestmark = pytest.mark.gpu
core = conftest.core
scenes = importlib.import_module("path-tracing_b200.scenes")
f32 = np.float32
W, H = 64, 48
MAX = 24  # samples per pixel the replay tests render at most
FIRST = dict(min_samples=4, max_samples=MAX, batch=4, threshold=0.1, min_pass_items=1)
SECOND = dict(FIRST, threshold=0.03)
# cases whose blocks stop at several counts under FIRST (measured on the B200: feature 4 / 12 / 24, default 16 / 20 / 24);
# in the emissive test room every 8x4 block is still noisy at 24 samples, so there FIRST is a uniform 24-sample render
MULTI_LEVEL = ("feature", "default")


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


def make_scene(name, request, w=W, h=H):
    """(scene, bounce count, light-sampling mode) of a test case."""
    if name == "feature":
        return scenes.feature_scene(), 8, "reference"
    if name == "default":
        return request.getfixturevalue("default_scene"), 8, "reference"
    return es.room(w, h), 6, name.split("/")[1]


def open_renderer(s, mode, w=W, h=H):
    r = core.Renderer(0)
    r.update_scene_data(s)
    r.set_light_sampling(mode)
    r.on_resize(w, h)
    return r


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.fixture(scope="module", params=["feature", "room/reference", "room/emissive_mis", "default"])
def case(request):
    """A renderer on the case's scene, with the per-sample images (one sample into a cleared target) and the uniform
    accumulation after each of MAX samples rendered one at a time."""
    s, bounces, mode = make_scene(request.param, request)
    r = open_renderer(s, mode)
    p = s.default_params(bounces)
    singles = []
    for i in range(MAX):
        r.on_resize(W, H)
        r.render(1, params=p, first_sample=i)
        singles.append(r.read_accumulation()[..., :3].copy())
    r.on_resize(W, H)
    snaps = []
    for i in range(MAX):
        r.render(1, params=p)
        snaps.append(r.read_accumulation().copy())
    yield request.param, r, p, np.stack(singles), np.stack(snaps)
    r.close()


def uniform_at(snaps, counts):
    """Per pixel, the uniform accumulation after counts[y, x] samples."""
    idx = np.broadcast_to((counts.astype(np.int64) - 1)[None, ..., None], (1,) + snaps.shape[1:])
    return np.take_along_axis(snaps, idx, 0)[0]


def check_identities(r, singles, snaps, state, info, ref_info):
    st = r.adaptive_statistics()
    assert np.array_equal(st["count"], state.count)
    assert np.array_equal(bits(st["mean"]), bits(state.mean)) and np.array_equal(bits(st["m2"]), bits(state.m2))
    assert info == ref_info, (info, ref_info)
    assert np.array_equal(bits(r.read_accumulation()), bits(uniform_at(snaps, st["count"])))
    return st


def test_identity_replay_and_continuation(case):
    name, r, p, singles, snaps = case
    r.on_resize(W, H)
    state = ar.State(H, W)
    info = r.render_adaptive(params=p, **FIRST)
    ref_info, _ = ar.render_adaptive(lambda s: singles[s], state, **FIRST)
    st = check_identities(r, singles, snaps, state, info, ref_info)
    first = st["count"].copy()
    print(f"{name}: threshold 0.1 -> counts {np.bincount(first.ravel())[4:].nonzero()[0] + 4}, {info}")
    if name in MULTI_LEVEL:  # blocks stopped at different counts: the next-level cap and the compaction of one level ran
        assert len(np.unique(first)) >= 2 and info["passes"] >= 2, (name, np.unique(first))
    # a second call with a lower threshold refines the same target; nothing is lowered and the identities still hold
    info = r.render_adaptive(params=p, **SECOND)
    ref_info, _ = ar.render_adaptive(lambda s: singles[s], state, **SECOND)
    st = check_identities(r, singles, snaps, state, info, ref_info)
    assert (st["count"] >= first).all()
    print(f"{name}: threshold 0.03 -> mean spp {st['count'].mean():.2f}, {info}")


def test_limits(case):
    name, r, p, singles, snaps = case
    # min_samples == max_samples is the uniform render of the whole frame
    r.on_resize(W, H)
    info = r.render_adaptive(min_samples=8, max_samples=8, batch=3, threshold=0.0, min_pass_items=1, params=p)
    assert info["passes"] == 1 and info["samples"] == W * H * 8 and (r.sample_counts() == 8).all()
    assert np.array_equal(bits(r.read_accumulation()), bits(snaps[7]))
    # a huge threshold stops every block at min_samples
    r.on_resize(W, H)
    info = r.render_adaptive(min_samples=6, max_samples=MAX, batch=4, threshold=1e30, min_pass_items=1, params=p)
    assert (r.sample_counts() == 6).all() and info["passes"] == 1 and info["unconverged_pixels"] == 0
    # threshold 0 sends every pixel with M2 > 0 to max_samples
    r.on_resize(W, H)
    info = r.render_adaptive(min_samples=4, max_samples=12, batch=4, threshold=0.0, min_pass_items=1, params=p)
    st = r.adaptive_statistics()
    assert (st["count"][st["m2"] > 0] == 12).all()
    assert info["unconverged_pixels"] == int((st["m2"] > 0).sum())
    state = ar.State(H, W)
    ref_info, _ = ar.render_adaptive(lambda s: singles[s], state, 4, 12, 4, 0.0, 1)
    assert info == ref_info and np.array_equal(st["count"], state.count)


@pytest.mark.parametrize("name", ["feature", "room/emissive_mis"])
def test_scheduling_independence(name, request):
    s, bounces, mode = make_scene(name, request)
    p = s.default_params(bounces)
    r = open_renderer(s, mode)
    try:
        results = []
        for tuning in ({}, {"pools": 1}, {"pools": 2, "slots": 1024}, {"sort_hits": 0}):
            for k, v in tuning.items():
                r.set_tuning(k, v)
            r.on_resize(W, H)
            r.render_adaptive(params=p, **FIRST)
            results.append((r.sample_counts(), bits(r.read_accumulation())))
            r.set_tuning("pools", 2)
            r.set_tuning("sort_hits", 1)
        for counts, acc in results[1:]:
            assert np.array_equal(counts, results[0][0]) and np.array_equal(acc, results[0][1])
    finally:
        r.close()


def test_output_paths(case):
    name, r, p, singles, snaps = case
    r.on_resize(W, H)
    r.render_adaptive(params=p, **FIRST)
    pp, hdr = r.postprocess(), r.postprocess(hdr=True)
    den = r.denoise(p, 5)
    den_pp = r.postprocess(denoised=True)
    counts = r.sample_counts()
    mean = r.read_accumulation()
    mean[..., :3] = mean[..., :3] / counts[..., None].astype(f32)
    mean[..., 3] = 1
    r.on_resize(W, H)
    set_accumulation(r, mean)
    assert np.array_equal(pp, r.postprocess(total_samples=1))
    assert np.array_equal(bits(hdr), bits(r.postprocess(hdr=True, total_samples=1)))
    assert np.array_equal(bits(den), bits(r.denoise(p, 5, total_samples=1)))
    assert np.array_equal(den_pp, r.postprocess(denoised=True))


def test_contract(case, request):
    name, r, p, singles, snaps = case
    if name != "feature":
        pytest.skip("one scene is enough for the API contract")
    L, h = r._L, r._h
    cp = p.to_c()
    counts = np.zeros((H, W), np.uint32)
    img = np.zeros((H, W, 4), np.uint8)
    out = np.zeros((H, W, 4), np.float32)
    pp = core.PostProcessParams(1.0, 1.0, 0.1, core.TONE_MAPPING_SDR)
    dn = core.DenoiseParams(5, 4.0, 128.0, 1.0)

    def call(params=cp, **kw):
        a = core.AdaptiveParams(**dict(dict(min_samples=4, max_samples=8, batch=2, min_pass_items=1, threshold=0.1), **kw))
        return L.pt_render_adaptive(h, C.addressof(params) if params is not None else None, C.addressof(a), None)

    def reads():
        return (L.pt_adaptive_readback(h, counts.ctypes.data, None, counts.size),
                L.pt_postprocess_adaptive(h, C.addressof(pp), core.OUTPUT_RGBA8_SRGB, img.ctypes.data, img.nbytes),
                L.pt_denoise_adaptive(h, C.addressof(cp), C.addressof(dn), out.ctypes.data, out.nbytes))

    # errors, each on an empty target
    r.on_resize(W, H)
    assert reads() == (-1, -1, -1)
    assert call(params=None) == -1
    assert L.pt_render_adaptive(h, C.addressof(cp), None, None) == -1
    assert call(min_samples=1) == -1 and call(min_samples=9) == -1 and call(batch=0) == -1
    for bad in (-1.0, float("nan"), float("inf")):
        assert call(threshold=bad) == -1
    nb = p.to_c()
    nb.bounce_count = 0
    assert call(params=nb) == -1
    assert call() == 0
    assert L.pt_adaptive_readback(h, counts.ctypes.data, None, counts.size - 1) == -1
    assert reads() == (0, 0, 0)
    assert r.stats()["kernel_launches"] == 2 + 1 + 5 + 1  # the denoiser's (guides, prepare, variance, 5 levels) + k_adaptive_mean
    assert L.pt_denoise_adaptive(h, C.addressof(cp), None, out.ctypes.data, out.nbytes) == -1
    # the mixing rules, both ways; pt_render_begin resets the record
    assert L.pt_render_samples(h, C.addressof(cp), 0, 1, None, 0) == -1
    assert L.pt_render_frames(h, C.addressof(cp), 0, 1, 2, None, 0) == -1
    assert "adaptive" in L.pt_last_error(h).decode()
    r.on_resize(W, H)
    assert reads() == (-1, -1, -1)
    # a uniform render after an adaptive one lists its pixels again, also when it asks for the tile set it rendered before
    # (the whole frame, in the fixture): the adaptive call left its last pass's pixels in the list
    r.render(1, params=p)
    assert np.array_equal(bits(r.read_accumulation()), bits(snaps[0]))
    assert call() == -1 and "uniform" in L.pt_last_error(h).decode()
    r.on_resize(W, H)
    assert call() == 0
    r.on_resize(W, H)
    r.render_adaptive(params=p, **FIRST)
    r.on_resize(W, H)
    r.render(4, params=p)
    assert np.array_equal(bits(r.read_accumulation()), bits(snaps[3]))
    r.on_resize(W, H)
    r.render_adaptive(params=p, **FIRST)
    r.on_resize(W, H)
    tiles = np.array([(0, 0, W, 20), (0, 20, 30, H), (30, 20, W, H)], conftest.pkg.scene.TILE)
    r.render(4, params=p, tiles=tiles)
    assert np.array_equal(bits(r.read_accumulation()), bits(snaps[3]))
    # pt_stats covers the whole call, not its last pass
    r.on_resize(W, H)
    info = r.render_adaptive(params=p, **FIRST)
    st = r.stats()
    assert info["passes"] > 1 and st["samples"] == info["samples"] and st["last_render_ms"] > 0
    assert st["kernel_launches"] >= 2 * (info["passes"] + 1) + 4 * info["passes"]
    # no scene, no target
    r2 = core.Renderer(0)
    try:
        a = core.AdaptiveParams(4, 8, 2, 1, 0.1)
        assert r2._L.pt_render_adaptive(r2._h, C.addressof(cp), C.addressof(a), None) == -5
        r2.update_scene_data(scenes.feature_scene())
        assert r2._L.pt_render_adaptive(r2._h, C.addressof(cp), C.addressof(a), None) == -6
        assert r2._L.pt_adaptive_readback(r2._h, counts.ctypes.data, None, counts.size) == -6
    finally:
        r2.close()


def test_adaptive_beats_uniform_at_equal_samples():
    """Emissive test room (emissive-MIS), 160x120: relMSE against a 1024-spp render of independent samples."""
    w, h = 160, 120
    s = es.room(w, h)
    p = s.default_params(6)
    r = open_renderer(s, "emissive_mis", w, h)
    try:
        r.render(1024, params=p, first_sample=1 << 20)
        ref = r.read_accumulation()[..., :3] / f32(1024)
        r.on_resize(w, h)
        info = r.render_adaptive(min_samples=16, max_samples=1024, batch=16, threshold=0.5, min_pass_items=1, params=p)
        counts = r.sample_counts()
        adaptive = r.read_accumulation()[..., :3] / counts[..., None].astype(f32)
        spp = int(round(info["samples"] / (w * h)))
        r.on_resize(w, h)
        r.render(spp, params=p)
        uniform = r.read_accumulation()[..., :3] / f32(spp)
    finally:
        r.close()
    ea, eu = metrics.rel_mse(adaptive, ref), metrics.rel_mse(uniform, ref)
    print(f"room/emissive_mis: {info}, counts {counts.min()}..{counts.max()}, at min_samples {(counts == 16).mean():.3f}, "
          f"uniform {spp} spp: relMSE adaptive {ea:.5f} uniform {eu:.5f} ratio {ea / eu:.4f}")
    # measured on an NVIDIA B200 (1000 W): ratio 0.9125 at a mean of 27.3 spp, 55 % of the pixels stopped at min_samples
    assert (counts == 16).mean() > 0.25 and ea < 0.95 * eu, ((counts == 16).mean(), ea, eu, ea / eu)


def test_adaptive_kernel_instances_do_not_spill():
    test_kernel_budgets.kernel_stats()  # builds the library if the log is missing
    found = 0
    for path in (test_kernel_budgets.LOG.replace("wavefront.ptxas.log", "adaptive.ptxas.log"), test_kernel_budgets.LOG):
        text = open(path).read()
        for m in re.finditer(r"Function properties for (\S*(k_adaptive_\w+?|k_resolveILb1E)E\S*)\n\s+(\d+) bytes stack frame, "
                             r"(\d+) bytes spill stores, (\d+) bytes spill loads\nptxas info\s+: Used (\d+) registers", text):
            found += 1
            print(f"{m[2]}: {m[6]} registers, stack {m[3]} bytes, spills {m[4]} / {m[5]} bytes (stores / loads)")
            assert int(m[3]) == 0 and int(m[4]) == 0 and int(m[5]) == 0, m[0]
    assert found == 5  # blocks, select, scatter, mean; resolve
