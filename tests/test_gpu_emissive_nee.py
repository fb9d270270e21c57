"""Emissive-triangle light sampling with MIS (PT_LIGHT_SAMPLING_EMISSIVE_MIS, DESIGN.md §3g) in the CUDA core: the
emitter table against the CPU reference's (tests/emissive_oracle.cpp) entry for entry, images against its emissive-MIS
mode within the bounds of test_gpu_configs.test_image_parity, path identity with the reference mode, and determinism
across scheduling, tiles, scene updates and mode switches."""
import importlib
import re

import numpy as np
import pytest

import conftest
import emissive_scenes as es
from emissive_oracle import EmissiveOracleScene
import metrics
import test_kernel_budgets
from scenes_small import SMALL, W, H

pytestmark = pytest.mark.gpu
scenes = importlib.import_module("path-tracing_b200.scenes")
sc = conftest.pkg.scene

CASES = ["default", "feature", "room"] + sorted(SMALL)


def build_case(name, default_scene):
    if name == "default":
        return default_scene, 8
    if name == "feature":
        return scenes.feature_scene(), 8
    if name == "room":
        return es.room(W, H), 6
    build, bounces, _ = SMALL[name]
    return build(), bounces


@pytest.fixture(scope="module", params=CASES)
def case(request, oracle_mod, default_scene):
    s, bounces = build_case(request.param, default_scene)
    r = conftest.core.Renderer(0)
    r.update_scene_data(s)
    r.set_light_sampling("emissive_mis")
    o = EmissiveOracleScene(s)
    o.set_light_sampling("emissive_mis")
    yield request.param, s, r, o, bounces
    r.close()


def test_emitter_table_equals_the_oracles(case):
    name, s, r, o, _ = case
    got, ref = r.emitter_table(), o.emitter_table()
    # chess, dragon and atrium have no emitters: there the mode is the reference mode
    assert (len(ref["flat_ids"]) > 0) == (name in ("default", "feature", "room", "street")), name
    for k in ref:
        assert (got[k] == ref[k]).all(), (name, k)


def test_image_parity_with_the_oracle(case):
    name, s, r, o, bounces = case
    p = s.default_params(bounce_count=bounces)
    spp = 16
    r.on_resize(W, H)
    r.render(spp, params=p)
    img, st = r.read_accumulation(), r.stats()
    ref, cnt = o.render(p, W, H, 0, spp)
    assert np.isfinite(img).all()
    assert st["samples"] == cnt["samples"] == W * H * spp
    assert metrics.close_fraction(img, ref, 1e-3) > (0.93 if name == "dragon" else 0.96), name
    assert metrics.rel_mse(img / spp, ref / spp) <= 1e-3, name
    assert metrics.flip(img / spp, ref / spp) <= 5e-3, name
    diverged = conftest.diverged_path_fraction(r, o, p, W, H, 0, 8)
    assert diverged <= (0.02 if name == "dragon" else 0.008), (name, diverged)


def test_paths_are_those_of_the_reference_mode(case):
    name, s, r, o, bounces = case
    p = s.default_params(bounce_count=bounces)
    counts = {}
    for mode in ("reference", "emissive_mis"):
        r.set_light_sampling(mode)
        r.on_resize(W, H)
        r.render(4, params=p, first_sample=0)
        st = r.stats()
        counts[mode] = (st["samples"], st["rays_closest"], st["hits"])
    r.set_light_sampling("emissive_mis")
    assert counts["reference"] == counts["emissive_mis"], name


def render_room(knobs=(), tiles=None, mode="emissive_mis", scene=None, spp=6):
    s = scene or es.room(96, 64)
    r = conftest.core.Renderer(0)
    try:
        for k, v in knobs:
            r.set_tuning(k, v)
        r.update_scene_data(s)
        r.set_light_sampling(mode)
        r.on_resize(96, 64)
        r.render(spp, params=s.default_params(6), tiles=tiles, first_sample=0)
        return r.read_accumulation().copy()
    finally:
        r.close()


def test_scheduling_and_tiles_do_not_change_the_image():
    ref = render_room()
    for knobs in ((("pools", 1), ("sort_hits", 0)), (("pools", 3), ("slots", 2000)), (("pools", 8), ("slots", 5000))):
        assert (render_room(knobs) == ref).all(), knobs
    tiles = np.array([(0, 0, 96, 21), (0, 21, 40, 64)], sc.TILE)
    part = render_room(tiles=tiles)
    inside = np.zeros((64, 96), bool)
    inside[:21] = True
    inside[21:, :40] = True
    assert (part[inside] == ref[inside]).all() and (part[~inside] == 0).all()


def test_scene_update_equals_a_fresh_upload():
    """Moving the lamps with pt_scene_update rebuilds the emitter table: the render equals a fresh upload's."""
    s = es.room(96, 64)
    moved = s.instances["transform"].copy()
    lamps = np.arange(len(moved) - 3, len(moved))
    moved[lamps, 3] += 0.4  # x of the 3x4 row-major translation
    moved[lamps, 11] -= 0.3
    p = s.default_params(6)
    r = conftest.core.Renderer(0)
    try:
        r.update_scene_data(s)
        r.set_light_sampling("emissive_mis")
        r.on_resize(96, 64)
        r.render(2, params=p, first_sample=0)  # builds the table of the unmoved scene
        r.update_scene(instance_transforms=moved)
        r.on_resize(96, 64)
        r.render(6, params=p, first_sample=0)
        updated = r.read_accumulation().copy()
        table = r.emitter_table()
    finally:
        r.close()
    s2 = es.room(96, 64)
    s2.instances["transform"] = moved
    fresh = render_room(scene=s2)
    assert (updated == fresh).all()
    r2 = conftest.core.Renderer(0)
    try:
        r2.update_scene_data(s2)
        fresh_table = r2.emitter_table()
    finally:
        r2.close()
    for k in table:
        assert (table[k] == fresh_table[k]).all(), k


def test_switching_the_mode_back_restores_the_reference_image():
    s = es.room(96, 64)
    p = s.default_params(6)
    fresh = render_room(mode="reference", scene=s)
    r = conftest.core.Renderer(0)
    try:
        r.update_scene_data(s)
        r.set_light_sampling("emissive_mis")
        r.on_resize(96, 64)
        r.render(6, params=p, first_sample=0)
        mis = r.read_accumulation().copy()
        r.set_light_sampling("reference")
        r.on_resize(96, 64)
        r.render(6, params=p, first_sample=0)
        back = r.read_accumulation().copy()
    finally:
        r.close()
    assert (back == fresh).all()
    assert not (mis == fresh).all()


def test_a_scene_without_emitters_renders_as_the_reference_mode():
    s = es.room(96, 64, emitters=False)
    assert (render_room(scene=s) == render_room(scene=s, mode="reference")).all()


def test_k_shade_emissive_register_budget():
    """k_shade_emissive: 128 registers at most, like k_shade (four 128-thread blocks per SM); its spills are reported."""
    test_kernel_budgets.kernel_stats()  # builds the library if the log is missing
    text = open(test_kernel_budgets.LOG).read()
    found = 0
    for m in re.finditer(r"Function properties for (\S*k_shade_emissiveILb([01])ELb([01])E\S*)\n\s+(\d+) bytes stack frame, "
                         r"(\d+) bytes spill stores, (\d+) bytes spill loads\nptxas info\s+: Used (\d+) registers", text):
        found += 1
        print(f"k_shade_emissive<{m[2]},{m[3]}>: {m[7]} registers, spills {m[5]} / {m[6]} bytes (stores / loads)")
        assert int(m[7]) <= 128, m[0]
    assert found == 4
