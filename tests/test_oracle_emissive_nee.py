"""Emissive-triangle light sampling with MIS (PT_LIGHT_SAMPLING_EMISSIVE_MIS, DESIGN.md §3g) in the CPU oracle: the
emitter table, the alias draw, path identity with the reference mode and convergence to the reference mode's image.
The mode's CPU reference is tests/emissive_oracle.cpp, which extends the oracle's code without changing it."""
import importlib

import numpy as np
import pytest
from scipy import stats

import emissive_scenes as es
from emissive_oracle import EmissiveOracleScene

scenes = importlib.import_module("path-tracing_b200.scenes")

W, H = 32, 24


@pytest.fixture(scope="module")
def room_scene():
    return es.room(W, H)


@pytest.mark.parametrize("name", ["default", "feature", "room"])
def test_emitter_set_and_weights_match_numpy(name, default_scene, oracle_mod, room_scene):
    s = {"default": default_scene, "feature": scenes.feature_scene(), "room": room_scene}[name]
    o = EmissiveOracleScene(s)
    t = o.emitter_table()
    ids, w = es.emitter_weights(s, o)
    assert len(ids) > 0 and (t["flat_ids"] == ids).all(), name
    # float32 corners and sums against float64: a weight of 2^24 moves by a few units at most
    assert np.abs(t["weights"].astype(np.float64) - w).max() <= 16, name
    assert t["weights"].max() == 2**24 and t["weights"].min() >= 1


def test_alias_table_is_exact_and_draws_match_the_weights(room_scene, oracle_mod):
    t = EmissiveOracleScene(room_scene).emitter_table()
    p = t["weights"] / t["weights"].sum()
    assert np.abs(es.alias_probabilities(t) - p).max() < 2.0**-31 * len(p)
    n = 10**6
    counts = np.bincount(es.alias_draws(t, n), minlength=len(p))
    chi2 = ((counts - n * p) ** 2 / (n * p)).sum()
    assert stats.chi2.sf(chi2, len(p) - 1) > 1e-3, (counts, n * p)


def test_the_reference_mode_is_the_oracles(room_scene, oracle_mod):
    p = room_scene.default_params(4)
    a, ca = oracle_mod.OracleScene(room_scene).render(p, W, H, 0, 4)
    b, cb = EmissiveOracleScene(room_scene).render(p, W, H, 0, 4)
    assert (a == b).all() and ca == cb


def test_a_scene_without_emitters_renders_bit_identically(oracle_mod):
    s = es.room(W, H, emitters=False)
    o = EmissiveOracleScene(s)
    p = s.default_params(4)
    a, ca = o.render(p, W, H, 0, 8)
    o.set_light_sampling("emissive_mis")
    assert len(o.emitter_table()["flat_ids"]) == 0
    b, cb = o.render(p, W, H, 0, 8)
    assert (a == b).all() and ca == cb


def test_paths_are_those_of_the_reference_mode(room_scene, oracle_mod):
    """The main rng stream is consumed as in the reference mode: every vertex, bounce and Russian-roulette decision is
    the same, only the collected radiance differs."""
    o = EmissiveOracleScene(room_scene)
    p = room_scene.default_params(6)
    a, ca = o.render(p, W, H, 0, 8)
    o.set_light_sampling("emissive_mis")
    b, cb = o.render(p, W, H, 0, 8)
    for k in ("samples", "rays_closest", "hits", "box_tests_closest", "tri_tests_closest"):
        assert ca[k] == cb[k], k
    assert not (a == b).all()
    o.set_light_sampling("reference")
    c, _ = o.render(p, W, H, 0, 8)
    assert (a == c).all()


# measured on this room (oracle, 1024 spp in 16 batches of 64, depth 4): the emissive-MIS mode's per-pixel variance of
# the batch means is 4.34x lower, averaged over the pixels; the bound keeps a margin for the estimate's own noise
VARIANCE_RATIO_MIN = 3.0


def test_both_modes_converge_to_the_same_image_with_less_variance(room_scene, oracle_mod):
    o = EmissiveOracleScene(room_scene)
    p = room_scene.default_params(4)
    batches, spp = 16, 64

    def batch_means(mode):
        o.set_light_sampling(mode)
        return np.stack([o.render(p, W, H, b * spp, spp)[0][..., :3] / spp for b in range(batches)])

    ref, mis = batch_means("reference"), batch_means("emissive_mis")
    # 8x8-pixel blocks of the luminance-like channel sum: batch means are independent, so the block means are too
    def blocks(x):
        return x.sum(-1).reshape(batches, H // 8, 8, W // 8, 8).mean((2, 4))

    br, bm = blocks(ref), blocks(mis)
    z = (br.mean(0) - bm.mean(0)) / np.sqrt(br.var(0, ddof=1) / batches + bm.var(0, ddof=1) / batches)
    assert np.abs(z).max() <= 4.0, z
    ir, im = ref.sum(-1).mean((1, 2)), mis.sum(-1).mean((1, 2))
    zi = (ir.mean() - im.mean()) / np.sqrt(ir.var(ddof=1) / batches + im.var(ddof=1) / batches)
    assert abs(zi) <= 3.0, zi
    ratio = ref.sum(-1).var(0, ddof=1).mean() / mis.sum(-1).var(0, ddof=1).mean()
    assert ratio >= VARIANCE_RATIO_MIN, ratio
