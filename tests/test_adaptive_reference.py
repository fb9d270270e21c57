"""The numpy reference of adaptive sampling (tests/adaptive_ref.py) against closed forms and hand-worked schedules; no GPU."""
import numpy as np
import pytest

import adaptive_ref as ar

f32 = np.float32


def constant(value, h, w):
    img = np.full((h, w, 3), value, f32)
    return lambda s: img


def noisy_blocks(h, w, noisy):
    """Sample s: 1 everywhere, plus noise of its own seed on the pixels of `noisy` (H, W bool)."""

    def sample(s):
        img = np.ones((h, w, 3), f32)
        img[noisy] += np.random.default_rng(s).uniform(0, 4, (int(noisy.sum()), 3)).astype(f32)
        return img

    return sample


@pytest.mark.parametrize("value", [0.0, 0.37, 5.0])
@pytest.mark.parametrize("threshold", [0.0, 0.02])
def test_constant_samples_stop_at_min_samples(value, threshold):
    h, w = 13, 21  # partial edge blocks on both sides
    st = ar.State(h, w)
    info, passes = ar.render_adaptive(constant(value, h, w), st, 5, 64, 3, threshold, 1)
    assert (st.m2 == 0).all() and (st.mean == f32(ar.luminance(np.full(3, value, f32)))).all()
    assert (st.count == 5).all()
    assert info == {"passes": 1, "min_count": 5, "max_count": 5, "unconverged_pixels": 0, "samples": h * w * 5}


def test_welford_matches_float64_statistics():
    rng = np.random.default_rng(3)
    for scale, n in ((1.0, 16), (100.0, 256), (1e-3, 1000)):
        stream = (rng.exponential(scale, (n, 7, 9)) * rng.uniform(0.5, 2, (1, 7, 9))).astype(f32)
        st = ar.State(7, 9)
        for l in stream:
            ar.welford(st, l)
        x = stream.astype(np.float64)
        assert (st.count == n).all()
        np.testing.assert_allclose(st.mean, x.mean(0), rtol=2e-5)
        np.testing.assert_allclose(st.m2 / (n - 1), x.var(0, ddof=1), rtol=2e-4)


def test_stop_rule_is_the_relative_standard_error():
    # var / n / (mean^2 + 0.01) <= t^2 with var = M2 / (n - 1)
    mean, n, t = f32(2.0), 10, 0.05
    limit = f32(t) * f32(t) * (mean * mean + ar.EPS) * f32(n) * f32(n - 1)
    assert ar.converged(n, mean, limit, t) and not ar.converged(n, mean, np.nextafter(limit, f32(np.inf)), t)
    assert ar.converged(n, mean, f32(0.0), 0.0) and not ar.converged(n, mean, f32(1e-30), 0.0)


def test_min_pass_items_and_batch_schedule():
    # a 16x8 frame: four 8x4 blocks, only the first one noisy (it never meets t = 1e-3 and runs to the cap)
    h, w = 8, 16
    noisy = np.zeros((h, w), bool)
    noisy[:4, :8] = True
    for mpi, ks in ((1, [4] + [4] * 24), (64, [4] + [4] * 24), (320, [4] + [10] * 9 + [6])):
        st = ar.State(h, w)
        info, passes = ar.render_adaptive(noisy_blocks(h, w, noisy), st, 2, 100, 4, 1e-3, mpi)
        # the first pass: one count level, max(n + batch, min_samples, n + ceil(mpi / A)) = 4 for all 128 pixels
        assert [k for _, k, _ in passes] == ks, mpi
        assert passes[0][2].all() and all((m == noisy).all() for _, _, m in passes[1:])
        assert (st.count[noisy] == 100).all() and (st.count[~noisy] == 4).all()
        assert info == {"passes": len(ks), "min_count": 4, "max_count": 100, "unconverged_pixels": 32,
                        "samples": 128 * 4 + 32 * 96}


def test_next_level_caps_a_pass_and_continuation_refines():
    h, w = 8, 16
    noisy = np.zeros((h, w), bool)
    noisy[:4, :8] = True
    noisy[4:, 8:] = True
    sample = noisy_blocks(h, w, noisy)
    st = ar.State(h, w)
    info, passes = ar.render_adaptive(sample, st, 2, 8, 2, 1e-3, 1)
    assert [k for _, k, _ in passes] == [2, 2, 2, 2]
    assert (st.count[noisy] == 8).all() and (st.count[~noisy] == 2).all()
    assert info["unconverged_pixels"] == 64 and info["samples"] == 128 * 2 + 64 * 6
    before = st.copy()
    # min_samples 12 re-activates the converged blocks at 2; the noisy ones wait at 8 (the next level caps the first pass)
    info, passes = ar.render_adaptive(sample, st, 12, 20, 16, 1e-3, 1)
    assert [(n, k) for n, k, _ in passes] == [(2, 6), (8, 12)]
    assert (passes[0][2] == ~noisy).all() and passes[1][2].all()
    assert (st.count == 20).all() and (st.count >= before.count).all()
    assert info == {"passes": 2, "min_count": 20, "max_count": 20, "unconverged_pixels": 64, "samples": 64 * 6 + 128 * 12}
    # the statistics do not depend on how the samples were split into passes
    once = ar.State(h, w)
    ar.render_adaptive(sample, once, 20, 20, 1, 0.0, 1)
    for a, b in ((st.count, once.count), (st.mean, once.mean), (st.m2, once.m2)):
        assert np.array_equal(a, b)


def test_blocks_move_together_on_partial_edges():
    h, w = 10, 21
    rng = np.random.default_rng(5)
    noisy = rng.uniform(size=(h, w)) < 0.1
    st = ar.State(h, w)
    ar.render_adaptive(noisy_blocks(h, w, noisy), st, 4, 40, 4, 0.05, 1)
    ids, nb = ar.block_ids(h, w)
    assert nb == 3 * 3
    for b in range(nb):
        c = st.count[ids == b]
        assert (c == c[0]).all()
        done = ar.converged(st.count[ids == b], st.mean[ids == b], st.m2[ids == b], 0.05).all()
        assert c[0] == 40 or (c[0] >= 4 and done), b
    assert (st.count[~noisy] >= 4).all() and (st.count[noisy] > 4).any()
