"""The CPU oracle against THE REFERENCE'S OWN COMPUTE SHADERS (SURVEY §8f rows 2 and 3): postprocess.comp,
bloomDownsample.comp, bloomUpsample.comp, composition.comp, toneMapping.comp and skinning.comp compiled as C++ against
the reference's vendored glm by the same mechanical transform as the ray-tracing stages (oracle/ref_overlay/
glsl2cpp.py --compute, build_glsl.sh -> oracle/_ref/libglsl_comp_ref.so).  The bar is BIT equality of

  * the post-process image after composition.comp and after toneMapping.comp, and bloom level 0 after the whole
    down / up-sampling chain (oracle/pt_oracle_post.cpp), incl. NaN / Inf marking, odd extents and frames too small
    for bloom — the harness's RGBA16F stores round with the compiler's _Float16, i.e. independently of the oracle's
    converter, and the bloom sampler (linear, clamp to edge: Vulkan's, "parity unpinned") is restated there;
  * every float of every skinned vertex (oracle/pt_oracle.cpp skinVertex).

This pin found one discrepancy when it was first run: `boneWeight * vec4(Position, 1) * transform` (skinning.comp:41)
groups from the left — the weighted point goes through the matrix — where oracle and core weighted the transformed
point (last bit of x / y on every second vertex).  Both follow the shader now.

Without the reference checkout the committed vectors of tests/golden/glsl_compute_vectors.npz pin the oracle, and the
comparisons with the compiled shaders compare with the SHA-256 of their output on the same inputs, recorded in
tests/golden/glsl_digests.json (make_glsl_digests.py)."""
import os

import numpy as np
import pytest

import glsl_cases as gc
import glsl_compute_cases as cc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "glsl_compute_vectors.npz")


@pytest.fixture(scope="module")
def glsl():
    """The compiled shaders, or None where libglsl_comp_ref.so is not built: the recorded digests stand in for their outputs."""
    from oracle import glsl_ref

    return glsl_ref if glsl_ref.comp_available() else None


@pytest.fixture(scope="module")
def live_glsl(glsl):
    if glsl is None:
        pytest.skip("libglsl_comp_ref.so not built and no reference checkout (golden vectors still pin the oracle)")
    return glsl


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def assert_same_bits(got, want, what):
    got, want = np.ascontiguousarray(got, np.float32), np.ascontiguousarray(want, np.float32)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    diff = got.view(np.uint32) != want.view(np.uint32)
    diff &= ~(np.isnan(got) & np.isnan(want))  # any NaN equals any NaN
    assert not diff.any(), f"{what}: {int(diff.sum())} of {diff.size} floats differ, first at {np.argwhere(diff)[:4].tolist()}"


def assert_shader_bits(key, got, want, what):
    """got == want bit for bit; with want None (no library), got == the compiled shaders' output recorded under key."""
    gc.check_recorded(key, got, want, assert_same_bits, what)


def oracle_post(oracle_mod, name):
    acc, total, exposure, threshold, intensity = cc.post_case(name)
    composed = oracle_mod.postprocess(acc, total, exposure, threshold, intensity, hdr=True)
    final = oracle_mod.postprocess(acc, total, exposure, threshold, intensity, hdr=True, tone_mapping_hdr=False)
    return composed, final


# ---- golden vectors (always run) --------------------------------------------------------------------------------
@pytest.mark.parametrize("name", cc.GOLDEN_POST)
def test_postprocess_chain_matches_the_golden_vectors(oracle_mod, golden, name):
    composed, final = oracle_post(oracle_mod, name)
    assert_same_bits(composed[..., :3], golden[f"post_{name}_composed"][..., :3], f"{name}: after composition.comp")
    assert_same_bits(final[..., :3], golden[f"post_{name}_final"][..., :3], f"{name}: after toneMapping.comp")
    assert (golden[f"post_{name}_final"][..., 3] == 1.0).all() and (final[..., 3] == 1.0).all()


@pytest.mark.parametrize("angle", cc.SKIN_ANGLES)
def test_skinning_matches_the_golden_vectors(oracle_mod, golden, angle):
    assert_same_bits(oracle_mod.skin_vertices(*cc.skin_case(angle)), golden[f"skin_{angle}"], f"skinning.comp at {angle} degrees")


# ---- the compiled shaders: live where the library is built, else their recorded digests ----------------------------
def test_golden_vectors_are_current(live_glsl, golden):
    for name in cc.GOLDEN_POST:
        acc, total, exposure, threshold, intensity = cc.post_case(name)
        b0, composed, final = live_glsl.postprocess(acc, total, exposure, threshold, intensity, tone_mapping_hdr=False)
        assert_same_bits(composed, golden[f"post_{name}_composed"], name)
        assert_same_bits(final, golden[f"post_{name}_final"], name)
        assert_same_bits(b0, golden[f"post_{name}_bloom0"], name)
    for angle in cc.SKIN_ANGLES:
        assert_same_bits(live_glsl.skin_vertices(*cc.skin_case(angle)), golden[f"skin_{angle}"], f"skin {angle}")


@pytest.mark.parametrize("case", [c[0] for c in cc.POST_CASES])
def test_postprocess_chain_bitwise(glsl, oracle_mod, case):
    acc, total, exposure, threshold, intensity = cc.post_case(case)
    composed, final = oracle_post(oracle_mod, case)
    g = glsl and glsl.postprocess(acc, total, exposure, threshold, intensity, tone_mapping_hdr=False)
    assert_shader_bits(f"post_{case}_composed", composed[..., :3], g and g[1][..., :3], f"{case}: after composition.comp")
    assert_shader_bits(f"post_{case}_final", final[..., :3], g and g[2][..., :3], f"{case}: after toneMapping.comp")
    if glsl:
        # toneMapping.comp in HDR mode is the identity
        _, _, g_hdr = glsl.postprocess(acc, total, exposure, threshold, intensity, tone_mapping_hdr=True)
        assert_same_bits(g_hdr, g[1], f"{case}: HDR tone mapping")


def test_postprocess_marks_nan_and_inf_like_the_shader(glsl, oracle_mod):
    """On the shader's image where the library is built, and on the oracle's."""
    acc, total, exposure, threshold, intensity = cc.post_case("defaults_96x54")
    images = [oracle_mod.postprocess(acc, total, exposure, 1e9, 0.0, hdr=True)]  # no bloom contribution
    if glsl:
        images.append(glsl.postprocess(acc, total, exposure, 1e9, 0.0, tone_mapping_hdr=True)[1])
    h, w = acc.shape[:2]
    for composed in images:
        assert composed[h // 2, w // 3, :3].tolist() == [5000.0, 0.0, 0.0]  # NaN -> red (postprocess.comp:24-25)
        assert composed[h // 3, w // 2, :3].tolist() == [0.0, 5000.0, 0.0]  # Inf -> green (:26-27)
        assert np.isinf(composed[h - 1, w - 1, :3]).all()  # finite in fp32, beyond binary16: the store overflows


@pytest.mark.parametrize("angle", [0.0, 5.0, 12.0, 47.5, 90.0, -33.0])
def test_skinning_bitwise(glsl, oracle_mod, angle):
    animated, idx, bones = cc.skin_case(angle)
    assert_shader_bits(f"skin_{angle}", oracle_mod.skin_vertices(animated, idx, bones), glsl and glsl.skin_vertices(animated, idx, bones),
                       f"skinning.comp at {angle} degrees")


def test_skinning_random_bones_bitwise(glsl, oracle_mod):
    """General (non-rigid, non-uniformly scaled) bone matrices and weights that do not sum to one."""
    animated, idx, _ = cc.skin_case(0.0)
    rng = np.random.default_rng(3)
    animated = animated.copy()
    animated["bone_weights"] = rng.random(animated["bone_weights"].shape, dtype=np.float32) * 0.6
    bones = (rng.standard_normal((4, 12)) * 0.7).astype(np.float32)
    bones[:, [0, 5, 10]] += 1.5  # keep the linear part invertible
    assert_shader_bits("skin_random_bones", oracle_mod.skin_vertices(animated, idx, bones), glsl and glsl.skin_vertices(animated, idx, bones),
                       "random bones")
