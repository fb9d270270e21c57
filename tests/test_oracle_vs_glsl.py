"""The CPU oracle against THE REFERENCE'S OWN SHADER CODE: Path-Tracing/Shaders/*.glsl, raygen.rgen,
closestHit.rchit, anyhit.rahit, occlusionAnyhit.rahit, miss.rmiss, occlusion.rmiss compiled as C++ against
the reference's vendored glm by a mechanical transform (oracle/ref_overlay/glsl2cpp.py, build_glsl.sh ->
oracle/_ref/libglsl_ref.so).  The bar is BIT equality: every function of SURVEY §8(a) rows a1-a3, a5-a16 on
the reference's unit-test grids (PTT/TestData.h) and 10^5 seeded random records each, closest-hit payloads,
and whole accumulation images (raygen main() driving the compiled any-hit / closest-hit / miss stages).
Only the two services the reference leaves to the Vulkan implementation — acceleration-structure traversal
and texture filtering — are shared with the oracle (callbacks); those stay "parity unpinned".

Where libglsl_ref.so cannot be built (no reference checkout) the committed golden vectors of
tests/golden/glsl_vectors.npz (generated from the same library by make_glsl_vectors.py) pin the oracle, and the live
comparisons compare with the SHA-256 of the library's output on the same inputs, recorded in
tests/golden/glsl_digests.json (make_glsl_digests.py)."""
import os

import numpy as np
import pytest

import glsl_cases as gc
import refdata as rd
import unit_inputs as ui

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "glsl_vectors.npz")
N_MODES = len(ui.MODE_NAMES)


@pytest.fixture(scope="module")
def glsl():
    """The compiled shaders, or None where libglsl_ref.so is not built: the recorded digests stand in for their outputs."""
    from oracle import glsl_ref

    return glsl_ref if glsl_ref.available() else None


@pytest.fixture(scope="module")
def live_glsl(glsl):
    if glsl is None:
        pytest.skip("libglsl_ref.so not built and no reference checkout (golden vectors still pin the oracle)")
    return glsl


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


def assert_bits(got, want, what):
    same = ui.bit_equal(got, want)
    assert same.all(), f"{what}: {int((~same).sum())} of {len(same)} records differ, first at {np.flatnonzero(~same)[:5].tolist()}"


def assert_shader_bits(key, got, want, what):
    """got == want bit for bit; with want None (no library), got == the compiled shaders' output recorded under key."""
    gc.check_recorded(key, got, want, assert_bits, what)


# ---- golden vectors (always run) -----------------------------------------------------------------------

def test_strides_match_the_header(oracle_mod):
    assert len(oracle_mod.TEST_IN) == len(oracle_mod.TEST_OUT) == N_MODES


@pytest.mark.parametrize("mode", range(N_MODES), ids=ui.MODE_NAMES)
def test_function_matches_golden_glsl_output(oracle_mod, golden, mode):
    assert_bits(oracle_mod.test_shading(mode, golden[f"in_{mode}"]), golden[f"out_{mode}"], ui.MODE_NAMES[mode])


def test_closest_hit_payloads_match_golden(oracle_mod, golden, default_scene):
    cases = gc.stage_scenes(default_scene)
    for name in ("default", "feature"):
        scene, params = cases[name][0], cases[name][1]
        ora = oracle_mod.OracleScene(scene)
        out = ora.closest_hit(params, golden[f"chit_{name}_hits"], golden[f"chit_{name}_rays"], golden[f"chit_{name}_in"])
        assert len(out) > 100
        assert_bits(out, golden[f"chit_{name}_out"], f"closestHit.rchit payloads, {name} scene")


def test_images_match_golden(oracle_mod, golden, default_scene):
    for name, (scene, params, w, h, first, frames, spp) in gc.stage_scenes(default_scene).items():
        ora = oracle_mod.OracleScene(scene)
        img, _ = ora.render_frames(params, w, h, first, frames, spp)
        want = golden[f"img_{name}"]
        assert np.isfinite(want).all() and want[..., :3].max() > 0.1
        assert_bits(img.reshape(-1, 4), want.reshape(-1, 4), f"accumulation image '{name}'")


def test_debug_pipeline_matches_golden(oracle_mod, golden, default_scene):
    cases = gc.stage_scenes(default_scene)
    for scene_name, mode, rf, hf in gc.DEBUG_GOLDEN:
        scene, params, w, h = cases[scene_name][:4]
        got = oracle_mod.OracleScene(scene).debug_render(params, w, h, mode, rf, hf)
        assert_bits(got.reshape(-1, 4), golden[gc.debug_key(scene_name, mode, rf, hf)].reshape(-1, 4),
                    f"debug pipeline, {scene_name} / {mode} / raygen {rf} / hit group {hf:#x}")


# ---- the compiled shaders: live where the library is built, else their recorded digests ------------------------------

GRIDS = {0: rd.grid_vec3_float, 1: rd.grid_vec3_float, 2: rd.grid_vec3_float, 3: rd.grid_dielectric, 4: rd.grid_schlick,
         5: rd.grid_reflection, 6: rd.grid_refraction, 7: rd.grid_sample_ggx, 8: rd.grid_lobe_pdfs}


@pytest.mark.parametrize("mode", sorted(GRIDS), ids=[ui.MODE_NAMES[m] for m in sorted(GRIDS)])
def test_reference_grids_bitwise(oracle_mod, glsl, mode):
    """The input grids of the reference's own unit tests (PTT/ShadingTest.cpp, BsdfTest.cpp, TestData.h)."""
    grid = GRIDS[mode]()
    assert_shader_bits(f"grid_{mode}", oracle_mod.test_shading(mode, grid), glsl and glsl.test_shading(mode, grid), ui.MODE_NAMES[mode])
    if mode == 6:
        grid = rd.grid_refraction(flip_l=True)
        assert_shader_bits("grid_6_flip_l", oracle_mod.test_shading(mode, grid), glsl and glsl.test_shading(mode, grid),
                           "EvaluateRefraction body")


@pytest.mark.parametrize("mode", range(N_MODES), ids=ui.MODE_NAMES)
def test_random_inputs_bitwise(oracle_mod, glsl, mode):
    x = ui.inputs(mode, 100_000, seed=3)
    assert_shader_bits(f"random_{mode}", oracle_mod.test_shading(mode, x), glsl and glsl.test_shading(mode, x), ui.MODE_NAMES[mode])


def test_golden_file_is_what_the_library_produces(live_glsl, golden):
    for mode in range(N_MODES):
        assert_bits(live_glsl.test_shading(mode, golden[f"in_{mode}"]), golden[f"out_{mode}"], f"golden {ui.MODE_NAMES[mode]}")


def test_closest_hit_payloads_bitwise(oracle_mod, glsl, default_scene):
    cases = gc.stage_scenes(default_scene)
    for name in ("default", "feature"):
        scene, params = cases[name][0], cases[name][1]
        ora = oracle_mod.OracleScene(scene)
        g = glsl and glsl.GlslScene(scene, ora)
        hits, rays, pin = gc.closest_hit_inputs(ora, oracle_mod, params, 96, 72)
        assert len(hits) > 1000
        assert_shader_bits(f"chit_{name}", ora.closest_hit(params, hits, rays, pin), g and g.closest_hit(params, hits, rays, pin),
                           f"payloads, {name}")


def _bitwise_images(oracle_mod, glsl, scene, params, w, h, first, frames, spp, key, what):
    ora = oracle_mod.OracleScene(scene)
    want = None
    if glsl:
        want, spinning = glsl.GlslScene(scene, ora).render(params, w, h, first, frames, spp)
        assert spinning == 0
        want = want.reshape(-1, 4)
    got, counters = ora.render_frames(params, w, h, first, frames, spp)
    assert np.isfinite(got).all() and got[..., :3].max() > 0.05, what
    assert_shader_bits(key, got.reshape(-1, 4), want, what)
    return counters


def test_images_bitwise(oracle_mod, glsl, default_scene):
    """raygen.rgen main() per pixel and frame (SampleCount 1, 2 and 3), compiled any-hit / closest-hit / miss."""
    for name, (scene, params, w, h, first, frames, spp) in gc.stage_scenes(default_scene).items():
        _bitwise_images(oracle_mod, glsl, scene, params, 2 * w, 2 * h, first, frames, spp, f"img_{name}", name)


def test_skybox_variants_bitwise(oracle_mod, glsl):
    sc = gc.sc
    rs = np.random.default_rng(5)
    fs = gc.scenes.feature_scene(width=48, height=36)
    sky = (rs.uniform(0, 1, (16, 32, 4)) * 255).astype(np.uint8)
    fs.skybox_2d = sc.Texture(sky, srgb=True)
    p = fs.default_params(bounce_count=4)
    p.miss_flags = sc.MISS_FLAGS_SKYBOX_2D
    _bitwise_images(oracle_mod, glsl, fs, p, 48, 36, 0, 2, 1, "img_sky_2d", "2-D skybox")
    fs.skybox_2d = None
    fs.skybox_cube = [sc.Texture(rs.uniform(0, 4, (8, 8, 4)).astype(np.float32), srgb=False) for _ in range(6)]
    p.miss_flags = sc.MISS_FLAGS_SKYBOX_CUBE
    _bitwise_images(oracle_mod, glsl, fs, p, 48, 36, 0, 2, 1, "img_sky_cube", "cube skybox")


def test_config_scenes_bitwise(oracle_mod, glsl):
    """The stand-ins of BASELINE configs 2-5 (alpha-tested cards + decals, attenuating glass, 64 point lights)."""
    import scenes_small

    for name, (make, bounces, _) in scenes_small.SMALL.items():
        scene = make()
        params = scene.default_params(bounce_count=bounces)
        # the camera was built for scenes_small.W x H: same aspect ratio at 64 x 48
        c = _bitwise_images(oracle_mod, glsl, scene, params, 64, 48, 0, 1, 2, f"img_config_{name}", name)
        assert c["rays_closest"] > 64 * 48


@pytest.mark.parametrize("mode", gc.DEBUG_MODES)
def test_debug_pipeline_bitwise(oracle_mod, glsl, default_scene, mode):
    """Debug/debugRaygen.rgen main() per pixel, dispatching to the compiled debugAnyhit / debugClosestHit / debugMiss (and
    occlusionAnyhit / occlusion.rmiss for the shadow rays), against pto_debug_render: every render mode x force-opaque,
    back-face culling and every hit-group flag, on the Default scene and the feature scene (decals, transmission, lights)."""
    cases = gc.stage_scenes(default_scene)
    for scene_name in ("default", "feature"):
        scene, params, w, h = cases[scene_name][:4]
        ora = oracle_mod.OracleScene(scene)
        g = glsl and glsl.GlslScene(scene, ora)
        for rf, hf in gc.DEBUG_FLAG_SETS:
            want = g and g.debug_render(params, w, h, mode, rf, hf).reshape(-1, 4)
            got = ora.debug_render(params, w, h, mode, rf, hf)
            assert np.isfinite(got).all() and got[..., :3].max() > 0.05
            assert_shader_bits(gc.debug_key(scene_name, mode, rf, hf), got.reshape(-1, 4), want,
                               f"{scene_name} / {mode} / raygen {rf} / hit group {hf:#x}")


def test_debug_miss_skyboxes_bitwise(oracle_mod, glsl):
    sc = gc.sc
    rs = np.random.default_rng(9)
    fs = gc.scenes.feature_scene(width=48, height=36)
    fs.skybox_2d = sc.Texture((rs.uniform(0, 1, (16, 32, 4)) * 255).astype(np.uint8), srgb=True)
    p = fs.default_params(bounce_count=4)
    p.miss_flags = sc.MISS_FLAGS_SKYBOX_2D
    ora = oracle_mod.OracleScene(fs)
    assert_shader_bits("dbg_miss_sky_2d", ora.debug_render(p, 48, 36, "color").reshape(-1, 4),
                       glsl and glsl.GlslScene(fs, ora).debug_render(p, 48, 36, "color").reshape(-1, 4), "debugMiss.rmiss, 2-D skybox")
    fs.skybox_2d = None
    fs.skybox_cube = [sc.Texture(rs.uniform(0, 4, (8, 8, 4)).astype(np.float32), srgb=False) for _ in range(6)]
    p.miss_flags = sc.MISS_FLAGS_SKYBOX_CUBE
    ora = oracle_mod.OracleScene(fs)
    assert_shader_bits("dbg_miss_sky_cube", ora.debug_render(p, 48, 36, "color").reshape(-1, 4),
                       glsl and glsl.GlslScene(fs, ora).debug_render(p, 48, 36, "color").reshape(-1, 4), "debugMiss.rmiss, cube skybox")
