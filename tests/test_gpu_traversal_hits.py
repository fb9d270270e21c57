"""The traversal the render runs, hit for hit.

k_extend and k_shadow trace through tracePersistent (dynamic ray fetch, deferred commits, straggler splitting with its
merge and decal hand-off); the standalone queries run the per-thread traverse().  pt_test_trace runs either on the same
rays, so the two can be compared bit for bit, and both are held against the oracle and a float64 brute force on ray sets
aimed at the places where traversals go wrong: vertices and edges of closed meshes seen from just inside, grazing rays
of a finely tessellated floor, ties between coincident instances, alpha-tested cards, NaN rays, and the subdivision
lines of reference-split triangles."""
import importlib

import numpy as np
import pytest

import conftest
import traversal_cases as tc
from test_gpu_traversal import compare_hits
from test_oracle_traversal import random_rays

pytestmark = pytest.mark.gpu
sc = conftest.pkg.scene
scenes = importlib.import_module("path-tracing_b200.scenes")

MODES = [dict(blocks=0, stats=False), dict(blocks=0, stats=True), dict(blocks=1, stats=False), dict(blocks=1, stats=True)]


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_same_hits(a, b, occlusion, what):
    if occlusion:
        diff = (a["instance"] != sc.NO_HIT) != (b["instance"] != sc.NO_HIT)
    else:
        diff = ((a["instance"] != b["instance"]) | (a["geometry"] != b["geometry"]) | (a["primitive"] != b["primitive"]) |
                (bits(a["t"]) != bits(b["t"])) | (bits(a["u"]) != bits(b["u"])) | (bits(a["v"]) != bits(b["v"])))
    assert not diff.any(), f"{what}: {int(diff.sum())} of {len(a)} rays differ, first at {np.flatnonzero(diff)[:8]}"


def effective_decal(hits, decals):
    """The decal k_shade applies: recorded (dist != -1) and in front of the hit (dist < t)."""
    on = (hits["instance"] != sc.NO_HIT) & (decals[:, 4] != -1) & (decals[:, 4] < hits["t"])
    return on, np.where(on[:, None], decals, 0)


def persistent_equals_per_thread(r, rays, occlusion=False, tag=""):
    """Every (blocks, stats) variant of the persistent traversal gives the per-thread answer bit for bit.  Returns the
    per-thread hits and the tail counters of the stats runs."""
    ref, ref_dec, tail = r.test_trace(rays, occlusion=occlusion, persistent=False)
    assert tail["stack_overflows"] == 0
    on_ref, dec_ref = effective_decal(ref, ref_dec)
    tails = {}
    for m in MODES:
        h, d, tail = r.test_trace(rays, occlusion=occlusion, persistent=True, **m)
        what = f"{tag} {'occlusion' if occlusion else 'closest'} persistent {m}"
        assert_same_hits(h, ref, occlusion, what)
        assert tail["stack_overflows"] == 0, what
        if not occlusion:
            on, dec = effective_decal(h, d)
            assert (on == on_ref).all() and (bits(dec) == bits(dec_ref)).all(), what
        if m["stats"]:
            tails[m["blocks"]] = tail
            assert tail["warp_drain_iterations"] > 0, what  # the drain mode (and its donations) ran
            print(f"{what}: {len(rays)} rays, tail {tail}")
    # the standalone queries are the per-thread traversal
    if occlusion:
        assert ((ref["instance"] != sc.NO_HIT) == (r.trace_occlusion(rays) != 0)).all()
    else:
        assert_same_hits(r.trace_closest(rays), ref, False, f"{tag} pt_trace_closest")
    return ref, tails


@pytest.fixture(scope="module")
def gpu():
    r = conftest.core.Renderer(0)
    yield r
    r.close()


def test_entry_point_rejects_mixed_tmin(gpu):
    pos, tris = tc.icosphere(1)
    gpu.update_scene_data(tc.mesh_scene(pos, tris))
    rays = tc.rays_of(np.zeros((4, 3), np.float32), np.tile(np.float32([0, 0, 1]), (4, 1)))
    rays["tmin"][2] = 1e-3
    with pytest.raises(conftest.core.PtError):
        gpu.test_trace(rays)
    rays["tmin"] = 1e-5
    h, _, _ = gpu.test_trace(rays)
    assert (h["instance"] == 0).all()


# ---------------------------------------------------------------------------------------------
# watertightness: vertices and edges of closed meshes, seen from just inside
# ---------------------------------------------------------------------------------------------
SIZE = 4.0  # mesh size: the closest origin (1e-5 of it) is still beyond tmin = 1e-5


def watertight_case(mesh):
    if mesh == "icosphere":
        pos, tris = tc.icosphere(3, SIZE)
    else:
        pos, tris = tc.tessellated_cube(16, SIZE)  # vertices on multiples of 1/2: planes exactly on the faces
    rays, inc, _ = tc.watertight_rays(pos, tris, np.random.default_rng(11))
    if mesh == "cube":
        ar, ai = tc.axis_rays(pos, tris, SIZE)
        rays, inc = np.concatenate([rays, ar]), np.concatenate([inc, ai])
    return pos, tris, tc.mesh_scene(pos, tris), rays, inc


@pytest.mark.parametrize("mesh", ["icosphere", "cube"])
def test_watertight_vertices_and_edges(gpu, oracle_mod, mesh):
    """No ray leaks through a closed mesh, with the per-thread or the persistent traversal: each one hits a triangle
    incident to its target, at the float64 distance."""
    pos, tris, s, rays, inc = watertight_case(mesh)
    gpu.update_scene_data(s)
    bf, t64 = oracle_mod.OracleScene(s).trace_closest_bruteforce_f64(rays)
    f = bf["instance"] != sc.NO_HIT  # (the float64 test is not watertight: it can miss exactly at a vertex)
    assert f.mean() > 0.99
    for persistent, m in [(False, {})] + [(True, m) for m in MODES]:
        what = f"{mesh} persistent={persistent} {m}"
        hits, _, tail = gpu.test_trace(rays, persistent=persistent, **m)
        occ, _, _ = gpu.test_trace(rays, occlusion=True, persistent=persistent, **m)
        assert tail["stack_overflows"] == 0
        leak = hits["instance"] == sc.NO_HIT
        assert not leak.any(), f"{what}: {int(leak.sum())} of {len(rays)} rays leak through the closed {mesh}"
        assert (occ["instance"] != sc.NO_HIT).all(), what
        ok = tc.incident_ok(hits["primitive"], tris, inc)
        assert ok.all(), f"{what}: {int((~ok).sum())} rays hit a triangle that does not touch their target"
        # t against float64: 1e-5 relative, plus the absolute rounding of the float32 vertex - origin differences
        err = np.abs(hits["t"][f] - t64[f])
        assert (err <= 1e-5 * t64[f] + 4 * np.finfo(np.float32).eps * SIZE).all(), (what, err.max())


@pytest.mark.parametrize("mesh", ["icosphere", "cube"])
def test_watertight_ties_persistent_equals_per_thread(gpu, mesh):
    """A ray through a shared vertex or edge meets several triangles at (nearly) the same t: the winner must not depend
    on the order the traversal visits them in.  (Before the box test widened its planes by their absolute rounding, a
    few rays in 10^3 of these sets resolved differently.)"""
    pos, tris, s, rays, inc = watertight_case(mesh)
    gpu.update_scene_data(s)
    persistent_equals_per_thread(gpu, rays, tag=mesh)


# ---------------------------------------------------------------------------------------------
# stragglers: grazing rays over a 262k-triangle floor, at ray counts around a fetch chunk and a warp
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def floor(gpu, oracle_mod):
    s = tc.floor_scene()
    gpu.update_scene_data(s)
    assert gpu.stats()["triangle_count"] >= 256 * 1024
    return s, oracle_mod.OracleScene(s)


@pytest.mark.parametrize("n", [1, 31, 32, 33, 95, 4103, 200003])
def test_stragglers(gpu, floor, n):
    s, o = floor
    gpu.update_scene_data(s)
    rays = tc.straggler_rays(np.random.default_rng(n), n)
    hits, tails = persistent_equals_per_thread(gpu, rays, tag=f"floor n={n}")
    rays["tmax"] = np.random.default_rng(n + 1).uniform(0.5, 80, n).astype(np.float32)
    persistent_equals_per_thread(gpu, rays, occlusion=True, tag=f"floor n={n}")
    if n <= 4103:
        rays["tmax"] = 1e4
        compare_hits(hits, o.trace_closest(rays), rays)


# ---------------------------------------------------------------------------------------------
# ties: one mesh instanced twice with one transform — every hit is a tie in t, the smaller flat id wins
# ---------------------------------------------------------------------------------------------
def test_coincident_instances_resolve_to_the_smaller_id(gpu):
    pos, tris = tc.icosphere(3, 1.0)
    gpu.update_scene_data(tc.mesh_scene(pos, tris, translations=((0.25, 0, 0), (0.25, 0, 0))))
    rs = np.random.default_rng(5)
    o = rs.normal(size=(20000, 3))
    o = 3 * o / np.linalg.norm(o, axis=1, keepdims=True)
    d = rs.uniform(-0.8, 0.8, o.shape) + [0.25, 0, 0] - o
    rays = tc.rays_of(o.astype(np.float32), (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32))
    hits, _ = persistent_equals_per_thread(gpu, rays, tag="ties")
    hit = hits["instance"] != sc.NO_HIT
    assert hit.mean() > 0.3 and (hits["instance"][hit] == 0).all()


# ---------------------------------------------------------------------------------------------
# alpha: the feature scene's cards and decals; shadow rays that end exactly on a surface
# ---------------------------------------------------------------------------------------------
def test_alpha_cards_and_decals(gpu, oracle_mod):
    s = scenes.feature_scene()
    gpu.update_scene_data(s)
    o = oracle_mod.OracleScene(s)
    rays = random_rays(np.random.default_rng(31), 60000, [-4, 0.2, -4], [4, 3.5, 4])
    hits, _ = persistent_equals_per_thread(gpu, rays, tag="feature")
    compare_hits(hits, o.trace_closest(rays), rays)
    _, decals, _ = gpu.test_trace(rays, persistent=False)
    assert effective_decal(hits, decals)[0].any()  # the set reaches the decal path
    rays["tmax"] = np.random.default_rng(32).uniform(0.05, 8, len(rays)).astype(np.float32)
    persistent_equals_per_thread(gpu, rays, occlusion=True, tag="feature")
    # shadow rays whose tmax is exactly the distance of the closest surface: that surface does not occlude
    hit = hits["instance"] != sc.NO_HIT
    sh = rays[hit].copy()
    sh["tmax"] = hits["t"][hit]
    occ, _ = persistent_equals_per_thread(gpu, sh, occlusion=True, tag="feature tmax = t")
    mismatch = (occ["instance"] != sc.NO_HIT) != (o.trace_occlusion(sh) != 0)
    assert not mismatch.any(), f"{int(mismatch.sum())} of {len(sh)} shadow rays ending on a surface disagree with the oracle"


def test_nan_rays_miss(gpu):
    pos, tris = tc.icosphere(2, 1.0)
    gpu.update_scene_data(tc.mesh_scene(pos, tris))
    rays, bad = tc.nan_rays(np.random.default_rng(9), 5000)
    hits, _ = persistent_equals_per_thread(gpu, rays, tag="nan")
    occ, _ = persistent_equals_per_thread(gpu, rays, occlusion=True, tag="nan")
    assert (hits["instance"][bad] == sc.NO_HIT).all() and (occ["instance"][bad] == sc.NO_HIT).all()
    assert (hits["instance"][~bad] != sc.NO_HIT).mean() > 0.9


# ---------------------------------------------------------------------------------------------
# reference splitting
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def split(oracle_mod):
    s, tri, cards = tc.split_scene()
    rs = np.random.default_rng(17)
    lines, target = tc.split_line_rays(tri, cards, rs)
    rand = random_rays(rs, 20000, [-3, -0.5, -3], [3, 2.5, 3])
    return s, tri, cards, lines, target, rand, oracle_mod.OracleScene(s)


def test_split_lines_hit_their_card(gpu, split):
    """Default splitting: the persistent traversal equals the per-thread one; a ray aimed at a subdivision line or point
    of a card hits that card wherever the float64 brute force says the card is the first thing it meets."""
    s, tri, cards, lines, target, rand, o = split
    gpu.set_tuning("split_threshold_x100", 400)
    gpu.update_scene_data(s)
    levels = tc.split_levels(tri, tc.threshold_of(400))
    assert set(np.unique(levels).tolist()) == {0, 1, 2, 3}
    assert gpu.stats()["bvh_reference_count"] == tc.reference_count(tri, 400)
    hits, _ = persistent_equals_per_thread(gpu, lines, tag="split lines")
    persistent_equals_per_thread(gpu, lines, occlusion=True, tag="split lines")
    bf, t64 = o.trace_closest_bruteforce_f64(lines)
    first = (bf["instance"] != sc.NO_HIT) & (bf["primitive"] == target - cards[0]) & (bf["geometry"] == 1)
    assert first.mean() > 0.5
    got = (hits["geometry"] == 1) & (hits["primitive"] == target - cards[0])
    assert got[first].all(), f"{int((~got[first]).sum())} of {int(first.sum())} rays miss the card they aim at"
    # t against float64 where the ray meets the card at a reasonable angle (t is ill-conditioned at grazing angles)
    c = tri[target].astype(np.float64)
    n = np.cross(c[:, 1] - c[:, 0], c[:, 2] - c[:, 0])
    cos = np.abs((n * lines["direction"]).sum(1)) / np.linalg.norm(n, axis=1)
    chk = first & (cos > 0.1)
    scale = np.abs(lines["origin"][chk]).max(1) + np.abs(c[chk]).max((1, 2))
    assert (np.abs(hits["t"][chk] - t64[chk]) <= 1e-5 * t64[chk] + 4 * np.finfo(np.float32).eps * scale).all()
    rh, _ = persistent_equals_per_thread(gpu, rand, tag="split random")
    compare_hits(rh, o.trace_closest(rand), rand)


def test_splitting_changes_nothing_but_the_tree(split):
    s, tri, cards, lines, target, rand, o = split
    rays = np.concatenate([lines, rand])
    occ_rays = rays.copy()
    occ_rays["tmax"] = np.random.default_rng(3).uniform(0.05, 6, len(rays)).astype(np.float32)
    ref = None
    with conftest.core.Renderer(0) as r:
        for thr in (0, 100, 400, 3200):
            for builder in (0, 1):
                for radius in (1, 8, 64, 200):  # 200 is clamped to 64
                    r.set_tuning("split_threshold_x100", thr)
                    r.set_tuning("bvh_builder", builder)
                    r.set_tuning("ploc_radius", radius)
                    r.update_scene_data(s)
                    st = r.stats()
                    what = f"threshold {thr / 100} builder {builder} radius {radius}"
                    assert st["triangle_count"] == len(tri), what
                    assert st["bvh_reference_count"] == tc.reference_count(tri, thr), what
                    got = (r.trace_closest(rays), r.trace_occlusion(occ_rays), r.test_trace(rays)[0],
                           r.test_trace(occ_rays, occlusion=True)[0])
                    if ref is None:
                        ref = got
                        continue
                    assert_same_hits(got[0], ref[0], False, what + " pt_trace_closest")
                    assert (got[1] == ref[1]).all(), what + " pt_trace_occlusion"
                    assert_same_hits(got[2], ref[0], False, what + " persistent closest")
                    assert_same_hits(got[3], ref[3], True, what + " persistent occlusion")
    assert ((ref[3]["instance"] != sc.NO_HIT) == (ref[1] != 0)).all()


@pytest.mark.parametrize("count", [4, 5])
def test_split_guard_on_tiny_scenes(count):
    """Four large triangles are one leaf and stay whole; five are split.  Either way the hits are those of the unsplit
    scene."""
    rs = np.random.default_rng(count)
    p = (rs.uniform(-1, 1, (count, 3, 3)) * [[4, 4, 4]] + rs.uniform(-0.05, 0.05, (count, 1, 3))).astype(np.float32)
    v = np.zeros(3 * count, sc.VERTEX)
    v["position"] = p.reshape(-1, 3)
    v["normal"], v["tangent"], v["bitangent"] = (0, 0, -1), (1, 0, 0), (0, 1, 0)
    b = scenes.SceneBuilder()
    g = b.add_geometry(v, np.arange(3 * count, dtype=np.uint32))
    b.add_instance(b.add_model([(g, b.add_material_mr(), None)]))
    s = b.build(*tc.camera())
    rays = random_rays(rs, 20000, [-3, -3, -3], [3, 3, 3])
    expect = tc.reference_count(p, 400)
    assert (expect == 4) if count == 4 else (expect > 5)
    out = []
    with conftest.core.Renderer(0) as r:
        for thr in (400, 0):
            r.set_tuning("split_threshold_x100", thr)
            r.update_scene_data(s)
            assert r.stats()["bvh_reference_count"] == (expect if thr else count)
            out.append((r.trace_closest(rays), r.test_trace(rays)[0]))
    for h in (out[0][0], out[0][1], out[1][1]):
        assert_same_hits(h, out[1][0], False, f"{count} triangles")


def test_render_is_identical_with_and_without_splitting(split):
    """The wavefront (k_extend / k_shade / k_shadow) over the split BVH renders the unsplit scene's image bit for bit."""
    s = split[0]
    params = s.default_params(bounce_count=4)
    imgs = []
    with conftest.core.Renderer(0) as r:
        for thr in (0, 400):
            r.set_tuning("split_threshold_x100", thr)
            r.update_scene_data(s)
            r.on_resize(64, 48)
            r.render(4, params=params)
            imgs.append(r.read_accumulation().copy())
    assert np.isfinite(imgs[0]).all() and imgs[0][..., :3].max() > 0
    assert np.array_equal(bits(imgs[0]), bits(imgs[1]))
