"""The case generators of the traversal hit-for-hit tests (traversal_cases.py), checked on the CPU: the meshes are closed
and share their vertices, the rays aim where they claim to, and split_levels replays k_split_count."""
import numpy as np
import pytest

import traversal_cases as tc

F = np.float32


@pytest.mark.parametrize("mesh", [lambda: tc.icosphere(3), lambda: tc.tessellated_cube(16)], ids=["icosphere", "cube"])
def test_meshes_are_closed_with_shared_vertices(mesh):
    pos, tris = mesh()
    assert len(np.unique(pos, axis=0)) == len(pos)  # every position stored once
    e = np.concatenate([tris[:, [0, 1]], tris[:, [1, 2]], tris[:, [2, 0]]]).astype(np.int64)
    directed, counts = np.unique(e, axis=0, return_counts=True)
    assert (counts == 1).all()  # consistently oriented
    assert len(tc.edges_of(tris)) * 2 == len(directed)  # every edge has two triangles


def test_cube_vertices_are_binary_fractions():
    pos, _ = tc.tessellated_cube(16)
    assert (pos * 8 == np.round(pos * 8)).all() and np.abs(pos).max() == 1


def test_watertight_rays_aim_at_their_targets():
    pos, tris = tc.icosphere(2)
    rays, inc, tgt = tc.watertight_rays(pos, tris, np.random.default_rng(1), per_target=1)
    p = pos.astype(np.float64)
    on_edge = np.linalg.norm(np.cross(tgt - p[inc[:, 0]], p[inc[:, 1]] - p[inc[:, 0]]), axis=1)
    assert (on_edge <= 1e-12).all()  # every target lies on its vertex / edge
    o, d = rays["origin"].astype(np.float64), rays["direction"].astype(np.float64)
    # the vertex targets: the ray passes the vertex within float32 rounding of its direction
    vert = inc[:, 0] == inc[:, 1]
    s = ((tgt - o) * d).sum(1)
    miss = np.linalg.norm(o + s[:, None] * d - tgt, axis=1)
    assert (s > 0).all() and (miss <= 1e-6).all()  # float32 rounding of the origin and the direction only
    assert (vert.sum() == len(pos) * 5) and (~vert).any()
    # the origins lie inside the mesh: behind every face plane
    n = np.cross(p[tris[:, 1]] - p[tris[:, 0]], p[tris[:, 2]] - p[tris[:, 0]])
    side = np.einsum("fk,rfk->rf", n, o[:, None, :] - p[tris[:, 0]][None])
    assert (side < 0).all() or (side > 0).all()


def test_axis_rays_are_axis_parallel_with_signed_zeros():
    pos, tris = tc.tessellated_cube(16)
    rays, inc = tc.axis_rays(pos, tris)
    d = rays["direction"]
    assert ((d != 0).sum(1) == 1).all()
    zero = d == 0
    assert np.signbit(d[zero]).any() and (~np.signbit(d[zero])).any()
    # the ray crosses its target exactly: the two other coordinates of the origin are the target's
    p = pos.astype(np.float64)
    tgt = 0.5 * (p[inc[:, 0]] + p[inc[:, 1]])
    assert (rays["origin"][zero] == tgt[zero]).all()


def test_split_levels_hand_worked():
    # 5 triangles: four unit-size ones around a big one.  Centroid bounds (0..4)^3 -> share = 64 / 5 = 12.8
    small = np.array([[0, 0, 0], [0.5, 0, 0], [0, 0.5, 0.5]], F)
    pos = [small + F(4) * np.array(c, F) for c in ((0, 0, 0), (1, 1, 1), (1, 0, 1), (0, 1, 0))]
    # the big one: box 8 x 8 x 8 = 512 -> r = 40: level 1 (40 > 4), level 2 (5 > 4), not 3 (0.625)
    big = np.array([[-2, -2, -2], [6, 6, 2], [2, 2, 6]], F)
    tri = np.stack(pos + [big])
    levels = tc.split_levels(tri, 4.0)
    # the centroid bounds include the big triangle's centre (2, 2, 2): still (0.125 .. 4.125)^3
    lo, hi = tri.min(1), tri.max(1)
    c = F(0.5) * (lo + hi)
    ext = c.max(0) - c.min(0)
    share = ext.prod(dtype=F) / F(5)
    r = F(512) / share
    expect = int(r > 4) + int(r / 8 > 4) + int(r / 64 > 4)
    assert levels.tolist() == [0, 0, 0, 0, expect] and expect == 2
    assert tc.reference_count(tri, 400) == 4 + 16
    assert tc.reference_count(tri, 0) == 5
    assert tc.reference_count(tri, 3200) == 4 + 4  # r = 40 > 32: one level
    # the guard: 4 triangles are one leaf and are never split
    assert tc.split_levels(tri[1:], 4.0).tolist() == [0, 0, 0, 0]
    assert tc.reference_count(tri[1:], 400) == 4


def test_split_levels_caps_at_three_and_skips_non_finite():
    tri = np.zeros((6, 3, 3), F)
    tri[:, 1, 0] = tri[:, 2, 1] = 1e-3
    tri += F(10) * np.arange(6, dtype=F)[:, None, None]  # centroid bounds about 50^3 (the huge one is in the middle)
    # huge: box 1000^3 centred in the scene, r = 1e9 / (50^3 / 6) = 48000: past 4 even after three levels, capped at 3
    tri[0] = [[-480, -480, -480], [520, 520, -480], [20, 520, 520]]
    assert tc.split_levels(tri, 4.0).tolist() == [3, 0, 0, 0, 0, 0]
    assert tc.reference_count(tri, 400) == 64 + 5
    tri[1, 0, 0] = np.inf  # a non-finite box: the scene extent is infinite, nothing is split
    assert tc.split_levels(tri, 4.0).tolist() == [0] * 6


def test_threshold_rounding_matches_the_library():
    assert tc.threshold_of(400) == F(4.0) and tc.threshold_of(3200) == F(32.0)
    assert tc.threshold_of(1) == F(1) / F(100)


def test_split_scene_has_every_level():
    s, tri, cards = tc.split_scene()
    assert len(tri) == s.instanced_triangle_count()
    lv = tc.split_levels(tri, 4.0)
    assert set(np.unique(lv[cards]).tolist()) >= {1, 2, 3}
    assert (lv[: cards[0]] == 0).all()  # the small triangles stay whole
    rays, tid = tc.split_line_rays(tri, cards, np.random.default_rng(2))
    assert len(rays) == 3 * len(cards) * len(tc.subdivision_points())
    # barycentrics on multiples of 1/8 only, the level-3 lines included, all inside the card
    b = tc.subdivision_points()
    assert ((b * 8) == np.round(b * 8)).all() and ((b * 8) % 2 == 1).any()
    assert (b > 0).all() and (b.sum(1) < 1).all() and len(b) == 21
