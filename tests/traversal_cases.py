"""Scenes and ray sets that aim at the places where a BVH traversal goes wrong, each with what the answer must be.

Every mesh here stores each position once and every instance transform is the identity (or an exact translation), so
the triangles k_bake builds are known exactly: meshes are closed where they are meant to be, and a ray aimed at a vertex
or an edge really crosses it.  split_levels replays k_split_count (bvh_build.cu) in float32 to predict the references
the BVH is built from."""
import importlib

import numpy as np

sc = importlib.import_module("path-tracing_b200.scene")
scenes = importlib.import_module("path-tracing_b200.scenes")

F = np.float32
TMIN = 1e-5  # the tmin of the render's trace kernels
SPLIT_MAX_LEVEL = 3  # PT_SPLIT_MAX_LEVEL
MAX_LEAF_TRIS = 4  # PT_MAX_LEAF_TRIS: a scene this small is one leaf and is never split


# ---------------------------------------------------------------------------------------------
# closed meshes with shared vertices
# ---------------------------------------------------------------------------------------------
def icosphere(subdivisions: int, radius: float = 1.0):
    """Subdivided icosahedron: (positions (V, 3) float32, indices (T, 3)), every edge midpoint computed once."""
    t = (1 + 5 ** 0.5) / 2
    pos = [(-1, t, 0), (1, t, 0), (-1, -t, 0), (1, -t, 0), (0, -1, t), (0, 1, t), (0, -1, -t), (0, 1, -t),
           (t, 0, -1), (t, 0, 1), (-t, 0, -1), (-t, 0, 1)]
    pos = [np.array(p, np.float64) / np.linalg.norm(p) for p in pos]
    tris = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6),
            (7, 1, 8), (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10),
            (8, 6, 7), (9, 8, 1)]
    for _ in range(subdivisions):
        mid = {}

        def m(a, b):
            k = (min(a, b), max(a, b))
            if k not in mid:
                p = pos[a] + pos[b]
                pos.append(p / np.linalg.norm(p))
                mid[k] = len(pos) - 1
            return mid[k]

        tris = [q for a, b, c in tris for q in ((a, m(a, b), m(c, a)), (b, m(b, c), m(a, b)), (c, m(c, a), m(b, c)),
                                               (m(a, b), m(b, c), m(c, a)))]
    return (np.array(pos) * radius).astype(F), np.array(tris, np.uint32)


def tessellated_cube(n: int = 16, half: float = 1.0):
    """Axis-aligned cube [-half, half]^3, every face an n x n grid of quads split along one diagonal.  With half = 1 and
    n = 16 every vertex lies on a multiple of 1/8, so the BVH's quantised planes can fall exactly on the faces."""
    index = {}
    pos = []

    def vid(p):
        k = tuple(p)
        if k not in index:
            index[k] = len(pos)
            pos.append(k)
        return index[k]

    g = np.linspace(-half, half, n + 1)
    tris = []
    for axis in range(3):
        for side in (-half, half):
            for i in range(n):
                for j in range(n):
                    q = []
                    for di, dj in ((0, 0), (1, 0), (1, 1), (0, 1)):
                        p = [0.0, 0.0, 0.0]
                        p[axis] = side
                        p[(axis + 1) % 3], p[(axis + 2) % 3] = g[i + di], g[j + dj]
                        q.append(vid(p))
                    a, b, c, d = q if side > 0 else q[::-1]
                    tris += [(a, b, c), (a, c, d)]
    return np.array(pos, F), np.array(tris, np.uint32)


def mesh_vertices(pos: np.ndarray) -> np.ndarray:
    v = np.zeros(len(pos), sc.VERTEX)
    v["position"] = pos
    c = pos.astype(np.float64)
    n = c / np.maximum(np.linalg.norm(c, axis=1, keepdims=True), 1e-30)
    v["normal"] = n
    v["tangent"], v["bitangent"] = (1, 0, 0), (0, 1, 0)
    v["texcoords"] = 0.5 + 0.5 * c[:, :2] / max(1e-30, np.abs(c).max())
    return v


def edges_of(tris: np.ndarray) -> np.ndarray:
    """Unique undirected edges (E, 2) of a triangle list."""
    e = np.concatenate([tris[:, [0, 1]], tris[:, [1, 2]], tris[:, [2, 0]]]).astype(np.int64)
    return np.unique(np.sort(e, axis=1), axis=0)


def camera():
    return scenes.camera_matrices((0, 0, -4), (0, 0, 1), 32, 32), (32, 32)


def mesh_scene(pos: np.ndarray, tris: np.ndarray, translations=((0, 0, 0),)):
    """One geometry, instanced once per translation (exact: k_bake adds the translation last, and the tests use
    translations by small binary fractions)."""
    b = scenes.SceneBuilder()
    g = b.add_geometry(mesh_vertices(pos), tris.reshape(-1))
    m = b.add_model([(g, b.add_material_mr(color=(0.8, 0.8, 0.8, 1)), None)])
    for t in translations:
        b.add_instance(m, scenes.translate(*t))
    return b.build(*camera())


def rays_of(origin, direction, tmax=1e4) -> np.ndarray:
    r = np.zeros(len(origin), sc.RAY)
    r["origin"], r["direction"] = origin, direction
    r["tmin"], r["tmax"] = TMIN, tmax
    return r


# ---------------------------------------------------------------------------------------------
# ray classes
# ---------------------------------------------------------------------------------------------
def watertight_rays(pos: np.ndarray, tris: np.ndarray, rs: np.random.Generator, per_target: int = 2,
                    distances=(1e-1, 1e-2, 1e-3, 1e-4, 1e-5)):
    """Rays from inside a closed, convex mesh (centred on the origin) aimed at its vertices and at points of its edges
    (midpoints and quarter points), starting `distance * size` away from the target.  Returns (rays, incident): incident
    (N, 2) holds the targeted vertex twice or the targeted edge's two vertices; every ray must hit a triangle that
    contains both.  Also returns the targets (N, 3) float64.  The mesh's size is the largest coordinate."""
    size = float(np.abs(pos).max())
    p = pos.astype(np.float64)
    e = edges_of(tris)
    targets = [p, 0.5 * (p[e[:, 0]] + p[e[:, 1]]), 0.75 * p[e[:, 0]] + 0.25 * p[e[:, 1]]]
    incident = [np.stack([np.arange(len(p))] * 2, 1), e, e]
    tgt = np.concatenate(targets)
    inc = np.concatenate(incident)
    origins, dirs, incs, tgts = [], [], [], []
    for d in distances:
        for _ in range(per_target):
            # towards the inside: the inward direction (to the centre) tilted at random by up to ~35 degrees
            inward = -tgt / np.linalg.norm(tgt, axis=1, keepdims=True)
            w = inward + 0.4 * rs.normal(size=tgt.shape) / np.sqrt(3)
            w /= np.linalg.norm(w, axis=1, keepdims=True)
            o = (tgt + d * size * w).astype(F)
            dd = (tgt - o.astype(np.float64))
            origins.append(o)
            dirs.append((dd / np.linalg.norm(dd, axis=1, keepdims=True)).astype(F))
            incs.append(inc)
            tgts.append(tgt)
    o = np.concatenate(origins)
    # near a convex corner the tilted origin can end up outside the mesh: keep the rays that start behind every face
    a, n = p[tris[:, 0].astype(np.int64)], np.cross(p[tris[:, 1]] - p[tris[:, 0]], p[tris[:, 2]] - p[tris[:, 0]])
    inside = np.ones(len(o), bool)
    for k in range(0, len(o), 2048):
        oc = o[k:k + 2048].astype(np.float64)
        inside[k:k + 2048] = (oc @ n.T < (a * n).sum(1)).all(1)
    return (rays_of(o[inside], np.concatenate(dirs)[inside]), np.concatenate(incs)[inside], np.concatenate(tgts)[inside])


def axis_rays(pos: np.ndarray, tris: np.ndarray, half: float = 1.0):
    """Axis-parallel rays of a tessellated_cube: from inside, along +-x / +-y / +-z with the two other components +0 or
    -0, through every vertex and every grid-edge midpoint strictly inside a face.  The ray crosses its target exactly
    (the coordinates are binary fractions).  Returns (rays, incident) like watertight_rays."""
    e = edges_of(tris)
    p = pos.astype(np.float64)
    cand = [(p, np.stack([np.arange(len(p))] * 2, 1)), (0.5 * (p[e[:, 0]] + p[e[:, 1]]), e)]
    origins, dirs, incs = [], [], []
    rs = np.random.default_rng(7)
    for pts, inc in cand:
        on_face = np.abs(np.abs(pts) - half) == 0
        keep = on_face.sum(1) == 1  # strictly inside one face
        pts, inc = pts[keep], inc[keep]
        axis = np.argmax(on_face[keep], 1)
        sign = np.sign(pts[np.arange(len(pts)), axis])
        for depth in (0.5, 1e-3, 1e-5):
            o = pts.copy()
            o[np.arange(len(o)), axis] -= sign * depth * half
            d = np.zeros_like(o)
            # the two other components: +0 or -0 at random
            d[:] = np.where(rs.random(d.shape) < 0.5, 0.0, -0.0)
            d[np.arange(len(d)), axis] = sign
            origins.append(o.astype(F))
            dirs.append(d.astype(F))
            incs.append(inc)
    return rays_of(np.concatenate(origins), np.concatenate(dirs)), np.concatenate(incs)


def incident_ok(hit_prim: np.ndarray, tris: np.ndarray, incident: np.ndarray) -> np.ndarray:
    """Per ray: the hit primitive (an index into tris) contains both vertices of `incident`."""
    ok = hit_prim < len(tris)
    t = tris[np.where(ok, hit_prim, 0)].astype(np.int64)
    has = lambda v: (t == v[:, None]).any(1)  # noqa: E731
    return ok & has(incident[:, 0]) & has(incident[:, 1])


def floor_scene(n: int = 363):
    """A gently undulating floor of 2 n^2 triangles (n = 363: 263538) and a box on it: the grazing rays of straggler
    splitting."""
    v, i = scenes.grid(n, n, 40.0, 40.0, height=lambda x, z: 0.05 * np.sin(1.3 * x) * np.cos(0.7 * z))
    b = scenes.SceneBuilder()
    g = b.add_geometry(v, i)
    bv, bi = scenes.box(2.0, 1.0, 2.0)
    g2 = b.add_geometry(bv, bi)
    mat = b.add_material_mr(color=(0.7, 0.7, 0.7, 1))
    b.add_instance(b.add_model([(g, mat, None), (g2, mat, scenes.translate(3.0, 0.5, 1.0))]))
    return b.build(*camera())


def straggler_rays(rs: np.random.Generator, n: int):
    """Grazing rays from far outside the floor (each visits thousands of nodes) mixed 1:3 with short rays."""
    graze = rs.random(n) < 0.25
    o = np.empty((n, 3))
    d = np.empty((n, 3))
    ang = rs.uniform(0, 2 * np.pi, n)
    o[:, 0], o[:, 2] = 60 * np.cos(ang), 60 * np.sin(ang)
    o[:, 1] = rs.uniform(0.06, 0.3, n)
    tgt = np.stack([rs.uniform(-15, 15, n), np.zeros(n), rs.uniform(-15, 15, n)], 1)
    d[:] = tgt - o
    # short rays: from just above the floor, steeply down or sideways
    o2 = np.stack([rs.uniform(-18, 18, n), rs.uniform(0.1, 2.0, n), rs.uniform(-18, 18, n)], 1)
    d2 = rs.normal(size=(n, 3))
    d2[:, 1] = -np.abs(d2[:, 1]) - 0.2
    o = np.where(graze[:, None], o, o2)
    d = np.where(graze[:, None], d, d2)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return rays_of(o.astype(F), d.astype(F))


def nan_rays(rs: np.random.Generator, n: int):
    """Rays as k_extend meets them after total internal reflection: NaN directions (normalize(0)), a few zero and
    infinite ones, among ordinary rays.  Only the ordinary ones can hit."""
    o = rs.uniform(-2.5, 2.5, (n, 3))
    d = rs.uniform(-0.3, 0.3, (n, 3)) - o  # the ordinary rays aim at the middle of the scene
    r = rays_of(o.astype(F), (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(F))
    bad = rs.random(n) < 0.5
    kind = rs.integers(0, 4, n)
    d = r["direction"]
    d[bad & (kind == 0)] = np.nan
    d[bad & (kind == 1), 0] = np.nan
    d[bad & (kind == 2)] = 0.0
    d[bad & (kind == 3), 2] = np.inf
    return r, bad


# ---------------------------------------------------------------------------------------------
# reference splitting
# ---------------------------------------------------------------------------------------------
def split_levels(tri_pos: np.ndarray, threshold: float) -> np.ndarray:
    """k_split_count in float32: the subdivision level (0..3) of every triangle of (n, 3, 3) baked positions at a split
    threshold (the value of "split_threshold_x100" / 100 as the library rounds it).  The BVH then holds
    sum(4 ** level) references."""
    p = np.asarray(tri_pos, F)
    n = len(p)
    levels = np.zeros(n, np.int64)
    thr = F(threshold)
    if not thr > 0 or n <= MAX_LEAF_TRIS:
        return levels
    lo, hi = p.min(1), p.max(1)
    c = F(0.5) * (lo + hi)
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        ext = np.maximum(c.max(0) - c.min(0), F(1e-20))
        share = ((ext[0] * ext[1]) * ext[2]) / F(n)
        d = hi - lo
        r = ((d[:, 0] * d[:, 1]) * d[:, 2]) / share
        active = np.ones(n, bool)
        for _ in range(SPLIT_MAX_LEVEL):
            active &= (r > thr) & np.isfinite(r)
            levels += active
            r = np.where(active, r * F(0.125), r)
    return levels


def threshold_of(split_threshold_x100: int) -> float:
    """The float the library makes of the tuning value: (float)value / 100.0f."""
    return F(split_threshold_x100) / F(100)


def reference_count(tri_pos: np.ndarray, split_threshold_x100: int) -> int:
    """bvh_reference_count the build must report."""
    levels = split_levels(tri_pos, threshold_of(split_threshold_x100))
    total = int((4 ** levels).sum())
    return total if total < (1 << 29) else len(levels)


def _alpha_texture(n: int = 32) -> np.ndarray:
    """Leaf-like alpha: an opaque disc with a transparent ring and holes (RGBA8)."""
    y, x = np.mgrid[0:n, 0:n] / (n - 1) * 2 - 1
    r = np.hypot(x, y)
    a = np.where((r < 0.9) & ~((r > 0.45) & (r < 0.55)) & ~((np.abs(x) < 0.08) & (y > 0)), 255, 0)
    rgba = np.zeros((n, n, 4), np.uint8)
    rgba[..., 0], rgba[..., 1], rgba[..., 2], rgba[..., 3] = 60 + 120 * (x > 0), 140, 40 + 100 * (y > 0), a
    return rgba


def split_scene(seed: int = 3, small: int = 4000, cards: int = 60):
    """Many small triangles and randomly oriented large alpha-tested cards — a small version of the atrium's foliage.
    Returns (scene, tri_pos (n, 3, 3) float32 in flattened order, card_ids (flat ids of the cards))."""
    rs = np.random.default_rng(seed)
    # small triangles in a 4 x 2 x 4 box
    c = rs.uniform([-2, 0, -2], [2, 2, 2], (small, 1, 3))
    p_small = (c + rs.normal(scale=0.03, size=(small, 3, 3))).astype(F)
    # cards: big triangles, sizes 0.5 .. 2.5, random orientation, centres in the same box
    sizes = rs.uniform(0.5, 2.5, cards)
    q, _ = np.linalg.qr(rs.normal(size=(cards, 3, 3)))
    tri = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0]]) - 1 / 3
    centres = rs.uniform([-2, 0, -2], [2, 2, 2], (cards, 3))
    p_cards = (np.einsum("cij,kj->cki", q, tri) * sizes[:, None, None] + centres[:, None, :]).astype(F)
    b = scenes.SceneBuilder()

    def geometry(p, opaque, uv):
        v = np.zeros(3 * len(p), sc.VERTEX)
        v["position"] = p.reshape(-1, 3)
        n = np.cross(p[:, 1] - p[:, 0], p[:, 2] - p[:, 0]).astype(np.float64)
        n /= np.maximum(np.linalg.norm(n, axis=1, keepdims=True), 1e-30)
        v["normal"] = np.repeat(n, 3, 0)
        v["tangent"], v["bitangent"] = (1, 0, 0), (0, 1, 0)
        v["texcoords"] = np.tile(uv, (len(p), 1))
        return b.add_geometry(v, np.arange(3 * len(p), dtype=np.uint32), is_opaque=opaque)

    g0 = geometry(p_small, True, np.array([[0, 0], [1, 0], [0, 1]], F))
    # (card texture coordinates off the texel grid: a subdivision point is never a bilinear tie at alpha 0.5)
    g1 = geometry(p_cards, False, np.array([[0.013, 0.021], [0.971, 0.034], [0.027, 0.983]], F))
    leaf = b.add_texture(_alpha_texture(), srgb=True)
    m0 = b.add_material_mr(color=(0.6, 0.6, 0.6, 1))
    m1 = b.add_material_mr(color=(1, 1, 1, 1), color_idx=leaf)
    b.add_instance(b.add_model([(g0, m0, None), (g1, m1, None)]))
    b.add_light((2, 2, 2), (0, 4, 0))
    s = b.build(scenes.camera_matrices((0, 1, -6), (0, 0, 1), 64, 48), (64, 48))
    return s, np.concatenate([p_small, p_cards]), np.arange(small, small + cards)


def subdivision_points(levels_max: int = 3):
    """Barycentrics (b1, b2) on the level-1, -2 and -3 subdivision lines and points inside a triangle: every (i, j) / 2^L
    with i, j > 0 and i + j < 2^L.  (Points on the triangle's own edges are left out: whether a ray through the edge of
    a lone triangle hits is a tie either way.)"""
    pts = set()
    for L in range(1, levels_max + 1):
        m = 2 ** L
        for i in range(1, m):
            for j in range(1, m - i):
                pts.add((i / m, j / m))
    return np.array(sorted(pts))


def split_line_rays(tri_pos: np.ndarray, card_ids: np.ndarray, rs: np.random.Generator, distances=(0.05, 0.7, 6.0)):
    """Rays at the subdivision lines and points of every card, from several distances and random sides.  Returns
    (rays, target flat id)."""
    bary = subdivision_points()
    p = tri_pos[card_ids].astype(np.float64)
    b1, b2 = bary[:, 0], bary[:, 1]
    tgt = (1 - b1 - b2)[None, :, None] * p[:, None, 0] + b1[None, :, None] * p[:, None, 1] + b2[None, :, None] * p[:, None, 2]
    tgt = tgt.reshape(-1, 3)
    ids = np.repeat(card_ids, len(bary))
    origins, dirs, tid = [], [], []
    for dist in distances:
        w = rs.normal(size=tgt.shape)
        w /= np.linalg.norm(w, axis=1, keepdims=True)
        o = (tgt + dist * w).astype(F)
        d = tgt - o
        origins.append(o)
        dirs.append((d / np.linalg.norm(d, axis=1, keepdims=True)).astype(F))
        tid.append(ids)
    return rays_of(np.concatenate(origins), np.concatenate(dirs)), np.concatenate(tid)
