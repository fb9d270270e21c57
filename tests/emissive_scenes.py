"""Scenes and numpy restatements for the emissive-triangle light sampling tests (DESIGN.md §3g)."""
import importlib

import numpy as np

scenes = importlib.import_module("path-tracing_b200.scenes")
sc = importlib.import_module("path-tracing_b200.scene")


def room(width=32, height=24, emitters=True, point_light=True):
    """A closed box room (rough walls) lit by several untextured emissive quads of different sizes and colours under
    the ceiling, and one point light."""
    b = scenes.SceneBuilder()
    # ior 1: no Fresnel term, so the lobe the reference samples and the pdf evaluateBSDF reports agree and its BSDF-sampled
    # estimator is unbiased (with ior 1.5 the sampled lobe follows F(V.H) of the sampled half vector but the pdf follows
    # F of the outgoing direction's half vector, and the two modes converge to slightly different images)
    wall = b.add_material_mr(color=(0.7, 0.7, 0.7, 1), roughness=0.8, ior=1.0)
    red = b.add_material_mr(color=(0.8, 0.2, 0.2, 1), roughness=0.6, ior=1.0)
    g_quad = b.add_geometry(*scenes.quad(1.0, 1.0))
    size = 4.0

    def place(model, *transforms):
        t = np.eye(4)
        for m in transforms:
            t = t @ m
        b.add_instance(model, t)

    m_wall = b.add_model([(g_quad, wall, None)])
    m_red = b.add_model([(g_quad, red, None)])
    place(m_wall, scenes.scale(size))                                                              # floor, facing +y
    place(m_wall, scenes.translate(0, size, 0), scenes.rotate_x(180), scenes.scale(size))          # ceiling
    place(m_wall, scenes.translate(0, size / 2, -size / 2), scenes.rotate_x(90), scenes.scale(size))   # back
    place(m_red, scenes.translate(-size / 2, size / 2, 0), scenes.rotate_y(90), scenes.rotate_x(90), scenes.scale(size))
    place(m_wall, scenes.translate(size / 2, size / 2, 0), scenes.rotate_y(-90), scenes.rotate_x(90), scenes.scale(size))
    place(m_wall, scenes.translate(0, size / 2, size / 2), scenes.rotate_x(-90), scenes.scale(size))   # front
    lamps = [((1.0, 0.9, 0.7), 12.0, 0.6, (-1.0, -1.0)), ((0.4, 0.6, 1.0), 30.0, 0.3, (1.0, -0.5)),
             ((1.0, 0.3, 0.2), 8.0, 0.9, (0.2, 1.0))]
    for color, intensity, s, (x, z) in lamps:
        m = b.add_material_mr(color=(1, 1, 1, 1), emissive=color, emissive_intensity=intensity if emitters else 0.0)
        place(b.add_model([(g_quad, m, None)]), scenes.translate(x, size - 0.05, z), scenes.rotate_x(180), scenes.scale(s))
    if point_light:
        b.add_light((3.0, 3.0, 3.0), (0.5, 2.0, 0.5), 1.0, 0.0, 0.3)
    camera = scenes.camera_matrices((0.0, 2.0, 1.9), (0.0, -0.1, -1.0), width, height, fov_deg=70)
    return b.build(camera, (width, height))


def flat_triangles(s):
    """Flattened triangles (instance, mesh in model, primitive) in float64: corners (n, 3, 3), uvs (n, 3, 2), material
    ids, opaque flags."""
    P, UV, MAT, OPQ = [], [], [], []
    for inst in s.instances:
        inst_m = np.vstack([inst["transform"].reshape(3, 4).astype(np.float64), [0, 0, 0, 1]])
        m = s.models[int(inst["model_index"])]
        for j in range(int(m["mesh_count"])):
            rec = s.mesh_records[int(m["mesh_offset"]) + j]
            g = s.geometries[int(rec["geometry_index"])]
            mesh_m = np.vstack([s.transforms[int(rec["transform_index"])].reshape(3, 4).astype(np.float64), [0, 0, 0, 1]])
            idx = s.indices[int(g["index_offset"]):int(g["index_offset"]) + int(g["index_length"])].astype(np.int64)
            v = s.vertices[idx + int(g["vertex_offset"])]
            p = np.c_[v["position"].astype(np.float64), np.ones(len(v))] @ (inst_m @ mesh_m).T
            P.append(p[:, :3].reshape(-1, 3, 3))
            UV.append(v["texcoords"].astype(np.float64).reshape(-1, 3, 2))
            MAT.append(np.full(len(idx) // 3, int(rec["material_id"]), np.uint32))
            OPQ.append(np.full(len(idx) // 3, bool(g["is_opaque"])))
    return np.concatenate(P), np.concatenate(UV), np.concatenate(MAT), np.concatenate(OPQ)


def emissive_fields(s, material_id):
    mtype, index = material_id & 0xFF, material_id >> 8
    table = {sc.MATERIAL_TYPE_MR: s.mr_materials, sc.MATERIAL_TYPE_SG: s.sg_materials}.get(mtype, s.phong_materials)
    m = table[index]
    return np.asarray(m["emissive_color"], np.float64), float(m["emissive_intensity"]), int(m["emissive_idx"])


def emitter_weights(s, oracle_scene):
    """The emitter set (flat ids) and integer weights restated in numpy (float64): opaque triangles whose material has
    intensity > 0 and a non-zero emissive colour or a texture other than the black built-in slots 4, 6, 7; power =
    area x luminance((colour + textureGrad at the UV centroid over the UV extent) x intensity)."""
    P, UV, MAT, OPQ = flat_triangles(s)
    ids, power = [], []
    for f in range(len(P)):
        color, intensity, slot = emissive_fields(s, int(MAT[f]))
        if not OPQ[f] or not intensity > 0 or (not color.any() and slot in (4, 6, 7)):
            continue
        area = 0.5 * np.linalg.norm(np.cross(P[f, 1] - P[f, 0], P[f, 2] - P[f, 0]))
        u, v = UV[f].mean(0)
        du, dv = np.ptp(UV[f][:, 0]), np.ptp(UV[f][:, 1])
        t = oracle_scene.texture_sample(slot, np.array([u, v, du, 0, 0, dv], np.float32))[0, :3].astype(np.float64)
        e = (t + color) * intensity
        p = area * max(0.2126 * e[0] + 0.7152 * e[1] + 0.0722 * e[2], 0.0)
        if p > 0:
            ids.append(f)
            power.append(p)
    power = np.array(power)
    w = np.maximum(1, np.rint(power / power.max() * 2.0**24)) if len(power) else power
    return np.array(ids, np.uint32), w


def alias_probabilities(t):
    """The exact selection probability of every entry implied by an alias table."""
    n = len(t["weights"])
    keep = t["alias_threshold"].astype(np.float64) / 2.0**32
    p = keep / n
    np.add.at(p, t["alias_index"].astype(np.int64), (1.0 - keep) / n)
    return p


def alias_draws(t, count, seed=7):
    """count draws through the table with 32-bit bucket and fraction words, as the renderers draw."""
    rs = np.random.default_rng(seed)
    n = len(t["weights"])
    hi = rs.integers(0, 2**32, count, dtype=np.uint64)
    lo = rs.integers(0, 2**32, count, dtype=np.uint64)
    bucket = ((hi * np.uint64(n)) >> np.uint64(32)).astype(np.int64)
    keep = lo < t["alias_threshold"][bucket].astype(np.uint64)
    return np.where(keep, bucket, t["alias_index"][bucket].astype(np.int64))
