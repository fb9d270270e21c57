"""numpy reference of the temporal denoiser (path-tracing_b200/csrc/temporal.cu, DESIGN.md §3j).

Follows k_temporal_reproject operation for operation in float32 (the library is built with -fmad=false): the pixel-centre
primary ray of constructPrimaryRay, the world point, Cramer's rule in the previous camera, the 2x2 bilinear taps with their
depth and normal tests, and the moving averages.  Prepare, the 7x7 variance and the a-trous levels are denoise_ref's.  The
reference also marks the pixels where one of its decisions lies within 1e-5 relative of its threshold (a tap test, s > 0,
an image bound, the 1e-3 weight floor): there a last-bit difference could flip it."""
import numpy as np

import denoise_ref as dr

F = np.float32
DEPTH_TOLERANCE = F(0.02)
NORMAL_TOLERANCE = F(0.9)
MIN_HISTORY_WEIGHT = F(1e-3)
MAX_HISTORY = F(65535)
MOMENTS_HISTORY = F(4)
MARGIN = 1e-5


def _mul_point(m, x, y, z, w):
    """mulPoint (shading.cuh): (M * vec4).xyz of a column-major 4x4, summed pairwise."""
    m = np.asarray(m, F).reshape(-1)
    return [(m[r] * x + m[4 + r] * y) + (m[8 + r] * z + m[12 + r] * w) for r in range(3)]


def _dot(a, b):
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]


def _cross(a, b):
    return [a[1] * b[2] - b[1] * a[2], a[2] * b[0] - b[2] * a[0], a[0] * b[1] - b[0] * a[1]]


def camera_rays(view, proj, width, height):
    """constructPrimaryRay's pixel-centre ray of every pixel, lens_radius = 0: origin (3,) and direction (H, W, 3)."""
    px = np.arange(width, dtype=F)[None, :] + F(0.5)
    py = np.arange(height, dtype=F)[:, None] + F(0.5)
    dx = np.broadcast_to(px / F(width) * F(2) - F(1), (height, width))
    dy = np.broadcast_to(py / F(height) * F(2) - F(1), (height, width))
    target = _mul_point(proj, dx, dy, F(1), F(1))
    inv = F(1) / np.sqrt(_dot(target, target))
    d0 = [c * inv for c in target]
    origin = np.array(_mul_point(view, F(0), F(0), F(0), F(1)), F)
    return origin, np.stack(_mul_point(view, d0[0], d0[1], d0[2], F(0)), -1).astype(F)


def reproject(view, proj, prev_view, prev_proj, t, width, height):
    """The previous pixel position (x', y') of the world point X = O + t D of every pixel, its distance |X - O'| from the
    previous camera, whether it lies in front of it (s > 0), and the marks of those decisions.  A camera whose matrices are
    bit-identical to the previous ones maps every pixel onto itself."""
    origin, d = camera_rays(view, proj, width, height)
    t = np.asarray(t, F)
    X = [origin[k] + t * d[..., k] for k in range(3)]
    pv = np.asarray(prev_view, F).reshape(-1)
    r = [X[k] - pv[12 + k] for k in range(3)]
    dist = np.sqrt(_dot(r, r))
    identity = np.array_equal(np.asarray(view, F).view(np.uint32), np.asarray(prev_view, F).view(np.uint32)) and \
        np.array_equal(np.asarray(proj, F).view(np.uint32), np.asarray(prev_proj, F).view(np.uint32))
    if identity:
        xp = np.broadcast_to(np.arange(width, dtype=F)[None, :], t.shape).copy()
        yp = np.broadcast_to(np.arange(height, dtype=F)[:, None], t.shape).copy()
        return {"x": xp, "y": yp, "dist": dist, "front": np.ones(t.shape, bool), "mark": np.zeros(t.shape, bool), "identity": True}
    pp = np.asarray(prev_proj, F).reshape(-1)
    A = _mul_point(pv, pp[0], pp[1], pp[2], F(0))
    B = _mul_point(pv, pp[4], pp[5], pp[6], F(0))
    C = _mul_point(pv, pp[8] + pp[12], pp[9] + pp[13], pp[10] + pp[14], F(0))
    det = F(_dot(A, _cross(B, C)))
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        d1, d2, d3 = _dot(r, _cross(B, C)), _dot(A, _cross(r, C)), _dot(A, _cross(B, r))
        s = d3 / det
        xp = (d1 / d3 + F(1)) * F(0.5) * F(width) - F(0.5)
        yp = (d2 / d3 + F(1)) * F(0.5) * F(height) - F(0.5)
        mark = np.abs(s) <= MARGIN * np.fmax(np.abs(s), np.fmax(np.abs(d1 / det), np.abs(d2 / det)))
        for v, n in ((xp, width), (yp, height)):
            for bound in (-1, 0, n - 1, n):
                mark |= np.abs(v - F(bound)) <= MARGIN * max(1, abs(bound))
    return {"x": xp, "y": yp, "dist": dist, "front": s > 0, "mark": mark, "identity": False}


def step(g, view, proj, prev, alpha=0.2, alpha_moments=0.2):
    """k_temporal_reproject: g is denoise_ref.prepare's output of this frame; prev is None (no history) or the previous
    state: {"view", "proj", "t" (invalid = -1), "n" (normals), "irr" (H, W, 4) = (I.rgb, length), "moments" (H, W, 2)}.
    Returns the new state (the same keys, for the next step) with "mark"."""
    h, w = g["t"].shape
    valid = g["valid"]
    sw = np.zeros((h, w), F)
    s4 = np.zeros((h, w, 4), F)
    sm = np.zeros((h, w, 2), F)
    mark = np.zeros((h, w), bool)
    if prev is not None:
        rp = reproject(view, proj, prev["view"], prev["proj"], g["t"], w, h)
        mark |= rp["mark"]
        with np.errstate(invalid="ignore"):
            inside = rp["front"] & (rp["x"] >= -1) & (rp["x"] < w) & (rp["y"] >= -1) & (rp["y"] < h)
            fx0 = np.floor(np.where(inside, rp["x"], F(0))).astype(F)
            fy0 = np.floor(np.where(inside, rp["y"], F(0))).astype(F)
        x0, y0 = fx0.astype(np.int64), fy0.astype(np.int64)
        fx, fy = np.where(inside, rp["x"], F(0)) - fx0, np.where(inside, rp["y"], F(0)) - fy0
        for k in range(4):
            qx, qy = x0 + (k & 1), y0 + (k >> 1)
            ok = inside & valid & (qx >= 0) & (qy >= 0) & (qx < w) & (qy < h)
            cx, cy = np.clip(qx, 0, w - 1), np.clip(qy, 0, h - 1)
            tq, nq = prev["t"][cy, cx], prev["n"][cy, cx]
            dev = np.abs(tq - rp["dist"])
            tol = DEPTH_TOLERANCE * rp["dist"]
            cos = _dot([nq[..., j] for j in range(3)], [g["n"][..., j] for j in range(3)])
            with np.errstate(invalid="ignore"):
                mark |= ok & (tq >= 0) & (np.abs(dev - tol) <= MARGIN * tol)
                mark |= ok & (tq >= 0) & (np.abs(cos - NORMAL_TOLERANCE) <= MARGIN * NORMAL_TOLERANCE)
                ok &= (tq >= 0) & (dev <= tol) & (cos >= NORMAL_TOLERANCE)
            wk = np.where(ok, ((fx if k & 1 else F(1) - fx) * (fy if k >> 1 else F(1) - fy)).astype(F), F(0))
            sw = np.where(ok, sw + wk, sw)
            s4 = np.where(ok[..., None], s4 + wk[..., None] * prev["irr"][cy, cx], s4)
            sm = np.where(ok[..., None], sm + wk[..., None] * prev["moments"][cy, cx], sm)
        mark |= valid & (np.abs(sw - MIN_HISTORY_WEIGHT) <= MARGIN * MIN_HISTORY_WEIGHT)
    keep = sw >= MIN_HISTORY_WEIGHT
    with np.errstate(invalid="ignore", divide="ignore"):
        hist = np.where(keep[..., None], s4 / sw[..., None], F(0)).astype(F)
        mom = np.where(keep[..., None], sm / sw[..., None], F(0)).astype(F)
    n = np.fmin(hist[..., 3] + F(1), MAX_HISTORY)
    a, am = np.fmax(F(alpha), F(1) / n), np.fmax(F(alpha_moments), F(1) / n)
    i = g["irr"]
    irr = hist[..., :3] + a[..., None] * (i - hist[..., :3])
    l = dr.luminance(i)
    m1 = mom[..., 0] + am * (l - mom[..., 0])
    m2 = mom[..., 1] + am * (l * l - mom[..., 1])
    v = valid[..., None]
    out = {
        "view": np.asarray(view, F), "proj": np.asarray(proj, F), "t": g["t"], "n": g["n"],
        "irr": np.where(v, np.concatenate([irr, n[..., None]], -1), F(0)).astype(F),
        "moments": np.where(v, np.stack([m1, m2], -1), F(0)).astype(F),
    }
    out["mark"] = valid & mark
    return out


def filter_state(g, albedo, state, iterations=5, sigma_luminance=4.0, sigma_normal=128.0, sigma_depth=1.0):
    """The filter of pt_denoise_temporal on a state: the variance (temporal where n >= 4, else the 7x7 estimate on I), K
    a-trous levels and the remodulation; K = 0 is I * max(albedo, 1e-3).  Invalid pixels keep c.  (H, W, 4), A = 1."""
    v = g["valid"]
    I = state["irr"][..., :3]
    out = np.concatenate([g["c"], np.ones(g["c"].shape[:2] + (1,), F)], -1)
    if iterations > 0:
        gi = dict(g, irr=I)
        m = state["moments"]
        var = np.where(state["irr"][..., 3] >= MOMENTS_HISTORY, np.fmax(F(0), m[..., 1] - m[..., 0] * m[..., 0]),
                       dr.variance(gi, sigma_normal, sigma_depth)).astype(F)
        for k in range(iterations):
            I, var = dr.atrous_level(gi, I, var, 1 << k, sigma_luminance, sigma_normal, sigma_depth)
            I, var = np.where(v[..., None], I, F(0)).astype(F), np.where(v, var, F(0)).astype(F)
    out[v, :3] = I[v] * np.fmax(np.asarray(albedo, F)[..., :3], dr.ALBEDO_FLOOR)[v]
    return out


def denoise_temporal(accum, total_samples, albedo_t, normal, view, proj, prev, iterations=5, sigma_luminance=4.0,
                     sigma_normal=128.0, sigma_depth=1.0, alpha=0.2, alpha_moments=0.2):
    """pt_denoise_temporal on host arrays (prev = None: no history).  Returns (output (H, W, 4), state)."""
    g = dr.prepare(accum, total_samples, albedo_t, normal)
    state = step(g, view, proj, prev, alpha, alpha_moments)
    return filter_state(g, albedo_t, state, iterations, sigma_luminance, sigma_normal, sigma_depth), state
