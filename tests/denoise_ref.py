"""numpy reference of the denoiser (path-tracing_b200/csrc/denoise.cu, DESIGN.md §3h).

Follows the kernels operation for operation in float32 (the library is built with -fmad=false, so neither side contracts
a multiply-add): the same sums in the same tap order, the same ε values.  Only expf / powf may differ from numpy's in the
last bits."""
import numpy as np

F = np.float32
ALBEDO_FLOOR = F(1e-3)
EPS_DEPTH = F(1e-4)
EPS_LUMINANCE = F(1e-10)
VARIANCE_RADIUS = 3
H5 = np.array([0.0625, 0.25, 0.375, 0.25, 0.0625], F)  # B3 spline (1, 4, 6, 4, 1) / 16


def luminance(c):
    return F(0.2126) * c[..., 0] + F(0.7152) * c[..., 1] + F(0.0722) * c[..., 2]


def shifted(a, dx, dy, fill):
    """out[y, x] = a[y + dy, x + dx], `fill` where that lies outside the image."""
    h, w = a.shape[:2]
    out = np.full_like(a, fill)
    y0, y1 = min(h, max(0, -dy)), max(0, min(h, h - dy))
    x0, x1 = min(w, max(0, -dx)), max(0, min(w, w - dx))
    if y0 < y1 and x0 < x1:
        out[y0:y1, x0:x1] = a[y0 + dy : y1 + dy, x0 + dx : x1 + dx]
    return out


def normal_weight(n_p, n_q, sigma_normal):
    d = n_p[..., 0] * n_q[..., 0] + n_p[..., 1] * n_q[..., 1] + n_p[..., 2] * n_q[..., 2]
    return np.power(np.fmax(F(0), d), F(sigma_normal))


def depth_weight(t_p, t_q, grad, dx, dy, sigma_depth):
    return np.exp(-np.abs(t_p - t_q) / (F(sigma_depth) * np.abs(grad[..., 0] * F(dx) + grad[..., 1] * F(dy)) + EPS_DEPTH))


def depth_slope(t, tb, tf):
    db, df = t - tb, tf - t
    hb, hf = tb >= 0, tf >= 0
    return np.where(hb & hf, np.where(np.abs(df) <= np.abs(db), df, db), np.where(hf, df, np.where(hb, db, F(0)))).astype(F)


def prepare(accum, total_samples, albedo_t, normal):
    """k_denoise_prepare: mean radiance c, validity, (N, t) taps, demodulated irradiance and the depth gradient."""
    c = accum[..., :3].astype(F) / F(total_samples)
    t = albedo_t[..., 3].astype(F)
    with np.errstate(invalid="ignore", over="ignore"):
        valid = (t >= 0) & np.isfinite(c).all(-1)
        irr = np.where(valid[..., None], c / np.fmax(albedo_t[..., :3].astype(F), ALBEDO_FLOOR), F(0)).astype(F)
        grad = np.stack([depth_slope(t, shifted(t, -1, 0, F(-1)), shifted(t, 1, 0, F(-1))),
                         depth_slope(t, shifted(t, 0, -1, F(-1)), shifted(t, 0, 1, F(-1)))], -1)
    return {"c": c, "valid": valid, "t": np.where(valid, t, F(-1)).astype(F), "n": normal[..., :3].astype(F), "irr": irr, "grad": grad}


def variance(g, sigma_normal, sigma_depth):
    """k_denoise_variance: luminance variance over the 7x7 window, taps weighted by w_n * w_z (the centre by 1), moments
    taken about l_p."""
    lp = luminance(g["irr"])
    sw, s1, s2 = (np.zeros_like(lp) for _ in range(3))
    for dy in range(-VARIANCE_RADIUS, VARIANCE_RADIUS + 1):
        for dx in range(-VARIANCE_RADIUS, VARIANCE_RADIUS + 1):
            t_q = shifted(g["t"], dx, dy, F(-1))
            ok = t_q >= 0
            if dx == 0 and dy == 0:
                w = np.ones_like(lp)
            else:
                with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
                    w = normal_weight(g["n"], shifted(g["n"], dx, dy, F(0)), sigma_normal) * depth_weight(
                        g["t"], t_q, g["grad"], dx, dy, sigma_depth)
            w = np.where(ok, w, F(0)).astype(F)
            d = luminance(shifted(g["irr"], dx, dy, F(0))) - lp
            sw = sw + w
            s1 = s1 + w * d
            s2 = s2 + w * d * d
    with np.errstate(invalid="ignore", divide="ignore"):
        m1 = s1 / sw
        var = np.fmax(F(0), s2 / sw - m1 * m1)
    return np.where(g["valid"], var, F(0)).astype(F)


def atrous_level(g, irr, var, step, sigma_luminance, sigma_normal, sigma_depth, return_weights=False):
    """k_atrous at step 2^k: (irradiance, variance) of the next level; with return_weights also the 25 normalised tap
    weights h w / sum(h w) of every pixel, (H, W, 25)."""
    sv, sk = np.zeros_like(var), np.zeros_like(var)
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            ok = shifted(g["t"], dx, dy, F(-1)) >= 0
            k = F((2 - abs(dx)) * (2 - abs(dy)))
            sv = sv + np.where(ok, k * shifted(var, dx, dy, F(0)), F(0))
            sk = sk + np.where(ok, k, F(0))
    with np.errstate(invalid="ignore", divide="ignore"):
        denom_l = F(sigma_luminance) * np.sqrt(sv / sk) + EPS_LUMINANCE
    lp = luminance(irr)
    acc, svar, sw = np.zeros_like(irr), np.zeros_like(var), np.zeros_like(var)
    taps = []
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            t_q = shifted(g["t"], dx * step, dy * step, F(-1))
            i_q = shifted(irr, dx * step, dy * step, F(0))
            v_q = shifted(var, dx * step, dy * step, F(0))
            if dx == 0 and dy == 0:
                w = np.ones_like(var)
            else:
                with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
                    w = normal_weight(g["n"], shifted(g["n"], dx * step, dy * step, F(0)), sigma_normal) * depth_weight(
                        g["t"], t_q, g["grad"], dx * step, dy * step, sigma_depth) * np.exp(-np.abs(lp - luminance(i_q)) / denom_l)
            hw = np.where(t_q >= 0, F(H5[dx + 2] * H5[dy + 2]) * w, F(0)).astype(F)
            acc = acc + hw[..., None] * i_q
            svar = svar + hw * hw * v_q
            sw = sw + hw
            taps.append(hw)
    with np.errstate(invalid="ignore", divide="ignore"):
        out = acc / sw[..., None], svar / (sw * sw)
    if return_weights:
        with np.errstate(invalid="ignore", divide="ignore"):
            return out, np.stack(taps, -1) / sw[..., None]
    return out


def denoise(accum, total_samples, albedo_t, normal, iterations=5, sigma_luminance=4.0, sigma_normal=128.0, sigma_depth=1.0):
    """pt_denoise on host arrays: accum (H, W, 4) sum, albedo_t (H, W, 4) = (albedo, t), normal (H, W, >= 3).
    Returns (H, W, 4) float32 mean radiance with A = 1."""
    g = prepare(accum, total_samples, albedo_t, normal)
    out = np.concatenate([g["c"], np.ones(g["c"].shape[:2] + (1,), F)], -1)
    if iterations == 0:
        return out
    irr, var = g["irr"], variance(g, sigma_normal, sigma_depth)
    v = g["valid"]
    for k in range(iterations):
        irr, var = atrous_level(g, irr, var, 1 << k, sigma_luminance, sigma_normal, sigma_depth)
        # invalid pixels take no part: keep their (unread) entries finite so that a 0 weight cancels them
        irr, var = np.where(v[..., None], irr, F(0)).astype(F), np.where(v, var, F(0)).astype(F)
    out[v, :3] = irr[v] * np.fmax(albedo_t[..., :3].astype(F), ALBEDO_FLOOR)[v]
    return out
