"""numpy float32 reference of adaptive sampling (DESIGN.md §3i, pt_render_adaptive): the per-pixel Welford update of the
samples' luminance, the stop rule of an 8x4 block and the pass schedule, replayed from per-sample radiance images.

Every operation is a float32 operation in the order the kernels perform it (the library is built with -fmad=false), so
the statistics and the schedule match the device bit for bit."""
import numpy as np

f32 = np.float32
EPS = f32(0.01)  # the relMSE denominator's epsilon (metrics.rel_mse)
BLOCK_W, BLOCK_H = 8, 4
DEFAULT_MIN_PASS_ITEMS = 1 << 21
NONE = 0xFFFFFFFF


def luminance(rgb):
    rgb = np.asarray(rgb, f32)
    return (f32(0.2126) * rgb[..., 0] + f32(0.7152) * rgb[..., 1]) + f32(0.0722) * rgb[..., 2]


class State:
    """Per pixel: count (uint32), mean and m2 (float32), as pt_adaptive_readback returns them."""

    def __init__(self, height, width):
        self.count = np.zeros((height, width), np.uint32)
        self.mean = np.zeros((height, width), f32)
        self.m2 = np.zeros((height, width), f32)

    def copy(self):
        s = State(*self.count.shape)
        s.count, s.mean, s.m2 = self.count.copy(), self.mean.copy(), self.m2.copy()
        return s


def welford(state, lum, mask=None):
    """One sample of luminance lum (H, W) for the pixels in mask: n += 1; d = l - mean; mean += d / n; M2 += d (l - mean)."""
    m = np.ones(state.count.shape, bool) if mask is None else mask
    l = np.asarray(lum, f32)[m]
    n = state.count[m] + np.uint32(1)
    d = l - state.mean[m]
    mean = state.mean[m] + d / n.astype(f32)
    state.m2[m] = state.m2[m] + d * (l - mean)
    state.mean[m] = mean
    state.count[m] = n


def converged(count, mean, m2, threshold):
    """M2 <= t^2 (mean^2 + 0.01) n (n - 1), evaluated left to right in float32."""
    t = f32(threshold)
    n = np.asarray(count, np.uint32)
    return m2 <= t * t * (mean * mean + EPS) * n.astype(f32) * (n - np.uint32(1)).astype(f32)


def block_ids(height, width):
    """(H, W) index of the 8x4 block (aligned at (0, 0), row-major over blocks) of every pixel, and the block count."""
    bw, bh = -(-width // BLOCK_W), -(-height // BLOCK_H)
    y, x = np.mgrid[0:height, 0:width]
    return (y // BLOCK_H) * bw + x // BLOCK_W, bw * bh


def evaluate(state, min_samples, max_samples, threshold):
    """Per block: its count, whether it is active, and its pixels that miss the threshold."""
    ids, nb = block_ids(*state.count.shape)
    bad = np.bincount(ids.ravel(), (~converged(state.count, state.mean, state.m2, threshold)).ravel(), nb).astype(np.int64)
    count = np.zeros(nb, np.int64)
    count[ids.ravel()] = state.count.ravel()  # the pixels of a block share their count
    active = (count < min_samples) | ((count < max_samples) & (bad > 0))
    return count, active, bad, ids


def render_adaptive(sample, state, min_samples, max_samples, batch, threshold, min_pass_items=0):
    """Replays pt_render_adaptive on `state` (changed in place).  sample(s) is the (H, W, 3) radiance of sample s of every
    pixel.  Returns pt_adaptive_info as a dict and the list of passes (n, k, pixel mask)."""
    mpi = min_pass_items or DEFAULT_MIN_PASS_ITEMS
    passes, total = [], 0
    cache = {}
    while True:
        count, active, bad, ids = evaluate(state, min_samples, max_samples, threshold)
        if not active.any():
            break
        n = int(count[active].min())
        above = count[active & (count > n)]
        nxt = int(above.min()) if above.size else NONE
        mask = (active & (count == n))[ids]
        a = int(mask.sum())
        to = min(max_samples, nxt, max(n + batch, min_samples, n + -(-mpi // a)))
        for s in range(n, to):
            if s not in cache:
                cache[s] = luminance(sample(s))
            welford(state, cache[s], mask)
        passes.append((n, to - n, mask))
        total += a * (to - n)
    count, active, bad, _ = evaluate(state, min_samples, max_samples, threshold)
    info = {"passes": len(passes), "min_count": int(state.count.min()), "max_count": int(state.count.max()),
            "unconverged_pixels": int(bad[count >= max_samples].sum()), "samples": total}
    return info, passes
