"""Seeded FP32 input sets for the denoiser's parity tests: the edge inputs of the filter (misses, non-finite inputs,
sample counts below two, clamped moments, albedo floors, depth ramps and scales, facets of nearly parallel normals) at
shapes that are not multiples of the 16x16 launch block.  Each set is the five arrays rt_denoise takes, with unit
normals for hits and (albedo 1, normal 0, depth -1) for misses as the feature kernel writes them, plus the counts it
claims, which tests/test_denoise_host.py recounts from the arrays (test infrastructure, like denoise_reference.py)."""
from __future__ import annotations

import numpy as np

SHAPES = [(1, 1), (1, 37), (37, 1), (3, 5), (16, 16), (17, 33), (33, 17), (7, 300)]  # (height, width)
KINDS = [
    "miss_block", "miss_border", "miss_single",
    "nonfinite_color", "nonfinite_albedo", "nonfinite_normal", "nonfinite_depth", "demod_overflow",
    "n0", "n1", "n2", "n64", "m2_zero", "m2_negative", "n_mixed",
    "albedo_edges", "depth_ramps", "depth_tiny", "depth_huge", "facets",
]
# the claim each kind exists for: it must be positive at every shape
DEFINES = {
    "miss_block": "misses", "miss_border": "misses", "miss_single": "misses",
    "nonfinite_color": "invalid", "nonfinite_albedo": "invalid", "nonfinite_normal": "invalid", "nonfinite_depth": "invalid",
    "demod_overflow": "invalid", "n0": "few_samples", "n1": "few_samples", "n_mixed": "few_samples",
    "m2_negative": "negative_m2", "albedo_edges": "zero_albedo",
}
N_BASE = 16
LIGHT, DARK = np.array([0.8, 0.6, 0.4]), np.array([0.05, 0.1, 0.2])


def _long_axis(H, W):
    """Position of every pixel along the image's longer axis, and that axis' length."""
    y, x = np.mgrid[0:H, 0:W]
    return (x, W) if W >= H else (y, H)


def _rot_y(deg):
    r = np.radians(deg)
    return np.array([np.sin(r), 0.0, np.cos(r)])


def _block(H, W, y0, y1, x0, x1):
    """Mask of rows [y0, y1) x columns [x0, x1), given as fractions of the image, at least one pixel on each axis."""
    m = np.zeros((H, W), bool)
    r0, c0 = min(int(y0 * H), H - 1), min(int(x0 * W), W - 1)
    m[r0:max(r0 + 1, int(y1 * H)), c0:max(c0 + 1, int(x1 * W))] = True
    return m


def make_case(kind: str, H: int, W: int, seed: int = 0):
    """(color, albedo, normal, depth, moments) as float32 arrays, and the counts the set claims."""
    rng = np.random.default_rng([seed, KINDS.index(kind), H, W])
    pos, L = _long_axis(H, W)
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    # base: hits on a gently tilted plane facing the camera, 4-pixel bands of two contrasting colours with noise
    band = (pos // 4) % 2 == 0
    mean = np.where(band[..., None], LIGHT, DARK)
    albedo = np.where(band[..., None], [0.7, 0.5, 0.3], [0.2, 0.4, 0.6]) * rng.uniform(0.9, 1.1, (H, W, 1))
    sd = 0.15 * mean * rng.uniform(0.5, 1.5, (H, W, 3))
    color = mean + sd * rng.standard_normal((H, W, 3))
    normal = np.zeros((H, W, 3))
    normal[..., 2] = 1.0
    depth = 2.0 + 0.01 * x + 0.005 * y
    n = np.full((H, W), float(N_BASE))
    m2 = sd * sd * (n - 1)[..., None]
    miss = np.zeros((H, W), bool)

    if kind == "miss_block":
        miss = _block(H, W, 0.25, 0.75, 0.3, 0.7)
        color[~miss] = np.where(band[~miss, None], [0.9, 0.9, 0.9], [0.02, 0.02, 0.02])  # contrasting hits around the sky
    elif kind == "miss_border":
        miss = _block(H, W, 0.0, 0.5, 0.0, 0.4)
    elif kind == "miss_single":
        miss = _block(H, W, 0.5, 0.5, 0.5, 0.5)
    elif kind == "m2_zero":
        color = mean.copy()  # noiseless bands: the luminance stop is a hard edge between them
        m2[:] = 0.0
    elif kind == "m2_negative":
        neg = rng.random((H, W)) < 0.3
        neg.flat[rng.integers(H * W)] = True
        m2[neg] = -np.abs(m2[neg]) - 1e-3
    elif kind in ("n0", "n1", "n2", "n64"):
        n[:] = float(kind[1:])
        m2 = sd * sd * np.maximum(n - 1, 0)[..., None]
        if kind == "n0":
            color[:] = 0.0
    elif kind == "n_mixed":
        few = rng.random((H, W)) < 0.1
        few.flat[rng.integers(H * W)] = True
        n[few] = rng.integers(0, 2, few.sum())
        m2[few] = 0.0
    elif kind == "albedo_edges":
        third = np.minimum(3 * pos // L, 2)
        albedo[third == 0] = [0.0, 0.5, 0.7]       # zero channel
        albedo[third == 1] = 0.0                   # all-zero: both floors of the filter apply
        albedo[third == 2] = [1.5, 2.0, 1.2]       # above 1
        color[third == 1] = 0.01 * rng.uniform(0.5, 1.5, (int((third == 1).sum()), 3))
        albedo[0, 0] = [0.6, 0.0, 0.0]             # every shape has a zero channel
    elif kind == "depth_ramps":
        # planar ramps of several slopes, one diagonal (both gradient components non-zero), jumps between them
        third = np.minimum(3 * pos // L, 2)
        depth = np.select([third == 0, third == 1, third == 2],
                          [3.0 + 0.05 * x, 6.0 + 0.03 * x - 0.04 * y, 4.0 + 0.4 * x + 0.25 * y])
        color = mean * (1.0 + 0.2 * rng.standard_normal((H, W, 1)))
    elif kind == "depth_tiny":
        depth = 1e-3 * (1.0 + 0.05 * x + 0.02 * y + 0.5 * (pos >= L // 2))
    elif kind == "depth_huge":
        depth = 1e4 * (1.0 + 0.001 * x + 0.002 * y + 0.3 * (pos >= L // 2))
    elif kind == "facets":
        # 0 | 4 deg | 90 deg | 8 deg facets along the long axis: w_n = cos^128 in its middle range and 0
        q = np.minimum(4 * pos // L, 3)
        for k, deg in enumerate((0.0, 4.0, 90.0, 8.0)):
            normal[q == k] = _rot_y(deg)
        m2 *= 4.0  # noisy enough that the luminance stop lets the normals decide

    color[miss] = color[miss] * 1.5
    albedo[miss] = 1.0
    normal[miss] = 0.0
    depth[miss] = -1.0
    sums = color * n[..., None]
    moments = np.concatenate([sums, m2, n[..., None], (3.0 * n)[..., None]], axis=-1)
    c, a, nm, z, m = (v.astype(np.float32) for v in (color, albedo, normal, depth, moments))

    invalid = np.zeros((H, W), bool)
    if kind.startswith("nonfinite_"):
        target = {"color": c, "albedo": a, "normal": nm, "depth": z}[kind[len("nonfinite_"):]]
        for (fy, fx), v in zip(((0.5, 0.5), (0.0, 0.99), (0.99, 0.0)), (np.nan, np.inf, -np.inf)):
            p = (min(int(fy * H), H - 1), min(int(fx * W), W - 1))
            if target.ndim == 3:
                target[p + (int(rng.integers(3)),)] = v
            else:
                target[p] = v
            invalid[p] = True
    elif kind == "demod_overflow":
        p = (H // 2, W // 2)
        c[p], a[p] = (3e38, 0.5, 0.5), (1e-3, 0.5, 0.5)  # finite colour; c / max(a, 1e-3) overflows FP32
        invalid[p] = True
    claims = {
        "misses": int((miss & ~invalid).sum()),
        "invalid": int(invalid.sum()),
        "few_samples": int((m[..., 6] < 2).sum()),
        "negative_m2": int((m[..., 3:6] < 0).any(-1).sum()),
        "zero_albedo": int((a == 0).any(-1).sum()),
    }
    return (c, a, nm, z, m), claims


OPTIONS = [
    ("defaults", {}),
    ("sl1.5", {"sigmaLuminance": 1.5}),
    ("sn16", {"sigmaNormal": 16.0}),
    ("sz4", {"sigmaDepth": 4.0}),
    ("zeros", {"sigmaLuminance": 0, "sigmaNormal": 0, "sigmaDepth": 0}),  # a sigma of 0 selects its default
]


def parity_sets():
    """(id, kind, (H, W), options) for the GPU parity test: every kind at three shapes, every shape, every iteration
    count 0..8 and every option set at least once."""
    out = []
    for r in range(3):
        for i, kind in enumerate(KINDS):
            H, W = SHAPES[(i + 3 * r) % len(SHAPES)]
            name, opts = OPTIONS[(i + r) % len(OPTIONS)]
            opts = {**opts, "iterations": (i + 4 * r) % 9}
            out.append((f"{kind}-{H}x{W}-it{opts['iterations']}-{name}", kind, (H, W), opts))
    return out
