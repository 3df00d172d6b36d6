"""Float64 numpy restatement of the denoiser (csrc/rt_denoise.cuh): the specification of the filter that rt_denoise and
rt_camera_render_denoised run in FP32 on the device (test infrastructure, like parity_stats.py).

The spatial filter of SVGF (Schied et al., HPG 2017) without its temporal part, on one image (the region):

* prepare: demodulate i = c / max(a, 1e-3); luminance variance of the pixel mean (sum_c w_c sd_c)^2 / n over
  max(lum(a), 1e-3)^2 with sd_c = sqrt(M2_c / (n - 1)), +inf (unknown: luminance weights 1) when n < 2; depth gradient by
  central differences, one-sided at the image border and next to misses.  A pixel whose colour, albedo, normal, depth or
  demodulated colour is not finite is passed through unchanged and is no neighbour's tap.  The demodulated colour is
  the FP32 quotient the filter stores: a finite colour over a small albedo (3e38 / 1e-3) overflows there, although it
  is finite in float64.
* K a-trous passes, step 2^k, taps h = (1,4,6,4,1)/16 x itself, weight h * w_n * w_z * w_l:
    w_n = max(0, n_p.n_q)^sigma_n for two hits, 1 for two misses, 0 for a hit and a miss;
    w_z = exp(-|z_p - z_q| / (sigma_z |grad z_p . (q - p)| + 1e-3 z_p + 1e-10)) for two hits, else 1;
    w_l = exp(-|l_p - l_q| / (sigma_l sqrt(max(g3x3(var)_p, var_q)) + 1e-10)), g3x3 = (1/4, 1/2, 1/4) blur over the taps
    the filter reads (the larger variance: bright Monte-Carlo pixels are the noisy ones, and a stop scaled by the
    centre's variance alone moves energy out of them and not back).
  colour = sum w i / sum w, variance = sum w^2 var / (sum w)^2.
* finish: remodulate by max(a, 1e-3).
"""
from __future__ import annotations

import numpy as np

LUM = np.array([0.299, 0.587, 0.114])
ALBEDO_MIN = 1e-3
DEFAULTS = {"iterations": 5, "sigmaLuminance": 4.0, "sigmaNormal": 128.0, "sigmaDepth": 1.0}
H5 = np.array([1, 4, 6, 4, 1], np.float64) / 16
K3 = np.array([0.25, 0.5, 0.25])


def options(opts=None):
    o = dict(DEFAULTS)
    for k, v in (opts or {}).items():
        if k == "iterations" or v:  # a sigma of 0 selects its default, as in rt_denoise_opts
            o[k] = v
    return o


def _shift(a, dx, dy, fill):
    """out[y, x] = a[y + dy, x + dx] where inside the image, else `fill`."""
    H, W = a.shape[:2]
    out = np.full_like(a, fill)
    if abs(dx) >= W or abs(dy) >= H:
        return out
    ys, yd = slice(max(dy, 0), H + min(dy, 0)), slice(max(-dy, 0), H + min(-dy, 0))
    xs, xd = slice(max(dx, 0), W + min(dx, 0)), slice(max(-dx, 0), W + min(-dx, 0))
    out[yd, xd] = a[ys, xs]
    return out


def _inside(H, W, dx, dy):
    return _shift(np.ones((H, W), bool), dx, dy, False)


def prepare(color, albedo, normal, depth, moments):
    c, a, n, z, m = (np.asarray(x, np.float64) for x in (color, albedo, normal, depth, moments))
    ac = np.maximum(a, ALBEDO_MIN)
    with np.errstate(all="ignore"):
        i = c / ac
        ns = m[..., 6]
        m2 = np.where(m[..., 3:6] > 0, m[..., 3:6], 0.0)
        sd = (np.sqrt(m2 / (ns - 1)[..., None]) * LUM).sum(-1)
        la = np.maximum(a @ LUM, ALBEDO_MIN)
        var = np.where(ns >= 2, sd * sd / ns / (la * la), np.inf)
        i32 = np.asarray(color, np.float32) / np.maximum(np.asarray(albedo, np.float32), np.float32(ALBEDO_MIN))
    fin = lambda x: np.isfinite(x).all(-1)  # noqa: E731
    valid = fin(c) & fin(a) & fin(n) & np.isfinite(z) & fin(i32)
    hit = valid & (z >= 0)
    usable = np.isfinite(z) & (z >= 0)
    H, W = z.shape
    grad = np.zeros((H, W, 2))
    for ax, (dx, dy) in enumerate(((1, 0), (0, 1))):
        zl, zh = _shift(z, -dx, -dy, np.nan), _shift(z, dx, dy, np.nan)
        ul, uh = _shift(usable, -dx, -dy, False), _shift(usable, dx, dy, False)
        g = np.where(ul & uh, 0.5 * (zh - zl), np.where(uh, zh - z, np.where(ul, z - zl, 0.0)))
        grad[..., ax] = np.where(hit, g, 0.0)
    return {"i": np.where(valid[..., None], i, np.nan), "var": np.where(valid, var, np.nan), "valid": valid,
            "n": n, "z": z, "grad": grad, "ac": ac, "color": c}


def atrous_pass(P, i, var, step, o):
    valid, n, z, grad = P["valid"], P["n"], P["z"], P["grad"]
    H, W = z.shape
    # 3x3 variance blur over the valid in-image taps
    gv = np.zeros((H, W))
    gw = np.zeros((H, W))
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            ok = _shift(valid, dx, dy, False)
            w = K3[dx + 1] * K3[dy + 1]
            gv += np.where(ok, w * _shift(np.nan_to_num(var, nan=0.0, posinf=0.0), dx, dy, 0.0), 0.0)
            gv = np.where(ok & np.isposinf(_shift(var, dx, dy, 0.0)), np.inf, gv)
            gw += np.where(ok, w, 0.0)
    with np.errstate(all="ignore"):
        gv = gv / gw
        lum = i @ LUM
        miss = z < 0
        z_eps = 1e-3 * z + 1e-10
        sw = np.zeros((H, W))
        si = np.zeros((H, W, 3))
        sv = np.zeros((H, W))
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                sx, sy = dx * step, dy * step
                ok = valid & _shift(valid, sx, sy, False)
                iq, vq, nq, zq = (_shift(x, sx, sy, np.nan) for x in (i, var, n, z))
                miss_q = zq < 0
                ok &= miss == miss_q
                wn = np.maximum((n * nq).sum(-1), 0.0) ** o["sigmaNormal"]
                dz = o["sigmaDepth"] * np.abs(grad[..., 0] * sx + grad[..., 1] * sy)
                wz = np.exp(-np.abs(z - zq) / (dz + z_eps))
                w = H5[dx + 2] * H5[dy + 2] * np.where(miss, 1.0, wn * wz)
                w = w * np.exp(-np.abs(lum - iq @ LUM) / (o["sigmaLuminance"] * np.sqrt(np.maximum(gv, vq)) + 1e-10))
                ok &= w > 0
                w = np.where(ok, w, 0.0)
                sw += w
                si += w[..., None] * np.where(ok[..., None], iq, 0.0)
                sv += np.where(ok, w * w * vq, 0.0)
        i2 = si / sw[..., None]
        v2 = sv / (sw * sw)
    return np.where(valid[..., None], i2, i), np.where(valid, v2, var)


def denoise(color, albedo, normal, depth, moments, opts=None):
    """The filtered colour [H,W,3] (float64) of one image."""
    o = options(opts)
    P = prepare(color, albedo, normal, depth, moments)
    i, var = P["i"], P["var"]
    for k in range(int(o["iterations"])):
        i, var = atrous_pass(P, i, var, 1 << k, o)
    return np.where(P["valid"][..., None], i * P["ac"], P["color"])


def gamma_rgb8(linear):
    """writeColorToBuffer (the rule of write_pixel): sqrt gamma, floor(255.999 c), Uint8Clamped (NaN/negative -> 0)."""
    with np.errstate(invalid="ignore"):
        v = np.floor(255.999 * np.sqrt(np.asarray(linear, np.float32).astype(np.float64)))
    return np.where(v > 0, np.minimum(v, 255), 0).astype(np.uint8)
