"""CPU oracle of the mask zoom (TEST INFRASTRUCTURE ONLY): a float64 numpy restatement of
``scipy.ndimage.zoom(a, (h / H, w / W))`` with scipy's defaults (order=3, mode='constant', prefilter=True, grid_mode=False) for
2-D arrays, as the inpainting-with-text handler shrinks its spectrogram mask to the latent grid (inpaint_with_text.py).

The operation is separable and linear, so it is applied along one axis at a time (the axes commute):
- ``prefilter_line``: the cubic B-spline prefilter, pole z = sqrt(3) - 2, mirror boundary (x[-k] = x[k], x[n-1+k] = x[n-1-k]),
  with scipy's exact causal and anticausal initialisations; a line of length 1 is left unchanged;
- ``interpolate_line``: output o samples the input coordinate x = o * ((n - 1) / (out - 1)) (0 when out = 1) as the sum of the
  coefficients floor(x) - 1 .. floor(x) + 2, mirrored with period 2n - 2, weighted by the cubic B-spline.
``prefilter_axis`` exposes the coefficients of one axis.  Pinned against scipy itself in tests/test_zoom_oracle.py."""
from __future__ import annotations

import numpy as np

POLE = np.sqrt(3.0) - 2.0
GAIN = (1.0 - POLE) * (1.0 - 1.0 / POLE)

__all__ = ["POLE", "GAIN", "zoom_shape", "prefilter_line", "prefilter_axis", "mirror", "bspline3_weights", "interpolate_line", "zoom"]


def zoom_shape(shape, out_shape=None, factors=None):
    """scipy's output shape: round(n * factor) per axis (Python's round), or ``out_shape`` as given."""
    if out_shape is not None:
        return tuple(int(v) for v in out_shape)
    return tuple(int(round(n * f)) for n, f in zip(shape, factors))


def prefilter_line(x: np.ndarray) -> np.ndarray:
    """Cubic B-spline coefficients of one line, in scipy's order of operations (gain, causal init and recursion, anticausal init
    and recursion)."""
    c = np.asarray(x, dtype=np.float64) * GAIN
    n = len(c)
    if n == 1:
        return np.asarray(x, dtype=np.float64).copy()
    z = POLE
    zn1 = z ** (n - 1)
    c0 = c[0] + zn1 * c[n - 1]
    zi = z
    for i in range(1, n - 1):
        c0 += zi * (c[i] + zn1 * c[n - 1 - i])
        zi *= z
    c[0] = c0 / (1.0 - zn1 * zn1)
    for i in range(1, n):
        c[i] += z * c[i - 1]
    c[n - 1] = z / (z * z - 1.0) * (z * c[n - 2] + c[n - 1])
    for i in range(n - 2, -1, -1):
        c[i] = z * (c[i + 1] - c[i])
    return c


def prefilter_axis(a: np.ndarray, axis: int) -> np.ndarray:
    """The prefilter along one axis of a 2-D array (every line along ``axis``)."""
    return np.apply_along_axis(prefilter_line, axis, np.asarray(a, dtype=np.float64))


def mirror(k: int, n: int) -> int:
    """Index k of a line of n coefficients, mirrored at both ends with period 2n - 2."""
    if n == 1:
        return 0
    p = 2 * n - 2
    k = abs(k) % p
    return p - k if k >= n else k


def bspline3_weights(t: float):
    """Cubic B-spline weights of the coefficients floor(x) - 1 .. floor(x) + 2 at t = x - floor(x)."""
    u = 1.0 - t
    return (u * u * u / 6.0, (3.0 * t * t * (t - 2.0) + 4.0) / 6.0, (3.0 * u * u * (u - 2.0) + 4.0) / 6.0, t * t * t / 6.0)


def interpolate_line(c: np.ndarray, out: int) -> np.ndarray:
    """``out`` samples of the spline with coefficients c, at x = o * ((n - 1) / (out - 1))."""
    n = len(c)
    step = (n - 1) / (out - 1) if out > 1 else 0.0
    res = np.empty(out)
    for o in range(out):
        x = o * step
        f = int(np.floor(x))
        w = bspline3_weights(x - f)
        res[o] = sum(wj * c[mirror(f - 1 + j, n)] for j, wj in enumerate(w))
    return res


def zoom(a: np.ndarray, out_shape) -> np.ndarray:
    """float64 zoom of a 2-D array to ``out_shape`` (h, w): prefilter and interpolate along axis 0, then along axis 1."""
    a = np.asarray(a, dtype=np.float64)
    assert a.ndim == 2
    h, w = (int(v) for v in out_shape)
    cols = prefilter_axis(a, 0)
    mid = np.stack([interpolate_line(cols[:, j], h) for j in range(a.shape[1])], axis=1)          # [h, W]
    rows = prefilter_axis(mid, 1)
    return np.stack([interpolate_line(rows[i], w) for i in range(h)], axis=0)                     # [h, w]
