"""Mask zoom without a GPU: the float64 restatement of scipy.ndimage.zoom (order 3, mode 'constant', prefilter, grid_mode False)
in tests/zoom_oracle.py pinned against scipy itself, and the argument checks of codec.zoom / ds_mask_zoom_workspace /
ds_mask_zoom, which run before any device work."""
import ctypes as C
import os

import numpy as np
import pytest
import scipy.ndimage as nd
import torch

from diffusynth_b200 import _lib, codec
from tests import zoom_oracle as Z

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (in shape, out shape): the latent grids of the spectrogram image (513 x T) and of the encoder's input (512 x 4w), odd and tiny
# grids, up- and down-sampling, the identity, and out = 1 / in = 1 on either axis
SIZES = [((513, 257), (128, 64)), ((512, 256), (128, 64)), ((37, 11), (128, 30)), ((3, 2), (7, 5)), ((1, 9), (4, 4)),
         ((128, 64), (128, 64)), ((513, 1025), (128, 1)), ((9, 1), (4, 3)), ((5, 7), (1, 1)), ((6, 40), (1, 13)), ((2, 2), (9, 1)),
         ((64, 16), (128, 64)), ((100, 3), (17, 250))]


def _scipy(a, out_shape):
    H, W = a.shape
    h, w = out_shape
    ref = nd.zoom(a, (h / H, w / W))
    assert ref.shape == (h, w)
    return ref


@pytest.mark.parametrize("shape_in,shape_out", SIZES)
def test_oracle_matches_scipy(shape_in, shape_out):
    rng = np.random.default_rng(shape_in[0] * 1000 + shape_in[1])
    soft = rng.random(shape_in)                                           # soft mask in [0, 1)
    binary = (rng.random(shape_in) > 0.5).astype(np.float64)             # binary mask
    rect = np.zeros(shape_in)
    rect[shape_in[0] // 3: 2 * shape_in[0] // 3 + 1, shape_in[1] // 4:] = 1.0
    for a in (soft, binary, rect):
        err = np.abs(Z.zoom(a, shape_out) - _scipy(a, shape_out)).max()
        assert err <= 1e-12, (shape_in, shape_out, err)


def test_binary_mask_overshoots_as_scipy_does():
    """An order-3 zoom of a binary mask rings: the values the blend receives lie outside [0, 1]."""
    b = (np.random.default_rng(0).random((513, 257)) > 0.5).astype(np.float32)
    got = Z.zoom(b, (128, 64))
    ref = _scipy(b, (128, 64))
    assert ref.dtype == np.float32 and np.abs(got - ref).max() <= 1e-6
    assert got.min() < -0.4 and got.max() > 1.45


def test_prefiltered_coefficients_per_axis():
    """The coefficients of each axis are scipy's spline_filter1d (mode 'mirror'), and the spline through them passes through the
    samples (interpolation at x = o reproduces the input)."""
    a = np.random.default_rng(3).random((37, 11))
    for axis in (0, 1):
        c = Z.prefilter_axis(a, axis)
        assert np.abs(c - nd.spline_filter1d(a, order=3, axis=axis, mode="mirror")).max() <= 1e-12
    for line in (a[:, 4], a[7], a[:1, 0], a[:2, 0]):
        c = Z.prefilter_line(line)
        assert np.abs(Z.interpolate_line(c, len(line)) - line).max() <= 1e-12
    assert Z.prefilter_line(np.array([0.3]))[0] == 0.3                   # a line of length 1 is unchanged


def test_mirror_and_weights():
    assert [Z.mirror(k, 4) for k in range(-3, 8)] == [3, 2, 1, 0, 1, 2, 3, 2, 1, 0, 1]
    assert [Z.mirror(k, 1) for k in (-1, 0, 1, 2)] == [0, 0, 0, 0]
    for t in (0.0, 0.25, 0.5, 0.999):
        assert abs(sum(Z.bspline3_weights(t)) - 1.0) <= 1e-15
    assert Z.zoom_shape((513, 257), factors=(128 / 513, 64 / 257)) == (128, 64)


def _arr(vals):
    return (C.c_longlong * len(vals))(*vals)


def test_mask_zoom_argument_errors_without_gpu():
    lib = _lib.load()
    nbytes = C.c_longlong(0)
    ins, outs = _arr([513, 257, 3, 2]), _arr([128, 64, 7, 5])
    assert lib.ds_mask_zoom_workspace(ins, outs, 2, C.byref(nbytes)) == 0
    need = nbytes.value
    assert need >= 8 * (513 * 257 + 3 * 2 + 128 * 257 + 7 * 2)        # float64 coefficients and intermediate
    cap = 16384                                                          # DS_MASK_ZOOM_MAX_DIM
    bad = (([513, 0, 3, 2], [128, 64, 7, 5]),                             # a non-positive dimension, in or out
           ([513, 257, -3, 2], [128, 64, 7, 5]),
           ([513, 257, 3, 2], [128, 0, 7, 5]),
           ([513, 257, 3, 2], [128, 64, 7, -5]),
           ([cap + 1, 257, 3, 2], [128, 64, 7, 5]),                      # a dimension above DS_MASK_ZOOM_MAX_DIM
           ([513, 257, 3, 2], [128, 64, 7, cap + 1]),
           ([513, 257, 3, 1 << 40], [128, 64, 7, 5]))
    for i, o in bad:
        assert lib.ds_mask_zoom_workspace(_arr(i), _arr(o), 2, C.byref(nbytes)) == -1
        assert b"ds_mask_zoom_workspace" in lib.ds_last_error()
        assert lib.ds_mask_zoom(C.c_void_p(16), C.c_void_p(16), _arr(i), _arr(o), 2, C.c_void_p(16), 1 << 40, None) == -1
        assert b"ds_mask_zoom" in lib.ds_last_error()
    assert lib.ds_mask_zoom_workspace(_arr([cap, cap]), _arr([cap, cap]), 1, C.byref(nbytes)) == 0     # the cap itself is accepted
    assert lib.ds_mask_zoom_workspace(None, outs, 2, C.byref(nbytes)) == -1
    assert lib.ds_mask_zoom_workspace(ins, None, 2, C.byref(nbytes)) == -1
    assert lib.ds_mask_zoom_workspace(ins, outs, 2, None) == -1
    assert lib.ds_mask_zoom_workspace(ins, outs, 0, C.byref(nbytes)) == -1
    assert lib.ds_mask_zoom_workspace(ins, outs, -1, C.byref(nbytes)) == -1
    assert lib.ds_mask_zoom(None, C.c_void_p(16), ins, outs, 2, C.c_void_p(16), need, None) == -1
    assert lib.ds_mask_zoom(C.c_void_p(16), None, ins, outs, 2, C.c_void_p(16), need, None) == -1
    assert lib.ds_mask_zoom(C.c_void_p(16), C.c_void_p(16), ins, outs, 2, None, need, None) == -1
    assert lib.ds_mask_zoom(C.c_void_p(16), C.c_void_p(16), None, outs, 2, C.c_void_p(16), need, None) == -1
    assert lib.ds_mask_zoom(C.c_void_p(16), C.c_void_p(16), ins, outs, 0, C.c_void_p(16), need, None) == -1
    assert lib.ds_mask_zoom(C.c_void_p(16), C.c_void_p(16), ins, outs, 2, C.c_void_p(16), need - 1, None) == -1
    assert b"workspace" in lib.ds_last_error()


def test_python_surface_rejects_bad_arguments_before_the_device():
    a = np.zeros((16, 8), np.float32)
    for kw in (dict(order=1), dict(mode="nearest"), dict(cval=0.5), dict(prefilter=False), dict(grid_mode=True),
               dict(output=np.float64)):
        with pytest.raises(NotImplementedError):
            codec.zoom(a, 0.5, **kw)
    with pytest.raises(NotImplementedError):
        codec.zoom(a, 0.5, None, 0)                                         # order passed positionally
    for bad in (0.0, -1.0, float("nan"), (0.5, 0.5, 0.5), 1e-3):           # 1e-3: an empty output
        with pytest.raises(ValueError):
            codec.zoom(a, bad)
    with pytest.raises(ValueError):
        codec.zoom(np.zeros(16, np.float32), 0.5)                           # 1-D
    with pytest.raises(ValueError):
        codec.zoom(np.zeros((2, 2, 16, 8), np.float32), 0.5)                # 4-D
    with pytest.raises(ValueError):
        codec.zoom([a, np.zeros(5, np.float32)], 0.5)                       # a list item that is not 2-D
    with pytest.raises(ValueError):
        codec.zoom([], 0.5)
    with pytest.raises(ValueError):
        codec.zoom(np.zeros((0, 16, 8), np.float32), 0.5)
    with pytest.raises(ValueError):
        codec.zoom(a, 2000.0)                                               # above DS_MASK_ZOOM_MAX_DIM
    with pytest.raises(ValueError):
        codec.zoom_packed(torch.zeros(128), [(16, 8)], (0, 4))


def test_product_code_never_imports_the_zoom_oracle():
    pkg = os.path.join(ROOT, "diffusynth_b200")
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            txt = open(os.path.join(pkg, f)).read()
            assert "zoom_oracle" not in txt and "from tests" not in txt and "import tests" not in txt, f
