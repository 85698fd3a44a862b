"""Timbre morphs without a GPU: the float64 rows of tests/morph_oracle.py against the reference's golden interpolation rows and the
properties slerp must have, the ascending inversion coefficient table, and the argument checks of ds_morph_rows_workspace /
ds_morph_rows and of TextToTimbre.morph / invert, which all run before any device work."""
import ctypes as C

import numpy as np
import pytest
import torch

from diffusynth_b200 import _lib, codec
from oracle import cases, ds_oracle as O
from tests import morph_oracle as M


def test_linear_rows_reproduce_the_reference_golden(golden):
    """sampler2.npz["interp_init"]: generate_linear_noise((3, 4, 16, 64), first_endpoint=e0, second_endpoint=e1) of the reference."""
    e0, e1 = cases.randn((4, 16, 64), 93), cases.randn((4, 16, 64), 94)
    rows = M.linear_rows(e0.numpy()[None], e1.numpy()[None], 3)
    g = golden["sampler2"]["interp_init"].astype(np.float64)
    assert np.linalg.norm(rows - g) / np.linalg.norm(g) <= 1e-6


@pytest.mark.parametrize("frames", [2, 3, 5, 33])
def test_slerp_frames_0_and_last_are_the_endpoints(frames):
    e0, e1 = cases.randn((3, 4, 16, 64), 1).numpy(), cases.randn((3, 4, 16, 64), 2).numpy()
    rows = M.slerp_rows(e0, e1, frames).reshape((3, frames) + e0.shape[1:])
    assert np.array_equal(rows[:, 0], e0.astype(np.float64)) and np.array_equal(rows[:, -1], e1.astype(np.float64))


def test_slerp_preserves_the_norm_of_orthogonal_equal_norm_endpoints():
    x = cases.randn((4 * 128 * 64,), 3).double().numpy()
    y = cases.randn((4 * 128 * 64,), 4).double().numpy()
    y -= (x @ y) / (x @ x) * x                      # Gram-Schmidt: <x, y> = 0
    y *= np.linalg.norm(x) / np.linalg.norm(y)
    rows = M.slerp_rows(x[None], y[None], 9)
    norms = np.linalg.norm(rows, axis=1)
    assert np.abs(norms / np.linalg.norm(x) - 1.0).max() < 1e-12
    lin = M.linear_rows(x[None], y[None], 9)        # the reference's linear midpoint shrinks to sqrt(0.5) of the norm
    assert abs(np.linalg.norm(lin[4]) / np.linalg.norm(x) - np.sqrt(0.5)) < 1e-12


def test_identical_antipodal_and_zero_endpoints_take_the_linear_rows():
    x = cases.randn((2, 4, 16, 64), 5).numpy()
    for e1 in (x, -x, x * 0.0, x * (1.0 + 1e-15)):
        rows = M.slerp_rows(x, e1, 5)
        assert np.isfinite(rows).all()
        assert np.array_equal(rows, M.linear_rows(x, e1, 5))
    mid = M.slerp_rows(x, -x, 3).reshape((2, 3) + x.shape[1:])[:, 1]
    assert np.abs(mid).max() == 0.0                 # antipodal: the linear midpoint is zero, not NaN


def test_inversion_coefficients_ascend_and_end_at_pure_noise():
    sch = O.Schedule(1000)
    sch.respace(list(np.linspace(0, 999, 20, dtype=np.int32)))
    co = M.invert_coefficients(sch, 3.0)
    assert co.shape == (20, 8)
    assert np.all(np.diff(co[:, 1]) < 0)            # sqrt(a_t) falls along the ascending steps
    assert np.array_equal(co[:-1, 2], co[1:, 1])     # step t lands where step t+1 reads: sqrt(a_next[t]) = sqrt(a[t+1])
    assert co[-1, 2] == 0.0 and co[-1, 3] == 1.0     # a_next = 0 after the last step: the result is the noise prediction
    assert np.all(co[:, 4] == 0.0) and np.all(co[:, 5] == 3.0)
    np.testing.assert_array_equal(co[:, 0], np.float32(np.sqrt(np.float32(1.0 - sch.alphas_cumprod.astype(np.float32)))))


def test_oracle_inversion_of_a_linear_model_reaches_its_noise():
    """The last step has a_next = 0, so it returns the model's eps of its input: the input itself for the identity model."""
    sch = O.Schedule(1000)
    sch.respace(list(np.linspace(0, 999, 5, dtype=np.int32)))
    x0 = cases.randn((2, 4, 8, 8), 6)
    imgs = M.ddim_invert(lambda x, t, c: x, sch, x0, torch.zeros(2, 3), None, 1.0)
    assert len(imgs) == 6 and torch.equal(imgs[-1], imgs[-2])     # a_next = 0: x_next = eps(x) = x


def test_morph_rows_argument_errors_without_gpu():
    lib = _lib.load()
    nbytes = C.c_longlong(-1)
    n, L = 4 * 128 * 64, 512
    assert lib.ds_morph_rows_workspace(3, 5, n, L, 1, C.byref(nbytes)) == 0
    need = nbytes.value
    assert need >= 3 * 3 * 8                                           # float64 (dot, |e0|^2, |e1|^2) per sequence at least
    assert lib.ds_morph_rows_workspace(3, 5, n, L, 0, C.byref(nbytes)) == 0 and nbytes.value == 0
    P16 = C.c_void_p(16)
    bad = [(0, 5, n, L, 1), (-1, 5, n, L, 1), (3, 1, n, L, 1), (3, 0, n, L, 0), (3, 5, 0, L, 1), (3, 5, -4, L, 1), (3, 5, n + 2, L, 1),
           (3, 5, n, 0, 1), (3, 5, n, -1, 0), (3, 5, n, L, 2), (3, 5, n, L, -1),
           (1 << 20, 1 << 10, 1 << 36, L, 0)]                             # P * N * n overflows int64
    for P, N, nn, LL, path in bad:
        assert lib.ds_morph_rows_workspace(P, N, nn, LL, path, C.byref(nbytes)) == -1, (P, N, nn, LL, path)
        assert b"ds_morph_rows_workspace" in lib.ds_last_error()
        assert lib.ds_morph_rows(P16, P16, P16, P16, P, N, nn, LL, path, P16, P16, P16, 1 << 40, None) == -1
        assert b"ds_morph_rows" in lib.ds_last_error()
    assert lib.ds_morph_rows_workspace(3, 5, n, L, 1, None) == -1
    for k in range(6):                                                 # each of e0, e1, c0, c1, noise, cond null
        ptrs = [P16] * 6
        ptrs[k] = None
        assert lib.ds_morph_rows(*ptrs[:4], 3, 5, n, L, 1, *ptrs[4:], P16, need, None) == -1
    assert lib.ds_morph_rows(P16, P16, P16, P16, 3, 5, n, L, 1, P16, P16, None, need, None) == -1
    assert lib.ds_morph_rows(P16, P16, P16, P16, 3, 5, n, L, 1, P16, P16, P16, need - 1, None) == -1
    assert b"workspace" in lib.ds_last_error()


def test_python_surface_rejects_bad_arguments_before_the_device():
    from diffusynth_b200.pipeline import TextToTimbre
    pipe = TextToTimbre(None, None, device="cpu")                     # no networks: every check below runs before they are used
    e, c = torch.zeros(2, 4, 128, 64), torch.zeros(2, 512)
    ok = dict(first_noise=e, second_noise=e, first_cond=c, second_cond=c, uncond=None, frames=3)
    for change in (dict(frames=1), dict(frames=0), dict(frames=2.5), dict(frames=True), dict(path="cosine"),
                   dict(first_noise=torch.zeros(2, 4, 128, 32)),       # not the train width
                   dict(second_noise=torch.zeros(3, 4, 128, 64)),      # P mismatch between noises
                   dict(first_cond=torch.zeros(3, 512)),               # P mismatch between noise and condition
                   dict(second_cond=torch.zeros(2, 256)),              # L mismatch
                   dict(first_cond=torch.zeros(2, 512, dtype=torch.long)),
                   dict(first_noise=torch.zeros(4, 128)), dict(first_cond=torch.zeros(2, 2, 512))):
        with pytest.raises(ValueError):
            pipe.morph(**dict(ok, **change))
    pipe.noise_strategy = "non_repeat"
    with pytest.raises(ValueError):
        pipe.morph(**ok)
    pipe.noise_strategy = "repeat"
    with pytest.raises(ValueError):
        pipe.invert(torch.zeros(2, 4, 128, 32), c)
    with pytest.raises(ValueError):
        pipe.invert(e, torch.zeros(3, 512))
    with pytest.raises(ValueError):
        codec.morph_rows(e, e, c, c, 3, path="spherical")
