"""tests/attn_oracle.py (float64 linear attention at the level of the chunk partials) against oracle/ds_oracle.py, and proof that the
per-chunk gates used by tests/test_gpu_attention.py are tight: each of a set of plausible kernel mistakes, applied to the float64
reference, moves its metric by at least 10x the gate."""
import numpy as np
import pytest
import torch

from oracle import ds_oracle as O
from tests import attn_oracle as A

HID = 128


def _sd_attn(C, L, seed, cat):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    p = "a."
    sd = {p + "fn.norm.weight": 1 + 0.2 * r(C), p + "fn.norm.bias": 0.2 * r(C),
          p + "fn.fn.to_qkv.weight": r(3 * HID, C, 1, 1) * (2 / C ** 0.5),
          p + "fn.fn.label_key.weight": r(HID, L) * 0.3, p + "fn.fn.label_key.bias": r(HID) * 0.3,
          p + "fn.fn.to_out.0.weight": r(C, HID, 1, 1) * 0.1, p + "fn.fn.to_out.0.bias": r(C) * 0.1,
          p + "fn.fn.to_out.1.weight": 1 + 0.1 * r(C), p + "fn.fn.to_out.1.bias": 0.1 * r(C)}
    second = "label_value" if cat else "label_query"
    sd[p + f"fn.fn.{second}.weight"], sd[p + f"fn.fn.{second}.bias"] = r(HID, L) * 0.3, r(HID) * 0.3
    return sd


@pytest.mark.parametrize("cat", [False, True])
@pytest.mark.parametrize("H,W", [(24, 22), (1, 5), (32, 33)])
def test_unet_attention_matches_ds_oracle(cat, H, W):
    C, L, N = 96, 16, 2
    sd = _sd_attn(C, L, 3 + cat, cat)
    x = torch.randn(N, C, H, W, generator=torch.Generator().manual_seed(9), dtype=torch.float64) * 1.7 + 0.3
    cemb = torch.randn(N, L, generator=torch.Generator().manual_seed(10), dtype=torch.float64)
    with torch.no_grad():
        ref = (O.linear_attention_cat if cat else O.linear_attention_add)(sd, "a.", x, cemb).numpy().reshape(N, C, H * W)
    got = (A.linear_cat_block if cat else A.linear_add_block)(sd, "a.", x.numpy().reshape(N, C, H * W), cemb.numpy())
    assert np.abs(got - ref).max() / np.abs(ref).max() < 1e-12


@pytest.mark.parametrize("skip", [False, True])
def test_vq_attention_matches_ds_oracle(skip):
    C, N, H, W = 80, 2, 16, 40
    g = torch.Generator().manual_seed(5)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    sd = {"v.to_qkv.weight": r(96, C, 1, 1) * 0.3, "v.to_out.weight": r(C, 32, 1, 1) * 0.2, "v.to_out.bias": r(C) * 0.1}
    if skip:
        sd["v.nin_shortcut.weight"], sd["v.nin_shortcut.bias"] = r(C, C, 1, 1) * 0.1, r(C) * 0.1
    x = r(N, C, H, W)
    with torch.no_grad():
        ref = O.vq_linear_attention(sd, "v.", x).numpy().reshape(N, C, H * W)
    got = A.vq_attention_block(sd, "v.", x.numpy().reshape(N, C, H * W))
    assert np.abs(got - ref).max() / np.abs(ref).max() < 1e-12


@pytest.mark.parametrize("npix", [1, 129, 513, 2600])
@pytest.mark.parametrize("label", [None, -80.0, 0.0, 80.0])
def test_chunk_quantities_merge_to_ctx(npix, label):
    rng = np.random.default_rng(npix)
    N, H = 2, 2
    k = rng.standard_normal((N, H, 32, npix)) * 20
    v = rng.standard_normal((N, H, 32, npix)) + 0.5
    lk = lv = None
    if label is not None:
        lk = rng.standard_normal((N, H, 32)) + label + k.max()
        lv = rng.standard_normal((N, H, 32))
    lse, avg, _ = A.chunk_quantities(k, v)
    assert lse.shape[2] == A.chunks_of(npix)
    ref = A.context(k, v, lk, lv)
    assert np.abs(A.merge(lse, avg, lk, lv) - ref).max() <= 1e-12 * np.abs(ref).max()


# ------------------------------------------------------------------ the gates are tight
# the two producers' gate parameters, as tests/test_gpu_attention.py uses them
FUSED = dict(u_p=A.U_BF16, u_v=A.U_BF16, p_flush=2.0 ** -26)
SEPARATE = dict(u_p=A.U_FP16, u_v=0.0, p_floor=2.0 ** -25)


def _ratio(got, ref, gate):
    r = np.linalg.norm(np.atleast_1d(got - ref).reshape(gate.shape + (-1,)), axis=-1) / gate
    return np.where(np.isfinite(r), r, np.inf).max()


def _case(npix, seed=0, kscale=1.5):
    rng = np.random.default_rng(seed)
    k = rng.standard_normal((1, 2, 32, npix)) * kscale
    v = rng.standard_normal((1, 2, 32, npix)) + 0.3
    return k, v


@pytest.mark.parametrize("prod", [FUSED, SEPARATE], ids=["fused", "separate"])
def test_gate_catches_dropped_last_pixel(prod):
    """A ragged chunk (npix = 517: 5 valid pixels in chunk 1) that loses its last valid pixel."""
    k, v = _case(517)
    lse, avg, _ = A.chunk_quantities(k, v)
    g_lse, g_avg = A.chunk_gates(k, v, **prod)
    lse2, avg2, _ = A.chunk_quantities(k[..., :-1], v[..., :-1])
    r = max(_ratio(lse2[:, :, 1], lse[:, :, 1], g_lse[:, :, 1]), _ratio(avg2[:, :, 1], avg[:, :, 1], g_avg[:, :, 1]))
    assert r >= 10, r


@pytest.mark.parametrize("prod", [FUSED, SEPARATE], ids=["fused", "separate"])
@pytest.mark.parametrize("npix", [517, 514])
def test_gate_catches_invalid_pixel(prod, npix):
    """One pixel past the end of the sample included with k = 0 (v = 0), as a mask off by one would."""
    k, v = _case(npix, 1)
    lse, avg, _ = A.chunk_quantities(k, v)
    g_lse, g_avg = A.chunk_gates(k, v, **prod)
    k2, v2 = np.concatenate([k, np.zeros(k.shape[:3] + (1,))], -1), np.concatenate([v, np.zeros(v.shape[:3] + (1,))], -1)
    lse2, avg2, _ = A.chunk_quantities(k2, v2)
    c = A.chunks_of(npix) - 1
    r = max(_ratio(lse2[:, :, c], lse[:, :, c], g_lse[:, :, c]), _ratio(avg2[:, :, c], avg[:, :, c], g_avg[:, :, c]))
    assert r >= 10, r


@pytest.mark.parametrize("prod", [FUSED, SEPARATE], ids=["fused", "separate"])
def test_gate_catches_swapped_heads(prod):
    """Heads 1 and 2 exchanged in q', in the partials and in M."""
    rng = np.random.default_rng(3)
    N, C, npix = 2, 96, 700
    q, k, v = (rng.standard_normal((N, 4, 32, npix)) * s for s in (1.5, 1.5, 1.0))
    wout = rng.standard_normal((C, HID)) * 0.1
    qp = A.q_prime(q)
    lse, avg, vsq = A.chunk_quantities(k, v)
    g_lse, g_avg = A.chunk_gates(k, v, **prod)
    M = A.fold(A.merge(lse, avg), wout)
    g_M = A.m_gate(A.ctx_gate(lse, avg, vsq, g_lse, g_avg), wout, M, A.U_FP16)
    g_q = A.q_gate(qp, A.U_FP16)
    sw = [0, 2, 1, 3]
    assert _ratio(qp[:, sw], qp, g_q) >= 10
    assert _ratio(avg[:, sw], avg, g_avg) >= 10 and _ratio(lse[:, sw], lse, g_lse) >= 10
    Msw = A.fold(A.merge(lse[:, sw], avg[:, sw]), wout)
    assert _ratio(Msw.reshape(N, C, 4, 32).transpose(0, 2, 1, 3), M.reshape(N, C, 4, 32).transpose(0, 2, 1, 3), g_M) >= 10


def test_gate_catches_per_head_ftz_stabiliser():
    """A per-head stabiliser without the per-row fallback (the fused kernel's former rule): P = exp2(rl2 acc - mh) with ONE mh per
    head, taken from the bare product rl2 acc of the item's first 128-pixel tile (the per-row constant tk[d] reported through m),
    and ex2.approx.ftz flushing below 2^-126.
    At mu / sigma = 50 of the block input whole rows of a head lose every pixel: Z = 0, log Z + m = -inf."""
    rng = np.random.default_rng(0)
    C, mu = 96, 50.0
    x = (mu + rng.standard_normal((1, C, A.CHUNK))).astype(np.float16).astype(np.float64)
    w = (rng.standard_normal((3 * HID, C)) * (2 / C ** 0.5)).astype(np.float16).astype(np.float64)
    mean, rstd = A.group_norm_stats(x)
    q, k, v = A.split_heads(A.qkv_logits(x, w, mean=mean, rstd=rstd), 4)
    lse, avg, _ = A.chunk_quantities(k, v)
    g_lse, g_avg = A.chunk_gates(k, v, **FUSED)
    bare = np.log2(np.e) * rstd[0] * np.einsum("oc,cn->on", w[HID:2 * HID], x[0]).reshape(4, 32, -1)     # rl2 acc
    tk = (k[0] * np.log2(np.e) - bare)[..., 0]                                                            # per-row constant
    mh = bare[..., :A.TILE].max(axis=(1, 2), keepdims=True)
    e = bare - mh
    p = np.where(e < -126, 0.0, np.exp2(e))
    with np.errstate(divide="ignore", invalid="ignore"):
        Z = p.sum(-1)
        lse_bad = (np.log(Z) + (mh[..., 0] + tk) * np.log(2))[None, :, None]
        avg_bad = (np.einsum("hdn,hen->hde", p, v[0]) / Z[..., None])[None, :, None]
    assert (Z == 0).sum() > 0
    assert _ratio(lse_bad, lse, g_lse) >= 10 and _ratio(avg_bad, avg, g_avg) >= 10


def test_gates_cover_fp_reordering():
    """The gates are not too tight either: the same quantities from float32 inputs (a reordering-level change) pass them."""
    k, v = _case(1100, 4, 20.0)
    lse, avg, _ = A.chunk_quantities(k, v)
    g_lse, g_avg = A.chunk_gates(k, v, **SEPARATE)
    lse2, avg2, _ = A.chunk_quantities(k.astype(np.float32).astype(np.float64), v.astype(np.float32).astype(np.float64))
    assert _ratio(lse2, lse, g_lse) < 1 and _ratio(avg2, avg, g_avg) < 1
