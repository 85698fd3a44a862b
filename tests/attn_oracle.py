"""Float64 restatement of the linear-attention core (CPU only), at the level of the kernels' chunk partials.

Three variants, all with dim_head = 32:
  linear_add  (LinearCrossAttentionAdd, diffusion_components.py:271-293): PreNorm GroupNorm(1, C), to_qkv, + the per-sample bias
              (label_query | label_key | 0), q' = softmax_d(q) * scale, ctx = softmax_n(k) v^T, M = Wout . ctx
  linear_cat  (LinearCrossAttention, diffusion_components.py:171-207): the same without the bias on q / k; the condition adds one
              extra key / value token (label_key, label_value) to the sequence
  VQGAN       (LinearAttention, VQGAN.py:261-272): no norm, one head, q' = q (neither soft-maxed nor scaled)

Chunk quantities.  attn.cu's partial of (sample, head, 512-pixel chunk c) is S[32][32], Z[32], m[32] with m in natural-log units.
Whatever stabiliser a producer picks, a correct partial satisfies
    log Z_c[d] + m_c[d] = lse_c[d]   = logsumexp over the chunk's valid pixels of k[d]
    S_c[d] / Z_c[d]     = avg_c[d]   = sum_n softmax_chunk(k[d])_n v[:, n]
so both producers are checked per chunk against the same values, and a bad chunk cannot hide in the merge.

Tolerances (``chunk_gates``) come from the producer's operand types; see the docstring there.
"""
from __future__ import annotations

import numpy as np

DH = 32
CHUNK = 512                      # pixels per partial (ds_attn_chunks)
TILE = 128                       # pixels per MMA tile of the fused kernel / sub-chunk of the separate one
U_FP16, U_BF16 = 2.0 ** -11, 2.0 ** -8      # unit roundoff (half an ulp at 1) of IEEE half and bfloat16


def chunks_of(npix: int) -> int:
    return (npix + CHUNK - 1) // CHUNK


def group_norm_stats(x: np.ndarray, eps: float = 1e-5):
    """x [N, C, n] -> (mean [N], rstd [N]) of GroupNorm(1, C), float64."""
    x = np.asarray(x, np.float64)
    mean = x.mean(axis=(1, 2))
    var = ((x - mean[:, None, None]) ** 2).mean(axis=(1, 2))
    return mean, 1.0 / np.sqrt(var + eps)


def qkv_logits(x, w, gamma=None, beta=None, sbias=None, mean=None, rstd=None, norm=True, eps=1e-5):
    """PreNorm + 1x1 to_qkv (no bias) + per-sample bias.  x [N, C, n], w [3*hid, C], sbias [N, 3*hid] or None.
    mean / rstd override the GroupNorm statistics (a kernel that is handed them in fp32 is compared on the same values)."""
    x = np.asarray(x, np.float64)
    w = np.asarray(w, np.float64)
    if norm:
        if mean is None:
            mean, rstd = group_norm_stats(x, eps)
        xn = (x - np.asarray(mean, np.float64)[:, None, None]) * np.asarray(rstd, np.float64)[:, None, None]
        if gamma is not None:
            xn = xn * np.asarray(gamma, np.float64)[None, :, None]
        if beta is not None:
            xn = xn + np.asarray(beta, np.float64)[None, :, None]
    else:
        xn = x
    out = np.einsum("oc,bcn->bon", w, xn)
    if sbias is not None:
        out = out + np.asarray(sbias, np.float64)[:, :, None]
    return out


def split_heads(qkv: np.ndarray, heads: int):
    """[N, 3*hid, n] -> q, k, v each [N, heads, 32, n]."""
    N, _, n = qkv.shape
    q, k, v = np.split(qkv, 3, axis=1)
    return tuple(t.reshape(N, heads, DH, n) for t in (q, k, v))


def logsumexp(a: np.ndarray, axis: int = -1) -> np.ndarray:
    m = np.max(a, axis=axis, keepdims=True)
    m = np.where(np.isfinite(m), m, 0.0)
    return np.squeeze(m, axis) + np.log(np.sum(np.exp(a - m), axis=axis))


def softmax(a: np.ndarray, axis: int) -> np.ndarray:
    e = np.exp(a - a.max(axis=axis, keepdims=True))
    return e / e.sum(axis=axis, keepdims=True)


def q_prime(q: np.ndarray, soft: bool = True, scale: float = DH ** -0.5) -> np.ndarray:
    """softmax over the 32 head channels * scale (U-Net), or q itself (VQGAN).  q [N, H, 32, n]."""
    return softmax(q, axis=2) * scale if soft else q.copy()


def context(k: np.ndarray, v: np.ndarray, label_k=None, label_v=None) -> np.ndarray:
    """ctx[b,h,d,e] = sum_n softmax_n(k)[d,n] v[e,n]; label_k / label_v [N, H, 32] add one extra key / value token."""
    if label_k is not None:
        k = np.concatenate([k, label_k[..., None]], axis=-1)
        v = np.concatenate([v, label_v[..., None]], axis=-1)
    return np.einsum("bhdn,bhen->bhde", softmax(k, axis=-1), v)


def chunk_quantities(k: np.ndarray, v: np.ndarray):
    """Per (sample, head, chunk, row d): lse [N,H,c,32], avg [N,H,c,32,32], and the p-weighted second moment of v
    vsq [N,H,c,32] = sum_n softmax_chunk(k[d])_n |v[:, n]|^2 (the scale the per-row gates are relative to)."""
    N, H, _, n = k.shape
    nc = chunks_of(n)
    lse = np.empty((N, H, nc, DH))
    avg = np.empty((N, H, nc, DH, DH))
    vsq = np.empty((N, H, nc, DH))
    for c in range(nc):
        kc, vc = k[..., c * CHUNK:(c + 1) * CHUNK], v[..., c * CHUNK:(c + 1) * CHUNK]
        lse[:, :, c] = logsumexp(kc, axis=-1)
        w = softmax(kc, axis=-1)
        avg[:, :, c] = np.einsum("bhdn,bhen->bhde", w, vc)
        vsq[:, :, c] = np.einsum("bhdn,bhn->bhd", w, (vc ** 2).sum(axis=2))
    return lse, avg, vsq


def merge(lse: np.ndarray, avg: np.ndarray, label_k=None, label_v=None) -> np.ndarray:
    """ctx from the chunk quantities (what attn_reduce_kernel computes from S, Z, m)."""
    tot = lse if label_k is None else np.concatenate([lse, label_k[:, :, None, :]], axis=2)
    L = logsumexp(tot, axis=2)
    w = np.exp(lse - L[:, :, None, :])
    ctx = np.einsum("bhcd,bhcde->bhde", w, avg)
    if label_k is not None:
        ctx = ctx + np.exp(label_k - L)[..., None] * label_v[:, :, None, :]
    return ctx


def chunk_weights(lse: np.ndarray, label_k=None) -> np.ndarray:
    """omega[b,h,c,d] = share of chunk c in row d's soft-max over the whole sequence (label token included)."""
    tot = lse if label_k is None else np.concatenate([lse, label_k[:, :, None, :]], axis=2)
    return np.exp(lse - logsumexp(tot, axis=2)[:, :, None, :])


def fold(ctx: np.ndarray, wout: np.ndarray) -> np.ndarray:
    """M[b, c, h*32 + d] = sum_e Wout[c, h*32 + e] ctx[b, h, d, e]  (attn_fold_kernel)."""
    N, H = ctx.shape[:2]
    C = wout.shape[0]
    return np.einsum("che,bhde->bchd", np.asarray(wout, np.float64).reshape(C, H, DH), ctx).reshape(N, C, H * DH)


def apply_out(M: np.ndarray, qp: np.ndarray) -> np.ndarray:
    """to_out's 1x1 convolution on ctx^T q' as the per-sample matrix M: out[b, c, n] = sum_(h,d) M[b, c, h*32+d] q'[b, h, d, n]."""
    N, H, _, n = qp.shape
    return np.einsum("bcj,bjn->bcn", M, qp.reshape(N, H * DH, n))


# ---------------------------------------------------------------- end-to-end restatements (pinned to oracle/ds_oracle.py)
def _gn(x, g, b, eps=1e-5):
    mean, rstd = group_norm_stats(x, eps)
    return (x - mean[:, None, None]) * rstd[:, None, None] * g[None, :, None] + b[None, :, None]


def _np(sd, key):
    return sd[key].detach().double().numpy()


def linear_add_block(sd, p: str, x: np.ndarray, cemb: np.ndarray, heads: int = 4) -> np.ndarray:
    """Residual(PreNorm(LinearCrossAttentionAdd)) through the chunked path: x [N, C, n] -> [N, C, n]."""
    w = _np(sd, p + "fn.fn.to_qkv.weight")[:, :, 0, 0]
    hid = heads * DH
    sb = np.zeros((x.shape[0], 3 * hid))
    sb[:, :hid] = cemb @ _np(sd, p + "fn.fn.label_query.weight").T + _np(sd, p + "fn.fn.label_query.bias")
    sb[:, hid:2 * hid] = cemb @ _np(sd, p + "fn.fn.label_key.weight").T + _np(sd, p + "fn.fn.label_key.bias")
    qkv = qkv_logits(x, w, _np(sd, p + "fn.norm.weight"), _np(sd, p + "fn.norm.bias"), sb)
    q, k, v = split_heads(qkv, heads)
    return _finish(sd, p + "fn.fn.", x, q_prime(q), merge(*chunk_quantities(k, v)[:2]), norm=True)


def linear_cat_block(sd, p: str, x: np.ndarray, cemb: np.ndarray, heads: int = 4) -> np.ndarray:
    """Residual(PreNorm(LinearCrossAttention)) ("linear_cat"): the condition is one extra key / value token."""
    w = _np(sd, p + "fn.fn.to_qkv.weight")[:, :, 0, 0]
    N = x.shape[0]
    qkv = qkv_logits(x, w, _np(sd, p + "fn.norm.weight"), _np(sd, p + "fn.norm.bias"))
    q, k, v = split_heads(qkv, heads)
    lk = (cemb @ _np(sd, p + "fn.fn.label_key.weight").T + _np(sd, p + "fn.fn.label_key.bias")).reshape(N, heads, DH)
    lv = (cemb @ _np(sd, p + "fn.fn.label_value.weight").T + _np(sd, p + "fn.fn.label_value.bias")).reshape(N, heads, DH)
    return _finish(sd, p + "fn.fn.", x, q_prime(q), merge(*chunk_quantities(k, v)[:2], lk, lv), norm=True)


def vq_attention_block(sd, p: str, x: np.ndarray) -> np.ndarray:
    """VQGAN LinearAttention (one head, q' = q), with the optional nin_shortcut."""
    w = _np(sd, p + "to_qkv.weight")[:, :, 0, 0]
    q, k, v = split_heads(qkv_logits(x, w, norm=False), 1)
    M = fold(merge(*chunk_quantities(k, v)[:2]), _np(sd, p + "to_out.weight")[:, :, 0, 0])
    out = apply_out(M, q_prime(q, soft=False)) + _np(sd, p + "to_out.bias")[None, :, None]
    if (p + "nin_shortcut.weight") in sd:
        out = out + np.einsum("oc,bcn->bon", _np(sd, p + "nin_shortcut.weight")[:, :, 0, 0], x) + _np(sd, p + "nin_shortcut.bias")[None, :, None]
    return out


def _finish(sd, p, x, qp, ctx, norm):
    M = fold(ctx, _np(sd, p + "to_out.0.weight")[:, :, 0, 0])
    out = apply_out(M, qp) + _np(sd, p + "to_out.0.bias")[None, :, None]
    return _gn(out, _np(sd, p + "to_out.1.weight"), _np(sd, p + "to_out.1.bias")) + x


# ---------------------------------------------------------------- gates
def logit_error(A: np.ndarray, C: int) -> np.ndarray:
    """Absolute error of an fp32 logit whose terms have absolute sum A over C products: sqrt(C) * 2^-22 * A, four times the
    typical error sqrt(C) u_fp32 A of a C-term fp32 sum (the products of 16-bit operands are exact in fp32)."""
    return np.sqrt(C) * 2.0 ** -22 * A


def chunk_gates(k, v, u_p: float, u_v: float, dk=0.0, dv=0.0, p_floor: float = 0.0, p_flush: float = 0.0):
    """Per (sample, head, chunk, row) gates of a producer whose P = exp(k - m) is rounded with unit roundoff u_p and whose V is
    rounded with u_v (0 when V is the stored operand itself).  A valid pixel contributes p_n (1 + delta_n) to Z and
    p_n (1 + delta_n) v_n (1 + delta'_n) to S, so
        log Z + m - lse  = sum_n p_n delta_n / Z
        S / Z - avg      = sum_n p_n delta_n (v_n - avg) / Z + sum_n p_n delta'_n v_n / Z.
    Round-to-nearest errors are independent with |delta| <= u and variance <= u^2 / 3, which gives the standard deviations
        s_lse = sqrt(sum_n var_n) / Z,   s_avg = sqrt(sum_n (var_n |v_n - avg|^2 + p_n^2 u_v^2 / 3 |v_n|^2)) / Z,
    var_n = (u_p^2 p_n^2 + p_floor^2) / 3 (p_floor: the absolute spacing of P's subnormals, relative to the chunk's row maximum).
    The gates are 6 standard deviations plus the logit error dk (a relative error of every p) and the error dv of v before its
    rounding (absolute), plus 2^-18 (fp32 sums, the approximate exponentials, m stored in fp32):
        g_lse = 6 s_lse + dk + 2^-18
        g_avg = 6 s_avg + (2 dk + 2^-18) sqrt(vsq) + dv sqrt(32)            (a 32-vector norm per row)
    p_flush: pixels whose p, relative to the chunk's row maximum, is below p_flush may be flushed to 0 by the producer (an
    approximate exponential that flushes below 2^-126 under a stabiliser up to 2^100 above the row's maximum: p_flush = 2^-26).
    Their whole contribution is added to the gates: b_n = p_n [p_n < p_flush] / Z, g_lse += sum_n b_n,
    g_avg += sum_n b_n |v_n - avg|.
    dk: scalar or array broadcastable to [N, H, 32, n]; dv: scalar or array broadcastable to [N, H, n]."""
    N, H, _, n = k.shape
    nc = chunks_of(n)
    g_lse = np.empty((N, H, nc, DH))
    g_avg = np.empty((N, H, nc, DH))
    dk = np.broadcast_to(np.asarray(dk, np.float64), k.shape)
    dv = np.broadcast_to(np.asarray(dv, np.float64), (N, H, n))
    for c in range(nc):
        sl = slice(c * CHUNK, (c + 1) * CHUNK)
        kc, vc = k[..., sl], v[..., sl]
        p = np.exp(kc - kc.max(axis=-1, keepdims=True))
        Z = p.sum(axis=-1)
        var = (u_p ** 2 * p ** 2 + p_floor ** 2) / 3.0
        avg = np.einsum("bhdn,bhen->bhde", p, vc) / Z[..., None]
        dev2 = ((vc[:, :, None, :, :] - avg[..., None]) ** 2).sum(axis=3)               # [N, H, d, n]
        vn2 = (vc ** 2).sum(axis=2)[:, :, None, :]
        s_lse = np.sqrt(var.sum(axis=-1)) / Z
        s_avg = np.sqrt((var * dev2 + p ** 2 * (u_v ** 2 / 3.0) * vn2).sum(axis=-1)) / Z
        vsq = (p * vn2).sum(axis=-1) / Z
        dkc = (dk[..., sl] * p).sum(axis=-1) / Z
        dkm = dk[..., sl].max(axis=-1)
        b = np.where(p < p_flush, p, 0.0) / Z[..., None]
        g_lse[:, :, c] = 6 * s_lse + dkc + 2.0 ** -18 + b.sum(axis=-1)
        g_avg[:, :, c] = (6 * s_avg + (2 * dkm + 2.0 ** -18) * np.sqrt(vsq) + dv[..., sl].max(axis=-1)[..., None] * np.sqrt(DH)
                          + (b * np.sqrt(dev2)).sum(axis=-1))
    return g_lse, g_avg


def ctx_gate(lse, avg, vsq, g_lse, g_avg, label_k=None) -> np.ndarray:
    """Per (sample, head, row) gate on ctx: ctx = sum_c omega_c avg_c, where chunk c's avg errs by at most g_avg and its weight
    omega_c by a factor exp(+-2 g_lse) (its own lse and, through the normaliser, the others'):
        g_ctx = sum_c omega_c (g_avg_c + 4 g_lse_c |avg_c|) ."""
    om = chunk_weights(lse, label_k)
    return (om * (g_avg + 4 * g_lse * np.linalg.norm(avg, axis=-1))).sum(axis=2)


def m_gate(g_ctx: np.ndarray, wout: np.ndarray, M_ref: np.ndarray, u_out: float) -> np.ndarray:
    """Per (sample, head) gate on ||M - M_ref||_F: the block is Wout_head dctx^T, so ||dM||_F <= ||Wout_head||_2 ||dctx||_F (spectral
    norm), plus the rounding of M to the 16-bit output type (u_out ||M_ref||)."""
    N, H = g_ctx.shape[:2]
    C = wout.shape[0]
    w = np.asarray(wout, np.float64).reshape(C, H, DH)
    wn = np.array([np.linalg.norm(w[:, h], ord=2) for h in range(H)])             # [H]
    mr = np.linalg.norm(M_ref.reshape(N, M_ref.shape[1], H, DH), axis=(1, 3))     # [N, H]
    return wn[None, :] * np.linalg.norm(g_ctx, axis=-1) + u_out * mr


def q_gate(qp_ref: np.ndarray, u_out: float, dq=0.0, soft: bool = True) -> np.ndarray:
    """Per (sample, head) gate on ||q' - q'_ref||: the 16-bit rounding of the output (u_out per element, relative), a logit error dq
    (softmax: q' (dq_j - mean dq) -> 2 dq relative), and the spacing 2^-24 of IEEE-half subnormals per element."""
    N, H, _, n = qp_ref.shape
    nrm = np.sqrt((qp_ref ** 2).sum(axis=(2, 3)))
    return (u_out + (2 * dq if soft else 0.0) + 2.0 ** -18) * nrm + 2.0 ** -25 * np.sqrt(DH * n)
