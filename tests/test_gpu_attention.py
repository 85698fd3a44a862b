"""Every linear-attention entry point through the C ABI against the float64 restatement in tests/attn_oracle.py, per chunk:

  producers  ds_attn_qkv_ctx      (fused PreNorm + to_qkv + q soft-max + partial context, heads = 4)
             ds_attn_ctx_partial  (separate path: q_mode 0 with 4 heads, q_mode 1 = the VQGAN's one head)
  finalize   ds_attn_finalize, ds_attn_finalize_cat (attn_reduce_kernel + attn_fold_kernel)

Each case checks that every partial and output is finite (the buffers start as NaN, so every partial was written), q' per
(sample, head), log Z + m - lse and S / Z - avg per (sample, head, chunk, row), and M per (sample, head).  The gates are
derived from the operand types in attn_oracle.chunk_gates / ctx_gate / m_gate / q_gate:
  fused     P and V are bfloat16 (unit roundoff 2^-8), the logits are fp32 sums of C exact products of 16-bit operands
  separate  k and v are the stored 16-bit operands themselves, p = exp(k - m) is IEEE half (2^-11, subnormal spacing 2^-24)
  both      S, Z and the merge accumulate in fp32; q' and M are rounded to the 16-bit activation type (EPS16).
Inputs are seeded and rounded to the 16-bit type before the oracle sees them."""
import numpy as np
import pytest
import torch

from diffusynth_b200 import _lib, ops
from diffusynth_b200._lib import check
from tests import attn_oracle as A
from tests.gpu_util import EPS16

pytestmark = pytest.mark.gpu
HID, HEADS, DH = 128, 4, 32
PART = DH * DH + 2 * DH
LN2E = np.log2(np.e)


def _r16(a: np.ndarray) -> np.ndarray:
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(ops.ACT).double().numpy()


def _dev16(a: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(ops.ACT).cuda()


def _part_buffer(lib, N, heads, npix):
    return torch.full((lib.ds_attn_part_floats(N, heads, npix),), float("nan"), dtype=torch.float32, device="cuda")


def _read_partials(part, N, heads, npix):
    nc = A.chunks_of(npix)
    p = part[:N * heads * nc * PART].double().cpu().numpy().reshape(N, heads, nc, PART)
    S, Z, m = p[..., :DH * DH].reshape(N, heads, nc, DH, DH), p[..., DH * DH:DH * DH + DH], p[..., DH * DH + DH:]
    return S, Z, m


def _ratio(err_norm, gate):
    r = err_norm / gate
    return float(np.where(np.isfinite(r), r, np.inf).max())


def _check(tag, k, v, S, Z, m, g_lse, g_avg, qp=None, qp_ref=None, g_q=None, M=None, M_ref=None, g_M=None):
    """The per-chunk / per-block assertions shared by every case (arrays in the oracle's layouts)."""
    lse, avg, _ = A.chunk_quantities(k, v)
    with np.errstate(divide="ignore", invalid="ignore"):
        e_lse = np.abs(np.log(Z) + m - lse)
        e_avg = np.linalg.norm(S / Z[..., None] - avg, axis=-1)
    r = {"lse": _ratio(e_lse, g_lse), "avg": _ratio(e_avg, g_avg)}
    if qp is not None:
        r["q"] = _ratio(np.sqrt(((qp - qp_ref) ** 2).sum(axis=(2, 3))), g_q)
    if M is not None:
        N, C = M_ref.shape[:2]
        blk = lambda t: t.reshape(N, C, -1, DH)
        r["M"] = _ratio(np.sqrt(((blk(M[:, :C]) - blk(M_ref)) ** 2).sum(axis=(1, 3))), g_M)
    worst = max(r, key=r.get)
    print(f"\n{tag}: error / gate  " + "  ".join(f"{n} {x:.3f}" for n, x in r.items()) +
          f"   max |log Z + m - lse| {np.nanmax(e_lse):.2e}, rows with Z = 0: {int((Z == 0).sum())} of {Z.size}")
    assert np.isfinite(S).all() and np.isfinite(Z).all() and np.isfinite(m).all(), f"{tag}: non-finite partial"
    assert (Z > 0).all(), f"{tag}: {int((Z == 0).sum())} rows of the partials lost every pixel (Z = 0)"
    if qp is not None:
        assert np.isfinite(qp).all(), f"{tag}: non-finite q'"
    if M is not None:
        # (the 16-bit store saturates: a non-finite M shows up as +-65504)
        assert np.isfinite(M).all() and (np.abs(M) < 65504).all(), f"{tag}: non-finite or saturated M"
        assert not M[:, C:].any(), f"{tag}: rows of M past C are not zero"
    assert r[worst] <= 1.0, f"{tag}: {worst} error {r[worst]:.3g} x its gate"


def _finalize(lib, part, wout, N, heads, npix, C, Cout_pad, label=None):
    M = torch.full((N, Cout_pad, heads * DH), float("nan"), dtype=ops.ACT, device="cuda")
    wd = torch.from_numpy(np.ascontiguousarray(wout, np.float32)).cuda()
    s = ops._stream()
    if label is None:
        check(lib.ds_attn_finalize(part.data_ptr(), wd.data_ptr(), M.data_ptr(), N, heads, npix, C, Cout_pad, s), "finalize")
    else:
        lk, lv = (torch.from_numpy(np.ascontiguousarray(t.reshape(N, -1), np.float32)).cuda() for t in label)
        check(lib.ds_attn_finalize_cat(part.data_ptr(), lk.data_ptr(), lv.data_ptr(), lk.stride(0), wd.data_ptr(), M.data_ptr(),
                                       N, heads, npix, C, Cout_pad, s), "finalize_cat")
    torch.cuda.synchronize()
    return M.double().cpu().numpy()


def _labels(rng, lse, where):
    """The linear_cat extra token: its logit far above every chunk's lse (+100), far below (-100), or comparable."""
    N, H = lse.shape[:2]
    base = {"above": lse.max(axis=2) + 100.0, "below": lse.min(axis=2) - 100.0, "comparable": lse.max(axis=2)}[where]
    return base + rng.standard_normal((N, H, DH)), rng.standard_normal((N, H, DH))


def _m_part(lse, avg, vsq, g_lse, g_avg, wout, label):
    lk, lv = label if label is not None else (None, None)
    M_ref = A.fold(A.merge(lse, avg, lk, lv), wout)
    g_ctx = A.ctx_gate(lse, avg, vsq, g_lse, g_avg, lk)
    return M_ref, A.m_gate(g_ctx, wout, M_ref, EPS16)


# ---------------------------------------------------------------------------------------------------- separate path
def _k_logits(rng, shape, kind, npix):
    """k for the separate path: 'std' ~ 1.5 N(0,1); 'wide' spans +-60 natural units with per-row offsets;
    'outlier' adds +90 to tile 2 of every chunk over a row maximum of tile 1."""
    if kind == "std":
        return rng.standard_normal(shape) * 1.5
    k = rng.uniform(-20, 20, shape) + rng.uniform(-40, 40, shape[:-1] + (1,))
    if kind == "outlier":
        k = rng.standard_normal(shape) * 2
        for c0 in range(0, npix, A.CHUNK):
            t2 = slice(c0 + 2 * A.TILE, min(c0 + 3 * A.TILE, npix))
            k[..., t2] += 90.0
    return k


SEPARATE_CASES = [
    # (q_mode, heads, N, npix, C, Cout_pad, k kind, finalize label)
    *[(0, 4, 1, n, 96, 96, "std", None) for n in (1, 5, 127, 128, 129, 511, 512, 513, 4097)],
    (0, 4, 3, 4097, 96, 112, "wide", None),
    (0, 4, 3, 2100, 96, 96, "outlier", "above"),
    (0, 4, 2, 32768, 192, 192, "wide", "below"),
    (0, 4, 1, 32769, 64, 64, "std", "comparable"),
    (1, 1, 2, 131072, 80, 96, "std", None),          # the decoder's 80-channel level (512 x 256): 256 chunks
    (1, 1, 1, 32769, 160, 160, "wide", None),
    (1, 1, 2, 513, 80, 96, "outlier", None),
]


@pytest.mark.parametrize("q_mode,heads,N,npix,C,Cout_pad,kind,label", SEPARATE_CASES)
def test_ctx_partial_per_chunk(q_mode, heads, N, npix, C, Cout_pad, kind, label):
    lib = _lib.load()
    rng = np.random.default_rng(npix * 7 + heads + q_mode)
    hid = heads * DH
    q = rng.standard_normal((N, heads, DH, npix)) * (1.5 if q_mode == 0 else 1.0)
    k = _k_logits(rng, (N, heads, DH, npix), kind, npix)
    v = rng.standard_normal((N, heads, DH, npix)) + rng.standard_normal((N, heads, DH, 1))
    q, k, v = _r16(q), _r16(k), _r16(v)
    qkv = np.concatenate([t.reshape(N, hid, npix) for t in (q, k, v)], axis=1).transpose(0, 2, 1)     # [N, npix, 3 hid]
    qkv_d = _dev16(qkv)
    qp_d = torch.full((N, npix + 8, hid), float("nan"), dtype=ops.ACT, device="cuda")                   # 8 guard rows per sample
    part = _part_buffer(lib, N, heads, npix)
    scale = DH ** -0.5 if q_mode == 0 else 1.0
    # q' rows are [N][npix][hid]: write through a view with the guard rows at the end of the buffer
    qp_flat = qp_d.view(-1)
    check(lib.ds_attn_ctx_partial(qkv_d.data_ptr(), qp_flat.data_ptr(), part.data_ptr(), N, heads, npix, q_mode, scale, ops._stream()), "ctx")
    torch.cuda.synchronize()
    qp = qp_flat[:N * npix * hid].double().cpu().numpy().reshape(N, npix, heads, DH).transpose(0, 2, 3, 1)
    assert torch.isnan(qp_flat[N * npix * hid:].float()).all(), "q' written past the end of the batch"
    S, Z, m = _read_partials(part, N, heads, npix)

    dk = 2.0 ** -21 * (1.0 + 2 * np.abs(k).max())                            # __expf(k - m): fp32 argument and ex2.approx
    g_lse, g_avg = A.chunk_gates(k, v, A.U_FP16, 0.0, dk=dk, p_floor=2.0 ** -25)
    lse, avg, vsq = A.chunk_quantities(k, v)
    wout = rng.standard_normal((C, hid)) * 0.1
    lab = _labels(rng, lse, label) if label is not None else None
    M = _finalize(lib, part, wout, N, heads, npix, C, Cout_pad, lab)
    M_ref, g_M = _m_part(lse, avg, vsq, g_lse, g_avg, wout, lab)
    if q_mode == 0:
        qp_ref = A.q_prime(q, scale=scale)
        g_q = A.q_gate(qp_ref, EPS16, dq=2.0 ** -21 * (1.0 + 2 * np.abs(q).max()))
    else:
        assert np.array_equal(qp, q), "q_mode 1 must copy q bit for bit"
        qp_ref, g_q = q, A.q_gate(q, 0.0, soft=False)
    _check(f"separate q_mode={q_mode} heads={heads} N={N} npix={npix} C={C}/{Cout_pad} k={kind} label={label}",
           k, v, S, Z, m, g_lse, g_avg, qp, qp_ref, g_q, M, M_ref, g_M)


# ---------------------------------------------------------------------------------------------------- fused path
FUSED_CASES = [
    # (N, C, npix, x_batch_mod, mu/sigma, with stats, with sbias, logit range, finalize label)
    *[(1, 96, n, 0, 0.3, True, True, "std", None) for n in (1, 5, 127, 129, 511, 513, 4097)],
    (3, 64, 640, 0, 0.3, True, True, "std", None),
    (3, 192, 1100, 0, 0.3, True, True, "std", None),
    (3, 384, 700, 0, 0.3, True, True, "std", None),
    (2, 96, 4097, 0, 20.0, True, True, "std", None),
    (2, 96, 4097, 0, 50.0, True, True, "std", None),
    (2, 384, 1024, 0, 50.0, True, True, "std", None),
    (4, 96, 1500, 2, "mixed", True, True, "std", None),                 # x_batch_mod: two very different samples, each used twice
    (2, 96, 1000, 0, 0.3, False, True, "std", None),                    # d_stats_in NULL: no norm
    (2, 96, 1500, 0, 0.3, True, False, "std", "above"),                 # d_sbias NULL + finalize_cat (the U-Net's linear_cat)
    (2, 96, 1500, 0, 0.3, True, False, "std", "below"),
    (2, 192, 1500, 0, 0.3, True, False, "std", "comparable"),
    (2, 96, 4097, 0, 0.3, True, True, "wide", None),                   # k logits spanning +-60
    (2, 96, 2600, 0, 0.3, True, True, "outlier", None),                # tiles 2 / 3 of chunks 0 / 3 ~90 above tile 1
    (2, 96, 1300, 0, 0.3, True, True, "q50", None),                    # q logits x 50
    (1, 64, 32768, 0, 0.3, True, True, "std", None),                   # 64 chunks (the reduce keeps every weight)
    (1, 64, 32769, 0, 20.0, True, True, "std", "comparable"),          # 65 chunks: the reduce's recompute branch
]


def _fused_inputs(rng, N, C, npix, mod, mu, rng_kind):
    n_in = mod if mod else N
    x = rng.standard_normal((n_in, C, npix))
    if mu == "mixed":
        x[0] = x[0] * 0.5 + 0.2
        x[1] = x[1] * 30.0 - 600.0
    else:
        x = x + mu
    w = rng.standard_normal((3 * HID, C)) * (2 / C ** 0.5)
    if rng_kind == "wide":
        w[HID:2 * HID] *= 4.0
    if rng_kind == "q50":
        w[:HID] *= 50.0
    if rng_kind == "outlier":
        # 8 pixels of tile 2 of chunk 0 and of tile 3 of chunk 3 move along k row 5 of head 1 (unit direction u): that row's
        # logit there rises ~90 natural units above its maximum over tile 1
        u = w[HID + DH + 5] / np.linalg.norm(w[HID + DH + 5])
        for p0 in (2 * A.TILE + 40, 3 * A.CHUNK + 3 * A.TILE + 7):
            x[:, :, p0:p0 + 8] += 52.0 * u[None, :, None]
    gamma = 2.0 ** rng.integers(-1, 2, C)           # powers of two: folding gamma into the 16-bit weights stays exact
    beta = rng.standard_normal(C) * 0.2
    return _r16(x), _r16(w), gamma, beta


@pytest.mark.parametrize("N,C,npix,mod,mu,stats,sbias,rng_kind,label", FUSED_CASES)
def test_qkv_ctx_per_chunk(N, C, npix, mod, mu, stats, sbias, rng_kind, label):
    lib = _lib.load()
    rng = np.random.default_rng(npix * 13 + C + N)
    x, w, gamma, beta = _fused_inputs(rng, N, C, npix, mod, mu, rng_kind)
    n_in = x.shape[0]
    pc = ops.pack_conv_s1(torch.from_numpy(w).float().view(3 * HID, C, 1, 1), None, torch.from_numpy(gamma).float(),
                          torch.from_numpy(beta).float()).to("cuda")
    mean64, rstd64 = A.group_norm_stats(x)
    mean, rstd = mean64.astype(np.float32), rstd64.astype(np.float32)
    st = ops.given_stats(torch.from_numpy(mean), torch.from_numpy(rstd), npix * C)
    sb = rng.standard_normal((N, 3 * HID)) * 0.5
    sb[:, 2 * HID:] = 0
    sb = sb.astype(np.float32).astype(np.float64)
    sbd = torch.from_numpy(sb).float().cuda()
    xd = _dev16(x.transpose(0, 2, 1))                                     # NHWC [n_in][npix][C]
    qp_flat = torch.full((N * npix * HID + 8 * HID,), float("nan"), dtype=ops.ACT, device="cuda")
    part = _part_buffer(lib, N, HEADS, npix)
    check(lib.ds_attn_qkv_ctx(xd.data_ptr(), C, mod, st.buf.data_ptr() if stats else None, st.slots, pc.weight.data_ptr(),
                              pc.e1.data_ptr(), pc.e2.data_ptr(), sbd.data_ptr() if sbias else None, sbd.stride(0),
                              qp_flat.data_ptr(), part.data_ptr(), N, HEADS, npix, DH ** -0.5, ops._stream()), "qkv_ctx")
    torch.cuda.synchronize()
    qp = qp_flat[:N * npix * HID].double().cpu().numpy().reshape(N, npix, HEADS, DH).transpose(0, 2, 3, 1)
    assert torch.isnan(qp_flat[N * npix * HID:].float()).all(), "q' written past the end of the batch"
    S, Z, m = _read_partials(part, N, HEADS, npix)

    # oracle on the same operands: x and W as rounded, gamma exact, the fp32 statistics the kernel is handed
    src = [i % mod if mod else i for i in range(N)]
    xs = x[src]
    mn, rs = (mean[src], rstd[src]) if stats else (np.zeros(N), np.ones(N))
    qkv = A.qkv_logits(xs, w, gamma, beta, sb if sbias else None, mean=mn, rstd=rs)
    q, k, v = A.split_heads(qkv, HEADS)
    # absolute sum of the terms of every logit (fp32: rstd * sum_c |W' x| + |mean rstd e1| + |e2| + |bias|) -> its fp32 error
    wf = w * gamma[None, :]
    terms = np.einsum("oc,bcn->bon", np.abs(wf), np.abs(xs)) * np.asarray(rs, np.float64)[:, None, None]
    terms += (np.abs(np.asarray(mn, np.float64) * np.asarray(rs, np.float64))[:, None] * np.abs(wf.sum(axis=1))[None, :])[..., None]
    terms += (np.abs(w @ beta)[None, :] + (np.abs(sb) if sbias else 0.0))[..., None]
    dq, dk, dv = (A.logit_error(t, C) for t in np.split(terms, 3, axis=1))
    dq, dk = dq.reshape(q.shape) * LN2E + 2.0 ** -21, dk.reshape(k.shape) * LN2E + 2.0 ** -21    # (+ ex2.approx)
    dv = dv.reshape(v.shape).max(axis=2)
    g_lse, g_avg = A.chunk_gates(k, v, A.U_BF16, A.U_BF16, dk=dk, dv=dv, p_flush=2.0 ** -26)
    lse, avg, vsq = A.chunk_quantities(k, v)
    if rng_kind == "outlier":      # the case is what it claims: some row's tile 2 is >= 88 above its tile-1 maximum
        jump = k[..., 2 * A.TILE:3 * A.TILE].max(-1) - k[..., :A.TILE].max(-1)
        assert 88 <= jump.max() <= 120, jump.max()
    if rng_kind == "wide":
        assert k.max() - k.min() >= 100
    wout = rng.standard_normal((C, HID)) * 0.1
    lab = _labels(rng, lse, label) if label is not None else None
    Cp = ops.pad16(C) if C % 16 else C + 16                               # Cout_pad > C
    M = _finalize(lib, part, wout, N, HEADS, npix, C, Cp, lab)
    M_ref, g_M = _m_part(lse, avg, vsq, g_lse, g_avg, wout, lab)
    qp_ref = A.q_prime(q)
    g_q = A.q_gate(qp_ref, EPS16, dq=dq.max(axis=(2, 3)))
    _check(f"fused N={N} C={C} npix={npix} mod={mod} mu={mu} stats={stats} sbias={sbias} {rng_kind} label={label}",
           k, v, S, Z, m, g_lse, g_avg, qp, qp_ref, g_q, M, M_ref, g_M)
