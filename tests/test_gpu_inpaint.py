"""Inpainting with text on the GPU: the mask zoom (ds_mask_zoom) of a ragged batch against scipy.ndimage.zoom itself and the float64
oracle (tests/zoom_oracle.py), its batch independence and determinism, the codec.zoom drop-in, and TextToTimbre.inpaint against the
oracle pipeline, against the sampler it wires up, and in its two limiting cases (keep everything, regenerate everything)."""
import numpy as np
import pytest
import scipy.ndimage as nd
import torch

from diffusynth_b200 import _lib, codec, weights as W
from oracle import cases, ds_oracle as O
from tests import zoom_oracle as Z
from tests.gpu_util import rel
from tests.test_gpu_resample import _counting

pytestmark = pytest.mark.gpu

BF16_TOL = 1e-2
# (in shape, out shape, kind): the spectrogram image's grid (513 x T), the encoder's (512 x 4w), a long upload, odd and tiny grids
RAGGED = [((513, 257), (128, 64), "binary"), ((512, 256), (128, 64), "soft"), ((513, 1025), (128, 1), "soft"),
          ((37, 11), (128, 30), "binary"), ((1, 9), (128, 64), "soft"), ((3, 2), (128, 30), "soft"), ((128, 64), (128, 64), "binary"),
          ((513, 257), (128, 30), "rect")]


def _mask(shape, kind, seed):
    rng = np.random.default_rng(seed)
    if kind == "soft":
        return rng.random(shape).astype(np.float32)
    if kind == "binary":
        return (rng.random(shape) > 0.5).astype(np.float32)
    m = np.ones(shape, np.float32)                                          # keep all but a time-frequency rectangle
    H, W_ = shape
    m[H // 5: H // 2, W_ // 3: 2 * W_ // 3] = 0.0
    return m


def _scipy(a, out_shape):
    ref = nd.zoom(a, (out_shape[0] / a.shape[0], out_shape[1] / a.shape[1]))
    assert ref.shape == tuple(out_shape) and ref.dtype == np.float32
    return ref


def _ragged():
    masks = [_mask(s, kind, 10 + k) for k, (s, _, kind) in enumerate(RAGGED)]
    packed = torch.from_numpy(np.concatenate([m.reshape(-1) for m in masks])).cuda()
    return masks, packed, [s for s, _, _ in RAGGED], [o for _, o, _ in RAGGED]


def _split(out, outs):
    return [p.view(o) for p, o in zip(torch.split(out, [h * w for h, w in outs]), outs)]


def test_ragged_batch_against_scipy_and_oracle():
    masks, packed, ins, outs = _ragged()
    got = _split(codec.zoom_packed(packed, ins, outs), outs)
    worst_scipy = worst_oracle = 0.0
    for m, o, g, (s, _, kind) in zip(masks, outs, got, RAGGED):
        g = g.cpu().numpy().astype(np.float64)
        e_s = np.abs(g - _scipy(m, o)).max()
        e_o = np.abs(g - Z.zoom(m, o)).max()
        print(f"\n{s} -> {o} ({kind}): max |err| vs scipy {e_s:.2e}, vs oracle {e_o:.2e}, range [{g.min():.4f}, {g.max():.4f}]")
        worst_scipy, worst_oracle = max(worst_scipy, e_s), max(worst_oracle, e_o)
    print(f"worst max |err|: vs scipy {worst_scipy:.2e}, vs oracle {worst_oracle:.2e}")
    assert worst_scipy <= 1e-5 and worst_oracle <= 1e-5
    ring = got[0].cpu().numpy()                                              # the binary 513 x 257 mask rings as scipy's does
    assert ring.min() < -0.4 and ring.max() > 1.4
    assert abs(ring.min() - _scipy(masks[0], (128, 64)).min()) <= 1e-5 and abs(ring.max() - _scipy(masks[0], (128, 64)).max()) <= 1e-5


def test_batched_items_equal_items_alone_and_calls_repeat():
    masks, packed, ins, outs = _ragged()
    batch = _split(codec.zoom_packed(packed, ins, outs), outs)
    again = _split(codec.zoom_packed(packed, ins, outs), outs)
    for k, m in enumerate(masks):
        alone = codec.zoom_packed(torch.from_numpy(m.reshape(-1)).cuda(), [ins[k]], outs[k]).view(outs[k])
        assert torch.equal(alone, batch[k]) and torch.equal(again[k], batch[k]), RAGGED[k]


def test_zoom_dropin_layouts():
    a = _mask((513, 257), "binary", 1)
    one = codec.zoom(a, (128 / 513, 64 / 257))                              # [H, W] numpy -> numpy
    assert isinstance(one, np.ndarray) and one.dtype == np.float32 and one.shape == (128, 64)
    assert np.abs(one - _scipy(a, (128, 64))).max() <= 1e-5
    b = np.stack([a, _mask((513, 257), "soft", 2)])
    two = codec.zoom(b, (128 / 513, 64 / 257))                              # [B, H, W]
    assert isinstance(two, np.ndarray) and two.shape == (2, 128, 64) and np.array_equal(two[0], one)
    dev = codec.zoom(torch.from_numpy(b).cuda(), (128 / 513, 64 / 257))     # tensor in, tensor out
    assert dev.is_cuda and torch.equal(dev.cpu(), torch.from_numpy(two))
    c = _mask((37, 11), "soft", 3)
    parts = codec.zoom([a, c], [(128 / 513, 64 / 257), (2.0, 3.0)])        # a list of different shapes, one zoom per item
    assert [p.shape for p in parts] == [(128, 64), (74, 33)] and np.array_equal(parts[0], one)
    assert np.abs(parts[1] - nd.zoom(c, (2.0, 3.0))).max() <= 1e-5
    assert codec.zoom(c, 2.0).shape == nd.zoom(c, 2.0).shape                 # scipy's round(n * zoom)


# ---- TextToTimbre.inpaint ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pipe():
    from diffusynth_b200 import TextToTimbre
    return TextToTimbre.random_init(device="cuda", seed=0, perturb_norm=True, batch_invariant=True)     # the oracle's weights


@pytest.fixture(scope="module")
def guide(pipe):
    return pipe.encode_audio(torch.from_numpy(cases.synthetic_wave(seed=33)).float()[None].cuda())      # [1, 4, 128, 64]


def _row_masks(B, seed=0):
    """B different 513 x 257 masks in the spectrogram's orientation: keep the upload except one time-frequency region per row."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(B):
        m = np.ones((513, 257), np.float32)
        f0, t0 = rng.integers(0, 300), rng.integers(0, 150)
        m[f0: f0 + rng.integers(60, 200), t0: t0 + rng.integers(40, 100)] = 0.0
        out.append(m)
    return out


def test_inpaint_pipeline_parity(pipe, guide):
    """Deployed networks, B = 2, 3 steps, CFG 6, a different 513 x 257 mask per row, against the oracle's p_sample_loop with the
    scipy-zoomed masks, then its quantiser, decoder and iSTFT."""
    B, steps = 2, 3
    masks = _row_masks(B)
    draws = W.host_noise(21, 1 + steps, B)
    cond, uncond = W.synthetic_conditions(B, 512)
    out = pipe.inpaint(guide, masks, cond.cuda(), uncond.cuda(), steps=steps, cfg_scale=6, noise_feed=draws)
    usd, vsd = W.unet_random_state_dict(seed=0), W.vqgan_random_state_dict(seed=1)
    _, dec_plan = W.vqgan_layer_plan(W.VQGAN_DEPLOYED)
    sch = O.Schedule(1000)
    sch.respace(list(np.linspace(0, 999, steps, dtype=np.int32)))
    mk = torch.from_numpy(np.stack([_scipy(m, (128, 64)) for m in masks]))[:, None]
    with torch.no_grad():
        ref = O.sample_loop(lambda x, t, c: O.unet_forward(usd, x, t, c), sch, (B, 4, 128, 64), cond, uncond, 6, draws,
                            guide=guide.cpu().repeat(B, 1, 1, 1), mask=mk, inpaint=True)
        q_same, idx = O.vq_quantize(out.latents.cpu(), vsd["_vq_vae._embedding.weight"])
        spec = O.vqgan_decode(vsd, dec_plan, q_same)
    wave_ref = np.stack([O.spectrogram_to_waveform(s.numpy().astype(np.float64)) for s in spec])
    e_lat, e_spec, e_wave = rel(out.latents, ref[-1]), rel(out.spectrograms, spec), rel(out.waveforms, torch.from_numpy(wave_ref))
    print(f"\ninpainting: ({len(ref) - 1} U-Net steps) latent {e_lat:.2e}  spectrogram {e_spec:.2e}  waveform {e_wave:.2e}")
    assert len(ref) == steps + 1
    assert torch.equal(q_same, out.quantized.cpu()) and torch.equal(pipe.vqgan._vq_vae.last_indices.cpu(), idx)
    assert e_lat < BF16_TOL and e_spec < BF16_TOL and e_wave < 2 * BF16_TOL


def test_all_ones_mask_returns_the_guide(pipe, guide):
    """The last blend uses the coefficients (1, 0): where the mask is 1 the result is the guide latent, bit for bit."""
    B, steps = 2, 3
    cond, uncond = W.synthetic_conditions(B, 512)
    out = pipe.inpaint(guide, np.ones((513, 257), np.float32), cond.cuda(), uncond.cuda(), steps=steps,
                       noise_feed=W.host_noise(22, 1 + steps, B), decode=False)
    assert torch.equal(out.latents, guide.repeat(B, 1, 1, 1))


def test_all_zeros_mask_equals_modify_at_full_strength(pipe, guide):
    """Both start from q_sample(guide, T - 1, noise) over ``steps`` respaced steps, and a blend with m = 0 leaves the latent as it is."""
    B, steps = 2, 3
    cond, uncond = W.synthetic_conditions(B, 512)
    draws = W.host_noise(23, 1 + steps, B)
    a = pipe.inpaint(guide, np.zeros((2, 512, 256), np.float32), cond.cuda(), uncond.cuda(), steps=steps, noise_feed=draws)
    b = pipe.modify(guide, cond.cuda(), uncond.cuda(), steps=steps, strength=1.0, noise_feed=draws)
    assert torch.equal(a.latents, b.latents) and torch.equal(a.waveforms, b.waveforms)


def test_inpaint_equals_the_sampler_given_the_zoomed_mask(pipe, guide):
    from diffusynth_b200 import DiffSynthSampler
    B, steps = 2, 3
    masks = _row_masks(B, seed=5)
    cond, uncond = W.synthetic_conditions(B, 512)
    draws = W.host_noise(24, 1 + steps, B)
    got = pipe.inpaint(guide, masks, cond.cuda(), uncond.cuda(), steps=steps, noise_feed=draws, decode=False).latents
    s = DiffSynthSampler(1000, height=128, channels=4, noise_strategy=pipe.noise_strategy, mute=True, device="cuda", max_batchsize=B)
    s.respace(list(np.linspace(0, 999, steps, dtype=np.int32)))
    s.activate_classifier_free_guidance(6, uncond.cuda())
    s.noise_feed = draws[1:]
    mk = torch.from_numpy(np.stack(codec.zoom(masks, (128 / 513, 64 / 257))))[:, None].cuda()
    imgs, _ = s.inpaint_sample(pipe.unet, (B, 4, 128, 64), 1.0, guide.repeat(B, 1, 1, 1), mk, return_tensor=True, condition=cond.cuda(),
                               initial_noise=draws[0].cuda())
    assert torch.equal(imgs[-1], got)


def test_batch_rows_equal_rows_alone(pipe, guide):
    B, steps = 3, 3
    masks = _row_masks(B, seed=7)
    masks[1] = _mask((512, 256), "rect", 8)                                 # rows may come on different grids
    cond, uncond = W.synthetic_conditions(B, 512)
    draws = W.host_noise(25, 1 + steps, B)
    both = pipe.inpaint(guide, masks, cond.cuda(), uncond.cuda(), steps=steps, noise_feed=draws)
    for k in range(B):
        alone = pipe.inpaint(guide, [masks[k]], cond[k:k + 1].cuda(), uncond.cuda(), steps=steps, noise_feed=draws[:, k:k + 1])
        assert torch.equal(alone.latents[0], both.latents[k]) and torch.equal(alone.waveforms[0], both.waveforms[k]), k


def test_inpaint_issues_one_mask_zoom_whatever_the_batch(pipe, guide):
    counts = []
    for B in (2, 5):
        masks = [_mask(((513, 257), (512, 256), (37, 11))[k % 3], "rect", 30 + k) for k in range(B)]
        cond, uncond = W.synthetic_conditions(B, 512)
        pipe.inpaint(guide, masks, cond.cuda(), uncond.cuda(), steps=2)        # warm: sampler, graph and buffers of this batch
        real = _lib.load()
        proxy = _counting(real)
        _lib._lib = proxy
        try:
            pipe.inpaint(guide, masks, cond.cuda(), uncond.cuda(), steps=2)
        finally:
            _lib._lib = real
        counts.append(sorted(proxy.calls))
    print(f"\ninpaint library calls: {len(counts[0])} ({counts[0].count('ds_mask_zoom')} ds_mask_zoom)")
    assert counts[0] == counts[1] and counts[0].count("ds_mask_zoom") == 1 and counts[0].count("ds_mask_zoom_workspace") == 1
