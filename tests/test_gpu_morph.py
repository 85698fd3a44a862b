"""Timbre morphs on the GPU: the ds_morph_rows kernel against the sampler's generate_linear_noise (bit for bit) and the float64
oracle (tests/morph_oracle.py), its batch independence and determinism; Timbres.initial_noise fed back into generate; DDIM
inversion against the oracle loop on both graph paths and the generic loop; and TextToTimbre.morph against generate at its end
frames, against DiffSynthSampler.interpolate, and against the oracle pipeline."""
import numpy as np
import pytest
import torch

from diffusynth_b200 import _lib, codec, weights as W
from oracle import cases, ds_oracle as O
from tests import morph_oracle as M
from tests.gpu_util import rel
from tests.test_gpu_resample import _counting

pytestmark = pytest.mark.gpu

BF16_TOL = 1e-2
NZ = (4, 128, 64)
L = 512


def _endpoints(P, seed):
    e0, e1 = cases.randn((P,) + NZ, seed), cases.randn((P,) + NZ, seed + 1)
    c0, c1 = cases.randn((P, L), seed + 2), cases.randn((P, L), seed + 3)
    return e0.cuda(), e1.cuda(), c0.cuda(), c1.cuda()


# ---- the kernel ---------------------------------------------------------------------------------------------------------------
def test_linear_rows_equal_generate_linear_noise_bit_for_bit():
    from diffusynth_b200 import DiffSynthSampler
    P, N = 3, 5
    e0, e1, c0, c1 = _endpoints(P, 10)
    noise, cond = codec.morph_rows(e0, e1, c0, c1, N, "linear")
    s = DiffSynthSampler(1000, device="cuda", mute=True)
    for p in range(P):
        ref = s.generate_linear_noise((N,) + NZ, first_endpoint=e0[p], second_endpoint=e1[p])
        assert torch.equal(noise.view(P, N, *NZ)[p], ref), p
        for k in range(N):
            a = k / (N - 1)
            assert torch.equal(cond[p * N + k], a * c1[p] + (1 - a) * c0[p]), (p, k)
    c1[:, ::3] = c0[:, ::3]                                             # shared elements are copied, not re-rounded
    _, cond = codec.morph_rows(e0, e1, c0, c1, N, "linear")
    rows = cond.view(P, N, L)
    assert torch.equal(rows[:, :, ::3], c0[:, None, ::3].expand(P, N, -1))
    assert torch.equal(codec.morph_rows(e0, e1, c0, c0, N, "slerp")[1].view(P, N, L), c0[:, None].expand(P, N, L))


@pytest.mark.parametrize("P", [1, 3, 17])
@pytest.mark.parametrize("N", [2, 5, 33])
def test_slerp_rows_against_the_oracle(P, N):
    e0, e1, c0, c1 = _endpoints(P, 20 + P + N)
    noise, cond = codec.morph_rows(e0, e1, c0, c1, N, "slerp")
    ref = torch.from_numpy(M.slerp_rows(e0.cpu().numpy(), e1.cpu().numpy(), N))
    err = rel(noise.view(P * N, *NZ), ref)
    print(f"\nslerp P={P} N={N}: rel-L2 {err:.2e}")
    assert err <= 1e-6
    rows = noise.view(P, N, *NZ)
    assert torch.equal(rows[:, 0], e0) and torch.equal(rows[:, -1], e1)
    assert torch.equal(cond, codec.morph_rows(e0, e1, c0, c1, N, "linear")[1])      # conditions stay linear


def test_rows_repeat_and_do_not_depend_on_the_batch():
    P, N = 5, 7
    e0, e1, c0, c1 = _endpoints(P, 40)
    e1[1] = e0[1]                                                       # identical endpoints: the linear fallback
    e1[3] = -e0[3]                                                      # antipodal: the linear fallback, zero midpoint
    for path in ("linear", "slerp"):
        noise, cond = codec.morph_rows(e0, e1, c0, c1, N, path)
        again = codec.morph_rows(e0, e1, c0, c1, N, path)
        assert torch.equal(noise, again[0]) and torch.equal(cond, again[1]), path
        assert torch.isfinite(noise).all()
        for p in range(P):
            alone = codec.morph_rows(e0[p:p + 1], e1[p:p + 1], c0[p:p + 1], c1[p:p + 1], N, path)
            assert torch.equal(alone[0], noise[p * N:(p + 1) * N]) and torch.equal(alone[1], cond[p * N:(p + 1) * N]), (path, p)
    lin = codec.morph_rows(e0, e1, c0, c1, N, "linear")[0].view(P, N, -1)
    slerp = codec.morph_rows(e0, e1, c0, c1, N, "slerp")[0].view(P, N, -1)
    assert torch.equal(slerp[1], lin[1]) and torch.equal(slerp[3], lin[3]) and not torch.equal(slerp[0], lin[0])
    assert slerp[3, N // 2].abs().max().item() == 0.0


# ---- pipeline ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pipe():
    from diffusynth_b200 import TextToTimbre
    return TextToTimbre.random_init(device="cuda", seed=0, perturb_norm=True, batch_invariant=True)     # the oracle's weights


@pytest.mark.parametrize("width", [64, 40])
def test_generated_initial_noise_recreates_the_timbre(pipe, width):
    B = 2
    cond, uncond = W.synthetic_conditions(B, L)
    a = pipe.generate(cond.cuda(), uncond.cuda(), steps=2, width=width, seed=3)
    assert tuple(a.initial_noise.shape) == (B,) + NZ
    b = pipe.generate(cond.cuda(), uncond.cuda(), steps=2, width=width, noise_feed=[a.initial_noise])
    assert torch.equal(a.latents, b.latents) and torch.equal(a.waveforms, b.waveforms) and torch.equal(b.initial_noise, a.initial_noise)
    draws = W.host_noise(4, 3, B)                                     # a host feed: initial_noise is its draw 0
    c = pipe.generate(cond.cuda(), uncond.cuda(), steps=2, width=width, noise_feed=draws, decode=False)
    assert torch.equal(c.initial_noise.cpu(), draws[0])


@pytest.mark.parametrize("entry", ["modify", "inpaint", "synthesize_note"])
def test_one_draw_feed_runs_like_the_full_feed(pipe, entry):
    """A feed of draw 0 alone, as generate takes it: the step draws come from the RNG, and DDIM multiplies them by sigma = 0, so
    the result is the full feed's; initial_noise is draw 0 either way."""
    steps, B = 2, (1 if entry == "synthesize_note" else 2)
    guide = cases.vq_latents(B=1, seed=66).cuda()
    cond, uncond = W.synthetic_conditions(B, L)
    draws = W.host_noise(6, 1 + 2 * steps, B)                         # enough step draws for modify's int(steps / 0.5)
    mask = np.ones((513, 257), np.float32)
    mask[100:300, 60:180] = 0.0

    def run(feed):
        if entry == "modify":
            return pipe.modify(guide, cond.cuda(), uncond.cuda(), steps=steps, strength=0.5, noise_feed=feed)
        if entry == "inpaint":
            return pipe.inpaint(guide, mask, cond.cuda(), uncond.cuda(), steps=steps, noise_feed=feed)
        return pipe.synthesize_note(guide, cond.cuda(), 0.9, sample_steps=steps, noise_feed=feed)
    full, one = run(draws), run([draws[0]])
    assert torch.equal(one.latents, full.latents) and torch.equal(one.waveforms, full.waveforms)
    assert torch.equal(one.initial_noise.cpu(), draws[0]) and torch.equal(full.initial_noise.cpu(), draws[0])


def _small_unet(use_engine):
    from diffusynth_b200 import ConditionedUnet
    cfg, sd, _, _, cond = cases.unet_case("small_w16")
    net = ConditionedUnet(**{k: v for k, v in cfg.items() if k not in ("out_dim", "time_dim")}, device="cuda")
    net.load_state_dict(sd)
    net.use_engine = use_engine
    return net, sd, cond


@pytest.mark.parametrize("cfg_scale", [1.0, 3.0])
@pytest.mark.parametrize("use_engine", [True, False])
def test_invert_small_unet_against_the_oracle(cfg_scale, use_engine):
    from diffusynth_b200 import DiffSynthSampler
    net, sd, cond = _small_unet(use_engine)
    uncond = cases.randn((cond.shape[1],), 62)
    x0 = cases.randn((2, 4, 32, 64), 61)
    s = DiffSynthSampler(1000, device="cuda", mute=True, height=32, max_batchsize=2)
    s.respace(list(np.linspace(0, 999, 6, dtype=np.int32)))
    s.activate_classifier_free_guidance(cfg_scale, uncond.cuda())
    imgs, none = s.ddim_invert(net, x0.cuda(), cond.cuda())
    sch = O.Schedule(1000)
    sch.respace(list(np.linspace(0, 999, 6, dtype=np.int32)))
    assert none is None and np.array_equal(np.array([s._invert_coef(t) for t in range(6)]), M.invert_coefficients(sch, cfg_scale))
    with torch.no_grad():
        ref = M.ddim_invert(lambda x, t, c: O.unet_forward(sd, x, t, c), sch, x0, cond, uncond, cfg_scale)
    errs = [rel(a, b) for a, b in zip(imgs[1:], ref[1:])]
    print(f"\ninvert small_w16 cfg={cfg_scale} engine={use_engine}: per-step rel-L2 {' '.join(f'{e:.1e}' for e in errs)}")
    assert len(imgs) == 7 and torch.equal(imgs[0].cpu(), x0) and max(errs) < BF16_TOL


def test_invert_generic_model_against_the_oracle():
    from diffusynth_b200 import DiffSynthSampler
    cond, uncond = W.synthetic_conditions(2, 16, seed=91)
    x0 = cases.randn((2, 4, 16, 64), 63)
    s = DiffSynthSampler(1000, device="cuda", mute=True, height=16, max_batchsize=2)
    s.respace(list(np.linspace(0, 999, 6, dtype=np.int32)))
    s.activate_classifier_free_guidance(3.0, uncond.cuda())
    imgs, _ = s.ddim_invert(cases.toy_model, x0.cuda(), cond.cuda())
    sch = O.Schedule(1000)
    sch.respace(list(np.linspace(0, 999, 6, dtype=np.int32)))
    ref = M.ddim_invert(cases.toy_model, sch, x0, cond, uncond, 3.0)
    assert max(rel(a, b) for a, b in zip(imgs[1:], ref[1:])) < 1e-5      # fp32 throughout


def test_invert_deployed_against_the_oracle(pipe):
    B, steps = 2, 3
    lat = cases.vq_latents(B=B, seed=64)
    cond, _ = W.synthetic_conditions(B, L)
    got = pipe.invert(lat.cuda(), cond.cuda(), steps=steps)
    usd = W.unet_random_state_dict(seed=0)
    sch = O.Schedule(1000)
    sch.respace(list(np.linspace(0, 999, steps, dtype=np.int32)))
    with torch.no_grad():
        ref = M.ddim_invert(lambda x, t, c: O.unet_forward(usd, x, t, c), sch, lat, cond, None, 1.0)
    err = rel(got, ref[-1])
    print(f"\ninvert deployed B={B} steps={steps}: noise rel-L2 {err:.2e}")
    assert tuple(got.shape) == (B,) + NZ and err < BF16_TOL


def _calls(pipe, fn):
    real = _lib.load()
    proxy = _counting(real)
    _lib._lib = proxy
    try:
        fn()
    finally:
        _lib._lib = real
    return sorted(proxy.calls), pipe.last_launches


def test_invert_launches_as_generate_does(pipe):
    B, steps = 2, 3
    cond, uncond = W.synthetic_conditions(B, L)
    lat = cases.vq_latents(B=B, seed=65).cuda()
    for cfg_scale in (1.0, 6.0):
        u = uncond.cuda() if cfg_scale != 1.0 else None
        pipe.invert(lat, cond.cuda(), u, steps=steps, cfg_scale=cfg_scale)           # warm: sampler and graph of this shape
        pipe.generate(cond.cuda(), u, steps=steps, cfg_scale=cfg_scale, decode=False)
        inv = _calls(pipe, lambda: pipe.invert(lat, cond.cuda(), u, steps=steps, cfg_scale=cfg_scale))
        gen = _calls(pipe, lambda: pipe.generate(cond.cuda(), u, steps=steps, cfg_scale=cfg_scale, decode=False))
        print(f"\ninvert cfg={cfg_scale}: {inv[1]} graph launches, library calls {inv[0]}")
        assert inv == gen


@pytest.mark.parametrize("path", ["linear", "slerp"])
def test_morph_end_frames_equal_generate(pipe, path):
    P, N, steps = 2, 3, 2
    e0, e1, c0, c1 = _endpoints(P, 70)
    _, uncond = W.synthetic_conditions(1, L)
    m = pipe.morph(e0, e1, c0, c1, uncond.cuda(), N, path=path, steps=steps)
    m_idx = pipe.vqgan._vq_vae.last_indices.view(P, N, -1)
    assert tuple(m.latents.shape) == (P * N,) + NZ and torch.equal(m.initial_noise.reshape(P, N, *NZ)[:, 0], e0)
    for k, (e, c) in ((0, (e0, c0)), (N - 1, (e1, c1))):
        g = pipe.generate(c, uncond.cuda(), steps=steps, noise_feed=[e])
        g_idx = pipe.vqgan._vq_vae.last_indices.view(P, -1)
        rows = [p * N + k for p in range(P)]
        assert torch.equal(m.latents[rows], g.latents) and torch.equal(m_idx[:, k], g_idx), (path, k)
        assert torch.equal(m.quantized[rows], g.quantized) and torch.equal(m.waveforms[rows], g.waveforms), (path, k)


def test_linear_morph_with_equal_conditions_equals_interpolate(pipe):
    from diffusynth_b200 import DiffSynthSampler
    N, steps = 4, 2
    e0, e1, c0, _ = _endpoints(1, 80)
    _, uncond = W.synthetic_conditions(1, L)
    m = pipe.morph(e0[0], e1[0], c0[0], c0[0], uncond.cuda(), N, path="linear", steps=steps, decode=False)
    s = DiffSynthSampler(1000, device="cuda", mute=True, max_batchsize=N)
    s.respace(list(np.linspace(0, 999, steps, dtype=np.int32)))
    s.activate_classifier_free_guidance(6, uncond.cuda())
    imgs, init = s.interpolate(pipe.unet, (N,) + NZ, 1.0, first_endpoint=e0[0], second_endpoint=e1[0], return_tensor=True,
                               condition=c0.repeat(N, 1))
    assert torch.equal(init, m.initial_noise) and torch.equal(imgs[-1], m.latents)


def test_morph_is_one_graph_launch(pipe):
    P, N, steps = 2, 3, 2
    e0, e1, c0, c1 = _endpoints(P, 90)
    cond, uncond = W.synthetic_conditions(P * N, L)
    pipe.morph(e0, e1, c0, c1, uncond.cuda(), N, steps=steps)        # warm
    calls, launches = _calls(pipe, lambda: pipe.morph(e0, e1, c0, c1, uncond.cuda(), N, steps=steps))
    pipe.generate(cond.cuda(), uncond.cuda(), steps=steps)
    print(f"\nmorph P={P} N={N}: {launches} graph launches, library calls {calls}")
    assert launches == pipe.last_launches
    assert calls.count("ds_morph_rows") == 1 and calls.count("ds_morph_rows_workspace") == 1


def test_morph_against_the_oracle_pipeline(pipe):
    """P = 1, N = 3 at the deployed size, CFG 6, 3 DDIM steps: the slerp rows against the float64 oracle, then the oracle's loop from
    the kernel's rows under the linearly interpolated conditions, its quantiser, decoder and iSTFT."""
    N, steps = 3, 3
    e0, e1, c0, c1 = _endpoints(1, 100)
    _, uncond = W.synthetic_conditions(1, L)
    m = pipe.morph(e0[0], e1[0], c0[0], c1[0], uncond.cuda(), N, steps=steps)
    rows = m.initial_noise.cpu()
    e_rows = rel(rows, torch.from_numpy(M.slerp_rows(e0.cpu().numpy(), e1.cpu().numpy(), N)))
    cond = torch.from_numpy(M.linear_rows(c0.cpu().numpy(), c1.cpu().numpy(), N)).float()
    draws = torch.cat([rows[None], torch.zeros((steps, N) + NZ)])     # DDIM: the per-step draws are multiplied by sigma = 0
    usd, vsd = W.unet_random_state_dict(seed=0), W.vqgan_random_state_dict(seed=1)
    _, dec_plan = W.vqgan_layer_plan(W.VQGAN_DEPLOYED)
    sch = O.Schedule(1000)
    sch.respace(list(np.linspace(0, 999, steps, dtype=np.int32)))
    with torch.no_grad():
        ref = O.sample_loop(lambda x, t, c: O.unet_forward(usd, x, t, c), sch, (N,) + NZ, cond, uncond, 6, draws)
        q_same, idx = O.vq_quantize(m.latents.cpu(), vsd["_vq_vae._embedding.weight"])
        spec = O.vqgan_decode(vsd, dec_plan, q_same)
    wave_ref = np.stack([O.spectrogram_to_waveform(s.numpy().astype(np.float64)) for s in spec])
    e_lat, e_wave = rel(m.latents, ref[-1]), rel(m.waveforms, torch.from_numpy(wave_ref))
    print(f"\nmorph vs oracle: rows {e_rows:.2e}  latent {e_lat:.2e}  waveform {e_wave:.2e}")
    assert e_rows <= 1e-6
    assert torch.equal(q_same, m.quantized.cpu()) and torch.equal(pipe.vqgan._vq_vae.last_indices.cpu(), idx)
    assert e_lat < BF16_TOL and e_wave < 2 * BF16_TOL
