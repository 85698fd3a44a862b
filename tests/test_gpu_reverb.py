"""Convolution reverb on the GPU: ds_fftconvolve against scipy.signal.fftconvolve in float64 over a ragged batch in every mode, its
bit-exact relations (batched == alone, repeats, shared IR, accumulate, zero input), its shared peak, the codec.fftconvolve
layouts, and TextToTimbre.render_arrangement(impulse_response=...) against the oracle chain (tests/reverb_oracle.py) and the
reverb-free render."""
import numpy as np
import pytest
import scipy.signal
import torch

from diffusynth_b200 import _lib, codec, weights as W
from diffusynth_b200.pipeline import Timbres
from oracle import cases
from tests import arrangement_oracle as A
from tests import reverb_oracle as RV
from tests.gpu_util import rel
from tests.test_gpu_track import _counting

pytestmark = pytest.mark.gpu

# (N, M): single samples, the partition size and its neighbours on both sides, M > N, and a 10**6-sample item with a 3 s IR
PAIRS = [(1, 1), (1, 7), (2, 1024), (1023, 1025), (1024, 1024), (1025, 1023), (3000, 48000), (5000, 1), (50000, 3000),
         (1_000_000, 48000), (777, 2049), (2048, 1000)]


def _batch(pairs, seed=0):
    rng = np.random.default_rng(seed)
    xs = [rng.standard_normal(n).astype(np.float32) for n, _ in pairs]
    hs = [(rng.standard_normal(m) * np.exp(-np.arange(m) / max(m / 4, 1))).astype(np.float32) for _, m in pairs]
    return xs, hs


def _run(xs, hs, mode="full", h_index=None, **kw):
    hi = list(range(len(xs))) if h_index is None else h_index
    rng = [codec.fftconvolve_range(len(x), len(hs[i]), mode) for x, i in zip(xs, hi)]
    out = codec.fftconvolve_packed(torch.from_numpy(np.concatenate(xs)).cuda(), [len(x) for x in xs],
                                   torch.from_numpy(np.concatenate(hs)).cuda(), [len(h) for h in hs], hi,
                                   [s for s, _ in rng], [n for _, n in rng], **kw)
    return list(torch.split(out, [n for _, n in rng]))


@pytest.mark.parametrize("mode", codec.CONV_MODES)
def test_ragged_batch_against_scipy_float64(mode):
    xs, hs = _batch(PAIRS)
    got = _run(xs, hs, mode)
    errs = []
    for x, h, g in zip(xs, hs, got):
        ref = scipy.signal.fftconvolve(x.astype(np.float64), h.astype(np.float64), mode=mode)
        assert g.numel() == len(ref)
        errs.append(rel(g, torch.from_numpy(ref)))
    print(f"\nfftconvolve {mode}: rel-L2 vs scipy float64 per item " + " ".join(f"{n}x{m}:{e:.1e}" for (n, m), e in zip(PAIRS, errs)))
    assert max(errs) <= 1e-5


def test_batched_equals_alone_repeats_and_shared_ir():
    xs, hs = _batch(PAIRS, seed=1)
    for mode in codec.CONV_MODES:
        batched = _run(xs, hs, mode)
        again = _run(xs, hs, mode)
        for k in (0, 3, 6, 9, 11):
            alone = _run([xs[k]], [hs[k]], mode)[0]
            assert torch.equal(batched[k], alone), (mode, k)
        assert all(torch.equal(a, b) for a, b in zip(batched, again))
    # one shared IR (transformed once) equals per-item copies of it
    ir = hs[6]
    shared = _run(xs, [ir], h_index=[0] * len(xs))
    copies = _run(xs, [ir] * len(xs))
    assert all(torch.equal(a, b) for a, b in zip(shared, copies))


def test_accumulate_and_zero_input():
    xs, hs = _batch(PAIRS[:9], seed=2)
    conv = torch.cat(_run(xs, hs))
    prev = torch.randn(conv.numel(), device="cuda")
    out = prev.clone()
    got = _run(xs, hs, out=out, accumulate=True)
    assert got[0].data_ptr() == out.data_ptr() and torch.equal(out, prev + conv)
    zeros = torch.cat(_run([np.zeros_like(x) for x in xs], hs))
    assert not zeros.any()


def test_shared_peak_over_the_call():
    xs, hs = _batch([(30000, 4000), (30000, 4000), (1000, 5000)], seed=3)
    hs[1] = hs[1] * 3
    raw = torch.cat(_run(xs, hs))
    for peak in (0.8, 3.0):
        out = torch.cat(_run(xs, hs, target_peak=peak))
        top = float(out.abs().max())
        print(f"\npeak {peak}: max |out| {top!r}")
        assert abs(top - peak) <= 2 * np.spacing(np.float32(peak))
        sc = np.float32(peak) / np.float32(raw.abs().max().item())              # one factor for every item
        want = (raw * float(sc)).cpu()
        assert ((out.cpu() - want).abs() <= torch.from_numpy(np.spacing(want.abs().numpy()))).all()
    zero = torch.cat(_run([np.zeros(3000, np.float32)] * 2, hs[:2], target_peak=0.9))
    assert not zero.any()


def test_drop_in_layouts():
    rng = np.random.default_rng(4)
    x2, h1, h2 = rng.standard_normal((3, 5000)), rng.standard_normal(700), rng.standard_normal((3, 700))
    for mode in codec.CONV_MODES:
        got = codec.fftconvolve(x2[0], h1, mode)                                  # numpy in, numpy out
        ref = scipy.signal.fftconvolve(x2[0], h1, mode)
        assert isinstance(got, np.ndarray) and got.dtype == np.float32 and got.shape == ref.shape
        assert rel(torch.from_numpy(got), torch.from_numpy(ref)) <= 1e-5
        got = codec.fftconvolve(x2, h1, mode)                                     # [B, N] x [M]: one shared IR
        ref = scipy.signal.fftconvolve(x2, h1[None], mode, axes=-1)
        assert got.shape == ref.shape and rel(torch.from_numpy(got), torch.from_numpy(ref)) <= 1e-5
        got = codec.fftconvolve(torch.from_numpy(x2).cuda(), torch.from_numpy(h2).cuda(), mode)   # [B, N] x [B, M], tensors
        ref = scipy.signal.fftconvolve(x2, h2, mode, axes=-1)
        assert torch.is_tensor(got) and got.is_cuda and tuple(got.shape) == ref.shape and rel(got, torch.from_numpy(ref)) <= 1e-5
        xs, hs = [x2[0][:100], x2[1], x2[2][:3000]], [h2[0], h2[1][:50], h2[2][:4000]]            # list in, list out
        got = codec.fftconvolve(xs, hs, mode)
        assert isinstance(got, list) and len(got) == 3
        for g, x, h in zip(got, xs, hs):
            ref = scipy.signal.fftconvolve(x, h, mode)
            assert isinstance(g, np.ndarray) and g.shape == ref.shape and rel(torch.from_numpy(g), torch.from_numpy(ref)) <= 1e-5


def _ir(M, channels=1, seed=7):
    rng = np.random.default_rng(seed)
    ir = rng.standard_normal((channels, M)) * np.exp(-np.arange(M) / (M / 6))
    return (0.3 * ir).astype(np.float32)


def test_reverb_arrangement_issues_fixed_library_calls():
    """Everything render_arrangement(impulse_response=...) does after synthesis, whatever the number of tracks, notes and items, is
    one pitch shift, two mixes and one convolution with their workspace queries.  Synthesis is replaced by random waveforms."""
    from diffusynth_b200 import TextToTimbre
    rng = np.random.default_rng(2)
    pipe = TextToTimbre.__new__(TextToTimbre)
    pipe.channels, pipe.height = 4, 128

    def fake_rows(latents, conditions, widths, *rest):
        return [Timbres(None, None, None, torch.from_numpy(rng.standard_normal((1, 256 * (4 * w - 1))).astype(np.float32)).cuda())
                for w in widths]
    pipe._synthesize_rows = fake_rows
    lat, cond = torch.zeros(1, 4, 128, 64), torch.zeros(1, 512)
    ir = torch.from_numpy(_ir(4800, 2)).cuda()
    counts = []
    for n_tracks, n_notes in ((1, 3), (4, 30)):
        tracks = [(lat, cond, [(float(o), float(d), int(s), 0.5) for o, d, s in
                               zip(rng.uniform(0, 10, n_notes), rng.choice([0.5, 1.0, 2.0], n_notes), rng.integers(-12, 13, n_notes))],
                   1.0, 0.05, float(rng.uniform(-1, 1))) for _ in range(n_tracks)]
        real = _lib.load()
        proxy = _counting(real)
        _lib._lib = proxy
        try:
            out = pipe.render_arrangement(tracks, target_peak=0.9, stereo=True, impulse_response=ir,
                                          reverb_sends=list(rng.uniform(0, 1, n_tracks)))
        finally:
            _lib._lib = real
        assert out.dim() == 2 and out.shape[0] == 2 and abs(float(out.abs().max()) - 0.9) < 1e-6
        counts.append(sorted(proxy.calls))
    print(f"\nreverb arrangement library calls: {counts[0]}")
    assert counts[0] == counts[1] == sorted(["ds_pitch_shift_workspace", "ds_pitch_shift", "ds_mix_stereo_workspace", "ds_mix_stereo",
                                             "ds_mix_stereo_workspace", "ds_mix_stereo", "ds_fftconvolve_workspace", "ds_fftconvolve"])


def test_render_arrangement_reverb_matches_oracle_and_dry_render():
    from diffusynth_b200 import TextToTimbre
    pipe = TextToTimbre.random_init(device="cuda", seed=0, batch_invariant=True)
    steps, M = 3, 8000
    conds, _ = W.synthetic_conditions(3, 512)
    insts = [cases.vq_latents(B=1, seed=22 + k) for k in range(3)]
    pans, sends = [-0.7, 0.0, 0.45], [0.2, 0.8, 0.0]
    tracks = [(insts[k].cuda(), conds[k:k + 1].cuda(), notes, gain, fade, pans[k]) for k, (notes, gain, fade) in enumerate(A.HAND_NOTES)]
    plan = TextToTimbre.arrangement_plan(tracks, reverb_sends=sends)
    feeds = [W.host_noise(70 + r, 1 + steps, 1) for r in range(len(plan.rows))]
    track_feeds = [[feeds[r] for r, (k, _) in enumerate(plan.rows) if k == t] for t in range(3)]
    waves = []
    for t in range(3):
        durs = [d for k, d in plan.rows if k == t]
        ts = pipe.synthesize_notes(tracks[t][0], tracks[t][1], durs, sample_steps=steps, noise_feeds=track_feeds[t])
        waves += [x.waveforms[0].cpu().numpy().astype(np.float64) for x in ts]
    ir1, ir2 = _ir(M, 1), _ir(M, 2, seed=8)
    mono_tracks = [t[:5] for t in tracks]
    for stereo, ir, peak in ((False, ir1[0], 0.7), (False, ir1[0], None), (True, ir1[0], None), (True, ir2, 0.7), (True, ir2, None)):
        out = pipe.render_arrangement(tracks if stereo else mono_tracks, sample_steps=steps, target_peak=peak, noise_feeds=feeds,
                                      stereo=stereo, impulse_response=ir, reverb_sends=sends)
        want_shape = (2, plan.track_len + M - 1) if stereo else (plan.track_len + M - 1,)
        assert tuple(out.shape) == want_shape and out.dtype == torch.float32 and out.is_cuda
        ref = RV.render(waves, plan, ir, stereo, target_peak=peak)
        errs = [rel(out[c], torch.from_numpy(ref[c])) for c in (0, 1)] if stereo else [rel(out, torch.from_numpy(ref))]
        print(f"\nrender_arrangement reverb stereo={stereo} ir={tuple(np.shape(ir))} peak={peak}: rel-L2 vs oracle "
              + " ".join(f"{e:.2e}" for e in errs))
        assert max(errs) <= 1e-4
        if peak is not None:
            assert abs(float(out.abs().max()) - peak) <= 2 * np.spacing(np.float32(peak))
    # all sends 0: the reverb-free render, zero-extended by M - 1, bit for bit
    for stereo, peak in ((False, 0.7), (True, None), (True, 0.7)):
        ts = tracks if stereo else mono_tracks
        dry = pipe.render_arrangement(ts, sample_steps=steps, target_peak=peak, noise_feeds=feeds, stereo=stereo)
        wet = pipe.render_arrangement(ts, sample_steps=steps, target_peak=peak, noise_feeds=feeds, stereo=stereo,
                                      impulse_response=torch.from_numpy(ir2 if stereo else ir1[0]).cuda(), reverb_sends=[0.0] * 3)
        L = plan.track_len
        assert torch.equal(wet[..., :L], dry) and not wet[..., L:].any()
