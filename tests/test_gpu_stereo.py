"""Stereo arrangements on the GPU: the stereo mix (ds_mix_stereo) against the float64 oracle (tests/stereo_oracle.py), its shared
peak normalisation, its bit-exact relations to the mono arrangement mix and between mirrored pans, and
TextToTimbre.render_arrangement(stereo=True) against the oracle chain and the mono render."""
import numpy as np
import pytest
import torch

from diffusynth_b200 import _lib, codec, weights as W
from diffusynth_b200.pipeline import Timbres
from oracle import cases
from tests import arrangement_oracle as A
from tests import stereo_oracle as S
from tests.gpu_util import rel
from tests.test_gpu_arrangement import _note_graphs, _notes
from tests.test_gpu_track import _counting

pytestmark = pytest.mark.gpu


def _pans(n, seed=5):
    """Mixed pans: uniform in [-1, 1], with hard left, centre and hard right among them."""
    p = np.random.default_rng(seed).uniform(-1, 1, n).astype(np.float32)
    p[0], p[1], p[2], p[5] = -1.0, 0.0, 1.0, -1.0
    return p


def test_mix_stereo_against_oracle_and_deterministic():
    packed, offs, lengths, onsets, gains, fades, waves = _notes()
    pans = _pans(len(lengths))
    a = codec.mix_stereo(packed, offs, lengths, onsets, gains, pans, fades)
    b = codec.mix_stereo(packed, offs, lengths, onsets, gains, pans, fades)
    ref = S.mix_stereo(waves, onsets, gains.astype(np.float64), pans.astype(np.float64), fades)
    assert tuple(a.shape) == ref.shape and a.dtype == torch.float32 and a.is_contiguous()
    errs = [rel(a[c], torch.from_numpy(ref[c])) for c in (0, 1)]
    print(f"\nmix_stereo: {len(lengths)} notes, {a.shape[1]} samples, rel-L2 vs oracle L {errs[0]:.2e} R {errs[1]:.2e}")
    assert max(errs) <= 1e-6
    assert torch.equal(a, b)


def test_shared_peak_normalisation():
    packed, offs, lengths, onsets, gains, fades, waves = _notes(seed=11)
    pans = _pans(len(lengths), seed=6)
    raw = codec.mix_stereo(packed, offs, lengths, onsets, gains, pans, fades)
    for peak in (0.8, 3.0):
        a = codec.mix_stereo(packed, offs, lengths, onsets, gains, pans, fades, target_peak=peak)
        b = codec.mix_stereo(packed, offs, lengths, onsets, gains, pans, fades, target_peak=peak)
        ref = S.mix_stereo(waves, onsets, gains.astype(np.float64), pans.astype(np.float64), fades, target_peak=peak)
        top = float(a.abs().max())
        errs = [rel(a[c], torch.from_numpy(ref[c])) for c in (0, 1)]
        print(f"\npeak {peak}: max(|L|, |R|) {top!r}, rel-L2 vs oracle L {errs[0]:.2e} R {errs[1]:.2e}")
        assert abs(top - peak) <= 2 * np.spacing(np.float32(peak)) and max(errs) <= 1e-6
        assert torch.equal(a, b)
        # one common factor for both channels: the unnormalised mix times fl32(peak / max|raw|), to fp32 rounding
        sc = np.float32(peak) / np.float32(raw.abs().max().item())
        want = (raw * float(sc)).cpu()
        assert ((a.cpu() - want).abs() <= torch.from_numpy(np.spacing(want.abs().numpy()))).all()
    zero = codec.mix_stereo(torch.zeros(5000, device="cuda"), [0, 1000], [3000, 4000], [0, 2500], [1.0, 0.5], [0.3, -1.0], [100, 0],
                            target_peak=0.9)
    assert tuple(zero.shape) == (2, 6500) and not zero.any()


def _positive_zero(x):
    return bool((x.view(torch.int32) == 0).all())


def test_bit_exact_relations():
    packed, offs, lengths, onsets, gains, fades, _ = _notes(seed=3)
    K = len(lengths)
    for f, peak in ((fades, None), ([0] * K, None), (fades, 0.9), ([0] * K, 1.5)):
        mono = codec.mix_arrangement(packed, offs, lengths, onsets, gains, f, target_peak=peak)
        left = codec.mix_stereo(packed, offs, lengths, onsets, gains, [-1.0] * K, f, target_peak=peak)
        assert torch.equal(left[0], mono) and _positive_zero(left[1])                       # hard left: the mono mix and +0
        right = codec.mix_stereo(packed, offs, lengths, onsets, gains, [1.0] * K, f, target_peak=peak)
        assert torch.equal(right[1], mono) and _positive_zero(right[0])
        p = _pans(K, seed=8)
        a = codec.mix_stereo(packed, offs, lengths, onsets, gains, p, f, target_peak=peak)
        m = codec.mix_stereo(packed, offs, lengths, onsets, gains, -p, f, target_peak=peak)
        assert torch.equal(a, m.flip(0))                                                     # mirrored pans swap the channels
        c = codec.mix_stereo(packed, offs, lengths, onsets, gains, [0.0] * K, f, target_peak=peak)
        assert torch.equal(c[0], c[1])                                                       # centre: L == R
    # shift_and_mix with pans mixes through ds_mix_stereo
    srcs = [packed[:1000], packed[1000:4000]]
    st = codec.shift_and_mix(srcs, [0.0, 3.0], [0, 1, 0], [0, 500, 2000], [1.0, 0.5, -0.25], fades=[0, 100, 0], pans=[-1.0, -1.0, -1.0])
    mono = codec.shift_and_mix(srcs, [0.0, 3.0], [0, 1, 0], [0, 500, 2000], [1.0, 0.5, -0.25], fades=[0, 100, 0])
    assert tuple(st.shape) == (2, mono.numel()) and torch.equal(st[0], mono) and _positive_zero(st[1])


def test_stereo_arrangement_issues_fixed_library_calls():
    """Everything render_arrangement(stereo=True) does after synthesis, whatever the number of tracks, notes and items, is one pitch
    shift and one stereo mix with their workspace queries.  Synthesis is replaced by random waveforms of the rows' widths."""
    from diffusynth_b200 import TextToTimbre
    rng = np.random.default_rng(2)
    pipe = TextToTimbre.__new__(TextToTimbre)
    pipe.channels, pipe.height = 4, 128

    def fake_rows(latents, conditions, widths, *rest):
        return [Timbres(None, None, None, torch.from_numpy(rng.standard_normal((1, 256 * (4 * w - 1))).astype(np.float32)).cuda())
                for w in widths]
    pipe._synthesize_rows = fake_rows
    lat, cond = torch.zeros(1, 4, 128, 64), torch.zeros(1, 512)
    counts = []
    for n_tracks, n_notes in ((1, 3), (4, 30)):
        tracks = [(lat, cond, [(float(o), float(d), int(s), 0.5) for o, d, s in
                               zip(rng.uniform(0, 10, n_notes), rng.choice([0.5, 1.0, 2.0], n_notes), rng.integers(-12, 13, n_notes))],
                   1.0, 0.05, float(rng.uniform(-1, 1))) for _ in range(n_tracks)]
        real = _lib.load()
        proxy = _counting(real)
        _lib._lib = proxy
        try:
            out = pipe.render_arrangement(tracks, target_peak=0.9, stereo=True)
        finally:
            _lib._lib = real
        assert out.dim() == 2 and out.shape[0] == 2 and abs(float(out.abs().max()) - 0.9) < 1e-6
        counts.append(sorted(proxy.calls))
    print(f"\nstereo arrangement library calls: {counts[0]}")
    assert counts[0] == counts[1] == sorted(["ds_pitch_shift_workspace", "ds_pitch_shift", "ds_mix_stereo_workspace", "ds_mix_stereo"])


def test_render_arrangement_stereo_matches_oracle_and_mono():
    from diffusynth_b200 import TextToTimbre
    pipe = TextToTimbre.random_init(device="cuda", seed=0, batch_invariant=True)
    steps, peak = 3, 0.7
    conds, _ = W.synthetic_conditions(3, 512)
    insts = [cases.vq_latents(B=1, seed=22 + k) for k in range(3)]
    pans = [-0.7, 0.0, 0.45]
    tracks = [(insts[k].cuda(), conds[k:k + 1].cuda(), notes, gain, fade, pans[k]) for k, (notes, gain, fade) in enumerate(A.HAND_NOTES)]
    plan = TextToTimbre.arrangement_plan(tracks)
    feeds = [W.host_noise(70 + r, 1 + steps, 1) for r in range(len(plan.rows))]
    track_feeds = [[feeds[r] for r, (k, _) in enumerate(plan.rows) if k == t] for t in range(3)]

    out = pipe.render_arrangement(tracks, sample_steps=steps, target_peak=peak, noise_feeds=feeds, stereo=True)
    assert _note_graphs(pipe) == len(set(plan.widths)) == 3
    assert tuple(out.shape) == (2, plan.track_len) and out.dtype == torch.float32 and out.is_cuda

    waves = []
    for t in range(3):
        durs = [d for k, d in plan.rows if k == t]
        ts = pipe.synthesize_notes(tracks[t][0], tracks[t][1], durs, sample_steps=steps, noise_feeds=track_feeds[t])
        waves += [x.waveforms[0].cpu().numpy().astype(np.float64) for x in ts]
    ref = S.render(waves, plan, target_peak=peak)
    errs = [rel(out[c], torch.from_numpy(ref[c])) for c in (0, 1)]
    print(f"\nrender_arrangement(stereo): 3 tracks, {len(plan.note_item)} notes, {out.shape[1]} samples, rel-L2 vs oracle "
          f"L {errs[0]:.2e} R {errs[1]:.2e}, max(|L|, |R|) {float(out.abs().max())!r}")
    assert max(errs) <= 1e-4
    assert abs(float(out.abs().max()) - peak) <= 2 * np.spacing(np.float32(peak))

    # every track hard left: the left channel is the mono render bit for bit, the right channel +0
    left = pipe.render_arrangement([t[:5] + (-1.0,) for t in tracks], sample_steps=steps, target_peak=peak, noise_feeds=feeds,
                                   stereo=True)
    mono = pipe.render_arrangement([t[:5] for t in tracks], sample_steps=steps, target_peak=peak, noise_feeds=feeds)
    assert torch.equal(left[0], mono) and _positive_zero(left[1])
    # 5-tuple tracks in stereo are centred
    centred = pipe.render_arrangement([t[:5] for t in tracks], sample_steps=steps, noise_feeds=feeds, stereo=True)
    assert torch.equal(centred[0], centred[1])
