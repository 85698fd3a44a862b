"""Multi-instrument arrangements on the GPU: the arrangement mix (ds_mix_arrangement) against the float64 oracle
(tests/arrangement_oracle.py), bit for bit against ds_mix_track without fades, its peak normalisation, and
TextToTimbre.render_arrangement against the oracle chain and against render_track."""
import numpy as np
import pytest
import torch

from diffusynth_b200 import _lib, codec, weights as W
from diffusynth_b200.pipeline import Timbres
from oracle import cases
from tests import arrangement_oracle as A
from tests.gpu_util import rel
from tests.test_gpu_track import _counting

pytestmark = pytest.mark.gpu


def _notes(seed=9, n_notes=40):
    """A ragged mix: 5 sources of note lengths (one shorter than a mix tile), notes straddling tile boundaries, mixed signs of gain,
    and fades of 0, shorter than, equal to and longer than the note."""
    rng = np.random.default_rng(seed)
    srcs = [rng.standard_normal(n).astype(np.float32) for n in (30464, 48896, 65280, 1000, 7777)]
    note_src = [int(v) for v in rng.integers(0, len(srcs), n_notes)]
    lengths = [len(srcs[i]) for i in note_src]
    onsets = [int(v) for v in rng.integers(0, 200000, n_notes)]
    onsets[1] = 1023
    gains = rng.uniform(-1, 1, n_notes).astype(np.float32)
    fades = [int(v) for v in rng.integers(1, 20000, n_notes)]
    for k in range(0, n_notes, 4):
        fades[k] = 0
    fades[2], fades[3] = lengths[2], 10 * lengths[3]
    starts = np.concatenate([[0], np.cumsum([len(s) for s in srcs])[:-1]])
    packed = torch.from_numpy(np.concatenate(srcs)).cuda()
    waves = [srcs[i].astype(np.float64) for i in note_src]
    return packed, starts[note_src], lengths, onsets, gains, fades, waves


def test_mix_arrangement_against_oracle_and_deterministic():
    packed, offs, lengths, onsets, gains, fades, waves = _notes()
    a = codec.mix_arrangement(packed, offs, lengths, onsets, gains, fades)
    b = codec.mix_arrangement(packed, offs, lengths, onsets, gains, fades)
    ref = A.mix_arrangement(waves, onsets, gains.astype(np.float64), fades)
    e = rel(a, torch.from_numpy(ref))
    print(f"\nmix_arrangement: {len(lengths)} notes, {a.numel()} samples, rel-L2 vs oracle {e:.2e}")
    assert a.numel() == len(ref) and e <= 1e-6
    assert torch.equal(a, b)


def test_fade_free_mix_is_mix_track_bit_for_bit():
    packed, offs, lengths, onsets, gains, _, _ = _notes(seed=3)
    plain = codec.mix_track(packed, offs, lengths, onsets, gains)
    arr = codec.mix_arrangement(packed, offs, lengths, onsets, gains, [0] * len(lengths))
    assert torch.equal(arr, plain)
    longer = codec.mix_arrangement(packed, offs, lengths, onsets, gains, [0] * len(lengths), track_len=plain.numel() + 3000)
    assert torch.equal(longer, codec.mix_track(packed, offs, lengths, onsets, gains, track_len=plain.numel() + 3000))


def test_peak_normalisation():
    packed, offs, lengths, onsets, gains, fades, waves = _notes(seed=11)
    for peak in (0.8, 3.0):
        a = codec.mix_arrangement(packed, offs, lengths, onsets, gains, fades, target_peak=peak)
        b = codec.mix_arrangement(packed, offs, lengths, onsets, gains, fades, target_peak=peak)
        ref = A.mix_arrangement(waves, onsets, gains.astype(np.float64), fades, target_peak=peak)
        top = float(a.abs().max())
        e = rel(a, torch.from_numpy(ref))
        print(f"\npeak {peak}: max|track| {top!r}, rel-L2 vs oracle {e:.2e}")
        assert abs(top - peak) <= 2 * np.spacing(np.float32(peak)) and e <= 1e-6
        assert torch.equal(a, b)
    zero = codec.mix_arrangement(torch.zeros(5000, device="cuda"), [0, 1000], [3000, 4000], [0, 2500], [1.0, 0.5], [100, 0],
                                 target_peak=0.9)
    assert zero.numel() == 6500 and not zero.any()


def test_arrangement_issues_fixed_library_calls():
    """Everything render_arrangement does after synthesis -- whatever the number of tracks, notes and items -- is one pitch shift
    and one arrangement mix with their workspace queries.  Synthesis is replaced by random waveforms of the rows' widths."""
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
                   1.0, 0.05) for _ in range(n_tracks)]
        real = _lib.load()
        proxy = _counting(real)
        _lib._lib = proxy
        try:
            out = pipe.render_arrangement(tracks, target_peak=0.9)
        finally:
            _lib._lib = real
        assert abs(float(out.abs().max()) - 0.9) < 1e-6
        counts.append(sorted(proxy.calls))
    print(f"\narrangement library calls: {counts[0]}")
    assert counts[0] == counts[1] == sorted(["ds_pitch_shift_workspace", "ds_pitch_shift", "ds_mix_arrangement_workspace",
                                             "ds_mix_arrangement"])


def _note_graphs(pipe):
    return sum(len(s._graphs) for k, s in pipe._samplers.items() if k[0] == "note")


def test_render_arrangement_matches_oracle_and_render_track():
    from diffusynth_b200 import TextToTimbre
    pipe = TextToTimbre.random_init(device="cuda", seed=0, batch_invariant=True)
    steps, peak = 3, 0.7
    conds, _ = W.synthetic_conditions(3, 512)
    insts = [cases.vq_latents(B=1, seed=22 + k) for k in range(3)]
    tracks = [(insts[k].cuda(), conds[k:k + 1].cuda(), notes, gain, fade) for k, (notes, gain, fade) in enumerate(A.HAND_NOTES)]
    plan = TextToTimbre.arrangement_plan(tracks)
    feeds = [W.host_noise(70 + r, 1 + steps, 1) for r in range(len(plan.rows))]
    track_feeds = [[feeds[r] for r, (k, _) in enumerate(plan.rows) if k == t] for t in range(3)]

    out = pipe.render_arrangement(tracks, sample_steps=steps, target_peak=peak, noise_feeds=feeds)
    per_track_widths = sum(len({TextToTimbre.note_width(d) for _, d, _, _ in notes}) for notes, _, _ in A.HAND_NOTES)
    assert _note_graphs(pipe) == len(set(plan.widths)) == 3 < per_track_widths == 5      # one launch per width across tracks
    assert tuple(out.shape) == (plan.track_len,) and out.dtype == torch.float32 and out.is_cuda

    # the oracle chain from each track's synthesize_notes waveforms (rows of a track are its durations in order)
    waves = []
    for t in range(3):
        durs = [d for k, d in plan.rows if k == t]
        ts = pipe.synthesize_notes(tracks[t][0], tracks[t][1], durs, sample_steps=steps, noise_feeds=track_feeds[t])
        waves += [x.waveforms[0].cpu().numpy().astype(np.float64) for x in ts]
    ref = A.render(waves, plan, target_peak=peak)
    e = rel(out, torch.from_numpy(ref))
    print(f"\nrender_arrangement: 3 tracks, {len(plan.note_item)} notes, {len(plan.items)} pitch items, {out.numel()} samples, "
          f"rel-L2 vs oracle {e:.2e}, max|x| {float(out.abs().max())!r}")
    assert e <= 1e-4
    assert abs(float(out.abs().max()) - peak) <= 2 * np.spacing(np.float32(peak))

    # one track, gain 1, no fade, no peak: render_track's output bit for bit
    notes0 = A.HAND_NOTES[0][0]
    one = pipe.render_arrangement([(tracks[0][0], tracks[0][1], notes0, 1.0, 0.0)], sample_steps=steps, noise_feeds=track_feeds[0])
    alone = [pipe.render_track(tracks[t][0], tracks[t][1], A.HAND_NOTES[t][0], sample_steps=steps, noise_feeds=track_feeds[t])
             for t in range(3)]
    assert torch.equal(one, alone[0])

    # three tracks, gains 1, no fades: the sum of the three render_track outputs (summed in another order)
    flat = [(lat, cond, notes, 1.0, 0.0) for lat, cond, notes, _, _ in tracks]
    mix = pipe.render_arrangement(flat, sample_steps=steps, noise_feeds=feeds)
    total = torch.zeros_like(mix)
    for x in alone:
        total[:x.numel()] += x
    e_sum = rel(mix, total)
    print(f"3 tracks vs the sum of 3 render_track outputs: rel-L2 {e_sum:.2e}, max |diff| {float((mix - total).abs().max()):.2e}")
    assert e_sum <= 1e-6

