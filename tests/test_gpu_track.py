"""Note arrangements on the GPU: the batched pitch shift (ds_pitch_shift) stage by stage and end to end against the float64 oracle
(tests/pitch_oracle.py), the track mix (ds_mix_track), and TextToTimbre.render_track."""
import numpy as np
import pytest
import torch

from diffusynth_b200 import _lib, codec, weights as W
from oracle import cases, ds_oracle as O
from tests import pitch_oracle as P
from tests.gpu_util import rel

pytestmark = pytest.mark.gpu

SR = 16000
WIDTHS = [30, 48, 64]
STEPS = [-24, -12, -7, -0.5, 0, 5, 12]


def _signals():
    """A ragged batch: one item per n_steps, lengths 256 * (4W - 1) for W cycling through 30, 48, 64."""
    rng = np.random.default_rng(5)
    out = []
    for i in range(len(STEPS)):
        L = 256 * (4 * WIDTHS[i % 3] - 1)
        t = np.arange(L) / SR
        y = sum(a * np.sin(2 * np.pi * f * t + p) for a, f, p in zip(rng.uniform(0.2, 1, 3), rng.uniform(100, 2000, 3), rng.uniform(0, 6, 3)))
        y = y * np.exp(-t) + 0.05 * rng.standard_normal(L)
        out.append(y.astype(np.float32))
    return out


def crel(a, b):
    """rel-L2 of complex (or real) numpy arrays."""
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def _tone(L, f=440.0):
    t = np.arange(L) / SR
    return (np.sin(2 * np.pi * f * t) * np.exp(-t)).astype(np.float32)


def test_pitch_shift_stages_and_chain_against_oracle():
    ys = _signals()
    lengths = [len(y) for y in ys]
    stages = {}
    out = codec.pitch_shift_packed(torch.from_numpy(np.concatenate(ys)).cuda(), lengths, STEPS, stages=stages).cpu().numpy()
    ws = stages["workspace"].cpu()
    oD, oS, _, oY = stages["offsets"]
    fin = fout = yo = lo = 0
    worst = {}
    for y, n, L in zip(ys, STEPS, lengths):
        rate = 2.0 ** (-n / 12)
        T_in = 1 + L // 512
        T_out = len(np.arange(0, T_in, rate))
        n_ys = int(round(L / rate))
        D = torch.view_as_complex(ws[oD:].view(torch.float32)[2 * 1025 * fin:2 * 1025 * (fin + T_in)].view(T_in, 1025, 2)).numpy().T
        S = torch.view_as_complex(ws[oS:].view(torch.float32)[2 * 1025 * fout:2 * 1025 * (fout + T_out)].view(T_out, 1025, 2)).numpy().T
        ysg = ws[oY:].view(torch.float32)[yo:yo + n_ys].numpy().astype(np.float64)
        D64, S64 = D.astype(np.complex128), S.astype(np.complex128)
        e = dict(stft=crel(D64, O.stft(y.astype(np.float64), 2048, 512)),
                 vocoder=crel(S64, P.phase_vocoder(D64, rate, 512)),
                 istft=crel(ysg, P.istft_length(S64, 512, n_ys)))
        res = ysg if rate == 1.0 else P.resample_kaiser(ysg, rate)
        got = out[lo:lo + L].astype(np.float64)
        e["resample"] = crel(got, P.fix_length(res, L))
        e["chain"] = crel(got, P.pitch_shift(y.astype(np.float64), n))
        print(f"\nn_steps {n:+.1f} (L {L}): " + "  ".join(f"{k} {v:.2e}" for k, v in e.items()))
        for k, v in e.items():
            worst[k] = max(worst.get(k, 0.0), v)
        fin, fout, yo, lo = fin + T_in, fout + T_out, yo + n_ys, lo + L
    assert worst["stft"] <= 1e-5 and worst["istft"] <= 1e-5, worst
    assert worst["vocoder"] <= 1e-4 and worst["resample"] <= 1e-5, worst
    assert worst["chain"] <= 1e-4, worst


def test_batched_items_equal_items_shifted_alone():
    ys = [torch.from_numpy(y).cuda() for y in _signals()]
    batch = codec.pitch_shift(ys, STEPS)
    assert [b.numel() for b in batch] == [y.numel() for y in ys]
    for k in (0, 3, 4, 6):
        alone = codec.pitch_shift([ys[k]], STEPS[k])[0]
        assert torch.equal(alone, batch[k]), k
    same = torch.stack([ys[1], ys[4]])                        # a [B, L] tensor in, a [B, L] tensor out
    two = codec.pitch_shift(same, [STEPS[1], STEPS[4]])
    assert tuple(two.shape) == tuple(same.shape) and torch.equal(two[0], batch[1]) and torch.equal(two[1], batch[4])


def test_pitch_shift_moves_a_tone_on_device():
    L = 256 * (4 * 48 - 1)
    ns = [-12, -7, 5, 12]
    z = codec.pitch_shift(np.stack([_tone(L)] * len(ns)), ns)            # numpy in, numpy out
    assert isinstance(z, np.ndarray) and z.shape == (len(ns), L)
    for n, zk in zip(ns, z):
        peak = np.argmax(np.abs(np.fft.rfft(zk.astype(np.float64) * np.hanning(L)))) * SR / L
        assert abs(peak - 440.0 * 2 ** (n / 12)) <= SR / L, (n, peak)
    one = codec.pitch_shift(_tone(L), 0.0)                                  # 1-D drop-in of librosa.effects.pitch_shift(y, ...)
    assert one.shape == (L,) and rel(torch.from_numpy(one), torch.from_numpy(_tone(L))) < 1e-5


def test_mix_against_oracle_and_deterministic():
    rng = np.random.default_rng(9)
    srcs = [rng.standard_normal(n).astype(np.float32) for n in (30464, 48896, 65280, 1000)]
    note_src = [0, 1, 2, 3, 0, 1, 1, 2, 3, 0, 2, 2]
    onsets = [int(v) for v in rng.integers(0, 60000, len(note_src))]
    onsets[3] = 1023                                           # straddles a tile boundary
    gains = rng.uniform(-1, 1, len(note_src)).astype(np.float32)
    lengths = [len(s) for s in srcs]
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]])
    packed = torch.from_numpy(np.concatenate(srcs)).cuda()
    args = (packed, starts[note_src], np.asarray(lengths)[note_src], onsets, gains)
    a, b = codec.mix_track(*args), codec.mix_track(*args)
    ref = P.mix_track([srcs[i].astype(np.float64) for i in note_src], onsets, gains.astype(np.float64))
    e = rel(a, torch.from_numpy(ref))
    print(f"\nmix: {len(note_src)} notes, {a.numel()} samples, rel-L2 {e:.2e}")
    assert a.numel() == len(ref) and e <= 1e-5
    assert torch.equal(a, b)
    longer = codec.mix_track(*args, track_len=len(ref) + 5000)            # past the last note: silence
    assert torch.equal(longer[:len(ref)], a) and not longer[len(ref):].any()


def _counting(lib):
    class Counting:
        def __init__(self):
            self.calls = []

        def __getattr__(self, name):
            fn = getattr(lib, name)
            if not name.startswith("ds_"):
                return fn

            def wrapped(*a):
                self.calls.append(name)
                return fn(*a)
            return wrapped
    return Counting()


def test_pitch_and_mix_stage_issues_fixed_library_calls():
    rng = np.random.default_rng(2)
    counts = []
    for n_src, n_notes in ((3, 6), (10, 40)):
        srcs = [torch.from_numpy(rng.standard_normal(256 * (4 * WIDTHS[i % 3] - 1)).astype(np.float32)).cuda() for i in range(n_src)]
        semis = [float(s) for s in rng.integers(-12, 13, n_src)]
        note_src = [i % n_src for i in range(n_notes)]
        onsets = [int(v) for v in rng.integers(0, 100000, n_notes)]
        real = _lib.load()
        proxy = _counting(real)
        _lib._lib = proxy
        try:
            codec.shift_and_mix(srcs, semis, note_src, onsets, [0.5] * n_notes)
        finally:
            _lib._lib = real
        counts.append(sorted(proxy.calls))
    print(f"\npitch/mix library calls: {counts[0]}")
    assert counts[0] == counts[1] == sorted(["ds_pitch_shift_workspace", "ds_pitch_shift", "ds_mix_track_workspace", "ds_mix_track"])


def test_render_track_matches_oracle_shift_and_mix():
    from diffusynth_b200 import TextToTimbre
    pipe = TextToTimbre.random_init(device="cuda", seed=0, batch_invariant=True)
    steps = 3
    notes = [(0.0, 0.9, 0, 1.0), (0.4, 2.0, -5, 0.6), (0.8, 0.9, 7, 0.8), (1.1, 3.0, 12, 0.5), (1.5, 2.0, -5, 0.9), (2.0, 0.9, -12, 0.7)]
    plan = TextToTimbre.track_plan(notes)
    assert len(plan.durations) == 3 and len(plan.pairs) == 5                  # (2.0, -5) repeats
    feeds = [W.host_noise(60 + i, 1 + steps, 1) for i in range(len(plan.durations))]
    cond, _ = W.synthetic_conditions(1, 512)
    inst = cases.vq_latents(B=1, seed=22)
    track = pipe.render_track(inst.cuda(), cond.cuda(), notes, sample_steps=steps, noise_feeds=feeds)
    n_graphs = sum(len(s._graphs) for k, s in pipe._samplers.items() if k[0] == "note")
    assert n_graphs == len({TextToTimbre.note_width(d) for d in plan.durations}) == 3
    assert tuple(track.shape) == (plan.track_len,) and track.dtype == torch.float32 and track.is_cuda
    timbres = pipe.synthesize_notes(inst.cuda(), cond.cuda(), plan.durations, sample_steps=steps, noise_feeds=feeds)
    waves = [t.waveforms[0].cpu().numpy().astype(np.float64) for t in timbres]
    shifted = [P.pitch_shift(waves[d], s) for d, s in plan.pairs]
    ref = P.mix_track([shifted[p] for p in plan.note_pair], plan.onsets, plan.gains)
    e = rel(track, torch.from_numpy(ref))
    print(f"\nrender_track: {len(notes)} notes, {len(plan.pairs)} pitch-shifted pairs, {track.numel()} samples, rel-L2 vs oracle {e:.2e}")
    assert e <= 1e-4
