"""Clip queue over the sampler (inference.infer_coeffs_queue / infer_coeffs_many) and the per-clip Philox noise keys
(msmd_sample_extras.noise_keys) it relies on.

CPU: the windowing helper, the scheduler driven by a stub model, argument validation and the C struct layout.
GPU: keys vs the noise_clip_offset path, the queue vs each clip sampled alone, the audio wrapper."""
import ctypes
import math
import os
import shutil
import subprocess
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT, rel_l2

L, LP = 100, 10


# ---------------------------------------------------------------------------------------------------------- fixtures
class StubModel:
    """Stands in for MSMD in the host loop: a deterministic per-row function of every input the sampler sees (audio,
    previous motion / audio, x_T, indicator, shape, style and the noise key), recording the (clip id, seed) per call."""

    def __init__(self, d=8):
        g = torch.Generator().manual_seed(0)
        self.device = torch.device('cpu')
        self.start_motion_feat = torch.randn(1, LP, 67, generator=g)
        self.start_audio_feat = torch.randn(1, LP, d, generator=g)
        self.calls = []

    def sample(self, audio, shape, style, prev_motion, prev_audio, motion_at_T, indicator=None, noise_seed=None,
               clip_offset=0, noise_keys=None, **kw):
        N = audio.shape[0]
        if prev_motion is None:
            prev_motion = self.start_motion_feat.expand(N, -1, -1)
        if prev_audio is None:
            prev_audio = self.start_audio_feat.expand(N, -1, -1)
        if motion_at_T is None:
            motion_at_T = torch.zeros(N, L, 67)
        if noise_keys is None:
            noise_keys = torch.stack([torch.full((N,), int(noise_seed or 0)), clip_offset + torch.arange(N)], 1)
        self.calls.append([(int(i), int(s)) for s, i in noise_keys.tolist()])
        k = noise_keys.double()
        out = (motion_at_T + audio[..., :67].sum(-1, keepdim=True) + prev_motion[:, -1:] + prev_audio[:, :, :1].sum(1, keepdim=True)
               + shape.reshape(N, 1, -1)[..., :1] + style.reshape(N, 1, -1)[..., 1:2] + 0.5 * indicator[..., None]
               + (1e-3 * k[:, :1, None] + 1e-2 * k[:, 1:, None]).float())
        return out, motion_at_T, audio


def stub_args():
    return SimpleNamespace(n_motions=L, n_prev_motions=LP, use_indicator=True, fps=25)


def stub_clips(windows, pads, d=8):
    g = torch.Generator().manual_seed(5)
    feats = [torch.randn(w * L, d, generator=g) for w in windows]
    lens = [w * L - p for w, p in zip(windows, pads)]
    shape = torch.randn(len(windows), 100, generator=g)
    style = torch.randn(len(windows), 16, generator=g)
    x_T = torch.randn(len(windows), L, 67, generator=g)
    return feats, shape, style, lens, x_T


def reference_plan(n_samples, fps, n_motions, audio_unit):
    """inference.py:39-45 as the parent implementation of infer_coeffs wrote it."""
    clip_len = int(n_samples / 16000 * fps)
    n_audio_samples = round(audio_unit * n_motions)
    n_subdivision = 1 if clip_len <= n_motions else math.ceil(clip_len / n_motions)
    n_padding_audio_samples = n_audio_samples * n_subdivision - n_samples
    n_padding_frames = math.ceil(n_padding_audio_samples / audio_unit)
    padded = n_samples + n_padding_audio_samples if n_padding_audio_samples > 0 else n_samples
    return n_subdivision, padded, n_motions * n_subdivision - max(n_padding_frames, 0)


# --------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('audio_unit', [640.0, 633.3])
def test_plan_clip_matches_infer_coeffs_arithmetic(audio_unit):
    from msmd_b200.inference import plan_clip
    args = stub_args()
    one = round(audio_unit * L)
    lengths = [300, 16000, one - 1, one, one + 1,           # under one window, exactly L frames, just over
               one + 640, one + 641, 2 * one, 2 * one + 1,   # L + 1 frames, a window boundary
               64650, 127999, 320123, 959999]                # non-integer frame counts
    for n in lengths:
        assert plan_clip(n, args, audio_unit) == reference_plan(n, 25, L, audio_unit), n
    assert plan_clip(one, args, audio_unit)[0] == 1 and plan_clip(2 * one + 1, args, audio_unit)[0] in (2, 3)


def test_infer_coeffs_plans_through_the_helper():
    """infer_coeffs pads each clip to its own window count and keeps plan_clip's frames (stub encoder + sampler)."""
    from msmd_b200.inference import infer_coeffs
    m = StubModel(d=8)
    seen = []
    m.extract_audio_feature = lambda a, n: (seen.append(tuple(a.shape)), torch.zeros(a.shape[0], n, 8))[1]
    for n in (16000, 64000, 64640, 100100, 128000):
        want = reference_plan(n, 25, L, 640.0)
        out = infer_coeffs(m, stub_args(), torch.zeros(n), torch.zeros(1, 100), 640.0, torch.zeros(1, 16),
                           dynamic_threshold=None)
        assert out.shape == (1, want[2], 67) and seen[-1] == (1, want[1])


def test_queue_schedule_order_capacity_refill():
    from msmd_b200.inference import queue_schedule
    windows = [3, 1, 4, 1, 2, 2, 1]
    calls = queue_schedule(windows, 3)
    seen = [(k, w) for call in calls for k, w in call]
    assert sorted(seen) == sorted((k, w) for k, n in enumerate(windows) for w in range(n))
    done = set()
    for c, call in enumerate(calls):
        remaining = len(windows) - len(done)
        assert len(call) == min(3, remaining)                       # a finished clip's slot is refilled at once
        for k, w in call:
            assert w == 0 or (k, w - 1) in [x for prev in calls[:c] for x in prev]
        done |= {k for k, w in call if w == windows[k] - 1}
    assert [k for call in calls for k, w in call if w == 0] == list(range(len(windows)))   # admitted in order
    assert any({w == 0 for _, w in call} == {True, False} for call in calls)


def test_queue_matches_each_clip_alone_with_stub():
    """Every window of every clip runs exactly once and in order, at most max_clips in flight, windows mixed in one
    call, and each clip's codes equal infer_coeffs_batched on that clip alone with clip_offset = its id."""
    from msmd_b200.inference import infer_coeffs_batched, infer_coeffs_queue
    windows, pads = [3, 1, 4, 1, 2, 2, 1], [0, 30, 7, 0, 99, 0, 55]
    feats, shape, style, lens, x_T = stub_clips(windows, pads)
    ids = [11, 3, 40, 7, 1000, 5, 2]
    m = StubModel()
    codes, lengths = infer_coeffs_queue(m, stub_args(), feats, shape, style, lens, x_T, max_clips=3, clip_ids=ids,
                                        noise_seed=70)
    calls = m.calls
    assert lengths.tolist() == lens and codes.shape == (7, max(lens), 67)
    runs = [(i, s - 70) for call in calls for i, s in call]
    assert sorted(runs) == sorted((ids[k], w) for k, n in enumerate(windows) for w in range(n))
    for k, n in enumerate(windows):
        order = [w for i, w in runs if i == ids[k]]
        assert order == list(range(n))
    assert max(len(c) for c in calls) == 3
    assert any({s == 70 for _, s in call} == {True, False} for call in calls)
    for k in range(7):
        alone = infer_coeffs_batched(StubModel(), stub_args(), feats[k][None], shape[k:k + 1], style[k:k + 1],
                                     clip_len=lens[k], x_T=x_T[k:k + 1], noise_seed=70, clip_offset=ids[k])
        assert torch.allclose(codes[k, :lens[k]], alone[0], rtol=0, atol=1e-5), k
        assert not codes[k, lens[k]:].any()


def test_audio_batches_keep_encoder_capacity_within_budget():
    """extract_clip_features batches every padded length with one clip count: the encoder grows its workspace to
    (largest batch seen) x (longest clip seen), and that product stays within AUDIO_BATCH_SAMPLES over clips of 1-60 s.
    Each clip gets its own features back."""
    from msmd_b200 import inference as I
    g = torch.Generator().manual_seed(3)
    sizes = (16000 + torch.randint(0, 59 * 16000, (600,), generator=g)).tolist()
    audios = [torch.full((n,), float(k)) for k, n in enumerate(sizes)]
    seen = []

    def extract(wav, frames):
        seen.append(tuple(wav.shape))
        return wav[:, :1, None].expand(-1, frames, 4).clone()     # features = the clip's id

    m = SimpleNamespace(extract_audio_feature=extract)
    feats, lens = I.extract_clip_features(m, stub_args(), audios)
    assert max(n for n, _ in seen) * max(s for _, s in seen) <= I.AUDIO_BATCH_SAMPLES
    assert sum(n for n, _ in seen) == len(audios)
    for k, (f, n) in enumerate(zip(feats, sizes)):
        n_sub, padded, clip_len = I.plan_clip(n, stub_args(), 640.0)
        assert f.shape == (n_sub * L, 4) and bool((f == k).all()) and lens[k] == clip_len


def test_infer_coeffs_many_defaults_to_infer_coeffs_thresholding():
    from msmd_b200.inference import infer_coeffs_many
    m = StubModel(d=4)
    m.extract_audio_feature = lambda a, n: torch.zeros(a.shape[0], n, 4)
    got = []
    sample = m.sample
    m.sample = lambda *a, **kw: (got.append(kw.get('dynamic_threshold')), sample(*a, **kw))[1]
    audios = [torch.zeros(20000), torch.zeros(70000)]
    infer_coeffs_many(m, stub_args(), audios, torch.zeros(2, 100), torch.zeros(2, 16))
    assert got and all(d == (0, 1, 4) for d in got)
    got.clear()
    infer_coeffs_many(m, stub_args(), audios, torch.zeros(2, 100), torch.zeros(2, 16), dynamic_threshold=None)
    assert got and all(d is None for d in got)


def test_queue_argument_validation():
    from msmd_b200.inference import infer_coeffs_many, infer_coeffs_queue, queue_schedule
    feats, shape, style, lens, x_T = stub_clips([2, 1], [0, 10])
    args = stub_args()
    with pytest.raises(ValueError, match='no clips'):
        infer_coeffs_queue(StubModel(), args, [], [], None, [], [])
    with pytest.raises(ValueError, match='no clips'):
        infer_coeffs_many(StubModel(), args, [], [], None)
    with pytest.raises(ValueError, match='max_clips'):
        infer_coeffs_queue(StubModel(), args, feats, shape, style, lens, x_T, max_clips=0)
    with pytest.raises(ValueError, match='max_clips'):
        queue_schedule([1, 2], 0)
    with pytest.raises(ValueError):
        infer_coeffs_queue(StubModel(), args, feats, shape[:1], style, lens, x_T)
    with pytest.raises(ValueError):
        infer_coeffs_queue(StubModel(), args, feats, shape, style, lens[:1], x_T)
    with pytest.raises(ValueError):
        infer_coeffs_queue(StubModel(), args, feats, shape, style, lens, x_T, clip_ids=[0])
    with pytest.raises(ValueError, match='clip_len'):
        infer_coeffs_queue(StubModel(), args, feats, shape, style, [200, 101], x_T)
    with pytest.raises(ValueError, match='audio features'):
        infer_coeffs_queue(StubModel(), args, [feats[0][:150], feats[1]], shape, style, lens, x_T)


def test_sample_noise_keys_validation():
    """MSMD.sample checks noise_keys before any device work."""
    from helpers import make_msmd
    m, args = make_msmd('cpu', n_diff_steps=12)
    N = 2
    feat, shape, style = torch.zeros(N, L, 512), torch.zeros(N, 100), torch.zeros(N, 256)
    keys = torch.zeros(N, 2, dtype=torch.int64)
    for bad in (keys.int(), keys[:1], torch.zeros(N, 3, dtype=torch.int64), keys.float(), [[0, 0], [0, 1]]):
        with pytest.raises(ValueError, match='noise_keys'):
            m.sample(feat, shape, style, noise_keys=bad)
    for extra in (dict(noise=torch.zeros(13, N, L, 67)), dict(noise_seed=3), dict(clip_offset=4)):
        with pytest.raises(ValueError, match='noise_keys'):
            m.sample(feat, shape, style, noise_keys=keys, **extra)


def test_sample_extras_layout_matches_c_header(tmp_path):
    """ctypes' SampleExtras has the layout of msmd_sample_extras, noise_keys appended last."""
    from msmd_b200._engine import SampleExtras
    gcc = shutil.which('gcc')
    assert gcc, 'gcc is part of the image'
    src = tmp_path / 'layout.c'
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "msmd_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu\\n", sizeof(msmd_sample_extras), '
                   'offsetof(msmd_sample_extras, noise_clip_offset), offsetof(msmd_sample_extras, noise_keys)); return 0; }\n')
    exe = str(tmp_path / 'layout')
    subprocess.run([gcc, '-std=c99', '-Wall', '-Werror', '-I', os.path.join(ROOT, 'include'), str(src), '-o', exe], check=True)
    size, off_offset, off_keys = map(int, subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split())
    assert size == ctypes.sizeof(SampleExtras)
    assert off_offset == SampleExtras.noise_clip_offset.offset
    assert off_keys == SampleExtras.noise_keys.offset
    assert [f for f, _ in SampleExtras._fields_][-1] == 'noise_keys'


# --------------------------------------------------------------------------------------------------------------- GPU
T_SMALL = 12


def gpu_clips(windows, pads, seed=0, dev='cuda'):
    g = torch.Generator().manual_seed(seed)
    n = len(windows)
    feats = [torch.randn(w * L, 512, generator=g).to(dev) for w in windows]
    lens = [w * L - p for w, p in zip(windows, pads)]
    style = torch.randn(n, 256, generator=g).to(dev)
    shape = torch.zeros(n, 100, device=dev)
    x_T = torch.randn(n, L, 67, generator=g).to(dev)
    return feats, shape, style, lens, x_T


def alone(m, args, feats, shape, style, lens, x_T, k, seed, cid, **kw):
    from msmd_b200.inference import infer_coeffs_batched
    return infer_coeffs_batched(m, args, feats[k][None], shape[k:k + 1], style[k:k + 1], clip_len=lens[k], cfg_scale=1.4,
                                x_T=x_T[k:k + 1], noise_seed=seed, clip_offset=cid, **kw)[0]


@pytest.mark.gpu
def test_keys_equal_noise_clip_offset_path(built_lib):
    from helpers import make_msmd
    m, args = make_msmd('cuda', precision=None, n_diff_steps=T_SMALL)
    feats, shape, style, lens, x_T = gpu_clips([1] * 5, [0] * 5, seed=1)
    feat = torch.stack(feats)
    ind = torch.ones(5, L, device='cuda')
    a = m.sample(feat, shape, style, motion_at_T=x_T, indicator=ind, cfg_scale=1.4, noise_seed=123, clip_offset=9)[0]
    keys = torch.stack([torch.full((5,), 123), 9 + torch.arange(5)], 1).cuda()
    b = m.sample(feat, shape, style, motion_at_T=x_T, indicator=ind, cfg_scale=1.4, noise_keys=keys)[0]
    assert torch.isfinite(a).all() and torch.equal(a, b)


@pytest.mark.gpu
def test_per_clip_keys_equal_each_clip_alone(built_lib):
    """Different seeds and non-contiguous global ids in one call: each clip equals that clip sampled on its own."""
    from helpers import make_msmd
    m, args = make_msmd('cuda', precision=None, n_diff_steps=T_SMALL)
    feats, shape, style, lens, x_T = gpu_clips([1] * 4, [0] * 4, seed=2)
    feat = torch.stack(feats)
    ind = torch.ones(4, L, device='cuda')
    keys = [(7, 3), (11, 40), (7, 1000), (2 ** 40 + 3, 9)]
    got = m.sample(feat, shape, style, motion_at_T=x_T, indicator=ind, cfg_scale=1.4,
                   noise_keys=torch.tensor(keys, dtype=torch.int64, device='cuda'))[0]
    for n, (s, cid) in enumerate(keys):
        one = m.sample(feat[n:n + 1], shape[n:n + 1], style[n:n + 1], motion_at_T=x_T[n:n + 1], indicator=ind[:1],
                       cfg_scale=1.4, noise_seed=s, clip_offset=cid)[0]
        assert torch.equal(got[n], one[0]), n
    assert not torch.equal(got[0], got[2])


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['hybrid', 'fp32'])
def test_queue_equals_each_clip_alone(built_lib, precision):
    """7 clips of 1-4 windows (some with a padded last window), 3 in flight: every clip's codes equal
    infer_coeffs_batched on that clip alone with the same features, x_T, noise_seed and clip_offset = its id."""
    from helpers import make_msmd
    from msmd_b200.inference import infer_coeffs_queue
    m, args = make_msmd('cuda', precision=precision, n_diff_steps=T_SMALL)
    windows, pads = [3, 1, 4, 2, 1, 2, 3], [0, 40, 17, 0, 99, 1, 50]
    feats, shape, style, lens, x_T = gpu_clips(windows, pads, seed=3)
    ids = [4, 0, 21, 8, 13, 5, 300]
    codes, lengths = infer_coeffs_queue(m, args, feats, shape, style, lens, x_T, max_clips=3, clip_ids=ids,
                                        noise_seed=55, cfg_scale=1.4)
    assert lengths.tolist() == lens and codes.shape == (7, max(lens), 67) and torch.isfinite(codes).all()
    for k in range(7):
        one = alone(m, args, feats, shape, style, lens, x_T, k, 55, ids[k])
        assert one.shape == (lens[k], 67)
        assert torch.equal(codes[k, :lens[k]], one), (k, rel_l2(codes[k, :lens[k]], one))
        assert not codes[k, lens[k]:].any()


@pytest.mark.gpu
def test_noise_keys_with_z_is_rejected_by_the_library(built_lib):
    """msmd_sample_window_ex returns MSMD_ERR_INVALID, which the Python binding raises as ValueError."""
    from helpers import make_msmd
    m, args = make_msmd('cuda', precision=None, n_diff_steps=T_SMALL)
    feats, shape, style, lens, x_T = gpu_clips([1, 1], [0, 0], seed=4)
    m.sample(torch.stack(feats), shape, style, motion_at_T=x_T, indicator=torch.ones(2, L, device='cuda'), noise_seed=1)
    z = torch.zeros(T_SMALL + 1, 2, L, 67, device='cuda')
    keys = torch.zeros(2, 2, dtype=torch.int64, device='cuda')
    with pytest.raises(ValueError, match='noise_keys key the in-kernel noise'):
        m._eng.sample_window(x_T, z=z, noise_keys=keys)


@pytest.mark.gpu
def test_queue_at_benchmark_slot_count(built_lib):
    """64 clips in flight x 3 guidance entries = 192 sequences, mixed lengths: clips 0, 31 and 63 agree with the same
    clips sampled alone within 1e-3 (the alone-vs-batch bound of the 16-bit paths at this batch)."""
    from helpers import make_msmd
    from msmd_b200.inference import infer_coeffs_queue
    m, args = make_msmd('cuda', precision=None, n_diff_steps=T_SMALL)
    g = torch.Generator().manual_seed(9)
    K = 80
    windows = torch.randint(1, 4, (K,), generator=g).tolist()
    pads = torch.randint(0, 100, (K,), generator=g).tolist()
    feats, shape, style, lens, x_T = gpu_clips(windows, pads, seed=6)
    codes, lengths = infer_coeffs_queue(m, args, feats, shape, style, lens, x_T, max_clips=64, noise_seed=8, cfg_scale=1.4)
    assert lengths.tolist() == lens
    for k in (0, 31, 63):
        one = alone(m, args, feats, shape, style, lens, x_T, k, 8, k)
        err = rel_l2(codes[k, :lens[k]], one)
        print(f'clip {k}: queue vs alone rel-L2 {err:.2e}')
        assert err < 1e-3, (k, err)


def make_msmd_with_hubert():
    import torch.nn as nn  # noqa: F401
    import transformers
    from msmd_b200 import model as M
    from msmd_b200.utils import hubert
    from oracle import synth
    from oracle.ref_shims import pinned_args
    args = pinned_args(n_diff_steps=T_SMALL)
    m = M.MSMD(args, 'cpu', True, use_head_alpha=False, audio_encoder=hubert.HubertModel(transformers.HubertConfig()))
    m.load_state_dict(synth.fill_state_dict(synth.param_spec(m, skip=()), 1234), strict=False)
    return m.cuda().eval(), args


@pytest.mark.gpu
def test_infer_coeffs_many_lengths_and_features(built_lib):
    from msmd_b200.inference import extract_clip_features, infer_coeffs, infer_coeffs_many, plan_clip
    from oracle import synth
    m, args = make_msmd_with_hubert()
    sizes = [16000, 64000, 64640, 100100, 64000, 150000]
    audios = [synth.clip_audio(i, n).cuda() for i, n in enumerate(sizes)]
    style = torch.randn(len(sizes), 256, generator=torch.Generator().manual_seed(1)).cuda()
    shape = torch.zeros(len(sizes), 100, device='cuda')
    feats, lens = extract_clip_features(m, args, audios)
    for k, a in enumerate(audios):
        n_sub, padded, clip_len = plan_clip(len(a), args, 640.0)
        one = m.extract_audio_feature(F.pad(a, (0, padded - len(a)))[None], L * n_sub)[0]
        assert lens[k] == clip_len and feats[k].shape == one.shape
        assert rel_l2(feats[k], one) < 1e-5, (k, rel_l2(feats[k], one))
    codes, lengths = infer_coeffs_many(m, args, audios, shape, style, max_clips=4, noise_seed=3, cfg_scale=1.4)
    assert torch.isfinite(codes).all()
    for k, a in enumerate(audios):
        ref = infer_coeffs(m, args, a, shape[k:k + 1], 640.0, style[k:k + 1], cfg_scale=1.4, dynamic_threshold=None)
        assert int(lengths[k]) == ref.shape[1], k
