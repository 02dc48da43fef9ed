"""align_mask_width other than 1: the banded cross attention of the decoder layers (model.py:879-883,
model_common.enc_dec_mask).  Motion row i attends to memory columns [i-1-(w-1), i-1+(w-1)], the person token to all of
them, and w = 0 means no mask.

CPU: the oracle's general-width arithmetic against torch.nn.TransformerDecoder (the class the reference calls) with
memory_mask = alignment_mask; the module's mask buffer and state_dict layout; argument validation.
GPU: the engine's every-step banded path (tcgen05 cross-attention mode + the fp32-grade kernel) against the oracle."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2
from helpers import cpu_state_dict, make_msmd
from oracle import denoiser as D, synth

WIDTHS = (0, 2, 3)
F32_TOL = 1e-5


def _forward_args(i):
    return (i['motion'], i['audio'], i['person'], i['style'], i['prev_motion'], i['prev_audio'], i['step'], i['indicator'])


# ------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('w', [0, 1, 2, 3])
def test_oracle_matches_torch_transformer_decoder_with_memory_mask(w):
    """oracle.denoiser_forward vs the module's own nn.TransformerDecoder run with memory_mask = net.alignment_mask.
    Embedding and motion_dec are restated around it; the decoder stack is torch's."""
    m, args = make_msmd('cpu', align_mask_width=w)
    sd = cpu_state_dict(m)
    net = m.denoising_net
    sub = {k[len('denoising_net.'):]: v for k, v in sd.items() if k.startswith('denoising_net.')}
    i = synth.denoiser_inputs(2, 5)
    dyn, _, _ = D.denoiser_forward(sd, args, *_forward_args(i), keep_separate=True)
    te = sub['TE.pe'][0, i['step']]
    emb = F.linear(F.gelu(F.linear(te, sub['diff_step_map.0.weight'], sub['diff_step_map.0.bias'])),
                   sub['diff_step_map.2.weight'], sub['diff_step_map.2.bias']).unsqueeze(1)
    ptok = F.linear(i['person'], sub['person_proj.weight'], sub['person_proj.bias']) + emb
    feats = torch.cat([i['prev_motion'], i['motion']], 1)
    ind = torch.cat([torch.zeros(2, 10), i['indicator']], 1).unsqueeze(-1)
    x = torch.cat([ptok, F.linear(torch.cat([feats, ind], -1), sub['feature_proj.weight'], sub['feature_proj.bias'])],
                  1) + sub['PE']
    mem = torch.cat([i['prev_audio'], i['audio']], 1)
    with torch.no_grad():
        y = net.transformer.eval()(x, mem, memory_mask=net.alignment_mask)
        out = F.linear(F.gelu(F.linear(y[:, 1:], sub['motion_dec.0.weight'], sub['motion_dec.0.bias'])),
                       sub['motion_dec.2.weight'], sub['motion_dec.2.bias'])
    nb = args.num_of_basis
    assert rel_l2(dyn, out[..., :-nb]) <= 2e-6


@pytest.mark.parametrize('w', [0, 1, 2, 3, 200])
def test_module_mask_buffer_and_state_dict_layout(w):
    m, _ = make_msmd('cpu', align_mask_width=w)
    net = m.denoising_net
    keys = set(m.state_dict())
    ref_keys = set(make_msmd('cpu', align_mask_width=1)[0].state_dict())
    if w >= 1:
        assert torch.equal(net.alignment_mask, D.alignment_mask(10, 100, w))
        assert keys == ref_keys
    else:
        assert net.alignment_mask is None
        assert keys == ref_keys - {'denoising_net.alignment_mask'}


def test_mask_buffer_that_disagrees_with_the_width_raises():
    """A checkpoint loaded with strict=True overwrites the bool buffer, which the engine does not read: the host
    rejects it before any weight reaches the engine."""
    from msmd_b200 import _lib
    from msmd_b200.model import _check_alignment_mask
    m, _ = make_msmd('cpu', align_mask_width=2)
    _check_alignment_mask(m.denoising_net)
    m.denoising_net.alignment_mask.copy_(D.alignment_mask(10, 100, 3))
    with pytest.raises(_lib.MsmdError, match='align_mask_width=2'):
        _check_alignment_mask(m.denoising_net)
    m0, _ = make_msmd('cpu', align_mask_width=0)
    del m0.denoising_net.alignment_mask
    m0.denoising_net.register_buffer('alignment_mask', D.alignment_mask(10, 100, 1))
    with pytest.raises(_lib.MsmdError, match='no cross-attention mask'):
        _check_alignment_mask(m0.denoising_net)


def test_create_rejects_negative_width(built_lib):
    """msmd_create validates the configuration before it touches a device."""
    from msmd_b200 import _lib
    from msmd_b200._engine import MsmdConfig
    from msmd_b200.model import _engine_cfg
    m, _ = make_msmd('cpu', align_mask_width=1)
    cfg = _engine_cfg(m.denoising_net, 500, 'sample', 4, 'hybrid')
    cfg['align_mask_width'] = -1
    h = ctypes.c_void_p()
    assert _lib.lib().msmd_create(ctypes.byref(MsmdConfig(**cfg)), 0, ctypes.byref(h)) == -1    # MSMD_ERR_INVALID
    assert b'align_mask_width=-1' in _lib.lib().msmd_last_error()
    assert not h.value


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize('w', WIDTHS)
def test_forward_vs_oracle(built_lib, w):
    """Same bounds as the width-1 tests: fp32-grade 1e-5, and the 16-bit paths inside the error bounds the 'auto'
    hybrid schedule is sized from, with the same margins."""
    from msmd_b200.model import MSMD
    m, args = make_msmd('cuda', precision='hybrid', align_mask_width=w)
    i = synth.denoiser_inputs(5, 21)
    sd = cpu_state_dict(m)
    want = D.denoiser_forward(sd, args, *_forward_args(i))
    c = [v.cuda() for v in _forward_args(i)]
    errs = {p: rel_l2(m.denoising_net(*c, precise=p), want) for p in ('fp32', 'bf16', 'fp16')}
    print(f'w={w} x0_hat rel-L2 vs oracle: ' + ', '.join(f'{p} {e:.2e}' for p, e in errs.items()))
    assert errs['fp32'] < F32_TOL
    assert errs['bf16'] < MSMD.BF16_ERR_BOUND / 1.3
    assert errs['fp16'] < MSMD.FP16_ERR_BOUND / 1.8
    dyn, sta, alp = m.denoising_net(*c, keep_separate=True)
    wd, ws, wa = D.denoiser_forward(sd, args, *_forward_args(i), keep_separate=True)
    parts = [rel_l2(dyn, wd), rel_l2(sta, ws.unsqueeze(1).expand(sta.shape)), rel_l2(alp, wa)]
    assert max(parts) < F32_TOL, parts


@pytest.mark.gpu
@pytest.mark.parametrize('w', WIDTHS)
@pytest.mark.parametrize('mode', ['incremental', 'independent'])
def test_teacher_forced_steps_vs_oracle(built_lib, w, mode):
    """Default hybrid engine at T = 500: both ends of every schedule segment within 1e-3; the fp32-grade engine 1e-5."""
    T = 500
    mh, args = make_msmd('cuda', precision=None, n_diff_steps=T, align_mask_width=w)
    m32, _ = make_msmd('cuda', precision='fp32', n_diff_steps=T, align_mask_width=w)
    sd = cpu_state_dict(mh)
    k32, k16 = mh._precise_steps(), mh._fp16_steps()
    i = synth.sampler_inputs(3, T, 31)
    kw = dict(cfg_mode=mode, cfg_scale=[1.4, 1.4])
    for t in (500, 250, k16 + 1, k16, k32 + 1, k32, 1):
        x_t = synth.sampler_inputs(3, T, 300 + t)['x_T'] * (0.3 + 0.7 * t / T)
        want, _, _ = D.sample(sd, args, i['audio_feat'], i['shape'], i['style'], x_T=x_t, z=i['z'],
                              indicator=i['indicator'], t_start=t, n_steps=1, **kw)
        for name, m, tol in (('hybrid', mh, 1e-3), ('fp32', m32, F32_TOL)):
            got, _, _ = m.sample(i['audio_feat'].cuda(), i['shape'].cuda(), i['style'].cuda(), motion_at_T=x_t.cuda(),
                                 indicator=i['indicator'].cuda(), noise=i['z'].cuda(), t_start=t, n_steps=1, **kw)
            err = rel_l2(got, want)
            print(f'w={w} {mode} t={t:3d} {name:6s} rel-L2 {err:.2e}')
            assert err < tol, (w, mode, t, name, err)
    mh.check()


@pytest.mark.gpu
def test_benchmark_size_width2_vs_oracle(built_lib):
    """configs[2] shape (64 clips -> 192 sequences) at w = 2: teacher-forced steps at the segment ends for clips
    0 / 31 / 63 against the oracle run on those clips alone, and clip 31 sampled alone against the same clip in the
    batch over a run that crosses all three segments (bf16 graph replays, fp16, fp32-grade)."""
    from test_engine_gpu import CHECK, _bench_inputs, _sub
    T = 500
    i = _bench_inputs(T)
    sub = _sub(i, CHECK)
    dev = {k: v.cuda() for k, v in i.items()}
    mh, args = make_msmd('cuda', precision=None, n_diff_steps=T, align_mask_width=2)
    m32, _ = make_msmd('cuda', precision='fp32', n_diff_steps=T, align_mask_width=2)
    sd = cpu_state_dict(mh)
    k32, k16 = mh._precise_steps(), mh._fp16_steps()
    kw = dict(cfg_mode='incremental', cfg_scale=[1.4, 1.4])
    for t in (500, 250, k16 + 1, k16, k32 + 1, k32, 1):
        scale = 0.3 + 0.7 * t / T
        want, _, _ = D.sample(sd, args, sub['audio_feat'], sub['shape'], sub['style'], x_T=sub['x_T'] * scale, z=sub['z'],
                              indicator=sub['indicator'], t_start=t, n_steps=1, **kw)
        for name, m, tol in (('hybrid', mh, 1e-3), ('fp32', m32, F32_TOL)):
            got, _, _ = m.sample(dev['audio_feat'], dev['shape'], dev['style'], motion_at_T=dev['x_T'] * scale,
                                 indicator=dev['indicator'], noise=dev['z'], t_start=t, n_steps=1, **kw)
            errs = [rel_l2(got[c], want[j]) for j, c in enumerate(CHECK)]
            print(f'w=2 t={t:3d} {name:6s} rel-L2 of clips {CHECK}: ' + ' '.join(f'{e:.2e}' for e in errs))
            assert max(errs) < tol, (t, name, errs)
    t0 = k16 + 8
    for name, m, tol in (('hybrid', mh, 1e-3), ('fp32', m32, 1e-6)):
        run = lambda ix: m.sample(dev['audio_feat'][ix], dev['shape'][ix], dev['style'][ix], motion_at_T=dev['x_T'][ix],
                                  indicator=dev['indicator'][ix], noise=dev['z'][:, ix].contiguous(), t_start=t0,
                                  n_steps=t0, **kw)[0]
        batch, alone = run(torch.arange(64)), run([31])
        assert rel_l2(alone[0], batch[31]) < tol, name
    mh.check()


@pytest.mark.gpu
def test_windowed_driver_vs_oracle(built_lib):
    """inference.infer_coeffs_batched over 3 windows (the last one padded) at w = 2: the window carry-over and the
    cached step graphs reused by the later windows."""
    from msmd_b200.inference import infer_coeffs_batched
    T, N = 20, 2
    m, args = make_msmd('cuda', precision=None, n_diff_steps=T, align_mask_width=2)
    g = torch.Generator().manual_seed(41)
    feat = torch.randn(N, 300, 512, generator=g)
    shape = torch.zeros(N, 1, 100)
    style = torch.randn(N, 256, generator=g)
    x_T = torch.randn(N, 100, 67, generator=g)
    z = [synth.sampler_inputs(N, T, 50 + k)['z'] for k in range(3)]
    want = D.infer_coeffs(cpu_state_dict(m), args, feat, shape, style, 250, x_T, z, cfg_scale=1.4)
    got = infer_coeffs_batched(m, args, feat.cuda(), shape.cuda(), style.cuda(), clip_len=250, cfg_scale=1.4,
                               x_T=x_T.cuda(), noise=[zz.cuda() for zz in z])
    err = rel_l2(got, want)
    print(f'w=2 windowed driver, {T} steps x 3 windows, default engine: rel-L2 {err:.2e}')
    assert got.shape == (N, 250, 67) and err < 1e-3


@pytest.mark.gpu
def test_band_wider_than_the_memory_equals_no_mask(built_lib):
    """w = 200 covers every key of every row: bit for bit the w = 0 engine, in bf16 and in fp32-grade arithmetic."""
    T = 8
    i = synth.sampler_inputs(2, T, 61)
    c = {k: v.cuda() for k, v in i.items()}
    for precision in ('bf16', 'fp32'):
        out = []
        for w in (0, 200):
            m, _ = make_msmd('cuda', precision=precision, n_diff_steps=T, align_mask_width=w)
            x0, _, _ = m.sample(c['audio_feat'], c['shape'], c['style'], motion_at_T=c['x_T'], indicator=c['indicator'],
                                cfg_mode='incremental', cfg_scale=[1.4, 1.4], noise=c['z'])
            out.append(x0)
        assert torch.equal(out[0], out[1]), precision


@pytest.mark.gpu
def test_overwritten_mask_buffer_raises_through_the_module(built_lib):
    from msmd_b200 import _lib
    m, _ = make_msmd('cuda', align_mask_width=2)
    c = [v.cuda() for v in _forward_args(synth.denoiser_inputs(1, 3))]
    m.denoising_net(*c)
    m.denoising_net.alignment_mask.copy_(D.alignment_mask(10, 100, 1).cuda())
    with pytest.raises(_lib.MsmdError, match='does not match align_mask_width=2'):
        m.denoising_net(*c)
