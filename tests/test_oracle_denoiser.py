"""CPU: oracle/denoiser.py against the golden vectors produced from the unmodified reference
(DenoisingNetwork_MSMD.forward and MSMD.sample trajectories), plus host-side drop-in checks."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_l2
from helpers import cpu_state_dict, make_msmd
from oracle import denoiser as D, ref_shims, synth
from oracle.make_golden import DEN_GOLD, SAMP_GOLD, VAR_GOLD, VARIANTS, ref_msmd, variant_kwargs


@pytest.fixture(scope='module')
def msmd():
    return make_msmd('cpu')


def test_tables_match_module_buffers(msmd):
    m, args = msmd
    sd = cpu_state_dict(m)
    for k, v in D.cosine_schedule(args.n_diff_steps).items():
        assert torch.equal(v, sd['diffusion_sched.' + k]), k
    assert torch.equal(D.sinusoid_table(args.n_diff_steps + 1, 512), sd['denoising_net.TE.pe'][0])
    assert torch.equal(D.alignment_mask(10, 100, 1), sd['denoising_net.alignment_mask'])
    # the structure the CUDA path exploits: row 0 sees all memory, motion row i sees exactly column i-1
    mask = sd['denoising_net.alignment_mask']
    assert not mask[0].any() and all((~mask[i]).nonzero().flatten().tolist() == [i - 1] for i in range(1, 111))


def test_oracle_denoiser_matches_golden(msmd):
    m, args = msmd
    i = synth.denoiser_inputs(DEN_GOLD['N'], DEN_GOLD['seed'])
    got = D.denoiser_forward(cpu_state_dict(m), args, i['motion'], i['audio'], i['person'], i['style'],
                             i['prev_motion'], i['prev_audio'], i['step'], i['indicator'])
    want = np.load(os.path.join(GOLDEN, 'denoiser.npz'))['out']
    assert rel_l2(got, want) < 2e-6


def test_oracle_sampler_matches_golden():
    c = SAMP_GOLD
    m, args = make_msmd('cpu', n_diff_steps=c['T'])
    sd = cpu_state_dict(m)
    i = synth.sampler_inputs(c['N'], c['T'], c['seed'])
    gold = np.load(os.path.join(GOLDEN, 'sampler.npz'))
    for mode in ('incremental', 'independent'):
        traj, _, _ = D.sample(sd, args, i['audio_feat'], i['shape'], i['style'], x_T=i['x_T'], z=i['z'],
                              indicator=i['indicator'], cfg_mode=mode, cfg_scale=list(c['scales']), ret_traj=True)
        for t in range(c['T'], -1, -1):
            assert rel_l2(traj[t], gold[mode][t]) < 5e-6, (mode, t)


def test_cross_attention_is_step_invariant_for_motion_rows(msmd):
    """SURVEY section 0: with align_mask_width=1 the cross-attention output of rows >= 1 equals
    out_proj(v_proj(memory[i-1])) whatever the query is."""
    m, args = msmd
    sd = {k[len('denoising_net.'):]: v for k, v in cpu_state_dict(m).items() if k.startswith('denoising_net.')}
    p = 'transformer.layers.3.multihead_attn.'
    g = torch.Generator().manual_seed(0)
    mem = torch.randn(2, 110, 512, generator=g)
    outs = [D.mha(torch.randn(2, 111, 512, generator=g), mem, sd[p + 'in_proj_weight'], sd[p + 'in_proj_bias'],
                  sd[p + 'out_proj.weight'], sd[p + 'out_proj.bias'], 8, sd['alignment_mask']) for _ in range(2)]
    assert (outs[0][:, 1:] - outs[1][:, 1:]).abs().max() < 1e-6
    W, b = sd[p + 'in_proj_weight'], sd[p + 'in_proj_bias']
    v = torch.nn.functional.linear(mem, W[1024:], b[1024:])
    want = torch.nn.functional.linear(v, sd[p + 'out_proj.weight'], sd[p + 'out_proj.bias'])
    assert (outs[0][:, 1:] - want).abs().max() < 2e-6


def test_dropin_state_dict_layout(msmd):
    """SURVEY App. E keys/shapes, and key for key the reference module's (stored in tests/golden/ref_modules.npz; checked
    live too when the reference is mounted)."""
    m, args = msmd
    sd = m.state_dict()
    assert sd['denoising_net.PE'].shape == (1, 111, 512)
    assert sd['denoising_net.transformer.layers.7.multihead_attn.in_proj_weight'].shape == (1536, 512)
    assert sd['denoising_net.motion_dec.2.weight'].shape == (71, 256)
    assert sd['denoising_net.feature_proj.weight'].shape == (512, 68)
    assert sd['null_style_feat'].shape == (1, 1, 256) and sd['start_audio_feat'].shape == (1, 10, 512)
    g = np.load(os.path.join(GOLDEN, 'ref_modules.npz'))
    want = {k: tuple(int(n) for n in s.split(',') if n) for k, s in zip(g['state_dict_keys'], g['state_dict_shapes'])}
    if ref_shims.available():
        r = ref_shims.ref_modules()
        rm = r.model.get_diffusion_model(ref_shims.pinned_args(), 'cpu')
        assert {k: tuple(v.shape) for k, v in rm.state_dict().items() if not k.startswith('audio_encoder.')} == want
    assert {k: tuple(v.shape) for k, v in sd.items()} == want


def test_no_cpu_path_for_model(msmd):
    from msmd_b200 import _lib
    m, _ = msmd
    i = synth.sampler_inputs(1, 500)
    with pytest.raises(_lib.MsmdError):
        m.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'], indicator=i['indicator'])
    with pytest.raises(_lib.MsmdError):
        m(i['x_T'], i['audio_feat'], i['shape'])


def test_oracle_sampler_noise_target_matches_golden():
    """args.target == 'noise' (model.py:421-424): the posterior step with the network read as eps."""
    c = SAMP_GOLD
    m, args = make_msmd('cpu', n_diff_steps=c['T'], target='noise')
    sd = cpu_state_dict(m)
    i = synth.sampler_inputs(c['N'], c['T'], c['seed'])
    gold = np.load(os.path.join(GOLDEN, 'sampler_noise.npz'))['incremental']
    x = torch.from_numpy(gold[c['T']])
    for t in range(c['T'], 0, -1):       # teacher-forced: the random-weight eps recursion amplifies any difference
        nxt, _, _ = D.sample(sd, args, i['audio_feat'], i['shape'], i['style'], x_T=torch.from_numpy(gold[t]), z=i['z'],
                             indicator=i['indicator'], cfg_mode='incremental', cfg_scale=list(c['scales']), t_start=t,
                             n_steps=1)
        assert rel_l2(nxt, gold[t - 1]) < 5e-6, t


@pytest.mark.parametrize('use_indicator', [True, False])
def test_oracle_sampler_variants_match_reference(use_indicator):
    """Guidance sets other than the default (none / audio only / style only), sigma 'flexibility' > 0 and a model built
    without the indicator input, 4 sampling steps each: the oracle against the reference's outputs stored in
    tests/golden/sampler_variants.npz (every 3rd frame; see oracle/make_golden.py for how they were made) and, when the
    unmodified reference is mounted, against it live on every frame."""
    c = VAR_GOLD
    m, args = make_msmd('cpu', n_diff_steps=c['T'], use_indicator=use_indicator)
    sd = cpu_state_dict(m)
    gold = np.load(os.path.join(GOLDEN, 'sampler_variants.npz'))
    i = synth.sampler_inputs(c['N'], c['T'], c['seed'])
    ind = i['indicator'] if use_indicator else None
    ref = ref_msmd(c['weight_seed'], n_diff_steps=c['T'], use_indicator=use_indicator)[0] if ref_shims.available() else None
    for k, v in enumerate(VARIANTS):
        kw = variant_kwargs(v)
        got, _, _ = D.sample(sd, args, i['audio_feat'], i['shape'], i['style'], x_T=i['x_T'], z=i['z'], indicator=ind, **kw)
        assert rel_l2(got[:, ::c['stride']], gold[f'indicator{int(use_indicator)}_variant{k}']) < 5e-6, v
        if ref is not None:
            with ref_shims.inject_randn_like([i['z'][t] for t in range(c['T'], 1, -1)]):
                want, _, _ = ref.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'], indicator=ind, **kw)
            assert rel_l2(got, want) < 5e-6, v
