#!/usr/bin/env python
"""Generate tests/golden/*.npz from the UNMODIFIED reference (build container only).

    python -m oracle.make_golden [rot flame denoiser sampler style audio infer]

Each section seeds its inputs through oracle.synth (so tests can rebuild them without
the file), runs the reference modules imported from /root/reference via
oracle.ref_shims, and stores the reference outputs.  The GPU box has no reference:
tests there compare the CUDA path against these vectors and against the oracle.
"""
import os
import sys

import numpy as np
import torch

from . import ref_shims, synth

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')


def rot_inputs(n=256, seed=11):
    """Shared by the generator and the tests: random + edge-case rotations."""
    g = torch.Generator().manual_seed(seed)
    aa = torch.randn(n, 3, generator=g) * 1.3
    aa[:4] = 0.0                     # exact zero angle (series branch)
    aa[4:8] *= 1e-7                  # tiny angle
    aa[8] = torch.tensor([np.pi, 0, 0])
    aa[9] = torch.tensor([0, 3.1, 0])
    quat = torch.randn(n, 4, generator=g)
    quat[:4] = torch.tensor([1.0, 0, 0, 0])
    quat[4] = torch.tensor([-1.0, 0, 0, 0])
    quat2 = torch.randn(n, 4, generator=g)
    euler = (torch.rand(n, 3, generator=g) * 2 - 1) * 3.0
    euler[:2] = 0
    d6 = torch.randn(n, 6, generator=g)
    pts = torch.randn(n, 3, generator=g)
    return dict(aa=aa, quat=quat, quat2=quat2, euler=euler, d6=d6, pts=pts)


ROT_CONVENTIONS = ['XYZ', 'YXZ', 'ZYX', 'XZY', 'XYX', 'ZXZ', 'YZY']


def gen_rot():
    rc = ref_shims.ref_modules().rc
    lbs = ref_shims.ref_modules().lbs
    i = rot_inputs()
    o = {}
    mats = rc.euler_angles_to_matrix(i['euler'], 'YXZ')
    o['mats'] = mats
    o['quaternion_to_matrix'] = rc.quaternion_to_matrix(i['quat'])
    o['matrix_to_quaternion'] = rc.matrix_to_quaternion(mats)
    for c in ROT_CONVENTIONS:
        o[f'euler_angles_to_matrix_{c}'] = rc.euler_angles_to_matrix(i['euler'], c)
        o[f'matrix_to_euler_angles_{c}'] = rc.matrix_to_euler_angles(mats, c)
    o['axis_angle_to_quaternion'] = rc.axis_angle_to_quaternion(i['aa'])
    o['quaternion_to_axis_angle'] = rc.quaternion_to_axis_angle(rc.axis_angle_to_quaternion(i['aa']))
    o['axis_angle_to_matrix'] = rc.axis_angle_to_matrix(i['aa'])
    o['matrix_to_axis_angle'] = rc.matrix_to_axis_angle(mats)
    o['rotation_6d_to_matrix'] = rc.rotation_6d_to_matrix(i['d6'])
    o['matrix_to_rotation_6d'] = rc.matrix_to_rotation_6d(mats)
    o['axis_angle_to_rotation_6d'] = rc.axis_angle_to_rotation_6d(i['aa'])
    o['standardize_quaternion'] = rc.standardize_quaternion(i['quat'])
    o['quaternion_raw_multiply'] = rc.quaternion_raw_multiply(i['quat'], i['quat2'])
    o['quaternion_multiply'] = rc.quaternion_multiply(i['quat'], i['quat2'])
    o['quaternion_invert'] = rc.quaternion_invert(i['quat'])
    o['quaternion_apply'] = rc.quaternion_apply(i['quat'], i['pts'])
    o['batch_rodrigues'] = lbs.batch_rodrigues(i['aa'])
    o['euler_to_axis_angle_YXZ'] = rc.matrix_to_axis_angle(rc.euler_angles_to_matrix(i['euler'], 'YXZ'))
    np.savez_compressed(os.path.join(OUT, 'rot.npz'), **{k: v.numpy() for k, v in o.items()})
    print('rot.npz', len(o))


FLAME_GOLD = dict(B=6, n_shape=300, n_exp=100, seed=3)


def gen_flame():
    cfg = FLAME_GOLD
    raw = synth.flame_raw(0, synth.FLAME_V, 400)
    fl = ref_shims.ref_flame(raw, cfg['n_shape'], cfg['n_exp'])
    sh, ex, po, ey = synth.flame_inputs(cfg['B'], cfg['n_shape'], cfg['n_exp'], cfg['seed'])
    with torch.no_grad():
        v, lm2d, lm3d = fl(sh, ex, po, ey)
        v_nopose, _, _ = fl(sh, ex, None, None, return_lm2d=False, return_lm3d=False)
        v_noglob, _, _ = fl(sh, ex, po, ey, ignore_global_rot=True, return_lm2d=False, return_lm3d=False)
        # 100/50 reference default (flame.py:49-50)
        fl2 = ref_shims.ref_flame(raw, 100, 50)
        sh2, ex2, po2, ey2 = synth.flame_inputs(cfg['B'], 100, 50, cfg['seed'] + 1)
        v2, _, _ = fl2(sh2, ex2, po2, ey2, return_lm2d=False, return_lm3d=False)
    np.savez_compressed(os.path.join(OUT, 'flame.npz'), verts=v.numpy(), lm2d=lm2d.numpy(), lm3d=lm3d.numpy(),
                        verts_nopose=v_nopose.numpy(), verts_noglob=v_noglob.numpy(), verts_100_50=v2.numpy())
    print('flame.npz', v.shape)


DEN_GOLD = dict(N=3, seed=21, weight_seed=1234)
SAMP_GOLD = dict(N=2, T=12, seed=22, weight_seed=1234, scales=[1.4, 1.7])


def ref_msmd(weight_seed, **over):
    """Reference MSMD (model.py:73) with deterministic weights from synth.fill_state_dict."""
    m = ref_shims.ref_modules()
    args = ref_shims.pinned_args(**over)
    model = m.model.get_diffusion_model(args, 'cpu').eval()
    fill = synth.fill_state_dict(synth.param_spec(model), weight_seed)
    missing, unexpected = model.load_state_dict(fill, strict=False)
    assert not unexpected and all(k.startswith(('audio_encoder.', 'diffusion_sched.')) or k.endswith(('TE.pe', 'alignment_mask'))
                                  for k in missing), (missing[:5], unexpected[:5])
    return model, args


def gen_denoiser():
    c = DEN_GOLD
    model, args = ref_msmd(c['weight_seed'])
    i = synth.denoiser_inputs(c['N'], c['seed'])
    out = model.denoising_net(i['motion'], i['audio'], i['person'], i['style'], i['prev_motion'], i['prev_audio'],
                              i['step'], i['indicator'])
    np.savez_compressed(os.path.join(OUT, 'denoiser.npz'), out=out.numpy())
    print('denoiser.npz', out.shape)


def gen_sampler():
    c = SAMP_GOLD
    model, args = ref_msmd(c['weight_seed'], n_diff_steps=c['T'])
    i = synth.sampler_inputs(c['N'], c['T'], c['seed'])
    res = {}
    for mode in ('incremental', 'independent'):
        with ref_shims.inject_randn_like([i['z'][t] for t in range(c['T'], 1, -1)]):
            traj, _, _ = model.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'],
                                      indicator=i['indicator'], cfg_mode=mode, cfg_scale=list(c['scales']),
                                      ret_traj=True)
        res[mode] = torch.stack([traj[t] for t in range(c['T'] + 1)]).numpy()
    np.savez_compressed(os.path.join(OUT, 'sampler.npz'), **res)
    print('sampler.npz', res['incremental'].shape)


def gen_sampler_noise():
    """args.target == 'noise' (model.py:421-424: the network predicts eps, x_{t-1} = (x_t - c1 eps) / sqrt(alpha) + sigma z),
    with dynamic thresholding off; same inputs as gen_sampler."""
    c = SAMP_GOLD
    model, args = ref_msmd(c['weight_seed'], n_diff_steps=c['T'], target='noise')
    assert model.target == 'noise'
    i = synth.sampler_inputs(c['N'], c['T'], c['seed'])
    with ref_shims.inject_randn_like([i['z'][t] for t in range(c['T'], 1, -1)]):
        traj, _, _ = model.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'], indicator=i['indicator'],
                                  cfg_mode='incremental', cfg_scale=list(c['scales']), ret_traj=True)
    out = torch.stack([traj[t] for t in range(c['T'] + 1)]).numpy()
    np.savez_compressed(os.path.join(OUT, 'sampler_noise.npz'), incremental=out)
    print('sampler_noise.npz', out.shape, float(np.abs(out[0]).max()))


STYLE_GOLD = dict(N=5, L=100, seed=31, weight_seed=77)


def gen_style():
    c = STYLE_GOLD
    m = ref_shims.ref_modules()
    enc = m.style.get_style_encoder(ref_shims.pinned_args(), 'vae2').eval()
    enc.load_state_dict(synth.fill_state_dict(synth.param_spec(enc), c['weight_seed']), strict=False)
    g = torch.Generator().manual_seed(c['seed'])
    x = torch.randn(c['N'], c['L'], 67, generator=g)
    eps = torch.randn(c['N'], 256, generator=g)
    with ref_shims.inject_randn_like([eps]):
        out, mu, logvar = enc(x)
    x2 = torch.randn(3, 41, 67, generator=g)          # a shorter style clip
    with ref_shims.inject_randn_like([eps[:3]]):
        out2, mu2, logvar2 = enc(x2)
    np.savez_compressed(os.path.join(OUT, 'style.npz'), out=out.numpy(), mu=mu.numpy(), logvar=logvar.numpy(),
                        mu_short=mu2.numpy(), logvar_short=logvar2.numpy())
    print('style.npz', out.shape)


def style_inputs():
    c = STYLE_GOLD
    g = torch.Generator().manual_seed(c['seed'])
    x = torch.randn(c['N'], c['L'], 67, generator=g)
    eps = torch.randn(c['N'], 256, generator=g)
    x2 = torch.randn(3, 41, 67, generator=g)
    return x, eps, x2


AUDIO_GOLD = dict(weight_seed=4321, clips=2, samples=64000, frames=100, short_samples=48000, short_frames=75)


def audio_inputs():
    c = AUDIO_GOLD
    x = torch.stack([synth.clip_audio(i, c['samples']) for i in range(c['clips'])])
    xs = torch.stack([synth.clip_audio(9, c['short_samples'])])
    return x, xs


def gen_audio():
    c = AUDIO_GOLD
    m = ref_shims.ref_modules()
    res = {}
    for am in ('hubert', 'wav2vec2'):
        model = m.model.get_diffusion_model(ref_shims.pinned_args(audio_model=am), 'cpu').eval()
        fill = synth.fill_state_dict(synth.param_spec(model, skip=('denoising_net.',)), c['weight_seed'])
        missing, unexpected = model.load_state_dict(fill, strict=False)
        assert not unexpected
        x, xs = audio_inputs()
        res[am] = model.extract_audio_feature(x, c['frames']).numpy()
        res[am + '_short'] = model.extract_audio_feature(xs, c['short_frames']).numpy()
    np.savez_compressed(os.path.join(OUT, 'audio.npz'), **res)
    print('audio.npz', {k: v.shape for k, v in res.items()})


INFER_GOLD = dict(T=6, weight_seed=1234, samples=160000, clip_id=3)


def infer_inputs():
    """Config-1-shaped inputs (SURVEY 8(d)): one 10 s clip -> 3 windows, the last one padded by 50 frames."""
    c = INFER_GOLD
    audio = synth.clip_audio(c['clip_id'], c['samples'])
    style = synth.clip_style_eps(c['clip_id'])                    # any [1,256] vector serves as the style code here
    x_T = synth.clip_xT(c['clip_id'])
    z = [synth.clip_step_noise(c['clip_id'], w, c['T']).unsqueeze(1) for w in range(3)]
    return audio, style, x_T, z


def gen_infer():
    """inference.infer_coeffs end to end (audio -> HuBERT -> 3 windows), T=6 diffusion steps to keep the file
    small; noise injected: x_T through torch.randn (model.py:337), z through torch.randn_like (model.py:379)."""
    c = INFER_GOLD
    m = ref_shims.ref_modules()
    infer = ref_shims.ref_infer_coeffs()
    args = ref_shims.pinned_args(n_diff_steps=c['T'])
    model = m.model.get_diffusion_model(args, 'cpu').eval()
    fill = synth.fill_state_dict(synth.param_spec(model, skip=()), c['weight_seed'])
    model.load_state_dict(fill, strict=False)
    audio, style, x_T, z = infer_inputs()
    zs = [z[w][t] for w in range(3) for t in range(c['T'], 1, -1)]
    orig_randn = torch.randn
    torch.randn = lambda *a, **k: x_T.clone()
    try:
        with ref_shims.inject_randn_like(zs):
            out = infer(model, args, audio, torch.zeros(1, 1, 100), 640.0, style, cfg_scale=1.4, dynamic_threshold=None)
    finally:
        torch.randn = orig_randn
    feat = model.extract_audio_feature(torch.nn.functional.pad(audio, (0, 32000)).unsqueeze(0), 300)
    np.savez_compressed(os.path.join(OUT, 'infer.npz'), coeffs=out.numpy(), audio_feat=feat.numpy())
    print('infer.npz', out.shape)


SEP_GOLD = dict(N=1, T=5, seed=23, weight_seed=1234, scales=[1.4, 1.7], dt=(0.8, 0.5, 2.0))


def gen_separate():
    """MSMD.sample with dynamic thresholding (N=2) and MSMD.sample_separate (N=1: the reference's tiling of the
    static features, model.py:983-984, only works for batch 1)."""
    c = SEP_GOLD
    model, args = ref_msmd(c['weight_seed'], n_diff_steps=c['T'])
    res = {}
    i2 = synth.sampler_inputs(2, c['T'], c['seed'] + 1)
    for mode in ('incremental', 'independent'):
        with ref_shims.inject_randn_like([i2['z'][t] for t in range(c['T'], 1, -1)]):
            res['dt_' + mode] = model.sample(i2['audio_feat'], i2['shape'], i2['style'], motion_at_T=i2['x_T'],
                                             indicator=i2['indicator'], cfg_mode=mode, cfg_scale=list(c['scales']),
                                             dynamic_threshold=c['dt'])[0].numpy()
    i = synth.sampler_inputs(c['N'], c['T'], c['seed'])
    for mode in ('incremental', 'independent'):
        with ref_shims.inject_randn_like([i['z'][t] for t in range(c['T'], 1, -1)]):
            w = model.sample_separate(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'],
                                      indicator=i['indicator'], cfg_mode=mode, cfg_scale=list(c['scales']),
                                      dynamic_threshold=c['dt'], return_all_alpha=True)
        for k, v in zip(('x0', 'dyn', 'stat', 'alpha'), (w[0], w[3], w[4], w[5])):
            res[f'sep_{mode}_{k}'] = v.numpy()
    np.savez_compressed(os.path.join(OUT, 'separate.npz'), **res)
    print('separate.npz', {k: v.shape for k, v in res.items()})


DECODE_GOLD = dict(N=2, F=4, seed=41)


def decode_inputs():
    """Shared by the generator and the tests: 54-d DiffPoseTalk-layout coefficients + statistics, and 67-d MSMD codes
    (normalised) + their de-normalisation statistics (head rotation in Euler 'YXZ' degrees)."""
    c = DECODE_GOLD
    g = torch.Generator().manual_seed(c['seed'])
    r = lambda *s: torch.randn(*s, generator=g)
    motion54 = torch.cat([r(c['N'], c['F'], 50), 0.2 * r(c['N'], c['F'], 4)], -1)
    shape = r(c['N'], 100)
    stats54 = dict(exp_mean=0.1 * r(50), exp_std=0.5 + torch.rand(50, generator=g), pose_mean=0.05 * r(6),
                   pose_std=0.5 + torch.rand(6, generator=g), shape_mean=0.1 * r(100), shape_std=0.5 + torch.rand(100, generator=g))
    codes67 = r(c['N'], c['F'], 67)
    stats67 = dict(exp_mean=0.1 * r(64), exp_std=0.5 + torch.rand(64, generator=g), rot_mean=5.0 * r(3),
                   rot_std=10.0 + 10.0 * torch.rand(3, generator=g))
    return motion54, shape, stats54, codes67, stats67


def gen_decode():
    """(a) utils/common.py:140-196 get_coef_dict + coef_dict_to_vertices on the reference FLAME(100, 50);
    (b) the 67-d decode chain out of reference functions: inference.py:274-275 de-normalisation, Euler 'YXZ' degrees
    (Step2*.py:556-566) -> rotation_conversions.euler_angles_to_matrix -> matrix_to_axis_angle -> FLAME(300, 100)."""
    import math
    m = ref_shims.ref_modules()
    import utils.common as ref_common
    motion54, shape, stats54, codes67, stats67 = decode_inputs()
    raw = synth.flame_raw(0, synth.FLAME_V, 400)
    res = {}
    fl = ref_shims.ref_flame(raw, 100, 50)
    for name, kw in (('global', dict(with_global_pose=True)), ('noglobal', dict(with_global_pose=False))):
        cd = ref_common.get_coef_dict(motion54.clone(), shape, stats54, **kw)
        for k, v in cd.items():
            res[f'cd_{name}_{k}'] = v.numpy().copy()
        res[f'verts54_{name}'] = ref_common.coef_dict_to_vertices(cd, fl, flame_batch_size=5).numpy()
    cd = ref_common.get_coef_dict(motion54.clone(), shape, stats54, with_global_pose=True)   # (no stats: .view fails on the expanded shape, common.py:178)
    res['verts54_ignore_global'] = ref_common.coef_dict_to_vertices(cd, fl, ignore_global_rot=True).numpy()
    fl2 = ref_shims.ref_flame(raw, 300, 100)
    N, Fr, _ = codes67.shape
    exp = codes67[..., :-3] * stats67['exp_std'] + stats67['exp_mean']
    rot = codes67[..., -3:] * stats67['rot_std'] + stats67['rot_mean']
    aa = m.rc.matrix_to_axis_angle(m.rc.euler_angles_to_matrix(rot.reshape(-1, 3) * (math.pi / 180.0), 'YXZ'))
    expression = torch.zeros(N * Fr, 100)
    expression[:, :64] = exp.reshape(N * Fr, 64)
    v, _, _ = fl2(torch.zeros(N * Fr, 300), expression, torch.cat([aa, torch.zeros_like(aa)], 1), None,
                  return_lm2d=False, return_lm3d=False)
    res['verts67'] = v.view(N, Fr, -1, 3).numpy()
    res['aa67'] = aa.numpy()
    np.savez_compressed(os.path.join(OUT, 'decode.npz'), **res)
    print('decode.npz', {k: v.shape for k, v in res.items()})


def gen_denoiser_parts():
    """DenoisingNetwork_MSMD.forward(keep_separate=True) (model.py:972-973), same inputs as gen_denoiser."""
    c = DEN_GOLD
    model, args = ref_msmd(c['weight_seed'])
    i = synth.denoiser_inputs(c['N'], c['seed'])
    dyn, sta, alp = model.denoising_net(i['motion'], i['audio'], i['person'], i['style'], i['prev_motion'], i['prev_audio'],
                                        i['step'], i['indicator'], keep_separate=True)
    np.savez_compressed(os.path.join(OUT, 'denoiser_parts.npz'), dyn=dyn.numpy(), static=sta.numpy(), alphas=alp.numpy())
    print('denoiser_parts.npz', dyn.shape, sta.shape, alp.shape)


VAR_GOLD = dict(N=2, T=4, seed=5, weight_seed=1234, stride=3)     # every 3rd frame is stored (size)
VARIANTS = [dict(cfg_cond=[], flexibility=0.3), dict(cfg_cond=['audio'], flexibility=0.0),
            dict(cfg_cond=['style'], flexibility=0.5), dict(cfg_cond=['audio', 'style'], flexibility=1.0, cfg_mode='independent')]


def variant_kwargs(v):
    return dict(cfg_mode=v.get('cfg_mode', 'incremental'), cfg_cond=v['cfg_cond'], cfg_scale=[1.3, 1.6][:len(v['cfg_cond'])],
                flexibility=v['flexibility'])


def dropin_state_dict(weight_seed, **over):
    """state_dict of the package's drop-in MSMD with synth weights (key for key the reference's, see
    tests/test_oracle_denoiser.py::test_dropin_state_dict_layout)."""
    import torch.nn as nn
    from msmd_b200 import model as M
    m = M.MSMD(ref_shims.pinned_args(**over), 'cpu', True, use_head_alpha=False, regularize_alpha="None",
               audio_encoder=nn.Identity())
    m.load_state_dict(synth.fill_state_dict(synth.param_spec(m), weight_seed), strict=False)
    return {k: v.detach() for k, v in m.state_dict().items()}


# The two sections below store what tests compare with the reference live.  The committed files were written without the
# reference (source = 'oracle'): by oracle/denoiser.py, oracle/rotations.py and oracle/flame_lbs.py, unchanged since the
# commits whose live tests pinned them to the unmodified reference (sampler variants: rel-L2 < 5e-6; rotations: 3e-6
# absolute; FLAME vertices and lbs joints: rel-L2 < 1e-6).  With the reference mounted they are written from it.
def gen_sampler_variants():
    """MSMD.sample for guidance sets other than the default (none / audio only / style only / independent), sigma
    'flexibility' > 0, and models with and without the indicator input: 4 sampling steps each."""
    from . import denoiser as D
    c, live, res = VAR_GOLD, ref_shims.available(), {}
    i = synth.sampler_inputs(c['N'], c['T'], c['seed'])
    for use_indicator in (True, False):
        ind = i['indicator'] if use_indicator else None
        if live:
            ref, args = ref_msmd(c['weight_seed'], n_diff_steps=c['T'], use_indicator=use_indicator)
        else:
            sd = dropin_state_dict(c['weight_seed'], n_diff_steps=c['T'], use_indicator=use_indicator)
            args = ref_shims.pinned_args(n_diff_steps=c['T'], use_indicator=use_indicator)
        for k, v in enumerate(VARIANTS):
            if live:
                with ref_shims.inject_randn_like([i['z'][t] for t in range(c['T'], 1, -1)]):
                    out, _, _ = ref.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'], indicator=ind,
                                           **variant_kwargs(v))
            else:
                out, _, _ = D.sample(sd, args, i['audio_feat'], i['shape'], i['style'], x_T=i['x_T'], z=i['z'],
                                     indicator=ind, **variant_kwargs(v))
            res[f'indicator{int(use_indicator)}_variant{k}'] = out[:, ::c['stride']].numpy()
    res['source'] = np.array('reference' if live else 'oracle')
    np.savez_compressed(os.path.join(OUT, 'sampler_variants.npz'), **res)
    print('sampler_variants.npz', res['source'], len(res) - 1)


REF_MOD_GOLD = dict(rot_n=128, rot_seed=99, conventions=('ZYX', 'YZX'), raw_seed=5, V=300, n_shape=100, n_exp=50, B=16,
                    seed=8, stride=3)     # every 3rd vertex is stored (size)


def gen_ref_modules():
    """Euler conventions ZYX / YZX both ways, FLAME.forward and lbs (vertices + posed joints) on a 300-vertex model with
    100 + 50 betas, and the MSMD state_dict layout (key -> shape, audio encoder excluded)."""
    from . import flame_lbs, rotations as R
    c, live, res = REF_MOD_GOLD, ref_shims.available(), {}
    i = rot_inputs(n=c['rot_n'], seed=c['rot_seed'])
    assets = synth.flame_assets(c['raw_seed'], c['V'], c['n_shape'], c['n_exp'])
    sh, ex, po, ey = synth.flame_inputs(c['B'], c['n_shape'], c['n_exp'], c['seed'])
    full = flame_lbs.flame_full_pose(po, ey, c['B'])
    betas = torch.cat([sh, ex], 1)
    if live:
        m = ref_shims.ref_modules()
        for conv in c['conventions']:
            mats = m.rc.euler_angles_to_matrix(i['euler'], conv)
            res[f'euler_angles_to_matrix_{conv}'] = mats.numpy()
            res[f'matrix_to_euler_angles_{conv}'] = m.rc.matrix_to_euler_angles(mats, conv).numpy()
        fl = ref_shims.ref_flame(synth.flame_raw(c['raw_seed'], c['V'], 400), c['n_shape'], c['n_exp'])
        res['flame_verts'] = fl(sh, ex, po, ey, return_lm2d=False, return_lm3d=False)[0][:, ::c['stride']].numpy()
        v, j = m.lbs.lbs(betas, full, assets['v_template'][None].expand(c['B'], -1, -1), assets['shapedirs'],
                         assets['posedirs'], assets['J_regressor'], torch.tensor(assets['parents']), assets['lbs_weights'])
        sd = m.model.get_diffusion_model(ref_shims.pinned_args(), 'cpu').state_dict()
    else:
        for conv in c['conventions']:
            mats = R.euler_angles_to_matrix(i['euler'].numpy(), conv)
            res[f'euler_angles_to_matrix_{conv}'] = mats
            res[f'matrix_to_euler_angles_{conv}'] = R.matrix_to_euler_angles(mats, conv)
        res['flame_verts'] = flame_lbs.flame_forward(assets, sh, ex, po, ey)[:, ::c['stride']].numpy()
        v, j = flame_lbs.lbs(betas, full, assets['v_template'], assets['shapedirs'], assets['posedirs'],
                             assets['J_regressor'], assets['parents'], assets['lbs_weights'])
        sd = dropin_state_dict(1234)
    res['lbs_verts'], res['lbs_joints'] = v[:, ::c['stride']].numpy(), j.numpy()
    keys = sorted(k for k in sd if not k.startswith('audio_encoder.'))
    res['state_dict_keys'] = np.array(keys)
    res['state_dict_shapes'] = np.array([','.join(map(str, sd[k].shape)) for k in keys])
    res['source'] = np.array('reference' if live else 'oracle')
    np.savez_compressed(os.path.join(OUT, 'ref_modules.npz'), **res)
    print('ref_modules.npz', res['source'], len(keys), 'state_dict keys')


SECTIONS = dict(decode=gen_decode, denoiser_parts=gen_denoiser_parts, rot=gen_rot, flame=gen_flame, denoiser=gen_denoiser, sampler=gen_sampler, style=gen_style,
                audio=gen_audio, infer=gen_infer, separate=gen_separate, sampler_noise=gen_sampler_noise,
                sampler_variants=gen_sampler_variants, ref_modules=gen_ref_modules)
WITHOUT_REFERENCE = {'sampler_variants', 'ref_modules'}     # sections that can fall back to the pinned oracle


def main(argv):
    assert ref_shims.available() or (argv and set(argv) <= WITHOUT_REFERENCE), \
        f'needs the unmodified reference (MSMD_REFERENCE); without it only {sorted(WITHOUT_REFERENCE)}'
    os.makedirs(OUT, exist_ok=True)
    torch.set_grad_enabled(False)
    names = argv or list(SECTIONS)
    for n in names:
        SECTIONS[n]()


if __name__ == '__main__':
    main(sys.argv[1:])
