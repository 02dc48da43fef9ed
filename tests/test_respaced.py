"""Sampling on respaced (DDIM) timestep schedules: MSMD.sample(timesteps=, eta=) -> msmd_sample_window_sched.

CPU: the uniform respacing, the oracle's respaced sampler against the default one at eta = 1 on the full list, eta = 0
determinism, the hybrid segment bounds, argument validation and the C struct layout.
GPU: the engine against the default path and the oracle, noise keying, state left behind, the benchmark shape.

Identity note: at eta = 1 on the full list t = T..1 the respaced step is the posterior step only when
alpha_t = alpha_bar_t / alpha_bar_{t-1}.  The fp32 buffers of the cosine schedule break that in the last bits, and
1 - alpha_t ~ 1e-4 at small t amplifies it to ~1e-4 in the x0_hat coefficient at t = 2..10.  So the identity is checked
on exact_schedule(), a schedule whose fp32 tables satisfy it exactly; the cosine schedule is checked against the oracle."""
import ctypes
import os
import shutil
import subprocess

import pytest
import torch

from conftest import ROOT, rel_l2
from helpers import cpu_state_dict, make_msmd
from oracle import denoiser as D, synth
from respaced_oracle import sample_respaced

F32_TOL = 1e-5
L = 100


def exact_schedule(T):
    """Schedule buffers with alpha_bar_t = alpha_t * alpha_bar_{t-1} exactly in fp32: alpha_1 = 15/16, alpha_2 = 7/8,
    alpha_t = 3/4 after (the products need 4 + 3 + 1.6 (T - 2) mantissa bits: T <= 12)."""
    assert T <= 12
    a = torch.tensor([1.0, 15 / 16, 7 / 8] + [0.75] * (T - 2), dtype=torch.float64)[:T + 1]
    ab = torch.cumprod(a, 0)
    assert torch.equal(ab.float().double(), ab)
    b = 1 - a
    inflex = torch.zeros(T + 1, dtype=torch.float32)
    abf, bf = ab.float(), b.float()
    for t in range(1, T + 1):
        inflex[t] = ((1 - abf[t - 1]) / (1 - abf[t])) * bf[t]
    return dict(betas=bf, alphas=a.float(), alpha_bars=abf, sigmas_flex=torch.sqrt(bf), sigmas_inflex=torch.sqrt(inflex))


def exact_msmd(device, T=12, **kw):
    m, args = make_msmd(device, n_diff_steps=T, **kw)
    with torch.no_grad():
        for k, v in exact_schedule(T).items():
            getattr(m.diffusion_sched, k).copy_(v)
    return m, args


# --------------------------------------------------------------------------------------------------------------- CPU
def test_respaced_timesteps():
    from msmd_b200.model import respaced_timesteps
    assert respaced_timesteps(500, 500) == list(range(500, 0, -1))
    assert respaced_timesteps(500, 50) == list(range(500, 0, -10))
    for T in (12, 500, 1000):
        for k in range(1, T + 1):
            ts = respaced_timesteps(T, k)
            assert len(ts) == k and len(set(ts)) == k and ts[0] == T and ts[-1] >= 1
            assert all(a > b for a, b in zip(ts, ts[1:]))
    for bad in (0, 501):
        with pytest.raises(ValueError):
            respaced_timesteps(500, bad)


@pytest.mark.parametrize('target', ['sample', 'noise'])
@pytest.mark.parametrize('mode', ['incremental', 'independent'])
def test_oracle_eta1_full_list_equals_sample(target, mode):
    """eta = 1 on t = T..1 is the posterior step (on a schedule whose fp32 tables are consistent): teacher-forced single
    steps from the default trajectory, and (target 'sample') the free-running trajectory."""
    T = 12
    m, args = exact_msmd('cpu', T, target=target)
    sd = cpu_state_dict(m)
    i = synth.sampler_inputs(2, T, 22)
    kw = dict(indicator=i['indicator'], cfg_mode=mode, cfg_scale=[1.4, 1.7])
    full = list(range(T, 0, -1))
    traj, _, _ = D.sample(sd, args, i['audio_feat'], i['shape'], i['style'], x_T=i['x_T'], z=i['z'], ret_traj=True, **kw)
    for t in range(T, 0, -1):
        got, _, _ = sample_respaced(sd, args, i['audio_feat'], i['shape'], i['style'], full, 1.0, x_T=traj[t], z=i['z'],
                                      t_start=t, n_steps=1, **kw)
        want, _, _ = D.sample(sd, args, i['audio_feat'], i['shape'], i['style'], x_T=traj[t], z=i['z'], t_start=t,
                              n_steps=1, **kw)
        assert rel_l2(got, want) < 1e-6, (t, rel_l2(got, want))
    if target == 'sample':
        rt, _, _ = sample_respaced(sd, args, i['audio_feat'], i['shape'], i['style'], full, 1.0, x_T=i['x_T'], z=i['z'],
                                     ret_traj=True, **kw)
        assert sorted(rt) == list(range(T + 1))
        assert max(rel_l2(rt[t], traj[t]) for t in range(T + 1)) < 1e-6


def test_oracle_eta0_ignores_z():
    T = 12
    m, args = make_msmd('cpu', n_diff_steps=T)
    sd = cpu_state_dict(m)
    i = synth.sampler_inputs(2, T, 3)
    run = lambda z, eta: sample_respaced(sd, args, i['audio_feat'], i['shape'], i['style'], [12, 8, 5, 2], eta,
                                           x_T=i['x_T'], z=z, indicator=i['indicator'], cfg_scale=[1.4, 1.7])[0]
    assert torch.equal(run(i['z'], 0.0), run(torch.randn_like(i['z']), 0.0))
    assert not torch.equal(run(i['z'], 0.5), run(torch.randn_like(i['z']), 0.5))


def test_hybrid_segment_bounds():
    """On the 500-step cosine schedule, K = 50: fp32-grade for t <= 10 and fp16 for t <= 90 at eta = 0, t <= 30 / 200 at
    eta = 1; the default loop keeps 2 / 16."""
    from msmd_b200.model import respaced_timesteps
    m, _ = make_msmd('cpu', precision=None)
    ts = respaced_timesteps(500, 50)
    assert (m._precise_steps(None, ts, 0.0), m._fp16_steps(None, ts, 0.0)) == (10, 90)
    assert (m._precise_steps(None, ts, 1.0), m._fp16_steps(None, ts, 1.0)) == (30, 200)
    assert (m._precise_steps(), m._fp16_steps()) == (2, 16)
    assert m.auto_steps(m.FP16_ERR_BOUND, timesteps=ts, eta=0.0) == 10


def test_sample_argument_validation():
    m, _ = make_msmd('cpu', n_diff_steps=12)
    i = synth.sampler_inputs(1, 12, 1)
    call = lambda **kw: m.sample(i['audio_feat'], i['shape'], i['style'], indicator=i['indicator'], **kw)
    cases = [(dict(eta=0.5), 'eta applies'),
             (dict(timesteps=[12, 6], flexibility=0.5), 'flexibility'),
             (dict(timesteps=[12, 6, 6]), 'strictly decreasing'),
             (dict(timesteps=[6, 12]), 'strictly decreasing'),
             (dict(timesteps=[13, 6]), 'strictly decreasing'),
             (dict(timesteps=[12, 0]), 'strictly decreasing'),
             (dict(timesteps=[]), 'strictly decreasing'),
             (dict(timesteps=[12, 6], eta=1.5), 'eta must be'),
             (dict(timesteps=[12, 6], eta=-0.1), 'eta must be'),
             (dict(timesteps=[12, 6], t_start=7), 't_start')]
    for kw, msg in cases:
        with pytest.raises(ValueError, match=msg):
            call(**kw)


def test_schedule_layout_matches_c_header(tmp_path):
    from msmd_b200._engine import SampleSchedule
    gcc = shutil.which('gcc')
    assert gcc, 'gcc is part of the image'
    src = tmp_path / 'layout.c'
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "msmd_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu\\n", sizeof(msmd_sample_schedule), '
                   'offsetof(msmd_sample_schedule, timesteps), offsetof(msmd_sample_schedule, n_timesteps), '
                   'offsetof(msmd_sample_schedule, eta)); return 0; }\n')
    exe = str(tmp_path / 'layout')
    subprocess.run([gcc, '-std=c99', '-Wall', '-Werror', '-I', os.path.join(ROOT, 'include'), str(src), '-o', exe], check=True)
    got = list(map(int, subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()))
    assert got == [ctypes.sizeof(SampleSchedule), SampleSchedule.timesteps.offset, SampleSchedule.n_timesteps.offset,
                   SampleSchedule.eta.offset]


# --------------------------------------------------------------------------------------------------------------- GPU
PATHS = {'bf16': (0, 0), 'fp16': (0, 12), 'fp32': (12, 12)}     # (precise_last_steps, fp16_last_steps) of a 12-step model


@pytest.mark.gpu
@pytest.mark.parametrize('target', ['sample', 'noise'])
@pytest.mark.parametrize('mode', ['incremental', 'independent'])
def test_eta1_full_list_equals_default_path(built_lib, target, mode):
    """Teacher-forced single steps in each arithmetic of the hybrid engine: the respaced step at eta = 1 on the full list
    equals the default step within 1e-6; a free-running fp32-engine window within 1e-5."""
    T = 12
    m, args = exact_msmd('cuda', T, precision=None, target=target)
    i = {k: v.cuda() for k, v in synth.sampler_inputs(2, T, 22).items()}
    full = list(range(T, 0, -1))
    kw = dict(indicator=i['indicator'], cfg_mode=mode, cfg_scale=[1.4, 1.7], noise=i['z'])
    run = lambda x, **k2: m.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=x, **kw, **k2)[0]
    for path, (k32, k16) in PATHS.items():
        worst = 0.0
        for t in range(T, 0, -1):
            x = i['x_T'] * (0.3 + 0.7 * t / T)
            pk = dict(t_start=t, n_steps=1, precise_last_steps=k32, fp16_last_steps=k16)
            a, b = run(x, **pk), run(x, timesteps=full, eta=1.0, **pk)
            worst = max(worst, rel_l2(b, a))
        print(f'{target} {mode} {path}: worst step rel-L2 respaced vs default {worst:.1e}')
        assert worst < 1e-6, (path, worst)
    m.check()
    if target == 'sample':
        m32, _ = exact_msmd('cuda', T, precision='fp32', target=target)
        a = m32.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'], **kw)[0]
        b = m32.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'], timesteps=full, eta=1.0, **kw)[0]
        assert rel_l2(b, a) < F32_TOL


def _oracle_traj(sd, args, i, ts, eta, mode, **kw):
    traj, _, _ = sample_respaced(sd, args, i['audio_feat'], i['shape'], i['style'], ts, eta, x_T=i['x_T'], z=i['z'],
                                   indicator=i['indicator'], cfg_mode=mode, cfg_scale=[1.4, 1.7], ret_traj=True, **kw)
    return traj


@pytest.mark.gpu
@pytest.mark.parametrize('eta', [0.0, 0.5])
@pytest.mark.parametrize('target,mode', [('sample', 'incremental'), ('sample', 'independent'), ('noise', 'incremental')])
def test_k50_teacher_forced_steps_vs_oracle(built_lib, eta, target, mode):
    """Every visited step of K = 50 on the 500-step cosine schedule, teacher-forced from the oracle's trajectory: the
    default engine within 1e-3 (1e-5 on its fp32-grade steps), the fp32 engine within 1e-5.  Target 'noise' carries the
    network error eps_err scaled by |c1| |eps_hat| / |x_s| (c1 ~ 1e3 at t = 500, where alpha_bar ~ 1e-8): the bound adds
    that term."""
    from msmd_b200.model import respaced_timesteps, respaced_coefficients
    T = 500
    ts = respaced_timesteps(T, 50)
    mh, args = make_msmd('cuda', precision=None, n_diff_steps=T, target=target)
    m32, _ = make_msmd('cuda', precision='fp32', n_diff_steps=T, target=target)
    sd = cpu_state_dict(mh)
    i = synth.sampler_inputs(2, T, 22)
    traj = _oracle_traj(sd, args, i, ts, eta, mode)
    c0, c1, sig = respaced_coefficients(mh.diffusion_sched.alpha_bars, ts, eta, target)
    k32 = mh._precise_steps(None, ts, eta)
    dev = {k: v.cuda() for k, v in i.items()}
    kw = dict(indicator=dev['indicator'], cfg_mode=mode, cfg_scale=[1.4, 1.7], noise=dev['z'], timesteps=ts, eta=eta)
    worst = {'hybrid': 0.0, 'fp32': 0.0}
    for j, t in enumerate(ts):
        s = ts[j + 1] if j + 1 < len(ts) else 0
        x_t, want = traj[t].float(), traj[s]
        out_norm = 0.0
        if target == 'noise':       # |c1 eps_hat| recovered from the oracle step
            zt = i['z'][t].double() if s > 0 else 0.0
            out_norm = float((want - c0[j] * x_t.double() - sig[j] * zt).norm() / want.norm())
        for name, m, tol in (('hybrid', mh, F32_TOL if t <= k32 else 1e-3), ('fp32', m32, F32_TOL)):
            got, _, _ = m.sample(dev['audio_feat'], dev['shape'], dev['style'], motion_at_T=x_t.cuda(), t_start=t,
                                 n_steps=1, **kw)
            err = rel_l2(got, want)
            bound = tol + (2e-5 if tol == F32_TOL else 1e-2) * out_norm
            worst[name] = max(worst[name], err / bound)
            assert err < bound, (name, t, err, bound)
    print(f'K=50 eta={eta} {target} {mode}: worst error / bound', worst)
    mh.check()


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['incremental', 'independent'])
def test_k50_free_running_vs_oracle(built_lib, mode):
    """A free-running K = 50 window of the fp32 engine against the oracle at eta = 0.5 with external noise: every visited
    state, then dynamic thresholding and the sample_separate outputs."""
    from msmd_b200.model import respaced_timesteps
    T = 500
    ts = respaced_timesteps(T, 50)
    m, args = make_msmd('cuda', precision='fp32', n_diff_steps=T)
    sd = cpu_state_dict(m)
    i = synth.sampler_inputs(2, T, 5)
    dev = {k: v.cuda() for k, v in i.items()}
    kw = dict(indicator=dev['indicator'], cfg_mode=mode, cfg_scale=[1.4, 1.7], noise=dev['z'], timesteps=ts, eta=0.5)
    want = _oracle_traj(sd, args, i, ts, 0.5, mode)
    got, _, _ = m.sample(dev['audio_feat'], dev['shape'], dev['style'], motion_at_T=dev['x_T'], ret_traj=True, **kw)
    assert sorted(got) == sorted(ts + [0])
    errs = [rel_l2(got[t], want[t]) for t in ts + [0]]
    print('K=50 fp32 free-running rel-L2, worst / final:', max(errs), errs[-1])
    assert max(errs) < F32_TOL
    dt = (0.9, 1.0, 4.0)
    a = m.sample(dev['audio_feat'], dev['shape'], dev['style'], motion_at_T=dev['x_T'], dynamic_threshold=dt, **kw)[0]
    b, _, _ = sample_respaced(sd, args, i['audio_feat'], i['shape'], i['style'], ts, 0.5, x_T=i['x_T'], z=i['z'],
                                indicator=i['indicator'], cfg_mode=mode, cfg_scale=[1.4, 1.7], dynamic_threshold=dt)
    assert rel_l2(a, b) < F32_TOL
    sep = m.sample_separate(dev['audio_feat'], dev['shape'], dev['style'], motion_at_T=dev['x_T'],
                            indicator=dev['indicator'], cfg_mode=mode, cfg_scale=[1.4, 1.7], noise=dev['z'], timesteps=ts,
                            eta=0.5, return_all_alpha=True)
    ref = sample_respaced(sd, args, i['audio_feat'], i['shape'], i['style'], ts, 0.5, x_T=i['x_T'], z=i['z'],
                            indicator=i['indicator'], cfg_mode=mode, cfg_scale=[1.4, 1.7], separate=True)
    assert sep[5].shape[0] == len(ts) * 2
    for k, tol in ((0, F32_TOL), (3, F32_TOL), (4, F32_TOL), (5, F32_TOL)):
        assert rel_l2(sep[k], ref[k]) < tol, (k, rel_l2(sep[k], ref[k]))


@pytest.mark.gpu
def test_eta0_is_deterministic_and_queue_keys_its_noise(built_lib):
    """eta = 0 draws no noise: two seeds give equal codes.  eta = 0.5: the clip queue (3 clips in flight) gives every
    clip the codes of that clip sampled alone."""
    from msmd_b200.inference import infer_coeffs_batched, infer_coeffs_queue
    from msmd_b200.model import respaced_timesteps
    T = 12
    ts = respaced_timesteps(T, 4)
    m, args = make_msmd('cuda', precision=None, n_diff_steps=T)
    i = {k: v.cuda() for k, v in synth.sampler_inputs(3, T, 9).items()}
    run = lambda seed, eta: m.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'],
                                     indicator=i['indicator'], cfg_scale=1.4, noise_seed=seed, timesteps=ts, eta=eta)[0]
    assert torch.equal(run(1, 0.0), run(2, 0.0))
    assert not torch.equal(run(1, 0.5), run(2, 0.5))
    g = torch.Generator().manual_seed(4)
    windows, pads = [1, 3, 2, 1, 2], [0, 30, 0, 55, 10]
    feats = [torch.randn(w * L, 512, generator=g).cuda() for w in windows]
    lens = [w * L - p for w, p in zip(windows, pads)]
    style = torch.randn(len(windows), 256, generator=g).cuda()
    shape = torch.zeros(len(windows), 100, device='cuda')
    x_T = torch.randn(len(windows), L, 67, generator=g).cuda()
    codes, n = infer_coeffs_queue(m, args, feats, shape, style, lens, x_T, max_clips=3, noise_seed=7, cfg_scale=1.4,
                                  timesteps=ts, eta=0.5)
    for k in range(len(windows)):
        one = infer_coeffs_batched(m, args, feats[k][None], shape[k:k + 1], style[k:k + 1], clip_len=lens[k],
                                   cfg_scale=1.4, x_T=x_T[k:k + 1], noise_seed=7, clip_offset=k, timesteps=ts, eta=0.5)[0]
        assert torch.equal(codes[k, :lens[k]], one), k


@pytest.mark.gpu
def test_respaced_call_leaves_no_state_and_does_not_synchronise(built_lib):
    """A default call after respaced ones equals a fresh engine's, and a respaced call through the cached step graph
    returns long before the stream drains."""
    import time
    from msmd_b200.model import respaced_timesteps
    T, N = 500, 8
    m, args = make_msmd('cuda', n_diff_steps=T)
    i = {k: v.cuda() for k, v in synth.sampler_inputs(N, T, 3).items()}
    run = lambda mm, **kw: mm.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'],
                                     indicator=i['indicator'], cfg_scale=1.4, noise=i['z'], **kw)[0]
    run(m)
    r50 = run(m, timesteps=respaced_timesteps(T, 50), eta=0.5)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    t0 = time.perf_counter()
    r100 = run(m, timesteps=respaced_timesteps(T, 100), eta=0.0)
    host_ms = (time.perf_counter() - t0) * 1e3
    ev1.record()
    drained_at_return = ev1.query()
    torch.cuda.synchronize()
    dev_ms = ev0.elapsed_time(ev1)
    print(f'K=100 window, {3 * N} sequences: host returned after {host_ms:.1f} ms, device busy {dev_ms:.1f} ms')
    assert not drained_at_return and host_ms < 0.6 * dev_ms
    assert torch.equal(run(m, timesteps=respaced_timesteps(T, 50), eta=0.5), r50) and not torch.equal(r50, r100)
    m2, _ = make_msmd('cuda', n_diff_steps=T)
    assert torch.equal(run(m), run(m2))


@pytest.mark.gpu
def test_benchmark_size_k50_teacher_forced_steps_vs_oracle(built_lib):
    """configs[2] shape: 64 clips -> 192 sequences.  Teacher-forced K = 50 steps at eta = 0 at both ends of every segment
    of the hybrid schedule; clips 0 / 31 / 63 against the CPU oracle run on those clips alone."""
    from test_engine_gpu import CHECK, _bench_inputs, _sub
    from msmd_b200.model import respaced_timesteps
    T = 500
    ts = respaced_timesteps(T, 50)
    i = _bench_inputs(T)
    sub = _sub(i, CHECK)
    dev = {k: v.cuda() for k, v in i.items()}
    mh, args = make_msmd('cuda', precision=None, n_diff_steps=T)
    m32, _ = make_msmd('cuda', precision='fp32', n_diff_steps=T)
    sd = cpu_state_dict(mh)
    k32, k16 = mh._precise_steps(None, ts, 0.0), mh._fp16_steps(None, ts, 0.0)
    assert (k32, k16) == (10, 90)
    kw = dict(cfg_mode='incremental', cfg_scale=[1.4, 1.4])
    for t in (500, 250, 100, 90, 20, 10):
        scale = 0.3 + 0.7 * t / T
        want, _, _ = sample_respaced(sd, args, sub['audio_feat'], sub['shape'], sub['style'], ts, 0.0,
                                       x_T=sub['x_T'] * scale, z=sub['z'], indicator=sub['indicator'], t_start=t,
                                       n_steps=1, **kw)
        for name, m, tol in (('hybrid', mh, F32_TOL if t <= k32 else 1e-3), ('fp32', m32, F32_TOL)):
            got, _, _ = m.sample(dev['audio_feat'], dev['shape'], dev['style'], motion_at_T=dev['x_T'] * scale,
                                 indicator=dev['indicator'], noise=dev['z'], t_start=t, n_steps=1, timesteps=ts, eta=0.0,
                                 **kw)
            errs = [rel_l2(got[c], want[j]) for j, c in enumerate(CHECK)]
            print(f't={t:3d} {name:6s} rel-L2 of clips {CHECK}: ' + ' '.join(f'{e:.2e}' for e in errs))
            assert max(errs) < tol, (t, name, errs)
    mh.check()
