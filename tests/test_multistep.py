"""DPM-Solver++(2M) on respaced schedules: MSMD.sample(solver='dpmpp_2m', x0_prev=) -> msmd_sample_window_sched.

CPU: convergence on a Gaussian toy whose probability-flow ODE is closed-form, the first-order identity with DDIM, the
package planner against the float64 reference, the hybrid precision rule, argument validation and the C struct layout.
GPU: the identity in every arithmetic, teacher-forced and free-running windows against the reference, noise keying
and the clip queue, state left behind, and the benchmark shape."""
import ctypes
import math
import os
import shutil
import subprocess

import pytest
import torch

from conftest import ROOT, rel_l2
from helpers import cpu_state_dict, make_msmd
from oracle import synth
from multistep_oracle import respaced_update, sample_multistep
from test_respaced import PATHS, exact_msmd

F32_TOL = 1e-5
L = 100


def _cosine_alpha_bars():
    m, _ = make_msmd('cpu', precision=None)
    return m.diffusion_sched.alpha_bars.double()


# --------------------------------------------------------------------------------------------------------------- CPU
MU, SD, X_T = 0.3, 0.5, 1.3      # data N(MU, SD^2); the start state of the toy


def _toy_x0(x, A):
    """E[x0 | x_t] for Gaussian data: the exact data prediction."""
    return MU + math.sqrt(A) * SD ** 2 / (A * SD ** 2 + 1 - A) * (x - math.sqrt(A) * MU)


def _toy_exact(A_T, A):
    """The probability-flow ODE from x_T = X_T at alpha_bar A_T to alpha_bar A (A = 1: x_0)."""
    return math.sqrt(A) * MU + math.sqrt(A * SD ** 2 + 1 - A) * (X_T - math.sqrt(A_T) * MU) / math.sqrt(A_T * SD ** 2 + 1 - A_T)


def _toy_run(ab, K, solver):
    """The reference's update loop at eta = 0 with the exact x0_hat: {s: x_s} over the visited successors."""
    from msmd_b200.model import respaced_timesteps
    ts = respaced_timesteps(500, K)
    x, prev, out = torch.tensor(X_T, dtype=torch.float64), None, {}
    zero = torch.zeros((), dtype=torch.float64)
    for i, t in enumerate(ts):
        x0 = torch.tensor(_toy_x0(float(x), float(ab[t])), dtype=torch.float64)
        x, prev = respaced_update(ab, ts, i, 0.0, 'sample', x, x0, zero, solver, prev)
        out[ts[i + 1] if i + 1 < K else 0] = float(x)
    return out


def test_gaussian_toy_convergence():
    """2M beats DDIM at every K, by 10x from K = 20 on; observed orders at t = 100 from K = 50 to K = 100."""
    ab = _cosine_alpha_bars()
    exact0 = _toy_exact(float(ab[500]), 1.0)
    for K in (10, 20, 50, 100):
        e_ddim = abs(_toy_run(ab, K, 'ddim')[0] - exact0)
        e_2m = abs(_toy_run(ab, K, 'dpmpp_2m')[0] - exact0)
        print(f'K={K}: |x0 - exact| DDIM {e_ddim:.2e}, 2M {e_2m:.2e}')
        assert e_2m < e_ddim and (K < 20 or e_2m * 10 < e_ddim), (K, e_ddim, e_2m)
    exact100 = _toy_exact(float(ab[500]), float(ab[100]))
    order = {sv: math.log2(abs(_toy_run(ab, 50, sv)[100] - exact100) / abs(_toy_run(ab, 100, sv)[100] - exact100))
             for sv in ('ddim', 'dpmpp_2m')}
    print('observed order at t = 100:', order)
    assert order['dpmpp_2m'] >= 1.6 and 0.9 <= order['ddim'] <= 1.1, order


@pytest.mark.parametrize('target', ['sample', 'noise'])
def test_first_order_step_is_ddim(target):
    """A first-order 2M step has DDIM's coefficients at eta = 0 and eta = 1 (within 1e-12 in float64)."""
    from msmd_b200.model import dpmpp_2m_coefficients, respaced_coefficients, respaced_timesteps
    ab = _cosine_alpha_bars()
    for ts in (respaced_timesteps(500, 20), respaced_timesteps(500, 500), [400, 3, 1]):
        for eta in (0.0, 1.0):
            d0, d1, dsig = respaced_coefficients(ab, ts, eta, target)
            for j in range(len(ts)):
                c0, c1, c2, sig, _, _ = [v[0] for v in dpmpp_2m_coefficients(ab, ts, eta, target, start=j)]
                assert float(c2) == 0.0
                for got, want in ((c0, d0[j]), (c1, d1[j]), (sig, dsig[j])):
                    assert abs(float(got - want)) <= 1e-12 * max(1.0, abs(float(want))), (ts[j], eta, got, want)


@pytest.mark.parametrize('target', ['sample', 'noise'])
@pytest.mark.parametrize('eta', [0.0, 0.5])
def test_planner_matches_reference_update(target, eta):
    """x_s = c0 x_t + c1 out + c2 x0_p + sigma z and x0_t = a x_t + b out against the reference's lambda-form update, on
    random vectors: whole calls, calls from mid-list with and without x0_prev, and the step to s = 0."""
    from msmd_b200.model import dpmpp_2m_coefficients, respaced_timesteps
    ab = _cosine_alpha_bars()
    g = torch.Generator().manual_seed(3)
    ts = respaced_timesteps(500, 20)
    for start, first in ((0, True), (7, True), (7, False), (19, False)):
        c0, c1, c2, sig, a, b = dpmpp_2m_coefficients(ab, ts, eta, target, start=start, first=first)
        prev = None if first else (torch.randn(64, generator=g, dtype=torch.float64),
                                   torch.log(ab[ts[start - 1]].sqrt() / (1 - ab[ts[start - 1]]).sqrt()))
        x = torch.randn(64, generator=g, dtype=torch.float64)
        for j, i in enumerate(range(start, len(ts))):
            out = torch.randn(64, generator=g, dtype=torch.float64)
            z = torch.randn(64, generator=g, dtype=torch.float64) if i + 1 < len(ts) else torch.zeros(64, dtype=torch.float64)
            hp = prev[0] if prev is not None else torch.zeros_like(x)
            want, nprev = respaced_update(ab, ts, i, eta, target, x, out, z, 'dpmpp_2m', prev)
            got = c0[j] * x + c1[j] * out + c2[j] * hp + sig[j] * z
            assert rel_l2(got, want) < 1e-12, (start, first, ts[i], rel_l2(got, want))
            assert rel_l2(a[j] * x + b[j] * out, nprev[0]) < 1e-12
            if i + 1 == len(ts):     # x_0 = x0_t
                assert float(c2[j]) == 0.0 and float(sig[j]) == 0.0
                assert float(c0[j]) == float(a[j]) and float(c1[j]) == float(b[j])
            x, prev = want, nprev
    with pytest.raises(ValueError):
        dpmpp_2m_coefficients(ab, ts, eta, target, start=0, first=False)


def _feasible(m, ts, eta, solver, k32, k16, tol=1e-3):
    w1, w2 = m._output_weights(ts, eta, solver)
    e = lambda t: 0.0 if t <= k32 else (m.FP16_ERR_BOUND if t <= k16 else m.BF16_ERR_BOUND)
    return all(w1[j] * e(ts[j]) + (w2[j] * e(ts[j - 1]) if j else 0.0) <= tol for j in range(len(ts)))


@pytest.mark.parametrize('solver', ['ddim', 'dpmpp_2m'])
@pytest.mark.parametrize('K', [10, 20, 50, 500])
def test_hybrid_rule_feasible_and_minimal(solver, K):
    """The bounds keep every step within tol; lowering either to the next visited step below (or 0) breaks that.
    DDIM keeps the per-step bounds (the largest t whose |c1| err exceeds tol)."""
    from msmd_b200.model import respaced_coefficients, respaced_timesteps
    m, _ = make_msmd('cpu', precision=None)
    ts = respaced_timesteps(500, K)
    k32, k16 = m._precise_steps(None, ts, 0.0, solver), m._fp16_steps(None, ts, 0.0, solver)
    assert k32 in [0] + ts and k16 in [0] + ts and k16 >= k32
    assert _feasible(m, ts, 0.0, solver, k32, k16)
    lower = lambda k: max([t for t in ts if t < k] + [0])
    if k32 > 0:
        assert not _feasible(m, ts, 0.0, solver, lower(k32), ts[0])
    if k16 > k32:
        assert not _feasible(m, ts, 0.0, solver, k32, lower(k16))
    if solver == 'ddim':
        _, c1, _ = respaced_coefficients(m.diffusion_sched.alpha_bars, ts, 0.0, 'sample')
        per_step = lambda err: max([t for t, c in zip(ts, c1.abs().tolist()) if c * err > 1e-3] + [0])
        assert (k32, k16) == (per_step(m.FP16_ERR_BOUND), max(k32, per_step(m.BF16_ERR_BOUND)))


def test_hybrid_bounds_2m_pinned():
    """2M on the 500-step cosine schedule at eta = 0: K = 20 -> (100, 450), 4 fp32-grade, 14 fp16 and 2 bf16 steps;
    K = 50 -> (40, 210).  Its late-step coefficients exceed 1, so it needs more precise steps than DDIM (K = 20: one)."""
    from msmd_b200.model import respaced_timesteps
    m, _ = make_msmd('cpu', precision=None)
    bounds = lambda K, sv: (m._precise_steps(None, respaced_timesteps(500, K), 0.0, sv),
                            m._fp16_steps(None, respaced_timesteps(500, K), 0.0, sv))
    assert bounds(20, 'dpmpp_2m') == (100, 450)
    assert bounds(50, 'dpmpp_2m') == (40, 210)
    ts = respaced_timesteps(500, 20)
    assert [sum(t <= 100 for t in ts), sum(100 < t <= 450 for t in ts), sum(t > 450 for t in ts)] == [4, 14, 2]
    assert sum(t <= bounds(20, 'ddim')[0] for t in ts) == 1


def test_sample_argument_validation():
    m, _ = make_msmd('cpu', n_diff_steps=12)
    i = synth.sampler_inputs(1, 12, 1)
    call = lambda **kw: m.sample(i['audio_feat'], i['shape'], i['style'], indicator=i['indicator'], **kw)
    xp = torch.zeros(1, L, 67)
    cases = [(dict(solver='dpmpp_2m'), 'needs a respaced schedule'),
             (dict(timesteps=[12, 6], solver='dpmpp'), 'solver must be'),
             (dict(timesteps=[12, 6], x0_prev=xp), "x0_prev applies to solver='dpmpp_2m'"),
             (dict(timesteps=[12, 6], solver='dpmpp_2m', t_start=6, x0_prev=torch.zeros(1, L, 66)), 'x0_prev must be'),
             (dict(timesteps=[12, 6], solver='dpmpp_2m', t_start=6, x0_prev=xp), 'x0_prev must be a CUDA tensor'),
             (dict(timesteps=[12, 6], solver='dpmpp_2m', x0_prev=xp), 'x0_prev must be a CUDA tensor')]
    for kw, msg in cases:
        with pytest.raises(ValueError, match=msg):
            call(**kw)
    with pytest.raises(ValueError, match='solver'):
        m.sample_separate(i['audio_feat'], i['shape'], i['style'], indicator=i['indicator'], timesteps=[12, 6],
                          solver='dpmpp_2m')


def test_schedule_layout_matches_c_header(tmp_path):
    from msmd_b200._engine import SampleSchedule
    gcc = shutil.which('gcc')
    assert gcc, 'gcc is part of the image'
    src = tmp_path / 'layout.c'
    fields = ('timesteps', 'n_timesteps', 'eta', 'solver', 'x0_prev')
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "msmd_b200.h"\n'
                   'int main(void) { printf("%zu' + ' %zu' * len(fields) + '\\n", sizeof(msmd_sample_schedule)' +
                   ''.join(f', offsetof(msmd_sample_schedule, {f})' for f in fields) + '); return 0; }\n')
    exe = str(tmp_path / 'layout')
    subprocess.run([gcc, '-std=c99', '-Wall', '-Werror', '-I', os.path.join(ROOT, 'include'), str(src), '-o', exe], check=True)
    got = list(map(int, subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()))
    assert got == [ctypes.sizeof(SampleSchedule)] + [getattr(SampleSchedule, f).offset for f in fields]


# --------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize('target', ['sample', 'noise'])
def test_first_order_step_equals_ddim_on_gpu(built_lib, target):
    """Single-step 2M calls (first order) equal DDIM single-step calls at eta = 0 and 1 within 1e-6, in each arithmetic
    of the hybrid engine, on a schedule whose fp32 tables are exact."""
    T = 12
    m, _ = exact_msmd('cuda', T, precision=None, target=target)
    i = {k: v.cuda() for k, v in synth.sampler_inputs(2, T, 22).items()}
    full = list(range(T, 0, -1))
    kw = dict(indicator=i['indicator'], cfg_mode='incremental', cfg_scale=[1.4, 1.7], noise=i['z'], timesteps=full)
    run = lambda x, **k2: m.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=x, **kw, **k2)[0]
    for path, (k32, k16) in PATHS.items():
        for eta in (0.0, 1.0):
            worst = 0.0
            for t in range(T, 0, -1):
                x = i['x_T'] * (0.3 + 0.7 * t / T)
                pk = dict(t_start=t, n_steps=1, precise_last_steps=k32, fp16_last_steps=k16, eta=eta)
                worst = max(worst, rel_l2(run(x, solver='dpmpp_2m', **pk), run(x, **pk)))
            print(f'{target} {path} eta={eta}: worst step rel-L2 2M vs DDIM {worst:.1e}')
            assert worst < 1e-6, (path, eta, worst)
    m.check()


def _oracle(sd, args, i, ts, eta, mode, x0_hats=None, **kw):
    return sample_multistep(sd, args, i['audio_feat'], i['shape'], i['style'], ts, eta, x_T=i['x_T'], z=i['z'],
                            indicator=i['indicator'], cfg_mode=mode, cfg_scale=[1.4, 1.7], ret_traj=True,
                            x0_hats=x0_hats, **kw)[0]


@pytest.mark.gpu
@pytest.mark.parametrize('eta', [0.0, 0.5])
@pytest.mark.parametrize('target,mode', [('sample', 'incremental'), ('sample', 'independent'), ('noise', 'incremental')])
def test_k20_teacher_forced_steps_vs_oracle(built_lib, eta, target, mode):
    """Every visited step of K = 20 on the 500-step cosine schedule from the reference's x_t and, as x0_prev, its x0_p:
    the default engine within 1e-3 (1e-5 on its fp32-grade steps), the fp32 engine within 1e-5.  Target 'noise' adds
    the allowance of the DDIM test for |c1 eps_hat| / |x_s|."""
    from msmd_b200.model import dpmpp_2m_coefficients, respaced_timesteps
    T = 500
    ts = respaced_timesteps(T, 20)
    mh, args = make_msmd('cuda', precision=None, n_diff_steps=T, target=target)
    m32, _ = make_msmd('cuda', precision='fp32', n_diff_steps=T, target=target)
    sd = cpu_state_dict(mh)
    i = synth.sampler_inputs(2, T, 22)
    x0_hats = {}
    traj = _oracle(sd, args, i, ts, eta, mode, x0_hats)
    k32 = mh._precise_steps(None, ts, eta, 'dpmpp_2m')
    dev = {k: v.cuda() for k, v in i.items()}
    kw = dict(indicator=dev['indicator'], cfg_mode=mode, cfg_scale=[1.4, 1.7], noise=dev['z'], timesteps=ts, eta=eta,
              solver='dpmpp_2m')
    worst = {'hybrid': 0.0, 'fp32': 0.0}
    for j, t in enumerate(ts):
        s = ts[j + 1] if j + 1 < len(ts) else 0
        x_t, want = traj[t].float(), traj[s]
        xp = x0_hats[ts[j - 1]].float() if j else None
        out_norm = 0.0
        if target == 'noise':       # |c1 eps_hat| recovered from the reference step
            c0, _, c2, sig, _, _ = [v[0] for v in dpmpp_2m_coefficients(mh.diffusion_sched.alpha_bars, ts, eta, target,
                                                                        start=j, first=j == 0)]
            zt = i['z'][t].double() if s > 0 else 0.0
            hp = xp.double() if xp is not None else 0.0
            out_norm = float((want - c0 * x_t.double() - c2 * hp - sig * zt).norm() / want.norm())
        for name, m, tol in (('hybrid', mh, F32_TOL if t <= k32 else 1e-3), ('fp32', m32, F32_TOL)):
            got, _, _ = m.sample(dev['audio_feat'], dev['shape'], dev['style'], motion_at_T=x_t.cuda(), t_start=t,
                                 n_steps=1, x0_prev=None if xp is None else xp.cuda(), **kw)
            err = rel_l2(got, want)
            bound = tol + (2e-5 if tol == F32_TOL else 1e-2) * out_norm
            worst[name] = max(worst[name], err / bound)
            assert err < bound, (name, t, err, bound)
    print(f'K=20 2M eta={eta} {target} {mode}: worst error / bound', worst)
    mh.check()


@pytest.mark.gpu
def test_k20_free_running_vs_oracle(built_lib):
    """A free-running K = 20 window of the fp32 engine against the reference: every visited state at eta = 0 and at
    eta = 0.5 with external noise, then with dynamic thresholding."""
    from msmd_b200.model import respaced_timesteps
    T = 500
    ts = respaced_timesteps(T, 20)
    m, args = make_msmd('cuda', precision='fp32', n_diff_steps=T)
    sd = cpu_state_dict(m)
    i = synth.sampler_inputs(2, T, 5)
    dev = {k: v.cuda() for k, v in i.items()}
    mode = 'incremental'
    for eta in (0.0, 0.5):
        kw = dict(indicator=dev['indicator'], cfg_mode=mode, cfg_scale=[1.4, 1.7], noise=dev['z'], timesteps=ts, eta=eta,
                  solver='dpmpp_2m')
        want = _oracle(sd, args, i, ts, eta, mode)
        got, _, _ = m.sample(dev['audio_feat'], dev['shape'], dev['style'], motion_at_T=dev['x_T'], ret_traj=True, **kw)
        assert sorted(got) == sorted(ts + [0])
        errs = [rel_l2(got[t], want[t]) for t in ts + [0]]
        print(f'K=20 2M eta={eta} fp32 free-running rel-L2, worst / final:', max(errs), errs[-1])
        assert max(errs) < F32_TOL
    dt = (0.9, 1.0, 4.0)
    a = m.sample(dev['audio_feat'], dev['shape'], dev['style'], motion_at_T=dev['x_T'], dynamic_threshold=dt, **kw)[0]
    b, _, _ = sample_multistep(sd, args, i['audio_feat'], i['shape'], i['style'], ts, 0.5, x_T=i['x_T'], z=i['z'],
                               indicator=i['indicator'], cfg_mode=mode, cfg_scale=[1.4, 1.7], dynamic_threshold=dt)
    assert rel_l2(a, b) < F32_TOL


@pytest.mark.gpu
def test_2m_deterministic_and_queue_keys_its_noise(built_lib):
    """eta = 0 draws no noise: two seeds give equal codes.  eta = 0.5: the clip queue (3 clips in flight) gives every
    clip bitwise the codes of that clip sampled alone, so the history rows follow the slots and reset per call."""
    from msmd_b200.inference import infer_coeffs_batched, infer_coeffs_queue
    from msmd_b200.model import respaced_timesteps
    T = 12
    ts = respaced_timesteps(T, 5)
    m, args = make_msmd('cuda', precision=None, n_diff_steps=T)
    i = {k: v.cuda() for k, v in synth.sampler_inputs(3, T, 9).items()}
    run = lambda seed, eta: m.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'],
                                     indicator=i['indicator'], cfg_scale=1.4, noise_seed=seed, timesteps=ts, eta=eta,
                                     solver='dpmpp_2m')[0]
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
                                  timesteps=ts, eta=0.5, solver='dpmpp_2m')
    for k in range(len(windows)):
        one = infer_coeffs_batched(m, args, feats[k][None], shape[k:k + 1], style[k:k + 1], clip_len=lens[k],
                                   cfg_scale=1.4, x_T=x_T[k:k + 1], noise_seed=7, clip_offset=k, timesteps=ts, eta=0.5,
                                   solver='dpmpp_2m')[0]
        assert torch.equal(codes[k, :lens[k]], one), k


@pytest.mark.gpu
def test_2m_call_leaves_no_state_and_does_not_synchronise(built_lib):
    """A DDIM call after 2M calls equals a fresh engine's, a 2M call without x0_prev after 2M calls (one with x0_prev)
    equals a fresh engine's, and a 2M call through the cached step graph returns long before the stream drains."""
    import time
    from msmd_b200.model import respaced_timesteps
    T, N = 500, 8
    ts = respaced_timesteps(T, 50)
    m, _ = make_msmd('cuda', n_diff_steps=T)
    i = {k: v.cuda() for k, v in synth.sampler_inputs(N, T, 3).items()}
    run = lambda mm, **kw: mm.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'],
                                     indicator=i['indicator'], cfg_scale=1.4, noise=i['z'], **kw)[0]
    run(m, timesteps=ts, eta=0.5, solver='dpmpp_2m')
    run(m, timesteps=ts, t_start=ts[10], n_steps=5, solver='dpmpp_2m', x0_prev=i['x_T'] * 3.0)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    t0 = time.perf_counter()
    r2m = run(m, timesteps=ts, eta=0.0, solver='dpmpp_2m')
    host_ms = (time.perf_counter() - t0) * 1e3
    ev1.record()
    drained_at_return = ev1.query()
    torch.cuda.synchronize()
    dev_ms = ev0.elapsed_time(ev1)
    print(f'K=50 2M window, {3 * N} sequences: host returned after {host_ms:.1f} ms, device busy {dev_ms:.1f} ms')
    assert not drained_at_return and host_ms < 0.6 * dev_ms
    ddim = run(m, timesteps=ts, eta=0.0)
    m2, _ = make_msmd('cuda', n_diff_steps=T)
    assert torch.equal(run(m2, timesteps=ts, eta=0.0, solver='dpmpp_2m'), r2m)
    assert torch.equal(run(m2, timesteps=ts, eta=0.0), ddim) and not torch.equal(ddim, r2m)


@pytest.mark.gpu
def test_benchmark_size_2m_teacher_forced_steps_vs_oracle(built_lib):
    """configs[2] shape: 64 clips -> 192 sequences.  Teacher-forced K = 20 2M steps (eta = 0, with x0_prev after the
    first) at both ends of every segment of the hybrid schedule; clips 0 / 31 / 63 against the reference run on those
    clips alone."""
    from test_engine_gpu import CHECK, _bench_inputs, _sub
    from msmd_b200.model import respaced_timesteps
    T = 500
    ts = respaced_timesteps(T, 20)
    i = _bench_inputs(T)
    i['x0_prev'] = torch.tanh(i['x_T'].flip(1))
    sub = _sub(i, CHECK)
    sub['x0_prev'] = i['x0_prev'][torch.tensor(CHECK)]
    dev = {k: v.cuda() for k, v in i.items()}
    mh, args = make_msmd('cuda', precision=None, n_diff_steps=T)
    m32, _ = make_msmd('cuda', precision='fp32', n_diff_steps=T)
    sd = cpu_state_dict(mh)
    k32, k16 = mh._precise_steps(None, ts, 0.0, 'dpmpp_2m'), mh._fp16_steps(None, ts, 0.0, 'dpmpp_2m')
    assert (k32, k16) == (100, 450)
    kw = dict(cfg_mode='incremental', cfg_scale=[1.4, 1.4])
    for t in (500, 475, 450, 125, 100, 25):
        scale = 0.3 + 0.7 * t / T
        xp = dict(x0_prev=sub['x0_prev']) if t != ts[0] else {}
        want, _, _ = sample_multistep(sd, args, sub['audio_feat'], sub['shape'], sub['style'], ts, 0.0,
                                      x_T=sub['x_T'] * scale, z=sub['z'], indicator=sub['indicator'], t_start=t,
                                      n_steps=1, **xp, **kw)
        for name, m, tol in (('hybrid', mh, F32_TOL if t <= k32 else 1e-3), ('fp32', m32, F32_TOL)):
            got, _, _ = m.sample(dev['audio_feat'], dev['shape'], dev['style'], motion_at_T=dev['x_T'] * scale,
                                 indicator=dev['indicator'], noise=dev['z'], t_start=t, n_steps=1, timesteps=ts, eta=0.0,
                                 solver='dpmpp_2m', x0_prev=dev['x0_prev'] if xp else None, **kw)
            errs = [rel_l2(got[c], want[j]) for j, c in enumerate(CHECK)]
            print(f't={t:3d} {name:6s} rel-L2 of clips {CHECK}: ' + ' '.join(f'{e:.2e}' for e in errs))
            assert max(errs) < tol, (t, name, errs)
    mh.check()


@pytest.mark.gpu
def test_c_rules_raise(built_lib):
    """The library's own checks, through the engine handle (MSMD_ERR_INVALID -> ValueError): solver outside {0, 1},
    x0_prev with solver 0 or at the list's first entry, and solver 1 with cumulative_static."""
    from msmd_b200._engine import SOLVERS
    T = 12
    m, _ = make_msmd('cuda', n_diff_steps=T)
    i = {k: v.cuda() for k, v in synth.sampler_inputs(1, T, 2).items()}
    m.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'], indicator=i['indicator'], cfg_scale=1.4,
             timesteps=[12, 6, 2])
    eng = m._eng
    x = i['x_T']
    with pytest.raises(ValueError):
        eng.sample_window(x, timesteps=[12, 6, 2], solver='heun')
    SOLVERS['bad'] = 7
    try:
        with pytest.raises(ValueError, match='solver 7'):
            eng.sample_window(x, timesteps=[12, 6, 2], solver='bad')
    finally:
        del SOLVERS['bad']
    with pytest.raises(ValueError, match='x0_prev needs solver 1'):
        eng.sample_window(x, timesteps=[12, 6, 2], t_start=6, x0_prev=x)
    with pytest.raises(ValueError, match="first entry"):
        eng.sample_window(x, timesteps=[12, 6, 2], solver='dpmpp_2m', x0_prev=x)
    with pytest.raises(ValueError, match='cumulative_static'):
        eng.sample_window(x, timesteps=[12, 6, 2], solver='dpmpp_2m', separate=True)
