#!/usr/bin/env python
"""DPM-Solver++(2M) against DDIM on respaced schedules, on the configs[2] workload.

    python tools/multistep_bench.py [--rounds 3] [--out profiles/multistep.jsonl]

Workload: bench.py's `sampler` workload (configs[2]: 64 clips x 10 s, HuBERT audio encoder, style encoder, 3 guidance
entries, the package's default 'hybrid' engine, FLAME decode of every frame), built by bench.SamplerWorkload from
tools/synth.py, with its external noise z.  Arms, each the whole path audio -> vertices, all at eta = 0:
  ddim_K50 / ddim_K25 / ddim_K15 / ddim_K10    DDIM on respaced_timesteps(500, K);
  2m_K25 / 2m_K15 / 2m_K10                     DPM-Solver++(2M) on the same lists.
Reference: the codes of the fp32-grade engine running DDIM at eta = 0 on the full list t = 500..1, i.e. the
probability-flow ODE solved finely.  On the synthetic checkpoint an arm's rel-L2 to it measures solver plus
arithmetic error against that ODE solution, not perceptual quality.
After one warm-up run of each arm, the arms alternate for `rounds` rounds in one process; the time of a run is the host
clock around it, ending in a device synchronise.  Reported per arm: animation-seconds per second (median over the
rounds), the visited steps per arithmetic (bf16 / fp16 / fp32-grade), the rel-L2 of its codes to the reference, and the
card name, power limit and SM clock read in the same run.  One JSON line per arm."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault('HF_HUB_OFFLINE', '1')

import torch  # noqa: E402

from bench import ClockSampler, SamplerWorkload  # noqa: E402


def run_arm(wl, timesteps, eta, solver):
    """SamplerWorkload._run with a schedule and a solver: encoders, sampler, FLAME decode of the generated frames."""
    from msmd_b200.decode import decode_vertices
    from msmd_b200.inference import infer_coeffs_batched
    d = wl.dev
    total = wl.n_sub * 100
    audio = torch.nn.functional.pad(d['audio'], (0, total * 640 - d['audio'].shape[1]))
    audio_feat = wl.model.extract_audio_feature(audio, total)
    mu, logvar = wl.style_enc._stats(d['style_motion'])
    style = mu + d['style_eps'] * torch.exp(0.5 * logvar)
    codes = infer_coeffs_batched(wl.model, wl.args, audio_feat, d['shape'], style, clip_len=wl.frames, cfg_scale=1.4,
                                 x_T=d['x_T'], noise=d.get('z'), noise_seed=wl.seed, clip_offset=wl.lo,
                                 timesteps=timesteps, eta=eta, solver=solver)
    return codes, decode_vertices(wl.flame, codes, n_exp=100)


def segments(m, ts, solver):
    """visited steps per arithmetic of the hybrid schedule: (bf16, fp16, fp32-grade)"""
    k32, k16 = m._precise_steps(None, ts, 0.0, solver), m._fp16_steps(None, ts, 0.0, solver)
    return dict(bf16=sum(t > k16 for t in ts), fp16=sum(k32 < t <= k16 for t in ts), fp32_grade=sum(t <= k32 for t in ts),
                k16=k16, k32=k32)


def set_precision(m, precision):
    m.precision = m.denoising_net.precision = precision


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--out', default=None, help='also append the JSON lines to this file')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('multistep_bench: needs a CUDA device')
    from msmd_b200.model import respaced_timesteps
    dev = torch.device('cuda', 0)
    wl = SamplerWorkload()
    wl.setup(dev, 0)
    m = wl.model
    default_precision = m.precision
    set_precision(m, 'fp32')
    ref = run_arm(wl, respaced_timesteps(500, 500), 0.0, 'ddim')[0].double()
    set_precision(m, default_precision)
    arms = {f'ddim_K{k}': (respaced_timesteps(500, k), 'ddim') for k in (50, 25, 15, 10)}
    arms.update({f'2m_K{k}': (respaced_timesteps(500, k), 'dpmpp_2m') for k in (25, 15, 10)})

    def timed(name):
        ts, solver = arms[name]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = run_arm(wl, ts, 0.0, solver)
        torch.cuda.synchronize()
        return r, time.perf_counter() - t0

    codes = {name: timed(name)[0][0] for name in arms}        # warm-up: step graphs, encoder workspaces
    t = {name: [] for name in arms}
    with ClockSampler(0) as clk:
        for _ in range(a.rounds):
            for name in arms:
                (c, _), dt = timed(name)
                t[name].append(dt)
                codes[name] = c
    m.check()
    power = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit', '--format=csv,noheader,nounits'],
                           capture_output=True, text=True).stdout.strip()
    clocks = clk.summary()
    hw = dict(gpu=torch.cuda.get_device_name(dev), power_limit_w=power, sm_clock_mhz=clocks['sm_mhz'],
              sm_clock_max_mhz=clocks['sm_max_mhz'], clock_event_reasons=clocks['reasons'])
    anim_s = wl.units()
    lines = []
    for name, (ts, solver) in arms.items():
        med = statistics.median(t[name])
        err = float((codes[name].double() - ref).norm() / ref.norm())
        lines.append(dict(arm=name, solver=solver, steps=len(ts), eta=0.0, seconds=round(med, 3),
                          anim_s_per_s=round(anim_s / med, 1), seconds_all=[round(x, 3) for x in t[name]],
                          segments=segments(m, ts, solver), codes_rel_l2_vs_fp32_ode=err,
                          reference='fp32-grade engine, DDIM eta=0, K=500', clips=wl.clips, clip_seconds=wl.seconds,
                          windows=wl.n_sub, anim_seconds=anim_s, rounds=a.rounds, **hw))
    for ln in lines:
        print(json.dumps(ln))
    if a.out:
        with open(a.out, 'a') as f:
            for ln in lines:
                f.write(json.dumps(ln) + '\n')


if __name__ == '__main__':
    main()
