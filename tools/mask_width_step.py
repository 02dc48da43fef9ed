#!/usr/bin/env python
"""Per-step cost of the cross-attention alignment band: align_mask_width 1 (step-invariant cross attention, cached per
window) against 2 and 0 (banded / unmasked cross attention of every row on every step).

    python tools/mask_width_step.py [--rounds 5] [--replays 200] > profiles/mask_width_step.jsonl

One process builds three default-precision ('hybrid') engines of the configs[2] shape: 64 clips x 3 CFG entries = 192
sequences.  Each engine samples one full window to warm up its bf16 and fp16 step graphs.  Then, alternating the widths
over the rounds:
  * bf16_step_us  = CUDA-event time of `replays` replays of the captured bf16 step graph (t = 500 down), per step;
  * window_step_us = one full 500-step window (bf16 graph replays + fp16 + fp32-grade tail) / 500.
The medians over the rounds are reported.  anim_s_per_s is the sampler-only rate the window time implies
(64 clips x 4 s of motion per window).  It leaves out the audio encoder, style encoder and FLAME decode that bench.py
includes.  One JSON line per width, with the card name, power limit and the SM clock sampled during the timed region."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

from bench import ClockSampler  # noqa: E402
from tools import synth  # noqa: E402

CLIPS, T, WIDTHS = 64, 500, (1, 2, 0)


def build(w):
    from msmd_b200 import model as M
    args = synth.pinned_args(align_mask_width=w)
    m = M.MSMD(args, 'cpu', True, use_head_alpha=False, audio_encoder=nn.Identity())
    m.load_state_dict(synth.fill_state_dict(synth.param_spec(m), 1234), strict=False)
    return m.cuda().eval()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--replays', type=int, default=200)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('mask_width_step: needs a CUDA device')
    dev = torch.device('cuda', 0)
    i = {k: v.to(dev) for k, v in synth.sampler_inputs(CLIPS, T, 17).items()}
    models = {w: build(w) for w in WIDTHS}
    for w, m in models.items():         # warm-up: window caches, bf16 + fp16 step graphs, fp32-grade tail
        m.sample(i['audio_feat'], i['shape'], i['style'], motion_at_T=i['x_T'], indicator=i['indicator'],
                 cfg_scale=1.4, noise=i['z'])
    torch.cuda.synchronize()
    m_k32, m_k16 = models[1]._precise_steps(), models[1]._fp16_steps()   # the same 'auto' schedule for every width

    def timed(eng, n_steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.sample_window(i['x_T'], i['z'], 0, False, 1.4, 1.4, 0.0, t_start=T, n_steps=n_steps,
                          precise_last_steps=m_k32, fp16_last_steps=m_k16)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1000.0 / n_steps

    res = {w: dict(bf16=[], window=[]) for w in WIDTHS}
    with ClockSampler(0) as clk:
        for _ in range(a.rounds):
            for w in WIDTHS:
                m = models[w]
                # the window state (conditioning, caches) of this engine is still the one its warm-up opened
                res[w]['bf16'].append(timed(m._eng, a.replays))
                res[w]['window'].append(timed(m._eng, T))
    q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit', '--format=csv,noheader,nounits'],
                       capture_output=True, text=True).stdout.strip()
    clocks = clk.summary()
    for w in WIDTHS:
        win = statistics.median(res[w]['window'])
        print(json.dumps(dict(
            align_mask_width=w, clips=CLIPS, sequences=3 * CLIPS, precision='hybrid', k32=m_k32, k16=m_k16,
            bf16_step_us=round(statistics.median(res[w]['bf16']), 1), window_step_us=round(win, 1),
            anim_s_per_s=round(CLIPS * 4.0 / (win * T * 1e-6), 1), rounds=a.rounds, replays=a.replays,
            bf16_step_us_all=[round(x, 1) for x in res[w]['bf16']], window_step_us_all=[round(x, 1) for x in res[w]['window']],
            gpu=torch.cuda.get_device_name(dev), power_limit_w=q, sm_clock_mhz=clocks['sm_mhz'],
            sm_clock_max_mhz=clocks['sm_max_mhz'], clock_event_reasons=clocks['reasons'])))


if __name__ == '__main__':
    main()
