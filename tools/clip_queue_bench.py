#!/usr/bin/env python
"""Mixed-length clips: the clip queue (inference.infer_coeffs_many) against one infer_coeffs_batched call per
window-count group.

    python tools/clip_queue_bench.py [--clips 192] [--max-windows 8] [--rounds 3] [--out profiles/clip_queue.jsonl]

Workload: `clips` clips of 16 kHz synthetic audio (tools/synth.clip_audio), each a whole number of windows drawn
uniformly from 1..max_windows (whole windows, so that grouping by window count gives every clip its own exact result
and the two arms compute the same codes); HuBERT audio encoder; the package's default ('hybrid') engine at 500 steps,
3 guidance entries; at most 64 clips per sampler call (the configs[2] batch: 192 sequences).
  (a) grouped: clips grouped by window count, each group in chunks of <= 64 clips: extract_audio_feature +
      infer_coeffs_batched per chunk, global clip ids numbered chunk by chunk;
  (b) queue:   infer_coeffs_many over all clips in the caller's order, with the same global clip ids.
Each arm has its own model (own engine, own step graphs).  After one warm-up run of each, the arms alternate for
`rounds` rounds; the time of a run is the host clock around the whole arm, ending in a device synchronise.
Reported: animation-seconds per second of each arm (sum of clip lengths / 25 fps / time, median over the rounds), the
step-graph shapes of the queue (and of its draining tail, the calls with fewer than 64 clips) and the one-time cost of
the queue's first run (its sampler calls on an engine that exists but has captured no step graph yet, minus the median
warm time of the same calls: per new (format, shape) a graph capture, its instantiation and the eager first step; the
engine itself is created and loaded beforehand by a 2-step call of 64 clips, which runs without graphs, and that call's
time is reported separately as engine_setup_s), the per-clip relative L2 between the arms' codes, and the card
name, power limit and SM clock read in the same run.  One JSON line per arm, then a summary line."""
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

from bench import ClockSampler  # noqa: E402
from tools import synth  # noqa: E402

L, FPS, CHUNK, SEED = 100, 25, 64, 20261020


def build_model(args, device):
    import transformers
    from msmd_b200 import model as M
    from msmd_b200.utils import hubert
    m = M.MSMD(args, 'cpu', True, use_head_alpha=False, audio_encoder=hubert.HubertModel(transformers.HubertConfig()))
    m.load_state_dict(synth.fill_state_dict(synth.param_spec(m, skip=()), 1234), strict=False)
    return m.to(device).eval()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--clips', type=int, default=192)
    ap.add_argument('--max-windows', type=int, default=8)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--steps', type=int, default=500, help='diffusion steps (500 = the released schedule)')
    ap.add_argument('--out', default=None, help='also append the JSON lines to this file')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('clip_queue_bench: needs a CUDA device')
    from msmd_b200.inference import extract_clip_features, infer_coeffs_batched, infer_coeffs_queue, queue_schedule
    dev = torch.device('cuda', 0)
    args = synth.pinned_args(n_diff_steps=a.steps)
    K = a.clips
    windows = torch.randint(1, a.max_windows + 1, (K,), generator=torch.Generator().manual_seed(SEED)).tolist()
    audios = [synth.clip_audio(k, w * L * 640).to(dev) for k, w in enumerate(windows)]
    style = torch.cat([synth.clip_style_eps(k) for k in range(K)]).to(dev)
    shape = torch.zeros(K, 100, device=dev)
    x_T = torch.cat([synth.clip_xT(k) for k in range(K)]).to(dev)
    # arm (a)'s chunks and the global clip id each clip gets there (arm (b) uses the same ids)
    chunks, ids = [], [0] * K
    for w in sorted(set(windows)):
        group = [k for k in range(K) if windows[k] == w]
        for i in range(0, len(group), CHUNK):
            chunk = group[i:i + CHUNK]
            for j, k in enumerate(chunk):
                ids[k] = sum(len(c) for c in chunks) + j
            chunks.append(chunk)
    model_a, model_b = build_model(args, dev), build_model(args, dev)

    def arm_grouped():
        out = [None] * K
        for chunk in chunks:
            wav = torch.stack([audios[k] for k in chunk])
            feat = model_a.extract_audio_feature(wav, windows[chunk[0]] * L)
            codes = infer_coeffs_batched(model_a, args, feat, shape[chunk], style[chunk], cfg_scale=1.4, x_T=x_T[chunk],
                                         noise_seed=SEED, clip_offset=ids[chunk[0]])
            for j, k in enumerate(chunk):
                out[k] = codes[j]
        return out

    def arm_queue_sampler(feats, lens):
        return infer_coeffs_queue(model_b, args, feats, shape, style, lens, x_T, max_clips=CHUNK, clip_ids=ids,
                                  noise_seed=SEED, cfg_scale=1.4)

    def arm_queue():     # = infer_coeffs_many(model_b, args, audios, ...), split to time the sampler part on its own
        feats, lens = extract_clip_features(model_b, args, audios)
        return arm_queue_sampler(feats, lens)

    def timed(fn, *x):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn(*x)
        torch.cuda.synchronize()
        return r, time.perf_counter() - t0

    # queue: warm the audio encoder; create the engine at its full capacity (64 clips x 3 entries) and load its weights
    # with a 2-step call, which runs eagerly (no step graph); then the sampler calls cold (every step graph captured) and warm
    feats_b, lens_b = extract_clip_features(model_b, args, audios)
    torch.cuda.synchronize()
    n0 = min(K, CHUNK)
    _, t_setup = timed(lambda: model_b.sample(torch.stack([f[:L] for f in feats_b[:n0]]), shape[:n0], style[:n0],
                                              motion_at_T=x_T[:n0], indicator=torch.ones(n0, L, device=dev),
                                              cfg_scale=1.4, noise_seed=SEED, n_steps=2))
    _, t_cold = timed(arm_queue_sampler, feats_b, lens_b)
    _, t_warm0 = timed(arm_queue_sampler, feats_b, lens_b)
    arm_grouped()                                               # warm-up of arm (a): its graphs, its encoder
    torch.cuda.synchronize()
    t = dict(grouped=[], queue=[])
    with ClockSampler(0) as clk:
        for _ in range(a.rounds):
            res_a, dt = timed(arm_grouped)
            t['grouped'].append(dt)
            (codes_b, lengths), dt = timed(arm_queue)
            t['queue'].append(dt)
        warm_sampler = [timed(arm_queue_sampler, feats_b, lens_b)[1] for _ in range(2)] + [t_warm0]
    err = [float(((codes_b[k, :lengths[k]].double() - res_a[k].double()).norm() / res_a[k].double().norm()).item())
           for k in range(K)]
    calls = queue_schedule(windows, CHUNK)
    sizes = sorted({len(c) for c in calls})
    tail = [s for s in sizes if s < CHUNK]
    power = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit', '--format=csv,noheader,nounits'],
                           capture_output=True, text=True).stdout.strip()
    clocks = clk.summary()
    anim_s = sum(windows) * L / FPS
    hw = dict(gpu=torch.cuda.get_device_name(dev), power_limit_w=power, sm_clock_mhz=clocks['sm_mhz'],
              sm_clock_max_mhz=clocks['sm_max_mhz'], clock_event_reasons=clocks['reasons'])
    common = dict(clips=K, windows_total=sum(windows), anim_seconds=anim_s, max_clips=CHUNK, sequences=3 * CHUNK,
                  n_diff_steps=a.steps, precision=model_b.precision, k32=model_b._precise_steps(),
                  k16=model_b._fp16_steps(), rounds=a.rounds)
    lines = []
    for arm, calls_n in (('grouped', sum(windows[c[0]] for c in chunks)), ('queue', len(calls))):
        med = statistics.median(t[arm])
        lines.append(dict(arm=arm, sampler_calls=calls_n, seconds=round(med, 3), anim_s_per_s=round(anim_s / med, 1),
                          seconds_all=[round(x, 3) for x in t[arm]], **common, **hw))
    warm = statistics.median(warm_sampler)
    lines.append(dict(summary=True, speedup_queue_over_grouped=round(statistics.median(t['grouped']) / statistics.median(t['queue']), 3),
                      rel_l2_max=max(err), rel_l2_median=statistics.median(err), rel_l2_clip_max=int(max(range(K), key=err.__getitem__)),
                      queue_call_sizes=sizes, tail_call_sizes=tail,
                      step_graphs_queue=2 * len(sizes), step_graphs_tail=2 * len(tail),
                      queue_sampler_cold_s=round(t_cold, 3), queue_sampler_warm_s=round(warm, 3),
                      first_run_overhead_s=round(t_cold - warm, 3), engine_setup_s=round(t_setup, 3),
                      windows_hist={w: windows.count(w) for w in sorted(set(windows))}, **common, **hw))
    for ln in lines:
        print(json.dumps(ln))
    if a.out:
        with open(a.out, 'a') as f:
            for ln in lines:
                f.write(json.dumps(ln) + '\n')


if __name__ == '__main__':
    main()
