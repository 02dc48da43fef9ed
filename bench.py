#!/usr/bin/env python
"""bench.py — benchmark of the msmd_b200 hot path (contract: DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one pass of the hot path over one batch of synthetic input.
Workloads (BASELINE.json configs):
  sampler       configs[2] (default, the configuration `metric` is quoted on): 64 clips x 10 s per GPU through the WHOLE
                path - HuBERT audio encoder, style encoder, 3 windows x 500 CFG sampling steps, FLAME decode.  Arithmetic
                = the package default: every sampling step within 1e-3 of the fp32 reference (bf16 / fp16 / fp32-grade
                schedule).  The default line also carries `flame` (configs[1]) and `pure_bf16_mode` sub-records.
  flame         configs[1]: FLAME decode 8192 frames x 5023 vertices, 300 + 100 betas, fp32
  latency1      configs[0] on the GPU: ONE 10 s clip end to end (launch-bound regime)
  clips1024     configs[3]: 1024 clips x 10 s in total, sharded by clip over the ranks, codes + vertices gathered to
                rank-0 pinned host memory inside the timed region (strong scaling)
  wav2vec2_60s  configs[4]: wav2vec2 encoder, 60 s clips (encoder attention over T = 3000 tokens), 16 clips per GPU
Multi-GPU (torchrun, one rank per GPU): clips / frames are partitioned by rank, no collective on the data path; time =
max over ranks between two barriers.  `--impl reference` times the CPU oracle port of the path on the host cores (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault('HF_HUB_OFFLINE', '1')


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        d['_source'] = 'measured'
        return d
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, _source='fallback')


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(',')])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        sm = sorted(int(float(r[0])) for r in self.rows if len(r) >= 6 and r[0].replace('.', '').isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) >= 6 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 6 and r[2 + k].lower().startswith('active') for r in self.rows)]
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=(max(mx) if mx else None),
                    reasons=reasons, samples=len(sm))


def ncu_traffic(kernel_key):
    """dram read+write bytes per launch of a kernel from the committed `ncu --set full` summary (profiles/), or None."""
    p = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    try:
        return json.load(open(p)).get(kernel_key)
    except Exception:
        return None


DUMP_BYTES = 60 << 20      # --dump-outputs stays under 64 MB, .npy headers included


def dump_outputs(outputs, out_dir, max_bytes=DUMP_BYTES, seed=0):
    """Write each {name: tensor} as out_dir/<name>.npy in float32.  An output larger than an even share of max_bytes keeps
    a fixed seeded sample of its matrices (one per index of all but the last two dims, e.g. one mesh per frame), in
    ascending order: two builds run with the same arguments store the same entries."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = max_bytes // len(outputs)
    for name, t in outputs.items():
        rows = t.reshape(-1, *t.shape[max(1, t.dim() - 2):])
        k = share // (rows[0].numel() * 4)
        assert k > 0, f'{name}: one {tuple(rows.shape[1:])} matrix is larger than its {share}-byte share of the dump'
        if k < rows.shape[0]:
            idx = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(seed))[:k].sort().values
            t = rows[idx.to(rows.device)]
        np.save(os.path.join(out_dir, name + '.npy'), t.detach().float().cpu().numpy())


# --------------------------------------------------------------------------------------------
class FlameWorkload:
    """configs[1]: standalone FLAME lbs decode, 8192 frames x 5023 verts, 300 shape + 100 expr, fp32."""
    name = 'flame'
    metric = 'flame_vertex_frames_per_sec'
    unit = 'frames/s'
    dtype = 'f32 (fp16 two-term split x3 on tcgen05, 22-bit operands; fp32 accumulate / skinning)'
    kernel = 'flame_fused'
    scaling = 'weak'

    def __init__(self, frames=8192):
        self.frames = frames

    def config(self, world):
        return dict(workload='flame_decode_8192x5023_300+100_fp32 (BASELINE configs[1])', frames_per_gpu=self.frames,
                    verts=5023, n_shape=300, n_exp=100, parallelism=f'frames sharded x{world}, no collective',
                    l2_policy='per-step output 494 MB > 126 MB L2 (no reuse between steps)')

    def setup(self, device, rank, world=1):
        from types import SimpleNamespace
        from msmd_b200.utils.flame import FLAME
        from tools import synth
        raw = synth.flame_raw(0, synth.FLAME_V, 400)
        self.model = FLAME(SimpleNamespace(n_shape=300, n_exp=100, flame_lmk_embedding_path=None), raw=raw).to(device)
        host = synth.flame_inputs(self.frames, 300, 100, seed=rank)
        self.host = [t.pin_memory() for t in host]
        self.dev = [t.to(device) for t in host]
        self.host_out = torch.empty((self.frames, synth.FLAME_V, 3), dtype=torch.float32).pin_memory()
        self.device = device

    def units(self, world=1):
        return self.frames * world

    def launches_per_step(self):
        return 2  # flame_pose_kernel + fused blendshape/LBS kernel

    def step(self):
        sh, ex, po, ey = self.dev
        v, _, _ = self.model(sh, ex, po, ey, return_lm2d=False, return_lm3d=False)
        return v

    def profile_step(self):
        return self.step()

    def outputs(self, ret):
        """{name: tensor} of what step() returned."""
        return dict(vertices=ret)

    def step_e2e(self):
        sh, ex, po, ey = [h.to(self.device, non_blocking=True) for h in self.host]
        v, _, _ = self.model(sh, ex, po, ey, return_lm2d=False, return_lm3d=False)
        self.host_out.copy_(v, non_blocking=True)
        return v

    def e2e_bytes(self):
        return sum(h.numel() * 4 for h in self.host), self.host_out.numel() * 4

    def roofline(self, peaks, kernel_ms):
        # fused kernel = three-pass fp16 (two-term split, 22 mantissa bits) tcgen05 GEMM [B,436]x[436,15069] + LBS epilogue.
        # Tensor-bound: 3 passes x 2*B*15069*436 issued 16-bit tensor FLOPs against the measured burst cuBLAS bf16 peak;
        # the HBM floor (SURVEY 8(d): 534 MB minimal traffic at B=8192) is reported next to it.
        B = self.frames
        flops = 2.0 * B * 15069 * 436
        ach = 3.0 * flops / (kernel_ms * 1e-3) / 1e12
        pk = peaks['bf16_tflops']
        alg = B * 400 * 4 + B * 15 * 4 + 15069 * 436 * 4 + B * 15069 * 4
        return dict(bound='tensor', kernel=self.kernel + ' (tcgen05 cta_group::2 kind::f16 x3 + LBS epilogue)', achieved=ach, peak=pk,
                    unit='TFLOP/s', frac=ach / pk, traffic=ncu_traffic('flame_tc_kernel') if B == 8192 else None,
                    peak_source=peaks['_source'] + ' burst cuBLAS bf16; achieved = 3 passes x algorithmic fp32-equivalent FLOPs',
                    algorithmic_flops_per_launch=flops, issued_tensor_flops_per_launch=3.0 * flops, kernel_ms=kernel_ms,
                    hbm=dict(algorithmic_bytes=alg, achieved_gbs=alg / (kernel_ms * 1e-3) / 1e9, peak_gbs=peaks['hbm_gbs'],
                             frac=alg / (kernel_ms * 1e-3) / 1e9 / peaks['hbm_gbs']))

    def cpu_reference(self, seconds=10.0):
        """oracle port (oracle/flame_lbs.py) on the host cores, 512-frame batches like common.py:176-196."""
        from oracle import flame_lbs, synth
        torch.set_num_threads(os.cpu_count())
        assets = synth.flame_assets(0, synth.FLAME_V, 300, 100)
        sh, ex, po, ey = synth.flame_inputs(512, 300, 100, seed=0)
        flame_lbs.flame_forward(assets, sh, ex, po, ey)
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds or n == 0:
            flame_lbs.flame_forward(assets, sh, ex, po, ey)
            n += 512
        dt = time.perf_counter() - t0
        return dict(value=n / dt, unit=self.unit, cores=torch.get_num_threads(), kind='port',
                    sample=f'{n} frames in 512-frame batches, {dt:.1f} s, oracle/flame_lbs.py (torch CPU fp32)')

    def reference_workload(self):
        return 'CPU oracle port (oracle/flame_lbs.py, torch fp32): FLAME.forward on 512-frame batches (common.py:176-196), ' \
               '300 + 100 betas, 5023 vertices'


class SamplerWorkload:
    """Whole-path generation: audio encoder + style encoder + CFG sampling (3 entries, windows x 500 steps) + FLAME decode of
    the generated frames.  `clips` per GPU (weak scaling) or `total_clips` over all ranks (strong scaling, with the host
    gather of codes and vertices inside the timed region)."""
    metric = 'generated_animation_seconds_per_second'
    unit = 'animation-s/s'

    def __init__(self, name='sampler', clips=64, seconds=10.0, audio_model='hubert', total_clips=None, chunk=64,
                 baseline_cfg='configs[2]'):
        self.name, self.clips, self.seconds, self.audio_model = name, clips, seconds, audio_model
        self.total_clips, self.chunk, self.baseline_cfg = total_clips, chunk, baseline_cfg
        self.frames = int(seconds * 25)
        self.n_sub = -(-self.frames // 100)
        self.scaling = 'strong' if total_clips else 'weak'
        self.precision = 'hybrid'
        self.seed = 20261017

    # ---- description
    def dtype_str(self):
        m = self.model
        if m.precision == 'hybrid':
            k32, k16 = m._precise_steps(), m._fp16_steps()
            return (f'bf16 tcgen05 (t > {k16}) + one-pass fp16 tcgen05 ({k32} < t <= {k16}) + fp32-grade fp16x3 (t <= {k32}): '
                    'every sampling step <= 1e-3 rel-L2 of the fp32 reference')
        return {'bf16': 'bf16', 'fp16': 'fp16', 'fp32': 'fp32-grade (fp16x3)'}[m.precision]

    def config(self, world):
        per_gpu = self.clips if not self.total_clips else -(-self.total_clips // world)
        enc = 'HuBERT' if self.audio_model == 'hubert' else 'wav2vec2'
        d = dict(workload=f'{per_gpu} clips x {self.seconds:g} s @ 25 fps per GPU: {enc} audio encoder + style encoder + CFG sampler '
                          f'(3 entries, {self.n_sub} windows x 500 steps) + FLAME decode (BASELINE {self.baseline_cfg})',
                 clips_per_gpu=per_gpu, sequences=3 * min(per_gpu, self.chunk), rows=3 * min(per_gpu, self.chunk) * 111,
                 parallelism=f'clips sharded x{world}, no collective on the data path',
                 audio=f'synthetic 16 kHz audio [{per_gpu}, {int(self.seconds * 16000)}] (sines + noise, normalised)',
                 noise=('externally supplied z [501, clips, 100, 67], shared by the windows; x_T, style eps supplied'
                        if not self.total_clips and self.n_sub <= 3 else
                        'in-kernel Philox step noise keyed by (seed, window, GLOBAL clip id); x_T, style eps supplied per clip'),
                 l2_policy='per-layer activations (qkv 65 MB + h 87 MB + ...) exceed the 126 MB L2 every layer'
                 if per_gpu >= 32 else 'inputs are re-uploaded / re-encoded every step; activations fit L2 at this batch (the regime measured)')
        if self.total_clips:
            d['total_clips'] = self.total_clips
            d['gather'] = 'codes + vertices of every clip land in rank-0 pinned host memory inside the timed region ' \
                          '(NCCL gather of device tensors per 64-clip chunk + async D2H on a copy stream)'
        return d

    # ---- setup
    def setup(self, device, rank, world=1):
        from types import SimpleNamespace
        import transformers
        from msmd_b200 import model as M
        from msmd_b200.style_encoder import get_style_encoder
        from msmd_b200.utils import hubert, wav2vec2
        from msmd_b200.utils.flame import FLAME
        from msmd_b200.parallel import shard_range
        from tools import synth
        from tools.synth import pinned_args
        self.device, self.rank, self.world, self.V = device, rank, world, synth.FLAME_V
        self.args = pinned_args(audio_model=self.audio_model)
        enc = (hubert.HubertModel(transformers.HubertConfig()) if self.audio_model == 'hubert'
               else wav2vec2.Wav2Vec2Model(transformers.Wav2Vec2Config()))
        m = M.MSMD(self.args, 'cpu', True, use_head_alpha=False, audio_encoder=enc)
        m.load_state_dict(synth.fill_state_dict(synth.param_spec(m, skip=()), 1234), strict=False)
        m.precision = m.denoising_net.precision = self.precision
        self.model = m.to(device).eval()
        se = get_style_encoder(self.args, 'vae2')
        se.load_state_dict(synth.fill_state_dict(synth.param_spec(se), 77), strict=False)
        self.style_enc = se.to(device).eval()
        raw = synth.flame_raw(0, synth.FLAME_V, 400)
        self.flame = FLAME(SimpleNamespace(n_shape=300, n_exp=100, flame_lmk_embedding_path=None), raw=raw).to(device)
        if self.total_clips:
            self.lo, self.hi = shard_range(self.total_clips, rank, world)     # contiguous block of GLOBAL clip ids
        else:
            self.lo, self.hi = rank * self.clips, (rank + 1) * self.clips       # results do not depend on the GPU count
        N = self.hi - self.lo
        n_samp = int(self.seconds * 16000)
        ids = range(self.lo, self.hi)
        self.host = dict(audio=torch.stack([synth.clip_audio(i, n_samp) for i in ids]),
                         style_motion=torch.cat([synth.clip_style_motion(i) for i in ids]),
                         style_eps=torch.cat([synth.clip_style_eps(i) for i in ids]), shape=torch.zeros(N, 1, 100),
                         x_T=torch.cat([synth.clip_xT(i) for i in ids]))
        self.use_philox = bool(self.total_clips) or self.n_sub > 3
        if not self.use_philox:
            g = torch.Generator().manual_seed(1000 + rank)
            self.host['z'] = torch.randn(501, N, 100, 67, generator=g)
        self.host = {k: v.pin_memory() for k, v in self.host.items()}
        self.dev = {k: v.to(device) for k, v in self.host.items()}
        if self.total_clips:      # gather target: every clip's codes + vertices in rank-0 pinned host memory
            self.dist = torch.distributed if world > 1 else None
            self.copy_stream = torch.cuda.Stream(device)
            per = -(-self.total_clips // world)
            self.n_chunks = -(-per // self.chunk)
            if rank == 0:
                self.host_out = torch.empty((self.total_clips, self.frames, 67)).pin_memory()
                self.host_verts = torch.empty((self.total_clips, self.frames, synth.FLAME_V, 3)).pin_memory()
                if world > 1:
                    self.g_codes = torch.empty((2, world, self.chunk, self.frames, 67), device=device)
                    self.g_verts = torch.empty((2, world, self.chunk, self.frames, synth.FLAME_V, 3), device=device)
        else:
            self.host_out = torch.empty((N, self.frames, 67)).pin_memory()
            self.host_verts = torch.empty((N, self.frames, synth.FLAME_V, 3)).pin_memory()

    def units(self, world=1):
        n = self.total_clips if self.total_clips else self.clips * world
        return n * self.frames / 25.0

    def launches_per_step(self):
        per_layer = 8                                    # QKV, self-attn, out-proj, LN1/LN2, person-token block, FF1, FF2, LN3
        per_denoise = 1 + 8 * per_layer + 2 + 1          # embed + layers + motion_dec(2) + update (advances the step index)
        batches = 1 if not self.total_clips else -(-(self.hi - self.lo) // self.chunk)
        return batches * (self.n_sub * (500 * per_denoise + 8 * 2 + 12) + 3 + 118 + 22)   # + audio encoder + style encoder

    # ---- one batch of clips [a, b) of this rank's block
    def _run(self, d, a=0, b=None):
        from msmd_b200.inference import infer_coeffs_batched
        from msmd_b200.decode import decode_vertices
        b = d['audio'].shape[0] if b is None else b
        total = self.n_sub * 100
        audio = torch.nn.functional.pad(d['audio'][a:b], (0, total * 640 - d['audio'].shape[1]))   # inference.py:41-45
        audio_feat = self.model.extract_audio_feature(audio, total)                                # inference.py:46
        mu, logvar = self.style_enc._stats(d['style_motion'][a:b])
        style = mu + d['style_eps'][a:b] * torch.exp(0.5 * logvar)                                  # style_encoder.py:209-213
        noise = None if self.use_philox else d['z'][:, a:b]
        if noise is not None and not noise.is_contiguous():
            noise = noise.contiguous()
        codes = infer_coeffs_batched(self.model, self.args, audio_feat, d['shape'][a:b], style,
                                     clip_len=self.frames, cfg_scale=1.4, x_T=d['x_T'][a:b], noise=noise,
                                     noise_seed=self.seed, clip_offset=self.lo + a)
        verts = decode_vertices(self.flame, codes, n_exp=100)
        return codes, verts

    def _run_sharded(self, d):
        """configs[3]: this rank's block in chunks of `chunk` clips; each finished chunk is gathered to rank 0 (device
        buffers, double-buffered) and copied to pinned host memory on a side stream while the next chunk samples."""
        n_local = self.hi - self.lo
        per = -(-self.total_clips // self.world)
        cur = torch.cuda.current_stream()
        for ci in range(self.n_chunks):
            a, b = ci * self.chunk, min((ci + 1) * self.chunk, n_local)
            if b > a:
                codes, verts = self._run(d, a, b)
            if self.world == 1:
                ev = torch.cuda.Event()
                ev.record(cur)
                with torch.cuda.stream(self.copy_stream):
                    self.copy_stream.wait_event(ev)
                    self.host_out[a:b].copy_(codes, non_blocking=True)
                    self.host_verts[a:b].copy_(verts, non_blocking=True)
                    codes.record_stream(self.copy_stream)
                    verts.record_stream(self.copy_stream)
                continue
            # every rank contributes a full `chunk`-clip block (zero-padded past the end of its shard)
            full = lambda t, tail: t if (b - a) == self.chunk else torch.cat(
                [t, torch.zeros((self.chunk - max(b - a, 0),) + tail, device=self.device)])
            codes = full(codes if b > a else torch.zeros((0, self.frames, 67), device=self.device), (self.frames, 67))
            verts = full(verts if b > a else torch.zeros((0, self.frames, self.V, 3), device=self.device), (self.frames, self.V, 3))
            slot = ci & 1
            if self.rank == 0 and ci >= 2:
                cur.wait_stream(self.copy_stream)          # slot reuse: the D2H that read it two chunks ago has drained
            self.dist.gather(codes, list(self.g_codes[slot].unbind(0)) if self.rank == 0 else None, dst=0)
            self.dist.gather(verts, list(self.g_verts[slot].unbind(0)) if self.rank == 0 else None, dst=0)
            if self.rank == 0:
                ev = torch.cuda.Event()
                ev.record(cur)
                with torch.cuda.stream(self.copy_stream):
                    self.copy_stream.wait_event(ev)
                    for r in range(self.world):
                        n_r = max(0, min((r + 1) * per, self.total_clips) - r * per)        # clips of rank r
                        cnt = min((ci + 1) * self.chunk, n_r) - a                             # of which in this chunk
                        if cnt > 0:
                            g0 = r * per + a
                            self.host_out[g0:g0 + cnt].copy_(self.g_codes[slot, r, :cnt], non_blocking=True)
                            self.host_verts[g0:g0 + cnt].copy_(self.g_verts[slot, r, :cnt], non_blocking=True)
        cur.wait_stream(self.copy_stream)
        return None

    def step(self):
        if self.total_clips:
            return self._run_sharded(self.dev)
        return self._run(self.dev)

    def outputs(self, ret):
        """{name: tensor} of what step() produced: the codes and vertices it returned, or with total_clips the rank-0 host
        buffers every clip was gathered into."""
        codes, verts = (self.host_out, self.host_verts) if self.total_clips else ret
        return dict(codes=codes, vertices=verts)

    def profile_step(self):
        # 10 eager bf16 sampling steps of the window left open by the last step(): only the per-step GEMMs are timed
        eng = self.model._eng
        n = min(self.chunk, self.hi - self.lo)
        z = None if self.use_philox else self.dev['z'][:, :n].contiguous()
        eng.sample_window(self.dev['x_T'][:n], z, 0, False, 1.4, 1.4, 0.0, t_start=500, n_steps=10)

    def step_time_us(self):
        """one CUDA-graph-replayed bf16 sampling step of the open window (CUDA events around 200 replays)."""
        eng = self.model._eng
        n = min(self.chunk, self.hi - self.lo)
        z = None if self.use_philox else self.dev['z'][:, :n].contiguous()
        eng.sample_window(self.dev['x_T'][:n], z, 0, False, 1.4, 1.4, 0.0, t_start=500, n_steps=20)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        eng.sample_window(self.dev['x_T'][:n], z, 0, False, 1.4, 1.4, 0.0, t_start=500, n_steps=200)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / 200

    def step_e2e(self):
        d = {k: v.to(self.device, non_blocking=True) for k, v in self.host.items()}
        if self.total_clips:
            return self._run_sharded(d)
        codes, verts = self._run(d)
        self.host_out.copy_(codes, non_blocking=True)
        self.host_verts.copy_(verts, non_blocking=True)
        return codes

    def e2e_bytes(self):
        h2d = sum(v.numel() * 4 for v in self.host.values())
        n = self.hi - self.lo
        return h2d, n * self.frames * (67 + 5023 * 3) * 4

    @property
    def kernel(self):
        # dominant kernel = the FF1 GEMM (linear1 + GELU) of the decoder layers: largest single share of the step
        return f'gemm_{3 * min(self.chunk, self.hi - self.lo) * 111}x2048x512'

    def roofline(self, peaks, kernel_ms):
        S = 3 * min(self.chunk, self.hi - self.lo)
        M = S * 111
        flops = 2.0 * M * 2048 * 512                      # algorithmic FLOPs of one launch (SURVEY App. D-1: FFN linear1)
        ach = flops / (kernel_ms * 1e-3) / 1e12
        pk = peaks.get('bf16_tflops_sustained', peaks['bf16_tflops'])
        step_us = self.step_time_us()
        step_flops = S * 5.84e9                           # SURVEY 8(d): 5.84 GFLOP per sequence-step with the exact hoisting
        return dict(bound='tensor', kernel=self.kernel + ' (tcgen05 cta_group::2 bf16, bias+GELU epilogue)', achieved=ach, peak=pk,
                    unit='TFLOP/s', frac=ach / pk, traffic=ncu_traffic('gemm_ff1_pair') if S == 192 else None,
                    peak_source=peaks['_source'] + ' (sustained cuBLAS bf16)', algorithmic_flops_per_launch=flops,
                    kernel_ms=kernel_ms, timing='CUDA events around each launch on its stream, eager steps (msmd_profile_*)',
                    sampling_step=dict(us=step_us, flops=step_flops, tflops=step_flops / step_us / 1e6,
                                       frac=step_flops / step_us / 1e6 / pk,
                                       note='one CUDA-graph-replayed bf16 step of all layers (events around 200 replays)'))

    # ---- CPU baseline: the oracle port of the SAME path on the host cores, bounded sample
    def reference_workload(self):
        return (f'CPU oracle port (oracle/*.py, torch fp32, all host threads) of the same path on a BOUNDED sample: 8 clips x '
                f'{self.seconds:g} s - audio encoder + style encoder + FLAME decode in full, the CFG sampler (24 sequences) for a '
                f'few steps extrapolated to {self.n_sub} windows x 500 steps.  NOT the 64-clip batch the GPU arm runs.')

    def cpu_reference(self, seconds=15.0, clips=8):
        from oracle import audio as OA, decode as OD, denoiser as D, style as OS, synth
        from oracle.ref_shims import pinned_args
        import transformers
        from msmd_b200 import model as M
        from msmd_b200.style_encoder import get_style_encoder
        from msmd_b200.utils import hubert, wav2vec2
        torch.set_num_threads(os.cpu_count())
        args = pinned_args(audio_model=self.audio_model)
        enc = (hubert.HubertModel(transformers.HubertConfig()) if self.audio_model == 'hubert'
               else wav2vec2.Wav2Vec2Model(transformers.Wav2Vec2Config()))
        m = M.MSMD(args, 'cpu', True, use_head_alpha=False, audio_encoder=enc)
        m.load_state_dict(synth.fill_state_dict(synth.param_spec(m, skip=()), 1234), strict=False)
        sd = {k: v.detach() for k, v in m.state_dict().items()}
        se = get_style_encoder(args, 'vae2')
        se.load_state_dict(synth.fill_state_dict(synth.param_spec(se), 77), strict=False)
        ssd = {k: v.detach() for k, v in se.state_dict().items()}
        total = self.n_sub * 100
        secs_audio = min(self.seconds, 12.0)          # the encoder cost per second of audio is measured on <= 12 s
        with torch.no_grad():
            t0 = time.perf_counter()
            audio = torch.stack([synth.clip_audio(i, int(secs_audio * 16000)) for i in range(clips)])
            n_sub_a = -(-int(secs_audio * 25) // 100)
            audio = torch.nn.functional.pad(audio, (0, n_sub_a * 64000 - audio.shape[1]))
            t0 = time.perf_counter()
            feat = OA.extract_audio_feature(sd, audio, 25, n_sub_a * 100)
            t_audio = (time.perf_counter() - t0) * (total / (n_sub_a * 100))
            t0 = time.perf_counter()
            mu, logvar = OS.style_stats(ssd, torch.cat([synth.clip_style_motion(i) for i in range(clips)]))
            style = mu + torch.cat([synth.clip_style_eps(i) for i in range(clips)]) * torch.exp(0.5 * logvar)
            t_style = time.perf_counter() - t0
            i = synth.sampler_inputs(clips, 500, 0)
            kw = dict(x_T=i['x_T'], z=i['z'], indicator=i['indicator'], cfg_scale=1.4)
            D.sample(sd, args, feat[:, :100], i['shape'], style, n_steps=1, **kw)
            n, t0 = 0, time.perf_counter()
            while time.perf_counter() - t0 < seconds or n == 0:
                D.sample(sd, args, feat[:, :100], i['shape'], style, n_steps=2, **kw)
                n += 2
            dt = time.perf_counter() - t0
            t_sampler = dt / n * 500 * self.n_sub
            assets = synth.flame_assets(0, synth.FLAME_V, 300, 100)
            codes = torch.randn(clips, min(self.frames, 250), 67)
            t0 = time.perf_counter()
            OD.decode_vertices(assets, codes, 300, 100)
            t_flame = (time.perf_counter() - t0) * self.frames / codes.shape[1]
        per_batch = t_audio + t_style + t_sampler + t_flame
        return dict(value=clips * self.seconds / per_batch, unit=self.unit, cores=torch.get_num_threads(), kind='port',
                    seconds_per_8_clips=dict(audio_encoder=t_audio, style_encoder=t_style, sampler_extrapolated=t_sampler,
                                             flame_decode=t_flame),
                    sample=f'{clips} clips: encoders + FLAME decode in full, {n} sampling steps of {3 * clips} sequences in '
                           f'{dt:.1f} s extrapolated to {self.n_sub} x 500; oracle/*.py (torch CPU fp32)')


def make_workload(name):
    if name == 'flame':
        return FlameWorkload()
    if name == 'sampler':
        return SamplerWorkload()
    if name == 'latency1':
        return SamplerWorkload('latency1', clips=1, baseline_cfg='configs[0], run on the GPU')
    if name == 'clips1024':
        return SamplerWorkload('clips1024', total_clips=1024, baseline_cfg='configs[3]')
    if name == 'wav2vec2_60s':
        return SamplerWorkload('wav2vec2_60s', clips=16, seconds=60.0, audio_model='wav2vec2', baseline_cfg='configs[4]')
    raise ValueError(name)


WORKLOADS = ['sampler', 'flame', 'latency1', 'clips1024', 'wav2vec2_60s']
DEFAULT_WORKLOAD = 'sampler'
DEFAULT_STEPS = {'flame': (20, 5), 'sampler': (3, 3), 'latency1': (5, 3), 'clips1024': (2, 3), 'wav2vec2_60s': (2, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None)
    ap.add_argument('--warmup', type=int, default=None)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default=DEFAULT_WORKLOAD, choices=WORKLOADS)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip the flame / pure-bf16 sub-records of the default line')
    ap.add_argument('--precision', default='hybrid', choices=['hybrid', 'bf16', 'fp16', 'fp32'],
                    help="sampler arithmetic; 'hybrid' (default, headline) keeps every step within 1e-3 of the fp32 reference")
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy in float32, '
                         'under 64 MB in all: large outputs keep a fixed seeded sample of their frames')
    a = ap.parse_args()
    if a.steps is None:
        a.steps = DEFAULT_STEPS[a.workload][0]
    if a.warmup is None:
        a.warmup = DEFAULT_STEPS[a.workload][1]
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and a.impl == 'reference':
        ap.error('--dump-outputs writes what the GPU path computed; the reference arm only times the CPU oracle')
    rank = int(os.environ.get('RANK', 0))
    local = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    wl = make_workload(a.workload)

    if a.impl == 'reference':
        if rank != 0:
            return 0
        t0 = time.perf_counter()
        per = max(2.0, min(20.0, 60.0 / max(1, a.steps + a.warmup)))
        for _ in range(a.warmup):
            wl.cpu_reference(per)
        vals = [wl.cpu_reference(per) for _ in range(a.steps)]
        v = sum(x['value'] for x in vals) / len(vals)
        cb = dict(vals[-1], value=v)
        cfg = wl.config(a.gpus)
        cfg['gpu_arm_workload'] = cfg['workload']
        cfg['workload'] = wl.reference_workload()        # what THIS arm actually runs
        print(json.dumps(dict(impl='reference', metric=wl.metric, value=v, unit=wl.unit, n_gpus=a.gpus, steps=a.steps,
                              warmup=a.warmup, ms_per_step=1e3 * (time.perf_counter() - t0) / max(1, a.steps + a.warmup),
                              higher_is_better=True, scaling=wl.scaling, vs_baseline=None, dtype='f32', data='synthetic',
                              config=cfg, cpu_baseline=cb,
                              e2e=dict(value=v, unit=wl.unit, h2d_bytes_per_step=0, d2h_bytes_per_step=0))))
        return 0

    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=device)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    from msmd_b200 import _lib
    if isinstance(wl, SamplerWorkload):
        wl.precision = a.precision
    wl.setup(device, rank, world)
    peaks = load_peaks()
    W = max(3, a.warmup)      # timing rule: at least 3 untimed warm-up steps

    def timed(fn, steps, profile=False, warm=None):
        """(ms of `steps` timed calls of fn, what the last call returned)"""
        for _ in range(W if warm is None else warm):
            fn()
        barrier()
        if profile:
            _lib.lib().msmd_profile_reset()
            _lib.lib().msmd_profile_enable(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - 1):
            fn()
        last = fn()          # only the last result is held: each earlier one is freed before the next step allocates
        e1.record()
        barrier()
        if profile:
            _lib.lib().msmd_profile_enable(0)
        return max_over_ranks(e0.elapsed_time(e1)), last

    def kernel_time(w):
        timed(w.profile_step, 1, profile=True, warm=1)
        kms, kn = _lib.profile_query(w.kernel)
        if kn == 0:                                   # CTA-pair (cta_group::2) launches are tallied under a _pair suffix
            kms, kn = _lib.profile_query(w.kernel + '_pair')
        return kms / max(1, kn)

    with ClockSampler(local) as cs:
        ms, last = timed(wl.step, a.steps)
    clocks = cs.summary()
    if a.dump_outputs and rank == 0:
        dump_outputs(wl.outputs(last), a.dump_outputs)
    del last
    kernel_ms = kernel_time(wl)       # dominant-kernel duration, measured live with CUDA events on the launching stream
    ms_e2e = timed(wl.step_e2e, a.steps, warm=1)[0]
    h2d, d2h = wl.e2e_bytes()
    dtype = wl.dtype_str() if isinstance(wl, SamplerWorkload) else wl.dtype

    out = dict(metric=wl.metric, value=wl.units(world) * a.steps / (ms * 1e-3), unit=wl.unit, n_gpus=world,
               steps=a.steps, warmup=W, ms_per_step=ms / a.steps, higher_is_better=True, scaling=wl.scaling,
               vs_baseline=None, dtype=dtype, data='synthetic', config=wl.config(world), clocks=clocks,
               e2e=dict(value=wl.units(world) * a.steps / (ms_e2e * 1e-3), unit=wl.unit, h2d_bytes_per_step=h2d,
                        d2h_bytes_per_step=d2h),
               gpu_launches=wl.launches_per_step() * a.steps,
               roofline=wl.roofline(peaks, kernel_ms) if kernel_ms > 0 else None)
    if a.workload == 'clips1024' and rank == 0:
        # every clip's codes + vertices arrived in rank 0's pinned host buffers (written by the LAST timed step)
        torch.cuda.synchronize()
        ho, hv = wl.host_out, wl.host_verts
        per_clip = hv.reshape(hv.shape[0], -1).abs().amax(1)
        ok = bool(torch.isfinite(ho).all()) and bool((per_clip > 0).all()) and bool(torch.isfinite(per_clip).all())
        codes0, verts0 = wl._run(wl.dev, 0, min(wl.chunk, wl.hi - wl.lo))       # rank 0's first chunk, recomputed
        same = torch.equal(codes0.cpu(), ho[:codes0.shape[0]]) and torch.equal(verts0.cpu(), hv[:verts0.shape[0]])
        out['gather_check'] = dict(all_clips_present_and_finite=ok, first_chunk_bit_identical_to_recompute=bool(same),
                                   clips=int(ho.shape[0]), host_bytes=int(ho.numel() * 4 + hv.numel() * 4))
    if a.workload == 'latency1':
        out['latency'] = dict(ms_per_clip=ms / a.steps, ms_per_clip_e2e=ms_e2e / a.steps,
                              us_per_sampling_step=out['roofline']['sampling_step']['us'] if out['roofline'] else None,
                              note='one 10 s clip: 3 sequences x 111 tokens = 333 rows per GEMM (launch-bound regime)')
    extras = a.workload == 'sampler' and a.precision == 'hybrid' and not a.no_extras
    if extras:
        # (1) the same workload in pure bf16 (every step one bf16 graph replay): the looser-precision figure, for reference
        wl.model.precision = wl.model.denoising_net.precision = 'bf16'
        ms_b = timed(wl.step, 1, warm=1)[0]
        out['pure_bf16_mode'] = dict(value=wl.units(world) / (ms_b * 1e-3), unit=wl.unit, ms_per_step=ms_b, dtype='bf16',
                                     headline_over_this=(ms_b * a.steps) / ms,
                                     note='misses the 1e-3 per-step tolerance on the last ~9 of 500 steps (x0_hat error 6.5e-3 '
                                          'undamped at small t); the headline mode does not')
        wl.model.precision = wl.model.denoising_net.precision = 'hybrid'
        # (2) configs[1], the second half of BASELINE.json's metric: FLAME vertex frames/s, in the driver-run line
        torch.cuda.empty_cache()
        fw = FlameWorkload()
        fw.setup(device, rank, world)
        ms_f = timed(fw.step, 20, warm=5)[0]
        k_f = kernel_time(fw)
        ms_fe = timed(fw.step_e2e, 10, warm=2)[0]
        fh2d, fd2h = fw.e2e_bytes()
        out['flame'] = dict(metric=fw.metric, value=fw.units(world) * 20 / (ms_f * 1e-3), unit=fw.unit, ms_per_step=ms_f / 20,
                            dtype=fw.dtype, config=fw.config(world),
                            e2e=dict(value=fw.units(world) * 10 / (ms_fe * 1e-3), unit=fw.unit, h2d_bytes_per_step=fh2d,
                                     d2h_bytes_per_step=fd2h, note='PCIe-bound: 494 MB of vertices leave the GPU per step'),
                            roofline=fw.roofline(peaks, k_f) if k_f > 0 else None)
    if rank == 0:
        if world == 1 and not a.no_cpu_baseline:
            out['cpu_baseline'] = wl.cpu_reference(10.0)
            if extras:
                out['flame']['cpu_baseline'] = fw.cpu_reference(5.0)
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
