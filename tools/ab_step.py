"""A/B helper: graph-replay time of a sampling step + per-class eager times for chosen kernel classes.
python tools/ab_step.py [class ...]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bench import SamplerWorkload
from msmd_b200 import _lib
CL = int(os.environ.get("MSMD_AB_CLIPS", 64))
wl = SamplerWorkload(clips=CL, seconds=4.0)
wl.precision = os.environ.get("MSMD_PRECISION", "bf16")
wl.setup(torch.device('cuda', 0), 0)
d = dict(wl.dev)
g = torch.Generator(device='cuda').manual_seed(0)
af = torch.randn(CL, 100, 512, device='cuda', generator=g)
st = torch.randn(CL, 256, device='cuda', generator=g)
ind = torch.ones(CL, 100, device='cuda')
m = wl.model
m.sample(af, d['shape'], st, motion_at_T=d['x_T'], indicator=ind, cfg_scale=1.4, noise=d['z'], n_steps=4)
eng = m._eng
best = 1e9
for rep in range(3):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); x, _ = eng.sample_window(d['x_T'], d['z'], 0, False, 1.4, 1.4, 0.0, t_start=500, n_steps=150); e1.record()
    torch.cuda.synchronize()
    best = min(best, e0.elapsed_time(e1) / 150 * 1000)
_lib.lib().msmd_profile_reset(); _lib.lib().msmd_profile_enable(1)
eng.sample_window(d['x_T'], d['z'], 0, False, 1.4, 1.4, 0.0, t_start=500, n_steps=10)
torch.cuda.synchronize()
_lib.lib().msmd_profile_enable(0)
prof = _lib.profile_dump()
sel = ' '.join(f'{k}={prof[k][0] / prof[k][1] * 1000:.1f}us' for k in sys.argv[1:] if k in prof)
print(f'step {best:.1f} us (best of 3 x 150 graph replays)  {sel}  checksum {float(x.double().abs().sum()):.6f}')
