"""Python handle over the C-ABI denoiser/sampler engine (msmd_create ... msmd_sample_window)."""
import ctypes as C

import torch

from . import _lib


class MsmdConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        'n_motions', 'n_prev_motions', 'd_model', 'n_heads', 'n_layers', 'd_ff', 'd_style', 'd_shape',
        'motion_dim', 'n_basis', 'n_diff_steps', 'use_indicator', 'align_mask_width', 'target_noise',
        'max_seqs', 'precision')]


class SampleExtras(C.Structure):
    _fields_ = [('use_dynamic_threshold', C.c_int), ('dt_ratio', C.c_float), ('dt_min', C.c_float), ('dt_max', C.c_float),
                ('target_dynamic', C.c_void_p), ('cumulative_static', C.c_void_p), ('alpha_traj', C.c_void_p),
                ('precise_last_steps', C.c_int), ('fp16_last_steps', C.c_int), ('noise_clip_offset', C.c_int64),
                ('noise_keys', C.c_void_p)]


class SampleSchedule(C.Structure):
    """msmd_sample_schedule: a HOST int32 list of visited timesteps (strictly decreasing), eta, the solver (0 DDIM,
    1 DPM-Solver++(2M)) and an optional device x0_prev."""
    _fields_ = [('timesteps', C.POINTER(C.c_int32)), ('n_timesteps', C.c_int), ('eta', C.c_float), ('solver', C.c_int),
                ('x0_prev', C.c_void_p)]


SOLVERS = {'ddim': 0, 'dpmpp_2m': 1}


PRECISIONS = {'bf16': 0, 'fp32': 1, 'hybrid': 2, 'fp16': 3}
PATHS = {'bf16': 0, 'fp32': 1, 'fp16': 2}          # msmd_denoise_ex's `precise` argument


class DenoiserEngine:
    """One engine per (device, capacity).  Weights are (re)loaded when the owning module's parameters change."""

    def __init__(self, cfg: dict, device):
        device = torch.device(device)
        if device.type != 'cuda':
            raise _lib.MsmdError('msmd_b200 denoiser needs a CUDA device (no CPU path)')
        self.device = device
        self.cfg = MsmdConfig(**cfg)
        h = C.c_void_p()
        idx = device.index if device.index is not None else torch.cuda.current_device()
        _lib.check(_lib.lib().msmd_create(C.byref(self.cfg), idx, C.byref(h)))
        self._h = h
        self.weights_key = None
        self._keep = None

    def load_state_dict(self, sd):
        """sd: {state_dict key: tensor}; only 'denoising_net.*' and 'diffusion_sched.*' float entries are used."""
        items = [(k, v.detach().to(torch.float32).contiguous()) for k, v in sd.items()
                 if v.is_floating_point() and k.startswith(('denoising_net.', 'diffusion_sched.'))]
        n = len(items)
        names = (C.c_char_p * n)(*[k.encode() for k, _ in items])
        ptrs = (C.c_void_p * n)(*[v.data_ptr() for _, v in items])
        numel = (C.c_int64 * n)(*[v.numel() for _, v in items])
        with torch.cuda.device(self.device):
            torch.cuda.synchronize()
            _lib.check(_lib.lib().msmd_load_weights(self._h, names, ptrs, numel, n))

    def window_begin(self, audio, person, style, prev_motion, prev_audio, indicator, NX, E):
        f = lambda t: None if t is None else t.detach().to(self.device, torch.float32).contiguous()
        audio, person, style, prev_motion, prev_audio, indicator = map(f, (audio, person, style, prev_motion,
                                                                          prev_audio, indicator))
        S = audio.shape[0]
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().msmd_window_begin(self._h, _lib.dev_ptr(audio), _lib.dev_ptr(person),
                                                    _lib.dev_ptr(style), _lib.dev_ptr(prev_motion),
                                                    _lib.dev_ptr(prev_audio), _lib.dev_ptr(indicator), S, NX, E,
                                                    _lib.stream_ptr()))
        self.S, self.NX, self.E = S, NX, E

    def _path(self, precise):
        """precise: None = the most accurate arithmetic the engine holds (fp32-grade on 'fp32' / 'hybrid' engines);
        True / False = fp32-grade / the engine's 16-bit arithmetic; or a name from PATHS."""
        p = self.cfg.precision
        if isinstance(precise, str):
            return PATHS[precise]
        if precise is None:
            precise = p in (1, 2)
        return 1 if precise else (2 if p == 3 else 0)

    def _steps(self, steps):
        steps = steps.detach().to(torch.int64)
        if not steps.is_cuda:   # host-side step indices are range-checked before they index the embedding table
            if steps.numel() and (int(steps.min()) < 0 or int(steps.max()) > self.cfg.n_diff_steps):
                raise IndexError(f'diffusion step outside [0, {self.cfg.n_diff_steps}]')
        return steps.to(self.device).contiguous()

    def denoise(self, motion, steps, precise=None):
        motion = motion.detach().to(self.device, torch.float32).contiguous()
        steps = self._steps(steps)
        c = self.cfg
        out = torch.empty((self.S, c.n_prev_motions + c.n_motions, c.motion_dim), device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().msmd_denoise_ex(self._h, _lib.dev_ptr(motion), _lib.dev_ptr(steps, torch.int64),
                                                  _lib.dev_ptr(out), self._path(precise), _lib.stream_ptr()))
        return out

    def denoise_parts(self, motion, steps, precise=None):
        """keep_separate=True outputs (model.py:972-973): (dynamic [S,Lp+L,dm], static [S,Lp+L,nb,dm], alphas [S,Lp+L,nb])."""
        motion = motion.detach().to(self.device, torch.float32).contiguous()
        steps = self._steps(steps)
        c = self.cfg
        R = c.n_prev_motions + c.n_motions
        dyn = torch.empty((self.S, R, c.motion_dim), device=self.device)
        sta = torch.empty((self.S, R, c.n_basis, c.motion_dim), device=self.device)
        alp = torch.empty((self.S, R, c.n_basis), device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().msmd_denoise_parts(self._h, _lib.dev_ptr(motion), _lib.dev_ptr(steps, torch.int64),
                                                     _lib.dev_ptr(dyn), _lib.dev_ptr(sta), _lib.dev_ptr(alp),
                                                     self._path(precise), _lib.stream_ptr()))
        return dyn, sta, alp

    def check(self):
        """Synchronise and raise if an earlier fp32-grade call overflowed its operand split."""
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().msmd_check(self._h, _lib.stream_ptr()))

    def sample_window(self, x_T, z=None, seed=0, cfg_independent=False, scale0=0.0, scale1=0.0, flexibility=0.0,
                      t_start=None, n_steps=None, want_traj=False, dynamic_threshold=None, separate=False,
                      precise_last_steps=0, fp16_last_steps=0, noise_clip_offset=0, noise_keys=None, timesteps=None,
                      eta=0.0, solver='ddim', x0_prev=None):
        """noise_keys: int64 [N, 2] (seed, global clip id) per clip, keying each clip's in-kernel noise on its own
        (``seed`` and ``noise_clip_offset`` are then unused).  The library rejects it together with ``z``.
        timesteps: strictly decreasing visited steps of a respaced (DDIM) schedule with ``eta`` in [0, 1], or None for
        the default loop t_start, t_start - 1, ...  On a schedule t_start defaults to its first entry and n_steps to the
        entries from t_start on; ``traj`` then holds x_s at each visited successor s.  solver: 'ddim' or 'dpmpp_2m'
        (needs timesteps); x0_prev: [N, L, dm] data prediction of the list entry before t_start ('dpmpp_2m')."""
        c = self.cfg
        x_T = x_T.detach().to(self.device, torch.float32).contiguous()
        sched = ts = None
        if solver not in SOLVERS:
            raise ValueError(f'solver must be one of {sorted(SOLVERS)}, got {solver!r}')
        if x0_prev is not None:
            x0_prev = x0_prev.detach().to(self.device, torch.float32).contiguous()
            if x0_prev.shape != x_T.shape:
                raise ValueError(f'x0_prev must be [N, L, d] = {tuple(x_T.shape)}, got {tuple(x0_prev.shape)}')
        if timesteps is None and (solver != 'ddim' or x0_prev is not None):
            raise ValueError("solver='dpmpp_2m' and x0_prev need a respaced schedule: pass timesteps")
        if timesteps is not None:
            ts = (C.c_int32 * len(timesteps))(*[int(t) for t in timesteps])
            sched = SampleSchedule(ts, len(timesteps), float(eta), SOLVERS[solver], _lib.dev_ptr(x0_prev).value)
            t_start = int(timesteps[0]) if t_start is None else t_start
            if n_steps is None:
                later = [i for i, t in enumerate(timesteps) if int(t) == t_start]
                n_steps = len(timesteps) - later[0] if later else 1   # t_start off the list: the library rejects it
        t_start = c.n_diff_steps if t_start is None else t_start
        n_steps = t_start if n_steps is None else n_steps
        if z is not None:
            z = z.detach().to(self.device, torch.float32).contiguous()
            if tuple(z.shape) != (c.n_diff_steps + 1,) + tuple(x_T.shape):
                raise ValueError(f'noise must be [T+1, N, L, d] = {(c.n_diff_steps + 1,) + tuple(x_T.shape)}, got {tuple(z.shape)}')
        if noise_keys is not None:
            if noise_keys.dtype != torch.int64 or tuple(noise_keys.shape) != (x_T.shape[0], 2):
                raise ValueError(f'noise_keys must be int64 [N, 2] = {(x_T.shape[0], 2)}, got {noise_keys.dtype} '
                                 f'{tuple(noise_keys.shape)}')
            noise_keys = noise_keys.to(self.device).contiguous()
        out = torch.empty_like(x_T)
        traj = torch.zeros((c.n_diff_steps + 1,) + tuple(x_T.shape), device=self.device) if want_traj else None
        ex = SampleExtras()
        ex.precise_last_steps = int(precise_last_steps)
        ex.fp16_last_steps = int(fp16_last_steps)
        ex.noise_clip_offset = int(noise_clip_offset)
        ex.noise_keys = _lib.dev_ptr(noise_keys, torch.int64, 'noise_keys').value
        sep = None
        if dynamic_threshold:
            ex.use_dynamic_threshold = 1
            ex.dt_ratio, ex.dt_min, ex.dt_max = [float(v) for v in dynamic_threshold]
        if separate:
            sep = (torch.empty_like(x_T), torch.empty_like(x_T),
                   torch.empty((n_steps,) + tuple(x_T.shape[:2]) + (c.n_basis,), device=self.device))
            ex.target_dynamic, ex.cumulative_static, ex.alpha_traj = [t.data_ptr() for t in sep]
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().msmd_sample_window_sched(self._h, _lib.dev_ptr(x_T), _lib.dev_ptr(z), C.c_uint64(seed),
                                                           int(cfg_independent), float(scale0), float(scale1),
                                                           float(flexibility), int(t_start), int(n_steps),
                                                           _lib.dev_ptr(out), _lib.dev_ptr(traj), C.byref(ex),
                                                           None if sched is None else C.byref(sched), _lib.stream_ptr()))
        return (out, traj, sep) if separate else (out, traj)

    def __del__(self):
        try:
            if self._h:
                _lib.lib().msmd_destroy(self._h)
                self._h = None
        except Exception:
            pass
