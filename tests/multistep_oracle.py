"""Float64 reference for DPM-Solver++(2M) on respaced schedules, used by tests/test_multistep.py.

It is ``oracle.denoiser.sample`` with the 2M update written out in the lambda form, independently of the package's
planner (``model.dpmpp_2m_coefficients``): the network forward and the CFG entries come from the oracle unchanged, only
the loop over timesteps and the update differ."""
import torch

from oracle.denoiser import cfg_entries, denoiser_forward


def _lam(a):
    return torch.log(torch.sqrt(a) / torch.sqrt(1 - a))


def respaced_update(ab, ts, i, eta, target, x, out, zt, solver='ddim', prev=None):
    """The update of visited step ts[i] (successor s = ts[i + 1], or 0), in float64: x_t, the network output ``out`` and
    the noise z_t (zero when s = 0) -> (x_s, (x0_t, lambda_t)).  ``prev`` is the (x0, lambda) pair of the step before it
    (DPM-Solver++(2M) only; None: first order).  ``ab`` is the float64 alpha_bars table.
    solver='dpmpp_2m': with alpha = sqrt(A), sig = sqrt(1 - A), lam = log(alpha / sig), h = lam_s - lam_t and
    r = (lam_t - lam_p) / h,
      D = x0_t + (x0_t - x0_p) / (2 r)   (D = x0_t without p, and on the step to s = 0, where x_0 = x0_t)
      x_s = (sig_s / sig_t) e^{-eta h} x_t + alpha_s (1 - e^{-(1 + eta) h}) D + sig_s sqrt(1 - e^{-2 eta h}) z_t
    x0_t is the network output for 'sample' and (x_t - sig_t eps_hat) / alpha_t for 'noise'.
    solver='ddim': the DDIM step of tests/respaced_oracle.py (eta is DDIM's eta there)."""
    t = ts[i]
    s = ts[i + 1] if i + 1 < len(ts) else 0
    A, B = ab[t], (ab[s] if s > 0 else torch.ones((), dtype=torch.float64))
    if solver == 'dpmpp_2m':
        al_t, sg_t, lam_t = torch.sqrt(A), torch.sqrt(1 - A), _lam(A)
        x0 = (x - sg_t * out) / al_t if target == 'noise' else out
        if s == 0:
            return x0, (x0, lam_t)
        al_s, sg_s = torch.sqrt(B), torch.sqrt(1 - B)
        h = _lam(B) - lam_t
        D = x0
        if prev is not None:
            r = (lam_t - prev[1]) / h
            D = x0 + (x0 - prev[0]) / (2 * r)
        x_s = sg_s / sg_t * torch.exp(-eta * h) * x + al_s * (1 - torch.exp(-(1 + eta) * h)) * D \
            + sg_s * torch.sqrt(1 - torch.exp(-2 * eta * h)) * zt
        return x_s, (x0, lam_t)
    sigma = eta * torch.sqrt((1 - B) / (1 - A)) * torch.sqrt(torch.clamp(1 - A / B, min=0))
    r = torch.sqrt(torch.clamp(1 - B - sigma ** 2, min=0))
    if target == 'noise':
        c0 = torch.sqrt(B / A)
        c1 = r - torch.sqrt(B) * torch.sqrt(1 - A) / torch.sqrt(A)
    else:
        c0 = r / torch.sqrt(1 - A)
        c1 = torch.sqrt(B) - torch.sqrt(A) * c0
    x0 = (x - torch.sqrt(1 - A) * out) / torch.sqrt(A) if target == 'noise' else out
    return c0 * x + c1 * out + sigma * zt, (x0, None)


def sample_multistep(sd, cfg, audio_feat, shape_coef_or_feat, style_feat, timesteps, eta, prev_motion=None,
                     prev_audio=None, x_T=None, z=None, indicator=None, cfg_mode=None, cfg_cond=None, cfg_scale=1.15,
                     ret_traj=False, n_steps=None, t_start=None, dynamic_threshold=None, x0_prev=None, x0_hats=None):
    """``sample`` with DPM-Solver++(2M) on the strictly decreasing ``timesteps`` (from ``t_start``, default the first
    entry, for ``n_steps`` entries), eta in [0, 1], the update of ``respaced_update``.  The first step is first order
    unless ``x0_prev`` (the data prediction of the entry before t_start) is given.  z_t = z[t] (or torch.randn) is drawn
    only when s > 0.  The network output is the CFG-combined, optionally thresholded output of ``sample``.
    Returns like ``sample``; ret_traj gives {t: x_t} over the visited t and the last successor; the state stays float64.
    ``x0_hats``: a dict that receives x0_t per visited t."""
    N = audio_feat.shape[0]
    sched = {k[len('diffusion_sched.'):]: v for k, v in sd.items() if k.startswith('diffusion_sched.')}
    ab = sched['alpha_bars'].double()
    ts = [int(t) for t in timesteps]
    cfg_mode = cfg_mode or cfg.cfg_mode
    if cfg_cond is None:
        cfg_cond = [c for c in cfg.guiding_conditions.split(',') if c in ('style', 'audio')]
    cfg_cond = [c for c in cfg_cond if c in ('audio', 'style')]
    if not isinstance(cfg_scale, list):
        cfg_scale = [cfg_scale] * len(cfg_cond)
    if cfg_cond:
        cfg_cond, cfg_scale = zip(*sorted(zip(cfg_cond, cfg_scale), key=lambda x: ['audio', 'style'].index(x[0])))
    shape_feat = shape_coef_or_feat
    if style_feat is None:
        style_feat = sd['null_style_feat'].expand(N, -1, -1)
    if shape_feat.ndim == 2:
        shape_feat = shape_feat.unsqueeze(1)
    if style_feat.ndim == 2:
        style_feat = style_feat.unsqueeze(1)
    if prev_motion is None:
        prev_motion = sd['start_motion_feat'].expand(N, -1, -1)
    if prev_audio is None:
        prev_audio = sd['start_audio_feat'].expand(N, -1, -1)
    if x_T is None:
        x_T = torch.randn(N, cfg.n_motions, 67)
    audio_in, person_in = cfg_entries(sd, cfg, audio_feat, shape_feat, style_feat, cfg_mode, cfg_cond)
    E = len(audio_in)
    audio_in = torch.cat(audio_in, 0)
    person_in = torch.cat(person_in, 0)
    pm = torch.cat([prev_motion] * E, 0)
    pa = torch.cat([prev_audio] * E, 0)
    ind = torch.cat([indicator] * E, 0) if indicator is not None else None
    st = torch.cat([style_feat] * E, 0)
    pos = ts.index(t_start if t_start is not None else ts[0])
    visit = ts[pos:pos + n_steps] if n_steps else ts[pos:]
    x = x_T.double()
    prev = (x0_prev.double(), _lam(ab[ts[pos - 1]])) if x0_prev is not None else None
    traj = {visit[0]: x_T}
    for t in visit:
        i = ts.index(t)
        s = ts[i + 1] if i + 1 < len(ts) else 0
        zt = (z[t] if z is not None else torch.randn_like(x_T)).double() if s > 0 else torch.zeros_like(x)
        step = torch.full((N * E,), t, dtype=torch.long)
        res = denoiser_forward(sd, cfg, torch.cat([x.float()] * E, 0), audio_in, person_in, st, pm, pa, step, ind)
        if dynamic_threshold:
            q, lo, hi = dynamic_threshold
            a = res[:, -cfg.n_motions:].reshape(N * E, -1).abs()
            thr = torch.clamp(torch.quantile(a, q, dim=1), min=lo, max=hi)[:, None, None]
            res = torch.clamp(res, min=-thr, max=thr)
        parts = [c[:, -cfg.n_motions:] for c in res.chunk(E)]
        tgt = parts[0]
        for k in range(E - 1):       # the CFG recursion of sample, aliasing included
            ref_k = tgt if (cfg_mode == 'independent' or k == 0) else parts[k]
            tgt = tgt + cfg_scale[k] * (parts[k + 1] - ref_k)
        x, prev = respaced_update(ab, ts, i, eta, cfg.target, x, tgt.double(), zt, 'dpmpp_2m', prev)
        if x0_hats is not None:
            x0_hats[t] = prev[0]
        traj[s] = x
    if ret_traj:
        return traj, x_T, audio_feat
    return x, x_T, audio_feat
