"""The denoiser engine across the architectures and batch sizes msmd_create accepts, against a float64 oracle.

Every other test of the engine runs the released architecture (1 + 10 + 100 tokens, motion_dim 67, 4 bases, d_ff 2048,
8 layers).  Inside the accepted envelope the kernels change code path: self-attention masks every key column at T <= 96
(TAIL16 = false) and only the last 16 above; T = 112 fills the attention tile; the person-token kernel cuts the memory
into 14 parts of 8 keys, some empty when Tk < 104; n_prev_motions = 0 leaves no context rows and an audio-only memory;
motion_dim sets the embedding's K padding, the decoder's N and the dec2 row stride.  Batch sizes move the GEMM tile
dispatch (M = S T: 64-wide tiles up to 512 rows, single-CTA tiles below 2048, CTA pairs above), the attention's jobs per
CTA (8 S jobs on 148 CTAs) and the person-token kernel's sequence groups (16 per group, at most 18 clusters).

CPU: the oracle against the modules' own torch layers in float64 at every configuration used here, and the float32
oracle against the float64 one.  GPU: the forward in all three arithmetics of one hybrid engine and teacher-forced
sampling steps of the default engine, per configuration; then the released architecture at S = 300 ... 1 sequences on
one engine, and a 100-clip (300-sequence) sampling step.  The 16-bit bounds are the ones the hybrid schedule is sized
from (MSMD.BF16_ERR_BOUND / FP16_ERR_BOUND): if they failed at some configuration, the default engine's 1e-3 per-step
contract would fail there too."""
import copy
import ctypes
import time

import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2
from helpers import cpu_state_dict, make_msmd
from oracle import denoiser as D, synth
from oracle.ref_shims import pinned_args

F32_TOL = 1e-5
# id -> overrides of the pinned configuration (T = 1 + n_prev_motions + n_motions tokens, Tk = T - 1 memory keys)
CONFIGS = {
    'A': {},                                                     # T = 111: the released architecture
    'B': dict(n_prev_motions=11),                                # T = 112: full attention tile, 7 keys in the last part
    'C': dict(n_motions=86),                                     # T = 97: smallest T of the TAIL16 kernel
    'D': dict(n_motions=85),                                     # T = 96: largest T of the fully masked kernel
    'E': dict(n_motions=50),                                     # T = 61: empty person-token key parts
    'E-w2': dict(n_motions=50, align_mask_width=2),              # banded cross-attention at a short T
    'F': dict(n_prev_motions=0),                                 # T = 101: no context rows, audio-only memory
    'G': dict(n_motions=1, n_prev_motions=0),                    # T = 2: one key
    'H': dict(n_layers=1, mlp_ratio=1, num_of_basis=1, use_indicator=False, d_style=128),   # d_ff 512, person 228
}
MOTION_DIMS = (50, 54, 76)                                       # 76 + 4 bases = 80 = the dec2 row stride
ALL = list(CONFIGS) + [f'I-dm{dm}' for dm in MOTION_DIMS]       # I: bare network (MSMD itself fixes motion_dim 67)
ARITHMETICS = ('fp32', 'fp16', 'bf16')
N_FWD = 3
BATCHES = (300, 37, 19, 18, 5, 4, 1)                           # descending: one engine created for 300 serves them all
NX_BIG = 100                                                   # clips of the large sampling step (x 3 guidance entries)
CFG_SCALE = [1.4, 1.4]


def _bounds():
    """(whole batch, each sequence) rel-L2 bound per arithmetic: the 16-bit batch margins of test_denoiser_gpu."""
    from msmd_b200.model import MSMD
    return {'fp32': (F32_TOL, F32_TOL), 'fp16': (MSMD.FP16_ERR_BOUND / 1.8, MSMD.FP16_ERR_BOUND),
            'bf16': (MSMD.BF16_ERR_BOUND / 1.3, MSMD.BF16_ERR_BOUND)}


def _build(cid, device, precision=None):
    """(MSMD or None, network, args, oracle key prefix).  precision None = the package default ('hybrid')."""
    if cid.startswith('I-'):
        from msmd_b200.model import DenoisingNetwork_MSMD
        args = pinned_args()
        net = DenoisingNetwork_MSMD(args, 'cpu', motion_feat_dim=int(cid[len('I-dm'):]), use_head_alpha=False)
        _, unexpected = net.load_state_dict(synth.fill_state_dict(synth.param_spec(net)), strict=False)
        assert not unexpected
        if precision is not None:
            net.precision = precision
        return None, net.to(device).eval(), args, ''
    m, args = make_msmd(device, precision=precision, **CONFIGS[cid])
    return m, m.denoising_net, args, 'denoising_net.'


def _forward_inputs(net, N, seed):
    i = synth.denoiser_inputs(N, seed, L=net.n_motions, Lp=net.n_prev_motions, dm=net.motion_feat_dim,
                              d_style=net.style_feat_dim)
    if not net.use_indicator:
        i['indicator'] = None
    return i


def _forward_args(i):
    return [i[k] for k in ('motion', 'audio', 'person', 'style', 'prev_motion', 'prev_audio', 'step', 'indicator')]


def _cast(x, dtype):
    if isinstance(x, dict):
        return {k: _cast(v, dtype) for k, v in x.items()}
    if isinstance(x, list):
        return [_cast(v, dtype) for v in x]
    return x.to(dtype) if isinstance(x, torch.Tensor) and x.is_floating_point() else x


def _oracle(sd, args, i, prefix, dtype=torch.float64, keep_separate=False):
    return D.denoiser_forward(_cast(sd, dtype), args, *_cast(_forward_args(i), dtype), prefix=prefix,
                              keep_separate=keep_separate)


def _seq_errs(got, want):
    return [rel_l2(got[s], want[s]) for s in range(want.shape[0])]


# ------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize('cid', ALL)
def test_oracle_matches_torch_layers_in_float64(cid):
    """oracle.denoiser_forward in float64 against the module's own layers in float64: nn.TransformerDecoder with
    memory_mask = alignment_mask, the static-basis nn.Sequential stacks, with the embedding, motion_dec and the
    basis mix (model.py:945-995) restated around them."""
    m, net, args, prefix = _build(cid, 'cpu')
    sd = cpu_state_dict(m if m is not None else net)
    i = _cast(_forward_inputs(net, N_FWD, 7), torch.float64)
    dyn, sta, alp = _oracle(sd, args, i, prefix, keep_separate=True)
    out = _oracle(sd, args, i, prefix)
    net = copy.deepcopy(net).double().eval()
    N, Lp = i['motion'].shape[0], net.n_prev_motions
    nb = net.num_of_basis
    with torch.no_grad():
        emb = net.diff_step_map(net.TE.pe[0, i['step']]).unsqueeze(1)
        ptok = net.person_proj(i['person']) + emb
        feats = torch.cat([i['prev_motion'], i['motion']], 1)
        if net.use_indicator:
            ind = torch.cat([torch.zeros(N, Lp, dtype=torch.float64), i['indicator']], 1).unsqueeze(-1)
            feats = torch.cat([feats, ind], -1)
        x = torch.cat([ptok, net.feature_proj(feats)], 1) + net.PE
        mem = torch.cat([i['prev_audio'], i['audio']], 1)
        y = net.transformer(x, mem, memory_mask=net.alignment_mask)
        o = net.motion_dec(y[:, 1:])
        static = torch.stack([net.static_feature_mapping[b](i['style'])[:, 0] for b in range(nb)], 1)
    w_dyn, w_alp = o[..., :-nb], o[..., -nb:]
    w_full = w_dyn + torch.cat([w_alp @ static[:, :, :-3], static[:, :, -3:].sum(1, keepdim=True).expand(-1, o.shape[1], -1)],
                               -1)
    errs = [rel_l2(dyn, w_dyn), rel_l2(alp, w_alp), rel_l2(sta, static), rel_l2(out, w_full)]
    assert out.dtype == torch.float64 and out.shape == (N, Lp + net.n_motions, net.motion_feat_dim)
    assert max(errs) < 1e-12, (cid, errs)


@pytest.mark.parametrize('cid', ALL)
def test_float32_oracle_within_2e6_of_float64(cid):
    """The float32 oracle, which the other GPU tests compare with, stays well inside the 1e-5 fp32-grade bound."""
    m, net, args, prefix = _build(cid, 'cpu')
    sd = cpu_state_dict(m if m is not None else net)
    i = _forward_inputs(net, N_FWD, 8)
    err = rel_l2(_oracle(sd, args, i, prefix, torch.float32), _oracle(sd, args, i, prefix))
    assert err < 2e-6, (cid, err)


def test_zero_bases_are_rejected(built_lib):
    """num_of_basis = 0 has no reference result (out[:, :, :-0] is empty, torch.stack([]) raises): the host raises
    before a device is touched, and msmd_create refuses it too."""
    from msmd_b200 import _lib
    from msmd_b200._engine import MsmdConfig
    from msmd_b200.model import _engine_cfg
    m0, _ = make_msmd('cpu', num_of_basis=0)
    with pytest.raises(ValueError, match='num_of_basis=0'):
        _engine_cfg(m0.denoising_net, 500, 'sample', 4, 'hybrid')
    m, _ = make_msmd('cpu')
    cfg = _engine_cfg(m.denoising_net, 500, 'sample', 4, 'hybrid')
    cfg['n_basis'] = 0
    h = ctypes.c_void_p()
    assert _lib.lib().msmd_create(ctypes.byref(MsmdConfig(**cfg)), 0, ctypes.byref(h)) == -1    # MSMD_ERR_INVALID
    assert b'n_basis=0' in _lib.lib().msmd_last_error()
    assert not h.value


# ------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope='module', params=ALL)
def config_case(request, built_lib):
    """One configuration on CUDA with the package-default (hybrid) engine, its forward inputs and the float64 oracle's
    forward, whole and in parts (computed once, shared by every arithmetic)."""
    cid = request.param
    m, net, args, prefix = _build(cid, 'cuda')
    sd = cpu_state_dict(m if m is not None else net)
    i = _forward_inputs(net, N_FWD, 21)
    want = _oracle(sd, args, i, prefix)
    parts = _oracle(sd, args, i, prefix, keep_separate=True)
    return dict(cid=cid, m=m, net=net, args=args, sd=sd, i=i, want=want, parts=parts)


@pytest.mark.gpu
def test_forward_vs_float64_oracle(config_case):
    """fp32-grade below 1e-5; fp16 / bf16 below the schedule's bounds with the usual margins over the batch and below
    the bounds themselves on every sequence; the keep_separate parts fp32-grade below 1e-5."""
    c = config_case
    net, want = c['net'], c['want']
    assert net.precision == 'hybrid'
    dev = [None if v is None else v.cuda() for v in _forward_args(c['i'])]
    bounds = _bounds()
    for p in ARITHMETICS:
        got = net(*dev, precise=p)
        assert got.shape == want.shape
        whole, per = rel_l2(got, want), _seq_errs(got, want)
        print(f"config {c['cid']:6s} forward {p}: batch rel-L2 {whole:.2e}, worst sequence {max(per):.2e}")
        assert whole < bounds[p][0] and max(per) < bounds[p][1], (c['cid'], p, whole, per)
    dyn, sta, alp = net(*dev, keep_separate=True, precise='fp32')
    wd, ws, wa = c['parts']
    parts = [rel_l2(dyn, wd), rel_l2(sta, ws.unsqueeze(1).expand(sta.shape)), rel_l2(alp, wa)]
    print(f"config {c['cid']:6s} keep_separate fp32: dynamic / static / alphas rel-L2 " +
          ' / '.join(f'{e:.2e}' for e in parts))
    assert max(parts) < F32_TOL, (c['cid'], parts)


@pytest.mark.gpu
@pytest.mark.parametrize('cfg_cond', [None, []], ids=['E3', 'E1'])
def test_teacher_forced_steps_vs_float64_oracle(config_case, cfg_cond):
    """Single sampling steps of the default engine (bf16 at t = 500, fp16 at the top of its segment, fp32-grade at
    t = 1) from a given state, 'incremental' guidance with both conditions (E = 3) and without guidance (E = 1):
    within 1e-3, and 1e-5 at t = 1."""
    c = config_case
    m, args = c['m'], c['args']
    if m is None:
        pytest.skip('MSMD fixes motion_dim 67: the bare-network configurations are forward only')
    assert m.precision == 'hybrid' and m.precise_last_steps == 'auto' and m.fp16_last_steps == 'auto'
    T, N = args.n_diff_steps, 3
    k16 = m._fp16_steps()
    assert m._precise_steps() < k16 < 500
    kw = dict(L=args.n_motions, d_style=args.d_style)
    i = synth.sampler_inputs(N, T, 31, **kw)
    ind = i['indicator'] if args.use_indicator else None
    g = dict(cfg_mode='incremental', cfg_cond=cfg_cond, cfg_scale=CFG_SCALE)
    sd64 = _cast(c['sd'], torch.float64)
    for t, tol in ((500, 1e-3), (k16, 1e-3), (1, F32_TOL)):
        x_t = synth.sampler_inputs(N, 1, 300 + t, **kw)['x_T'] * (0.3 + 0.7 * t / T)
        want, _, _ = D.sample(sd64, args, *_cast([i['audio_feat'], i['shape'], i['style']], torch.float64),
                              x_T=x_t.double(), z={t: i['z'][t].double()}, indicator=_cast(ind, torch.float64),
                              t_start=t, n_steps=1, **g)
        got, _, _ = m.sample(i['audio_feat'].cuda(), i['shape'].cuda(), i['style'].cuda(), motion_at_T=x_t.cuda(),
                             indicator=None if ind is None else ind.cuda(), noise=i['z'].cuda(), t_start=t, n_steps=1,
                             **g)
        errs = _seq_errs(got, want)
        print(f"config {c['cid']:6s} E={3 if cfg_cond is None else 1} t={t:3d}: "
              f"rel-L2 {rel_l2(got, want):.2e}, worst clip {max(errs):.2e}")
        assert rel_l2(got, want) < tol and max(errs) < tol, (c['cid'], t, errs)
    m.check()


@pytest.fixture(scope='module')
def batch_case(built_lib):
    """The released architecture on one hybrid engine, with the float64 oracle of the largest batch (every smaller
    batch is a prefix of it)."""
    m, args = make_msmd('cuda', precision='hybrid')
    i = synth.denoiser_inputs(BATCHES[0], 41)
    t0 = time.time()
    want = _oracle(cpu_state_dict(m), args, i, 'denoising_net.')
    print(f'float64 oracle, {BATCHES[0]} sequences: {time.time() - t0:.1f} s')
    return m, i, want


@pytest.mark.gpu
def test_batch_sizes_on_one_engine(batch_case):
    """S = 300, 37, 19, 18, 5, 4, 1 in that order on the engine created for 300: every sequence of every batch in all
    three arithmetics.  300 > 16 x 18 gives every person-token cluster more than one group of 16; 18 / 19 straddle the
    CTA-pair GEMM switch and one attention job per CTA; 4 / 5 the 64-wide tile switch; 37 is two jobs on each of 148
    CTAs."""
    m, i, want = batch_case
    net = m.denoising_net
    bounds = _bounds()
    eng = None
    for S in BATCHES:
        dev = [v[:S].cuda() for v in _forward_args(i)]
        for p in ARITHMETICS:
            got = net(*dev, precise=p)
            errs = _seq_errs(got, want[:S])
            print(f'S={S:3d} forward {p}: worst sequence rel-L2 {max(errs):.2e} (sequence {errs.index(max(errs))})')
            assert max(errs) < bounds[p][1], (S, p, [(s, e) for s, e in enumerate(errs) if e >= bounds[p][1]])
        eng = eng or net._eng
        assert net._eng is eng and eng.cfg.max_seqs == BATCHES[0]


@pytest.fixture(scope='module')
def big_sample_case(built_lib):
    """100 clips with both guidance conditions (300 sequences) on the default engine, the states and step noise of
    t = 500, the top of the fp16 segment and t = 1, and the float64 oracle's step from each (clips are independent,
    so the batched oracle is the oracle of every clip alone)."""
    m, args = make_msmd('cuda', precision=None)
    T = args.n_diff_steps
    i = synth.sampler_inputs(NX_BIG, 1, 51)
    sd64 = _cast(cpu_state_dict(m), torch.float64)
    steps = {}
    t0 = time.time()
    for t in (500, m._fp16_steps(), 1):
        g = torch.Generator().manual_seed(600 + t)
        x_t = torch.randn(NX_BIG, args.n_motions, 67, generator=g) * (0.3 + 0.7 * t / T)
        z_t = torch.randn(NX_BIG, args.n_motions, 67, generator=g) if t > 1 else torch.zeros(NX_BIG, args.n_motions, 67)
        want, _, _ = D.sample(sd64, args, *_cast([i['audio_feat'], i['shape'], i['style']], torch.float64),
                              x_T=x_t.double(), z={t: z_t.double()}, indicator=i['indicator'].double(), t_start=t,
                              n_steps=1, cfg_mode='incremental', cfg_scale=CFG_SCALE)
        steps[t] = (x_t, z_t, want)
    print(f'float64 oracle, {NX_BIG} clips x 3 entries x {len(steps)} steps: {time.time() - t0:.1f} s')
    return m, args, i, steps


@pytest.mark.gpu
def test_sampling_step_at_300_sequences(big_sample_case):
    """One teacher-forced step of 100 clips x 3 guidance entries at t = 500 (bf16), the top of the fp16 segment and
    t = 1 (fp32-grade): every clip within 1e-3 of the oracle, and 1e-5 at t = 1."""
    m, args, i, steps = big_sample_case
    T = args.n_diff_steps
    z = torch.zeros((T + 1, NX_BIG, args.n_motions, 67), device='cuda')     # the engine takes noise indexed by t
    for t, (x_t, z_t, want) in steps.items():
        z.zero_()
        z[t] = z_t.cuda()
        got, _, _ = m.sample(i['audio_feat'].cuda(), i['shape'].cuda(), i['style'].cuda(), motion_at_T=x_t.cuda(),
                             indicator=i['indicator'].cuda(), noise=z, t_start=t, n_steps=1, cfg_mode='incremental',
                             cfg_scale=CFG_SCALE)
        errs = _seq_errs(got, want)
        tol = F32_TOL if t == 1 else 1e-3
        print(f'{NX_BIG} clips x 3 entries t={t:3d}: worst clip rel-L2 {max(errs):.2e} (clip {errs.index(max(errs))})')
        assert max(errs) < tol, (t, [(n, e) for n, e in enumerate(errs) if e >= tol])
    assert m._eng.S == 3 * NX_BIG
    m.check()
