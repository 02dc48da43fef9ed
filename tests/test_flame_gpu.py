"""GPU parity: FLAME decode through the drop-in FLAME module / lbs() vs oracle and golden vectors.
Tolerance: vertices <= 1e-5 relative L2 (BASELINE.json north_star)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_l2
from oracle import flame_lbs, synth
from oracle.make_golden import FLAME_GOLD

pytestmark = pytest.mark.gpu
TOL = 1e-5


def make_flame(V, n_shape, n_exp, seed=0, impl=0):
    from msmd_b200.utils.flame import FLAME
    from types import SimpleNamespace
    raw = synth.flame_raw(seed, V, 400)
    cfg = SimpleNamespace(n_shape=n_shape, n_exp=n_exp, flame_lmk_embedding_path=None)
    m = FLAME(cfg, raw=raw, lmk_embeddings=synth.flame_lmk_embeddings(raw['f'].shape[0])).cuda()
    m.impl = impl
    return m


@pytest.mark.parametrize('impl', [0, 1])
def test_flame_matches_golden(built_lib, impl):
    g = np.load(os.path.join(GOLDEN, 'flame.npz'))
    c = FLAME_GOLD
    fl = make_flame(synth.FLAME_V, c['n_shape'], c['n_exp'], impl=impl)
    sh, ex, po, ey = [t.cuda() for t in synth.flame_inputs(c['B'], c['n_shape'], c['n_exp'], c['seed'])]
    v, lm2d, lm3d = fl(sh, ex, po, ey)
    print(f'FLAME impl {impl}: vertices rel-L2 vs reference golden = {rel_l2(v, g["verts"]):.2e}')
    assert rel_l2(v, g['verts']) < TOL
    assert rel_l2(lm2d, g['lm2d']) < TOL and rel_l2(lm3d, g['lm3d']) < TOL
    v, _, _ = fl(sh, ex, None, None, return_lm2d=False, return_lm3d=False)
    assert rel_l2(v, g['verts_nopose']) < TOL
    v, _, _ = fl(sh, ex, po, ey, ignore_global_rot=True, return_lm2d=False, return_lm3d=False)
    assert rel_l2(v, g['verts_noglob']) < TOL
    fl2 = make_flame(synth.FLAME_V, 100, 50, impl=impl)
    sh2, ex2, po2, ey2 = [t.cuda() for t in synth.flame_inputs(c['B'], 100, 50, c['seed'] + 1)]
    v, _, _ = fl2(sh2, ex2, po2, ey2, return_lm2d=False, return_lm3d=False)
    assert rel_l2(v, g['verts_100_50']) < TOL


@pytest.mark.parametrize('impl', [0, 1])
@pytest.mark.parametrize('B', [1, 63, 130, 517])
def test_flame_ragged_batches_vs_oracle(built_lib, impl, B):
    """Batch sizes that are not tile multiples; rotation-matrix input (pose2rot=False) as well."""
    assets = synth.flame_assets(0, synth.FLAME_V, 300, 100)
    fl = make_flame(synth.FLAME_V, 300, 100, impl=impl)
    sh, ex, po, ey = synth.flame_inputs(B, 300, 100, seed=B)
    want = flame_lbs.flame_forward(assets, sh, ex, po, ey)
    got, _, _ = fl(sh.cuda(), ex.cuda(), po.cuda(), ey.cuda(), return_lm2d=False, return_lm3d=False)
    assert rel_l2(got, want) < TOL
    full = flame_lbs.flame_full_pose(po, ey, B)
    Rm = flame_lbs.rodrigues(full.reshape(-1, 3)).reshape(B, 5 * 9)
    got2, _, _ = fl(sh.cuda(), ex.cuda(), torch.cat([Rm[:, :9], Rm[:, 18:27]], 1).cuda(), Rm[:, 27:].cuda(),
                    pose2rot=False, return_lm2d=False, return_lm3d=False)
    assert rel_l2(got2, want) < TOL


@pytest.mark.parametrize('impl', [0, 1])
def test_flame_odd_coefficient_count_vs_oracle(built_lib, impl):
    """101 + 50 coefficients: the tensor-core pose kernel reads them in pairs and needs an even count, so an odd
    count runs the CUDA-core pose kernel."""
    assets = synth.flame_assets(0, synth.FLAME_V, 101, 50)
    fl = make_flame(synth.FLAME_V, 101, 50, impl=impl)
    sh, ex, po, ey = synth.flame_inputs(130, 101, 50, seed=5)
    want = flame_lbs.flame_forward(assets, sh, ex, po, ey)
    got, _, _ = fl(sh.cuda(), ex.cuda(), po.cuda(), ey.cuda(), return_lm2d=False, return_lm3d=False)
    assert rel_l2(got, want) < TOL


def test_flame_small_mesh_and_lbs_function(built_lib):
    """lbs() drop-in (verts AND posed joints) on a mesh whose 3V is not a tile multiple."""
    from msmd_b200.utils.lbs import lbs
    V = 301
    assets = synth.flame_assets(2, V, 100, 50)
    sh, ex, po, ey = synth.flame_inputs(40, 100, 50, seed=4)
    betas = torch.cat([sh, ex], 1)
    full = flame_lbs.flame_full_pose(po, ey, 40)
    vw, jw = flame_lbs.lbs(betas, full, assets['v_template'], assets['shapedirs'], assets['posedirs'],
                           assets['J_regressor'], assets['parents'], assets['lbs_weights'])
    d = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in assets.items()}
    vg, jg = lbs(betas.cuda(), full.cuda(), d['v_template'][None].expand(40, -1, -1), d['shapedirs'], d['posedirs'],
                 d['J_regressor'], torch.tensor(d['parents']).cuda(), d['lbs_weights'])
    assert rel_l2(vg, vw) < TOL and rel_l2(jg, jw) < TOL


def test_flame_known_answers(built_lib):
    fl = make_flame(synth.FLAME_V, 300, 100)
    z, _, _ = fl(torch.zeros(2, 300).cuda(), torch.zeros(2, 100).cuda(), return_lm2d=False, return_lm3d=False)
    assert (z - fl.v_template).abs().max() < 3e-7
    e, _, _ = fl(torch.zeros(0, 300).cuda(), torch.zeros(0, 100).cuda(), torch.zeros(0, 6).cuda(),
                 torch.zeros(0, 6).cuda(), return_lm2d=False, return_lm3d=False)
    assert e.shape == (0, synth.FLAME_V, 3)


def test_flame_full_size_properties(built_lib):
    """Config 2 (8192 x 5023, 300+100): impl 0 vs impl 1 agree; a sampled subset matches the oracle;
    decoding is batch-order equivariant."""
    B = 8192
    fl = make_flame(synth.FLAME_V, 300, 100)
    sh, ex, po, ey = [t.cuda() for t in synth.flame_inputs(B, 300, 100, 0)]
    v0, _, _ = fl(sh, ex, po, ey, return_lm2d=False, return_lm3d=False)
    fl.impl = 1
    v1, _, _ = fl(sh, ex, po, ey, return_lm2d=False, return_lm3d=False)
    print(f'FLAME B=8192: tensor-core vs SIMT path rel-L2 = {rel_l2(v0, v1):.2e}')
    assert rel_l2(v0, v1) < TOL
    idx = torch.arange(0, B, 331)
    assets = synth.flame_assets(0, synth.FLAME_V, 300, 100)
    want = flame_lbs.flame_forward(assets, sh[idx].cpu(), ex[idx].cpu(), po[idx].cpu(), ey[idx].cpu())
    assert rel_l2(v0[idx], want) < TOL
    fl.impl = 0
    perm = torch.randperm(B, device='cuda')
    vp, _, _ = fl(sh[perm], ex[perm], po[perm], ey[perm], return_lm2d=False, return_lm3d=False)
    assert torch.equal(vp, v0[perm])
