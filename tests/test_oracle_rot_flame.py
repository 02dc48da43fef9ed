"""CPU: the oracle (oracle/rotations.py, oracle/flame_lbs.py) against the committed golden
vectors produced from the unmodified reference (oracle/make_golden.py), and - when
the reference is mounted (MSMD_REFERENCE) - against the reference modules directly."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_l2
from oracle import flame_lbs, ref_shims, rotations as R, synth
from oracle.make_golden import FLAME_GOLD, REF_MOD_GOLD, ROT_CONVENTIONS, rot_inputs


@pytest.fixture(scope='module')
def gold():
    return np.load(os.path.join(GOLDEN, 'rot.npz'))


def oracle_rot_outputs(gold):
    i = {k: v.numpy() for k, v in rot_inputs().items()}
    mats = gold['mats']
    o = {'quaternion_to_matrix': R.quaternion_to_matrix(i['quat']),
         'matrix_to_quaternion': R.matrix_to_quaternion(mats),
         'axis_angle_to_quaternion': R.axis_angle_to_quaternion(i['aa']),
         'quaternion_to_axis_angle': R.quaternion_to_axis_angle(gold['axis_angle_to_quaternion']),
         'axis_angle_to_matrix': R.axis_angle_to_matrix(i['aa']),
         'matrix_to_axis_angle': R.matrix_to_axis_angle(mats),
         'rotation_6d_to_matrix': R.rotation_6d_to_matrix(i['d6']),
         'matrix_to_rotation_6d': R.matrix_to_rotation_6d(mats),
         'axis_angle_to_rotation_6d': R.axis_angle_to_rotation_6d(i['aa']),
         'standardize_quaternion': R.standardize_quaternion(i['quat']),
         'quaternion_raw_multiply': R.quaternion_raw_multiply(i['quat'], i['quat2']),
         'quaternion_multiply': R.quaternion_multiply(i['quat'], i['quat2']),
         'quaternion_invert': R.quaternion_invert(i['quat']),
         'quaternion_apply': R.quaternion_apply(i['quat'], i['pts']),
         'batch_rodrigues': flame_lbs.rodrigues(torch.from_numpy(i['aa'])).numpy(),
         'euler_to_axis_angle_YXZ': R.matrix_to_axis_angle(R.euler_angles_to_matrix(i['euler'], 'YXZ'))}
    for c in ROT_CONVENTIONS:
        o[f'euler_angles_to_matrix_{c}'] = R.euler_angles_to_matrix(i['euler'], c)
        o[f'matrix_to_euler_angles_{c}'] = R.matrix_to_euler_angles(mats, c)
    return o


def test_oracle_rotations_match_golden(gold):
    out = oracle_rot_outputs(gold)
    assert set(out) | {'mats'} == set(gold.files)
    for k, v in out.items():
        # fp32 libm differences only (numpy vs torch); axis-angle of near-pi rotations is ill-conditioned
        tol = 2e-5 if 'axis_angle' in k and k.startswith(('quaternion_to', 'matrix_to', 'euler_to')) else 3e-6
        assert np.abs(v - gold[k]).max() <= tol, k


def test_oracle_rotation_known_answers():
    """Closed-form KATs (SURVEY section 4): identity, 90-degree turns, round trips."""
    assert np.array_equal(R.axis_angle_to_matrix(np.zeros((1, 3), np.float32))[0], np.eye(3, dtype=np.float32))
    assert torch.equal(flame_lbs.rodrigues(torch.zeros(1, 3))[0], torch.eye(3))
    rz = R.euler_angles_to_matrix(np.array([[0, 0, np.pi / 2]], np.float32), 'XYZ')[0]
    assert np.allclose(rz, [[0, -1, 0], [1, 0, 0], [0, 0, 1]], atol=1e-7)
    e = (np.random.default_rng(0).uniform(-1, 1, (64, 3)) * 1.2).astype(np.float32)
    back = R.matrix_to_euler_angles(R.euler_angles_to_matrix(e, 'YXZ'), 'YXZ')
    assert np.abs(back - e).max() < 5e-6
    q = R.axis_angle_to_quaternion(e)
    assert np.abs(R.quaternion_to_axis_angle(q) - e).max() < 5e-6
    for bad in ('XY', 'XXY', 'XAZ'):
        with pytest.raises(ValueError):
            R.euler_angles_to_matrix(e, bad)


def test_oracle_flame_matches_golden():
    g = np.load(os.path.join(GOLDEN, 'flame.npz'))
    c = FLAME_GOLD
    assets = synth.flame_assets(0, synth.FLAME_V, c['n_shape'], c['n_exp'])
    sh, ex, po, ey = synth.flame_inputs(c['B'], c['n_shape'], c['n_exp'], c['seed'])
    assert rel_l2(flame_lbs.flame_forward(assets, sh, ex, po, ey), g['verts']) < 1e-6
    assert rel_l2(flame_lbs.flame_forward(assets, sh, ex), g['verts_nopose']) < 1e-6
    assert rel_l2(flame_lbs.flame_forward(assets, sh, ex, po, ey, ignore_global_rot=True), g['verts_noglob']) < 1e-6
    a2 = synth.flame_assets(0, synth.FLAME_V, 100, 50)
    sh2, ex2, po2, ey2 = synth.flame_inputs(c['B'], 100, 50, c['seed'] + 1)
    assert rel_l2(flame_lbs.flame_forward(a2, sh2, ex2, po2, ey2), g['verts_100_50']) < 1e-6


def test_oracle_flame_known_answers():
    """FLAME(0,0,0) ~= template (3e-8, not bit exact: the chain re-adds joint offsets);
    a global-only rotation is R (v - j0) + j0."""
    assets = synth.flame_assets(1, 257, 300, 100)
    z = flame_lbs.flame_forward(assets, torch.zeros(3, 300), torch.zeros(3, 100))
    assert (z - assets['v_template']).abs().max() < 2e-7
    pose = torch.zeros(1, 6)
    pose[0, :3] = torch.tensor([0.3, -0.2, 0.5])
    v = flame_lbs.flame_forward(assets, torch.zeros(1, 300), torch.zeros(1, 100), pose)
    Rm = flame_lbs.rodrigues(pose[:, :3])[0]
    j0 = assets['J_regressor'][0] @ assets['v_template']
    want = (assets['v_template'] - j0) @ Rm.T + j0
    assert (v[0] - want).abs().max() < 1e-6


def test_oracle_against_reference_modules():
    """Euler conventions ZYX / YZX both ways, FLAME.forward and lbs (vertices and posed joints) on a 300-vertex model
    with 100 + 50 betas: the oracle against the reference's outputs stored in tests/golden/ref_modules.npz (every 3rd
    vertex; see oracle/make_golden.py for how they were made) and, when the unmodified reference is mounted, against it
    live."""
    c = REF_MOD_GOLD
    g = np.load(os.path.join(GOLDEN, 'ref_modules.npz'))
    m = ref_shims.ref_modules() if ref_shims.available() else None
    i = rot_inputs(n=c['rot_n'], seed=c['rot_seed'])
    for conv in c['conventions']:
        mats = R.euler_angles_to_matrix(i['euler'].numpy(), conv)
        assert np.abs(mats - g[f'euler_angles_to_matrix_{conv}']).max() < 3e-6
        got = R.matrix_to_euler_angles(g[f'euler_angles_to_matrix_{conv}'], conv)
        assert np.abs(got - g[f'matrix_to_euler_angles_{conv}']).max() < 3e-6
        if m is not None:
            want = m.rc.euler_angles_to_matrix(i['euler'], conv)
            assert np.abs(mats - want.numpy()).max() < 3e-6
            got = R.matrix_to_euler_angles(want.numpy(), conv)
            assert np.abs(got - m.rc.matrix_to_euler_angles(want, conv).numpy()).max() < 3e-6
    assets = synth.flame_assets(c['raw_seed'], c['V'], c['n_shape'], c['n_exp'])
    sh, ex, po, ey = synth.flame_inputs(c['B'], c['n_shape'], c['n_exp'], c['seed'])
    verts = flame_lbs.flame_forward(assets, sh, ex, po, ey)
    assert rel_l2(verts[:, ::c['stride']], g['flame_verts']) < 1e-6
    # joints (lbs returns J_transformed)
    full = flame_lbs.flame_full_pose(po, ey, c['B'])
    v2, j2 = flame_lbs.lbs(torch.cat([sh, ex], 1), full, assets['v_template'], assets['shapedirs'],
                           assets['posedirs'], assets['J_regressor'], assets['parents'], assets['lbs_weights'])
    assert rel_l2(v2[:, ::c['stride']], g['lbs_verts']) < 1e-6 and rel_l2(j2, g['lbs_joints']) < 1e-6
    if m is not None:
        fl = ref_shims.ref_flame(synth.flame_raw(c['raw_seed'], c['V'], 400), c['n_shape'], c['n_exp'])
        with torch.no_grad():
            want, _, _ = fl(sh, ex, po, ey, return_lm2d=False, return_lm3d=False)
        assert rel_l2(verts, want) < 1e-6
        vr, jr = m.lbs.lbs(torch.cat([sh, ex], 1), full, assets['v_template'][None].expand(c['B'], -1, -1),
                           assets['shapedirs'], assets['posedirs'], assets['J_regressor'],
                           torch.tensor(assets['parents']), assets['lbs_weights'])
        assert rel_l2(v2, vr) < 1e-6 and rel_l2(j2, jr) < 1e-6
