"""CPU: the oracle's restatement of the source-domain preparation steps (oracle/msgchn_oracle.py: init_step / head_step) against the
fixtures written by the REAL reference's stage-1 / stage-2 loops (oracle/gen_golden_prepare.py; src/init_main.py:482-522,
src/head_main.py:437-480).  fp32 vs fp32: the tolerances only cover summation order."""
import glob
import os

import pytest
import torch

from oracle import msgchn_oracle as O
from golden_util import GOLDEN_DIR, nrel, rel
from golden_util import fixture_threads  # noqa: F401  (pytest fixture)
from tta_depth_completion_b200.external_model_adapt import add_head_state

pytestmark = pytest.mark.usefixtures('fixture_threads')

# a bias in front of a train-mode BatchNorm has an analytically zero gradient: both sides hold rounding noise there and Adam turns its
# SIGN into +-lr steps, so these tensors are only bounded by the distance Adam can move them
NOISE_GRAD = ('pred.0.bias', 'conv1_rgb_meta.conv1_meta.1.bias')
PREP = sorted(os.path.basename(p)[:-3] for p in glob.glob(os.path.join(GOLDEN_DIR, 'prep_*.pt')))


def prep_frame(case, t):
    image, sparse, dense = O.synthetic_frame(case['seq_seed'], t, case['n'], case['h'], case['w'], case['dataset'])
    if case.get('density'):
        g = torch.Generator().manual_seed(77 + t)
        sparse = dense * (torch.rand(dense.shape, generator=g) < case['density']).float()
    return image, sparse, dense


def prep_initial_state(case):
    """the state the reference trained from: the fitted miniature checkpoint + the layers its `prepare_parameters` re-creates from
    torch's global RNG under the fixture's seed (the generator asserted that add_head_state reproduces them bit for bit)"""
    sd = {k: v.clone() for k, v in O.get_checkpoint(case['ckpt'], case['prepare_mode']).items()}
    torch.manual_seed(case['seed'])
    if case['stage'] == 'init':
        sd = {k: v for k, v in sd.items() if not k.startswith(('conv1_rgb_meta', 'proj', 'pred'))}
        fresh = add_head_state({}, case['init_mode'])
    else:
        fresh = {}
        add_head_state(fresh, 'head_selfsup_ema')
        add_head_state(fresh, 'head_selfsup_ema')
    sd.update(fresh)
    return sd, fresh


def test_fixtures_present():
    assert len(PREP) >= 4


@pytest.mark.parametrize('name', PREP)
def test_oracle_matches_reference_preparation(name):
    fx = torch.load(os.path.join(GOLDEN_DIR, name + '.pt'), weights_only=False)
    case = fx['case']
    sd, fresh = prep_initial_state(case)
    assert abs(O.checkpoint_digest(fresh) - fx['digest0']) < 1e-9 * max(1.0, abs(fx['digest0']))
    names = fx['trained']
    state = O.AdamState(names, sd)
    for t, want in enumerate(fx['steps']):
        image, sparse, dense = prep_frame(case, t)
        if case['stage'] == 'init':
            res = O.init_step(sd, state, image, sparse, dense, lr=case['lr'], max_input_depth=case['max_input_depth'], return_grads=True)
        else:
            res = O.head_step(sd, state, image, sparse, lr=case['lr'], max_input_depth=case['max_input_depth'], return_grads=True)
        assert rel(res['loss'], want['loss']) < 2e-5, (t, res['loss'], want['loss'])
        for k in names:
            assert k in NOISE_GRAD or rel(float(res['grads'][k].norm()), want['grad_norm'][k]) < 2e-3 or want['grad_norm'][k] < 1e-7, (t, k)
    for k in names:
        if k in NOISE_GRAD:
            assert float((sd[k] - fx['params_after'][k]).abs().max()) <= 2 * case['lr'] * case['steps'], k
            continue
        assert nrel(sd[k], fx['params_after'][k]) < 2e-5, k
    for k, v in fx['buffers_after'].items():
        if k in sd:
            assert nrel(sd[k].float(), v.float()) < 1e-5, k
    if case['stage'] == 'init':
        assert nrel(res['output_depth'], fx['output_depth']) < 1e-5
        for k in names:
            assert k in NOISE_GRAD or nrel(state.m[k], fx['exp_avg'][k]) < 2e-3, k
    else:
        for k, v in fx['proj_t_after_s8'].items():
            assert torch.equal(sd[k].flatten()[::8], v), k          # the EMA copy is plain fp32 arithmetic: bit-exact
        for k in names:
            if k in NOISE_GRAD:
                continue
            assert nrel(state.m[k].flatten()[::16], fx['exp_avg_s16'][k]) < 2e-3, k
            assert nrel(state.v[k].flatten()[::16], fx['exp_avg_sq_s16'][k]) < 4e-3, k
