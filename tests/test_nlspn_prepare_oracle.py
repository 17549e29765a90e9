"""CPU: the oracle's restatement of the stage-2 step on the NLSPN back-end (oracle/nlspn_oracle.py: head_step) against the fixtures written
by the REAL reference's stage-2 loop (oracle/gen_golden_nlspn_prepare.py; src/head_main.py:259-278, 437-480).  fp32 vs fp32: the
tolerances only cover summation order."""
import glob
import os

import pytest
import torch

from oracle import nlspn_oracle as NO
from oracle import msgchn_oracle as O
from golden_util import GOLDEN_DIR, nrel, rel
from golden_util import fixture_threads  # noqa: F401  (pytest fixture)
from tta_depth_completion_b200.nlspn_prepare import fresh_head_state, HEAD_TRAINED

pytestmark = pytest.mark.usefixtures('fixture_threads')

# a bias in front of a train-mode BatchNorm has an analytically zero gradient: both sides hold rounding noise there and Adam turns its SIGN
# into +-lr steps, so these tensors are only bounded by the distance Adam can move them
NOISE_GRAD = ('proj.0.bias', 'proj.3.bias', 'pred.0.bias')      # proj.3.bias: a constant through pred.0 into pred's BatchNorm
PREP = sorted(os.path.basename(p)[:-3] for p in glob.glob(os.path.join(GOLDEN_DIR, 'nlspn_prep_head_*.pt')))
S = 128


def initial_state(case):
    """the state the reference trained from: the seeded checkpoint + the heads its `prepare_parameters` re-creates from torch's global RNG
    under the fixture's seed (the generator asserted that fresh_head_state reproduces them bit for bit)"""
    sd = {k: v.clone() for k, v in NO.make_synthetic_checkpoint(case['ckpt_seed']).items()}
    torch.manual_seed(case['seed'])
    fresh = fresh_head_state()
    sd.update(fresh)
    return sd, fresh


def test_fixtures_present():
    assert len(PREP) >= 2
    assert HEAD_TRAINED == NO.HEAD_TRAINED


@pytest.mark.parametrize('name', PREP)
def test_oracle_matches_reference_stage2(name):
    fx = torch.load(os.path.join(GOLDEN_DIR, name + '.pt'), weights_only=False)
    case = fx['case']
    sd, fresh = initial_state(case)
    assert abs(O.checkpoint_digest(fresh) - fx['digest_heads0']) < 1e-9 * max(1.0, abs(fx['digest_heads0']))
    names = fx['trained']
    state = O.AdamState(names, sd)
    for t, want in enumerate(fx['steps']):
        image, sparse, dense = NO.synthetic_frame(case['seq'], t, case['n'], case['h'], case['w'], case['dataset'])
        res = NO.head_step(sd, state, NO.normalize_image(image), torch.clamp(sparse, 0, case['cap']), lr=case['lr'], return_grads=True)
        assert rel(res['loss'], want['loss']) < 2e-5, (t, res['loss'], want['loss'])
        assert nrel(res['emb'][:4], want['emb_rows']) < 1e-4 and nrel(res['ref'][:4], want['ref_rows']) < 1e-4
        for k in names:
            assert k in NOISE_GRAD or rel(float(res['grads'][k].norm()), want['grad_norm'][k]) < 2e-3 or want['grad_norm'][k] < 1e-7, (t, k)
    for k in names:
        if k in NOISE_GRAD:
            assert float((sd[k].flatten()[::S] - fx['params_after_s128'][k]).abs().max()) <= 2 * case['lr'] * case['steps'], k
            continue
        upd = fx['update_norm'][k] * (1.0 / S) ** 0.5
        assert float((sd[k].flatten()[::S] - fx['params_after_s128'][k]).norm()) < 2e-2 * upd, k
        assert nrel(state.m[k].flatten()[::S], fx['exp_avg_s128'][k]) < 2e-3, k
        assert nrel(state.v[k].flatten()[::S], fx['exp_avg_sq_s128'][k]) < 4e-3, k
    for k, v in fx['buffers_after'].items():
        assert nrel(sd[k].float(), v.float()) < 1e-5, k
    for k, v in fx['proj_t_after_s128'].items():
        assert nrel(sd[k].flatten()[::S], v) < 1e-6, k          # EMA of a proj that is itself trained (equal up to the gradients' summation order)
