"""CPU: the reference-written checkpoint fixture (tests/golden/refckpt_*.ckpt.pth, oracle/gen_golden_ckpt.py) against the oracle --
restoring its 'net' + torch.optim.Adam state into the oracle and taking the next step reproduces what the reference did next."""
import os

import pytest
import torch

from golden_util import GOLDEN_DIR, load_golden, case_frame, rel, nrel, W_SD, W_SM, W_COS
from golden_util import fixture_threads  # noqa: F401  (pytest fixture)
from oracle import msgchn_oracle as O

pytestmark = pytest.mark.usefixtures('fixture_threads')

NAME = 'refckpt_2layers_kitti_1x64x128'


def test_oracle_continues_the_reference_checkpoint():
    fx = load_golden(NAME)
    case = fx['case']
    ck = torch.load(os.path.join(GOLDEN_DIR, NAME + '.ckpt.pth'), map_location='cpu', weights_only=False)
    assert set(ck.keys()) == {'net', 'optimizer', 'train_step'} and ck['train_step'] == case['steps_before']
    sd = {k: v.clone() for k, v in ck['net'].items()}
    names = O.adapt_parameter_names(sd)
    assert names == fx['adapt_names']
    state = O.AdamState(names, sd)
    for i, k in enumerate(names):
        st = ck['optimizer']['state'][i]
        state.m[k], state.v[k] = st['exp_avg'].clone(), st['exp_avg_sq'].clone()
        state.step = int(st['step'])
    image, sparse, _ = case_frame(case, case['steps_before'])
    res = O.tta_step(sd, state, image, sparse, lr=case['lr'], w_sd=W_SD, w_sm=W_SM, w_cos=W_COS, max_input_depth=case['max_input_depth'])
    for k in ('loss', 'loss_sparse_depth', 'loss_smooth', 'loss_cos'):
        assert rel(res[k], fx['step_after'][k]) < 1e-5, (k, res[k], fx['step_after'][k])
    for k in names:
        assert nrel(sd[k], fx['params_after'][k]) < 1e-5, k
        assert nrel(state.m[k], fx['exp_avg_after'][k]) < 1e-4, k
    assert state.step == fx['adam_step_after']
