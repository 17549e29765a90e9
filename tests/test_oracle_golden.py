"""The CPU oracle (oracle/msgchn_oracle.py) against the fixtures produced by the real reference
(oracle/gen_golden.py): this is what pins the oracle (SURVEY.md §8c: the reference has no golden
vectors of its own)."""
import pytest
import torch

from oracle import msgchn_oracle as O
from golden_util import golden_names, load_golden, case_frame, case_checkpoint, rel, nrel, W_SD, W_SM, W_COS
from golden_util import fixture_threads  # noqa: F401  (pytest fixture)

pytestmark = pytest.mark.usefixtures('fixture_threads')
# fp32 CPU vs fp32 CPU of the same torch build: only summation-order noise is expected
TOL_LOSS = 2e-5
TOL_TENSOR = 2e-5
# conv bias in front of a train-mode BatchNorm (network_exp_msg_chn_adapt.py:31-33): dL/db == 0 exactly
ZERO_GRAD = ('conv1_rgb_meta.conv1_meta.1.bias',)


@pytest.mark.parametrize('name', golden_names())
def test_oracle_matches_reference_fixture(name):
    fx = load_golden(name)
    case = fx['case']
    torch.manual_seed(0)
    sd = case_checkpoint(case)
    assert O.checkpoint_digest(sd) == pytest.approx(fx['digest'], rel=1e-12), 'checkpoint differs from the one the fixture was made with'
    names = O.adapt_parameter_names(sd, 'meta')
    assert names == fx['adapt_names']
    state = O.AdamState(names, sd)
    for t in range(case['steps']):
        image, sparse, _ = case_frame(case, t)
        res = O.tta_step(sd, state, image, sparse, lr=case['lr'], w_sd=W_SD, w_sm=W_SM, w_cos=W_COS,
                         max_input_depth=case['max_input_depth'], return_grads=True)
        g = fx['steps'][t]
        for k in ('loss', 'loss_smooth', 'loss_sparse_depth', 'loss_cos'):
            assert rel(res[k], g[k]) < TOL_LOSS, (t, k, res[k], g[k])
        assert int(res['validity'].sum()) == g['n_valid']
        if 'w_cos_eff' in g:       # the `loss_cos < 0.3` gate of src/external_model_adapt.py:424
            assert (res['loss_cos'] < 0.3) == (g['w_cos_eff'] == 0.0), (t, res['loss_cos'], g['w_cos_eff'])
        for k in names:
            if k in ZERO_GRAD:
                # analytically zero gradient: what the reference holds is fp32 rounding noise
                assert float(res['grads'][k].norm()) < 1e-4 * max(g['grad_norm'].values()), (t, k)
                continue
            assert rel(float(res['grads'][k].norm()), g['grad_norm'][k]) < 1e-3, (t, k)
            assert rel(float(sd[k].norm()), g['param_norm'][k]) < TOL_TENSOR, (t, k)
    # integer-valued outputs: bit exact
    assert torch.equal(res['validity'].to(torch.uint8), fx['validity_filtered'])
    assert torch.equal(res['sparse_depth'], fx['sparse_depth_filtered'])
    assert nrel(res['output_depth'], fx['output_depth']) < TOL_TENSOR
    assert nrel(res['emb'][:4], fx['emb_rows']) < 1e-4
    assert nrel(res['ref'][:4], fx['ref_rows']) < 1e-4
    for k in names:
        if k in ZERO_GRAD:
            # Adam turns the rounding noise into +-lr steps: bounded random walk, not reproducible
            assert float((sd[k] - fx['params_after'][k]).abs().max()) <= 2.001 * case['lr'] * case['steps'], k
            continue
        assert nrel(sd[k], fx['params_after'][k]) < TOL_TENSOR, k
        assert nrel(state.m[k], fx['exp_avg'][k]) < 1e-3, k
        assert nrel(state.v[k], fx['exp_avg_sq'][k]) < 1e-3, k
    for k, v in fx['buffers_after'].items():
        if k.endswith('num_batches_tracked'):
            assert int(sd[k]) == int(v), k
        else:
            assert nrel(sd[k], v) < 1e-4, k
    # eval-mode forward after adaptation (running statistics are used -> checks the double update)
    image, sparse, _ = case_frame(case, case['steps'] - 1)
    with torch.no_grad():
        out = O.model_forward(sd, image / 255.0, res['sparse_depth'], False, case['max_input_depth'])
    assert nrel(out, fx['eval_output_depth']) < TOL_TENSOR


def test_outlier_removal_inf_fill_is_equivalent():
    """SURVEY.md §8 a2: replacing the 10*max fill by +inf cannot change the result (this is the
    form the CUDA kernel uses, dropping the global max reduction)."""
    image, sparse, _ = O.synthetic_frame(3, 0, 2, 64, 96, 'kitti')
    v = O.validity_map(sparse)
    d_ref, v_ref = O.remove_outliers(sparse, v)
    filled = torch.where(v <= 0, torch.full_like(sparse, float('inf')), sparse)
    filled = torch.nn.functional.pad(filled, (3, 3, 3, 3), value=float('inf'))
    m = -torch.nn.functional.max_pool2d(-filled, 7, 1, 0)
    keep = ~(m < sparse - 1.5)
    v2 = v * keep.float()
    assert torch.equal(v2, v_ref) and torch.equal(sparse * v2, d_ref)
    assert 0 < int(v_ref.sum()) < int(v.sum())
