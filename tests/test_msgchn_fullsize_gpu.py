"""Parity of the dispatch that is BENCHMARKED: the MSG-CHN TTA step at the full BASELINE.json sizes (1x352x1216 `2layers`,
1x480x640 `1layer`), where the engine routes the 32->32 convolutions and their data gradients to the tcgen05 kernels
(csrc/conv_tc.cuh, conv_tc_s2.cuh, conv_tc_t2.cuh), against the CPU oracle run on the same seeded inputs -- and the small
reference fixtures run BOTH ways (every tcgen05 kernel forced on / all of them off) so that each kernel family is compared
with outputs of the real reference.

Tolerances (north star): filtered validity / filtered sparse depth bit-exact; per-step losses and adapted tensors after Adam:
test_msgchn_step_gpu.loss_tolerance / weight_tolerance (docstring there)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import msgchn_oracle as O
from golden_util import golden_names, load_golden, case_frame, case_checkpoint, rel, nrel, W_SD, W_SM, W_COS
from oracle_trace import trace_step, to_nchw
from test_msgchn_step_gpu import (make_model, report, ZERO_GRAD, eng_adapt_names, weight_tolerance, loss_tolerance, step_loss_tolerance, TOL_W,
                                  FWD_NAMES, GRAD_NAMES)

DEV = 'cuda'

FULL = [
    # name, checkpoint, prepare_mode, dataset, n, h, w, lr, cap
    ('kitti_2layers_fitted', 'kitti_2layers_a', 'meta_selfsup_seq_2layers_ema', 'kitti', 1, 352, 1216, 1e-4, 80.0),
    ('kitti_2layers_gate', 'kitti_2layers_b', 'meta_selfsup_seq_2layers_ema', 'kitti', 1, 352, 1216, 1e-4, 80.0),
    ('kitti_2layers_random', 0, 'meta_selfsup_seq_2layers_ema', 'kitti', 1, 352, 1216, 1e-4, 80.0),
    ('void_1layer_fitted', 'void_1layer_a', 'meta_selfsup_seq_1layer_ema', 'void', 1, 480, 640, 3e-3, 8.0),
    ('void_1layer_random', 1, 'meta_selfsup_seq_1layer_ema', 'void', 1, 480, 640, 3e-3, 8.0),
    ('kitti_2layers_batch2', 'kitti_2layers_a', 'meta_selfsup_seq_2layers_ema', 'kitti', 2, 176, 608, 1e-4, 80.0),
]
IDS = [c[0] for c in FULL]


def _sync_oracle_to_native(model, sd_o, state, names, t):
    """teacher forcing: the oracle takes the native path's weights, BatchNorm buffers and Adam moments, so that every step is an
    independent comparison from IDENTICAL state (a continual comparison multiplies the L1-sign-flip error of step t by the
    sensitivity of step t+1 -- at the indoor lr = 3e-3 the fitted network's loss doubles per step -- and stops measuring the kernels)"""
    sd_n = model.state_dict()
    for k in sd_o:
        sd_o[k].copy_(sd_n[k].detach().cpu().to(sd_o[k].dtype).view(sd_o[k].shape))
    for k in names:
        state.m[k] = model.model._m_views[k].detach().cpu().clone().view(sd_o[k].shape)
        state.v[k] = model.model._v_views[k].detach().cpu().clone().view(sd_o[k].shape)
    state.step = t


@pytest.mark.parametrize('case', FULL, ids=IDS)
def test_fullsize_steps_match_oracle(case):
    """3 TTA steps at the benchmarked size, native (tcgen05 dispatch) vs oracle; each step starts from the native path's own state
    (weights, BatchNorm buffers, Adam moments copied into the oracle), so the bounds are per step and carry no step-to-step allowance."""
    name, ckpt, mode, dataset, n, h, w, lr, cap = case
    tol_key = {'ckpt': ckpt if isinstance(ckpt, str) else None}          # fitted checkpoints: test_msgchn_step_gpu.loss_tolerance
    sd = O.get_checkpoint(ckpt, mode)
    model = make_model(mode, sd, cap)
    sd_o = {k: v.clone() for k, v in sd.items()}
    names = O.adapt_parameter_names(sd_o)
    state = O.AdamState(names, sd_o)
    for t in range(3):
        if t:
            _sync_oracle_to_native(model, sd_o, state, names, t)
        before = {k: sd_o[k].clone() for k in names}
        image, sparse, dense = O.synthetic_frame(11, t, n, h, w, dataset)
        model.tta_step(image.to(DEV), sparse.to(DEV), lr, W_SD, W_SM, W_COS)
        got = model.last_losses()
        res = O.tta_step(sd_o, state, image, sparse, lr=lr, max_input_depth=cap, return_grads=True)
        eng = model._last_engine
        assert torch.equal(eng.tensor('filtered_validity').view(n, 1, h, w).cpu(), res['validity']), t
        assert torch.equal(eng.tensor('filtered_depth').view(n, 1, h, w).cpu(), res['sparse_depth']), t
        # the L1 residual of a FITTED network is a few % of the depth itself, and the prediction carries the bf16 noise of the operands
        # (measured 6e-4 of the depth, for the oracle's own bf16 emulation as well): |d loss_sd| is bounded in units of the depth
        mean_depth = float(res['sparse_depth'][res['validity'] > 0].mean())
        for k in ('loss', 'loss_sparse_depth', 'loss_smooth', 'loss_cos'):
            report('%s step %d %-18s native %.6f oracle %.6f rel %.2e' % (name, t, k, got[k], res[k], rel(got[k], res[k])))
            ok = rel(got[k], res[k]) < loss_tolerance(tol_key)
            if k in ('loss', 'loss_sparse_depth') and tol_key['ckpt']:
                ok = ok or abs(got[k] - res[k]) < 5e-4 * mean_depth
            assert ok, (t, k, got[k], res[k], mean_depth)
        gate = 0.0 if res['loss_cos'] < 0.3 else W_COS
        assert got['w_cos_eff'] == pytest.approx(gate), (t, got, res['loss_cos'])
        e_out = nrel(model.last_output().cpu(), res['output_depth'])
        report('%s step %d output depth nrel %.3e' % (name, t, e_out))
        assert e_out < 2e-2, (t, e_out)
        sd_n = model.state_dict()
        for k in names:
            if k in ZERO_GRAD:
                continue
            e, upd = nrel(sd_n[k].cpu(), sd_o[k]), nrel(before[k], sd_o[k])
            report('%s step %d lr=%g %-40s weight nrel %.3e  (update/|w| %.3e, error/update %.3f)' % (name, t, lr, k, e, upd, e / max(upd, 1e-30)))
            if t == 0:
                # Adam's FIRST step is -lr * sign(g) (m / sqrt(v) = g / |g|): the two implementations can only differ where the sign of a
                # gradient component differs, i.e. on components inside the gradient noise of the bf16 operands / L1 sign flips.  Asserted:
                # few components flip, and every flipped one is a SMALL component of the oracle's gradient (a wrong backward flips large ones)
                g_o = res['grads'][k].flatten()
                d_n, d_o = (sd_n[k].cpu() - before[k]).flatten(), (sd_o[k] - before[k]).flatten()
                flipped = (torch.sign(d_n) != torch.sign(d_o)) & (d_o != 0)
                frac = float(flipped.float().mean())
                rms = float(g_o.pow(2).mean().sqrt())
                worst = float(g_o[flipped].abs().max()) if bool(flipped.any()) else 0.0
                report('%s step 0 %-40s first Adam step: %.2f %% of the signs differ, largest flipped |g| = %.3f rms(g)' % (name, k, 100 * frac, worst / max(rms, 1e-30)))
                assert frac < 0.12 and worst < 1.0 * rms, (k, frac, worst, rms)
            else:
                assert e < max(TOL_W, 0.25 * upd), (t, k, e, upd)


@pytest.mark.parametrize('case', FULL[:1] + FULL[3:4], ids=IDS[:1] + IDS[3:4])
def test_fullsize_blocks_against_oracle_trace(case):
    """One training forward + backward at the benchmarked size, block by block: every conv_tc / conv_tc_s2 / conv_tc_t2 role
    (forward, data gradient + mask + add, out2 / add2, stride 2 both ways) is hit inside the engine."""
    name, ckpt, mode, dataset, n, h, w, lr, cap = case
    tol_key = {'ckpt': ckpt if isinstance(ckpt, str) else None}          # fitted checkpoints: test_msgchn_step_gpu.loss_tolerance
    sd = O.get_checkpoint(ckpt, mode)
    model = make_model(mode, sd, cap)
    image, sparse, _ = O.synthetic_frame(12, 0, n, h, w, dataset)
    T, G, L, grads = trace_step({k: v.clone() for k, v in sd.items()}, image, sparse, cap, W_SD, W_SM, W_COS)
    eng = model.model._engine_for(image.to(DEV))
    eng.set_adam(0.0)
    model.tta_step(image.to(DEV), sparse.to(DEV), 0.0, W_SD, W_SM, W_COS)
    torch.cuda.synchronize()
    rep, worst = [], 0.0
    for nm in FWD_NAMES:
        got, want = to_nchw(eng.tensor(nm)), T[nm]
        e = nrel(got.reshape(want.shape), want)
        rep.append('%-14s %.3e' % (nm, e))
        worst = max(worst, e)
    report('%s forward blocks, worst %.3e' % (name, worst))
    assert worst < 2e-2, 'forward block mismatch:\n' + '\n'.join(rep)
    got_l = model.last_losses()
    for k in ('loss', 'loss_sparse_depth', 'loss_smooth', 'loss_cos'):
        assert rel(got_l[k], L[k]) < loss_tolerance(tol_key), (k, got_l[k], L[k])
    greport = []
    for nm in GRAD_NAMES:
        got, want = to_nchw(eng.tensor(nm)), G[nm]
        greport.append((nm, nrel(got.reshape(want.shape), want)))
    for k in eng_adapt_names(model):
        if k not in ZERO_GRAD:
            greport.append((k, nrel(model.model._grad_views[k].cpu(), grads[k])))
    for nm, e in greport:
        report('%s gradient %-44s nrel %.3e' % (name, nm, e))
    worst_g = max(e for _, e in greport)
    assert worst_g < 0.3, greport      # end-to-end gradients carry the L1 sign flips (see test_msgchn_step_gpu); cosine > 0.95


@pytest.mark.parametrize('force', ['tc_all', 'tc_off'])
@pytest.mark.parametrize('name', golden_names())
def test_fixtures_with_forced_dispatch(name, force):
    """The reference's own fixtures with every tcgen05 conv forced on at these small sizes (tc_min_pixels = 0) and with all of
    them off (mma.sync kernels): both dispatches must reproduce the reference."""
    fx = load_golden(name)
    case = fx['case']
    sd = case_checkpoint(case)
    opts = {'tc_min_pixels': 0, 'tc_s2_min_pixels': 0, 'tc_t2_min_pixels': 0, 'tc_head_min_pixels': 0} if force == 'tc_all' else {'tc_enabled': 0}
    model = make_model(case, sd, case['max_input_depth'], options=opts)
    for t in range(case['steps']):
        image, sparse, _ = case_frame(case, t)
        model.tta_step(image.to(DEV), sparse.to(DEV), case['lr'], W_SD, W_SM, W_COS)
        got, g = model.last_losses(), fx['steps'][t]
        for k in ('loss', 'loss_smooth', 'loss_sparse_depth', 'loss_cos'):
            prev = fx['steps'][t - 1][k] if t else None
            assert rel(got[k], g[k]) < step_loss_tolerance(case, t, g[k], prev), (force, t, k, got[k], g[k])
    out = model.last_output().cpu()
    assert nrel(out, fx['output_depth']) < 2e-2, nrel(out, fx['output_depth'])
    sd_after = model.state_dict()
    for k in fx['adapt_names']:
        if k in ZERO_GRAD:
            continue
        e, upd = nrel(sd_after[k].cpu(), fx['params_after'][k]), nrel(sd[k], fx['params_after'][k])
        report('%s [%s] %-40s weight nrel %.3e (update/|w| %.3e)' % (name, force, k, e, upd))
        assert e < weight_tolerance(upd), (force, k, e, upd)


def test_fused_proj3_pred0_equals_two_gemms():
    """emb = pred(proj(z)): proj.3 and pred.0 are two Linear layers with nothing between them; the engine runs them as ONE GEMM with
    W = W_pred0 W_proj3 (fp32 product at pack time).  Against the two-GEMM form (option fuse_projpred = 0): same embedding up to the
    bf16 rounding of the intermediate the fused form no longer has, same losses."""
    mode, cap = 'meta_selfsup_seq_2layers_ema', 80.0
    sd = O.get_checkpoint('kitti_2layers_a', mode)
    image, sparse, _ = O.synthetic_frame(14, 0, 1, 64, 128, 'kitti')
    outs = []
    for fuse in (1, 0):
        model = make_model(mode, sd, cap, options={'fuse_projpred': fuse})
        model.tta_step(image.to(DEV), sparse.to(DEV), 0.0, W_SD, W_SM, W_COS)
        eng = model._last_engine
        outs.append((eng.tensor('emb').float().cpu(), model.last_losses()))
    e = nrel(outs[0][0], outs[1][0])
    assert e < 1e-2, e
    assert rel(outs[0][1]['loss_cos'], outs[1][1]['loss_cos']) < 1e-3
    assert outs[0][1]['loss_sparse_depth'] == outs[1][1]['loss_sparse_depth']          # nothing else moved
