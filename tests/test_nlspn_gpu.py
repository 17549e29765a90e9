"""GPU tier: the B200 NLSPN propagation kernels (through the C ABI / nlspn_prop.py) against the oracle, the fixtures generated
by the reference's own NLSPN class, torchvision's DCNv2, and -- where oracle/build_ref_dcn.py has built oracle/_ref/dcn_ref.so
from the reference's source -- the reference's own DCN CUDA kernels.  Tolerances: fp32 arithmetic in a different summation order
-> 1e-5 relative (norm-wise) on values and gradients; scatter-accumulated gradients (fp32 atomics, as in the reference) 1e-4."""
import importlib.machinery
import importlib.util
import os

import numpy as np
import pytest
import torch

from oracle import nlspn_prop_oracle as P

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
DEV = 'cuda'


@pytest.fixture(scope='module')
def NP():
    from tta_depth_completion_b200 import nlspn_prop
    return nlspn_prop


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def load(name):
    return torch.load(os.path.join(GOLDEN, name + '.pt'), weights_only=False)


def dcn_ref():
    path = os.path.join(ROOT, 'oracle', '_ref', 'dcn_ref.so')
    if not os.path.exists(path):
        return None
    loader = importlib.machinery.ExtensionFileLoader('dcn_ref', path)
    spec = importlib.util.spec_from_loader('dcn_ref', loader)
    mod = importlib.util.module_from_spec(spec)
    loader.exec_module(mod)
    return mod


def rand_case(seed, n, h, w, k):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, 1, h, w, generator=g)
    off = torch.randn(n, 2 * k * k, h, w, generator=g) * 2.5
    m = torch.rand(n, k * k, h, w, generator=g)
    wt = torch.randn(1, 1, k, k, generator=g)
    b = torch.randn(1, generator=g)
    go = torch.randn(n, 1, h, w, generator=g)
    return x, off, m, wt, b, go


@pytest.mark.parametrize('n,h,w,k,pad', [(1, 19, 37, 3, 1), (2, 24, 40, 1, 0), (1, 33, 65, 3, 1)])
def test_mdconv_matches_oracle(NP, n, h, w, k, pad):
    x, off, m, wt, b, go = rand_case(3, n, h, w, k)
    want = P.mdconv_forward(*(t.numpy() for t in (x, off, m, wt, b)), 1, pad, 1)
    gwant = P.mdconv_backward(*(t.numpy() for t in (x, off, m, wt, b)), go.numpy(), 1, pad, 1)
    dx, doff, dm, dw, db = (t.to(DEV).requires_grad_(True) for t in (x, off, m, wt, b))
    out = NP.ModulatedDeformConvFunction.apply(dx, doff, dm, dw, db, 1, pad, 1, 1, 1, 64)
    assert rel(out, torch.from_numpy(want)) < 1e-5
    out.backward(go.to(DEV))
    for got, ref_, name, tol in ((dx.grad, gwant[0], 'grad_input', 1e-4), (doff.grad, gwant[1], 'grad_offset', 1e-5),
                                 (dm.grad, gwant[2], 'grad_mask', 1e-5), (dw.grad, gwant[3], 'grad_weight', 1e-4), (db.grad, gwant[4], 'grad_bias', 1e-4)):
        assert rel(got, torch.from_numpy(np.ascontiguousarray(ref_))) < tol, name


def reference_mdconv(impl, x, off, m, wt, b, go, k, pad):
    """(output, [grad_input, grad_offset, grad_mask, grad_weight, grad_bias]) of a reference DCNv2 on CPU tensors:
    'reference_kernels': the reference's own CUDA kernels (oracle/_ref/dcn_ref.so);
    'torchvision': torchvision's deform_conv2d with a mask (the reference's offset layout and bilinear border rule) on the CPU,
    in float32 as the reference -- a sampling position rounded differently can land in the neighbouring cell, where the offset
    gradient jumps (in float64, about 1e-2 of it moves at 352x1216)."""
    if impl == 'reference_kernels':
        ref = dcn_ref()
        if ref is None:
            pytest.skip('oracle/_ref/dcn_ref.so not built (oracle/build_ref_dcn.py builds it from the reference\'s source tree)')
        x, off, m, wt, b, go = (t.to(DEV) for t in (x, off, m, wt, b, go))
        want = ref.modulated_deform_conv_forward(x, wt, b, off, m, k, k, 1, 1, pad, pad, 1, 1, 1, 1, 64)
        return want, ref.modulated_deform_conv_backward(x, wt, b, off, m, go, k, k, 1, 1, pad, pad, 1, 1, 1, 1, 64)
    tvops = pytest.importorskip('torchvision.ops')
    cpu = [t.clone().requires_grad_(True) for t in (x, off, m, wt, b)]
    want = tvops.deform_conv2d(cpu[0], cpu[1], cpu[3], cpu[4], stride=1, padding=pad, dilation=1, mask=cpu[2])
    want.backward(go)
    return want, [t.grad for t in cpu]


@pytest.mark.parametrize('n,h,w,k,pad', [(2, 40, 72, 3, 1), (1, 40, 72, 1, 0), (1, 352, 1216, 3, 1)])
@pytest.mark.parametrize('impl', ['reference_kernels', 'torchvision'])
def test_mdconv_matches_reference_dcn(NP, impl, n, h, w, k, pad):
    x, off, m, wt, b, go = rand_case(4, n, h, w, k)
    want, gwant = reference_mdconv(impl, x, off, m, wt, b, go, k, pad)
    dx, doff, dm, dw, db = (t.to(DEV).requires_grad_(True) for t in (x, off, m, wt, b))
    out = NP.ModulatedDeformConvFunction.apply(dx, doff, dm, dw, db, 1, pad, 1, 1, 1, 64)
    assert rel(out, want) < 1e-5
    out.backward(go.to(DEV))
    for got, ref_, name, tol in ((dx.grad, gwant[0], 'grad_input', 1e-4), (doff.grad, gwant[1], 'grad_offset', 1e-5),
                                 (dm.grad, gwant[2], 'grad_mask', 1e-5), (dw.grad, gwant[3], 'grad_weight', 1e-3), (db.grad, gwant[4], 'grad_bias', 1e-3)):
        assert rel(got, ref_) < tol, (name, rel(got, ref_))


@pytest.mark.parametrize('name', ['nlspn_prop_1x24x40', 'nlspn_prop_2x17x23'])
def test_propagation_matches_reference_fixture(NP, name):
    fx = load(name)
    offset_aff = fx['offset_aff'].to(DEV).requires_grad_(True)
    conf = fx['confidence'].to(DEV).requires_grad_(True)
    feat_init = fx['feat_init'].to(DEV).requires_grad_(True)
    mod = NP.NLSPNPropagation(prop_time=fx['case']['prop_time']).to(DEV)
    assert abs(float(mod.aff_scale_const) - fx['aff_scale_const']) < 1e-7
    y, feats, offset, aff, _ = mod(feat_init, offset_aff, conf, fx['sparse'].to(DEV))
    assert torch.equal(offset.cpu(), fx['offset'])                    # pure data movement: bit-exact
    assert rel(aff, fx['aff']) < 1e-6
    for got, key in ((feats[0], 'feat_1'), (feats[8], 'feat_9'), (feats[-1], 'feat_out'), (y, 'feat_out')):
        assert rel(got, fx[key]) < 1e-5, key
    (y * fx['probe'].to(DEV)).sum().backward()
    for got, key in ((feat_init.grad, 'g_feat_init'), (offset_aff.grad, 'g_offset_aff'), (conf.grad, 'g_confidence')):
        assert rel(got, fx[key]) < 1e-4, (key, rel(got, fx[key]))


def test_fused_loop_equals_stepwise_dcn_calls(NP):
    """the fused propagation == 18 separate ModulatedDeformConvFunction calls with autograd in between (what the reference runs)"""
    n, h, w = 1, 48, 80
    feat_init, sparse, offset_aff, conf = (t.to(DEV) for t in P.synthetic_prop_inputs(7, n, h, w, offset_std=1.5))
    offset_aff[:, 16:] *= 0.3
    offset, aff = NP.offset_affinity(offset_aff, conf, 4.0, True)
    a = [t.clone().requires_grad_(True) for t in (feat_init, offset, aff)]
    b = [t.clone().requires_grad_(True) for t in (feat_init, offset, aff)]
    y1 = NP.propagate(a[0], a[1], a[2], sparse, 18)
    ones, zero = torch.ones((1, 1, 3, 3), device=DEV), torch.zeros(1, device=DEV)
    mask_fix = (sparse > 0).float()
    f = b[0]
    for _ in range(18):
        f = (1.0 - mask_fix) * f + mask_fix * sparse
        f = NP.ModulatedDeformConvFunction.apply(f, b[1], b[2], ones, zero, 1, 1, 1, 1, 1, 64)
    assert rel(y1, f) < 1e-6
    probe = torch.randn_like(y1)
    (y1 * probe).sum().backward()
    (f * probe).sum().backward()
    for u, v, nm in zip(a, b, ('feat_init', 'offset', 'aff')):
        assert rel(u.grad, v.grad) < 1e-4, nm


def test_full_size_properties(NP):
    """352x1216: identity at zero offset / centre affinity, linearity without input preservation, and the adjoint identity
    <P f, g> == <f, P^T g> that ties backward to forward"""
    n, h, w = 1, 352, 1216
    g = torch.Generator().manual_seed(9)
    f1 = torch.randn(n, 1, h, w, generator=g).to(DEV)
    f2 = torch.randn(n, 1, h, w, generator=g).to(DEV)
    offset = torch.zeros(n, 18, h, w, device=DEV)
    aff = torch.zeros(n, 9, h, w, device=DEV)
    aff[:, 4] = 1.0
    assert torch.equal(NP.propagate(f1, offset, aff, None, 18), f1)
    offset = (torch.randn(n, 18, h, w, generator=g) * 2.0).to(DEV)
    offset[:, 8:10] = 0
    araw = torch.randn(n, 9, h, w, generator=g).to(DEV) * 0.05
    araw[:, 4] = 1.0 - (araw.sum(1) - araw[:, 4])
    y1, y2 = NP.propagate(f1, offset, araw, None, 6), NP.propagate(f2, offset, araw, None, 6)
    y12 = NP.propagate(2.0 * f1 - 3.0 * f2, offset, araw, None, 6)
    assert rel(y12, 2.0 * y1 - 3.0 * y2) < 1e-5
    fin = f1.clone().requires_grad_(True)
    y = NP.propagate(fin, offset, araw, None, 6)
    y.backward(f2)
    lhs, rhs = float((y.detach().double() * f2.double()).sum()), float((f1.double() * fin.grad.double()).sum())
    assert abs(lhs - rhs) <= 1e-4 * max(abs(lhs), abs(rhs), 1.0), (lhs, rhs)


def test_errors_are_loud(NP):
    x, off, m, wt, b, _ = rand_case(1, 1, 8, 8, 3)
    with pytest.raises(RuntimeError):
        NP.ModulatedDeformConvFunction.apply(x, off, m, wt, b, 1, 1, 1, 1, 1, 64)                        # CPU tensors: no fallback
    dx, doff, dm, dw, db = (t.to(DEV) for t in (x, off, m, wt, b))
    with pytest.raises(RuntimeError):
        NP.ModulatedDeformConvFunction.apply(dx.expand(1, 1, 8, 8).transpose(2, 3), doff, dm, dw, db, 1, 1, 1, 1, 1, 64)    # non-contiguous
    with pytest.raises(RuntimeError):
        NP.ModulatedDeformConvFunction.apply(dx.repeat(1, 2, 1, 1), doff, dm, dw.repeat(1, 2, 1, 1), db, 1, 1, 1, 1, 1, 64)  # C_in = 2
    with pytest.raises(RuntimeError):
        NP.propagate(dx, doff, dm[:, :8], None, 18)                                                      # 8 affinities instead of 9
