"""Epilogue operands of the 32-channel tcgen05 convolutions (ReLU-derivative mask, add / add2 addends, the bilinear x2 `up2`
addend, and mask / add of the transposed stride-2 kernel): every variant at ragged strip widths, widths below one strip, and
batches whose per-CTA row ranges cross strips and images, checked bit for bit where the mma.sync kernel computes the same
fp32 expression, and by identities of the kernel itself (a zero addend, an all-positive mask) where it does not."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = 'cuda'

# (n, h, w): ragged last strip (1216, 514, 258), below one strip (100, 38); n = 3 with h not a multiple of the rows per CTA,
# so CTA ranges cross strips and images
S1_SHAPES = [(1, 352, 1216), (1, 40, 514), (3, 21, 514), (2, 33, 258), (3, 50, 258), (1, 12, 100), (2, 7, 38)]
UP2_SHAPES = [(1, 352, 1216), (1, 38, 514), (3, 50, 258), (2, 38, 258), (1, 14, 100), (2, 6, 38)]     # half sizes 19x257, 25x129, ...
T2_SHAPES = [(1, 176, 608), (1, 20, 257 * 2), (3, 17, 129 * 2), (2, 9, 50), (1, 5, 16)]


@pytest.fixture(scope='module')
def ops():
    from tta_depth_completion_b200 import ops as _ops
    return _ops


def _rand(g, *shape):
    return torch.randn(shape, generator=g).to(DEV).to(torch.bfloat16)


def _weights(ops, g, kind):
    wt = (torch.randn((32, 32, 3, 3), generator=g) * (2.0 / 288) ** 0.5).to(DEV)
    return ops.pack_conv_weight(wt, kind), (torch.randn(32, generator=g) * 0.1).to(DEV)


@pytest.mark.parametrize('n,h,w', S1_SHAPES)
def test_conv_tc_mask_add_variants_match_mma(ops, n, h, w):
    from tta_depth_completion_b200 import _lib
    g = torch.Generator().manual_seed(31 + h + w)
    wp, bias = _weights(ops, g, 'conv_fwd')
    wi = ops.pack_conv_weight_tc(wp)
    x, m, a = _rand(g, n, h, w, 32), _rand(g, n, h, w, 32), _rand(g, n, h, w, 32)
    # mask only, mask + add (the data gradients)
    want = ops.conv3x3(x, wp, None, ops.MODE_S1, ops.PRO_NONE, mask=m, mask_mode=ops.MASK_RELU)
    assert torch.equal(ops.conv3x3_tc(x, wp, None, mask=m, wimage=wi), want), 'mask'
    want = ops.conv3x3(x, wp, None, ops.MODE_S1, ops.PRO_NONE, mask=m, mask_mode=ops.MASK_RELU, add=a)
    assert torch.equal(ops.conv3x3_tc(x, wp, None, mask=m, add=a, wimage=wi), want), 'mask + add'
    # out aliases add: the backward accumulates in place
    acc = a.clone()
    _lib.check(_lib.lib().ptta_conv3x3_tc(_lib.ptr(x), _lib.ptr(acc), _lib.ptr(wi), None, n, h, w, 0, 0, _lib.ptr(m), _lib.ptr(acc),
                                          torch.cuda.current_stream().cuda_stream), 'conv3x3_tc in place')
    assert torch.equal(acc, want), 'mask + add in place'
    # add only (with bias and relu_out), and add2 + out2 (decoder sums)
    xr = torch.relu(x)
    base = ops.conv3x3_tc(xr, wp, bias, wimage=wi)
    assert torch.equal(base, ops.conv3x3(x, wp, bias, ops.MODE_S1, ops.PRO_RELU)), 'plain'
    zero = torch.zeros_like(a)
    assert torch.equal(ops.conv3x3_tc(xr, wp, bias, add=zero, wimage=wi), base), 'add of zeros'
    want = ops.conv3x3(x, wp, bias, ops.MODE_S1, ops.PRO_RELU, add=a)
    assert torch.equal(ops.conv3x3_tc(xr, wp, bias, add=a, wimage=wi), want), 'add'
    assert torch.equal(ops.conv3x3_tc(xr, wp, bias, add=a, relu_out=True, wimage=wi), torch.relu(want)), 'add + relu_out'
    o, o2 = ops.conv3x3_tc_ex(xr, wp, bias, add2=a, wimage=wi)
    assert torch.equal(o, base), 'add2: out'
    assert torch.equal(o2, torch.relu((base.float() + a.float()).to(torch.bfloat16))), 'add2: out2 = ReLU(out + add2)'
    o, o2 = ops.conv3x3_tc_ex(xr, wp, bias, add=a, wimage=wi)
    assert torch.equal(o, want) and torch.equal(o2, torch.relu(want)), 'add + out2'
    with pytest.raises(RuntimeError):
        ops.conv3x3_tc_ex(xr, wp, bias, mask=m, wimage=wi)        # a mask with out2 is not a variant the network uses


@pytest.mark.parametrize('n,h,w', UP2_SHAPES)
def test_conv_tc_up2_odd_half_sizes(ops, n, h, w):
    g = torch.Generator().manual_seed(41 + h + w)
    wp, bias = _weights(ops, g, 'conv_fwd')
    x = torch.relu(_rand(g, n, h, w, 32))
    half = _rand(g, n, h // 2, w // 2, 32)
    base = ops.conv3x3_tc(x, wp, bias)
    out, out_relu = ops.conv3x3_tc_up2(x, wp, torch.zeros_like(half), bias)
    assert torch.equal(out, base) and torch.equal(out_relu, torch.relu(base)), 'up2 of zeros'
    out, out_relu = ops.conv3x3_tc_up2(x, wp, half, bias)
    assert torch.equal(out_relu, torch.relu(out.float()).to(torch.bfloat16))
    # reference: the plain kernel's bf16(conv + bias) plus F.interpolate (align_corners = True) of the same bf16 map
    up = F.interpolate(half.float().permute(0, 3, 1, 2), scale_factor=2, mode='bilinear', align_corners=True).permute(0, 2, 3, 1)
    ref = base.float() + up                                    # base = bf16(conv + bias): one extra rounding of <= 2^-9 relative
    err = (out.float() - ref).abs()
    tol = 2.0 ** -7 * torch.maximum(ref.abs(), base.float().abs()) + 1e-3 * float(ref.pow(2).mean().sqrt())
    assert not bool((err > tol).any()), 'up2: %d elements off, max err %.3g' % (int((err > tol).sum()), float(err.max()))


@pytest.mark.parametrize('n,h,w', T2_SHAPES)
def test_conv_tc_t2_mask_add_variants(ops, n, h, w):
    from tta_depth_completion_b200 import _lib
    g = torch.Generator().manual_seed(51 + h + w)
    wp, bias = _weights(ops, g, 'convT_fwd')
    x = _rand(g, n, h, w, 32)
    m, a = _rand(g, n, 2 * h, 2 * w, 32), _rand(g, n, 2 * h, 2 * w, 32)
    base = ops.conv3x3_tc_t2(x, wp, None)
    ones, zero = torch.ones_like(m), torch.zeros_like(a)
    # identities of the kernel itself: bit for bit
    assert torch.equal(ops.conv3x3_tc_t2(x, wp, None, mask=ones, add=zero), base), 't2 all-positive mask + zero add'
    assert torch.equal(ops.conv3x3_tc_t2(x, wp, None, add=zero), base), 't2 zero add'
    assert torch.equal(ops.conv3x3_tc_t2(x, wp, None, mask=m), torch.where(m.float() > 0, base, torch.zeros_like(base))), 't2 mask'
    # against mma.sync: equal up to the summation order of the 4-tap output class (as the transposed-kernel test in test_ops_gpu.py)
    want = ops.conv3x3(x, wp, None, ops.MODE_T2, ops.PRO_NONE, mask=m, mask_mode=ops.MASK_RELU, add=a)
    got = ops.conv3x3_tc_t2(x, wp, None, mask=m, add=a)
    d = (got.float() - want.float()).abs()
    assert float((d > 0).float().mean()) < 1e-3 and bool((d <= want.float().abs() * 2.0 ** -7 + 1e-6).all()), 't2 mask + add'
    acc = a.clone()
    wi = torch.empty((9 * 32 * 32,), dtype=torch.bfloat16, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(_lib.lib().ptta_pack_conv_weight_tc_t2(_lib.ptr(wp), _lib.ptr(wi), st), 'pack')
    _lib.check(_lib.lib().ptta_conv3x3_tc_t2(_lib.ptr(x), _lib.ptr(acc), _lib.ptr(wi), None, n, h, w, 0, _lib.ptr(m), _lib.ptr(acc), st),
               'conv3x3_tc_t2 in place')
    assert torch.equal(acc, got), 't2 mask + add in place'


def test_conv_tc_operand_variants_graph_replay(ops):
    """the operand variants captured in one CUDA graph replay to exactly the eager results"""
    g = torch.Generator().manual_seed(61)
    n, h, w = 3, 50, 516          # the half-size map feeds the transposed conv: W / 2 even
    wp, bias = _weights(ops, g, 'conv_fwd')
    wpT, _ = _weights(ops, g, 'convT_fwd')
    wi = ops.pack_conv_weight_tc(wp)
    x, m, a = _rand(g, n, h, w, 32), _rand(g, n, h, w, 32), _rand(g, n, h, w, 32)
    xr, half, xs = torch.relu(x), _rand(g, n, h // 2, w // 2, 32), _rand(g, n, h // 2, w // 2, 32)

    def run():
        return [ops.conv3x3_tc(x, wp, None, mask=m, wimage=wi), ops.conv3x3_tc(x, wp, None, mask=m, add=a, wimage=wi),
                *ops.conv3x3_tc_ex(xr, wp, bias, add2=a, wimage=wi), *ops.conv3x3_tc_up2(xr, wp, half, bias),
                ops.conv3x3_tc_t2(xs, wpT, None, mask=m, add=a)]
    eager = run()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        run()                       # weight images and tensor maps are made outside the capture
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=s):
            outs = run()
    for _ in range(2):
        for o in outs:
            o.zero_()
        gr.replay()
        torch.cuda.synchronize()
        for i, (e, o) in enumerate(zip(eager, outs)):
            assert torch.equal(e, o), 'graph replay differs from eager (output %d)' % i
