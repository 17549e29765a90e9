"""Thin torch-tensor wrappers over the stand-alone operators of libptta_b200.so.

Layouts: feature maps are NHWC bf16 tensors [N,H,W,C]; single-channel maps fp32 [N,H,W] (or [N,1,H,W]);
images fp32 NCHW.  No operator here has a PyTorch fallback."""
import ctypes

import torch

from . import _lib
from ._lib import check, ptr, c_void_p

MODE_S1, MODE_S2, MODE_T2 = 0, 1, 2
PRO_NONE, PRO_RELU, PRO_BN_LEAKY = 0, 1, 2
MASK_NONE, MASK_RELU, MASK_BN_LEAKY = 0, 1, 2


def _stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def _need(t, dtype, name):
    if t.dtype != dtype or not t.is_cuda or not t.is_contiguous():
        raise TypeError('%s must be a contiguous CUDA %s tensor' % (name, dtype))


def outlier_removal(sparse_depth, kernel_size=7, threshold=1.5):
    """validity map + OutlierRemoval.remove_outliers (src/tta_main.py:583-586, src/net_utils.py:766-811).
    Returns (filtered_sparse_depth, filtered_validity_map), same shape as the input."""
    _need(sparse_depth, torch.float32, 'sparse_depth')
    n = sparse_depth.shape[0]
    h, w = sparse_depth.shape[-2:]
    d = torch.empty_like(sparse_depth)
    v = torch.empty_like(sparse_depth)
    check(_lib.lib().ptta_outlier_removal(ptr(sparse_depth), ptr(d), ptr(v), n, h, w, kernel_size, threshold, _stream()), 'outlier_removal')
    return d, v


def pyramid(depth, max_input_depth=None):
    """clamp + validity-normalised /2 and /4 average pooling (network_exp_msg_chn_adapt.py:479,487,492)."""
    _need(depth, torch.float32, 'depth')
    n = depth.shape[0]
    h, w = depth.shape[-2:]
    dc = torch.empty_like(depth)
    d2 = torch.empty((n, 1, h // 2, w // 2), dtype=torch.float32, device=depth.device)
    d4 = torch.empty((n, 1, h // 4, w // 4), dtype=torch.float32, device=depth.device)
    cap = -1.0 if max_input_depth is None else float(max_input_depth)
    check(_lib.lib().ptta_pyramid(ptr(depth), ptr(dc), ptr(d2), ptr(d4), n, h, w, cap, 0 if max_input_depth is None else 1, _stream()),
          'pyramid')
    return dc, d2, d4


def pack_conv_weight(weight, role):
    """fp32 Conv2d [Cout,Cin,3,3] / ConvTranspose2d [Cin,Cout,3,3] weight -> bf16 [9][O][I] operand.
    role: 'conv_fwd', 'conv_dgrad_s1', 'conv_dgrad_s2', 'convT_fwd', 'convT_dgrad'."""
    _need(weight, torch.float32, 'weight')
    a, b = weight.shape[0], weight.shape[1]
    if role == 'conv_fwd':
        o, i, so, si, flip = a, b, b * 9, 9, 0
    elif role == 'conv_dgrad_s1':
        o, i, so, si, flip = b, a, 9, b * 9, 1
    elif role == 'conv_dgrad_s2':
        o, i, so, si, flip = b, a, 9, b * 9, 0
    elif role == 'convT_fwd':          # weight [Cin, Cout, 3, 3]
        o, i, so, si, flip = b, a, 9, b * 9, 0
    elif role == 'convT_dgrad':
        o, i, so, si, flip = a, b, b * 9, 9, 0
    else:
        raise ValueError(role)
    out = torch.empty((9, o, i), dtype=torch.bfloat16, device=weight.device)
    check(_lib.lib().ptta_pack_conv_weight(ptr(weight), ptr(out), o, i, so, si, flip, _stream()), 'pack_conv_weight')
    return out


def conv3x3(x, wpack, bias=None, mode=MODE_S1, prologue=PRO_NONE, pro_scale=None, pro_shift=None, slope=0.2,
            mask=None, mask_mode=MASK_NONE, mask_scale=None, mask_shift=None, add=None):
    _need(x, torch.bfloat16, 'x')
    _need(wpack, torch.bfloat16, 'wpack')
    n, h, w, cin = x.shape
    cout = wpack.shape[1]
    if wpack.shape[2] != cin:
        raise ValueError('weight operand expects %d input channels, x has %d' % (wpack.shape[2], cin))
    if mode == MODE_S1:
        ho, wo = h, w
    elif mode == MODE_S2:
        ho, wo = (h + 1) // 2, (w + 1) // 2
    else:
        ho, wo = 2 * h, 2 * w
    out = torch.empty((n, ho, wo, cout), dtype=torch.bfloat16, device=x.device)
    check(_lib.lib().ptta_conv3x3(ptr(x), ptr(out), ptr(wpack), ptr(bias), n, h, w, cin, cout, mode, prologue, ptr(pro_scale),
                                  ptr(pro_shift), slope, ptr(mask), mask_mode, ptr(mask_scale), ptr(mask_shift), ptr(add), _stream()),
          'conv3x3')
    return out


def pack_conv_weight_tc(wpack):
    """[9][32][32] bf16 pack -> the tcgen05 kernel's 18 KB shared-memory weight image"""
    _need(wpack, torch.bfloat16, 'wpack')
    if tuple(wpack.shape) != (9, 32, 32):
        raise ValueError('pack_conv_weight_tc handles 32->32 channels only')
    image = torch.empty((9 * 32 * 32,), dtype=torch.bfloat16, device=wpack.device)
    check(_lib.lib().ptta_pack_conv_weight_tc(ptr(wpack), ptr(image), _stream()), 'pack_conv_weight_tc')
    return image


def conv3x3_tc(x, wpack, bias=None, relu_in=False, relu_out=False, mask=None, add=None, variant=0, wimage=None):  # variant: unused
    """32->32 stride-1 conv on tcgen05 (same operand conventions as conv3x3 with MODE_S1, no ReLU-on-load).
    Pass `wimage` (pack_conv_weight_tc) to skip the per-call weight-image kernel."""
    _need(x, torch.bfloat16, 'x')
    n, h, w, cin = x.shape
    if cin != 32:
        raise ValueError('conv3x3_tc handles 32->32 channels only')
    if wimage is None:
        wimage = pack_conv_weight_tc(wpack)
    out = torch.empty_like(x)
    check(_lib.lib().ptta_conv3x3_tc(ptr(x), ptr(out), ptr(wimage), ptr(bias), n, h, w, 1 if relu_in else 0, 1 if relu_out else 0,
                                     ptr(mask), ptr(add), _stream()), 'conv3x3_tc')
    return out


def conv3x3_tc_ex(x, wpack, bias=None, relu_out=False, mask=None, add=None, add2=None, wimage=None):
    """conv3x3_tc with the second output: returns (out, out2) with out2 = ReLU(bf16(out) [+ add2])"""
    _need(x, torch.bfloat16, 'x')
    n, h, w, cin = x.shape
    if wimage is None:
        wimage = pack_conv_weight_tc(wpack)
    out, out2 = torch.empty_like(x), torch.empty_like(x)
    check(_lib.lib().ptta_conv3x3_tc_ex(ptr(x), ptr(out), ptr(out2), ptr(wimage), ptr(bias), n, h, w, 1 if relu_out else 0, ptr(mask), ptr(add),
                                        ptr(add2), _stream()), 'conv3x3_tc_ex')
    return out, out2


def conv3x3_tc_up2(x, wpack, half, bias=None):
    """(conv(x) + bias + up2(half), ReLU of it) in one pass of the tcgen05 conv; half: [n, h/2, w/2, 32]"""
    _need(x, torch.bfloat16, 'x')
    _need(half, torch.bfloat16, 'half')
    n, h, w, _ = x.shape
    wimage = pack_conv_weight_tc(wpack)
    out, out2 = torch.empty_like(x), torch.empty_like(x)
    check(_lib.lib().ptta_conv3x3_tc_up2(ptr(x), ptr(out), ptr(out2), ptr(wimage), ptr(bias), ptr(half), n, h, w, _stream()), 'conv3x3_tc_up2')
    return out, out2


def conv3x3_tc_s2(x, wpack, bias=None, relu_out=False, mask=None, add=None, want_relu_copy=False):
    """32->32 stride-2 conv on tcgen05 (operand conventions of conv3x3 with MODE_S2, no ReLU-on-load); H, W even.
    Returns out, or (out, relu(out)) with want_relu_copy."""
    _need(x, torch.bfloat16, 'x')
    _need(wpack, torch.bfloat16, 'wpack')
    n, h, w, cin = x.shape
    if cin != 32 or tuple(wpack.shape) != (9, 32, 32):
        raise ValueError('conv3x3_tc_s2 handles 32->32 channels only')
    image = torch.empty((9 * 32 * 32,), dtype=torch.bfloat16, device=x.device)
    check(_lib.lib().ptta_pack_conv_weight_tc_s2(ptr(wpack), ptr(image), _stream()), 'pack_conv_weight_tc_s2')
    out = torch.empty((n, h // 2, w // 2, 32), dtype=torch.bfloat16, device=x.device)
    out2 = torch.empty_like(out) if want_relu_copy else None
    check(_lib.lib().ptta_conv3x3_tc_s2(ptr(x), ptr(out), ptr(out2), ptr(image), ptr(bias), n, h, w, 1 if relu_out else 0, ptr(mask), ptr(add),
                                        _stream()), 'conv3x3_tc_s2')
    return (out, out2) if want_relu_copy else out


def conv3x3_tc_t2(x, wpack, bias=None, relu_out=False, mask=None, add=None):
    """32->32 transposed stride-2 conv on tcgen05 (operand conventions of conv3x3 with MODE_T2, no ReLU-on-load); W even.
    x: [n, h, w, 32] -> [n, 2h, 2w, 32]"""
    _need(x, torch.bfloat16, 'x')
    _need(wpack, torch.bfloat16, 'wpack')
    n, h, w, cin = x.shape
    if cin != 32 or tuple(wpack.shape) != (9, 32, 32):
        raise ValueError('conv3x3_tc_t2 handles 32->32 channels only')
    image = torch.empty((9 * 32 * 32,), dtype=torch.bfloat16, device=x.device)
    check(_lib.lib().ptta_pack_conv_weight_tc_t2(ptr(wpack), ptr(image), _stream()), 'pack_conv_weight_tc_t2')
    out = torch.empty((n, 2 * h, 2 * w, 32), dtype=torch.bfloat16, device=x.device)
    check(_lib.lib().ptta_conv3x3_tc_t2(ptr(x), ptr(out), ptr(image), ptr(bias), n, h, w, 1 if relu_out else 0, ptr(mask), ptr(add), _stream()),
          'conv3x3_tc_t2')
    return out


def conv3x3_wgrad(x, gout, prologue=PRO_NONE, pro_scale=None, pro_shift=None, slope=0.2):
    _need(x, torch.bfloat16, 'x')
    _need(gout, torch.bfloat16, 'gout')
    n, h, w, cin = x.shape
    cout = gout.shape[3]
    L = _lib.lib()
    ws = torch.empty(L.ptta_conv3x3_wgrad_workspace_bytes(n, h, w, cin, cout), dtype=torch.uint8, device=x.device)
    dw = torch.empty((cout, cin, 3, 3), dtype=torch.float32, device=x.device)
    check(L.ptta_conv3x3_wgrad(ptr(x), ptr(gout), ptr(dw), ptr(ws), n, h, w, cin, cout, prologue, ptr(pro_scale), ptr(pro_shift), slope,
                               _stream()), 'conv3x3_wgrad')
    return dw


def stem_conv(planes, weight, bias=None, scale=None, shift=None, mask=None):
    """planes: list of 1..3 fp32 tensors [N,H,W] (each contiguous) -> NHWC bf16 [N,H,W,32]."""
    cin = len(planes)
    n, h, w = planes[0].shape
    for p in planes:
        _need(p, torch.float32, 'plane')
    _need(weight, torch.float32, 'weight')
    pl = (ctypes.c_void_p * 3)(*[planes[min(k, cin - 1)].data_ptr() for k in range(3)])
    st = (ctypes.c_longlong * 3)(*[h * w] * 3)
    sc = (ctypes.c_float * 3)(*(list(scale) if scale is not None else [1.0] * cin) + [1.0] * (3 - cin))
    sh = (ctypes.c_float * 3)(*(list(shift) if shift is not None else [0.0] * cin) + [0.0] * (3 - cin))
    out = torch.empty((n, h, w, 32), dtype=torch.bfloat16, device=weight.device)
    check(_lib.lib().ptta_stem_conv(pl, st, sc, sh, cin, ptr(weight), ptr(bias), ptr(mask), ptr(out), n, h, w, _stream()), 'stem_conv')
    return out


def stem_conv_tc(planes, weight, bias=None, scale=None, shift=None, mask=None, relu_out=False):
    """stem_conv on tcgen05 (csrc/stem_tc.cuh); device weights [32, cin, 3, 3]"""
    cin = len(planes)
    n, h, w = planes[0].shape
    for p in planes:
        _need(p, torch.float32, 'plane')
    _need(weight, torch.float32, 'weight')
    pl = (ctypes.c_void_p * 3)(*[planes[min(k, cin - 1)].data_ptr() for k in range(3)])
    st = (ctypes.c_longlong * 3)(*[h * w] * 3)
    sc = (ctypes.c_float * 3)(*(list(scale) if scale is not None else [1.0] * cin) + [1.0] * (3 - cin))
    sh = (ctypes.c_float * 3)(*(list(shift) if shift is not None else [0.0] * cin) + [0.0] * (3 - cin))
    out = torch.empty((n, h, w, 32), dtype=torch.bfloat16, device=weight.device)
    image = torch.empty(2048, dtype=torch.bfloat16, device=weight.device)
    check(_lib.lib().ptta_stem_conv_tc(pl, st, sc, sh, cin, ptr(weight), ptr(bias), ptr(mask), ptr(out), ptr(image), 1 if relu_out else 0,
                                       n, h, w, _stream()), 'stem_conv_tc')
    return out


def stem_conv_const(planes, weight, bias=None, scale=None, shift=None, mask=None, relu_out=False):
    """stem_conv with HOST weights [32, cin, 3, 3] / bias [32] (CPU tensors): by-value kernel parameters, constant-bank operands"""
    cin = len(planes)
    n, h, w = planes[0].shape
    wh = weight.detach().cpu().contiguous().float()
    bh = None if bias is None else bias.detach().cpu().contiguous().float()
    pl = (ctypes.c_void_p * 3)(*[planes[min(k, cin - 1)].data_ptr() for k in range(3)])
    st = (ctypes.c_longlong * 3)(*[h * w] * 3)
    sc = (ctypes.c_float * 3)(*(list(scale) if scale is not None else [1.0] * cin) + [1.0] * (3 - cin))
    sh = (ctypes.c_float * 3)(*(list(shift) if shift is not None else [0.0] * cin) + [0.0] * (3 - cin))
    out = torch.empty((n, h, w, 32), dtype=torch.bfloat16, device=planes[0].device)
    check(_lib.lib().ptta_stem_conv_const(pl, st, sc, sh, cin, ctypes.c_void_p(wh.data_ptr()), ctypes.c_void_p(bh.data_ptr()) if bh is not None else None,
                                          ptr(mask), ptr(out), 1 if relu_out else 0, n, h, w, _stream()), 'stem_conv_const')
    return out


def head_conv_const(x, weight_9x32, bias=0.0, add=None, relu_in=True, out=None, accumulate=False):
    """head_conv with a HOST [9, 32] weight (CPU tensor)"""
    _need(x, torch.bfloat16, 'x')
    n, h, w, _ = x.shape
    wh = weight_9x32.detach().cpu().contiguous().float()
    if out is None:
        out = torch.empty((n, h, w), dtype=torch.float32, device=x.device)
    check(_lib.lib().ptta_head_conv_const(ptr(x), ctypes.c_void_p(wh.data_ptr()), float(bias), ptr(add), ptr(out), n, h, w, 1 if relu_in else 0,
                                          1 if accumulate else 0, _stream()), 'head_conv_const')
    return out


def head_conv_tc(x, weight_9x32, bias=0.0, add=None, out=None):
    """32 -> 1 conv on tcgen05 (no ReLU-on-load: pass ReLU(x) where the layer reads its input through one)"""
    _need(x, torch.bfloat16, 'x')
    _need(weight_9x32, torch.float32, 'weight')
    n, h, w, _ = x.shape
    image = torch.empty(9 * 16 * 32, dtype=torch.bfloat16, device=x.device)
    check(_lib.lib().ptta_pack_head_weight_tc(ptr(weight_9x32), ptr(image), _stream()), 'pack_head_weight_tc')
    if out is None:
        out = torch.empty((n, h, w), dtype=torch.float32, device=x.device)
    check(_lib.lib().ptta_head_conv_tc(ptr(x), ptr(image), float(bias), ptr(add), ptr(out), n, h, w, _stream()), 'head_conv_tc')
    return out


def head_conv(x, weight_9x32, bias=0.0, add=None, relu_in=True, out=None, accumulate=False):
    _need(x, torch.bfloat16, 'x')
    _need(weight_9x32, torch.float32, 'weight')
    n, h, w, _ = x.shape
    if out is None:
        out = torch.empty((n, h, w), dtype=torch.float32, device=x.device)
    check(_lib.lib().ptta_head_conv(ptr(x), ptr(weight_9x32), float(bias), ptr(add), ptr(out), n, h, w, 1 if relu_in else 0,
                                    1 if accumulate else 0, _stream()), 'head_conv')
    return out


def up2_1ch(a, b=None, c=None):
    _need(a, torch.float32, 'a')
    n, h, w = a.shape
    out = torch.empty((n, 2 * h, 2 * w), dtype=torch.float32, device=a.device)
    check(_lib.lib().ptta_up2_1ch(ptr(a), ptr(b), ptr(c), ptr(out), n, h, w, _stream()), 'up2_1ch')
    return out


def up2_1ch_adjoint(g_hi):
    _need(g_hi, torch.float32, 'g_hi')
    n, H, W = g_hi.shape
    out = torch.empty((n, H // 2, W // 2), dtype=torch.float32, device=g_hi.device)
    check(_lib.lib().ptta_up2_1ch_adjoint(ptr(g_hi), ptr(out), n, H // 2, W // 2, 0, _stream()), 'up2_1ch_adjoint')
    return out


def add_up2_c32(x, half):
    _need(x, torch.bfloat16, 'x')
    _need(half, torch.bfloat16, 'half')
    n, h, w, _ = half.shape
    out = torch.empty_like(x)
    check(_lib.lib().ptta_add_up2_c32(ptr(x), ptr(half), ptr(out), n, h, w, _stream()), 'add_up2_c32')
    return out


def up2_c32_adjoint(g_hi):
    _need(g_hi, torch.bfloat16, 'g_hi')
    n, H, W, c = g_hi.shape
    out = torch.empty((n, H // 2, W // 2, c), dtype=torch.bfloat16, device=g_hi.device)
    check(_lib.lib().ptta_up2_c32_adjoint(ptr(g_hi), ptr(out), n, H // 2, W // 2, 0, _stream()), 'up2_c32_adjoint')
    return out


def gemm_bf16(a, b, bias=None):
    """a [M,K] bf16, b [N,K] bf16 (nn.Linear weight layout) -> [M,N] bf16"""
    _need(a, torch.bfloat16, 'a')
    _need(b, torch.bfloat16, 'b')
    m, k = a.shape
    n = b.shape[0]
    out = torch.empty((m, n), dtype=torch.bfloat16, device=a.device)
    check(_lib.lib().ptta_gemm_bf16(ptr(a), ptr(b), ptr(out), ptr(bias), m, n, k, _stream()), 'gemm_bf16')
    return out


def gemm_bf16_tc(a, b, bias=None):
    """tcgen05 variant of gemm_bf16 (N % 256 == 0, K % 64 == 0)"""
    _need(a, torch.bfloat16, 'a')
    _need(b, torch.bfloat16, 'b')
    m, k = a.shape
    n = b.shape[0]
    out = torch.empty((m, n), dtype=torch.bfloat16, device=a.device)
    check(_lib.lib().ptta_gemm_bf16_tc(ptr(a), ptr(b), ptr(out), ptr(bias), m, n, k, _stream()), 'gemm_bf16_tc')
    return out


def adam_flat(param, grad, exp_avg, exp_avg_sq, lr, step, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
    for t in (param, grad, exp_avg, exp_avg_sq):
        _need(t, torch.float32, 'adam tensor')
    check(_lib.lib().ptta_adam_flat(ptr(param), ptr(grad), ptr(exp_avg), ptr(exp_avg_sq), param.numel(), lr, betas[0], betas[1], eps,
                                    weight_decay, step, _stream()), 'adam_flat')


def eval_metrics(output_depth, ground_truth, min_depth, max_depth):
    """MAE / RMSE (mm) and iMAE / iRMSE (1/km) over the pixels with min_depth <= gt <= max_depth, gt > 0, computed on the device
    (src/eval_utils.py:117-175 as called from src/tta_main.py:760-798; the reference moves both maps to the CPU first).
    Returns a dict of floats (one 20-byte D2H read)."""
    _need(output_depth, torch.float32, 'output_depth')
    _need(ground_truth, torch.float32, 'ground_truth')
    if output_depth.numel() != ground_truth.numel():
        raise ValueError('output_depth and ground_truth differ in size')
    L = _lib.lib()
    ws = torch.empty(L.ptta_eval_metrics_workspace_bytes(), dtype=torch.uint8, device=output_depth.device)
    res = torch.empty(5, dtype=torch.float32, device=output_depth.device)
    check(L.ptta_eval_metrics(ptr(output_depth), ptr(ground_truth), output_depth.numel(), float(min_depth), float(max_depth), ptr(ws), ptr(res),
                              _stream()), 'eval_metrics')
    v = res.cpu()
    return {'mae': float(v[0]), 'rmse': float(v[1]), 'imae': float(v[2]), 'irmse': float(v[3]), 'count': int(v[4])}


def inpaint_biharmonic(depth):
    """In place on a contiguous CUDA fp32 [N,1,H,W] map: every pixel that is exactly 0 becomes
    skimage.restoration.inpaint_biharmonic of its sample, clipped to the range of the sample's known pixels (the reference's eval-time
    hole filling, src/nlspn_model_adapt.py:124-127 -> src/data_utils.py:327-354), solved exactly in fp64 on the device.  One read of a
    4 x N word summary; when it shows holes, the solve runs and its status word is read back.  A sample whose pixels are all 0 raises
    ValueError, as the reference's empty `min` does.  Returns `depth`."""
    _need(depth, torch.float32, 'depth')
    if depth.dim() != 4 or depth.shape[1] != 1:
        raise ValueError('inpaint_biharmonic expects [N,1,H,W], got %s' % (tuple(depth.shape),))
    n, _, h, w = depth.shape
    L = _lib.lib()
    summary = torch.empty(4 * n + 4, dtype=torch.int32, device=depth.device)
    check(L.ptta_inpaint_plan(ptr(depth), n, h, w, ptr(summary), _stream()), 'inpaint_plan')
    host = summary.cpu()
    holes = host[0:4 * n:4]
    if not bool(holes.any()):
        return depth
    full = (holes == h * w).nonzero().flatten().tolist()
    if full:
        raise ValueError('zero-size array to reduction operation minimum which has no identity (sample %d of the prediction is 0 everywhere)'
                         % full[0])
    nbytes = ctypes.c_size_t()
    check(L.ptta_inpaint_workspace_bytes(c_void_p(host.data_ptr()), n, h, w, ctypes.byref(nbytes)), 'inpaint_workspace_bytes')
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=depth.device)
    check(L.ptta_inpaint_solve(ptr(depth), n, h, w, ptr(summary), ptr(ws), nbytes.value, _stream()), 'inpaint_solve')
    status = int(summary[4 * n])
    if status:
        raise RuntimeError('inpaint_biharmonic: solve status %d (%s)' % (status, 'non-positive pivot' if status == 1 else 'workspace too small'))
    return depth


def input_stage(image_u8_hwc, depth_u16, crop_shape=None, crop_type=('bottom',), depth_multiplier=256.0):
    """Decoded 8-bit RGB [N,H0,W0,3] (uint8) and 16-bit depth [N,H0,W0] (int16/uint16 bit pattern) -> (image fp32 NCHW in [0,255],
    sparse depth, validity map), cropped like the reference's default crop (src/datasets.py:83-170: horizontally centred, vertically
    centred or at the bottom).  src/data_utils.py:134-200 on the device; the frames cross PCIe in their compact types."""
    if image_u8_hwc.dtype != torch.uint8 or not image_u8_hwc.is_cuda or not image_u8_hwc.is_contiguous():
        raise TypeError('image must be a contiguous CUDA uint8 tensor [N,H0,W0,3]')
    if depth_u16.dtype not in (torch.int16, torch.uint16) or not depth_u16.is_cuda or not depth_u16.is_contiguous():
        raise TypeError('depth must be a contiguous CUDA 16-bit integer tensor [N,H0,W0]')
    n, h0, w0, _ = image_u8_hwc.shape
    h, w = (h0, w0) if crop_shape is None else crop_shape
    x0 = (w0 - w) // 2
    y0 = (h0 - h) if 'bottom' in crop_type else (h0 - h) // 2
    image = torch.empty((n, 3, h, w), dtype=torch.float32, device=image_u8_hwc.device)
    depth = torch.empty((n, 1, h, w), dtype=torch.float32, device=image_u8_hwc.device)
    validity = torch.empty_like(depth)
    check(_lib.lib().ptta_input_stage(ptr(image_u8_hwc), ptr(depth_u16), ptr(image), ptr(depth), ptr(validity), n, h0, w0, y0, x0, h, w,
                                      float(depth_multiplier), _stream()), 'input_stage')
    return image, depth, validity


# ---- host-side PNG decoding (csrc/png_host.cu; SURVEY.md section 8 f2) --------------------------------------------------------------
def _file_bytes(src):
    if isinstance(src, (bytes, bytearray, memoryview)):
        return bytes(src)
    with open(src, 'rb') as f:
        return f.read()


def png_info(src):
    """(width, height, channels, bit_depth) of a PNG file (path or bytes) -- header only"""
    data = _file_bytes(src)
    w, h, c, d = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    check(_lib.lib().ptta_png_info(data, len(data), ctypes.byref(w), ctypes.byref(h), ctypes.byref(c), ctypes.byref(d)), 'png_info')
    return w.value, h.value, c.value, d.value


def _decode_png(src, out, fn_name, dtype, channels):
    import numpy as np
    data = _file_bytes(src)
    w, h, _, _ = png_info(data)
    shape = (h, w, channels) if channels > 1 else (h, w)
    if out is None:
        out = np.empty(shape, dtype=dtype)
    if isinstance(out, torch.Tensor):            # e.g. a pinned staging buffer: decoded in place, no intermediate copy
        if out.is_cuda or not out.is_contiguous() or tuple(out.shape) != shape or out.element_size() != np.dtype(dtype).itemsize:
            raise TypeError('out must be a contiguous host tensor of shape %s' % (shape,))
        p, nbytes = out.data_ptr(), out.numel() * out.element_size()
    else:
        if out.dtype != dtype or not out.flags['C_CONTIGUOUS'] or out.shape != shape:
            raise TypeError('out must be a C-contiguous %s array of shape %s' % (np.dtype(dtype).name, shape))
        p, nbytes = out.ctypes.data, out.nbytes
    check(getattr(_lib.lib(), fn_name)(data, len(data), c_void_p(p), nbytes), fn_name)
    return out


def decode_png_rgb8(src, out=None):
    """what `np.asarray(Image.open(path).convert('RGB'))` holds (src/data_utils.py:149-152): uint8 [H, W, 3]; `out` may be a numpy array or a
    (pinned) host torch tensor to decode into"""
    import numpy as np
    return _decode_png(src, out, 'ptta_png_decode_rgb8', np.uint8, 3)


def decode_png_gray16(src, out=None):
    """what `np.array(Image.open(path))` holds for a 16-bit (or 8-bit) grey depth map (src/data_utils.py:186, 219): uint16 [H, W]"""
    import numpy as np
    return _decode_png(src, out, 'ptta_png_decode_gray16', np.uint16, 1)
