"""Eval-time hole filling on the device (ops.inpaint_biharmonic, csrc/inpaint.cuh) against the CPU oracle (oracle/inpaint_oracle.py,
scikit-image 0.18's algorithm): every filled pixel within 1e-5 x (max - min) of the sample's known range, every other pixel untouched."""
import warnings

import numpy as np
import pytest
import torch

from oracle import inpaint_oracle as IO

pytestmark = pytest.mark.gpu


def _field(n, h, w, seed):
    g = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    d = np.empty((n, 1, h, w), np.float32)
    for b in range(n):
        a = g.uniform(0.5, 2.0, size=4)
        d[b, 0] = 20 + 10 * a[0] * np.sin(x / (7 * a[1])) + 8 * a[2] * np.cos(y / (5 * a[3])) + g.random((h, w))
    return d


def _check(d):
    from tta_depth_completion_b200 import ops
    ref = IO.inpainting(d)
    got_t = torch.from_numpy(d).cuda()
    ops.inpaint_biharmonic(got_t)
    got = got_t.cpu().numpy()
    holes = d == 0
    assert np.array_equal(got[~holes], d[~holes])
    for b in range(d.shape[0]):
        known = d[b][~holes[b]]
        tol = 1e-5 * float(known.max() - known.min())
        err = np.abs(got[b] - ref[b]).max()
        assert err <= tol, (b, err, tol)
    return got


def test_scattered_single_pixels():
    d = _field(1, 48, 96, 0)
    g = np.random.default_rng(10)
    d[0, 0][g.random((48, 96)) < 0.01] = 0.0
    _check(d)


def test_blobs():
    d = _field(1, 64, 96, 1)
    d[0, 0, 10:22, 15:40] = 0.0
    d[0, 0, 30:50, 60:70] = 0.0
    d[0, 0, 40:43, 20:23] = 0.0
    _check(d)


def test_components_touching_edge_and_corner():
    d = _field(1, 40, 56, 2)
    d[0, 0, 0:6, 10:30] = 0.0          # top edge
    d[0, 0, 15:25, 50:56] = 0.0        # right edge
    d[0, 0, 33:40, 0:9] = 0.0          # bottom-left corner
    d[0, 0, 0, 0] = 0.0                # single corner pixel
    d[0, 0, 1, 55] = 0.0               # one pixel from the top-right corner
    _check(d)


def test_two_holes_two_pixels_apart():
    d = _field(1, 24, 32, 3)
    d[0, 0, 10, 10] = 0.0
    d[0, 0, 10, 12] = 0.0              # within stencil reach: one component
    d[0, 0, 15, 20] = 0.0
    d[0, 0, 17, 20] = 0.0
    d[0, 0, 4, 4] = 0.0
    d[0, 0, 6, 7] = 0.0                # out of reach of (4, 4): two components
    _check(d)


def test_top_band():
    d = _field(1, 48, 160, 4)
    d[0, 0, 0:8, :] = 0.0
    _check(d)


def test_batch_of_three_with_a_sample_without_holes():
    d = _field(3, 40, 64, 5)
    g = np.random.default_rng(11)
    d[0, 0][g.random((40, 64)) < 0.05] = 0.0
    d[2, 0, 5:20, 30:50] = 0.0
    d[2, 0, 0:3, 0:64] = 0.0
    got = _check(d)
    assert np.array_equal(got[1], d[1])


def test_no_holes_untouched_and_all_zero_sample_raises():
    from tta_depth_completion_b200 import ops
    d = torch.from_numpy(_field(2, 16, 24, 6)).cuda()
    ref = d.clone()
    ops.inpaint_biharmonic(d)
    assert torch.equal(d, ref)
    d[1] = 0.0
    with pytest.raises(ValueError):
        ops.inpaint_biharmonic(d)


def test_wrapper_eval_forward_fills_holes_like_the_reference():
    """a synthetic NLSPN checkpoint with id_dec0.0.bias shifted negative: the eval prediction has holes, and the wrapper returns
    oracle.inpainting(engine eval output) without a warning"""
    from tta_depth_completion_b200 import synthetic
    from tta_depth_completion_b200.nlspn_model_adapt import NLSPNModel_Adapt
    dev = torch.device('cuda:0')
    n, h, w = 1, 32, 64
    image, sparse, _ = synthetic.synthetic_frame(3, 0, n, h, w, 'kitti')
    image = synthetic.normalize_image_imagenet(image).to(dev)
    sparse = sparse.to(dev)
    base = synthetic.make_nlspn_checkpoint(0)
    for shift in (8.0, 9.0, 10.0, 7.0, 11.0, 6.0, 12.0):
        sd = {k: v.clone() for k, v in base.items()}
        sd['id_dec0.0.bias'] -= shift
        m = NLSPNModel_Adapt(device=dev, offset=True)
        m._prepare_head(synthetic.NLSPN_PREPARE_MODE)
        m.load_state_dict(sd)
        m.eval()
        eng = m._engine_for(image)
        eng.repack_adapted()
        with torch.no_grad():
            raw = eng.forward(image, sparse, training=False).clone()
        frac = float((raw == 0).float().mean())
        if 0.002 <= frac <= 0.6:
            break
    assert 0.002 <= frac <= 0.6, frac
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter('always')
        out = m.forward(image, sparse, loss_type='pretrain')
    assert not [r for r in rec if issubclass(r.category, RuntimeWarning)], [str(r.message) for r in rec]
    assert not hasattr(m, 'warn_on_holes')
    raw = raw.cpu().numpy()
    ref = IO.inpainting(raw)
    got = out.cpu().numpy()
    holes = raw == 0
    assert np.array_equal(got[~holes], raw[~holes])
    known = raw[~holes]
    assert np.abs(got - ref).max() <= 1e-5 * float(known.max() - known.min())
