"""Shared-model mode of the NLSPN back-end (one model over all GPUs: SyncBatchNorm sums of every train-mode BatchNorm and the gradient
mean all-reduce fused with Adam, through NVLink peer memory, csrc/peer_comm.cuh).  On one GPU the world-1 plumbing and the refusals run;
the world-2 check needs two GPUs of one node (tools/shared_check.py --model nlspn under torch.distributed.run)."""
import json
import os
import subprocess
import sys

import pytest
import torch

from golden_util import rel

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H, W, CAP, LR = 64, 128, 80.0, 3e-4


def make_model(sd, syncbn=True):
    from tta_depth_completion_b200 import ExternalModel_Adapt, synthetic
    m = ExternalModel_Adapt('nlspn', 0.0, 100.0, max_input_depth=CAP, offset=True, dataset_name='kitti', device=torch.device('cuda:0'))
    m._prepare_head(synthetic.NLSPN_PREPARE_MODE)
    m.load_state_dict(sd)
    if syncbn:
        m.convert_syncbn()
    m.set_image_normalization([1.0 / (255.0 * s) for s in synthetic.IMAGENET_STD],
                              [-mu / s for mu, s in zip(synthetic.IMAGENET_MEAN, synthetic.IMAGENET_STD)])
    m.train()
    return m


@pytest.mark.parametrize('graph', [False, True])
def test_world1_shared_step_equals_plain_step(graph):
    """world 1: the communicator exists, the step is the plain step -- step 0 bit-identical (same kernels on the same inputs), gradients
    within the atomics bound of the propagation backward"""
    from tta_depth_completion_b200 import sharding, synthetic
    dev = torch.device('cuda:0')
    sd = synthetic.make_nlspn_checkpoint(0)
    a, b = make_model(sd), make_model(sd)
    comm = sharding.enable_shared_model(b)
    assert comm.world == 1 and comm.grad_floats == b.model._base.flat_g.numel()
    img_a, sp_a = torch.empty((1, 3, H, W), device=dev), torch.empty((1, 1, H, W), device=dev)
    img_b, sp_b = torch.empty_like(img_a), torch.empty_like(sp_a)
    stream = torch.cuda.Stream(dev)            # a step can only be captured on a non-default stream
    with torch.cuda.stream(stream):
        for t in range(3):
            image, sparse, _ = synthetic.synthetic_frame(5, t, 1, H, W, 'kitti')
            img_a.copy_(image.to(dev)); sp_a.copy_(sparse.to(dev)); img_b.copy_(img_a); sp_b.copy_(sp_a)
            a.tta_step(img_a, sp_a, LR, 1.0, 1.0, 0.1, graph=graph)
            sharding.shared_model_step(b, img_b, sp_b, LR, 1.0, 1.0, 0.1, graph=graph)
            ea, eb = a.model._engines[(1, H, W)], b.model._engines[(1, H, W)]
            assert eb._comm is comm
            la, lb = a.last_losses(), b.last_losses()
            if t == 0:
                assert torch.equal(ea.B['output'], eb.B['output']) and torch.equal(ea.emb, eb.emb) and torch.equal(ea.ref, eb.ref)
                assert la == lb, (la, lb)
                for k in ea.adapt_names:
                    assert float((ea.grads[k] - eb.grads[k]).norm()) <= 5e-2 * float(ea.grads[k].norm()) + 1e-7, k
            else:
                assert rel(la['loss'], lb['loss']) < 6e-2, (t, la, lb)
    torch.cuda.synchronize()
    assert comm.error() == 0
    if graph:
        assert eb._graph is not None and int(eb.adam_step_dev.item()) == 3


def test_shared_nlspn_refusals():
    """enable_shared_model without convert_syncbn, the autograd path and the stage-2 head_step on a shared model raise"""
    from tta_depth_completion_b200 import sharding, synthetic
    dev = torch.device('cuda:0')
    sd = synthetic.make_nlspn_checkpoint(1)
    with pytest.raises(RuntimeError, match='convert_syncbn'):
        sharding.enable_shared_model(make_model(sd, syncbn=False))
    m = make_model(sd)
    sharding.enable_shared_model(m)
    image, sparse, _ = synthetic.synthetic_frame(5, 0, 1, H, W, 'kitti')
    image, sparse = image.to(dev), sparse.to(dev)
    with pytest.raises(RuntimeError, match='shared model'):
        m.forward(image=synthetic.normalize_image_imagenet(image.cpu()).to(dev), sparse_depth=sparse,
                  loss_type='adapt_meta_selfsup_seq_ema_reverse')
    with pytest.raises(RuntimeError, match='shared model'):
        m.head_step(image, sparse, 1e-3)
    # the eval forward keeps local statistics and stays available
    m.eval()
    out = m.forward(image=synthetic.normalize_image_imagenet(image.cpu()).to(dev), sparse_depth=sparse, loss_type='pretrain')
    assert tuple(out.shape) == (1, 1, H, W) and bool(torch.isfinite(out).all())


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs of one node')
def test_world2_nlspn_replicas_identical_and_equal_to_the_big_batch():
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1', '--master-port', '29733',
           os.path.join(ROOT, 'tools', 'shared_check.py'), '--model', 'nlspn']
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    line = [l for l in res.stdout.splitlines() if l.startswith('{')][-1]
    out = json.loads(line)
    assert out['world'] == 2 and out['model'] == 'nlspn'
    for key in ('eager', 'graph'):
        assert out[key]['comm_error'] == 0 and out[key]['exchanges_per_step'] == 125
        assert 'step0_grad_worst' in out[key]


def _comm_world1(grad_floats):
    from tta_depth_completion_b200 import sharding
    return sharding.PeerCommunicator(grad_floats)


def test_world1_exchange_kernels_equal_plain_kernels():
    """the communicator-aware entry points on a one-rank communicator: the rank-order sum is 0 + the local sum and the count rows x 1, so
    BatchNorm statistics, BatchNorm backward and Adam must equal the plain kernels bit for bit -- over several steps (epoch advance, both
    slot parities, low and high exchange ids), eager and replayed from a CUDA graph"""
    from tta_depth_completion_b200 import _lib
    from tta_depth_completion_b200._lib import check, ptr, c_void_p
    L = _lib.lib()
    dev = torch.device('cuda:0')
    g = torch.Generator().manual_seed(31)
    n_adam = 46000
    comm = _comm_world1(n_adam)
    cases = []
    for rows, c, act in ((1000, 64, 1), (4096, 192, 2), (515, 1024, 1)):
        nblk = L.ptta_nl_reduce_blocks(rows, c)
        t = {'x': (torch.randn((rows, c), generator=g) * 1.5 + 0.3).to(dev).to(torch.bfloat16),
             'dy': torch.randn((rows, c), generator=g).to(dev).to(torch.bfloat16),
             'dy_b': torch.randn((rows, c), generator=g).to(dev).to(torch.bfloat16),
             'gamma': (1 + 0.1 * torch.randn(c, generator=g)).to(dev), 'beta': (0.1 * torch.randn(c, generator=g)).to(dev)}
        t['y'] = torch.relu(t['x'].float()).to(torch.bfloat16) if act == 1 else t['x'].clone()
        for side in ('p', 'c'):
            t['partial_' + side] = torch.empty(2 * c * nblk, device=dev)
            for k in ('mean', 'rstd', 'scale', 'shift', 'dgamma', 'dbeta'):
                t[k + '_' + side] = torch.zeros(c, device=dev)
            t['rm_' + side], t['rv_' + side] = torch.zeros(c, device=dev), torch.ones(c, device=dev)
            t['coef_' + side] = torch.empty(3 * c, device=dev)
            t['dx_' + side], t['gskip_' + side] = torch.empty_like(t['x']), torch.empty_like(t['x'])
        cases.append((rows, c, act, t))
    ad = {k: torch.randn(n_adam, generator=g).to(dev) * s for k, s in (('p', 1.0), ('g', 1e-2), ('m', 1e-3))}
    ad['v'] = torch.rand(n_adam, generator=g).to(dev) * 1e-4
    adam = {side: {k: v.clone() for k, v in ad.items()} for side in ('p', 'c')}
    hyper = torch.tensor([3e-4, 0.9, 0.999, 1e-8, 0.0], dtype=torch.float64, device=dev)
    steps = {side: torch.zeros(1, dtype=torch.int32, device=dev) for side in ('p', 'c')}

    def one_step(st):
        for k, (rows, c, act, t) in enumerate(cases):
            for side in ('p', 'c'):
                a = (ptr(t['x']), c, rows, c, ptr(t['gamma']), ptr(t['beta']), 1e-5, ptr(t['partial_' + side]), ptr(t['mean_' + side]),
                     ptr(t['rstd_' + side]), ptr(t['scale_' + side]), ptr(t['shift_' + side]), ptr(t['rm_' + side]), ptr(t['rv_' + side]), None, 0.1)
                if side == 'p':
                    check(L.ptta_nl_bn_stats(*a, st))
                else:
                    check(L.ptta_nl_bn_stats_comm(*a, comm.handle, k, st))
            for side in ('p', 'c'):
                a = (ptr(t['dy']), c, ptr(t['dy_b']), c, ptr(t['y']), act, ptr(t['x']), ptr(t['mean_' + side]), ptr(t['rstd_' + side]), ptr(t['gamma']),
                     ptr(t['partial_' + side]), ptr(t['dgamma_' + side]), ptr(t['dbeta_' + side]), ptr(t['coef_' + side]), ptr(t['dx_' + side]),
                     ptr(t['gskip_' + side]), rows, c)
                if side == 'p':
                    check(L.ptta_nl_bn_backward(*a, st))
                else:
                    check(L.ptta_nl_bn_backward_comm(*a, comm.handle, 253 + k, st))      # up to the last exchange id
        p_, c_ = adam['p'], adam['c']
        check(L.ptta_adam_flat_dev(ptr(p_['p']), ptr(p_['g']), ptr(p_['m']), ptr(p_['v']), n_adam, ptr(hyper), ptr(steps['p']), st))
        check(L.ptta_adam_flat_dev_comm(ptr(c_['p']), ptr(c_['g']), ptr(c_['m']), ptr(c_['v']), n_adam, ptr(hyper), ptr(steps['c']), comm.handle, 7, st))
        check(L.ptta_comm_advance(comm.handle, st))

    def compare(step):
        torch.cuda.synchronize()
        for rows, c, act, t in cases:
            for k in ('mean', 'rstd', 'scale', 'shift', 'rm', 'rv', 'dgamma', 'dbeta', 'coef', 'dx', 'gskip'):
                assert torch.equal(t[k + '_p'], t[k + '_c']), (step, rows, c, k)
        for k in ('p', 'g', 'm', 'v'):
            assert torch.equal(adam['p'][k], adam['c'][k]), (step, 'adam', k)
        assert torch.equal(steps['p'], steps['c'])

    stream = torch.cuda.Stream(dev)
    with torch.cuda.stream(stream):
        for s in range(3):
            one_step(c_void_p(stream.cuda_stream))
            compare(s)
        graph = torch.cuda.CUDAGraph()
        torch.cuda.synchronize()
        with torch.cuda.graph(graph):
            one_step(c_void_p(torch.cuda.current_stream().cuda_stream))
        for s in range(3, 6):
            graph.replay()
            compare(s)
    assert int(steps['c'].item()) == 6
    assert comm.error() == 0


@pytest.mark.parametrize('graph', [False, True])
def test_world1_exchanging_step_equals_plain_step(graph):
    """the whole NLSPN step through the exchanging kernels on a one-rank communicator (set_comm(..., exchange_at_world1=True)): one stream,
    125 exchanges per step, the epoch advanced at the end; step 0 computes the plain step's forward and losses bit for bit, the gradients
    within the atomics bound of the propagation backward"""
    from tta_depth_completion_b200 import synthetic
    from tta_depth_completion_b200.nlspn_engine import NlspnEngine
    dev = torch.device('cuda:0')
    engines = [NlspnEngine(synthetic.make_nlspn_checkpoint(3), 1, H, W, dev) for _ in range(2)]
    a, b = engines
    comm = _comm_world1(b.flat_g.numel())
    b.set_comm(comm, exchange_at_world1=True)
    for e in engines:
        e.set_image_normalization([1.0 / (255.0 * s) for s in synthetic.IMAGENET_STD],
                                  [-mu / s for mu, s in zip(synthetic.IMAGENET_MEAN, synthetic.IMAGENET_STD)])
    img_d, sp_d = torch.empty((1, 3, H, W), device=dev), torch.empty((1, 1, H, W), device=dev)
    stream = torch.cuda.Stream(dev)
    with torch.cuda.stream(stream):
        for t in range(3):
            image, sparse, _ = synthetic.synthetic_frame(7, t, 1, H, W, 'kitti')
            img_d.copy_(image.to(dev)); sp_d.copy_(sparse.to(dev))
            for e in engines:
                e.tta_step(img_d, img_d, sp_d, LR, 1.0, 1.0, 0.1, CAP, graph=graph)
            la, lb = a.read_losses(), b.read_losses()
            assert b.exchanges_per_step == 125
            if t == 0:
                assert torch.equal(a.B['output'], b.B['output']) and torch.equal(a.emb, b.emb) and torch.equal(a.ref, b.ref)
                assert la == lb, (la, lb)
                for k in a.adapt_names:
                    assert float((a.grads[k] - b.grads[k]).norm()) <= 5e-2 * float(a.grads[k].norm()) + 1e-7, k
            else:
                assert rel(la['loss'], lb['loss']) < 6e-2, (t, la, lb)
    torch.cuda.synchronize()
    assert comm.error() == 0
    assert int(b.adam_step_dev.item()) == 3
    if graph:
        assert b._graph is not None
