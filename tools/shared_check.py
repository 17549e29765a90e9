#!/usr/bin/env python
"""Shared-model mode check, launched as `python -m torch.distributed.run --nproc-per-node W tools/shared_check.py` (W >= 2 GPUs of one node).

Every rank adapts the SAME model on its own batch-1 frame per step through the peer-memory path (SyncBatchNorm sums + gradient all-reduce
fused with Adam, csrc/peer_comm.cuh).  Checked: (1) the adapted tensors, BatchNorm buffers and Adam moments are BIT-IDENTICAL on all
ranks after every step; (2) they equal a single-GPU step on the batch of all W frames (what DDP + SyncBatchNorm is defined to reproduce)
up to fp32 summation order; (3) the CUDA-graph replay of the step gives the same result as eager launches.  Prints one JSON line.
`--stage init | head` runs the same three checks on the source-domain preparation steps (the reference's src/init_main.py and
src/head_main.py are DDP + SyncBatchNorm trainers: one model, every rank its own batch, gradients averaged).
`--model nlspn` runs the NLSPN back-end's shared-model step instead (check_nlspn below); `--model msg_chn` is the default."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from tta_depth_completion_b200 import ExternalModel_Adapt, sharding, synthetic

MODE, CAP, LR = 'meta_selfsup_seq_2layers_ema', 80.0, 1e-4
H, W_, STEPS = 64, 128, 3


STAGE, MODEL = 'tta', 'msg_chn'
for _i, _a in enumerate(sys.argv):
    if _a == '--stage':
        STAGE = sys.argv[_i + 1]
    if _a == '--model':
        MODEL = sys.argv[_i + 1]


def run_step(model, image, sparse, dense, graph):
    if STAGE == 'tta':
        sharding.shared_model_step(model, image, sparse, LR, 1.0, 1.0, 0.1, graph=graph)
    elif STAGE == 'init':
        model.init_step(image, sparse, dense, 1e-3, graph=graph)
    else:
        model.head_step(image, sparse, 1e-3, graph=graph)


def make_model(dev, sd):
    m = ExternalModel_Adapt('msg_chn', 0.0, 100.0, max_input_depth=CAP, device=dev)
    # the kernel dispatch depends on the pixel count of a map (N x H x W): force the tcgen05 kernels everywhere, so that the per-rank
    # batch-1 engines and the single-GPU batch-W engine run the SAME kernels and differ by summation order only
    m.model.engine_options = {'tc_min_pixels': 0, 'tc_s2_min_pixels': 0, 'tc_t2_min_pixels': 0, 'tc_head_min_pixels': 0, 'tc_stem_min_pixels': 0}
    m._prepare_head(MODE)
    m.load_state_dict(sd)
    if STAGE == 'head':
        torch.manual_seed(11)                                   # the same fresh heads on every rank (src/head_main.py:268)
        m.prepare_parameters('head_selfsup_ema')
    m.set_image_normalization((1 / 255.0,) * 3, (0.0,) * 3)
    m.train()
    return m


def nrel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def main():
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ.get('LOCAL_RANK', '0'))
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    dist.init_process_group('nccl', device_id=dev)
    sd = synthetic.get_checkpoint('kitti_2layers_a', MODE) if synthetic.fitted_checkpoint_available('kitti_2layers_a') else synthetic.make_synthetic_checkpoint(0, MODE)
    out = {'world': world}
    torch.cuda.set_stream(torch.cuda.Stream(dev))          # a step can only be captured on a non-default stream
    for use_graph in (False, True):
        model = make_model(dev, sd)
        comm = sharding.enable_shared_model(model)
        losses = []
        for t in range(STEPS):
            image, sparse, dense = synthetic.synthetic_frame(40, t * world + rank, 1, H, W_, 'kitti')
            run_step(model, image.to(dev), sparse.to(dev), dense.to(dev), use_graph)
            losses.append(model.last_losses()['loss'])
            # (1) replicas identical, bit for bit
            flat = torch.cat([model.model._flat['param'], model.model._flat['m'], model.model._flat['v'], model.model._flat['grad']])
            gathered = [torch.empty_like(flat) for _ in range(world)]
            dist.all_gather(gathered, flat)
            for r in range(world):
                assert torch.equal(gathered[r], gathered[0]), 'replicas differ at step %d (rank %d vs 0, graph=%s)' % (t, r, use_graph)
            bufs = torch.cat([v.float().flatten() for k, v in model.state_dict().items() if 'running' in k])
            gb = [torch.empty_like(bufs) for _ in range(world)]
            dist.all_gather(gb, bufs)
            for r in range(world):
                assert torch.equal(gb[r], gb[0]), 'BatchNorm buffers differ at step %d' % t
        assert comm.error() == 0, 'peer exchange %d timed out' % (comm.error() - 1)
        lt = torch.tensor(losses, device=dev, dtype=torch.float64)
        dist.all_reduce(lt)
        mean_losses = (lt / world).tolist()
        key = 'graph' if use_graph else 'eager'
        out[key] = {'mean_loss': mean_losses}
        # (2) single-GPU step on the whole batch (rank 0 only)
        if rank == 0:
            big = make_model(dev, sd)
            big_losses = []
            for t in range(STEPS):
                frames = [synthetic.synthetic_frame(40, t * world + r, 1, H, W_, 'kitti') for r in range(world)]
                image = torch.cat([f[0] for f in frames]).to(dev)
                sparse = torch.cat([f[1] for f in frames]).to(dev)
                dense = torch.cat([f[2] for f in frames]).to(dev)
                if STAGE == 'tta':
                    big.tta_step(image, sparse, LR, 1.0, 1.0, 0.1)
                elif STAGE == 'init':
                    big.init_step(image, sparse, dense, 1e-3)
                else:
                    big.head_step(image, sparse, 1e-3)
                big_losses.append(big.last_losses()['loss'])
            sa, sb = model.state_dict(), big.state_dict()
            errs = {}
            for k in model.model._adapt_names:
                if k in ('conv1_rgb_meta.conv1_meta.1.bias', 'pred.0.bias'):     # bias in front of a train-mode BatchNorm: analytically zero gradient, pure rounding noise
                    continue
                upd = nrel(sd[k].to(dev), sb[k])
                errs[k] = (nrel(sa[k], sb[k]), upd)
            worst = max(e / max(u, 1e-30) for e, u in errs.values())
            buf_err = max(nrel(sa[k].float(), sb[k].float()) for k in sa if 'running' in k)
            loss_err = max(abs(a - b) / abs(b) for a, b in zip(mean_losses, big_losses))
            out[key].update(worst_error_over_update=worst, bn_buffer_error=buf_err, loss_error=loss_err, big_batch_loss=big_losses)
            assert loss_err < 2e-3, (mean_losses, big_losses)
            assert buf_err < 1e-4, buf_err
            assert worst < 0.05, errs           # fp32 summation order only (per-rank wgrad partial sums vs one sum) through Adam's 1/sqrt(v)
        dist.barrier()
    out['stage'] = STAGE
    if rank == 0:
        print(json.dumps(out), flush=True)
    dist.destroy_process_group()


# ---- NLSPN back-end ------------------------------------------------------------------------------------------------------------------
# 64x128 frames, synthetic NLSPN checkpoint; sequence NL_SEQ, frame t*W + r on rank r (the big batch stacks them in rank order)
NL_SEQ, NL_LR, NL_STEPS = 23, 3e-4, 3
# Bounds, with the values measured on the first run (2 ranks time-sliced on one B200, profiles/nlspn_shared_check_2ranks.json; eager | graph):
#   step-0 loss, mean of the ranks' losses vs the big batch's: measured 0.0 | 0.0 -> bound 1e-5
#   step-0 gradients, norm-relative per tensor: measured worst 1.01e-2 | 1.02e-2 (conv4.0.bn1.bias), median 5.6e-3 | 5.4e-3 -> the atomics
#     bound of the NLSPN tests, 5e-2 (the fp32 atomics of the propagation backward sum in a different order on every run and the bf16
#     backward chain amplifies them; a world-size factor on the BatchNorm affine gradients would be an error of 1.0).  No tensor excluded.
#   weights after 3 steps, max |diff|: measured 1.5e-3 | 1.2e-3 -> the bound of test_graph_replay_equals_eager, 2.4 lr per step = 2.16e-3
#   norm-relative on conv2.0.bn1.weight / dec2.1.weight: measured 9.8e-5 / 3.3e-5 | 9.1e-5 / 3.8e-5 -> the same test's 5e-3
#   w_cos_eff (loss_cos >= 0.3 on every rank and in the big batch, so the cosine term is on): 0.1 for both ranks and the big batch, all steps
NL_GRAD_BOUND, NL_LOSS_BOUND = 5e-2, 1e-5


def make_nlspn_model(dev, sd):
    m = ExternalModel_Adapt('nlspn', 0.0, 100.0, max_input_depth=CAP, offset=True, dataset_name='kitti', device=dev)
    m._prepare_head(synthetic.NLSPN_PREPARE_MODE)
    m.load_state_dict(sd)
    m.convert_syncbn()
    m.set_image_normalization([1.0 / (255.0 * s) for s in synthetic.IMAGENET_STD],
                              [-mu / s for mu, s in zip(synthetic.IMAGENET_MEAN, synthetic.IMAGENET_STD)])
    m.train()
    return m


def check_nlspn():
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ.get('LOCAL_RANK', '0'))
    # one GPU per rank (NCCL for the checker's own gathers); on a node with fewer GPUs than ranks the ranks share them, time-sliced
    # (gloo for the gathers; NCCL refuses two ranks on one device) -- the exchanges and the numerics are the same, the timing is not
    n_dev = torch.cuda.device_count()
    shared_gpu = n_dev < world
    dev = torch.device('cuda', local % n_dev)
    torch.cuda.set_device(dev)
    if shared_gpu:
        dist.init_process_group('gloo')
    else:
        dist.init_process_group('nccl', device_id=dev)
    sd = synthetic.make_nlspn_checkpoint(0)
    out = {'world': world, 'model': 'nlspn', 'gpus': min(n_dev, world), 'gpu_name': torch.cuda.get_device_name(dev),
           'frames': [1, 3, H, W_], 'sequence': NL_SEQ, 'steps': NL_STEPS}
    torch.cuda.set_stream(torch.cuda.Stream(dev))
    img_d = torch.empty((1, 3, H, W_), device=dev)
    sp_d = torch.empty((1, 1, H, W_), device=dev)
    for use_graph in (False, True):
        model = make_nlspn_model(dev, sd)
        comm = sharding.enable_shared_model(model)
        model.model._engine_for(img_d)
        eng = model.model._engines[(1, H, W_)]           # parameters, gradients and moments are shared by all engines of the model
        names = eng.adapt_names
        losses, grads0 = [], None
        for t in range(NL_STEPS):
            image, sparse, _ = synthetic.synthetic_frame(NL_SEQ, t * world + rank, 1, H, W_, 'kitti')
            img_d.copy_(image.to(dev)); sp_d.copy_(sparse.to(dev))
            sharding.shared_model_step(model, img_d, sp_d, NL_LR, 1.0, 1.0, 0.1, graph=use_graph)
            losses.append(model.last_losses())
            if t == 0:
                grads0 = {k: eng.grads[k].clone() for k in names}        # the averaged gradient (written back by the fused Adam)
            # (1) replicas identical, bit for bit: parameters, averaged gradients, Adam moments
            flat = torch.cat([eng.flat_p, eng.flat_g, eng.flat_m, eng.flat_v])
            if shared_gpu:
                flat = flat.cpu()
            gathered = [torch.empty_like(flat) for _ in range(world)]
            dist.all_gather(gathered, flat)
            for r in range(world):
                assert torch.equal(gathered[r], gathered[0]), 'replicas differ at step %d (rank %d vs 0, graph=%s)' % (t, r, use_graph)
        assert comm.error() == 0, 'peer exchange %d timed out' % (comm.error() - 1)
        per_rank = [None] * world
        dist.all_gather_object(per_rank, losses)
        key = 'graph' if use_graph else 'eager'
        out[key] = {'exchanges_per_step': eng.exchanges_per_step, 'comm_error': comm.error(),
                    'w_cos_eff_per_rank': [[l['w_cos_eff'] for l in pr] for pr in per_rank]}
        if use_graph:
            out[key]['graph_replayed'] = eng._graph is not None
            assert eng._graph is not None
        # (2) the single-GPU step on the batch of all W frames (rank 0)
        if rank == 0:
            big = make_nlspn_model(dev, sd)
            beng = None
            big_losses, big_grads0 = [], None
            for t in range(NL_STEPS):
                frames = [synthetic.synthetic_frame(NL_SEQ, t * world + r, 1, H, W_, 'kitti') for r in range(world)]
                image = torch.cat([f[0] for f in frames]).to(dev)
                sparse = torch.cat([f[1] for f in frames]).to(dev)
                big.tta_step(image, sparse, NL_LR, 1.0, 1.0, 0.1)
                big_losses.append(big.last_losses())
                beng = big.model._base
                if t == 0:
                    big_grads0 = {k: beng.grads[k].clone() for k in names}
            mean0 = sum(pr[0]['loss'] for pr in per_rank) / world
            loss_err = abs(mean0 - big_losses[0]['loss']) / abs(big_losses[0]['loss'])
            w_big = [l['w_cos_eff'] for l in big_losses]
            gerr = {k: nrel(grads0[k], big_grads0[k]) for k in names}
            worst_g = max(gerr, key=gerr.get)
            sa, sb = model.state_dict(), big.state_dict()
            werr = {k: float((sa[k] - sb[k]).abs().max()) for k in names}
            worst_w = max(werr, key=werr.get)
            moved = {k: nrel(sa[k], sb[k]) for k in names if k.endswith('dec2.1.weight') or k.endswith('conv2.0.bn1.weight')}
            out[key].update(step0_loss_mean_over_ranks=mean0, step0_big_batch_loss=big_losses[0]['loss'], step0_loss_error=loss_err,
                            w_cos_eff_big_batch=w_big, step0_grad_worst=(worst_g, gerr[worst_g]),
                            step0_grad_median=sorted(gerr.values())[len(gerr) // 2], weights_max_abs_diff=(worst_w, werr[worst_w]),
                            weights_max_abs_bound=2.4 * NL_LR * NL_STEPS, weights_nrel_moved=moved)
            print(json.dumps({key: out[key]}), file=sys.stderr, flush=True)      # the measured values, also when a bound below fails
            assert all(pr[t]['w_cos_eff'] == w_big[t] for pr in per_rank for t in range(NL_STEPS)), \
                ('ranks and the big batch disagree on w_cos_eff: pick other data', out[key]['w_cos_eff_per_rank'], w_big)
            assert loss_err < NL_LOSS_BOUND, out[key]
            assert gerr[worst_g] <= NL_GRAD_BOUND, out[key]
            assert werr[worst_w] <= 2.4 * NL_LR * NL_STEPS, out[key]
            assert all(v < 5e-3 for v in moved.values()), out[key]
        dist.barrier()
    if rank == 0:
        print(json.dumps(out), flush=True)
    dist.destroy_process_group()


if __name__ == '__main__':
    check_nlspn() if MODEL == 'nlspn' else main()
