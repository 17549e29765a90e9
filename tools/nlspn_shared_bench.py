#!/usr/bin/env python
"""Throughput of the NLSPN shared-model mode (one model over all GPUs: SyncBatchNorm over the ranks, gradient mean all-reduce fused with
Adam, csrc/peer_comm.cuh) against the shards mode (one model per GPU, `bench.py --workload nlspn`), at 352x1216, in one call:

    python tools/nlspn_shared_bench.py [--gpus 2,8] [--steps 50] [--warmup 5] [--out FILE]

launches, for every world size W in --gpus that the node has, `torch.distributed.run --nproc-per-node W` of this script in worker mode
(the shared step at per-GPU batch 1 and 2, replayed from its CUDA graph) and of `bench.py --workload nlspn --gpus W` (shards), reads the
card name and power limit, and prints one JSON line (also written to --out).  Frames/s = W x batch x steps / the slowest rank's time
between two device events around the timed steps (frames already on the device)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
H, W_, LR, CAP = 352, 1216, 3e-4, 80.0
RING = 4


def worker(args):
    import torch
    import torch.distributed as dist
    from tta_depth_completion_b200 import ExternalModel_Adapt, sharding, synthetic
    rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ.get('LOCAL_RANK', '0'))
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    dist.init_process_group('nccl', device_id=dev)
    sd = synthetic.make_nlspn_checkpoint(0)
    stream = torch.cuda.Stream(dev)
    results, comms = {}, []
    for batch in (1, 2):
        m = ExternalModel_Adapt('nlspn', 0.0, 100.0, max_input_depth=CAP, offset=True, dataset_name='kitti', device=dev)
        m._prepare_head(synthetic.NLSPN_PREPARE_MODE)
        m.load_state_dict(sd)
        m.convert_syncbn()
        m.set_image_normalization([1.0 / (255.0 * s) for s in synthetic.IMAGENET_STD],
                                  [-mu / s for mu, s in zip(synthetic.IMAGENET_MEAN, synthetic.IMAGENET_STD)])
        m.train()
        comm = sharding.enable_shared_model(m)
        frames = [[x.to(dev) for x in synthetic.synthetic_frame(1 + rank, i, batch, H, W_, 'kitti')[:2]] for i in range(RING)]
        img_d, sp_d = torch.empty_like(frames[0][0]), torch.empty_like(frames[0][1])
        with torch.cuda.stream(stream):
            for i in range(args.warmup + 2):                 # first call eager, second captures, then replays
                img_d.copy_(frames[i % RING][0]); sp_d.copy_(frames[i % RING][1])
                sharding.shared_model_step(m, img_d, sp_d, LR, 1.0, 1.0, 0.1, graph=True)
            torch.cuda.synchronize(dev)
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for i in range(args.steps):
                img_d.copy_(frames[i % RING][0], non_blocking=True); sp_d.copy_(frames[i % RING][1], non_blocking=True)
                sharding.shared_model_step(m, img_d, sp_d, LR, 1.0, 1.0, 0.1, graph=True)
            e1.record(stream)
            torch.cuda.synchronize(dev)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = float(ms[0])
        eng = m.model._engines[(batch, H, W_)]
        err = comm.error()
        losses = m.last_losses()
        results['batch%d' % batch] = {'adapted_frames_per_sec': world * batch * args.steps / (ms / 1e3), 'ms_per_step': ms / args.steps,
                                      'per_gpu_batch': batch, 'exchanges_per_step': eng.exchanges_per_step, 'graph_replayed': eng._graph is not None,
                                      'comm_error': err, 'last_losses_rank0': losses}
        assert err == 0, 'peer exchange %d timed out' % (err - 1)
        comms.append(comm)                                    # kept alive until every rank is done with the peer blocks
    dist.barrier()
    if rank == 0:
        print(json.dumps({'world': world, 'steps': args.steps, 'warmup': args.warmup, 'shared': results}), flush=True)
    dist.destroy_process_group()


def stream_layout_leg(args):
    """One GPU: the plain NLSPN step with the zero-image branch on its own stream (the default) and on the main stream (the layout of the
    shared-model step, without its exchanges), per-GPU batch 1 and 2, CUDA graph replay -- the part of the shared mode's cost that one GPU
    can show"""
    import torch
    from tta_depth_completion_b200 import synthetic
    from tta_depth_completion_b200.nlspn_engine import NlspnEngine
    dev = torch.device('cuda', 0)
    stream = torch.cuda.Stream(dev)
    res = {}
    for batch in (1, 2):
        frames = [[x.to(dev) for x in synthetic.synthetic_frame(1, i, batch, H, W_, 'kitti')[:2]] for i in range(RING)]
        img_d, sp_d = torch.empty_like(frames[0][0]), torch.empty_like(frames[0][1])
        for two in (True, False):
            eng = NlspnEngine(synthetic.make_nlspn_checkpoint(0), batch, H, W_, dev)
            eng.two_streams = two
            eng.set_image_normalization([1.0 / (255.0 * s) for s in synthetic.IMAGENET_STD],
                                        [-mu / s for mu, s in zip(synthetic.IMAGENET_MEAN, synthetic.IMAGENET_STD)])
            with torch.cuda.stream(stream):
                for i in range(args.warmup + 2):
                    img_d.copy_(frames[i % RING][0]); sp_d.copy_(frames[i % RING][1])
                    eng.tta_step(img_d, img_d, sp_d, LR, 1.0, 1.0, 0.1, CAP, graph=True)
                torch.cuda.synchronize(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for i in range(args.steps):
                    img_d.copy_(frames[i % RING][0], non_blocking=True); sp_d.copy_(frames[i % RING][1], non_blocking=True)
                    eng.tta_step(img_d, img_d, sp_d, LR, 1.0, 1.0, 0.1, CAP, graph=True)
                e1.record(stream)
                torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1)
            res['batch%d_%s' % (batch, 'two_streams' if two else 'one_stream')] = {'adapted_frames_per_sec': batch * args.steps / (ms / 1e3),
                                                                                    'ms_per_step': ms / args.steps}
            del eng
            torch.cuda.empty_cache()
    return res


def last_json(text):
    lines = [l for l in text.splitlines() if l.startswith('{')]
    return json.loads(lines[-1]) if lines else None


def launch(world, script_args, port):
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(world), '--master-addr', '127.0.0.1',
           '--master-port', str(port)] + script_args
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=1800)
    if res.returncode != 0:
        raise RuntimeError('%s failed (%d):\n%s\n%s' % (' '.join(cmd), res.returncode, res.stdout[-3000:], res.stderr[-3000:]))
    return last_json(res.stdout)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--worker', action='store_true', help=argparse.SUPPRESS)
    ap.add_argument('--gpus', default='2,8', help='world sizes to measure (those the node has)')
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--out', help='also write the JSON line to this file')
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError('nlspn_shared_bench.py needs CUDA devices (there is no CPU fallback)')
    n_dev = torch.cuda.device_count()
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True)
    out = {'metric': 'adapted_frames_per_sec', 'unit': 'frames/s', 'frame': [3, H, W_], 'gpus_on_node': n_dev,
           'cards': sorted(set(l.strip() for l in q.stdout.splitlines() if l.strip())),
           'config': 'NLSPN ProxyTTA (meta_bn after convert_syncbn), synthetic KITTI-shape frames, lr %g, w_sd/w_smooth/w_cos 1/1/0.1; '
                     'shared: one model over all ranks (SyncBatchNorm + gradient mean all-reduce fused with Adam through peer memory), '
                     'CUDA graph replay; shards: bench.py --workload nlspn (one model per GPU, no collective)' % LR,
           'runs': {}}
    out['w1_stream_layout'] = stream_layout_leg(args)
    port = 29741
    for world in [int(w) for w in args.gpus.split(',')]:
        if world > n_dev:
            out['runs']['w%d' % world] = 'not measured: the node has %d GPUs' % n_dev
            continue
        shared = launch(world, [os.path.abspath(__file__), '--worker', '--steps', str(args.steps), '--warmup', str(args.warmup)], port)
        shards = launch(world, [os.path.join(ROOT, 'bench.py'), '--workload', 'nlspn', '--gpus', str(world), '--steps', str(args.steps),
                                '--warmup', str(args.warmup)], port + 1)
        port += 2
        out['runs']['w%d' % world] = {'shared': shared['shared'],
                                      'shards': {'adapted_frames_per_sec': shards['value'], 'ms_per_step': shards['ms_per_step'],
                                                 'per_gpu_batch': 1, 'clocks': shards.get('clocks')}}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
