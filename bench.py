#!/usr/bin/env python
"""Benchmark of the ProxyTTA per-frame adaptation step (BASELINE.json: adapted frames/s, fwd+bwd+update, 352x1216).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload kitti|void|nlspn|prepare_init|prepare_head|prepare_head_nlspn] [--batch B]
                    [--dump-outputs DIR]

One "step" = src/tta_main.py:583-633 of the reference for one batch: outlier removal, forward (real + zero-image
branch + proxy heads), the three losses, backward to the adapted meta layer, Adam.  Workload at N=1 = BASELINE.json
configs[1]: MSG-CHN `meta_selfsup_seq_2layers_ema`, batch 1, synthetic KITTI-shape 3x352x1216 frames, ~5 % sparse depth,
continual adaptation over consecutive frames of one synthetic sequence.  With N GPUs every rank adapts its own model on
its own sequence shard (no collective; "scaling": "weak").

Printed JSON (rank 0, one line): the contract keys + `roofline` (dominant kernel, timed alone with CUDA events inside
this script), `cpu_baseline` (the oracle port on the host cores, bounded sample), `e2e` (same metric through the
facade with HOST pinned inputs, H2D inside the timed region, loss read back D2H every step) and `clocks`.

`--impl reference`: the reference's own CPU path -- here the oracle port of it (the reference is PyTorch-eager Python
that cannot travel to the GPU box; oracle/msgchn_oracle.py is pinned against its outputs, tests/golden/) -- timed on
all host cores on the same workload.

`--dump-outputs DIR`: after the timed steps, what the last timed step handed its caller (output depth where the step makes one,
loss values, adapted or trained parameters) is written to DIR/<name>.npy.  Inputs and starting weights are seeded, so two builds
run with the same arguments can be compared file by file."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch

WORKLOADS = {
    # name: (H, W, dataset, prepare_mode, lr, max_input_depth)
    'kitti': (352, 1216, 'kitti', 'meta_selfsup_seq_2layers_ema', 1e-4, 80.0),
    'void': (480, 640, 'void', 'meta_selfsup_seq_1layer_ema', 3e-3, 8.0),
    # BASELINE.json configs[3]: NLSPN back-end (ResNet34 encoder/decoder + 18-step non-local propagation), adapt_mode meta_bn
    'nlspn': (352, 1216, 'kitti', 'meta_selfsup_seq_1layer_ema', 3e-4, 80.0),
    # the NLSPN back-end on synthetic VOID-shape indoor frames (480x640, ~0.5 % density, depth cap 8 m)
    'nlspn_void': (480, 640, 'void', 'meta_selfsup_seq_1layer_ema', 3e-4, 8.0),
}
# SURVEY.md section 8 f3: the source-domain preparation stages on the KITTI-shape workload (src/init_main.py / src/head_main.py steps)
PREPARE = {'prepare_init': 'init', 'prepare_head': 'head', 'prepare_head_nlspn': 'head'}
for _k in PREPARE:
    WORKLOADS[_k] = (352, 1216, 'kitti', 'meta_selfsup_seq_2layers_ema', 1e-3, 80.0)
# stage 2 on the NLSPN back-end (tta_depth_completion_b200/nlspn_prepare.py)
WORKLOADS['prepare_head_nlspn'] = (352, 1216, 'kitti', 'meta_selfsup_seq_1layer_ema', 1e-3, 80.0)
NLSPN_GFLOP_STEP = 3445.9        # SURVEY.md section 8d: forward 2 227.0 + required dgrad 1 201.1 + wgrad 17.8 at 1x352x1216
W_SD, W_SM, W_COS = 1.0, 1.0, 0.1
RING = 8                      # distinct frames cycled through (device-resident for `value`, pinned host for `e2e`)
CONV_GFLOP_R1 = 2 * 9 * 32 * 32 * 352 * 1216 / 1e9      # 32->32 3x3 s1 @352x1216: SURVEY.md section 8(d) / Appendix A


def load_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            p = json.load(f)
        return {'hbm_gbs': p['hbm_gbs'], 'bf16_tflops': p['bf16_tflops'], 'bf16_tflops_sustained': p.get('bf16_tflops_sustained'),
                'source': 'measured (MEASURED_PEAKS.json)'}
    except Exception:
        return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback (B200_PROFILING.md)'}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs"""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace('.', '').isdigit())
        reasons = set()
        for s in self.samples:
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), s[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': float(self.samples[0][1]), 'reasons': sorted(reasons),
                'samples': len(self.samples)}


class HostPrefetcher:
    """Double-buffered input staging for the end-to-end leg: the H2D copy of frame t+1 (pinned host -> device staging buffer, on
    its own copy stream) is issued right after step t is launched, so it overlaps the step; the step's fixed input buffers are then
    filled by a device-to-device copy on the compute stream.  Every frame still crosses PCIe inside the timed region -- this is
    what a prefetching data loader does for the reference's `inputs.to(device)` (src/tta_main.py:521-523)."""

    def __init__(self, pinned, img_d, sp_d, compute_stream, dev):
        self.pinned, self.img_d, self.sp_d, self.compute = pinned, img_d, sp_d, compute_stream
        self.copy = torch.cuda.Stream(dev)
        self.stage = [(torch.empty_like(img_d), torch.empty_like(sp_d)) for _ in range(2)]
        self.ready = [torch.cuda.Event() for _ in range(2)]
        self.consumed = [torch.cuda.Event() for _ in range(2)]
        self.issued = 0

    def prefetch(self, i):
        k = i % 2
        with torch.cuda.stream(self.copy):
            self.copy.wait_event(self.consumed[k])           # the D2D copy that read this staging slot two frames ago is done
            self.stage[k][0].copy_(self.pinned[i % len(self.pinned)][0], non_blocking=True)
            self.stage[k][1].copy_(self.pinned[i % len(self.pinned)][1], non_blocking=True)
            self.ready[k].record(self.copy)

    def take(self, i):
        k = i % 2
        self.compute.wait_event(self.ready[k])
        self.img_d.copy_(self.stage[k][0], non_blocking=True)
        self.sp_d.copy_(self.stage[k][1], non_blocking=True)
        self.consumed[k].record(self.compute)


class LossReader:
    """Reads every step's loss block back to pinned host memory WITHOUT stalling the stream: the D2H copy of step t is enqueued right
    after step t, its event is waited for only after step t+1 has been launched (the reference's progress bar reads the loss
    synchronously every step, src/tta_main.py:801; nothing downstream needs it before the next frame)."""

    def __init__(self, stream):
        self.stream = stream
        self.host = [torch.empty(5, dtype=torch.float32).pin_memory() for _ in range(2)]
        self.ev = [torch.cuda.Event() for _ in range(2)]
        self.pending = None
        self.last = None

    def enqueue(self, dev_losses, i):
        k = i % 2
        self.host[k].copy_(dev_losses, non_blocking=True)
        self.ev[k].record(self.stream)
        prev, self.pending = self.pending, k
        if prev is not None:
            self.collect(prev)

    def collect(self, k):
        self.ev[k].synchronize()
        self.last = self.host[k].tolist()

    def drain(self):
        if self.pending is not None:
            self.collect(self.pending)
            self.pending = None
        return self.last


def make_frames(workload, batch, count, seq_seed):
    from tta_depth_completion_b200 import synthetic          # seeded input generators (SURVEY.md section 8d); no oracle on the product arm
    h, w, dataset = WORKLOADS[workload][:3]
    frames = []
    for t in range(count):
        image, sparse, _ = synthetic.synthetic_frame(seq_seed, t, batch, h, w, dataset)
        frames.append((image.contiguous(), sparse.contiguous()))
    return frames


def make_checkpoint(workload):
    from tta_depth_completion_b200 import synthetic
    return synthetic.make_synthetic_checkpoint(0, WORKLOADS[workload][3])


DUMP_LIMIT_BYTES = 64 << 20
NPY_HEADER_BYTES = 128          # what np.save writes in front of a 1-D or small-rank float array


def dump_outputs(out_dir, arrays):
    """`--dump-outputs`: {name: CPU tensor or Python float} -> out_dir/<name>.npy (tensors as float32, scalars as float64), at most
    DUMP_LIMIT_BYTES of files in all.  Arrays are written smallest first; one that does not fit in what the smaller ones left, split
    evenly over it and the larger ones, is replaced by a fixed sample of its flattened values (indices drawn with seed 0, kept in
    ascending order), so that runs with the same arguments write the same elements."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: (v.float().numpy() if isinstance(v, torch.Tensor) else np.float64(v)) for k, v in arrays.items()}
    left = DUMP_LIMIT_BYTES
    for i, (name, a) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].nbytes)):
        share = left // (len(arrays) - i) - NPY_HEADER_BYTES
        if a.nbytes > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False))]
        path = os.path.join(out_dir, name + '.npy')
        np.save(path, a)
        left -= os.path.getsize(path)


# ------------------------------------------------------------------------------------------------------------
def nlspn_cpu_sample(args, steps, warmup):
    """NLSPN oracle port on the host cores.  A full 352x1216 step needs ~25 GB of fp32 activations and minutes on CPU, so the
    bounded sample is a HALF-resolution frame (176x608, 1/4 of the pixels; every layer's work scales with the pixel count) and
    the throughput is scaled by 1/4."""
    from oracle import msgchn_oracle as O
    from oracle import nlspn_oracle as NO
    h, w, dataset, mode, lr, cap = WORKLOADS[args.workload]
    hs, ws = h // 2, w // 2
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = NO.make_synthetic_checkpoint(0)
    names = NO.adapt_parameter_names(sd, 'meta_bn')
    state = O.AdamState(names, sd)
    frames = [NO.synthetic_frame(1, t, args.batch, hs, ws, dataset)[:2] for t in range(2)]
    for i in range(warmup):
        NO.tta_step(sd, state, *frames[i % 2], lr=lr, w_sd=W_SD, w_sm=W_SM, w_cos=W_COS, max_input_depth=cap)
    t0 = time.perf_counter()
    for i in range(steps):
        NO.tta_step(sd, state, *frames[i % 2], lr=lr, w_sd=W_SD, w_sm=W_SM, w_cos=W_COS, max_input_depth=cap)
    dt = time.perf_counter() - t0
    value = 0.25 * args.batch * steps / dt
    return value, dt, {'value': value, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                       'sample': '%d TTA step(s) of oracle/nlspn_oracle.py (torch %s CPU fp32) on %dx3x%dx%d frames = 1/4 of the pixels of the '
                                 'workload, %.1f s/step, throughput scaled by 1/4' % (steps, torch.__version__, args.batch, hs, ws, dt / steps)}


def prepare_state(workload):
    """(state dict the stage trains from, names of the trained tensors): the seeded synthetic checkpoint; stage 1 starts from a freshly
    drawn meta layer (prepare_parameters), stage 2 from freshly drawn heads -- here the checkpoint's own (equivalent for timing)"""
    sd = make_checkpoint(workload)
    if PREPARE[workload] == 'init':
        names = [k for k in sd if 'meta' in k and k.endswith(('weight', 'bias'))]
    else:
        names = ['pred.0.weight', 'pred.0.bias', 'pred.1.weight', 'pred.1.bias', 'pred.3.weight', 'pred.3.bias']
    return sd, names


def prepare_frames(workload, batch, count, seq_seed):
    from tta_depth_completion_b200 import synthetic
    h, w, dataset = WORKLOADS[workload][:3]
    return [tuple(t.contiguous() for t in synthetic.synthetic_frame(seq_seed, t, batch, h, w, dataset)) for t in range(count)]


def prepare_cpu_steps(args, steps, warmup):
    """oracle port of the stage's step (oracle/msgchn_oracle.py: init_step / head_step) on all host cores; returns seconds per step"""
    from oracle import msgchn_oracle as O
    h, w, dataset, mode, lr, cap = WORKLOADS[args.workload]
    torch.set_num_threads(os.cpu_count() or 1)
    if args.workload == 'prepare_head_nlspn':
        from oracle import nlspn_oracle as NO
        sd = NO.make_synthetic_checkpoint(0)
        state = O.AdamState(list(NO.HEAD_TRAINED), sd)
        frames = prepare_frames(args.workload, args.batch, 2, 1)
        for i in range(warmup):
            NO.head_step(sd, state, NO.normalize_image(frames[i % 2][0]), torch.clamp(frames[i % 2][1], 0, cap), lr=lr)
        t0 = time.perf_counter()
        for i in range(steps):
            NO.head_step(sd, state, NO.normalize_image(frames[i % 2][0]), torch.clamp(frames[i % 2][1], 0, cap), lr=lr)
        return (time.perf_counter() - t0) / steps
    sd, names = prepare_state(args.workload)
    state = O.AdamState(names, sd)
    frames = prepare_frames(args.workload, args.batch, 2, 1)

    def one(i):
        image, sparse, dense = frames[i % 2]
        if PREPARE[args.workload] == 'init':
            O.init_step(sd, state, image, sparse, dense, lr=lr, max_input_depth=cap)
        else:
            O.head_step(sd, state, image, sparse, lr=lr, max_input_depth=cap)
    for i in range(warmup):
        one(i)
    t0 = time.perf_counter()
    for i in range(steps):
        one(i)
    return (time.perf_counter() - t0) / steps


def run_reference(args):
    """CPU arm: the oracle port of the reference step on all host cores."""
    from oracle import msgchn_oracle as O
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    if args.workload in PREPARE:
        steps, warm = args.steps, min(args.warmup, 1)
        dt = prepare_cpu_steps(args, steps, warm)
        value = args.batch / dt
        h, w = WORKLOADS[args.workload][:2]
        cb = {'value': value, 'unit': 'frames/s', 'cores': os.cpu_count() or 1, 'kind': 'port',
              'sample': '%d full-size %s steps (%dx3x%dx%d) of oracle/%s_oracle.py, torch %s CPU fp32, %.2f s/step' % (
                  steps, PREPARE[args.workload], args.batch, h, w, 'nlspn' if args.workload == 'prepare_head_nlspn' else 'msgchn', torch.__version__, dt)}
        print(json.dumps({'impl': 'reference', 'metric': 'trained_frames_per_sec', 'value': value, 'unit': 'frames/s', 'n_gpus': args.gpus,
                          'steps': steps, 'warmup': warm, 'ms_per_step': 1e3 * dt, 'higher_is_better': True, 'scaling': 'weak',
                          'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(args), 'cpu_baseline': cb,
                          'e2e': {'value': value, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}), flush=True)
        return
    if args.workload.startswith('nlspn'):
        steps = args.steps
        value, dt, cb = nlspn_cpu_sample(args, steps, min(args.warmup, 1))
        print(json.dumps({'impl': 'reference', 'metric': 'adapted_frames_per_sec', 'value': value, 'unit': 'frames/s', 'n_gpus': args.gpus,
                          'steps': steps, 'warmup': min(args.warmup, 1), 'ms_per_step': 1e3 * 4.0 * dt / steps, 'higher_is_better': True,
                          'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(args),
                          'cpu_baseline': cb, 'e2e': {'value': value, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}),
              flush=True)
        return
    h, w, dataset, mode, lr, cap = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = make_checkpoint(args.workload)
    names = O.adapt_parameter_names(sd, 'meta')
    state = O.AdamState(names, sd)
    frames = make_frames(args.workload, args.batch, min(RING, args.steps + args.warmup), 1)
    for i in range(args.warmup):
        O.tta_step(sd, state, *frames[i % len(frames)], lr=lr, w_sd=W_SD, w_sm=W_SM, w_cos=W_COS, max_input_depth=cap)
    t0 = time.perf_counter()
    for i in range(args.steps):
        O.tta_step(sd, state, *frames[(args.warmup + i) % len(frames)], lr=lr, w_sd=W_SD, w_sm=W_SM, w_cos=W_COS, max_input_depth=cap)
    dt = time.perf_counter() - t0
    value = args.batch * args.steps / dt
    line = {
        'impl': 'reference', 'metric': 'adapted_frames_per_sec', 'value': value, 'unit': 'frames/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args),
        'cpu_baseline': {'value': value, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                         'sample': '%d full-size TTA steps (%dx%dx%d) of the oracle port, torch %s CPU fp32, after %d warm-up' % (
                             args.steps, args.batch, h, w, torch.__version__, args.warmup)},
        'e2e': {'value': value, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'ranks_note': 'ONE CPU process (rank 0) on all %d host cores whatever --gpus is: the host has one set of cores, so this value does not '
                      'grow with N -- compare it with the N=1 product line only' % cores,
    }
    print(json.dumps(line), flush=True)


def workload_config(args):
    h, w, dataset, mode, lr, cap = WORKLOADS[args.workload]
    if args.workload in PREPARE:
        what = {'init': 'stage-1 meta-layer initialisation (src/init_main.py:482-522: forward init_meta_seq_ema, masked L2 against the ground truth, '
                        'backward to the meta layer, Adam)',
                'head': 'stage-2 predictor-head training (src/head_main.py:437-480: frozen network on the frame and on the zero image, EMA copy of '
                        'proj, cosine loss, backward to pred.*, Adam)'}[PREPARE[args.workload]]
        if args.workload == 'prepare_head_nlspn':
            what = ('stage-2 predictor-head training on the NLSPN back-end (src/head_main.py:437-480 with nlspnmodel_adapt.py:1014-1060: both ResNet34 '
                    'encoders with eval-mode BatchNorm on the frame and on the zero image, EMA copy of proj, cosine loss, backward to proj.* and pred.*, Adam)')
        return {'workload': '%s source-domain preparation, %s, synthetic %s-shape %dx3x%dx%d frames, prepare_mode %s, lr %g, one step per '
                            'batch, %d-frame ring (per-step working set >> L2)' % ('NLSPN' if args.workload == 'prepare_head_nlspn' else 'MSG-CHN', what,
                                                                                  dataset.upper(), args.batch, h, w, mode, lr, RING),
                'batch': args.batch, 'height': h, 'width': w}
    if args.workload.startswith('nlspn'):
        return {'workload': 'NLSPN ProxyTTA continual adaptation (ResNet34 encoder/decoder, 18-step non-local propagation), synthetic ' + dataset.upper() + '-shape '
                            '%dx3x%dx%d frames, prepare_mode %s, adapt_mode meta_bn after convert_syncbn (94 tensors), lr %g, w_sd/w_smooth/w_cos %g/%g/%g, '
                            'Adam(0.9,0.999,1e-8)' % (args.batch, h, w, mode, lr, W_SD, W_SM, W_COS),
                'batch_per_gpu': args.batch, 'parallelism': 'independent sequence shard per GPU (no collective)',
                'l2': 'ring of %d distinct frames; per-step working set (~7 GB of activations) exceeds the 126 MB L2' % RING}
    return {'workload': 'MSG-CHN ProxyTTA continual adaptation, synthetic %s-shape %dx3x%dx%d frames, prepare_mode %s, adapt_mode meta, '
                        'lr %g, w_sd/w_smooth/w_cos %g/%g/%g, Adam(0.9,0.999,1e-8)' % (dataset.upper(), args.batch, h, w, mode, lr, W_SD, W_SM,
                                                                                       W_COS),
            'batch_per_gpu': args.batch,
            'parallelism': {'shards': 'independent sequence shard per GPU (no collective)',
                            'shared': 'shared model (DDP + SyncBatchNorm semantics): BatchNorm sums and the mean all-reduce of the flat adapted-gradient buffer '
                                      'through NVLink peer memory inside the engine kernels, all-reduce fused with Adam, whole step one CUDA graph',
                            'shared_nccl': 'shared model, round-1 form: local BatchNorm statistics, torch.distributed (NCCL) all-reduce of the gradient buffer, '
                                           'separate Adam launch, eager'}[getattr(args, 'mode', 'shards')],
            'l2': 'ring of %d distinct frames; per-step working set (~1.5 GB of activations) exceeds the 126 MB L2' % RING}


def cpu_baseline_sample(args, budget_s=25.0):
    """oracle port on the host cores, bounded sample (1 warm-up + up to 3 timed full-size steps)"""
    from oracle import msgchn_oracle as O
    h, w, dataset, mode, lr, cap = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = make_checkpoint(args.workload)
    names = O.adapt_parameter_names(sd, 'meta')
    state = O.AdamState(names, sd)
    frames = make_frames(args.workload, args.batch, 2, 1)
    O.tta_step(sd, state, *frames[0], lr=lr, w_sd=W_SD, w_sm=W_SM, w_cos=W_COS, max_input_depth=cap)
    n, t0 = 0, time.perf_counter()
    while n < 3 and (n == 0 or time.perf_counter() - t0 < budget_s):
        O.tta_step(sd, state, *frames[n % 2], lr=lr, w_sd=W_SD, w_sm=W_SM, w_cos=W_COS, max_input_depth=cap)
        n += 1
    dt = time.perf_counter() - t0
    return {'value': args.batch * n / dt, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
            'sample': '%d full-size TTA step(s) (%dx3x%dx%d) of oracle/msgchn_oracle.py (torch %s CPU fp32) after 1 warm-up, %.1f s/step' % (
                n, args.batch, h, w, torch.__version__, dt / n)}


def time_dominant_kernel(dev, peaks, iters=40):
    """The 32->32 3x3 stride-1 conv at full resolution (the layer shape that carries most FLOPs and most bytes of the step) on
    the tcgen05 kernel, timed alone with CUDA events on its launch stream.  The 40 launches are replayed from a CUDA graph so that
    the host's per-launch cost (ctypes + torch.empty) is not in the number; inputs rotate over 8 x 27 MB maps (> L2)."""
    from tta_depth_completion_b200 import ops
    h, w = 352, 1216
    g = torch.Generator().manual_seed(0)
    wt = (torch.randn((32, 32, 3, 3), generator=g) * (2.0 / 288) ** 0.5).to(dev)
    wi = ops.pack_conv_weight_tc(ops.pack_conv_weight(wt, 'conv_fwd'))
    bias = torch.zeros(32, device=dev)
    xs = [torch.relu(torch.randn((1, h, w, 32), device=dev)).to(torch.bfloat16) for _ in range(8)]
    stream = torch.cuda.Stream(dev)
    with torch.cuda.stream(stream):
        for i in range(3):
            ops.conv3x3_tc(xs[i % 8], None, bias, wimage=wi)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            for i in range(iters):
                ops.conv3x3_tc(xs[i % 8], None, bias, wimage=wi)
        graph.replay()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        graph.replay()
        e1.record(stream)
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / iters
    tflops = CONV_GFLOP_R1 / ms          # GFLOP / ms == TFLOP/s
    alg_bytes = 2 * h * w * 32 * 2 + 9 * 32 * 32 * 2 + 128
    gbs = alg_bytes / ms / 1e6
    traffic = None
    try:
        with open(os.path.join(ROOT, 'profiles', 'dominant_kernel_traffic.json')) as f:
            traffic = json.load(f).get('dram_bytes_per_launch')
    except Exception:
        pass
    # 144 FLOP per byte is below the ridge (bf16 peak / HBM peak = 253 FLOP/B): the layer is HBM-bound, so that is the
    # roofline it is reported against; the tensor-pipe figures are given next to it (SURVEY.md section 8d caveat)
    return {'kernel': 'conv3x3_tc_kernel: 3x3 32->32 s1 @352x1216 (NHWC bf16, tcgen05 + TMEM, TMA-fed, fp32 accumulate, bias epilogue)',
            'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': gbs / peaks['hbm_gbs'],
            'traffic': traffic, 'us_per_launch': 1e3 * ms, 'algorithmic_bytes_per_launch': alg_bytes,
            'gflop_per_launch': CONV_GFLOP_R1, 'tensor_tflops_achieved': tflops, 'tensor_frac': tflops / peaks['bf16_tflops'],
            'flop_per_byte': CONV_GFLOP_R1 * 1e9 / alg_bytes,
            'peak_source': peaks['source'] + ', burst figures (kernel timed alone, 40 launches replayed from a CUDA graph)'}


def time_convg_kernel(dev, peaks, iters=24):
    """dominant kernel of the NLSPN step: the 64->64 3x3 stride-1 conv of resnet34.layer1 at full resolution (12 forward + 12
    data-gradient launches per step) on the general-channel tcgen05 kernel, timed alone with CUDA events over a ring of 6 inputs
    (6 x 55 MB > L2).  31.6 GFLOP per 110 MB = 288 FLOP/B is above the ridge, so it is reported against the bf16 tensor peak."""
    from tta_depth_completion_b200.convg import ConvG, FWD
    h, w = 352, 1216
    g = torch.Generator().manual_seed(0)
    wt = (torch.randn((64, 64, 3, 3), generator=g) * (2.0 / 576) ** 0.5).to(dev)
    op = ConvG('s1', FWD, wt, 64, 64)
    xs = [torch.randn((1, h, w, 64), device=dev).to(torch.bfloat16) for _ in range(6)]
    outs = [torch.empty((1, h, w, 64), dtype=torch.bfloat16, device=dev) for _ in range(6)]
    stream = torch.cuda.Stream(dev)
    with torch.cuda.stream(stream):
        for i in range(3):
            op(xs[i], out=outs[i])
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):          # replayed from a CUDA graph: no host cost between the launches
            for i in range(iters):
                op(xs[i % 6], out=outs[i % 6])
        graph.replay()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        graph.replay()
        e1.record(stream)
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / iters
    gflop = 2 * 9 * 64 * 64 * h * w / 1e9
    alg_bytes = 2 * h * w * 64 * 2 + 9 * 64 * 64 * 2
    tflops = gflop / ms
    traffic = None
    try:
        with open(os.path.join(ROOT, 'profiles', 'convg_kernel_traffic.json')) as f:
            traffic = json.load(f).get('dram_bytes_per_launch')
    except Exception:
        pass
    return {'kernel': 'convg_kernel: 3x3 64->64 s1 @352x1216 (NHWC bf16, tcgen05 + TMEM, TMA loads and stores, fp32 accumulate)',
            'bound': 'tensor', 'achieved': tflops, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s', 'frac': tflops / peaks['bf16_tflops'],
            'traffic': traffic, 'us_per_launch': 1e3 * ms, 'gflop_per_launch': gflop, 'algorithmic_bytes_per_launch': alg_bytes,
            'hbm_gbs_achieved': alg_bytes / ms / 1e6, 'flop_per_byte': gflop * 1e9 / alg_bytes,
            'peak_source': peaks['source'] + ', burst figure (kernel timed alone, %d launches replayed from a CUDA graph)' % iters}


def run_native_nlspn(args):
    """BASELINE.json configs[3]: NLSPN ProxyTTA at 352x1216, one adapting model per GPU, no collective."""
    from tta_depth_completion_b200 import synthetic as NO
    from tta_depth_completion_b200.nlspn_engine import NlspnEngine
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py needs a CUDA device: the TTA step has no CPU fallback (use --impl reference for the CPU arm)')
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    h, w, dataset, mode, lr, cap = WORKLOADS[args.workload]
    peaks = load_peaks()
    eng = NlspnEngine(NO.make_nlspn_checkpoint(0), args.batch, h, w, dev)
    mean, std = NO.IMAGENET_MEAN, NO.IMAGENET_STD
    eng.set_image_normalization([1.0 / (255.0 * s) for s in std], [-m / s for m, s in zip(mean, std)])
    frames = [NO.synthetic_frame(1 + rank, t, args.batch, h, w, dataset)[:2] for t in range(RING)]
    dev_frames = [(i.to(dev), s.to(dev)) for i, s in frames]
    pinned = [(i.pin_memory(), s.pin_memory()) for i, s in frames]
    img_d, sp_d = torch.empty_like(dev_frames[0][0]), torch.empty_like(dev_frames[0][1])
    stream = torch.cuda.Stream(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def step(graph=None):
        eng.tta_step(img_d, img_d, sp_d, lr, W_SD, W_SM, W_COS, cap, graph=args.graph if graph is None else graph)

    with torch.cuda.stream(stream):
        img_d.copy_(dev_frames[0][0]); sp_d.copy_(dev_frames[0][1])
        step(False)
        l0 = eng.launches
        step(False)
        launches_per_step = eng.launches - l0
        step(); step()                                   # graph mode: first call eager, second captures
        for i in range(args.warmup):
            img_d.copy_(dev_frames[i % RING][0], non_blocking=True); sp_d.copy_(dev_frames[i % RING][1], non_blocking=True)
            step()
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(args.steps):
            img_d.copy_(dev_frames[(args.warmup + i) % RING][0], non_blocking=True); sp_d.copy_(dev_frames[(args.warmup + i) % RING][1], non_blocking=True)
            step()
        e1.record(stream)
        barrier()
        ms_total = e0.elapsed_time(e1)
        sampler.stop_flag = True
        losses = eng.read_losses()
        if args.dump_outputs and rank == 0:             # taken before the e2e leg adapts the model further
            dumped = dict(losses, output_depth=eng.B['output'].cpu(),
                          adapted_parameters=torch.cat([eng.params[k].reshape(-1) for k in eng.adapt_names]).cpu())
        pre = HostPrefetcher(pinned, img_d, sp_d, stream, dev)
        pre.consumed[0].record(stream); pre.consumed[1].record(stream)
        pre.prefetch(0)
        for i in range(3):
            pre.take(i)
            pre.prefetch(i + 1)
            step()
            eng.read_losses()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        reader = LossReader(stream)
        for i in range(3, 3 + args.steps):
            pre.take(i)
            pre.prefetch(i + 1)
            step()
            reader.enqueue(eng.loss_ws[:20].view(torch.float32), i)   # D2H of this step's losses, read one step later
        reader.drain()
        f1.record(stream)
        barrier()
        ms_e2e = f0.elapsed_time(f1)
    if world > 1:
        t = torch.tensor([ms_total, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e = float(t[0]), float(t[1])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    frames_total = world * args.batch * args.steps
    h2d = frames[0][0].numel() * 4 + frames[0][1].numel() * 4
    line = {'metric': 'adapted_frames_per_sec', 'value': frames_total / (ms_total / 1e3), 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_total / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16', 'data': 'synthetic', 'config': workload_config(args),
            'e2e': {'value': frames_total / (ms_e2e / 1e3), 'unit': 'frames/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 20,
                    'ms_per_step': ms_e2e / args.steps,
                    'input_staging': 'pinned host frames, double-buffered: the H2D copy of frame t+1 runs on a copy stream while step t computes; every step\'s loss block is copied D2H to pinned memory and read by the host after the next step has been launched (no per-step stream stall)'},
            'gpu_launches': launches_per_step * args.steps, 'launches_per_step': launches_per_step, 'cuda_graph': bool(args.graph),
            'clocks': sampler.summary(), 'last_losses': losses,
            'step_tflops': NLSPN_GFLOP_STEP * (h * w / (352.0 * 1216.0)) * args.batch / (ms_total / args.steps),
            'step_tflops_note': 'algorithmic work per step (%.1f GFLOP at 352x1216, scaled by the pixel count, x batch: SURVEY.md 8d) / ms_per_step' % NLSPN_GFLOP_STEP}
    if world == 1 and not args.no_extras:
        line['roofline'] = time_convg_kernel(dev, peaks)
        line['cpu_baseline'] = nlspn_cpu_sample(args, 1, 1)[2]
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


E2E_PASSES = 5


def time_dropin_leg(model, pinned, lr, cap, dev, stream, steps, barrier):
    """the reference driver's per-frame lines on the drop-in classes, timed with host frames (see the caller's comment)"""
    from tta_depth_completion_b200 import OutlierRemoval
    params = model.adapt_parameters('meta')
    opt = torch.optim.Adam(params, lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0)
    outlier = OutlierRemoval(7, 1.5)

    def one(i):
        image = pinned[i % len(pinned)][0].to(dev, non_blocking=False)
        sparse = pinned[i % len(pinned)][1].to(dev, non_blocking=False)
        model.train()
        validity = torch.where(sparse > 0, torch.ones_like(sparse), sparse)
        fsd, fvm = outlier.remove_outliers(sparse_depth=sparse, validity_map=validity)
        out, emb, ref = model.forward(image=image / 255.0, sparse_depth=fsd, intrinsics=None, crop_mask=None,
                                      loss_type='adapt_meta_selfsup_seq_ema_reverse')
        loss, info = model.compute_loss(input_rgb=image.detach(), output_depth=out, sparse_depth=fsd.detach(), validity_map=fvm.detach(),
                                        embedding=emb, reference=ref, w_loss_sparse_depth=W_SD, w_loss_smoothness=W_SM, w_loss_cos=W_COS,
                                        loss_type='adapt')
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss.item()

    for i in range(3):
        one(i)
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record(stream)
    for i in range(steps):
        one(3 + i)
    g1.record(stream)
    barrier()
    return g0.elapsed_time(g1)


def gpu_eager_baseline(args, dev, steps=10):
    """Reported baseline, like cpu_baseline: the PyTorch restatement of the reference step (oracle/msgchn_oracle.py, pinned against the
    real reference) run EAGERLY on this GPU through cuDNN / cuBLAS in fp32, with TF32 off and on -- the closest stand-in on the GPU box
    for "the reference's existing GPU path" (the reference itself cannot travel).  It back-propagates only to the adapted tensors
    (225 GFLOP/step instead of the 400 GFLOP the reference's autograd executes), so it flatters the reference."""
    from oracle import msgchn_oracle as O
    h, w, dataset, mode, lr, cap = WORKLOADS[args.workload]
    out = {'unit': 'frames/s', 'kind': 'port on GPU (torch %s eager, cuDNN/cuBLAS fp32)' % torch.__version__, 'steps': steps}
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    try:
        for tf32 in (False, True):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            sd = {k: v.to(dev) for k, v in make_checkpoint(args.workload).items()}
            names = O.adapt_parameter_names(sd, 'meta')
            state = O.AdamState(names, sd)
            frames = [(i.to(dev), s.to(dev)) for i, s in make_frames(args.workload, args.batch, 4, 1)]
            for i in range(3):
                O.tta_step(sd, state, *frames[i % 4], lr=lr, w_sd=W_SD, w_sm=W_SM, w_cos=W_COS, max_input_depth=cap)
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            for i in range(steps):
                O.tta_step(sd, state, *frames[i % 4], lr=lr, w_sd=W_SD, w_sm=W_SM, w_cos=W_COS, max_input_depth=cap)
            torch.cuda.synchronize(dev)
            out['tf32_on' if tf32 else 'tf32_off'] = args.batch * steps / (time.perf_counter() - t0)
            del sd, state, frames
    except Exception as e:          # a baseline leg must never take the bench line down
        out['error'] = '%s: %s' % (type(e).__name__, e)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
        torch.cuda.empty_cache()
    return out


def time_gemm_tn_kernel(dev, peaks, rows, iters=40):
    """the Linear weight gradient dW = dY^T X (rows x 512 x 512) of the stage-2 step on tcgen05 (csrc/gemm_tn_tc.cuh), timed alone"""
    import ctypes
    from tta_depth_completion_b200 import _lib
    L = _lib.lib()
    g = torch.Generator().manual_seed(0)
    As = [torch.randn(rows, 512, generator=g).to(dev, torch.bfloat16) for _ in range(4)]
    Bs = [torch.randn(rows, 512, generator=g).to(dev, torch.bfloat16) for _ in range(4)]
    c = torch.empty(512, 512, device=dev)
    ws = torch.empty(L.ptta_gemm_tn_workspace_bytes(rows, 512, 512), dtype=torch.uint8, device=dev)
    stream = torch.cuda.Stream(dev)
    with torch.cuda.stream(stream):
        st = ctypes.c_void_p(stream.cuda_stream)

        def launch(i):
            _lib.check(L.ptta_gemm_tn_bf16_tc(_lib.ptr(As[i % 4]), _lib.ptr(Bs[i % 4]), _lib.ptr(c), _lib.ptr(ws), rows, 512, 512, st), 'gemm_tn')
        for i in range(3):
            launch(i)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            for i in range(iters):
                launch(i)
        graph.replay()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        graph.replay()
        e1.record(stream)
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / iters
    gflop = 2.0 * rows * 512 * 512 / 1e9
    tflops = gflop / ms
    traffic = None
    try:
        with open(os.path.join(ROOT, 'profiles', 'gemm_tn_kernel_traffic.json')) as f:
            traffic = json.load(f).get('dram_bytes_per_launch')
    except Exception:
        pass
    return {'kernel': 'gemm_tn_tc_kernel + gemm_tn_reduce_kernel: dW[512][512] = dY^T X over %d rows (bf16 operands MN-major, tcgen05 + TMEM, '
                      'TMA-fed, fp32 split-K partial tiles)' % rows,
            'bound': 'tensor', 'achieved': tflops, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s', 'frac': tflops / peaks['bf16_tflops'],
            'traffic': traffic, 'us_per_launch': 1e3 * ms, 'gflop_per_launch': gflop,
            'algorithmic_bytes_per_launch': 2 * rows * 512 * 2 + 512 * 512 * 4,
            'note': 'bounded by the L2 -> SM operand traffic (each operand is read by every tile of the other dimension: 164 MB for 54.8 MB of '
                    'DRAM reads, profiles/r2_gemm_tn_ncu_details.txt), not by the tensor pipe',
            'peak_source': peaks['source'] + ', burst figures (kernel timed alone, 40 launches replayed from a CUDA graph)'}


def run_native_prepare(args):
    """`--workload prepare_init | prepare_head`: the source-domain preparation steps (SURVEY section 8 f3) in the same harness as the TTA
    step -- device-resident graph replays for `value`, pinned host frames + H2D + a blocking loss read every step for `e2e`."""
    from tta_depth_completion_b200 import ExternalModel_Adapt
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py needs a CUDA device: the preparation steps have no CPU fallback (use --impl reference for the CPU arm)')
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    stage = PREPARE[args.workload]
    h, w, dataset, mode, lr, cap = WORKLOADS[args.workload]
    peaks = load_peaks()
    nlspn = args.workload == 'prepare_head_nlspn'
    model = ExternalModel_Adapt('nlspn' if nlspn else 'msg_chn', 0.0, 100.0, max_input_depth=cap, offset=True, device=dev)
    model._prepare_head(mode)
    if nlspn:
        from tta_depth_completion_b200 import synthetic
        model.load_state_dict(synthetic.make_nlspn_checkpoint(0))
    else:
        model.load_state_dict(make_checkpoint(args.workload))
    torch.manual_seed(0)
    if stage == 'head':
        model.prepare_parameters('head_selfsup_ema')            # src/head_main.py:268 (draws fresh heads)
    if nlspn:
        model.convert_syncbn()                                  # :278
        model.set_image_normalization([1.0 / (255.0 * s_) for s_ in synthetic.IMAGENET_STD],
                                      [-m_ / s_ for m_, s_ in zip(synthetic.IMAGENET_MEAN, synthetic.IMAGENET_STD)])
    else:
        model.set_image_normalization((1 / 255.0,) * 3, (0.0,) * 3)
    model.train()
    frames = prepare_frames(args.workload, args.batch, RING, 1 + rank)
    dev_frames = [tuple(t.to(dev) for t in f) for f in frames]
    pinned = [tuple(t.pin_memory() for t in f) for f in frames]
    stream = torch.cuda.Stream(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def run_step(f, graph):
        if stage == 'init':
            model.init_step(f[0], f[1], f[2], lr, graph=graph)
        else:
            model.head_step(f[0], f[1], lr, graph=graph)
    with torch.cuda.stream(stream):
        run_step(dev_frames[0], False)
        eng = model._last_engine
        count = (lambda: eng.launches + eng.eng.launches) if nlspn else eng.launch_count
        l0 = count()
        run_step(dev_frames[0], False)
        launches_per_step = count() - l0
        for i in range(max(3, args.warmup)):
            run_step(dev_frames[i % RING], args.graph)
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(args.steps):
            run_step(dev_frames[(args.warmup + i) % RING], args.graph)
        e1.record(stream)
        barrier()
        ms_total = e0.elapsed_time(e1)
        sampler.stop_flag = True
        losses = model.last_losses()
        if args.dump_outputs and rank == 0:             # taken before the e2e passes train further
            from tta_depth_completion_b200.nlspn_prepare import HEAD_TRAINED
            sd = model.state_dict()
            trained = HEAD_TRAINED if nlspn else model.model._adapt_names
            dumped = dict(losses, trained_parameters=torch.cat([sd[k].reshape(-1) for k in trained]).cpu())
            if stage == 'init':
                dumped['output_depth'] = model.last_output().cpu()
        # end to end: pinned host frames -> H2D -> step -> D2H loss read (synchronising), every step
        passes = []
        for _ in range(E2E_PASSES):
            barrier()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(stream)
            for i in range(args.steps):
                f = tuple(t.to(dev, non_blocking=True) for t in pinned[i % RING])
                run_step(f, args.graph)
                model.last_losses()
            f1.record(stream)
            barrier()
            passes.append(f0.elapsed_time(f1))
        ms_e2e = sorted(passes)[len(passes) // 2]
    if world > 1:
        t = torch.tensor([ms_total, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e = float(t[0]), float(t[1])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    frames_total = world * args.batch * args.steps
    h2d = sum(t.numel() * 4 for t in (frames[0] if stage == 'init' else frames[0][:2]))
    line = {'metric': 'trained_frames_per_sec', 'value': frames_total / (ms_total / 1e3), 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': max(3, args.warmup), 'ms_per_step': ms_total / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16', 'data': 'synthetic', 'config': workload_config(args),
            'e2e': {'value': frames_total / (ms_e2e / 1e3), 'unit': 'frames/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4 if nlspn else 20,
                    'ms_per_step': ms_e2e / args.steps, 'passes_ms': passes,
                    'input_staging': 'pinned host frames copied H2D on the compute stream every step, blocking loss read every step'},
            'gpu_launches': launches_per_step * args.steps, 'launches_per_step': launches_per_step, 'cuda_graph': bool(args.graph),
            'clocks': sampler.summary(), 'last_losses': losses}
    if world == 1 and not args.no_extras:
        if nlspn:
            line['roofline'] = time_convg_kernel(dev, peaks)        # the encoders' 64->64 convolutions: the step's dominant kernel
        else:
            line['roofline'] = time_gemm_tn_kernel(dev, peaks, args.batch * (h // 4) * (w // 4)) if stage == 'head' else time_dominant_kernel(dev, peaks)
        dt = prepare_cpu_steps(args, 2, 1)
        line['cpu_baseline'] = {'value': args.batch / dt, 'unit': 'frames/s', 'cores': os.cpu_count() or 1, 'kind': 'port',
                                'sample': '2 full-size %s steps (%dx3x%dx%d) of oracle/%s_oracle.py (torch %s CPU fp32) after 1 warm-up, %.2f s/step' % (
                                    stage, args.batch, h, w, 'nlspn' if nlspn else 'msgchn', torch.__version__, dt)}
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


def run_native(args):
    if args.workload.startswith('nlspn'):
        return run_native_nlspn(args)
    if args.workload in PREPARE:
        return run_native_prepare(args)
    from tta_depth_completion_b200 import ExternalModel_Adapt
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py needs a CUDA device: the TTA step has no CPU fallback (use --impl reference for the CPU arm)')
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    h, w, dataset, mode, lr, cap = WORKLOADS[args.workload]
    peaks = load_peaks()

    model = ExternalModel_Adapt('msg_chn', 0.0, 100.0, max_input_depth=cap, device=dev)
    model.model.engine_options = dict((k, int(v)) for k, v in (o.split('=') for o in args.engine_opt))      # dispatch experiments
    model._prepare_head(mode)
    model.load_state_dict(make_checkpoint(args.workload))
    model.set_image_normalization((1 / 255.0,) * 3, (0.0,) * 3)
    model.train()
    frames = make_frames(args.workload, args.batch, RING, seq_seed=1 + rank)          # rank r adapts on sequence shard r
    dev_frames = [(i.to(dev), s.to(dev)) for i, s in frames]
    pinned = [(i.pin_memory(), s.pin_memory()) for i, s in frames]
    stream = torch.cuda.Stream(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident throughput (`value`) -------------------------------------------------------------------
    # every step: D2D copy of the next ring frame into the step's fixed input buffers, then the whole step replayed from
    # its CUDA graph (--no-graph: the same kernels launched eagerly)
    use_graph = args.graph and args.mode != 'shared_nccl'
    if args.mode in ('shared', 'shared_nccl'):
        # BASELINE.json configs[4]: one shared model, every rank adapts on its own batch.  'shared': SyncBatchNorm sums and the mean
        # all-reduce of the flat adapted-gradient buffer (74 080 floats) go through NVLink peer memory INSIDE the engine's kernels (the
        # all-reduce fused with Adam), the step replays from one CUDA graph.  'shared_nccl': the round-1 form kept as the baseline --
        # eager launches, local BatchNorm statistics, torch.distributed all_reduce + div + a separate Adam launch.
        from tta_depth_completion_b200 import sharding
        if args.mode == 'shared':
            comm = sharding.enable_shared_model(model)

        def run_step(img, sp, graph=False):
            sharding.shared_model_step(model, img, sp, lr, W_SD, W_SM, W_COS, graph=graph)
    else:
        def run_step(img, sp, graph=False):
            model.tta_step(img, sp, lr, W_SD, W_SM, W_COS, graph=graph)
    img_d = torch.empty_like(dev_frames[0][0])
    sp_d = torch.empty_like(dev_frames[0][1])
    eng = None
    with torch.cuda.stream(stream):
        # launches per step are counted on one eager step (graph replays do not pass through the launch counter)
        img_d.copy_(dev_frames[0][0]); sp_d.copy_(dev_frames[0][1])
        run_step(img_d, sp_d)
        eng = model._last_engine
        l0 = eng.launch_count()
        run_step(img_d, sp_d)
        launches_per_step = eng.launch_count() - l0
        for i in range(args.warmup):
            img, sp = dev_frames[i % RING]
            img_d.copy_(img, non_blocking=True); sp_d.copy_(sp, non_blocking=True)
            run_step(img_d, sp_d, graph=use_graph)
        barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(args.steps):
            img, sp = dev_frames[(args.warmup + i) % RING]
            img_d.copy_(img, non_blocking=True); sp_d.copy_(sp, non_blocking=True)
            for _ in range(args.inner_iter):                # src/tta_main.py:579: `inner_iter` adaptation steps on every batch
                run_step(img_d, sp_d, graph=use_graph)
        e1.record(stream)
        barrier()
        ms_total = e0.elapsed_time(e1)
        sampler.stop_flag = True
        losses = model.last_losses()
        if args.dump_outputs and rank == 0:             # taken before the e2e and drop-in legs adapt the model further
            dumped = dict(losses, output_depth=model.last_output().cpu(),
                          adapted_parameters=torch.cat([p.detach().reshape(-1) for p in model.adapt_parameters('meta')]).cpu())

        # ---- end to end: host pinned inputs -> H2D -> step -> D2H loss read, every step -------------------------------
        # E2E_PASSES passes of `steps` steps each, every pass bracketed like the device-resident region; the MEDIAN pass is reported
        # (a single 20-step pass is a 30 ms region: one host hiccup moved it by 20 % in round 1)
        pre = HostPrefetcher(pinned, img_d, sp_d, stream, dev)
        pre.consumed[0].record(stream); pre.consumed[1].record(stream)
        nwarm = max(3, args.warmup)
        pre.prefetch(0)
        for i in range(nwarm):
            pre.take(i)
            pre.prefetch(i + 1)
            run_step(img_d, sp_d, graph=use_graph)
            model.last_losses()
        e2e_passes, i0 = [], nwarm
        for _ in range(E2E_PASSES):
            barrier()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(stream)
            reader = LossReader(stream)
            for i in range(i0, i0 + args.steps):
                pre.take(i)                                 # frame i: staged by the copy stream while step i-1 was running
                pre.prefetch(i + 1)
                for _ in range(args.inner_iter):
                    run_step(img_d, sp_d, graph=use_graph)
                reader.enqueue(model.last_losses_device(), i)   # D2H of this step's losses; looked at after the next step is launched
            e2e_losses = reader.drain()
            f1.record(stream)
            barrier()
            e2e_passes.append(f0.elapsed_time(f1))
            i0 += args.steps
        ms_e2e = sorted(e2e_passes)[len(e2e_passes) // 2]

        # ---- end to end through the reference driver's OWN calls (src/tta_main.py:583-633): OutlierRemoval.remove_outliers ->
        # model.forward -> model.compute_loss -> loss.backward() -> torch.optim.Adam.step(), host pinned frames, blocking `.to(device)`
        # and a `.item()` read of the loss every step as the reference's progress bar does -- the "no change to the driver" path
        ms_dropin = None
        if args.mode == 'shards' and not args.no_extras and world == 1:
            ms_dropin = time_dropin_leg(model, pinned, lr, cap, dev, stream, args.steps, barrier)

    if world > 1:
        t = torch.tensor([ms_total, ms_e2e, ms_dropin or 0.0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e = float(t[0]), float(t[1])
        ms_dropin = float(t[2]) if ms_dropin else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    frames_total = world * args.batch * args.steps
    h2d = frames[0][0].numel() * 4 + frames[0][1].numel() * 4
    line = {
        'metric': 'adapted_frames_per_sec', 'value': frames_total / (ms_total / 1e3), 'unit': 'frames/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_total / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic', 'config': workload_config(args),
        'e2e': {'value': frames_total / (ms_e2e / 1e3), 'unit': 'frames/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 20,
                'ms_per_step': ms_e2e / args.steps, 'passes_ms': e2e_passes, 'passes': 'median of %d passes of %d steps' % (E2E_PASSES, args.steps),
                'input_staging': 'pinned host frames, double-buffered: the H2D copy of frame t+1 runs on a copy stream while step t computes; every step\'s loss block is copied D2H to pinned memory and read by the host after the next step has been launched (no per-step stream stall)'},
        'gpu_launches': (launches_per_step or 0) * args.steps,
        'launches_per_step': launches_per_step, 'cuda_graph': use_graph,
        'clocks': sampler.summary(),
        'last_losses': losses,
    }
    if args.engine_opt:
        line['engine_options'] = args.engine_opt
    if args.inner_iter != 1:
        line['config']['inner_iter'] = args.inner_iter
        line['config']['workload'] += ', inner_iter %d (TTA steps per frame, src/tta_main.py:579)' % args.inner_iter
        line['gpu_launches'] *= args.inner_iter
    gflop_step = {'kitti': 210.5, 'void': 152.8}[args.workload] * args.batch
    line['step_tflops'] = gflop_step / (ms_total / args.steps)
    line['step_tflops_note'] = 'work performed per step (%.1f GFLOP: fwd + required dgrad/wgrad, rgb_encoder(0) cached, SURVEY.md 8d) / ms_per_step' % gflop_step
    if ms_dropin:
        line['e2e_dropin'] = {'value': frames_total / (ms_dropin / 1e3), 'unit': 'frames/s', 'ms_per_step': ms_dropin / args.steps,
                              'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4,
                              'path': 'the reference driver\'s own lines (src/tta_main.py:583-633) on the drop-in classes: OutlierRemoval.remove_outliers, '
                                      'ExternalModel_Adapt.forward, .compute_loss, loss.backward(), torch.optim.Adam.step(); blocking .to(device) of pinned '
                                      'host frames and loss.item() every step; kernels launched eagerly (no CUDA graph)'}
    if world == 1 and not args.no_extras:
        line['roofline'] = time_dominant_kernel(dev, peaks)
        line['gpu_eager_baseline'] = gpu_eager_baseline(args, dev)
        line['cpu_baseline'] = cpu_baseline_sample(args)
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='native', choices=['native', 'reference'])
    ap.add_argument('--workload', default='kitti', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=1)
    ap.add_argument('--mode', default='shards', choices=['shards', 'shared', 'shared_nccl'], help='shards: independent sequence shard per GPU, no collective (default); shared: one shared model, NCCL all-reduce of the adapted-parameter gradients (BASELINE.json configs[4])')
    ap.add_argument('--no-graph', dest='graph', action='store_false', help='launch the step kernels eagerly instead of replaying the captured CUDA graph')
    ap.add_argument('--inner-iter', type=int, default=1, help='adaptation steps per frame (src/tta_main.py:579; the indoor script bash/adapt/adapt_msgchn_scenenet.sh runs 3); a bench "step" is then one FRAME = inner_iter TTA steps')
    ap.add_argument('--no-extras', action='store_true', help='skip the roofline / cpu_baseline legs (profiling runs)')
    ap.add_argument('--engine-opt', action='append', default=[], metavar='NAME=VALUE', help='ptta_msgchn_set_option on the engine (dispatch experiments, e.g. tc_min_pixels=1000); not for headline runs')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step computed to DIR/<name>.npy (float32 / float64, at most 64 MB in all)')
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.steps is None:
        if args.impl == 'reference':          # a CPU step of these workloads takes seconds to minutes
            args.steps = 5 if args.workload in PREPARE else 3 if args.workload.startswith('nlspn') else 10
        else:
            args.steps = 200
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs records the native path (--impl native)')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_native(args)


if __name__ == '__main__':
    main()
