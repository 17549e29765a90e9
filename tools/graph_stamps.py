#!/usr/bin/env python
"""GPU experiment: in-situ kernel start times of a REPLAYED step graph (profiling build, python -m tta_depth_completion_b200.build stamps).
Run with PTTA_B200_LIB=tta_depth_completion_b200/lib/libptta_b200_stamps.so: python tools/graph_stamps.py [workload] [--one-stream].
--one-stream sets the engine option two_streams = 0, so the replayed graph launches in the order of one eager trace of the same step,
which gives the kernel names."""
import sys, os, ctypes, io, contextlib, subprocess
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
from tta_depth_completion_b200 import ExternalModel_Adapt, _lib
dev = torch.device('cuda:0')
args = [a for a in sys.argv[1:] if a != '--one-stream']
one_stream = '--one-stream' in sys.argv[1:]
wl = args[0] if args else 'kitti'
h, w, dataset, mode, lr, cap = bench.WORKLOADS[wl]
model = ExternalModel_Adapt('msg_chn', 0.0, 100.0, max_input_depth=cap, device=dev)
model._prepare_head(mode)
if one_stream:
    model.model.engine_options = {'two_streams': 0}
model.load_state_dict(bench.make_checkpoint(wl))
model.set_image_normalization((1 / 255.0,) * 3, (0.0,) * 3)
model.train()
frames = [(i.to(dev), s.to(dev)) for i, s in bench.make_frames(wl, 1, 4, 1)]
L = ctypes.CDLL(os.environ['PTTA_B200_LIB'])
st = torch.cuda.Stream(dev)
with torch.cuda.stream(st):
    for i in range(6):
        model.tta_step(frames[i % 4][0], frames[i % 4][1], lr, 1.0, 1.0, 0.1, graph=True)
    torch.cuda.synchronize()
    L.ptta_stamps_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    model.tta_step(frames[2][0], frames[2][1], lr, 1.0, 1.0, 0.1, graph=True)
    e1.record(st)
    torch.cuda.synchronize()
buf = (ctypes.c_ulonglong * 8192)()
n = L.ptta_stamps_read(buf, 8192) - 1000000
ts = sorted(buf[i] for i in range(n))
print('graph replay: %.1f us by events; %d kernel stamps spanning %.1f us' % (e0.elapsed_time(e1) * 1e3, n, (ts[-1] - ts[0]) / 1e3))
# names: eager trace of the same step (stdout of the C side)
eng = model._last_engine
F3 = ctypes.c_float * 3
sys.stdout.flush()
r, wfd = os.pipe(); saved = os.dup(1); os.dup2(wfd, 1)
with torch.cuda.stream(st):
    _lib.check(_lib.lib().ptta_msgchn_trace_step(eng.handle, _lib.ptr(frames[0][0]), F3(1 / 255.0, 1 / 255.0, 1 / 255.0), F3(0, 0, 0),
                                                 _lib.ptr(frames[0][1]), cap, 1.0, 1.0, 0.1, ctypes.c_void_p(st.cuda_stream)), 'trace_step')
os.dup2(saved, 1); os.close(wfd)
names = [l.split()[-1] for l in os.read(r, 1 << 20).decode().splitlines() if l.strip()]
if one_stream and len(names) == n:
    agg = {}
    for i in range(n):
        d = ((ts[i + 1] if i + 1 < n else ts[-1]) - ts[i]) / 1e3
        print('%8.1f  +%6.1f  %s' % ((ts[i] - ts[0]) / 1e3, d, names[i]))
        a = agg.setdefault(names[i], [0, 0.0]); a[0] += 1; a[1] += d
    print('---- start-to-start by kernel')
    for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        print('%-22s %3d launches  %7.1f us  avg %5.1f' % (k, a[0], a[1], a[1] / a[0]))
else:
    print('(%d names vs %d stamps: per-kernel attribution needs --one-stream)' % (len(names), n))
    gaps = [(ts[i + 1] - ts[i]) / 1e3 for i in range(n - 1)]
    print('start-to-start gaps: median %.1f us, max %.1f us' % (sorted(gaps)[len(gaps) // 2], max(gaps)))
