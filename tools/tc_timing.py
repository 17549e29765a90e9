#!/usr/bin/env python
"""GPU experiment: tcgen05 conv vs mma.sync conv, timed from a CUDA graph of 40 back-to-back launches (no host launch cost)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from tta_depth_completion_b200 import ops, _lib
dev = 'cuda'
g = torch.Generator().manual_seed(0)
wt = (torch.randn((32, 32, 3, 3), generator=g) * (2.0 / 288) ** 0.5).to(dev)
wp = ops.pack_conv_weight(wt, 'conv_fwd'); wi = ops.pack_conv_weight_tc(wp); bias = torch.zeros(32, device=dev)


def timeit(fn, xs, iters=40, graph=True):
    for i in range(3):
        fn(xs[i % len(xs)])
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        if graph:
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr, stream=s):
                for i in range(iters):
                    fn(xs[i % len(xs)])
            run = gr.replay
        else:
            def run():
                for i in range(iters):
                    fn(xs[i % len(xs)])
        run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        run()
        e1.record(s)
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3


import subprocess
print(subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True).stdout.strip(),
      '| library', _lib.LIB_PATH, flush=True)


def rotation(shape, bytes_each):
    """enough distinct buffers that one pass over them exceeds the 126 MB L2 (>= 300 MB), as the step streams its maps"""
    cnt = max(2, min(64, int(300e6 / bytes_each)))
    return [torch.randn(shape, device=dev).to(torch.bfloat16) for _ in range(cnt)]


# operands rotate with the input: mask / add / add2 / up2 are a different buffer for every launch of the graph
for shape in [(1, 352, 1216), (4, 352, 1216), (1, 176, 608), (1, 88, 304)]:
    n, h, w = shape
    xs = rotation((n, h, w, 32), n * h * w * 64)
    ms = rotation((n, h, w, 32), n * h * w * 64)
    hs = rotation((n, h // 2, w // 2, 32), n * h * w * 16)
    k = len(xs)
    ops_ = list(range(k))
    res = []
    res.append('tc %.1f' % timeit(lambda x: ops.conv3x3_tc(x, wp, bias, wimage=wi), xs))
    res.append('warm %.1f' % timeit(lambda x: ops.conv3x3_tc(x, wp, bias, wimage=wi), xs[:1]))
    res.append('out2 %.1f' % timeit(lambda i: ops.conv3x3_tc_ex(xs[i], wp, bias, wimage=wi), ops_))
    res.append('add2+out2 %.1f' % timeit(lambda i: ops.conv3x3_tc_ex(xs[i], wp, bias, add2=ms[(i + 1) % k], wimage=wi), ops_))
    res.append('mask %.1f' % timeit(lambda i: ops.conv3x3_tc(xs[i], wp, bias, mask=ms[i], wimage=wi), ops_))
    res.append('mask+add %.1f' % timeit(lambda i: ops.conv3x3_tc(xs[i], wp, bias, mask=ms[i], add=ms[(i + 1) % k], wimage=wi), ops_))
    res.append('up2+out2 %.1f' % timeit(lambda i: ops.conv3x3_tc_up2(xs[i], wp, hs[i % len(hs)], bias), ops_))
    res.append('mma %.1f' % timeit(lambda x: ops.conv3x3(x, wp, bias, ops.MODE_S1, ops.PRO_RELU), xs))
    gb = 2 * n * h * w * 64 / 1e3
    print(shape, ' | '.join(res), '| tc %.0f GB/s' % (gb / float(res[0].split()[1])), flush=True)
    del xs, ms, hs

# transposed stride-2 (input sizes; output, mask and add are 2x): the backward's data gradients run it with mask + add
wtT = (torch.randn((32, 32, 3, 3), generator=g) * (2.0 / 288) ** 0.5).to(dev)
wpT = ops.pack_conv_weight(wtT, 'convT_fwd')
for shape in [(1, 176, 608), (1, 88, 304), (1, 44, 152)]:
    n, h, w = shape
    xs = rotation((n, h, w, 32), 5 * n * h * w * 64)
    ms = rotation((n, 2 * h, 2 * w, 32), 5 * n * h * w * 64)
    k = len(xs)
    ops_ = list(range(k))
    res = ['t2 tc %.1f' % timeit(lambda x: ops.conv3x3_tc_t2(x, wpT, bias), xs),
           't2 tc mask+add %.1f' % timeit(lambda i: ops.conv3x3_tc_t2(xs[i], wpT, None, mask=ms[i], add=ms[(i + 1) % k]), ops_),
           't2 mma %.1f' % timeit(lambda x: ops.conv3x3(x, wpT, bias, ops.MODE_T2, ops.PRO_RELU), xs)]
    print(shape, ' | '.join(res), flush=True)
    del xs, ms
