import sys, os, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tta_depth_completion_b200 import _lib
from tta_depth_completion_b200._lib import ptr, c_void_p
L = _lib.lib()
dev = torch.device('cuda:0')
a = torch.zeros(64, device=dev); b = torch.zeros(64, device=dev)
st = torch.cuda.Stream(dev)
with torch.cuda.stream(st):
    s = c_void_p(st.cuda_stream)
    for _ in range(3):
        L.ptta_nl_clamp0(ptr(a), ptr(b), 64, s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        s = c_void_p(torch.cuda.current_stream().cuda_stream)
        for i in range(500):
            L.ptta_nl_clamp0(ptr(a if i % 2 == 0 else b), ptr(b if i % 2 == 0 else a), 64, s)
    g.replay(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st); g.replay(); e1.record(st); torch.cuda.synchronize()
    print('graph of 500 dependent empty-ish kernels: %.2f us per kernel' % (e0.elapsed_time(e1) * 1e3 / 500))
