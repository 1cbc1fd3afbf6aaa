"""Correlation at the bench shape: accuracy vs the oracle on a small case, timing of the active path (FN2_CORR_NOTC=1 ->
FP32 fast path) with algorithmic GB/s and TFLOP/s."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from flownet2_b200 import ops
from oracle import oracle as O
r = np.random.default_rng(0)
cl = torch.channels_last
for (N, C, H, W, s2, md) in [(2, 64, 40, 56, 2, 20), (1, 32, 21, 37, 2, 20), (1, 32, 24, 30, 1, 10)]:
    a = r.standard_normal((N, C, H, W)).astype(np.float32); b = r.standard_normal((N, C, H, W)).astype(np.float32)
    ta = torch.from_numpy(a).cuda().contiguous(memory_format=cl); tb = torch.from_numpy(b).cuda().contiguous(memory_format=cl)
    got = ops.correlation(ta, tb, md, 1, md, 1, s2).contiguous().cpu().numpy()
    want = O.correlation_fwd(a, b, md, 1, md, 1, s2, 0, False)
    print((N, C, H, W, s2, md), "max err %.3e (scale %.2f)" % (float(np.abs(got - want).max()), float(np.abs(want).max())), flush=True)
for (N, H, W) in [(4, 56, 128), (8, 40, 56)]:
    a = torch.randn(N, 256, H, W, device="cuda").contiguous(memory_format=cl)
    b = torch.randn(N, 256, H, W, device="cuda").contiguous(memory_format=cl)
    out = torch.empty(N, 441, H, W, device="cuda").contiguous(memory_format=cl)
    for _ in range(3):
        ops.correlation(a, b, 20, 1, 20, 1, 2, out=out)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        ops.correlation(a, b, 20, 1, 20, 1, 2, out=out)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    by = 4.0 * N * H * W * (2 * 256 + 441); fl = 2.0 * 441 * 256 * N * H * W
    print("NOTC=%s (%d,256,%d,%d): %.3f ms  %.0f GB/s algorithmic  %.1f TFLOP/s" % (os.environ.get("FN2_CORR_NOTC", "0"), N, H, W, ms, by / ms / 1e6, fl / ms / 1e9), flush=True)
