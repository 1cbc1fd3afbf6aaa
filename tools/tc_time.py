import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C, torch
from flownet2_b200 import ops, lib, check, fn2_conv_desc
cl = torch.channels_last
l = lib()
for (N, Ci, H, W, Co, k, s, p) in [(4, 473, 56, 128, 256, 3, 1, 1), (4, 12, 448, 1024, 64, 7, 2, 3), (4, 82, 448, 1024, 16, 3, 1, 1), (4, 64, 448, 1024, 64, 3, 2, 1), (4, 162, 224, 512, 32, 3, 1, 1)]:
    Cp = (Ci + 31) // 32 * 32 if Ci >= 32 else (Ci + 3) // 4 * 4
    x = torch.randn(N, Cp, H, W, device="cuda").contiguous(memory_format=cl)[:, :Ci]
    w = torch.randn(Co, Ci, k, k, device="cuda") * 0.02
    b = torch.zeros(Co, device="cuda")
    d = fn2_conv_desc(Ci, Co, k, k, s, s, p, p, 0, 1, 1, 0.1, 2)
    nf = C.c_size_t(); check(l.fn2_conv_packed_floats(C.byref(d), Ci, C.byref(nf)))
    packed = torch.empty(nf.value, device="cuda")
    check(l.fn2_conv_pack_weights(C.byref(d), Ci, C.c_void_p(w.data_ptr()), C.c_void_p(packed.data_ptr()), None))
    Ho = (H + 2 * p - k) // s + 1; Wo = (W + 2 * p - k) // s + 1
    out = torch.empty(N, Co, Ho, Wo, device="cuda").contiguous(memory_format=cl)
    dx, do = ops.desc(x), ops.desc(out)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    wb = C.c_size_t(); check(l.fn2_conv_workspace_bytes(C.byref(d), N, H, W, C.byref(wb)))
    wsbuf = torch.empty(max(wb.value, 4) // 4, device="cuda") if os.environ.get("TC_TIME_WS", "1") == "1" else None
    wsp, wsn = (C.c_void_p(wsbuf.data_ptr()), wb.value) if wsbuf is not None else (None, 0)
    for _ in range(3):
        check(l.fn2_conv_forward(C.byref(d), C.byref(dx), C.c_void_p(packed.data_ptr()), C.c_void_p(b.data_ptr()), C.byref(do), wsp, wsn, st))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        check(l.fn2_conv_forward(C.byref(d), C.byref(dx), C.c_void_p(packed.data_ptr()), C.c_void_p(b.data_ptr()), C.byref(do), wsp, wsn, st))
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    steps = k * k * ((Ci + 31) // 32)
    tiles = N * ((Ho * Wo + 127) // 128) * max(1, Co // (128 if Co % 128 == 0 else 64 if Co % 64 == 0 else 32 if Co % 32 == 0 else 16))
    rounds = (tiles + 147) // 148
    print("%s: %.3f ms, %d tiles (%d rounds) x %d steps -> %.0f cycles/step @1.9GHz" % ((N, Ci, H, W, Co, k, s), ms, tiles, rounds, steps, ms * 1e-3 * 1.9e9 / rounds / steps), flush=True)
