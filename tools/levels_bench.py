"""Warm, graph-replayed timings of the three inference kernels of a FlowStep (affine1x1_fwd, fused conv kernel, fused
Conv2dZeros + coupling) at every level of the CIFAR model, rotating over enough buffers to exceed the L2:
    python tools/levels_bench.py [B]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from nf_distillation_b200 import ops
dev = "cuda"
B = int(sys.argv[1]) if len(sys.argv) > 1 else 2048
hid = 512
bf16 = torch.bfloat16


def time_graph(fn, reps, nbuf):
    for i in range(nbuf): fn(i)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(reps): fn(i % nbuf)
    g.replay(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


tot = 0.0
for (C, H) in ((12, 16), (24, 8), (48, 4)):
    W = H
    M = B * H * W
    K1p, K3p = ops.round_up(9 * C // 2, 64), ops.round_up(9 * C, 64)
    nb = max(3, int(200e6 // (M * hid * 2)) + 1)
    nb = min(nb, 8)
    xs = [torch.randn(B, C, H, W, device=dev) for _ in range(nb)]
    ys = [torch.empty(B, C, H, W, device=dev) for _ in range(nb)]
    cols = [torch.empty(M, K1p, device=dev, dtype=bf16) for _ in range(nb)]
    h2 = [(torch.randn(M, hid, device=dev).clamp_min(0) * 0.5).to(bf16) for _ in range(nb)]
    Wf, bfv, sl = torch.randn(C, C, device=dev) * 0.3, torch.randn(C, device=dev) * 0.1, torch.zeros(1, device=dev)
    ld, ld1 = torch.zeros(B, device=dev), torch.zeros(B, device=dev)
    W1 = (torch.randn(hid, K1p, device=dev) * 0.1).to(bf16)
    W2 = (torch.randn(hid, hid, device=dev) * 0.05).to(bf16)
    B3 = (torch.randn(K3p, hid, device=dev) * 0.02).to(bf16)
    b1, b2, b3 = torch.zeros(hid, device=dev), torch.zeros(hid, device=dev), torch.zeros(C, device=dev)
    ta = time_graph(lambda i: ops.affine1x1_fwd(xs[i], Wf, bfv, sl, ys[i], cols[i], K1p, ld, ld1, B, C, H, W), 16, nb)
    if ops.cnet_fused_supported(hid, K1p, M):
        tc = time_graph(lambda i: ops.cnet_fwd_fused(cols[i], K1p, W1, W2, b1, b2, h2[i], M, hid), 16, nb)
    else:
        tc = float("nan")
    tp = time_graph(lambda i: ops.pconv_coupling_fwd(h2[i], B3, K3p, b3, ys[i], None, ld, B, C, H, W, hid, False), 16, nb)
    hb_a, hb_p = M * (8.0 * C + 2.0 * K1p), M * (2.0 * hid + 4.0 * C)
    fl = 2.0 * M * hid * (9 * C // 2 + hid)
    print(f"C={C:2d} {H}x{W} M={M}: affine1x1_fwd {ta:6.1f} us ({hb_a/ta/1e3:5.0f} GB/s) | fused conv {tc:6.1f} us "
          f"({fl/tc/1e6:5.0f} TFLOP/s) | pconv_coupling {tp:6.1f} us ({hb_p/tp/1e3:5.0f} GB/s) | sum {ta+tc+tp:6.1f}")
    tot += ta + tc + tp
print(f"sum over levels {tot:.1f} us per FlowStep triple; x32 teacher steps = {tot*32/1e3:.2f} ms")
