"""csrc/dgrad_col2im.cu: the coupling net's first-conv input gradient fused with its col2im and affine1x1_bwd.

The fused kernel computes the same tcgen05 products as the gemm_nt (EPI_F32) dgrad it replaces, sums the nine taps in
col2im_gather's order and runs affine1x1_bwd's fmaf chain, so dx must be bit-identical to that pair of kernels. dW' and
db' are fp32 sums whose order differs (per-CTA partials meeting in global atomics): 1e-6 of their max.
"""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
dev = "cuda"


def rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-12)).item()


def test_supported_shapes():
    from nf_distillation_b200 import ops
    for C, H in ((12, 16), (12, 8), (24, 8), (24, 4), (48, 8), (48, 4), (48, 2)):
        assert ops.conv1_dgrad_affine_bwd_supported(C, H, H, 512), (C, H)
    assert ops.conv1_dgrad_affine_bwd_supported(12, 16, 16, 256)
    for C, H, W, hid in ((12, 32, 32, 512),    # CelebA level 0: an image is larger than a tile
                         (24, 16, 16, 512), (48, 16, 16, 512), (96, 4, 4, 512), (12, 16, 16, 96), (12, 12, 12, 512)):
        assert not ops.conv1_dgrad_affine_bwd_supported(C, H, W, hid), (C, H, W, hid)


@pytest.mark.gpu
@pytest.mark.parametrize("C,H,B,hid", [
    (12, 16, 2048, 512), (12, 16, 64, 512), (12, 16, 37, 512),
    (24, 8, 2048, 512), (24, 8, 64, 512), (24, 8, 37, 512),
    (48, 4, 2048, 512), (48, 4, 64, 512), (48, 4, 37, 512),
    (12, 8, 9, 256),      # four images per tile, ragged last tile
    (48, 2, 7, 64),       # 2x2 maps, one k-block
    (48, 8, 5, 256),      # one 8x8 image per tile
])
def test_fused_matches_gemm_plus_affine1x1_bwd(C, H, B, hid):
    from nf_distillation_b200 import ops
    W, CH = H, C // 2
    M, K1p = B * H * W, ops.round_up(9 * CH, 64)
    g = torch.Generator(device=dev).manual_seed(1000 + 7 * B + C + hid)
    dpre1 = (torch.randn(M, hid, device=dev, generator=g) * (torch.rand(M, hid, device=dev, generator=g) > 0.5)
             ).bfloat16()
    B1T = torch.zeros(K1p, hid, device=dev, dtype=torch.bfloat16)
    B1T[:9 * CH] = (torch.randn(9 * CH, hid, device=dev, generator=g) * 0.03).bfloat16()   # row = tap*CH + ci
    dy = torch.randn(B, C, H, W, device=dev, generator=g)
    x = torch.randn(B, C, H, W, device=dev, generator=g)
    Wf = torch.randn(C, C, device=dev, generator=g) * 0.3
    assert ops.conv1_dgrad_affine_bwd_supported(C, H, W, hid)

    dcol = torch.empty(M, K1p, device=dev)
    ops.gemm_nt(dpre1, B1T, M, K1p, hid, ops.EPI_F32, dcol)
    dx_u, dW_u, db_u = torch.empty_like(x), torch.zeros(C, C, device=dev), torch.zeros(C, device=dev)
    ops.affine1x1_bwd(dy, dcol, K1p, x, Wf, dx_u, dW_u, db_u, B, C, H, W)
    dx_f, dW_f, db_f = torch.full_like(x, float("nan")), torch.zeros(C, C, device=dev), torch.zeros(C, device=dev)
    ops.conv1_dgrad_affine_bwd(dpre1, B1T, K1p, dy, x, Wf, dx_f, dW_f, db_f, B, C, H, W, hid)
    torch.cuda.synchronize()
    assert torch.equal(dx_f, dx_u), rel(dx_f, dx_u)
    assert rel(dW_f, dW_u) < 1e-6 and rel(db_f, db_u) < 1e-6, (rel(dW_f, dW_u), rel(db_f, db_u))

    # and against torch: conv_transpose of the bf16 operands in fp32, then the affine backward
    import torch.nn.functional as F
    w1 = B1T[:9 * CH].float().view(3, 3, CH, hid).permute(3, 2, 0, 1)          # conv#1 weight [hid, CH, ky, kx]
    dmap = dpre1.float().view(B, H, W, hid).permute(0, 3, 1, 2)
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        dy1 = F.conv_transpose2d(dmap, w1, padding=1)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    dys = dy.clone()
    dys[:, :CH] += dy1
    dx_t = torch.einsum("oc,bohw->bchw", Wf, dys)
    dW_t = torch.einsum("bohw,bchw->oc", dys, x)
    assert rel(dx_f, dx_t) < 1e-4 and rel(dW_f, dW_t) < 1e-4 and rel(db_f, dys.sum((0, 2, 3))) < 1e-4


def _flowstep_grads(C, H, B, monkeypatch, fused):
    """One student FlowStep forward + backward; returns the input gradient, the parameter gradients and which of the
    two conv#1-dgrad paths its backward ran."""
    from nf_distillation_b200 import functional, ops
    from nf_distillation_b200.models.flows import FlowStep
    calls = {"fused": 0, "affine1x1_bwd": 0}

    def spy(name, fn):
        def wrapped(*a, **k):
            calls[name] += 1
            return fn(*a, **k)
        return wrapped

    monkeypatch.setattr(functional, "USE_FUSED_DGRAD1", fused)
    monkeypatch.setattr(ops, "conv1_dgrad_affine_bwd", spy("fused", ops.conv1_dgrad_affine_bwd))
    monkeypatch.setattr(ops, "affine1x1_bwd", spy("affine1x1_bwd", ops.affine1x1_bwd))
    torch.manual_seed(5)
    st = FlowStep(in_channels=C, hidden_channels=512, actnorm_scale=1.0, flow_permutation="invconv",
                  flow_coupling="affine", LU_decomposed=True)
    for m in st.modules():
        if hasattr(m, "inited"):
            m.inited = True
    g = torch.Generator().manual_seed(6)
    with torch.no_grad():
        for p in st.parameters():
            if p.abs().max() == 0:
                p.copy_(torch.randn(p.shape, generator=g) * 0.05)
    st = st.to(dev)
    x = torch.randn(B, C, H, H, generator=g).to(dev).requires_grad_(True)
    ld0 = torch.zeros(B, device=dev)
    wy = torch.randn(B, C, H, H, generator=g).to(dev)
    y, ld = st(x, logdet=ld0)
    ((y * wy).sum() + ld.sum()).backward()
    torch.cuda.synchronize()
    return x.grad, {n: p.grad.clone() for n, p in st.named_parameters()}, calls


@pytest.mark.gpu
@pytest.mark.parametrize("C,H,B", [(12, 16, 40), (24, 8, 9), (48, 4, 130)])
def test_flowstep_backward_dispatch_and_parity(C, H, B, monkeypatch):
    """FlowStep2dFn.backward runs the fused kernel where it is supported; NFK_FUSED_DGRAD1=0 keeps gemm_nt +
    affine1x1_bwd. Input gradients are bit-identical, parameter gradients agree to fp32 summation order."""
    dx_f, g_f, calls_f = _flowstep_grads(C, H, B, monkeypatch, True)
    assert calls_f == {"fused": 1, "affine1x1_bwd": 0}, calls_f
    dx_u, g_u, calls_u = _flowstep_grads(C, H, B, monkeypatch, False)
    assert calls_u == {"fused": 0, "affine1x1_bwd": 1}, calls_u
    assert torch.equal(dx_f, dx_u), rel(dx_f, dx_u)
    for n in g_u:
        assert rel(g_f[n], g_u[n]) < 1e-5, (n, rel(g_f[n], g_u[n]))


@pytest.mark.gpu
def test_unsupported_shape_keeps_the_two_kernel_path(monkeypatch):
    """32x32 maps (CelebA level 0) are larger than a tile: the backward keeps gemm_nt + affine1x1_bwd."""
    _, _, calls = _flowstep_grads(12, 32, 3, monkeypatch, True)
    assert calls == {"fused": 0, "affine1x1_bwd": 1}, calls
