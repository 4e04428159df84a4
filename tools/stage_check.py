"""Stage-by-stage check of one 2-D FlowStep's forward and backward kernel sequence (functional.FlowStep2dFn): every
kernel's output is compared with plain torch fp32 arithmetic applied to THAT kernel's own inputs (the CUDA path's
intermediates), so a deviation is attributed to one kernel instead of to "bf16 rounding somewhere"."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
import torch.nn.functional as F
import test_headline_parity_gpu as T
from nf_distillation_b200 import functional as Fn, ops
dev = "cuda"
BF = torch.bfloat16


RESULTS = []


def stats(name, got, ref, bf16=False):
    """fp32 outputs: max|d| / max|ref|. bf16 outputs: additionally the fraction of elements that differ at all (a
    1-ulp rounding flip where the fp32 pre-rounding values differ in summation order)."""
    got, ref = got.float(), ref.float()
    d = (got - ref).abs()
    scale = ref.abs().max().item() + 1e-30
    err = d.max().item() / scale
    nz = (d > 0).float().mean().item() if bf16 else None
    RESULTS.append((name, err, nz))
    print(f"  {name:12s} max|d|/max|ref| {err:.2e}" + (f"  mismatching elements {nz:.2e}" if bf16 else ""))


def run(C, H, B, hid=512):
    """Returns [(stage, max|d|/max|ref|, mismatch fraction or None)] for one FlowStep at (C, H, B)."""
    del RESULTS[:]
    st, sd = T.make_step(C, hid, 100 + C)
    st = st.to(dev)
    W = H
    M, cin = B * H * W, C // 2
    K1p, K3p = ops.round_up(9 * cin, 64), ops.round_up(9 * C, 64)
    g = torch.Generator().manual_seed(C)
    x = torch.randn(B, C, H, H, generator=g).to(dev); ld0 = torch.randn(B, generator=g).to(dev)
    g_out = torch.randn(B, C, H, H, generator=g).to(dev); g_ld = torch.randn(B, generator=g).to(dev)
    print(f"=== C={C} H={H} B={B} M={M} K1p={K1p} K3p={K3p}")
    pctx = Fn.PrepCtx([st], False)
    with torch.no_grad():
        pctx.build()
    Wf, bf, sl = pctx.consts[0]
    k = Fn.StepConsts(Wf, bf, sl, *pctx.cops[0])
    with torch.no_grad():
        y, ld_out, (col, h1, h2, hsave, m1, m2) = Fn.flowstep2d_forward(x, ld0, k, hid, keep=True)
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        # ---- forward stages
        y_aff = torch.einsum("oi,bihw->bohw", Wf, x) + bf.view(1, -1, 1, 1)
        stats("y1 (affine)", y[:, :cin], y_aff[:, :cin])
        colr = F.unfold(y[:, :cin], 3, padding=1)                  # [B, cin*9, HW] index ci*9 + tap
        colr = colr.view(B, cin, 9, H * W).permute(0, 3, 2, 1).reshape(M, 9 * cin)   # k = tap*cin + ci
        stats("col", col[:, :9 * cin], colr.to(BF), bf16=True)
        h1r = torch.relu(col.float() @ k.B1.float().T + k.bias1).to(BF)
        stats("h1", h1, h1r, bf16=True)
        h2r = torch.relu(h1.float() @ k.B2.float().T + k.bias2).to(BF)
        stats("h2", h2, h2r, bf16=True)
        w3 = k.B3[:9 * C].float().view(3, 3, C, hid).permute(2, 3, 0, 1).contiguous()       # [co, k, ky, kx]
        hmap = h2.float().view(B, H, W, hid).permute(0, 3, 1, 2)
        conv3 = F.conv2d(hmap, w3, k.bias3, padding=1)
        stats("hsave", hsave.view(B, H, W, C).permute(0, 3, 1, 2), conv3)
        shift, logit = conv3[:, 0::2], conv3[:, 1::2]
        s = torch.sigmoid(logit + 2)
        z2 = (y_aff[:, cin:] + shift) * s
        stats("z2", y[:, cin:], z2)
        stats("logdet", ld_out, ld0 + sl * H * W + torch.log(s).flatten(1).sum(1))
        # ---- backward stages (the sequence of FlowStep2dFn.backward)
        dbias3 = torch.zeros(C, device=dev)
        dy = torch.empty_like(x)
        dhcol = torch.empty(M, K3p, device=dev, dtype=BF)
        ops.coupling_bwd(g_out, g_ld, y, hsave, dy, dhcol, K3p, dbias3, B, C, H, W)
        hs = hsave.view(B, H, W, C).permute(0, 3, 1, 2)
        sg = torch.sigmoid(hs[:, 1::2] + 2)
        dsh = g_out[:, cin:] * sg
        dlg = (g_out[:, cin:] * y[:, cin:] + g_ld.view(-1, 1, 1, 1)) * (1 - sg)
        dh = torch.stack((dsh, dlg), 2).flatten(1, 2)               # [B, C, H, W] interleaved shift / logit
        stats("dy2", dy[:, cin:], dsh); stats("dy1", dy[:, :cin], g_out[:, :cin])
        stats("dbias3", dbias3, dh.sum((0, 2, 3)))
        # dhcol[m, tap*C + co] = dh[co] at pixel (y - dy, x - dx), tap = (dy+1)*3 + (dx+1): transposed-conv im2col
        dhp = F.pad(dh, (1, 1, 1, 1))
        cols = []
        for tap in range(9):
            oy, ox = tap // 3 - 1, tap % 3 - 1
            cols.append(dhp[:, :, 1 - oy:1 - oy + H, 1 - ox:1 - ox + W])
        dhcol_r = torch.stack(cols, 1).permute(0, 3, 4, 1, 2).reshape(M, 9 * C)
        stats("dhcol", dhcol[:, :9 * C], dhcol_r.to(BF), bf16=True)
        dpre2 = torch.empty(M, hid, device=dev, dtype=BF); dbias2 = torch.zeros(hid, device=dev)
        dpre1 = torch.empty(M, hid, device=dev, dtype=BF); dbias1 = torch.zeros(hid, device=dev)
        fused_bwd = ops.cnet_fused_supported(hid, K3p) and M >= 8192
        if fused_bwd:     # the path FlowStep2dFn.backward takes at this size: both dgrads in one kernel
            ops.cnet_bwd_fused(dhcol, K3p, k.B3T, k.B2T, m2, m1, dpre2, dpre1, dbias2, dbias1, M, hid)
        else:
            ops.gemm_nt(dhcol, k.B3T, M, hid, K3p, ops.EPI_MASK_BF16, dpre2, aux=m2, colsum=dbias2)
        dpre2_r = ((dhcol.float() @ k.B3T.float().T) * (h2 > 0)).to(BF)
        stats("dpre2", dpre2, dpre2_r, bf16=True)
        stats("dbias2", dbias2, dpre2.float().sum(0))
        stats("B3T==B3^T", k.B3T, k.B3.T)
        dB3 = torch.zeros(K3p, hid, device=dev); ops.gemm_tn(dhcol, h2, K3p, hid, M, dB3)
        stats("dB3", dB3, dhcol.float().T @ h2.float())
        if not fused_bwd:
            ops.gemm_nt(dpre2, k.B2T, M, hid, hid, ops.EPI_MASK_BF16, dpre1, aux=m1, colsum=dbias1)
        dpre1_r = ((dpre2.float() @ k.B2T.float().T) * (h1 > 0)).to(BF)
        stats("dpre1", dpre1, dpre1_r, bf16=True)
        stats("dbias1", dbias1, dpre1.float().sum(0))
        dB2 = torch.zeros(hid, hid, device=dev); ops.gemm_tn(dpre2, h1, hid, hid, M, dB2)
        stats("dB2", dB2, dpre2.float().T @ h1.float())
        dcol = torch.empty(M, K1p, device=dev); ops.gemm_nt(dpre1, k.B1T, M, K1p, hid, ops.EPI_F32, dcol)
        stats("dcol", dcol, dpre1.float() @ k.B1T.float().T)
        dB1 = torch.zeros(hid, K1p, device=dev); ops.gemm_tn(dpre1, col, hid, K1p, M, dB1)
        stats("dB1", dB1, dpre1.float().T @ col.float())
        dx = torch.empty_like(x); dWf = torch.zeros(C, C, device=dev); dbf = torch.zeros(C, device=dev)
        ops.affine1x1_bwd(dy, dcol, K1p, x, Wf, dx, dWf, dbf, B, C, H, W)
        # col2im of dcol -> gradient of y1, added to dy1
        dc = dcol[:, :9 * cin].view(B, H * W, 9, cin).permute(0, 3, 2, 1).reshape(B, cin * 9, H * W)
        dy1c = F.fold(dc, (H, W), 3, padding=1)
        dyt = torch.cat((dy[:, :cin] + dy1c, dy[:, cin:]), 1)
        stats("dx", dx, torch.einsum("oi,bohw->bihw", Wf, dyt))
        stats("dWf", dWf, torch.einsum("bohw,bihw->oi", dyt, x))
        stats("dbf", dbf, dyt.sum((0, 2, 3)))
    return list(RESULTS)


if __name__ == "__main__":
    for C, H, B in ((12, 16, 40), (24, 8, 136), (48, 4, 520)):
        run(C, H, B)
