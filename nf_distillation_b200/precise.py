"""fp32-class ("bf16x3") execution of the 2-D FlowStep: the reference's convolutions are fp32
(/root/reference/models/layers.py:209,249, models/flows.py:25-34); this mode runs them on the same tcgen05 GEMM tiles
with every operand split into two bf16 parts (h + m) laid side by side along K, so that ONE pass of the unchanged
tensor-core GEMM accumulates the three significant partial products hh + hm + mh in fp32 (csrc/split3.cu): 2^-16 per
product instead of bf16's 2^-8. Measured against fp64 (tools/x3_check.py): 5e-6 of max|out| per GEMM, against 3e-7
for an fp32 SIMT matmul and 2e-3 for plain bf16 operands.

That 5e-6 is the floor of this hardware path, not of the split: the six-term form (h + m + l, hh+hm+hl+mh+mm+lh,
layouts 2 / 3 of split3.cu) measures the same 2e-6..5e-6, because the tensor core's fp32 accumulator does not carry
terms 2^-16 below the running sum. Consequence for GRADIENTS: of the ~5 M ReLU units of a FlowStep at M = 10 240 pixels
about 20 have a pre-activation within 5e-6 of zero and get the other mask than in the fp32 reference; each such unit
moves the weight-gradient entries of its row / the bias gradient of its channel by O(1/sqrt(M)) ~ 1e-2 of their size
(the log-scale gradients, which weight every unit by its pre-activation, stay at 5e-6). So outputs, log-dets and loss
terms are at fp32 level (2e-6), gradients at 1e-3 in relative L2 / <= 1e-2 in max-norm on conv#1 / conv#2 weights and
biases and 1e-5 elsewhere — 5-10x below the bf16 mode, and the same effect any two fp32 implementations show once
their summation orders differ by more than the distance of a pre-activation to zero.

It is selected per model (`model.set_precision("bf16x3")`), costs ~3x the tensor-core work plus unfused fp32
intermediates, and exists so that parity with the reference can be shown at fp32 level (KD taps 1e-4, gradients 1e-3)
and benchmarked beside the bf16 mode.

Both directions train: FlowStep2dX3Fn (forward pass) and FlowStep2dReverseX3Fn (inverse pass, through which the
perceptual term's gradient reaches the student) share one split backward of the coupling net (_coupling_net_backward),
fed by an fp32 dh (coupling_bwd_f32 / coupling_inv_bwd_f32 of csrc/split3.cu). Additive steps run the affine arithmetic
with the pinned logit rows of FlowStep._coupling_params_2d (s == 1.0f), as in the bf16 mode.

Parameter-space work (folding the ActNorm scales into the conv weights, the LU product of the invertible 1x1 conv) is
plain differentiable tensor arithmetic on [C, C] / [hid, K] tensors here; everything per pixel runs in libnfk kernels.
The inverse pass takes its inverse-direction affine from the batched prep kernel (functional.PrepCtx), whose backward
applies the inverse's chain rule, so no matrix inverse enters the autograd graph.
"""
from __future__ import annotations

import torch

from . import ops
from ._lib import LIB, check

BF16, F32 = torch.bfloat16, torch.float32
A3, B3, A6, B6 = 0, 1, 2, 3          # operand layouts of csrc/split3.cu
TERMS = {A3: 3, B3: 3, A6: 6, B6: 6}
# column block (in units of K) holding the h / m part of each A layout, for the two-part wgrads
H_OFF = {A3: 0, A6: 0}
M_OFF = {A3: 2, A6: 3}


def _st():
    return torch.cuda.current_stream().cuda_stream


def split_rows(src, K, pattern):
    """fp32 [rows, Ksrc <= K] -> bf16 [rows, terms*K] in the given operand layout (zero padded to K columns)."""
    src = src.contiguous()
    rows, Ksrc = src.shape
    out = torch.empty(rows, TERMS[pattern] * K, device=src.device, dtype=BF16)
    ops._count()
    check(LIB.nfk_split3_rows(src.data_ptr(), src.stride(0), rows, K, Ksrc, pattern, out.data_ptr(), _st()),
          "nfk_split3_rows")
    return out


def im2col_split(src, layout, Ctot, c0, Cc, B, H, W, flip, Kp, pattern=A3):
    out = torch.empty(B * H * W, TERMS[pattern] * Kp, device=src.device, dtype=BF16)
    ops._count()
    check(LIB.nfk_im2col3x3_split3(src.data_ptr(), layout, Ctot, c0, Cc, B, H, W, int(flip), Kp, pattern,
                                   out.data_ptr(), _st()), "nfk_im2col3x3_split3")
    return out


def act_split(pre, mode, gate=None, colsum=None, pattern=A3):
    M, N = pre.shape
    out = torch.empty(M, TERMS[pattern] * N, device=pre.device, dtype=BF16)
    ops._count()
    check(LIB.nfk_act_split3(pre.data_ptr(), M, N, mode, None if gate is None else gate.data_ptr(),
                             0 if gate is None else gate.stride(0), pattern, out.data_ptr(),
                             None if colsum is None else colsum.data_ptr(), _st()), "nfk_act_split3")
    return out


def gemm_split(As, Bs, M, N, bias=None):
    """fp32 [M, N] = As @ Bs^T over the K-concatenated split operands (+ bias)."""
    assert As.shape[1] == Bs.shape[1]
    out = torch.empty(M, N, device=As.device, dtype=F32)
    ops.gemm_nt(As, Bs, M, N, As.shape[1], ops.EPI_F32, out, bias=bias)
    return out


def wgrad_split(As, Ka, pa, Bs, Kb, pb, Kpix):
    """fp32 [Ka, Kb] = sum over pixels of A^T B, A = h + m and B = h + m taken from split operands in layout pa / pb:
    three split-K tensor-core GEMMs accumulating into one output (hh + hm + mh)."""
    out = torch.zeros(Ka, Kb, device=As.device, dtype=F32)
    ah, am, bh, bm = H_OFF[pa] * Ka, M_OFF[pa] * Ka, H_OFF[pb] * Kb, M_OFF[pb] * Kb
    for ao, bo in ((ah, bh), (ah, bm), (am, bh)):
        ops._count()
        check(LIB.nfk_gemm_tn_bf16(As.data_ptr() + 2 * ao, As.stride(0), Bs.data_ptr() + 2 * bo, Bs.stride(0), Ka, Kb,
                                   Kpix, out.data_ptr(), out.stride(0), ops.sm_count(), _st()), "nfk_gemm_tn_bf16")
    return out


def _padded(t, rows, cols):
    if t.shape == (rows, cols):
        return t.contiguous()
    out = torch.zeros(rows, cols, device=t.device, dtype=F32)
    out[:t.shape[0], :t.shape[1]] = t
    return out


# ------------------------------------------------------------------------------------------------ parameter space
def folded_params(step):
    """(Wf, bf, sl, W1f, b1f, W2f, b2f, W3f, b3f) of a FlowStep as DIFFERENTIABLE fp32 tensors:
    fused ActNorm o invconv (layers.py:101-142,376-397) and the conv weights with the ActNorm / exp(3 logs) scales
    folded in (layers.py:223-228,257-260), laid out for the im2col GEMMs (k = tap*Cin + ci, rows of W3f = tap*Cout + co)."""
    C = step.in_channels
    iv = step.invconv
    lower, upper, log_s, p, sign_s, weight = iv.lu_tensors()
    dev = step.actnorm.bias.device
    if weight is None:
        eye = torch.eye(C, device=dev)
        Lm = torch.tril(lower, -1) + eye
        Um = torch.triu(upper, 1) + torch.diag(sign_s * torch.exp(log_s))
        Wm = p @ (Lm @ Um)
        ld_w = log_s.sum()
    else:
        Wm, ld_w = weight, torch.slogdet(weight)[1]
    e = torch.exp(step.actnorm.logs.view(-1))
    Wf = Wm * e.view(1, -1)
    bf = Wf @ step.actnorm.bias.view(-1)
    sl = (step.actnorm.logs.sum() + ld_w).view(1)
    return (Wf, bf, sl, *folded_coupling(step))


def folded_coupling(step):
    """(W1f, b1f, W2f, b2f, W3f, b3f) of folded_params(): the coupling-net part alone (the inverse pass takes its
    affine from the prep kernel)."""
    C, hid = step.in_channels, step.hidden_channels
    cin = C // 2
    w1, b1, l1, w2, b2, l2, w3, b3, l3 = step._coupling_params_2d()
    e1, e2, e3 = torch.exp(l1.view(-1)), torch.exp(l2.view(-1)), torch.exp(3.0 * l3.view(-1))
    W1f = (w1 * e1.view(-1, 1, 1, 1)).permute(0, 2, 3, 1).reshape(hid, 9 * cin)
    W2f = w2.view(hid, hid) * e2.view(-1, 1)
    W3f = (w3 * e3.view(-1, 1, 1, 1)).permute(2, 3, 0, 1).reshape(9 * C, hid)
    return W1f, b1.view(-1) * e1, W2f, b2.view(-1) * e2, W3f, b3.view(-1) * e3


def _coupling_net(y, B, C, H, W, hid, K1p, K3p, W1f, b1f, W2f, b2f, W3f):
    """conv3x3 -> ReLU -> conv1x1 -> ReLU -> per-tap products P of the last conv, three-term split products."""
    M, cin = B * H * W, C // 2
    col = im2col_split(y, 0, C, 0, cin, B, H, W, False, K1p, A3)
    h1 = act_split(gemm_split(col, split_rows(W1f, K1p, B3), M, hid, bias=b1f), 0, pattern=A3)
    pre2 = gemm_split(h1, split_rows(W2f, hid, B3), M, hid, bias=b2f)
    h2 = act_split(pre2, 0, pattern=A3)
    P = gemm_split(h2, split_rows(_padded(W3f, K3p, hid), hid, B3), M, K3p)
    return col, h1, h2, P


def _coupling_net_backward(dh, col, h1, h2, B, C, H, W, hid, K1p, K3p, W1f, W2f, W3f):
    """Backward of _coupling_net in either direction, from the fp32 pixel-major dh [M, C] (shift / logit interleaved) to
    the first conv's per-tap input gradient dcol [M, K1p] fp32 (column = tap*(C/2) + ci), with the weight and bias
    gradients: (dcol, dW1, dbias1, dW2, dbias2, dW3)."""
    M, cin = B * H * W, C // 2
    dev = dh.device
    dhcol = im2col_split(dh, 1, C, 0, C, B, H, W, True, K3p, A3)                        # [M, 3 K3p]
    # conv#3 dgrad (NT GEMM against W3f^T [hid, K3p]), ReLU mask of h2, bias gradient as fp32 column sums
    dbias2 = torch.zeros(hid, device=dev, dtype=F32)
    dpre2 = act_split(gemm_split(dhcol, split_rows(_padded(W3f.t(), hid, K3p), K3p, B3), M, hid), 1, gate=h2,
                      colsum=dbias2)
    dW3 = wgrad_split(dhcol, K3p, A3, h2, hid, A3, M)[:9 * C]
    dbias1 = torch.zeros(hid, device=dev, dtype=F32)
    dpre1 = act_split(gemm_split(dpre2, split_rows(W2f.t().contiguous(), hid, B3), M, hid), 1, gate=h1,
                      colsum=dbias1)
    dW2 = wgrad_split(dpre2, hid, A3, h1, hid, A3, M)
    dcol = gemm_split(dpre1, split_rows(_padded(W1f.t(), K1p, hid), hid, B3), M, K1p)
    dW1 = wgrad_split(dpre1, hid, A3, col, K1p, A3, M)[:, :9 * cin]
    return dcol, dW1.contiguous(), dbias1, dW2, dbias2, dW3.contiguous()


class FlowStep2dX3Fn(torch.autograd.Function):
    """FlowStep.normal_flow (models/flows.py:142-171) with fp32-class coupling-net arithmetic; inputs are x, logdet and
    the folded parameter tensors of folded_params() (autograd carries their gradients back to the reference
    parameters)."""

    @staticmethod
    def forward(ctx, x, ld_in, hid, Wf, bf, sl, W1f, b1f, W2f, b2f, W3f, b3f):
        B, C, H, W = x.shape
        M, cin = B * H * W, C // 2
        K1p, K3p = ops.round_up(9 * cin, 64), ops.round_up(9 * C, 64)
        dev = x.device
        x = x.contiguous()
        Wf, bf, sl = Wf.contiguous(), bf.contiguous(), sl.contiguous()
        y = torch.empty_like(x)
        ld_out = torch.empty(B, device=dev, dtype=F32)
        ops.affine1x1_fwd(x, Wf, bf, sl, y, None, 0, ld_in.contiguous(), ld_out, B, C, H, W)
        col, h1, h2, P = _coupling_net(y, B, C, H, W, hid, K1p, K3p, W1f, b1f.contiguous(), W2f, b2f.contiguous(), W3f)
        hsave = torch.empty(M, C, device=dev, dtype=F32)
        ops.coupling_fwd(P, K3p, b3f.contiguous(), y, hsave, ld_out, B, C, H, W, reverse=False)
        ctx.hid = hid
        ctx.save_for_backward(x, y, col, h1, h2, hsave, Wf, W1f, W2f, W3f)
        return y, ld_out

    @staticmethod
    def backward(ctx, g_out, g_ld):
        x, z_out, col, h1, h2, hsave, Wf, W1f, W2f, W3f = ctx.saved_tensors
        hid = ctx.hid
        B, C, H, W = x.shape
        M, cin = B * H * W, C // 2
        K1p, K3p = ops.round_up(9 * cin, 64), ops.round_up(9 * C, 64)
        dev = x.device
        g_out = torch.zeros_like(x) if g_out is None else g_out.contiguous()
        g_ld = torch.zeros(B, device=dev, dtype=F32) if g_ld is None else g_ld.contiguous()
        dy = torch.empty_like(x)
        dh = torch.empty(M, C, device=dev, dtype=F32)
        dbias3 = torch.zeros(C, device=dev, dtype=F32)
        ops._count()
        check(LIB.nfk_coupling_bwd_f32(g_out.data_ptr(), g_ld.data_ptr(), z_out.data_ptr(), hsave.data_ptr(),
                                       dy.data_ptr(), dh.data_ptr(), dbias3.data_ptr(), B, C, H, W, _st()),
              "nfk_coupling_bwd_f32")
        dcol, dW1, dbias1, dW2, dbias2, dW3 = _coupling_net_backward(dh, col, h1, h2, B, C, H, W, hid, K1p, K3p, W1f,
                                                                     W2f, W3f)
        dx = torch.empty_like(x)
        dWf = torch.zeros(C, C, device=dev, dtype=F32)
        dbf = torch.zeros(C, device=dev, dtype=F32)
        ops.affine1x1_bwd(dy, dcol, K1p, x, Wf, dx, dWf, dbf, B, C, H, W)
        dsl = (g_ld.sum() * float(H * W)).view(1)
        return dx, g_ld, None, dWf, dbf, dsl, dW1, dbias1, dW2, dbias2, dW3, dbias3


def flowstep2d_reverse_x3(z, ld_in, hid, inv_affine, W1f, b1f, W2f, b2f, W3f, b3f, keep=False):
    """FlowStep.reverse_flow (models/flows.py:173-202): coupling^-1 with the precise coupling net, then the inverse
    fused affine (inv_affine = (Wf, bf, sl) of the inverse direction, from the prep kernel). keep=True (training) also
    returns what FlowStep2dReverseX3Fn's backward reads: (zc = the post-coupling tensor, col, h1, h2, hsave); the
    outputs are the same bits."""
    B, C, H, W = z.shape
    cin = C // 2
    K1p, K3p = ops.round_up(9 * cin, 64), ops.round_up(9 * C, 64)
    col, h1, h2, P = _coupling_net(z, B, C, H, W, hid, K1p, K3p, W1f, b1f.contiguous(), W2f, b2f.contiguous(), W3f)
    zc, ld_mid = z.clone(), ld_in.clone()
    hsave = torch.empty(B * H * W, C, device=z.device, dtype=F32) if keep else None
    ops.coupling_fwd(P, K3p, b3f.contiguous(), zc, hsave, ld_mid, B, C, H, W, reverse=True)
    Wf, bf, sl = inv_affine
    x = torch.empty_like(z)
    ld_out = torch.empty_like(ld_mid)
    ops.affine1x1_fwd(zc, Wf, bf, sl, x, None, 0, ld_mid, ld_out, B, C, H, W)
    if keep:
        return x, ld_out, (zc, col, h1, h2, hsave)
    return x, ld_out


class FlowStep2dReverseX3Fn(torch.autograd.Function):
    """FlowStep.reverse_flow under autograd with fp32-class coupling-net arithmetic, the counterpart of
    functional.FlowStep2dReverseFn (the perceptual term's gradient reaches the student through its inverse pass,
    pl_module.py:229-243). The inverse-direction affine comes from the batched prep (token, pctx, idx as in the bf16 Fn:
    this step's backward deposits (dWf, dbf, g_ld) and PrepAllFn.backward applies the inverse chain rule); the
    coupling-net weights are the folded_params() tensors, so autograd carries their gradients to the reference
    parameters. Backward: dzc = Wf^T g_x (affine1x1_bwd without col2im, also dWf, dbf), dz2 = dzc2 / s and the fp32 dh
    (coupling_inv_bwd_f32), the coupling net's split backward to dcol, dz1 = dzc1 + col2im(dcol)."""

    @staticmethod
    def forward(ctx, z, ld_in, hid, token, pctx, idx, W1f, b1f, W2f, b2f, W3f, b3f):
        z = z.contiguous()
        Wf = pctx.consts[idx][0]
        x, ld_out, (zc, col, h1, h2, hsave) = flowstep2d_reverse_x3(z, ld_in.contiguous(), hid, pctx.consts[idx], W1f,
                                                                    b1f, W2f, b2f, W3f, b3f, keep=True)
        ctx.hid = hid
        ctx.pctx, ctx.idx = pctx, idx
        ctx.save_for_backward(zc, col, h1, h2, hsave, Wf, W1f, W2f, W3f)
        return x, ld_out

    @staticmethod
    def backward(ctx, g_x, g_ld):
        zc, col, h1, h2, hsave, Wf, W1f, W2f, W3f = ctx.saved_tensors
        hid = ctx.hid
        B, C, H, W = zc.shape
        M, cin = B * H * W, C // 2
        K1p, K3p = ops.round_up(9 * cin, 64), ops.round_up(9 * C, 64)
        dev = zc.device
        g_x = torch.zeros_like(zc) if g_x is None else g_x.contiguous()
        g_ld = torch.zeros(B, device=dev, dtype=F32) if g_ld is None else g_ld.contiguous()
        dzc = torch.empty_like(zc)
        dWf = torch.zeros(C, C, device=dev, dtype=F32)
        dbf = torch.zeros(C, device=dev, dtype=F32)
        ops.affine1x1_bwd(g_x, None, K1p, zc, Wf, dzc, dWf, dbf, B, C, H, W)
        dz = torch.empty_like(zc)
        dh = torch.empty(M, C, device=dev, dtype=F32)
        dbias3 = torch.zeros(C, device=dev, dtype=F32)
        ops._count()
        check(LIB.nfk_coupling_inv_bwd_f32(dzc.data_ptr(), g_ld.data_ptr(), zc.data_ptr(), hsave.data_ptr(),
                                           dz.data_ptr(), dh.data_ptr(), dbias3.data_ptr(), B, C, H, W, _st()),
              "nfk_coupling_inv_bwd_f32")
        dcol, dW1, dbias1, dW2, dbias2, dW3 = _coupling_net_backward(dh, col, h1, h2, B, C, H, W, hid, K1p, K3p, W1f,
                                                                     W2f, W3f)
        ops.col2im_add(dcol, K1p, dz, B, C, H, W)
        ctx.pctx.grads[ctx.idx] = (dWf, C, dbf, g_ld, B, float(H * W))
        return dz, g_ld, None, None, None, None, dW1, dbias1, dW2, dbias2, dW3, dbias3
