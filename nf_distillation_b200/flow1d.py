"""1-D (tabular) FlowStep: host glue for the fused kernels in csrc/flow1d.cu (reference: is_1d branches of
models/flows.py:37-52,142-202 and models/layers.py:76,117,410-411)."""
from __future__ import annotations

import torch

from . import functional as Fn
from . import ops

F32 = torch.float32


def affine_rows(x4, Wf, bf, sl, y, ld_in, ld_out):
    """Stand-alone y = W x + b for [B, D] rows (or [B, C, 1, 1])."""
    B, C, H, W = x4.shape
    if H * W != 1:
        raise NotImplementedError("stand-alone 2-D ActNorm / InvertibleConv1x1 kernels exist for C in {12,24,48,96}")
    ops.affine_rows(x4, Wf, bf, sl, y, ld_in, ld_out, B, C, 1.0)


def _mlp_params(step):
    b = step.block
    ws = [b[i].weight for i in (0, 2, 4, 6, 8, 10)]
    bs = [b[i].bias for i in (0, 2, 4, 6, 8, 10)]
    return ws, bs


def _pack(step, reverse, with_bwd, affine, ws, bs):
    """affine = (Wf, bf, sl) of this direction (functional.affine_item with transpose=1)."""
    D, Cc, hid = step.in_channels, step.condition_features, step.hidden_channels
    Wf, bf, sl = affine
    tf, tb, tg, n_act, offs = ops.flow1d_sizes(D, Cc, hid)
    dev = Wf.device
    PF = torch.empty(tf, device=dev, dtype=F32)
    PB = torch.empty(tb, device=dev, dtype=F32) if with_bwd else None
    ops.flow1d_pack(Wf, bf, ws, bs, D, Cc, hid, PF, PB)
    return Wf, sl, PF, PB, (tg, n_act, offs)


def _consts(step, reverse):
    """No-grad path: packed weights cached until a parameter changes (frozen teacher, sampling)."""
    def build():
        ws, bs = _mlp_params(step)
        inv = tuple(None if t is None else t.detach() for t in step.invconv.lu_tensors())
        affine = Fn.build_affine(step.actnorm.bias.detach(), step.actnorm.logs.detach(), inv, step.in_channels,
                                 reverse, True)
        return _pack(step, reverse, False, affine, [w.detach() for w in ws], [b.detach() for b in bs])
    return Fn.cached(step, ("1d", reverse), build)


class FlowStep1dFn(torch.autograd.Function):
    """Differentiable 1-D FlowStep in either direction (the tabular configs train through the inverse pass:
    perceptual L1 on reverse-pass samples, conf/training/tabular.yaml:11-19). The fused affine comes from the batched
    prep (functional.PrepCtx); its parameter-space backward is deferred to PrepAllFn.backward."""

    @staticmethod
    def forward(ctx, x, ld_in, cond, step, reverse, token, pctx, idx, *mlp):
        ws, bs = list(mlp[:6]), list(mlp[6:])
        D, Cc, hid = step.in_channels, step.condition_features, step.hidden_channels
        B = x.shape[0]
        x = x.contiguous()
        cond = None if cond is None else cond.contiguous()
        Wf, sl, PF, PB, (tg, n_act, offs) = _pack(step, reverse, True, pctx.consts[idx], ws, bs)
        acts = torch.empty(B, n_act, device=x.device, dtype=F32)
        y = torch.empty_like(x)
        ld_out = torch.empty(B, device=x.device, dtype=F32)
        ops.flow1d_fwd(x, cond, PF, sl, y, ld_in.contiguous(), ld_out, acts, B, D, Cc, hid, reverse)
        ctx.meta = (D, Cc, hid, reverse, tg, offs, cond is not None)
        ctx.pctx, ctx.idx = pctx, idx
        ctx.save_for_backward(x, acts, y, PB, *([cond] if cond is not None else []), *ws, *bs)
        return y, ld_out

    @staticmethod
    def backward(ctx, g_y, g_ld):
        D, Cc, hid, reverse, tg, offs, has_cond = ctx.meta
        saved = ctx.saved_tensors
        x, acts, y_out, PB = saved[:4]
        rest = saved[4:]
        cond = rest[0] if has_cond else None
        ws = rest[1:7] if has_cond else rest[0:6]
        B = x.shape[0]
        dev = x.device
        g_y = torch.zeros_like(x) if g_y is None else g_y.contiguous()
        g_ld = torch.zeros(B, device=dev, dtype=F32) if g_ld is None else g_ld.contiguous()
        G = torch.zeros(tg, device=dev, dtype=F32)
        dx = torch.empty_like(x)
        ops.flow1d_bwd(x, cond, acts, PB, y_out, g_y, g_ld, dx, G, B, D, Cc, hid, reverse)
        offG, offGB, ninp, _ = offs[0]
        dWf = G[offG:offG + D * ninp]          # [D, ninp] rows, the first D columns of each are dW'
        dbf = G[offGB:offGB + D]
        ctx.pctx.grads[ctx.idx] = (dWf, ninp, dbf, g_ld, B, 1.0)
        dws, dbs = [], []
        for l in range(1, 7):
            offG, offGB, ninp, _ = offs[l]
            nout, nin = ws[l - 1].shape
            dws.append(G[offG:offG + nout * ninp].view(nout, ninp)[:, :nin])
            dbs.append(G[offGB:offGB + nout])
        return (dx, g_ld, None, None, None, None, None, None, *dws, *dbs)


# ---------------------------------------------------------------------------------------- wide MLPs (inference)
def _wide_consts(step, reverse):
    """Frozen wide step (hidden width a multiple of 64 that does not fit the fused kernel, e.g. conf/teacher/rich.yaml:
    256): fused affine of this direction + the six Linear layers as zero-padded bf16 GEMM operands. Cached."""
    def build():
        D = step.in_channels
        inv = tuple(None if t is None else t.detach() for t in step.invconv.lu_tensors())
        Wf, bf, sl = Fn.build_affine(step.actnorm.bias.detach(), step.actnorm.logs.detach(), inv, D, reverse, True)
        ws, bs = _mlp_params(step)
        Wb, bb = [], []
        for w, b in zip(ws, bs):
            nout, nin = w.shape
            n_p, k_p = ops.round_up(nout, 16), ops.round_up(nin, 64)
            wp = torch.zeros(n_p, k_p, device=w.device, dtype=torch.bfloat16)
            wp[:nout, :nin] = w.detach()
            bp = torch.zeros(n_p, device=w.device, dtype=F32)
            bp[:nout] = b.detach()
            Wb.append(wp)
            bb.append(bp)
        return Wf, bf, sl, Wb, bb
    return Fn.cached(step, ("1dw", reverse), build)


def _flowstep1d_wide(step, x, cond, ld, reverse):
    """Inference of a 1-D FlowStep whose coupling MLP is too wide for shared memory: the affine on the fp32 row kernel,
    the MLP as tcgen05 GEMMs (bf16 operands, fp32 accumulate, bias+ReLU epilogues; 1e-2 tolerance class like the 2-D
    coupling nets), tanh / coupling as elementwise torch ops. Gradients are not built for this path."""
    Wf, bf, sl, Wb, bb = _wide_consts(step, reverse)
    B, D = x.shape
    D1, D2, hid = D // 2, D - D // 2, step.hidden_channels
    dev = x.device
    if not reverse:
        z = torch.empty_like(x)
        ld1 = torch.empty(B, device=dev, dtype=F32)
        ops.affine_rows(x, Wf, bf, sl, z, ld, ld1, B, D, 1.0)
    else:
        z, ld1 = x, ld
    k0 = Wb[0].shape[1]
    a0 = torch.zeros(B, k0, device=dev, dtype=torch.bfloat16)
    a0[:, :D1] = z[:, :D1]
    if cond is not None:
        a0[:, D1:D1 + cond.shape[1]] = cond
    h = a0
    for l in range(4):
        hn = torch.empty(B, hid, device=dev, dtype=torch.bfloat16)
        ops.gemm_nt(h, Wb[l], B, hid, h.shape[1], ops.EPI_BIAS_RELU_BF16, hn, bias=bb[l])
        h = hn
    t = torch.empty(B, hid, device=dev, dtype=F32)
    ops.gemm_nt(h, Wb[4], B, hid, hid, ops.EPI_F32, t, bias=bb[4])
    h = torch.tanh(t).to(torch.bfloat16)
    n6 = Wb[5].shape[0]
    o = torch.empty(B, n6, device=dev, dtype=F32)
    ops.gemm_nt(h, Wb[5], B, n6, hid, ops.EPI_F32, o, bias=bb[5])
    shift, logit = o[:, 0:2 * D2:2], o[:, 1:2 * D2:2] + 2.0
    ls = torch.nn.functional.logsigmoid(logit)
    if not reverse:
        out = torch.cat((z[:, :D1], (z[:, D1:] + shift) * torch.exp(ls)), 1)
        return out, ld1 + ls.sum(1)
    zc = torch.cat((z[:, :D1], z[:, D1:] * torch.exp(-ls) - shift), 1).contiguous()
    ld_mid = (ld1 - ls.sum(1)).contiguous()
    xo = torch.empty_like(zc)
    ld_out = torch.empty(B, device=dev, dtype=F32)
    ops.affine_rows(zc, Wf, bf, sl, xo, ld_mid, ld_out, B, D, 1.0)
    return xo, ld_out


def flowstep1d(step, input, y_onehot, logdet, reverse):
    from .models.layers import _as_logdet
    B = input.shape[0]
    ld = _as_logdet(logdet, B, input.device)
    want_ld = ld is not None
    if ld is None:
        ld = torch.zeros(B, device=input.device)
    cond = y_onehot if step.condition_features else None
    params = step._all_params()
    needs_grad = torch.is_grad_enabled() and (input.requires_grad or ld.requires_grad
                                              or any(p.requires_grad for p in params))
    if needs_grad:
        ws, bs = _mlp_params(step)
        pctx, idx, token = Fn.prep_for(step, bool(reverse))
        z, ld_out = FlowStep1dFn.apply(input, ld, cond, step, bool(reverse), token, pctx, idx, *ws, *bs)
    elif not ops.flow1d_supported(step.in_channels, step.condition_features, step.hidden_channels, False):
        z, ld_out = _flowstep1d_wide(step, input.contiguous(), None if cond is None else cond.contiguous().float(),
                                     ld.contiguous(), bool(reverse))
    else:
        Wf, sl, PF, _, _ = _consts(step, bool(reverse))
        x = input.contiguous()
        z = torch.empty_like(x)
        ld_out = torch.empty(B, device=x.device, dtype=F32)
        ops.flow1d_fwd(x, None if cond is None else cond.contiguous(), PF, sl, z, ld.contiguous(), ld_out, None, B,
                       step.in_channels, step.condition_features, step.hidden_channels, bool(reverse))
    return z, (ld_out if want_ld else None)
