"""Autograd glue between the drop-in nn.Modules (models/) and the libnfk kernels (ops.py).

Each torch.autograd.Function runs one reference layer (FlowStep, Split2d, prior->bpd, per-level KD MSE) as a short,
fixed sequence of kernel launches; saved tensors are exactly what the matching backward sequence reads.
"""
from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Optional

import torch

from . import ops

BF16 = torch.bfloat16
F32 = torch.float32
USE_FUSED_PCONV = os.environ.get("NFK_FUSED_PCONV", "1") != "0"
USE_FUSED_DGRAD1 = os.environ.get("NFK_FUSED_DGRAD1", "1") != "0"

# ---- weight gradients beside the backward chain (small batches) --------------------------------------------------
# A student FlowStep's backward is a chain of dependent launches: coupling_bwd -> both dgrads -> (3 weight-gradient
# GEMMs) -> conv#1 dgrad -> affine1x1_bwd. The weight gradients feed nothing in that chain (only the batched parameter
# chain rule at the very end of the pass), and at the reference's batch size every launch is one tile's latency, so
# they are issued on a second stream: fork after the dgrads, join at the start of the next step's backward (and in
# PrepAllFn.backward before their results are read). The buffers that stream reads are kept alive until the join.
# Large maps saturate the GPU anyway and keep the single stream (and do not hold a step's activations any longer).
WGRAD_STREAM_MAX_M = int(os.environ.get("NFK_WGRAD_STREAM_MAX_M", "65536"))   # 0 disables
_wgrad_streams: dict = {}
_wgrad_keepalive: list = []


def _wgrad_stream(dev):
    key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
    st = _wgrad_streams.get(key)
    if st is None:
        st = _wgrad_streams[key] = torch.cuda.Stream(device=dev)
    return st


def _join_wgrads(dev):
    """Make the current stream wait for the weight-gradient stream; then the buffers it was reading may be freed."""
    if _wgrad_keepalive:
        torch.cuda.current_stream(dev).wait_stream(_wgrad_stream(dev))
        _wgrad_keepalive.clear()

# ------------------------------------------------------------------------------------------------ parameter epoch
# The no-grad paths cache operands derived from the parameters (fused affine, folded bf16 conv weights, packed MLP /
# MADE weights) keyed on (data_ptr, _version) of the parameters. An optimiser step replayed from a CUDA graph (or a
# write through `.data`) changes the values without touching either, so every such key also carries this counter:
# whoever updates parameters behind autograd's back (train.KDTrainer after each replayed clip+Adam graph) calls
# `bump_param_epoch()`, which invalidates every cached operand of trainable modules at once.
_PARAM_EPOCH = [0]


def bump_param_epoch() -> None:
    _PARAM_EPOCH[0] += 1


def param_key(params) -> tuple:
    """Cache key of a parameter set: identity + version of every tensor, plus the global epoch when any of them is
    trainable (frozen modules — the teacher — keep their operands across optimiser steps)."""
    params = list(params)
    epoch = _PARAM_EPOCH[0] if any(p.requires_grad for p in params) else -1
    return (epoch, tuple((p.data_ptr(), p._version) for p in params))


# ------------------------------------------------------------------------------------------------ derived weights
@dataclass
class StepConsts:
    """Per-FlowStep tensors derived from the parameters (rebuilt whenever a parameter changes)."""
    Wf: torch.Tensor          # [C,C] fused ActNorm o invconv matrix (forward or inverse direction)
    bf: torch.Tensor          # [C]
    sl: torch.Tensor          # [1] +-(sum logs + sum log_s)
    B1: torch.Tensor = None   # bf16 GEMM operands of the coupling net
    B1T: torch.Tensor = None
    B2: torch.Tensor = None
    B2T: torch.Tensor = None
    B3: torch.Tensor = None
    B3T: torch.Tensor = None
    bias1: torch.Tensor = None
    bias2: torch.Tensor = None
    bias3: torch.Tensor = None


def build_affine(an_bias, an_logs, inv, C, reverse, transpose):
    """inv = (lower, upper, log_s, p, sign_s, weight) with unused entries None."""
    dev = an_bias.device
    Wf = torch.empty(C, C, device=dev, dtype=F32)
    bf = torch.empty(C, device=dev, dtype=F32)
    sl = torch.empty(1, device=dev, dtype=F32)
    lower, upper, log_s, p, sign_s, weight = inv
    ops.invconv_prep(an_bias, an_logs, lower, upper, log_s, p, sign_s, weight, C, reverse, transpose, Wf, bf, sl)
    return Wf, bf, sl


# ------------------------------------------------------------------------------------ batched affine build (K0)
class PrepCtx:
    """The fused ActNorm o invconv matrices of a set of FlowSteps built by ONE launch, and their deferred backward.

    Forward: `PrepAllFn` runs nfk_invconv_prep_batch (one CTA per step) and leaves (Wf, bf, sl) per step in
    `consts`. Each step's autograd Function takes the returned `token` as an input, so the autograd graph knows the
    steps depend on the prep; in its backward the step deposits (dWf, dbf, g_ld) in `grads` instead of running its own
    parameter-space kernel. `PrepAllFn.backward` runs after every step (it is their common ancestor) and turns all the
    deposits into parameter gradients with one nfk_invconv_prep_bwd_batch launch."""

    def __init__(self, steps, reverse: bool):
        self.steps = list(steps)
        self.reverse = bool(reverse)
        self.index = {id(s): i for i, s in enumerate(self.steps)}
        n = len(self.steps)
        self.consts = [None] * n     # (Wf, bf, sl) per step
        self.items = [None] * n
        self.grads = [None] * n      # deposits of the steps' backward: (dWf, ld, dbf, g_ld, B, pixels)
        self.cops = [None] * n       # 2-D steps: (B1, B1T, B2, B2T, B3, B3T, bias1, bias2, bias3)
        self.citems = [None] * n
        self.cgrads = [None] * n     # deposits: (dB1, dbias1, dB2, dbias2, dB3, dbias3)
        self.token = None

    def build(self):
        flat = []
        for st in self.steps:
            iv = st.invconv
            if iv.LU_decomposed:
                flat += [st.actnorm.bias, st.actnorm.logs, iv.lower, iv.upper, iv.log_s]
            else:   # plain weight (layers.py:366-375): same five slots, the matrix in the first, the others unused
                flat += [st.actnorm.bias, st.actnorm.logs, iv.weight, iv.weight, iv.weight]
        for st in self.steps:
            if not st.is_1d:
                flat += list(st._coupling_params_2d())
        self.token = PrepAllFn.apply(self, *flat)
        return self

    def lookup(self, step, reverse):
        i = self.index.get(id(step))
        return None if i is None or self.reverse != bool(reverse) else i


_PREP_STACK: list = []


class use_prep:
    """Context manager: steps called inside find their batched constants in `pctx` (None = no batching)."""

    def __init__(self, pctx):
        self.pctx = pctx

    def __enter__(self):
        if self.pctx is not None:
            _PREP_STACK.append(self.pctx)
        return self.pctx

    def __exit__(self, *exc):
        if self.pctx is not None:
            _PREP_STACK.pop()
            self.pctx.token = None   # every step has taken it; dropping it breaks the pctx <-> grad_fn reference cycle
        return False


def prep_for(step, reverse):
    """(pctx, index, token) of the innermost active batch that holds `step`, else a one-step batch built on the
    spot (whose token reference is dropped at once: see use_prep.__exit__)."""
    for pctx in reversed(_PREP_STACK):
        i = pctx.lookup(step, reverse)
        if i is not None:
            return pctx, i, pctx.token
    pctx = PrepCtx([step], reverse).build()
    token, pctx.token = pctx.token, None
    return pctx, 0, token


def prepare_steps(layers, reverse):
    """Batch every trainable FlowStep in `layers` (called by FlowNet.encode/decode under grad); reverse=True builds the
    inverse-direction matrices, and PrepAllFn.backward then applies the inverse's chain rule."""
    if not torch.is_grad_enabled():
        return None
    steps = [l for l in layers if getattr(l, "_batched_prep_ok", None) is not None and l._batched_prep_ok()
             and l.actnorm.logs.requires_grad]
    if len(steps) < 2:
        return None
    return PrepCtx(steps, reverse).build()


class PrepAllFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pctx, *flat):
        dev = flat[0].device
        sizes = [(st.in_channels * st.in_channels, st.in_channels, 1) for st in pctx.steps]
        total = sum(ops.round_up(a, 4) + ops.round_up(b, 4) + 4 for a, b, _ in sizes)
        buf = torch.empty(total, device=dev, dtype=F32)
        off = 0
        items = []
        for i, st in enumerate(pctx.steps):
            C = st.in_channels
            Wf = buf[off:off + C * C].view(C, C); off += ops.round_up(C * C, 4)
            bf = buf[off:off + C]; off += ops.round_up(C, 4)
            sl = buf[off:off + 1]; off += 4
            an_bias, an_logs, lower, upper, log_s = flat[5 * i:5 * i + 5]
            if st.invconv.LU_decomposed:
                it = ops.invconv_item(an_bias, an_logs, lower, upper, log_s, st.invconv.p, st.invconv.sign_s, None, C,
                                      pctx.reverse, st.is_1d, Wf, bf, sl)
            else:
                it = ops.invconv_item(an_bias, an_logs, None, None, None, None, None, lower, C, pctx.reverse,
                                      st.is_1d, Wf, bf, sl)
            items.append(it)
            pctx.consts[i] = (Wf, bf, sl)
            pctx.items[i] = it
        ops.invconv_prep_batch(items)
        # coupling-net GEMM operands of the 2-D steps, one launch
        off = 5 * len(pctx.steps)
        citems = []
        for i, st in enumerate(pctx.steps):
            if st.is_1d:
                continue
            cw = flat[off:off + 9]; off += 9
            C, hid = st.in_channels, st.hidden_channels
            cin, cout = C // 2, C
            K1p, K3p = ops.round_up(9 * cin, 64), ops.round_up(9 * cout, 64)
            e = lambda *s_: torch.empty(*s_, device=dev, dtype=BF16)
            B1, B2, B3 = e(hid, K1p), e(hid, hid), e(K3p, hid)
            B1T, B2T, B3T = e(K1p, hid), e(hid, hid), e(hid, K3p)
            bias = torch.empty(2 * hid + ops.round_up(cout, 4), device=dev, dtype=F32)
            bias1, bias2, bias3 = bias[:hid], bias[hid:2 * hid], bias[2 * hid:2 * hid + cout]
            it = ops.coupling_item(cw, cin, hid, cout, K1p, K3p, True, B1, B1T, B2, B2T, B3, B3T, bias1, bias2, bias3)
            citems.append(it)
            pctx.citems[i] = it
            pctx.cops[i] = (B1, B1T, B2, B2T, B3, B3T, bias1, bias2, bias3)
        ops.coupling_prep_batch(citems)
        ctx.pctx = pctx
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(*flat)
        return torch.empty(1, device=dev, dtype=F32)

    @staticmethod
    def backward(ctx, _g_token):
        pctx = ctx.pctx
        flat = ctx.saved_tensors
        dev = flat[0].device
        _join_wgrads(dev)      # the last steps' weight gradients may still be in flight on the second stream
        n = len(pctx.steps)
        live = [i for i in range(n) if pctx.grads[i] is not None]
        sizes = []
        for i in live:
            C = pctx.steps[i].in_channels
            sizes += [C, C, C * C, C * C, C]
        offs = [0]
        for sz in sizes:
            offs.append(offs[-1] + ops.round_up(sz, 4))
        arena = torch.empty(offs[-1], device=dev, dtype=F32)
        out = [None] * (5 * n)
        items = []
        for j, i in enumerate(live):
            C = pctx.steps[i].in_channels
            d = [arena[offs[5 * j + k]:offs[5 * j + k] + sizes[5 * j + k]] for k in range(5)]
            d_bias, d_logs = d[0].view_as(flat[5 * i]), d[1].view_as(flat[5 * i + 1])
            d_lower, d_upper, d_log_s = d[2].view(C, C), d[3].view(C, C), d[4]   # (d_log_s: [C], like log_s)
            dWf, dWf_ld, dbf, g_ld, B, pixels = pctx.grads[i]
            if pctx.steps[i].invconv.LU_decomposed:
                items.append(ops.invconv_bwd_item(pctx.items[i], dWf.data_ptr(), dWf_ld, dbf, g_ld, B, pixels, d_bias,
                                                  d_logs, d_lower, d_upper, d_log_s))
                out[5 * i:5 * i + 5] = [d_bias, d_logs, d_lower, d_upper, d_log_s]
            else:   # gradient of the plain weight lands in the first of its three slots
                items.append(ops.invconv_bwd_item(pctx.items[i], dWf.data_ptr(), dWf_ld, dbf, g_ld, B, pixels, d_bias,
                                                  d_logs, None, None, None, d_weight=d_lower))
                out[5 * i:5 * i + 5] = [d_bias, d_logs, d_lower, None, None]
        ops.invconv_prep_bwd_batch(items)
        pctx.grads = [None] * n
        # coupling-net parameters of the 2-D steps
        off = 5 * n
        cout_grads, citems = [], []
        for i, st in enumerate(pctx.steps):
            if st.is_1d:
                continue
            cw = flat[off:off + 9]; off += 9
            if pctx.cgrads[i] is None:
                cout_grads += [None] * 9
                continue
            total = sum(ops.round_up(t.numel(), 4) for t in cw)
            arena_c = torch.empty(total, device=dev, dtype=F32)
            o2, gout = 0, []
            for t in cw:
                gout.append(arena_c[o2:o2 + t.numel()].view_as(t)); o2 += ops.round_up(t.numel(), 4)
            citems.append(ops.coupling_bwd_item(pctx.citems[i], pctx.cgrads[i], gout))
            cout_grads += gout
        ops.coupling_prep_bwd_batch(citems)
        pctx.cgrads = [None] * n
        return (None, *out, *cout_grads)


def build_coupling_ops(cw, cin, hid, cout, with_t):
    """cw = (w1, b1, l1, w2, b2, l2, w3, b3, l3) reference parameters of get_block_2d."""
    dev = cw[0].device
    K1p, K3p = ops.round_up(9 * cin, 64), ops.round_up(9 * cout, 64)
    e = lambda *s: torch.empty(*s, device=dev, dtype=BF16)
    B1, B2, B3 = e(hid, K1p), e(hid, hid), e(K3p, hid)
    B1T, B2T, B3T = (e(K1p, hid), e(hid, hid), e(hid, K3p)) if with_t else (None, None, None)
    bias1 = torch.empty(hid, device=dev, dtype=F32)
    bias2 = torch.empty(hid, device=dev, dtype=F32)
    bias3 = torch.empty(cout, device=dev, dtype=F32)
    ops.coupling_prep(*cw, cin, hid, cout, K1p, K3p, B1, B1T, B2, B2T, B3, B3T, bias1, bias2, bias3, with_t)
    return B1, B1T, B2, B2T, B3, B3T, bias1, bias2, bias3


def _coupling_net(col, k: StepConsts, M, hid, K1p, K3p, keep):
    """conv3x3 -> ReLU -> conv1x1 -> ReLU -> per-tap products of the last conv3x3, all on tcgen05."""
    dev = col.device
    m1 = ops.relu_mask_like(M, hid, dev) if keep else None      # 1-bit ReLU masks for the backward epilogues
    m2 = ops.relu_mask_like(M, hid, dev) if keep else None
    h1 = torch.empty(M, hid, device=dev, dtype=BF16) if keep else None
    h2 = torch.empty(M, hid, device=dev, dtype=BF16)
    if ops.cnet_fused_supported(hid, K1p) and M >= 8192:
        # one kernel for conv#1 + conv#2: h1 stays in tensor memory (and is only written out when training)
        ops.cnet_fwd_fused(col, K1p, k.B1, k.B2, k.bias1, k.bias2, h2, M, hid, h1=h1, mask1=m1, mask2=m2)
    else:
        if h1 is None:
            h1 = torch.empty(M, hid, device=dev, dtype=BF16)
        ops.gemm_nt(col, k.B1, M, hid, K1p, ops.EPI_BIAS_RELU_BF16, h1, bias=k.bias1, aux=m1)
        ops.gemm_nt(h1, k.B2, M, hid, hid, ops.EPI_BIAS_RELU_BF16, h2, bias=k.bias2, aux=m2)
    return (h1, h2, m1, m2) if keep else (None, h2, None, None)


def _conv3_coupling(h2, k: StepConsts, y, hsave, ld, B, C, H, W, hid, K3p, reverse):
    """Conv2dZeros + affine coupling on y (in place) / ld (accumulated): one fused kernel where the shape allows it,
    otherwise per-tap GEMM into P followed by the col2im + coupling kernel."""
    M = B * H * W
    if USE_FUSED_PCONV and ops.pconv_coupling_supported(C, H, W, hid):
        ops.pconv_coupling_fwd(h2, k.B3, K3p, k.bias3, y, hsave, ld, B, C, H, W, hid, reverse)
        return
    P = torch.empty(M, K3p, device=h2.device, dtype=F32)
    ops.gemm_nt(h2, k.B3, M, K3p, hid, ops.EPI_F32, P)
    ops.coupling_fwd(P, K3p, k.bias3, y, hsave, ld, B, C, H, W, reverse=reverse)


def flowstep2d_forward(x, ld_in, k: StepConsts, hid, keep):
    """FlowStep.normal_flow (reference models/flows.py:142-171), 2-D affine coupling."""
    B, C, H, W = x.shape
    M, cin = B * H * W, C // 2
    K1p, K3p = ops.round_up(9 * cin, 64), ops.round_up(9 * C, 64)
    dev = x.device
    y = torch.empty_like(x)
    col = torch.empty(M, K1p, device=dev, dtype=BF16)
    ld_out = torch.empty(B, device=dev, dtype=F32)
    ops.affine1x1_fwd(x, k.Wf, k.bf, k.sl, y, col, K1p, ld_in, ld_out, B, C, H, W)
    h1, h2, m1, m2 = _coupling_net(col, k, M, hid, K1p, K3p, keep)
    hsave = torch.empty(M, C, device=dev, dtype=F32) if keep else None
    _conv3_coupling(h2, k, y, hsave, ld_out, B, C, H, W, hid, K3p, False)
    return y, ld_out, (col, h1, h2 if keep else None, hsave, m1, m2)


def flowstep2d_reverse(z, ld_in, k: StepConsts, hid, keep=False):
    """FlowStep.reverse_flow (reference models/flows.py:173-202): coupling^-1 -> invconv^-1 -> actnorm^-1.
    k.Wf / k.bf / k.sl hold the INVERSE affine here. keep=True (training) also returns what FlowStep2dReverseFn's
    backward reads: (zc = the post-coupling tensor, col, h1, h2, hsave, m1, m2); the outputs are the same bits."""
    B, C, H, W = z.shape
    M, cin = B * H * W, C // 2
    K1p, K3p = ops.round_up(9 * cin, 64), ops.round_up(9 * C, 64)
    dev = z.device
    col = torch.empty(M, K1p, device=dev, dtype=BF16)
    ops.affine1x1_fwd(z, None, None, None, None, col, K1p, None, None, B, C, H, W)   # im2col of z1 only
    h1, h2, m1, m2 = _coupling_net(col, k, M, hid, K1p, K3p, keep)
    hsave = torch.empty(M, C, device=dev, dtype=F32) if keep else None
    zc = z.clone()
    ld_mid = ld_in.clone()
    _conv3_coupling(h2, k, zc, hsave, ld_mid, B, C, H, W, hid, K3p, True)
    x = torch.empty_like(z)
    ld_out = torch.empty_like(ld_mid)
    ops.affine1x1_fwd(zc, k.Wf, k.bf, k.sl, x, None, 0, ld_mid, ld_out, B, C, H, W)
    if keep:
        return x, ld_out, (zc, col, h1, h2, hsave, m1, m2)
    return x, ld_out


def _grad_arena(C, hid, K1p, K3p, dev):
    """One zero-filled arena for every accumulate-into buffer of a 2-D step's backward:
    (arena, dbias3, dbias2, dbias1, dB3, dB2, dB1, dWf, dbf)."""
    sizes = [C, hid, hid, K3p * hid, hid * hid, hid * K1p, C * C, C]
    offs = [0]
    for s in sizes:
        offs.append(offs[-1] + ops.round_up(s, 4))
    arena = torch.zeros(offs[-1], device=dev, dtype=F32)
    dbias3, dbias2, dbias1, dB3, dB2, dB1, dWf, dbf = (arena[offs[i]:offs[i] + sizes[i]] for i in range(8))
    return (arena, dbias3, dbias2, dbias1, dB3.view(K3p, hid), dB2.view(hid, hid), dB1.view(hid, K1p),
            dWf.view(C, C), dbf)


def _coupling_net_backward(dhcol, col, h1, h2, m1, m2, B1T, B2T, B3T, dbias2, dbias1, dB3, dB2, dB1, arena, M, hid,
                           K1p, K3p):
    """Backward of the coupling net (direction-independent): from the bf16 im2col of dh [M, K3p] to the masked
    gradient at the first conv's output dpre1 [M, hid] bf16 (returned; the first conv's input gradient is left to the
    caller, see _conv1_dgrad), accumulating the three weight gradients and the two bias gradients.
    Small batches issue the weight gradients on the second stream (see WGRAD_STREAM_MAX_M)."""
    dev = dhcol.device
    dpre2 = torch.empty(M, hid, device=dev, dtype=BF16)
    dpre1 = torch.empty(M, hid, device=dev, dtype=BF16)
    if ops.cnet_fused_supported(hid, K3p) and M >= 8192:
        # both dgrads of the chain in ONE kernel: dpre2 stays in tensor memory as the second GEMM's A operand
        ops.cnet_bwd_fused(dhcol, K3p, B3T, B2T, m2, m1, dpre2, dpre1, dbias2, dbias1, M, hid)
    else:
        ops.gemm_nt(dhcol, B3T, M, hid, K3p, ops.EPI_MASK_BF16, dpre2, aux=m2, colsum=dbias2)
        ops.gemm_nt(dpre2, B2T, M, hid, hid, ops.EPI_MASK_BF16, dpre1, aux=m1, colsum=dbias1)
    if 0 < M <= WGRAD_STREAM_MAX_M:
        cur, side = torch.cuda.current_stream(dev), _wgrad_stream(dev)
        side.wait_stream(cur)                          # fork: dhcol / dpre2 / dpre1 and the zeroed arena exist
        with torch.cuda.stream(side):
            ops.gemm_tn(dhcol, h2, K3p, hid, M, dB3)
            ops.gemm_tn(dpre2, h1, hid, hid, M, dB2)
            ops.gemm_tn(dpre1, col, hid, K1p, M, dB1)
        _wgrad_keepalive.append((dhcol, dpre2, dpre1, h1, h2, col, arena))
    else:
        ops.gemm_tn(dhcol, h2, K3p, hid, M, dB3)
        ops.gemm_tn(dpre2, h1, hid, hid, M, dB2)
        ops.gemm_tn(dpre1, col, hid, K1p, M, dB1)
    return dpre1


def _conv1_dgrad(dpre1, B1T, M, K1p, hid):
    """The first conv's input gradient as per-tap products dcol [M, K1p] fp32 (column = tap*(C/2) + ci)."""
    dcol = torch.empty(M, K1p, device=dpre1.device, dtype=F32)
    ops.gemm_nt(dpre1, B1T, M, K1p, hid, ops.EPI_F32, dcol)
    return dcol


class FlowStep2dFn(torch.autograd.Function):
    """Differentiable 2-D FlowStep forward. Inputs: x, logdet and the prep token (see PrepCtx): the fused affine comes
    from pctx.consts[idx], the coupling net's bf16 GEMM operands from pctx.cops[idx]; parameter gradients are produced
    by PrepAllFn.backward from what this step's backward deposits in pctx."""

    @staticmethod
    def forward(ctx, x, ld_in, hid, token, pctx, idx):
        B, C, H, W = x.shape
        x = x.contiguous()
        Wf, bf, sl = pctx.consts[idx]
        k = StepConsts(Wf, bf, sl, *pctx.cops[idx])
        y, ld_out, (col, h1, h2, hsave, m1, m2) = flowstep2d_forward(x, ld_in.contiguous(), k, hid, keep=True)
        ctx.hid = hid
        ctx.pctx, ctx.idx = pctx, idx
        ctx.save_for_backward(x, y, col, h1, h2, hsave, m1, m2, Wf, k.B1T, k.B2T, k.B3T)
        return y, ld_out

    @staticmethod
    def backward(ctx, g_out, g_ld):
        (x, z_out, col, h1, h2, hsave, m1, m2, Wf, B1T, B2T, B3T) = ctx.saved_tensors
        hid = ctx.hid
        B, C, H, W = x.shape
        M, cin = B * H * W, C // 2
        K1p, K3p = ops.round_up(9 * cin, 64), ops.round_up(9 * C, 64)
        dev = x.device
        _join_wgrads(dev)      # the previous step's weight gradients (before anything here can reuse their buffers)
        g_out = torch.zeros_like(x) if g_out is None else g_out.contiguous()
        g_ld = torch.zeros(B, device=dev, dtype=F32) if g_ld is None else g_ld.contiguous()
        arena, dbias3, dbias2, dbias1, dB3, dB2, dB1, dWf, dbf = _grad_arena(C, hid, K1p, K3p, dev)

        dy = torch.empty_like(x)
        dhcol = torch.empty(M, K3p, device=dev, dtype=BF16)
        ops.coupling_bwd(g_out, g_ld, z_out, hsave, dy, dhcol, K3p, dbias3, B, C, H, W)
        dpre1 = _coupling_net_backward(dhcol, col, h1, h2, m1, m2, B1T, B2T, B3T, dbias2, dbias1, dB3, dB2, dB1, arena,
                                       M, hid, K1p, K3p)
        dx = torch.empty_like(x)
        if USE_FUSED_DGRAD1 and ops.conv1_dgrad_affine_bwd_supported(C, H, W, hid):
            # conv#1 dgrad + col2im + affine1x1_bwd in one kernel: the fp32 dcol never goes through HBM
            ops.conv1_dgrad_affine_bwd(dpre1, B1T, K1p, dy, x, Wf, dx, dWf, dbf, B, C, H, W, hid)
        else:
            dcol = _conv1_dgrad(dpre1, B1T, M, K1p, hid)
            ops.affine1x1_bwd(dy, dcol, K1p, x, Wf, dx, dWf, dbf, B, C, H, W)

        # the parameter-space chain rules (fused affine, folded conv operands) are deferred to PrepAllFn.backward:
        # one batched launch each for all steps of the pass
        ctx.pctx.grads[ctx.idx] = (dWf, C, dbf, g_ld, B, float(H * W))
        ctx.pctx.cgrads[ctx.idx] = (dB1, dbias1, dB2, dbias2, dB3, dbias3)
        return (dx, g_ld, None, None, None, None)


class FlowStep2dReverseFn(torch.autograd.Function):
    """Differentiable 2-D FlowStep INVERSE (reference models/flows.py:173-202), the counterpart of FlowStep2dFn for the
    perceptual term, whose gradient reaches the student through its inverse pass (pl_module.py:229-243). pctx holds
    the inverse-direction affine; the deposits feed PrepAllFn.backward's inverse chain rule.

    z = [z1, z2], h = NN(z1), zc2 = z2 / s - shift, x = Wf zc + bf. Backward: dzc = Wf^T g_x (affine1x1_bwd, also dWf,
    dbf), dz2 = dzc2 / s and dh (coupling_inv_bwd), the coupling net's backward to dcol, dz1 = dzc1 + col2im(dcol)."""

    @staticmethod
    def forward(ctx, z, ld_in, hid, token, pctx, idx):
        z = z.contiguous()
        Wf, bf, sl = pctx.consts[idx]
        k = StepConsts(Wf, bf, sl, *pctx.cops[idx])
        x, ld_out, (zc, col, h1, h2, hsave, m1, m2) = flowstep2d_reverse(z, ld_in.contiguous(), k, hid, keep=True)
        ctx.hid = hid
        ctx.pctx, ctx.idx = pctx, idx
        ctx.save_for_backward(zc, col, h1, h2, hsave, m1, m2, Wf, k.B1T, k.B2T, k.B3T)
        return x, ld_out

    @staticmethod
    def backward(ctx, g_x, g_ld):
        (zc, col, h1, h2, hsave, m1, m2, Wf, B1T, B2T, B3T) = ctx.saved_tensors
        hid = ctx.hid
        B, C, H, W = zc.shape
        M, cin = B * H * W, C // 2
        K1p, K3p = ops.round_up(9 * cin, 64), ops.round_up(9 * C, 64)
        dev = zc.device
        _join_wgrads(dev)
        g_x = torch.zeros_like(zc) if g_x is None else g_x.contiguous()
        g_ld = torch.zeros(B, device=dev, dtype=F32) if g_ld is None else g_ld.contiguous()
        arena, dbias3, dbias2, dbias1, dB3, dB2, dB1, dWf, dbf = _grad_arena(C, hid, K1p, K3p, dev)

        dzc = torch.empty_like(zc)
        ops.affine1x1_bwd(g_x, None, K1p, zc, Wf, dzc, dWf, dbf, B, C, H, W)
        dz = torch.empty_like(zc)
        dhcol = torch.empty(M, K3p, device=dev, dtype=BF16)
        ops.coupling_inv_bwd(dzc, g_ld, zc, hsave, dz, dhcol, K3p, dbias3, B, C, H, W)
        dpre1 = _coupling_net_backward(dhcol, col, h1, h2, m1, m2, B1T, B2T, B3T, dbias2, dbias1, dB3, dB2, dB1, arena,
                                       M, hid, K1p, K3p)
        ops.col2im_add(_conv1_dgrad(dpre1, B1T, M, K1p, hid), K1p, dz, B, C, H, W)

        ctx.pctx.grads[ctx.idx] = (dWf, C, dbf, g_ld, B, float(H * W))
        ctx.pctx.cgrads[ctx.idx] = (dB1, dbias1, dB2, dbias2, dB3, dbias3)
        return (dz, g_ld, None, None, None, None)


# ------------------------------------------------------------------------------------------------ Split2d
class Split2dFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, ld_in, w, bias, logs):
        B, C, H, W = x.shape
        x = x.contiguous()
        z1 = torch.empty(B, C // 2, H, W, device=x.device, dtype=F32)
        ld = ld_in.clone()
        ops.split2d_fwd(x, w, bias, logs, z1, ld, B, C, H, W)
        ctx.save_for_backward(x, w, bias, logs)
        return z1, ld

    @staticmethod
    def backward(ctx, g_z1, g_ld):
        x, w, bias, logs = ctx.saved_tensors
        B, C, H, W = x.shape
        dev = x.device
        g_ld = torch.zeros(B, device=dev, dtype=F32) if g_ld is None else g_ld.contiguous()
        g_z1 = None if g_z1 is None else g_z1.contiguous()
        dx = torch.empty_like(x)
        nw = w.numel()
        arena = torch.zeros(nw + 2 * C, device=dev, dtype=F32)
        dw, dbias, dlogs = arena[:nw].view_as(w), arena[nw:nw + C].view_as(bias), arena[nw + C:].view_as(logs)
        ops.split2d_bwd(x, w, bias, logs, g_z1, g_ld, dx, dw, dbias, dlogs, B, C, H, W)
        return dx, g_ld, dw, dbias, dlogs


class Split2dSqueezeFn(torch.autograd.Function):
    """Split2d followed by the next level's SqueezeLayer in ONE kernel each way (layers.py:293-327): returns z1, its
    space-to-depth copy [B, 4*C/2, H/2, W/2] and the log-det; the backward reads the squeezed tensor's gradient through
    the same index map (no permute / contiguous pass in either direction)."""

    @staticmethod
    def forward(ctx, x, ld_in, w, bias, logs):
        B, C, H, W = x.shape
        x = x.contiguous()
        z1 = torch.empty(B, C // 2, H, W, device=x.device, dtype=F32)
        z1_sq = torch.empty(B, 2 * C, H // 2, W // 2, device=x.device, dtype=F32)
        ld = ld_in.clone()
        ops.split2d_fwd(x, w, bias, logs, z1, ld, B, C, H, W, z1_sq=z1_sq)
        ctx.save_for_backward(x, w, bias, logs)
        return z1, z1_sq, ld

    @staticmethod
    def backward(ctx, g_z1, g_sq, g_ld):
        x, w, bias, logs = ctx.saved_tensors
        B, C, H, W = x.shape
        dev = x.device
        g_ld = torch.zeros(B, device=dev, dtype=F32) if g_ld is None else g_ld.contiguous()
        g_z1 = None if g_z1 is None else g_z1.contiguous()
        g_sq = None if g_sq is None else g_sq.contiguous()
        dx = torch.empty_like(x)
        nw = w.numel()
        arena = torch.zeros(nw + 2 * C, device=dev, dtype=F32)
        dw, dbias, dlogs = arena[:nw].view_as(w), arena[nw:nw + C].view_as(bias), arena[nw + C:].view_as(logs)
        ops.split2d_bwd(x, w, bias, logs, g_z1, g_ld, dx, dw, dbias, dlogs, B, C, H, W, g_z1_sq=g_sq)
        return dx, g_ld, dw, dbias, dlogs


def split2d_reverse(z1, w, bias, logs, eps, temperature):
    B, CH, H, W = z1.shape
    out = torch.empty(B, 2 * CH, H, W, device=z1.device, dtype=F32)
    ops.split2d_rev(z1.contiguous(), w, bias, logs, eps, temperature, out, B, 2 * CH, H, W)
    return out


class Split2dReverseFn(torch.autograd.Function):
    """Split2d reverse under autograd: cat(z1, z2) with z2 ~ N(mean(z1), exp(logs(z1)) * T) sampled by the split2d_rev
    kernel. The reference samples with torch.normal, whose derivative with respect to mean and std is zero, so z2 is a
    constant to autograd: z1 gets the pass-through half of the gradient and the Split2d parameters get none."""

    @staticmethod
    def forward(ctx, z1, w, bias, logs, eps, temperature):
        ctx.ch = z1.shape[1]
        return split2d_reverse(z1, w.detach(), bias.detach(), logs.detach(), eps, temperature)

    @staticmethod
    def backward(ctx, g):
        return g[:, :ctx.ch], None, None, None, None, None


# ------------------------------------------------------------------------------------------------ prior -> bpd
class PriorBpdFn(torch.autograd.Function):
    """bpd[b] = -(logdet[b] + log N(z_b; mean, exp(logs))) * scale (reference models/kd_flows.py:134-150)."""

    @staticmethod
    def forward(ctx, z, logdet, mean, logs, scale):
        B = z.shape[0]
        n = z[0].numel()
        z = z.contiguous()
        out = torch.empty(B, device=z.device, dtype=F32)
        ops.prior_bpd_fwd(z, mean, logs, logdet.contiguous(), B, n, scale, out)
        ctx.save_for_backward(z, mean, logs)
        ctx.scale = scale
        return out

    @staticmethod
    def backward(ctx, g):
        z, mean, logs = ctx.saved_tensors
        B = z.shape[0]
        n = z[0].numel()
        dz = torch.empty_like(z)
        dld = torch.empty(B, device=z.device, dtype=F32)
        ops.prior_bpd_bwd(z, mean, logs, g.contiguous(), B, n, ctx.scale, dz, dld)
        return dz, dld, None, None, None


# ------------------------------------------------------------------------------------------------ KD loss
class KdMseFn(torch.autograd.Function):
    """kd[b] = (1/L) sum_levels mean_i (s_i - t_i)^2 in one accumulation buffer (pl_module.py:266-282).
    Inputs: L student tensors followed by L teacher tensors (teacher is constant)."""

    @staticmethod
    def forward(ctx, *tensors):
        L = len(tensors) // 2
        s = [t.contiguous() for t in tensors[:L]]
        t = [t.contiguous() for t in tensors[L:]]
        B = s[0].shape[0]
        acc = torch.zeros(B, device=s[0].device, dtype=F32)
        for a, b in zip(s, t):
            n = a[0].numel()
            ops.kd_mse_fwd(a, b, B, n, 1.0 / (n * L), acc)
        ctx.save_for_backward(*s, *t)
        ctx.L = L
        return acc

    @staticmethod
    def backward(ctx, g):
        L = ctx.L
        saved = ctx.saved_tensors
        g = g.contiguous()
        grads = []
        for a, b in zip(saved[:L], saved[L:]):
            B, n = a.shape[0], a[0].numel()
            ds = torch.empty_like(a)
            ops.kd_mse_bwd(a, b, g, B, n, 1.0 / (n * L), ds)
            grads.append(ds)
        return (*grads, *([None] * L))


class KdNllLossFn(torch.autograd.Function):
    """NFModel.loss (pl_module.py:257-320) as ONE forward and ONE backward launch (csrc/loss_optim.cu): multi-level
    latent MSE + prior log-density / bits-per-dim objective + weighted sum + the four batch means.

    apply(spec, logdet_or_nll, z_last, perc, *student_levels) -> (means[4] = (nll, kd, perceptual, loss), nll[B], kd[B])
    spec: dict(teacher=[...], prior=(mean_row, logs_row) | None, nll_scale, w=(w_nll, w_kd, w_perc), sample_w).
    z_last None: `logdet_or_nll` already is the per-sample objective (models whose prior is not a fixed row)."""

    @staticmethod
    def forward(ctx, spec, ld_or_nll, z_last, perc, *s_levels):
        s = [t.contiguous() for t in s_levels]
        t = [x.detach().contiguous() for x in spec["teacher"]]
        assert len(s) == len(t)
        B = ld_or_nll.shape[0]
        dev = ld_or_nll.device
        ld_or_nll = ld_or_nll.contiguous()
        z_last = None if z_last is None else z_last.contiguous()
        perc = None if perc is None else perc.contiguous()
        mean, logs = spec["prior"] if spec.get("prior") is not None else (None, None)
        sw = spec.get("sample_w")
        sw = None if sw is None else sw.detach().to(F32).contiguous()
        w_nll, w_kd, w_perc = spec["w"]
        out = torch.empty(4 + 2 * B, device=dev, dtype=F32)
        means, nll, kd = out[:4], out[4:4 + B], out[4 + B:]
        ops.kd_nll_loss_fwd(s, t, z_last, mean, logs, ld_or_nll if z_last is not None else None,
                            spec.get("nll_scale", 1.0), None if z_last is not None else ld_or_nll, perc, sw,
                            w_nll, w_kd, w_perc, B, nll, kd, means)
        ctx.spec, ctx.sw, ctx.L, ctx.B = spec, sw, len(s), B
        ctx.has_z, ctx.has_perc = z_last is not None, perc is not None
        ctx.save_for_backward(z_last, mean, logs, *s, *t)
        ctx.mark_non_differentiable(nll, kd)
        return means, nll, kd

    @staticmethod
    def backward(ctx, g_means, _g_nll, _g_kd):
        z_last, mean, logs, *st = ctx.saved_tensors
        L, B = ctx.L, ctx.B
        s, t = st[:L], st[L:]
        spec = ctx.spec
        w_nll, w_kd, w_perc = spec["w"]
        dev = g_means.device
        needs = ctx.needs_input_grad
        ds = [torch.empty_like(a) if needs[4 + i] else None for i, a in enumerate(s)]
        dz = torch.empty_like(z_last) if ctx.has_z and needs[2] else None
        d_first = torch.empty(B, device=dev, dtype=F32) if needs[1] else None
        dperc = torch.empty(B, device=dev, dtype=F32) if ctx.has_perc and needs[3] else None
        ops.kd_nll_loss_bwd(s, t, ds, z_last if ctx.has_z else None, mean, logs, spec.get("nll_scale", 1.0), ctx.sw,
                            w_nll, w_kd, w_perc, B, g_means.contiguous(), None, None, dz,
                            d_first if ctx.has_z else None, None if ctx.has_z else d_first, dperc)
        return (None, d_first, dz, dperc, *ds)


def kd_mse(student_levels, teacher_levels) -> Optional[torch.Tensor]:
    if not student_levels:
        return None
    return KdMseFn.apply(*student_levels, *[t.detach() for t in teacher_levels])
