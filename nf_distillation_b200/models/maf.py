"""MAF / MADE with the same calling conventions as the Glow modules (forward -> (z, logdet), reverse, and a
``...GetAllOutputs`` wrapper returning (list[z], nll[B], None)) so NFModel.forward / loss work unchanged.

The reference repository names MAF in README.md:7 but ships NO MAF/MADE code (SURVEY.md §0.2), so there is nothing to be
in parity with: this follows Papamakarios et al. 2017 / Germain et al. 2015 and is checked against the repo's own
plain-PyTorch restatement (oracle/maf_oracle.py) — "parity unpinned".

MADE here: D -> H (ReLU) -> H (ReLU) -> 2D masked linears; hidden degrees are assigned in sorted order, which makes
the H x H mask block-lower-triangular so the tensor-core GEMM skips its structurally-zero k-blocks."""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from .. import functional as Fn
from .. import ops
from .layers import _as_logdet, _require_cuda

BF16, F32 = torch.bfloat16, torch.float32


def hidden_degrees(D: int, H: int) -> torch.Tensor:
    """Sorted degrees in [1, D-1], each value ~H/(D-1) times (D == 1 degenerates to all ones): the standard MADE
    assignment (Germain et al. 2015, eq. 12-13 with deterministic, evenly spread degrees). When H is a multiple of 8
    AND there are at least D-1 tiles of 8 units, the degree changes only on multiples of 8 units (whole MMA column
    tiles), which is what lets the inverse kernel feed a finished layer-2 tile straight from its accumulators into the
    output sums (csrc/maf_inverse.cu, push); every degree 1..D-1 still occurs. With fewer tiles than degrees the
    tile-aligned form would drop degrees (outputs 2..8 would see only degree-1 units), so the per-unit assignment is
    used and the inverse runs the pull kernel."""
    if D <= 1:
        return torch.ones(H, dtype=torch.int32)
    if H % 8 == 0 and H // 8 >= D - 1:
        tiles = H // 8
        return (torch.arange(tiles, dtype=torch.int64) * (D - 1) // tiles + 1).repeat_interleave(8).to(torch.int32)
    return (torch.arange(H, dtype=torch.int64) * (D - 1) // H + 1).to(torch.int32)


def _kb_ranges(deg_out, deg_in, bn, strict_rows=None):
    """k-block [begin, end) per n-tile for mask[o][k] = deg_out[o] >= deg_in[k] (both sorted ascending)."""
    H_out, H_in = len(deg_out), len(deg_in)
    nkb = H_in // 64
    begins, ends = [], []
    for n0 in range(0, H_out, bn):
        dmax = int(deg_out[min(n0 + bn, H_out) - 1])
        kmax = int((deg_in <= dmax).sum())          # inputs [0, kmax) can be non-zero
        begins.append(0)
        ends.append(max(1, min(nkb, (kmax + 63) // 64)))
    return begins, ends


def _kb_ranges_t(deg_out, deg_in, bn):
    """Transposed mask (dgrad): rows = inputs k, reduction over outputs o with deg_out[o] >= deg_in[k]."""
    H_out, H_in = len(deg_out), len(deg_in)
    nkb = H_out // 64
    begins, ends = [], []
    for n0 in range(0, H_in, bn):
        dmin = int(deg_in[n0])
        omin = int((deg_out < dmin).sum())          # outputs [omin, H_out) can be non-zero
        begins.append(min(nkb - 1, omin // 64))
        ends.append(nkb)
    return begins, ends


class _MadePlan:
    """What one degree assignment (deg1, deg2) fixes, derived on the host once per assignment (MADE._plan): sorted
    (both ascending), resident_ok (sorted, no degree 0: what the resident inverse and the reverse solve need), the
    k-block ranges of the H x H masked linear and of its transpose (full when unsorted), the fused kernel's
    kb2_end_half0, the resident inverse's job table (on the degrees' device), push flag and stream bytes, and the
    reverse solve's job table and stream bytes (None when not resident_ok or the shape does not fit the kernel).
    It holds the degree tensors it was built from, so no pointer in `key` can be reused while it is alive."""

    def __init__(self, made, key):
        self.key, self.deg1, self.deg2 = key, made.deg1, made.deg2
        d1, d2 = self.deg1.detach().cpu().long(), self.deg2.detach().cpu().long()
        D, H, Dp, N3p, bn = made.D, made.H, made.Dp, made.N3p, made.bn
        nkb = H // 64
        self.sorted = bool((d1[1:] >= d1[:-1]).all() and (d2[1:] >= d2[:-1]).all())
        self.resident_ok = self.sorted and bool(d1.min() >= 1 and d2.min() >= 1)
        if self.sorted:
            self.ranges, self.ranges_t = _kb_ranges(d2, d1, bn), _kb_ranges_t(d2, d1, bn)
            self.kb2_end_half0 = _kb_ranges(d2, d1, 256)[1][0] if H == 512 else nkb
        else:
            nt = (H + bn - 1) // bn
            self.ranges = self.ranges_t = ([0] * nt, [nkb] * nt)
            self.kb2_end_half0 = nkb
        self.jobs, self.push, self.nbytes, self.bwd_jobs, self.bwd_nbytes = None, False, 0, None, 0
        if not self.resident_ok:
            return
        edges = torch.arange(D + 1)
        cnt1, cnt2 = ((d[None, :] <= edges[:, None]).sum(1) for d in (d1, d2))   # cnt[d] = units of degree <= d
        dev = self.deg1.device
        if ops.made_inverse_resident_supported(D, H, Dp):
            jobs = None
            if made.push_inverse and ops.made_inverse_push_supported(D, H, Dp, N3p):
                jobs = ops.made_inverse_jobs(cnt1, cnt2, D, H, Dp, N3p, push=True)
                self.push = jobs is not None
            if jobs is None:
                jobs = ops.made_inverse_jobs(cnt1, cnt2, D, H, Dp)
            self.jobs, self.nbytes = jobs.to(dev), int(jobs[:, 5].sum()) * 16
        if ops.made_inverse_bwd_supported(D, H, N3p):
            jobs = ops.made_inverse_bwd_jobs(cnt1, cnt2, D, H, N3p)
            self.bwd_jobs, self.bwd_nbytes = jobs.to(dev), int(jobs[:, 5].sum()) * 16


class _MadeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, ld_in, made, flip, xb, w1, b1, w2, b2, w3, b3):
        x = x.contiguous()
        ops_ = made._operands((w1, b1, w2, b2, w3, b3), True)
        u, ld_out, ub, saved = made._run_forward(x, ld_in.contiguous(), ops_, b1, b2, flip, True, xb)
        ctx.made, ctx.flip = made, flip
        ctx.save_for_backward(x, *saved)
        ctx.mark_non_differentiable(ub)
        return u, ld_out, ub

    @staticmethod
    def backward(ctx, g_u, g_ld, _g_ub):
        made, flip = ctx.made, ctx.flip
        x, xb, h1, h2, m1, m2, out, B1T, B2T, B3T = ctx.saved_tensors
        B = x.shape[0]
        dev = x.device
        g_u = torch.zeros_like(x) if g_u is None else g_u.contiguous()
        g_ld = torch.zeros(B, device=dev, dtype=F32) if g_ld is None else g_ld.contiguous()
        grads = _made_grad_arena(made, dev)
        dx = torch.empty_like(x)
        dout = torch.empty(B, made.N3p, device=dev, dtype=BF16)
        ops.made_affine_bwd(x, out, made.N3p, g_u, g_ld, dx, dout, grads[0], B, made.D, flip)
        dxn, dw1, dw2, dw3 = _made_net_backward(made, dout, xb, h1, h2, m1, m2, B1T, B2T, B3T, grads, True)
        dx = dx + dxn[:, :made.D]
        db3, db2, db1 = grads[:3]
        return dx, g_ld, None, None, None, dw1, db1, dw2, db2, dw3, db3


def _made_grad_arena(made, dev):
    """Zeroed fp32 accumulators (db3, db2, db1, dB3, dB2, dB1) of one MADE layer's parameter gradients, one allocation."""
    D, H, Dp, N3p = made.D, made.H, made.Dp, made.N3p
    sizes = [2 * D, H, H, N3p * H, H * H, H * Dp]
    offs = [0]
    for s in sizes:
        offs.append(offs[-1] + ops.round_up(s, 4))
    arena = torch.zeros(offs[-1], device=dev, dtype=F32)
    db3, db2, db1, dB3, dB2, dB1 = (arena[offs[i]:offs[i] + sizes[i]] for i in range(6))
    return db3, db2, db1, dB3.view(N3p, H), dB2.view(H, H), dB1.view(H, Dp)


def _made_net_backward(made, dout, xb, h1, h2, m1, m2, B1T, B2T, B3T, grads, want_dx):
    """The masked network's backward at the forward's saved activations, from dout = [dmu | dalpha] (bf16 [B, N3p]):
    accumulates db2, db1 and dB3, dB2, dB1 into `grads` (_made_grad_arena; db3 is the caller's), returns
    (dxn [B, Dp] fp32 or None, dw1, dw2, dw3)."""
    D, H, Dp, N3p = made.D, made.H, made.Dp, made.N3p
    B = dout.shape[0]
    dev = dout.device
    _, db2, db1, dB3, dB2, dB1 = grads
    dpre2 = torch.empty(B, H, device=dev, dtype=BF16)
    ops.gemm_nt(dout, B3T, B, H, N3p, ops.EPI_MASK_BF16, dpre2, aux=m2, colsum=db2)
    ops.gemm_tn(dout, h2, N3p, H, B, dB3)
    dpre1 = torch.empty(B, H, device=dev, dtype=BF16)
    kb0, kb1 = made._plan().ranges_t
    ops.gemm_nt_ranged(dpre2, B2T, B, H, H, ops.EPI_MASK_BF16, dpre1, made.bn, kb0, kb1, aux=m1, colsum=db1)
    ops.gemm_tn(dpre2, h1, H, H, B, dB2)
    dxn = None
    if want_dx:
        dxn = torch.empty(B, Dp, device=dev, dtype=F32)
        ops.gemm_nt(dpre1, B1T, B, Dp, H, ops.EPI_F32, dxn)
    ops.gemm_tn(dpre1, xb, H, Dp, B, dB1)
    dw1, dw2, dw3 = (torch.empty(H, D, device=dev), torch.empty(H, H, device=dev),
                     torch.empty(2 * D, H, device=dev))
    ops.made_prep_bwd(dB1, dB2, dB3, made.deg1, made.deg2, D, H, Dp, dw1, dw2, dw3)
    return dxn, dw1, dw2, dw3


class _MadeInverseFn(torch.autograd.Function):
    """The sequential inverse x = MADE^-1(u) with gradients. The forward is the no-grad inverse unchanged (x is
    bit-identical); the backward recomputes the forward network at x (activations and ReLU masks), runs the reverse
    solve (MADE._inverse_solve) for g_u and dout = [mubar | alphabar], and the forward's parameter chain from dout."""

    @staticmethod
    def forward(ctx, u_in, ld_in, made, flip, w1, b1, w2, b2, w3, b3):
        u_in = u_in.contiguous()
        x, ld_out = made._run_inverse(u_in, ld_in, True, (w1, b1, w2, b2, w3, b3))
        ctx.made, ctx.flip = made, flip
        ctx.save_for_backward(u_in, x, w1, b1, w2, b2, w3, b3)
        return x, ld_out

    @staticmethod
    def backward(ctx, g_x, g_ld):
        made, flip = ctx.made, ctx.flip
        u_in, x, *params = ctx.saved_tensors
        B = x.shape[0]
        dev = x.device
        g_x = torch.zeros_like(x) if g_x is None else g_x.contiguous()
        g_ld = None if g_ld is None else g_ld.contiguous()
        ops_ = made._operands(params, True)
        xb = made._bf16_rows(x, None)
        h1, h2, out, m1, m2 = made._net(xb, B, ops_, params[1], params[3], keep=True)
        grads = _made_grad_arena(made, dev)
        g_u = torch.empty_like(x)
        dout = torch.empty(B, made.N3p, device=dev, dtype=BF16)
        made._inverse_solve(g_x, g_ld, u_in, out, m1, m2, ops_, flip, g_u, dout, grads[0])
        _, dw1, dw2, dw3 = _made_net_backward(made, dout, xb, h1, h2, m1, m2, ops_[1], ops_[3], ops_[5], grads, False)
        db3, db2, db1 = grads[:3]
        return g_u, g_ld, None, None, dw1, db1, dw2, db2, dw3, db3


class MADE(nn.Module):
    """One masked autoregressive layer: forward x -> u with logdet = -sum(alpha); reverse is the sequential inverse
    (one launch, activations resident in shared memory: csrc/maf_inverse.cu)."""

    def __init__(self, num_inputs: int, hidden_features: int, flip: bool):
        super().__init__()
        if hidden_features % 64:
            raise NotImplementedError("MADE hidden width must be a multiple of 64 (tcgen05 k-block)")
        D, H = num_inputs, hidden_features
        self.D, self.H, self.flip = D, H, bool(flip)
        self.Dp, self.N3p = ops.round_up(D, 64), ops.round_up(2 * D, 64)
        self.bn = 128 if H % 128 == 0 else 64
        self.fc1, self.fc2, self.fc3 = nn.Linear(D, H), nn.Linear(H, H), nn.Linear(H, 2 * D)
        with torch.no_grad():   # start close to the identity transform
            self.fc3.weight.mul_(0.1)
            self.fc3.bias.zero_()
        deg = hidden_degrees(D, H)
        self.register_buffer("deg1", deg.clone())
        self.register_buffer("deg2", deg.clone())
        self._plan_cache = None   # _MadePlan of the current degree buffers
        self._cache = None        # no-grad operands: [param_key, plan, operands, resident inverse's weight stream]
        self.push_inverse = True         # False: the pull kernel (h2 kept in shared memory) even for aligned degrees
        self.resident_inverse = True     # False: the D-pass GEMM inverse and reverse solve (the cross-checks in the tests)
        self.resident_mtiles = 0         # 16-sample tiles per warp in the resident inverse (0 = chosen by the library)

    def _plan(self):
        """The plan of the current degree buffers (a loaded checkpoint may carry other degrees than the constructor's)
        and push_inverse. Building one reads the degrees to the host, so the first eager call builds it: a CUDA graph
        captured after that finds it here."""
        d1, d2 = self.deg1, self.deg2
        key = (d1.data_ptr(), d1._version, d2.data_ptr(), d2._version, str(d1.device), self.push_inverse)
        if self._plan_cache is None or self._plan_cache.key != key:
            self._plan_cache = _MadePlan(self, key)
        return self._plan_cache

    # views of the plan: (job table on `dev`, push?) of the resident inverse, (job table, stream bytes) or None of
    # the reverse solve
    @property
    def _ranges(self):
        return self._plan().ranges

    def _inverse_jobs(self, dev):
        plan = self._plan()
        return (None if plan.jobs is None else plan.jobs.to(dev)), plan.push

    def _inverse_bwd_jobs(self, dev):
        plan = self._plan()
        return None if plan.bwd_jobs is None else (plan.bwd_jobs.to(dev), plan.bwd_nbytes)

    def _pack_stream(self, plan, ops_):
        ws = torch.zeros(max(plan.nbytes, 128), device=plan.jobs.device, dtype=torch.uint8)
        ops.made_inverse_pack(plan.jobs, ops_[0], ops_[2], ops_[4], self.N3p, self.D, self.H, self.Dp, plan.push, ws)
        return ws

    def _params(self):
        return (self.fc1.weight, self.fc1.bias, self.fc2.weight, self.fc2.bias, self.fc3.weight, self.fc3.bias)

    def _operands(self, params, with_t):
        w1, b1, w2, b2, w3, b3 = params
        dev = w1.device
        D, H, Dp, N3p = self.D, self.H, self.Dp, self.N3p
        e = lambda *s: torch.empty(*s, device=dev, dtype=BF16)
        B1, B2, B3 = e(H, Dp), e(H, H), e(N3p, H)
        B1T, B2T, B3T = (e(Dp, H), e(H, H), e(H, N3p)) if with_t else (None, None, None)
        ops.made_prep(w1, w2, w3, self.deg1, self.deg2, D, H, Dp, N3p, B1, B1T, B2, B2T, B3, B3T, with_t)
        b3p = torch.zeros(N3p, device=dev, dtype=F32)
        b3p[:2 * D] = b3
        return B1, B1T, B2, B2T, B3, B3T, b3p

    def _cached_operands(self):
        """The operands of the current parameters for no-grad calls, cached on param_key and the plan: made_prep bakes
        the degree masks into them."""
        key, plan = Fn.param_key(self._params()), self._plan()
        if self._cache is None or self._cache[0] != key or self._cache[1] is not plan:
            self._cache = [key, plan, self._operands(tuple(p.detach() for p in self._params()), False), None]
        return self._cache[2]

    def _cached_stream(self):
        """The resident inverse's packed weight stream of _cached_operands(), kept in the same cache entry, which holds
        the plan and operands it was packed from."""
        ops_ = self._cached_operands()
        if self._cache[3] is None:
            self._cache[3] = self._pack_stream(self._cache[1], ops_)
        return self._cache[3]

    def _net(self, xb, Bn, ops_, b1, b2, keep=False):
        """(mu | alpha) = masked MLP(xb) on the tensor cores; returns h1, h2, out (+ 1-bit ReLU masks if keep)."""
        B1, _, B2, _, B3, _, b3p = ops_
        dev = xb.device
        H, Dp, N3p = self.H, self.Dp, self.N3p
        plan = self._plan()
        m1 = ops.relu_mask_like(Bn, H, dev) if keep else None
        m2 = ops.relu_mask_like(Bn, H, dev) if keep else None
        h2 = torch.empty(Bn, H, device=dev, dtype=BF16)
        if ops.cnet_fused_supported(H, Dp, Bn):
            # both masked linears in ONE kernel (the coupling net's fused conv#1 -> conv#2 kernel: h1 stays in tensor
            # memory as the second GEMM's A operand and is only written out when training). The masks are zeros in the
            # bf16 weights here; skipping their k-blocks would save < what the h1 round trip through HBM costs.
            h1 = torch.empty(Bn, H, device=dev, dtype=BF16) if keep else None
            # k-blocks of the hidden weight that output channels [0, 256) can see (block-triangular mask): the rest
            # are exact zeros in B2 and are skipped
            ops.cnet_fwd_fused(xb, Dp, B1, B2, b1, b2, h2, Bn, H, h1=h1, mask1=m1, mask2=m2,
                               kb2_end_half0=plan.kb2_end_half0)
        else:
            h1 = torch.empty(Bn, H, device=dev, dtype=BF16)
            ops.gemm_nt(xb, B1, Bn, H, Dp, ops.EPI_BIAS_RELU_BF16, h1, bias=b1, aux=m1)
            kb0, kb1 = plan.ranges
            ops.gemm_nt_ranged(h1, B2, Bn, H, H, ops.EPI_BIAS_RELU_BF16, h2, self.bn, kb0, kb1, bias=b2, aux=m2)
        out = torch.empty(Bn, N3p, device=dev, dtype=F32)
        ops.gemm_nt(h2, B3, Bn, N3p, H, ops.EPI_F32, out, bias=b3p)
        return (h1, h2, out, m1, m2) if keep else (h1, h2, out)

    def _bf16_rows(self, x, xb):
        """bf16 zero-padded copy of x [B, Dp] for the first GEMM; reuses the copy the previous MADE layer's
        affine kernel already wrote (attached to its output as `_nfk_bf16`) when there is one."""
        Bn = x.shape[0]
        if xb is not None and xb.shape == (Bn, self.Dp) and xb.dtype == BF16 and xb.device == x.device:
            return xb
        xb = torch.empty(Bn, self.Dp, device=x.device, dtype=BF16)
        ops.rows_to_bf16(x, Bn, self.D, self.Dp, xb)
        return xb

    def _run_forward(self, x, ld_in, ops_, b1, b2, flip, keep, xb=None):
        """u = MADE(x) and ld_out = ld_in - sum alpha from the operands ops_; keep: also returns what _MadeFn's
        backward saves. ub is u's bf16 copy for the next layer's first GEMM."""
        Bn = x.shape[0]
        dev = x.device
        xb = self._bf16_rows(x, xb)
        res = self._net(xb, Bn, ops_, b1, b2, keep)
        h1, h2, out = res[:3]
        u = torch.empty_like(x)
        ub = torch.empty(Bn, self.Dp, device=dev, dtype=BF16)   # the next layer's GEMM operand
        ld_out = torch.empty(Bn, device=dev, dtype=F32)
        ops.made_affine_fwd(x, out, self.N3p, u, ub, self.Dp, ld_in, ld_out, Bn, self.D, flip)
        return u, ld_out, ub, ((xb, h1, h2, res[3], res[4], out, ops_[1], ops_[3], ops_[5]) if keep else None)

    def forward(self, input, y_onehot=None, logdet=None, reverse=False, **kwargs):
        _require_cuda(input, "MADE")
        Bn = input.shape[0]
        ld = _as_logdet(logdet, Bn, input.device)
        want = ld is not None
        if ld is None:
            ld = torch.zeros(Bn, device=input.device)
        params = self._params()
        if not reverse:
            xb_in = getattr(input, "_nfk_bf16", None)      # (bf16 copy, version of the tensor it was made from)
            xb_in = xb_in[0] if xb_in is not None and xb_in[1] == input._version else None
            if torch.is_grad_enabled() and (input.requires_grad or any(p.requires_grad for p in params)):
                u, ld_out, ub = _MadeFn.apply(input, ld, self, self.flip, xb_in, *params)
            else:
                x = input.contiguous()
                u, ld_out, ub, _ = self._run_forward(x, ld.contiguous(), self._cached_operands(), params[1].detach(),
                                                     params[3].detach(), self.flip, False,
                                                     xb_in if x is input else None)
            u._nfk_bf16 = (ub, u._version)   # bf16 copy for the next MADE layer (saves its conversion pass)
            return u, (ld_out if want else None)
        if torch.is_grad_enabled() and (input.requires_grad or ld.requires_grad or any(p.requires_grad for p in params)):
            x, ld_out = _MadeInverseFn.apply(input, ld, self, self.flip, *params)
            return x, (ld_out if want else None)
        return self._run_inverse(input.contiguous(), ld, want)

    def _run_inverse(self, u_in, ld, want, params=None):
        """x = MADE^-1(u_in) and (want) ld_out = ld + sum alpha, without gradients. params=None (frozen modules:
        no-grad calls): the operands and the packed weight stream come from _cached_operands / _cached_stream. Given
        params (the trainable path): both are rebuilt from them on every call, as the forward's _MadeFn does, because
        an optimiser that writes the parameters through raw pointers (FlatAdam) bumps no version, and a captured graph
        must contain the rebuild."""
        Bn = u_in.shape[0]
        plan = self._plan()
        resident = plan.jobs is not None and self.resident_inverse
        if params is None:
            params = self._params()
            ops_ = self._cached_operands()
            ws = self._cached_stream() if resident else None
        else:
            params = tuple(p.detach() for p in params)
            ops_ = self._operands(params, False)
            ws = self._pack_stream(plan, ops_) if resident else None
        b1, b2 = params[1].detach(), params[3].detach()
        if resident:
            # ONE launch: every hidden unit finalised once, in degree order, activations resident in shared memory
            x = torch.empty_like(u_in)
            ld_out = torch.empty(Bn, device=x.device, dtype=F32) if want else None
            ops.made_inverse_resident(u_in, ws, b1, b2, ops_[6], plan.jobs, plan.push, self.N3p, x,
                                      ld.contiguous() if want else None, ld_out, Bn, self.D, self.H, self.Dp,
                                      self.flip, self.resident_mtiles)
            return x, ld_out
        # fallback (unsorted degrees / shapes the resident kernel does not take): D passes of the three GEMMs,
        # activations in HBM / L2, one column of x fixed per pass
        x = torch.zeros_like(u_in)
        xb = torch.zeros(Bn, self.Dp, device=x.device, dtype=BF16)
        ld_out = torch.empty(Bn, device=x.device, dtype=F32)
        ldc = ld.contiguous()
        for i in range(self.D):
            _, _, out = self._net(xb, Bn, ops_, b1, b2)
            ops.made_inv_update(x, xb, self.Dp, u_in, out, self.N3p, ldc, ld_out, Bn, self.D, i, self.flip,
                                i == self.D - 1)
        return x, (ld_out if want else None)

    def _inverse_solve(self, g_x, g_ld, u_in, out, m1, m2, ops_, flip, g_u, dout, db3):
        """Reverse solve of the inverse's gradients at x (out, m1, m2 from the forward network recomputed at x):
        writes g_u, dout = [mubar | alphabar | 0] and adds dout's column sums to db3. One launch when the plan has
        the reverse solve's jobs (and resident_inverse is on); else D passes of the three dgrad GEMMs."""
        B = u_in.shape[0]
        D, H, Dp, N3p = self.D, self.H, self.Dp, self.N3p
        _, B1T, _, B2T, _, B3T, _ = ops_
        plan = self._plan()
        if plan.bwd_jobs is not None and self.resident_inverse:
            # (no memset: the pack writes every row the kernel multiplies; the bytes it leaves alone are only read
            # into MMA columns the kernel discards)
            ws = torch.empty(max(plan.bwd_nbytes, 128), device=u_in.device, dtype=torch.uint8)
            ops.made_inverse_bwd_pack(plan.bwd_jobs, B1T, B2T, B3T, D, H, N3p, ws)
            ops.made_inverse_bwd_resident(g_x, g_ld, out, m1, m2, u_in, ws, plan.bwd_jobs, g_u, dout, db3, B, D, H,
                                          N3p, flip, self.resident_mtiles)
            return
        dout.zero_()
        c = torch.empty(B, Dp, device=u_in.device, dtype=F32)
        dpre2 = torch.empty(B, H, device=u_in.device, dtype=BF16)
        dpre1 = torch.empty(B, H, device=u_in.device, dtype=BF16)
        kb0, kb1 = plan.ranges_t
        for d in reversed(range(D)):
            if d < D - 1:   # c = the network's input gradient for the rows finished so far
                ops.gemm_nt(dout, B3T, B, H, N3p, ops.EPI_MASK_BF16, dpre2, aux=m2)
                ops.gemm_nt_ranged(dpre2, B2T, B, H, H, ops.EPI_MASK_BF16, dpre1, self.bn, kb0, kb1, aux=m1)
                ops.gemm_nt(dpre1, B1T, B, Dp, H, ops.EPI_F32, c)
            ops.made_inv_bwd_update(c if d < D - 1 else None, Dp, g_x, g_ld, out, N3p, u_in, g_u, dout, db3, B, D, d,
                                    flip)


class MAFNet(nn.Module):
    """Stack of MADE layers with order reversal in between; `layers` / `output_shapes` like FlowNet."""

    def __init__(self, num_inputs, hidden_features, num_layers):
        super().__init__()
        self.layers = nn.ModuleList([MADE(num_inputs, hidden_features, flip=True) for _ in range(num_layers)])
        self.output_shapes = [[-1, num_inputs] for _ in range(num_layers)]

    def forward(self, input, y_onehot=None, logdet=0.0, reverse=False, temperature=None):
        outs = []
        z = input
        if not reverse:
            for layer in self.layers:
                z, logdet = layer(z, logdet=logdet, reverse=False)
                outs.append(z)
            return outs, logdet
        for layer in reversed(self.layers):
            z, _ = layer(z, logdet=None, reverse=True)
            outs.append(z)
        return outs


class MAFGetAllOutputs(nn.Module):
    """MAF density model with the GlowGetAllOutputs interface (is_1d semantics: nll in nats)."""

    def __init__(self, image_shape, hidden_channels, K, L=1, **unused):
        super().__init__()
        D = image_shape[0]
        self.is_1d = True
        self.y_condition = False
        self.learn_top = False
        self.flow = MAFNet(D, hidden_channels, K * L)
        self.register_buffer("prior_h", torch.zeros(1, 2 * D))

    def prior(self, data, y_onehot=None):
        batch = data.shape[0] if data is not None else (y_onehot.size(0) if y_onehot is not None else 32)
        h = self.prior_h.repeat(batch, 1)
        D = h.shape[1] // 2
        return h[:, :D], h[:, D:]

    def forward(self, x=None, y_onehot=None, z=None, temperature=None, reverse=False):
        from .. import functional as Fn
        if reverse:
            if z is None:
                mean, logs = self.prior(z, y_onehot)
                z = torch.normal(mean, torch.exp(logs) * (1.0 if temperature is None else temperature))
            return self.flow(z, reverse=True, temperature=temperature)
        _require_cuda(x, "MAF")
        logdet = torch.zeros(x.shape[0], device=x.device, dtype=F32)
        outs, logdet = self.flow(x, logdet=logdet, reverse=False)
        D = self.prior_h.shape[1] // 2
        nll = Fn.PriorBpdFn.apply(outs[-1], logdet, self.prior_h[0, :D].contiguous(),
                                  self.prior_h[0, D:].contiguous(), 1.0)
        return outs, nll, None


def create_maf_model(config) -> MAFGetAllOutputs:
    """config keys: image_shape=[D], hidden_channels=H, K=number of MADE layers (same keys as the Glow configs)."""
    return MAFGetAllOutputs(**config)
