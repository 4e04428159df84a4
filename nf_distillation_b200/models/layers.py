"""Drop-in mirror of the reference's models/layers.py: same class names, constructor arguments, parameter /
buffer names (=> identical ``state_dict`` keys) and call signatures; the arithmetic runs in libnfk CUDA kernels.

Reference line numbers refer to /root/reference/models/layers.py.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from .. import functional as Fn
from .. import ops
from .utils import compute_same_pad, split_feature  # noqa: F401  (re-exported like the reference)


def _require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise RuntimeError(f"{what}: nf_distillation_b200 has no CPU path; move the module and its inputs to CUDA")


def _as_logdet(logdet, B, device):
    """The reference threads logdet as a [B] tensor, a python float (0.0) or None (layers.py:129-142,296)."""
    if logdet is None:
        return None
    if torch.is_tensor(logdet) and logdet.dim() == 1 and logdet.shape[0] == B:
        return logdet.to(torch.float32)
    return torch.zeros(B, device=device, dtype=torch.float32) + logdet


# -------------------------------------------------------------------------------------------- Gaussian helpers
def gaussian_p(mean, logs, x):
    """Element-wise diagonal-Gaussian log density (layers.py:10-17)."""
    c = math.log(2 * math.pi)
    return -0.5 * (logs * 2.0 + ((x - mean) ** 2) / torch.exp(logs * 2.0) + c)


def gaussian_likelihood(mean, logs, x):
    """Summed over all non-batch dims (layers.py:20-23)."""
    return gaussian_p(mean, logs, x).flatten(1).sum(1)


def gaussian_sample(mean, logs, temperature=1):
    """z ~ N(mean, (exp(logs) * T)^2) from the global torch generator (layers.py:26-29).

    Written as normal_(0,1)*std+mean, which is what torch.normal(mean, std) does internally (same Philox draws), minus
    its host-side `std.min() >= 0` check: that check synchronises and cannot be captured in a CUDA graph, and
    exp(logs)*T with T >= 0 is non-negative by construction."""
    return torch.empty_like(mean).normal_().mul_(torch.exp(logs) * temperature).add_(mean)


def squeeze2d(input, factor):
    """Space-to-depth; out channel = c*f*f + fh*f + fw (layers.py:32-44)."""
    if factor == 1:
        return input
    B, C, H, W = input.size()
    assert H % factor == 0 and W % factor == 0, "H or W modulo factor is not 0"
    x = input.view(B, C, H // factor, factor, W // factor, factor)
    return x.permute(0, 1, 3, 5, 2, 4).contiguous().view(B, C * factor * factor, H // factor, W // factor)


def unsqueeze2d(input, factor):
    """Depth-to-space (layers.py:47-61)."""
    if factor == 1:
        return input
    f2 = factor ** 2
    B, C, H, W = input.size()
    assert C % f2 == 0, "C module factor squared is not 0"
    x = input.view(B, C // f2, factor, factor, H, W)
    return x.permute(0, 1, 4, 2, 5, 3).contiguous().view(B, C // f2, H * factor, W * factor)


# -------------------------------------------------------------------------------------------- ActNorm
class _ActNorm(nn.Module):
    """Per-channel affine (x + bias) * exp(logs) with log-det pixels * sum(logs) (layers.py:64-142).

    Inside a FlowStep the affine is folded into the invertible 1x1 conv (one kernel); called on its own it runs the
    same kernel with an identity mixing matrix. Data-dependent initialisation never runs in the reference pipeline
    (create_glow_model -> set_actnorm_init forces ``inited``), it is kept for API parity."""

    def __init__(self, num_features, scale=1.0, is_1d=False):
        super().__init__()
        self.is_1d = is_1d
        size = [1, num_features] + ([] if is_1d else [1, 1])
        self.bias = nn.Parameter(torch.zeros(*size))
        self.logs = nn.Parameter(torch.zeros(*size))
        self.num_features = num_features
        self.scale = scale
        self.inited = False

    def initialize_parameters(self, input):
        if not self.training:
            raise ValueError("In Eval mode, but ActNorm not inited")
        dims = [0] + ([] if self.is_1d else [2, 3])
        with torch.no_grad():
            bias = -input.mean(dim=dims, keepdim=True)
            var = ((input + bias) ** 2).mean(dim=dims, keepdim=True)
            self.bias.data.copy_(bias)
            self.logs.data.copy_(torch.log(self.scale / (var.sqrt() + 1e-6)))
            self.inited = True

    def forward(self, input, logdet=None, reverse=False):
        self._check_input_dim(input)
        _require_cuda(input, type(self).__name__)
        if not self.inited:
            self.initialize_parameters(input)
        if torch.is_grad_enabled() and (input.requires_grad or self.bias.requires_grad):
            # stand-alone differentiable use is off the hot path: plain tensor ops (FlowStep is the fused path)
            e = torch.exp(-self.logs) if reverse else torch.exp(self.logs)
            out = input * e - self.bias if reverse else (input + self.bias) * e
            if logdet is not None:
                pix = 1 if self.is_1d else input.shape[2] * input.shape[3]
                d = self.logs.sum() * pix
                logdet = logdet - d if reverse else logdet + d
            return out, logdet
        C = self.num_features
        eye = torch.eye(C, device=input.device)
        B = input.shape[0]
        x4 = input.contiguous().view(B, C, 1, 1) if self.is_1d else input.contiguous()
        Wf, bf, sl = Fn.build_affine(self.bias.detach(), self.logs.detach(), (None, None, None, None, None, eye), C,
                                     reverse, False)
        ld_in = _as_logdet(logdet, B, input.device)
        y = torch.empty_like(x4)
        ld_out = None if ld_in is None else torch.empty_like(ld_in)
        _affine_any(x4, Wf, bf, sl, y, ld_in, ld_out)
        return y.view_as(input), ld_out


def _affine_any(x4, Wf, bf, sl, y, ld_in, ld_out):
    B, C, H, W = x4.shape
    if C in (12, 24, 48, 96):
        ops.affine1x1_fwd(x4, Wf, bf, sl, y, None, 0, ld_in, ld_out, B, C, H, W)
    else:
        from .. import flow1d
        flow1d.affine_rows(x4, Wf, bf, sl, y, ld_in, ld_out)


class ActNorm2d(_ActNorm):
    def __init__(self, num_features, scale=1.0):
        super().__init__(num_features, scale, is_1d=False)

    def _check_input_dim(self, input):
        assert len(input.size()) == 4
        assert input.size(1) == self.num_features, (
            "[ActNorm]: input should be in shape as `B x C x H x W`, channels should be {} rather than {}".format(
                self.num_features, input.size()))


class ActNorm1d(_ActNorm):
    def __init__(self, num_features, scale=1.0):
        super().__init__(num_features, scale, is_1d=True)

    def _check_input_dim(self, input):
        assert len(input.size()) == 2
        assert input.size(1) == self.num_features, (
            "[ActNorm]: input should be in shape as `B x C`, channels should be {} rather than {}".format(
                self.num_features, input.size()))


# -------------------------------------------------------------------------------------------- small linear heads
class LinearZeros(nn.Module):
    """Zero-initialised Linear with exp(3*logs) output scale (layers.py:173-187). Only used by the conditional /
    learn_top heads (SURVEY §8f 'next'): a [B, classes] x [classes, 2C] product, kept as a library call."""

    def __init__(self, in_channels, out_channels, logscale_factor=3):
        super().__init__()
        self.linear = nn.Linear(in_channels, out_channels)
        self.linear.weight.data.zero_()
        self.linear.bias.data.zero_()
        self.logscale_factor = logscale_factor
        self.logs = nn.Parameter(torch.zeros(out_channels))

    def forward(self, input):
        return self.linear(input) * torch.exp(self.logs * self.logscale_factor)


# -------------------------------------------------------------------------------------------- coupling convs
class Conv2d(nn.Module):
    """3x3 / 1x1 'same' conv without bias followed by an ActNorm affine (layers.py:190-228). Parameter container:
    inside FlowStep the conv runs as a tcgen05 implicit-GEMM tile with the affine + ReLU fused in the epilogue."""

    def __init__(self, in_channels, out_channels, kernel_size=(3, 3), stride=(1, 1), padding="same",
                 do_actnorm=True, weight_std=0.05):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size, stride, bias=(not do_actnorm))
        torch.nn.init.xavier_normal_(self.conv.weight)
        if not do_actnorm:
            self.conv.bias.data.zero_()
        else:
            self.actnorm = ActNorm2d(out_channels)
        self.do_actnorm = do_actnorm
        self.kernel_size = tuple(kernel_size)

    def forward(self, input):
        raise NotImplementedError(
            "Conv2d is fused into FlowStep (conv -> ActNorm -> ReLU is one tcgen05 GEMM tile); call the FlowStep")


class Conv2dZeros(nn.Module):
    """Zero-initialised 3x3 conv + bias with exp(3*logs) output scale (layers.py:231-260). Parameter container for
    FlowStep / Split2d / learn_top."""

    def __init__(self, in_channels, out_channels, kernel_size=(3, 3), stride=(1, 1), padding="same",
                 logscale_factor=3):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size, stride)
        self.conv.weight.data.zero_()
        self.conv.bias.data.zero_()
        self.logscale_factor = logscale_factor
        self.logs = nn.Parameter(torch.zeros(out_channels, 1, 1))

    def forward(self, input, **kwargs):
        raise NotImplementedError("Conv2dZeros is fused into FlowStep / Split2d; call those modules")


class Permute2d(nn.Module):
    """Fixed channel permutation (reverse or shuffle), layers.py:263-290. No shipped config uses it."""

    def __init__(self, num_channels, shuffle):
        super().__init__()
        self.num_channels = num_channels
        self.indices = torch.arange(self.num_channels - 1, -1, -1, dtype=torch.long)
        self.indices_inverse = torch.zeros((self.num_channels), dtype=torch.long)
        for i in range(self.num_channels):
            self.indices_inverse[self.indices[i]] = i
        if shuffle:
            self.reset_indices()

    def reset_indices(self):
        shuffle_idx = torch.randperm(self.indices.shape[0])
        self.indices = self.indices[shuffle_idx]
        for i in range(self.num_channels):
            self.indices_inverse[self.indices[i]] = i

    def forward(self, input, reverse=False, **kwargs):
        assert len(input.size()) == 4
        idx = self.indices_inverse if reverse else self.indices
        return input.index_select(1, idx.to(input.device))


# -------------------------------------------------------------------------------------------- Split2d
class Split2d(nn.Module):
    """Multi-scale split (layers.py:293-313): forward scores z2 under N(mean(z1), exp(logs(z1))) and returns z1;
    reverse samples z2. One fused kernel each way (direct 3x3 conv + Gaussian log-density reduction)."""

    def __init__(self, num_channels):
        super().__init__()
        self.conv = Conv2dZeros(num_channels // 2, num_channels)

    def _params(self):
        c = self.conv
        return c.conv.weight, c.conv.bias, c.logs

    def forward(self, input, logdet=0.0, reverse=False, temperature=None, **kwargs):
        _require_cuda(input, "Split2d")
        w, b, l = self._params()
        B = input.shape[0]
        if reverse:
            eps = None
            if temperature is None or temperature != 0:
                eps = torch.randn_like(input)
            T = 1.0 if temperature is None else float(temperature)
            if torch.is_grad_enabled():
                # z2 is a constant to autograd like the reference's torch.normal draw: only z1's half flows back
                out = Fn.Split2dReverseFn.apply(input, w.detach(), b.detach(), l.detach(), eps, T)
            else:
                out = Fn.split2d_reverse(input, w.detach(), b.detach(), l.detach(), eps, T)
            return out, logdet
        ld = _as_logdet(logdet, B, input.device)
        if ld is None:
            ld = torch.zeros(B, device=input.device)
        if torch.is_grad_enabled() and (input.requires_grad or w.requires_grad):
            return Fn.Split2dFn.apply(input, ld, w, b, l)
        with torch.no_grad():
            return Fn.Split2dFn.apply(input, ld, w, b, l)


    def forward_with_squeeze(self, input, logdet=0.0):
        """Forward of this Split2d AND of the SqueezeLayer(2) that follows it in FlowNet, one kernel:
        returns (z1, squeeze2d(z1, 2), logdet)."""
        _require_cuda(input, "Split2d")
        w, b, l = self._params()
        ld = _as_logdet(logdet, input.shape[0], input.device)
        if ld is None:
            ld = torch.zeros(input.shape[0], device=input.device)
        if torch.is_grad_enabled() and (input.requires_grad or w.requires_grad):
            return Fn.Split2dSqueezeFn.apply(input, ld, w, b, l)
        with torch.no_grad():
            return Fn.Split2dSqueezeFn.apply(input, ld, w, b, l)


class SqueezeLayer(nn.Module):
    def __init__(self, factor):
        super().__init__()
        self.factor = factor

    def forward(self, input, logdet=None, reverse=False, **kwargs):
        out = unsqueeze2d(input, self.factor) if reverse else squeeze2d(input, self.factor)
        return out, logdet


# -------------------------------------------------------------------------------------------- invertible 1x1 conv
class InvertibleConv1x1(nn.Module):
    """LU-parametrised invertible channel mixing (layers.py:330-421). Parameters / buffers: p, sign_s, lower, log_s,
    upper (or ``weight`` when LU_decomposed is False)."""

    def __init__(self, num_channels, LU_decomposed, is_1d=False):
        super().__init__()
        self.is_1d = is_1d
        w_shape = [num_channels, num_channels]
        w_init = torch.linalg.qr(torch.randn(*w_shape))[0]
        if not LU_decomposed:
            self.weight = nn.Parameter(w_init.contiguous())   # (QR returns a column-major Q; the kernels read rows)
        else:
            p, lower, upper = torch.lu_unpack(*torch.linalg.lu_factor(w_init))
            s = torch.diag(upper)
            self.register_buffer("p", p)
            self.register_buffer("sign_s", torch.sign(s))
            self.lower = nn.Parameter(lower)
            self.log_s = nn.Parameter(torch.log(torch.abs(s)))
            self.upper = nn.Parameter(torch.triu(upper, 1))
            self.l_mask = torch.tril(torch.ones(w_shape), -1)
            self.eye = torch.eye(*w_shape)
        self.w_shape = w_shape
        self.LU_decomposed = LU_decomposed

    def lu_tensors(self):
        """(lower, upper, log_s, p, sign_s, weight) with unused entries None, as the prep kernel expects."""
        if self.LU_decomposed:
            return (self.lower, self.upper, self.log_s, self.p, self.sign_s, None)
        return (None, None, None, None, None, self.weight)

    def get_weight(self, input, reverse):
        """(weight, dlogdet) like the reference (layers.py:360-402), computed by the prep kernel."""
        C = self.w_shape[0]
        pix = 1 if self.is_1d else input.shape[2] * input.shape[3]
        z = torch.zeros(C, device=input.device)
        inv = tuple(None if t is None else t.detach() for t in self.lu_tensors())
        Wf, _, sl = Fn.build_affine(z, z, inv, C, reverse, False)
        w = Wf if self.is_1d else Wf.view(C, C, 1, 1)
        return w, (-sl[0] if reverse else sl[0]) * pix

    def forward(self, input, logdet=None, reverse=False):
        _require_cuda(input, "InvertibleConv1x1")
        C = self.w_shape[0]
        B = input.shape[0]
        z = torch.zeros(C, device=input.device)
        inv = tuple(None if t is None else t.detach() for t in self.lu_tensors())
        Wf, bf, sl = Fn.build_affine(z, z, inv, C, reverse, self.is_1d)
        x4 = input.contiguous().view(B, C, 1, 1) if self.is_1d else input.contiguous()
        ld_in = _as_logdet(logdet, B, input.device)
        y = torch.empty_like(x4)
        ld_out = None if ld_in is None else torch.empty_like(ld_in)
        _affine_any(x4, Wf, bf, sl, y, ld_in, ld_out)
        return y.view_as(input), ld_out
