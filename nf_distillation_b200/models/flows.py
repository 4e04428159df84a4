"""Drop-in mirror of the reference's models/flows.py (FlowStep / FlowNet / Glow): same constructor arguments,
module tree and call signatures. FlowStep runs as a fixed sequence of libnfk kernels (functional.py).

Reference line numbers refer to /root/reference/models/flows.py.
"""
from __future__ import annotations

import logging
import math

import torch
import torch.nn as nn

from .. import functional as Fn
from .. import ops
from .layers import (ActNorm1d, ActNorm2d, Conv2d, Conv2dZeros, InvertibleConv1x1, LinearZeros, Permute2d, Split2d,
                     SqueezeLayer, _as_logdet, _require_cuda, gaussian_likelihood, gaussian_sample)
from .utils import (can_fuse_dequant_squeeze, dequantize_and_squeeze, split_feature,
                    uniform_binning_correction)

logger = logging.getLogger(__name__)


def get_block_2d(in_channels, out_channels, hidden_channels):
    """conv3x3+ActNorm -> ReLU -> conv1x1+ActNorm -> ReLU -> zero-init conv3x3 (flows.py:25-34). The Sequential
    only holds the parameters (state_dict keys block.{0,2,4}.*); FlowStep executes it as three tcgen05 GEMMs."""
    return nn.Sequential(
        Conv2d(in_channels, hidden_channels),
        nn.ReLU(inplace=False),
        Conv2d(hidden_channels, hidden_channels, kernel_size=(1, 1)),
        nn.ReLU(inplace=False),
        Conv2dZeros(hidden_channels, out_channels),
    )


def get_block_1d(in_features, out_features, hidden_features):
    """6-Linear MLP, ReLU x4 then Tanh (flows.py:37-52); executed by the fused 1-D coupling kernel."""
    return nn.Sequential(
        nn.Linear(in_features, hidden_features), nn.ReLU(inplace=False),
        nn.Linear(hidden_features, hidden_features), nn.ReLU(inplace=False),
        nn.Linear(hidden_features, hidden_features), nn.ReLU(inplace=False),
        nn.Linear(hidden_features, hidden_features), nn.ReLU(inplace=False),
        nn.Linear(hidden_features, hidden_features), nn.Tanh(),
        nn.Linear(hidden_features, out_features),
    )


class _PermutationAsLU:
    """A fixed channel permutation (Permute2d: flow_permutation 'shuffle' / 'reverse', reference flows.py:85-95) in the
    LU parametrisation the kernels take: W = P (L + I)(U + diag(sign_s e^{log_s})) with L = U = 0, log_s = 0,
    sign_s = 1 is the permutation matrix itself and log|det W| = 0, so the step runs through the same fused
    ActNorm o 1x1 kernels (forward, inverse, training) as an invertible conv whose factors never train. Nothing here
    is a Parameter or a buffer: the reference's Permute2d has neither, so the state_dict keys stay identical."""

    LU_decomposed = True

    def __init__(self, perm: Permute2d):
        self.perm = perm
        self._key = None
        self.lower = self.upper = self.log_s = self.p = self.sign_s = None

    def sync(self, device):
        idx = self.perm.indices
        key = (tuple(idx.tolist()), str(device))
        if key != self._key:
            C = idx.numel()
            p = torch.zeros(C, C)
            p[torch.arange(C), idx.cpu()] = 1.0          # z[:, o] = x[:, indices[o]]  <=>  W[o, indices[o]] = 1
            self.p = p.to(device)
            self.lower, self.upper = torch.zeros(C, C, device=device), torch.zeros(C, C, device=device)
            self.log_s, self.sign_s = torch.zeros(C, device=device), torch.ones(C, device=device)
            self._key = key
        return self

    def lu_tensors(self):
        return (self.lower, self.upper, self.log_s, self.p, self.sign_s, None)


class FlowStep(nn.Module):
    """actnorm -> invertible 1x1 conv (or a fixed permutation) -> affine (or additive) coupling, forward and inverse
    (flows.py:55-202)."""

    def __init__(self, in_channels, hidden_channels, actnorm_scale, flow_permutation, flow_coupling, LU_decomposed,
                 is_1d=False, condition_features=0):
        super().__init__()
        self.is_1d = is_1d
        self.flow_coupling = flow_coupling
        self.flow_permutation_type = flow_permutation
        self.condition_features = condition_features
        self.in_channels = in_channels
        self.hidden_channels = hidden_channels

        self.actnorm = ActNorm1d(in_channels, actnorm_scale) if is_1d else ActNorm2d(in_channels, actnorm_scale)
        if flow_permutation == "invconv":
            self.invconv = InvertibleConv1x1(in_channels, LU_decomposed=LU_decomposed, is_1d=is_1d)
        elif flow_permutation == "shuffle":
            if is_1d:
                raise RuntimeError("Permutation is not supported is 1d mode")
            self.shuffle = Permute2d(in_channels, shuffle=True)
            self.invconv = _PermutationAsLU(self.shuffle)      # (plain attribute: not a sub-module, no state)
        else:
            if is_1d:
                raise RuntimeError("Permutation is not supported is 1d mode")
            self.reverse = Permute2d(in_channels, shuffle=False)
            self.invconv = _PermutationAsLU(self.reverse)

        if flow_coupling == "additive":
            out_block = in_channels - in_channels // 2
        elif flow_coupling == "affine":
            out_block = (in_channels - in_channels // 2) * 2
        else:
            raise NameError(f"Unknown coupling type: {flow_coupling}")
        in_block = in_channels // 2 + condition_features
        make = get_block_1d if is_1d else get_block_2d
        self.block = make(in_block, out_block, hidden_channels)
        self._cache = {}
        # arithmetic of the coupling-net GEMMs (2-D): "bf16" = bf16 operands, fp32 accumulate (default, the benched
        # mode); "bf16x3" = fp32-class split products (nf_distillation_b200/precise.py). Glow.set_precision sets it.
        self.precision = "bf16"

    # ---- parameter views in the order the kernels expect
    def _coupling_params_2d(self):
        b = self.block
        w3, b3, l3 = b[4].conv.weight, b[4].conv.bias, b[4].logs
        if self.flow_coupling == "additive":
            # z2 + block(z1) (reference flows.py:157-158) on the affine kernels with the scale pinned to one: the
            # Conv2dZeros gets interleaved 'logit' rows with zero weights and bias 30, so sigmoid(30 + 2) == 1.0f and
            # log sigmoid = -1.3e-14 per element. Built with differentiable ops: gradients reach the real rows only.
            w3 = torch.stack((w3, torch.zeros_like(w3)), 1).flatten(0, 1)
            b3 = torch.stack((b3, torch.full_like(b3, 30.0)), 1).flatten()
            l3 = torch.stack((l3, torch.zeros_like(l3)), 1).flatten(0, 1)
        return (b[0].conv.weight, b[0].actnorm.bias, b[0].actnorm.logs,
                b[2].conv.weight, b[2].actnorm.bias, b[2].actnorm.logs, w3, b3, l3)

    def _sync_permutation(self):
        if isinstance(self.invconv, _PermutationAsLU):
            self.invconv.sync(self.actnorm.bias.device)

    def _all_params(self):
        self._sync_permutation()
        inv = [t for t in self.invconv.lu_tensors() if t is not None]
        blk = list(self.block.parameters())
        return [self.actnorm.bias, self.actnorm.logs, *inv, *blk]

    def _consts(self, reverse: bool) -> Fn.StepConsts:
        """Derived tensors for the no-grad path (frozen teacher, sampling): rebuilt only when a parameter changed."""
        def build():
            inv = tuple(None if t is None else t.detach() for t in self.invconv.lu_tensors())
            Wf, bf, sl = Fn.build_affine(self.actnorm.bias.detach(), self.actnorm.logs.detach(), inv,
                                         self.in_channels, reverse, self.is_1d)
            if self.is_1d:
                return Fn.StepConsts(Wf, bf, sl)
            cw = tuple(t.detach() for t in self._coupling_params_2d())
            item, cops = Fn.coupling_operands(cw, self.in_channels, self.hidden_channels, False)
            ops.coupling_prep_batch([item])
            return Fn.StepConsts(Wf, bf, sl, *cops)
        return Fn.cached(self, reverse, build)

    def _check_actnorm_inited(self, input):
        """Reference layers.py:129-133: an ActNorm that was never initialised runs its data-dependent init on the first
        training batch and raises in eval mode. create_glow_model marks every ActNorm initialised (kd_flows.py:155-159),
        so this only matters for a Glow / FlowStep built directly. The step's own ActNorm is initialised from the input
        like the reference; the two ActNorms inside the coupling net would need the statistics of the hidden maps, which
        the fused kernels never materialise: those raise instead of silently running with zero bias / logs."""
        if not self.actnorm.inited:
            self.actnorm.initialize_parameters(input)      # (raises ValueError in eval mode, like the reference)
        if not self.is_1d:
            for blk in (self.block[0], self.block[2]):
                if not blk.actnorm.inited:
                    if not self.training:
                        raise ValueError("In Eval mode, but ActNorm not inited")
                    raise NotImplementedError(
                        "data-dependent ActNorm initialisation inside the fused coupling net is not built; build the "
                        "model with create_glow_model (or call set_actnorm_init()) as the reference pipeline does")

    def _check_supported(self, input):
        _require_cuda(input, "FlowStep")
        self._check_actnorm_inited(input)
        if self.is_1d and self.flow_coupling != "affine":
            raise NotImplementedError("additive coupling is built for the 2-D steps only (every 1-D config is affine)")
        self._sync_permutation()
        if self.is_1d:
            training = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
            wide_ok = not training and self.hidden_channels % 64 == 0      # GEMM path of flow1d._flowstep1d_wide
            if not wide_ok and not ops.flow1d_supported(self.in_channels, self.condition_features,
                                                        self.hidden_channels, training):
                raise NotImplementedError(
                    f"the fused 1-D FlowStep keeps the whole coupling MLP in shared memory; hidden_channels="
                    f"{self.hidden_channels} at D={self.in_channels} does not fit "
                    f"({'training: widths up to 48' if training else 'inference: widths up to 88'}). The tabular "
                    f"configs use 16 / 32. Frozen steps with a width that is a multiple of 64 (conf/teacher/rich.yaml: "
                    f"256) run on the tensor-core GEMM path instead; training them is not built.")
        if not self.is_1d:
            if self.condition_features:
                raise NotImplementedError("y-conditioned 2-D coupling is not built (no shipped image config uses it)")
            if self.hidden_channels % 64 or self.in_channels not in (12, 24, 48, 96):
                raise NotImplementedError("2-D FlowStep kernels need hidden_channels % 64 == 0 and "
                                          "C in {12, 24, 48, 96}")

    def forward(self, input, y_onehot=None, logdet=None, reverse=False):
        self._check_supported(input)
        if self.is_1d:
            from .. import flow1d
            return flow1d.flowstep1d(self, input, y_onehot, logdet, reverse)
        B = input.shape[0]
        ld = _as_logdet(logdet, B, input.device)
        want_ld = ld is not None
        if ld is None:
            ld = torch.zeros(B, device=input.device)
        params = self._all_params()
        needs_grad = torch.is_grad_enabled() and (input.requires_grad or ld.requires_grad
                                                  or any(p.requires_grad for p in params))
        if self.precision == "bf16x3":
            return self._forward_precise(input, ld, want_ld, reverse, needs_grad)
        if not reverse:
            if needs_grad:
                pctx, idx, token = Fn.prep_for(self, False)
                z, ld_out = Fn.FlowStep2dFn.apply(input, ld, self.hidden_channels, token, pctx, idx)
            else:
                z, ld_out, _ = Fn.flowstep2d_forward(input.contiguous(), ld.contiguous(), self._consts(False),
                                                     self.hidden_channels, keep=False)
        else:
            if needs_grad:
                # the perceptual term's gradient reaches the student through its inverse pass (pl_module.py:229-243)
                pctx, idx, token = Fn.prep_for(self, True)
                z, ld_out = Fn.FlowStep2dReverseFn.apply(input, ld, self.hidden_channels, token, pctx, idx)
            else:
                z, ld_out = Fn.flowstep2d_reverse(input.contiguous(), ld.contiguous(), self._consts(True),
                                                  self.hidden_channels)
        return z, (ld_out if want_ld else None)

    def _forward_precise(self, input, ld, want_ld, reverse, needs_grad):
        """fp32-class mode (precise.py): split-bf16 products on the same tensor-core tiles. Additive steps run the
        affine arithmetic with the pinned logit rows of _coupling_params_2d, as in the bf16 mode."""
        from .. import precise
        with torch.set_grad_enabled(needs_grad):
            if not reverse:
                z, ld_out = precise.FlowStep2dX3Fn.apply(input, ld, self.hidden_channels, *precise.folded_params(self))
            elif needs_grad:
                # the perceptual term's gradient reaches the student through its inverse pass (pl_module.py:229-243);
                # the inverse-direction affine and its chain rule come from the batched prep, as in the bf16 mode
                pctx, idx, token = Fn.prep_for(self, True)
                z, ld_out = precise.FlowStep2dReverseX3Fn.apply(input, ld, self.hidden_channels, token, pctx, idx,
                                                                *precise.folded_coupling(self))
            else:
                k = self._consts(True)
                z, ld_out = precise.flowstep2d_reverse_x3(input.contiguous(), ld.contiguous(), self.hidden_channels,
                                                          (k.Wf, k.bf, k.sl), *precise.folded_coupling(self))
        return z, (ld_out if want_ld else None)

    def normal_flow(self, input, y_onehot, logdet):
        return self.forward(input, y_onehot=y_onehot, logdet=logdet, reverse=False)

    def reverse_flow(self, input, y_onehot, logdet):
        return self.forward(input, y_onehot=y_onehot, logdet=logdet, reverse=True)


class FlowNet(nn.Module):
    """[Squeeze, K x FlowStep, Split2d] x (L-1) + [Squeeze, K x FlowStep] (flows.py:205-295)."""

    def __init__(self, image_shape, hidden_channels, K, L, actnorm_scale, flow_permutation, flow_coupling,
                 LU_decomposed, is_1d=False, condition_features=0):
        super().__init__()
        self.is_1d = is_1d
        self.layers = nn.ModuleList()
        self.output_shapes = []
        self.K = K
        self.L = L
        if not is_1d:
            H, W, C = image_shape
        else:
            C = image_shape[0]
        for i in range(L):
            if not is_1d:
                C, H, W = C * 4, H // 2, W // 2
                self.layers.append(SqueezeLayer(factor=2))
                self.output_shapes.append([-1, C, H, W])
            for _ in range(K):
                self.layers.append(FlowStep(in_channels=C, hidden_channels=hidden_channels,
                                            actnorm_scale=actnorm_scale, flow_permutation=flow_permutation,
                                            flow_coupling=flow_coupling, LU_decomposed=LU_decomposed, is_1d=is_1d,
                                            condition_features=condition_features))
                self.output_shapes.append([-1, C] if is_1d else [-1, C, H, W])
            if i < L - 1 and not is_1d:
                self.layers.append(Split2d(num_channels=C))
                self.output_shapes.append([-1, C // 2, H, W])
                C = C // 2

    def forward(self, input, y_onehot=None, logdet=0.0, reverse=False, temperature=None, _sq0=None):
        if reverse:
            return self.decode(input, y_onehot=y_onehot, temperature=temperature)
        return self.encode(input, y_onehot=y_onehot, logdet=logdet, _sq0=_sq0)

    def _encode_layers(self, z, y_onehot, logdet, sq0=None):
        """Generator over (layer output, logdet) in layer order. Squeezes are folded into their neighbours: the first
        one arrives precomputed from the dequantisation kernel (`sq0`), a SqueezeLayer(2) after a Split2d is produced
        by the Split2d kernel itself (layers.py:32-44 as an index map, no permute/contiguous pass)."""
        layers = self.layers
        i, n = 0, len(layers)
        while i < n:
            layer = layers[i]
            if i == 0 and sq0 is not None and isinstance(layer, SqueezeLayer) and layer.factor == 2:
                z = sq0
                yield z, logdet
                i += 1
                continue
            nxt = layers[i + 1] if i + 1 < n else None
            if (isinstance(layer, Split2d) and isinstance(nxt, SqueezeLayer) and nxt.factor == 2
                    and z.shape[2] % 2 == 0 and z.shape[3] % 2 == 0):
                z1, z, logdet = layer.forward_with_squeeze(z, logdet=logdet)
                yield z1, logdet
                yield z, logdet
                i += 2
                continue
            z, logdet = layer(z, y_onehot=y_onehot, logdet=logdet, reverse=False)
            yield z, logdet
            i += 1

    def encode(self, z, y_onehot=None, logdet=0.0, _sq0=None):
        with Fn.use_prep(Fn.prepare_steps(self.layers, False)):   # one K0 launch for every trainable step
            for z, logdet in self._encode_layers(z, y_onehot, logdet, _sq0):
                pass
        return z, logdet

    def decode(self, z, y_onehot=None, temperature=None):
        with Fn.use_prep(Fn.prepare_steps(self.layers, True)):
            for layer in reversed(self.layers):
                if isinstance(layer, Split2d):
                    z, _ = layer(z, logdet=0, reverse=True, temperature=temperature)
                else:
                    z, _ = layer(z, y_onehot=y_onehot, logdet=0, reverse=True)
        return z


class Glow(nn.Module):
    """Flow + prior + bits/dim objective (flows.py:298-438)."""

    def __init__(self, image_shape, hidden_channels, K, L, actnorm_scale, flow_permutation, flow_coupling,
                 LU_decomposed, y_classes, learn_top, y_condition, is_1d=False):
        super().__init__()
        self.flow = FlowNet(image_shape=image_shape, hidden_channels=hidden_channels, K=K, L=L,
                            actnorm_scale=actnorm_scale, flow_permutation=flow_permutation,
                            flow_coupling=flow_coupling, LU_decomposed=LU_decomposed, is_1d=is_1d,
                            condition_features=y_classes if y_condition else 0)
        self.is_1d = is_1d
        self.y_classes = y_classes
        self.y_condition = y_condition
        self.learn_top = learn_top
        if learn_top:
            C = self.flow.output_shapes[-1][1]
            self.learn_top_fn = LinearZeros(C * 2, C * 2) if is_1d else Conv2dZeros(C * 2, C * 2)
        if y_condition:
            C = self.flow.output_shapes[-1][1]
            self.project_ycond = LinearZeros(y_classes, 2 * C)
            self.project_class = LinearZeros(C, y_classes)
        last = self.flow.output_shapes[-1]
        self.register_buffer("prior_h", torch.zeros([1, last[1] * 2] + ([] if is_1d else [last[2], last[3]])))

    def prior(self, data, y_onehot=None):
        """(mean, logs) of the top-level Gaussian (flows.py:367-391); batch 32 when neither data nor y is given."""
        if data is not None:
            batch = data.shape[0]
        else:
            batch = y_onehot.size(0) if y_onehot is not None else 32
        h = self.prior_h.repeat(batch, *([1] * (self.prior_h.dim() - 1)))
        channels = h.size(1)
        if self.learn_top:
            if self.is_1d:
                h = self.learn_top_fn(h)
            else:
                # Conv2dZeros over the prior buffer (flows.py:344-352). The buffer is all zeros (it is created as zeros
                # and nothing ever writes it), so every tap of the 3x3 conv multiplies zero and what is left is one
                # constant per channel, (0 + bias) * exp(3 * logs): parameter-space arithmetic, no kernel.
                if self._prior_h_nonzero():
                    raise NotImplementedError("learn_top over a non-zero prior_h buffer is not built")
                f = self.learn_top_fn
                row = f.conv.bias * torch.exp(f.logs.view(-1) * f.logscale_factor)
                h = h + row.view(1, channels, 1, 1)
        if self.y_condition:
            assert y_onehot is not None
            yp = self.project_ycond(y_onehot)
            h = h + yp.view(h.shape[0], channels, *([1] * (h.dim() - 2)))
        return split_feature(h, "split")

    def _prior_h_nonzero(self):
        key = (self.prior_h.data_ptr(), self.prior_h._version)
        if getattr(self, "_ph_key", None) != key:
            self._ph_key, self._ph_nonzero = key, bool((self.prior_h != 0).any())
        return self._ph_nonzero

    def _prior_rows(self):
        """Batch-independent (mean, logs) rows when the prior is the fixed buffer (all shipped non-RICH configs)."""
        if self.learn_top or self.y_condition:
            return None
        h = self.prior_h
        c = h.shape[1] // 2
        return h[0, :c].contiguous().view(-1), h[0, c:].contiguous().view(-1)

    def forward(self, x=None, y_onehot=None, z=None, temperature=None, reverse=False):
        if reverse:
            return self.reverse_flow(z, y_onehot, temperature)
        return self.normal_flow(x, y_onehot)

    def _objective(self, x, z_last, logdet, y_onehot):
        """bpd = -(logdet + log p(z)) / (ln2 * CHW) in 2-D, nats in 1-D — one fused reduction kernel."""
        scale = 1.0 if self.is_1d else 1.0 / (math.log(2.0) * x.shape[1] * x.shape[2] * x.shape[3])
        rows = self._prior_rows()
        if rows is not None:
            return Fn.PriorBpdFn.apply(z_last, logdet, rows[0], rows[1], scale)
        mean, logs = self.prior(x, y_onehot)
        return -(logdet + gaussian_likelihood(mean, logs, z_last)) * scale

    def normal_flow(self, x, y_onehot=None):
        _require_cuda(x, "Glow")
        sq0 = None
        if self.is_1d:
            logdet = torch.zeros(x.shape[0], device=x.device, dtype=torch.float32)
        elif can_fuse_dequant_squeeze(x):
            x, logdet, sq0 = dequantize_and_squeeze(x)
        else:
            x, logdet = uniform_binning_correction(x)
        z, logdet = self.flow(x, y_onehot=y_onehot, logdet=logdet, reverse=False, _sq0=sq0)
        bpd = self._objective(x, z, logdet, y_onehot)
        y_logits = self.project_class(z.mean(2).mean(2)) if self.y_condition else None
        return z, bpd, y_logits

    def reverse_flow(self, z, y_onehot, temperature):
        if z is None:
            mean, logs = self.prior(z, y_onehot)
            z = gaussian_sample(mean, logs, temperature)
        return self.flow(z, y_onehot=y_onehot, temperature=temperature, reverse=True)

    def set_actnorm_init(self):
        for _, module in self.named_modules():
            if isinstance(module, (ActNorm2d, ActNorm1d)):
                module.inited = True

    def set_precision(self, precision: str):
        """Arithmetic of the 2-D coupling-net GEMMs: "bf16" (default: bf16 operands, fp32 accumulation) or "bf16x3"
        (fp32-class: every operand split hi + lo, three partial products; ~3x the tensor-core work). Everything else
        (z path, log-dets, Split2d, prior, losses, the whole 1-D path) is fp32 in both."""
        if precision not in ("bf16", "bf16x3"):
            raise ValueError("precision must be 'bf16' or 'bf16x3'")
        for layer in self.flow.layers:
            if isinstance(layer, FlowStep):
                layer.precision = precision
        return self
