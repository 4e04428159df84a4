"""TEST INFRASTRUCTURE ONLY — CPU restatement of the reference flow hot path (vklyukin/nf_distillation).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this file.
The product (nf_distillation_b200/) never does; it fails loudly if libnfk.so is missing.

What it is: a functional (no nn.Module), dtype-generic restatement of the reference's Glow / 1-D Glow forward,
inverse, log-det and KD-loss arithmetic, driven directly by a reference-format ``state_dict``. It runs on the
CPU in fp32 or fp64 with torch tensor ops. Every function cites the reference lines it follows.

Pinning: the reference ships no tests or golden vectors (SURVEY.md §4), so this oracle is pinned against outputs
of the UNMODIFIED reference code executed in the build container: oracle/make_golden.py imports
/root/reference/models, runs it on seeded inputs/weights and commits the vectors under tests/golden/;
tests/test_oracle_golden.py checks this file against them (and against the live reference when it is present).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
SD = Dict[str, Tensor]
LOG2PI = math.log(2.0 * math.pi)


# ------------------------------------------------------------------------------------------ bf16-operand mode
# The CUDA path runs the three convolutions of the 2-D coupling network (models/flows.py:25-34) on the tensor cores with
# bf16 OPERANDS and fp32 accumulation; everything else (z path, log-dets, Split2d, prior, losses) is fp32. With
# `bf16_operands()` active this oracle rounds exactly the same tensors at exactly the same places, so that a CUDA-vs-
# oracle difference that remains is summation order (1e-6), not operand rounding:
#   forward   conv inputs (z1, h1, h2) and the folded weights w*exp(logs) / w*exp(3 logs) are rounded to bf16, the biases
#             b*exp(logs) and all sums stay fp32, h1 / h2 are stored as bf16;
#   backward  (autograd) the gradients that the CUDA backward stores as bf16 GEMM operands are rounded too: d(pre2),
#             d(pre1) (after the ReLU mask) and the gradient of the Conv2dZeros output taps; weight / bias gradients and
#             the gradient of z1 are fp32 sums of those products.
# The default (flag off) is the reference's plain fp32 arithmetic; the fp32 bounds of the tests are stated against that.
_BF16 = {"on": False}


class bf16_operands:
    """Context manager: `with bf16_operands(): glow_forward(...)`."""

    def __init__(self, on: bool = True):
        self.on = on

    def __enter__(self):
        self.prev, _BF16["on"] = _BF16["on"], self.on
        return self

    def __exit__(self, *exc):
        _BF16["on"] = self.prev
        return False


class _Round(torch.autograd.Function):
    """Round to the nearest bf16 (kept in the tensor's own dtype) in the forward and / or the backward direction."""

    @staticmethod
    def forward(ctx, x, fwd, bwd):
        ctx.bwd = bwd
        return x.to(torch.bfloat16).to(x.dtype) if fwd else x.clone()

    @staticmethod
    def backward(ctx, g):
        return (g.to(torch.bfloat16).to(g.dtype) if ctx.bwd else g), None, None


def _q(x: Tensor, fwd: bool = True, bwd: bool = False) -> Tensor:
    return _Round.apply(x, fwd, bwd) if _BF16["on"] else x


# ------------------------------------------------------------------------------------------ model topology
def layer_plan(cfg: dict) -> List[Tuple[str, int, int, int]]:
    """List of (kind, C_in, H, W) in execution order, kind in {squeeze, step, split}.

    Follows FlowNet.__init__ (models/flows.py:234-269): per level [Squeeze, K x FlowStep, Split2d (not last)];
    the 1-D variant has no squeeze / split and image_shape = [D]."""
    plan = []
    if cfg.get("is_1d", False):
        C = cfg["image_shape"][0]
        for _ in range(cfg["L"] * cfg["K"]):
            plan.append(("step", C, 1, 1))
        return plan
    H, W, C = cfg["image_shape"]
    for lvl in range(cfg["L"]):
        plan.append(("squeeze", C, H, W))
        C, H, W = C * 4, H // 2, W // 2
        for _ in range(cfg["K"]):
            plan.append(("step", C, H, W))
        if lvl < cfg["L"] - 1:
            plan.append(("split", C, H, W))
            C //= 2
    return plan


# ------------------------------------------------------------------------------------------ primitive ops
def squeeze2d(x: Tensor) -> Tensor:
    """Space-to-depth x2, output channel = c*4 + fh*2 + fw (models/layers.py:32-44)."""
    B, C, H, W = x.shape
    x = x.reshape(B, C, H // 2, 2, W // 2, 2).permute(0, 1, 3, 5, 2, 4)
    return x.reshape(B, C * 4, H // 2, W // 2)


def unsqueeze2d(x: Tensor) -> Tensor:
    """Inverse of squeeze2d (models/layers.py:47-61)."""
    B, C, H, W = x.shape
    x = x.reshape(B, C // 4, 2, 2, H, W).permute(0, 1, 4, 2, 5, 3)
    return x.reshape(B, C // 4, H * 2, W * 2)


def gaussian_logp(mean: Tensor, logs: Tensor, x: Tensor) -> Tensor:
    """Per-sample diagonal-Gaussian log density (models/layers.py:10-23)."""
    lp = -0.5 * (2.0 * logs + (x - mean) ** 2 * torch.exp(-2.0 * logs) + LOG2PI)
    return lp.flatten(1).sum(1)


def actnorm(x: Tensor, bias: Tensor, logs: Tensor, logdet, reverse: bool) -> Tuple[Tensor, Optional[Tensor]]:
    """(x + b) * exp(logs) forward, x * exp(-logs) - b reverse; logdet +- pixels * sum(logs)
    (models/layers.py:101-142)."""
    pixels = 1 if x.dim() == 2 else x.shape[2] * x.shape[3]
    if reverse:
        y = x * torch.exp(-logs) - bias
    else:
        y = (x + bias) * torch.exp(logs)
    if logdet is not None:
        d = logs.sum() * pixels
        logdet = logdet - d if reverse else logdet + d
    return y, logdet


def invconv_matrix(sd: SD, pre: str, reverse: bool) -> Tuple[Tensor, Tensor]:
    """W = P (L o tril + I) (U o triu + diag(sign_s exp(log_s))), log|det W| = sum(log_s); the reverse uses
    U^-1 L^-1 P^-1 (models/layers.py:376-397). The non-LU branch (:366-375) uses slogdet / inverse."""
    if pre + "weight" in sd:
        w = sd[pre + "weight"]
        ld = torch.slogdet(w)[1]
        return (torch.inverse(w) if reverse else w), ld
    lower, upper, log_s = sd[pre + "lower"], sd[pre + "upper"], sd[pre + "log_s"]
    p, sign_s = sd[pre + "p"].to(lower.dtype), sd[pre + "sign_s"].to(lower.dtype)
    C = lower.shape[0]
    eye = torch.eye(C, dtype=lower.dtype)
    Lm = torch.tril(lower, -1) + eye
    Um = torch.triu(upper, 1) + torch.diag(sign_s * torch.exp(log_s))
    if reverse:
        w = torch.inverse(Um) @ (torch.inverse(Lm) @ torch.inverse(p))
    else:
        w = p @ (Lm @ Um)
    return w, log_s.sum()


def invconv(x: Tensor, sd: SD, pre: str, logdet, reverse: bool) -> Tuple[Tensor, Optional[Tensor]]:
    """2-D: z[b,o,h,w] = sum_i W[o,i] x[b,i,h,w]; 1-D: z = x @ W (models/layers.py:404-421)."""
    w, ld = invconv_matrix(sd, pre, reverse)
    if x.dim() == 2:
        z, pixels = x @ w, 1
    else:
        z, pixels = torch.einsum("oi,bihw->bohw", w, x), x.shape[2] * x.shape[3]
    if logdet is not None:
        logdet = logdet - ld * pixels if reverse else logdet + ld * pixels
    return z, logdet


def conv_actnorm(x: Tensor, sd: SD, pre: str) -> Tensor:
    """Conv2d: zero-pad 'same' -> bias-free conv -> ActNorm affine (models/layers.py:190-228)."""
    w = sd[pre + "conv.weight"]
    if _BF16["on"]:   # folded operand bf16(w * exp(logs)) and fp32 bias b * exp(logs) (prep.cu coupling_prep_kernel)
        e = torch.exp(sd[pre + "actnorm.logs"])                      # [1, Cout, 1, 1]
        wf = _q(w * e.view(-1, 1, 1, 1))
        y = F.conv2d(_q(x), wf, padding=(w.shape[2] // 2, w.shape[3] // 2))
        return y + sd[pre + "actnorm.bias"] * e
    y = F.conv2d(x, w, padding=(w.shape[2] // 2, w.shape[3] // 2))
    return (y + sd[pre + "actnorm.bias"]) * torch.exp(sd[pre + "actnorm.logs"])


def conv_zeros(x: Tensor, sd: SD, pre: str, bf16: bool = False) -> Tensor:
    """Conv2dZeros: zero-pad -> conv3x3 + bias -> * exp(3 * logs) (models/layers.py:231-260)."""
    w = sd[pre + "conv.weight"]
    if _BF16["on"] and bf16:
        e = torch.exp(sd[pre + "logs"] * 3.0)                        # [Cout, 1, 1]
        y = F.conv2d(_q(x), _q(w * e.view(-1, 1, 1, 1)), padding=(w.shape[2] // 2, w.shape[3] // 2))
        # the per-tap products leave the tensor cores in fp32; their GRADIENT is a bf16 dgrad / wgrad operand
        return _q(y, fwd=False, bwd=True) + (sd[pre + "conv.bias"] * e.view(-1)).view(1, -1, 1, 1)
    y = F.conv2d(x, w, sd[pre + "conv.bias"], padding=(w.shape[2] // 2, w.shape[3] // 2))
    return y * torch.exp(sd[pre + "logs"] * 3.0)


def coupling_net(x: Tensor, sd: SD, pre: str) -> Tensor:
    """get_block_2d (models/flows.py:25-34) or get_block_1d (:37-52), chosen by tensor rank."""
    if x.dim() == 4:
        # (bf16 mode: h1 / h2 are stored as bf16 and their pre-activation gradients are bf16 operands of the backward)
        h = _q(torch.relu(conv_actnorm(x, sd, pre + "0.")), bwd=True)
        h = _q(torch.relu(conv_actnorm(h, sd, pre + "2.")), bwd=True)
        return conv_zeros(h, sd, pre + "4.", bf16=True)
    h = x
    for i, act in zip((0, 2, 4, 6, 8, 10), ("relu", "relu", "relu", "relu", "tanh", None)):
        h = F.linear(h, sd[f"{pre}{i}.weight"], sd[f"{pre}{i}.bias"])
        if act == "relu":
            h = torch.relu(h)
        elif act == "tanh":
            h = torch.tanh(h)
    return h


def permute(x: Tensor, perm: Tensor, reverse: bool) -> Tensor:
    """Permute2d (models/layers.py:263-290): forward input[:, indices], reverse input[:, indices_inverse]; no log-det."""
    perm = torch.as_tensor(perm, dtype=torch.long)
    if reverse:
        inv = torch.empty_like(perm)
        inv[perm] = torch.arange(perm.numel())
        perm = inv
    return x[:, perm]


def flowstep(x: Tensor, sd: SD, pre: str, logdet: Tensor, reverse: bool, y_onehot=None,
             coupling: str = "affine", perm=None) -> Tuple[Tensor, Tensor]:
    """FlowStep.normal_flow / reverse_flow (models/flows.py:142-202): actnorm -> invconv (or, with `perm` = the
    step's Permute2d.indices, the fixed shuffle / reverse permutation, flows.py:85-95) -> coupling, where the affine
    coupling is z2 = (z2 + shift) * sigmoid(s + 2) with shift = h[:,0::2], s = h[:,1::2] and the additive one is
    z2 = z2 + h (flows.py:157-158)."""
    red = lambda t: t.flatten(1).sum(1)
    if not reverse:
        z, logdet = actnorm(x, sd[pre + "actnorm.bias"], sd[pre + "actnorm.logs"], logdet, False)
        if perm is None:
            z, logdet = invconv(z, sd, pre + "invconv.", logdet, False)
        else:
            z = permute(z, perm, False)
    else:
        z = x
    c1 = z.shape[1] // 2
    z1, z2 = z[:, :c1], z[:, c1:]
    arg = z1 if y_onehot is None else torch.cat((z1, y_onehot), 1)
    h = coupling_net(arg, sd, pre + "block.")
    if coupling == "additive":
        z2 = z2 - h if reverse else z2 + h
    else:
        shift, scale = h[:, 0::2], torch.sigmoid(h[:, 1::2] + 2.0)
        if reverse:
            z2 = z2 / scale - shift
            logdet = logdet - red(torch.log(scale))
        else:
            z2 = (z2 + shift) * scale
            logdet = logdet + red(torch.log(scale))
    z = torch.cat((z1, z2), 1)
    if reverse:
        if perm is None:
            z, logdet = invconv(z, sd, pre + "invconv.", logdet, True)
        else:
            z = permute(z, perm, True)
        z, logdet = actnorm(z, sd[pre + "actnorm.bias"], sd[pre + "actnorm.logs"], logdet, True)
    return z, logdet


def split2d_forward(x: Tensor, sd: SD, pre: str, logdet: Tensor) -> Tuple[Tensor, Tensor]:
    """Split2d forward (models/layers.py:309-313): keep z1, score z2 under N(mean, exp(logs)) predicted from z1
    with mean = h[:,0::2], logs = h[:,1::2]."""
    c1 = x.shape[1] // 2
    z1, z2 = x[:, :c1], x[:, c1:]
    h = conv_zeros(z1, sd, pre + "conv.")
    return z1, logdet + gaussian_logp(h[:, 0::2], h[:, 1::2], z2)


def split2d_reverse(z1: Tensor, sd: SD, pre: str, temperature: float, eps: Optional[Tensor]) -> Tensor:
    """Split2d reverse (models/layers.py:303-308): z2 = mean + exp(logs) * T * eps, eps ~ N(0,1) (eps=None -> 0,
    which equals the reference at temperature 0)."""
    h = conv_zeros(z1, sd, pre + "conv.")
    mean, logs = h[:, 0::2], h[:, 1::2]
    z2 = mean if eps is None else mean + torch.exp(logs) * temperature * eps
    return torch.cat((z1, z2), 1)


# ------------------------------------------------------------------------------------------ whole model
def prior(sd: SD, cfg: dict, batch: int, y_onehot: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """Glow.prior (models/flows.py:367-391): prior_h repeated, through learn_top_fn when learn_top (Conv2dZeros in 2-D,
    LinearZeros in 1-D: models/flows.py:344-352), plus the LinearZeros projection of y_onehot when y_condition
    (models/layers.py:173-187: linear(x) * exp(3 * logs)), split in halves."""
    h = sd["prior_h"]
    h = h.expand(batch, *h.shape[1:])
    if cfg.get("learn_top", False):
        if h.dim() == 4:
            h = conv_zeros(h, sd, "learn_top_fn.")
        else:
            h = torch.nn.functional.linear(h, sd["learn_top_fn.linear.weight"], sd["learn_top_fn.linear.bias"])
            h = h * torch.exp(sd["learn_top_fn.logs"] * 3.0)
    if cfg.get("y_condition", False):
        yp = torch.nn.functional.linear(y_onehot, sd["project_ycond.linear.weight"], sd["project_ycond.linear.bias"])
        yp = yp * torch.exp(sd["project_ycond.logs"] * 3.0)
        h = h + yp.view(batch, h.shape[1], *([1] * (h.dim() - 2)))
    c = h.shape[1] // 2
    return h[:, :c], h[:, c:]


def step_perm(cfg: dict, i: int):
    """Permute2d.indices of layer i for flow_permutation 'shuffle' / 'reverse' (they are plain attributes, not in the
    state_dict, so they travel in cfg["perm_indices"] = {str(layer index): [indices]}); None for 'invconv'."""
    if cfg.get("flow_permutation", "invconv") == "invconv":
        return None
    return cfg["perm_indices"][str(i)]


def glow_forward(sd: SD, cfg: dict, x: Tensor, noise: Optional[Tensor] = None, y_onehot: Optional[Tensor] = None):
    """GlowGetAllOutputs.normal_flow (models/kd_flows.py:121-152): returns (all layer outputs, bpd|nll [B]).

    `noise` is the dequantisation noise U(0, 1/256) the reference draws in uniform_binning_correction
    (models/utils.py:26-41); pass the recorded noise to reproduce a reference run, or None for no noise."""
    B = x.shape[0]
    is_1d = cfg.get("is_1d", False)
    if is_1d:
        logdet = torch.zeros(B, dtype=x.dtype)
        chw = 1
    else:
        chw = x.shape[1] * x.shape[2] * x.shape[3]
        if noise is not None:
            x = x + noise
        logdet = torch.full((B,), -math.log(256.0) * chw, dtype=x.dtype)
    outs = []
    z = x
    for i, (kind, C, H, W) in enumerate(layer_plan(cfg)):
        pre = f"flow.layers.{i}."
        if kind == "squeeze":
            z = squeeze2d(z)
        elif kind == "step":
            z, logdet = flowstep(z, sd, pre, logdet, False, y_onehot=y_onehot if cfg.get("y_condition") else None,
                                 coupling=cfg.get("flow_coupling", "affine"), perm=step_perm(cfg, i))
        else:
            z, logdet = split2d_forward(z, sd, pre, logdet)
        outs.append(z)
    mean, logs = prior(sd, cfg, B, y_onehot)
    objective = logdet + gaussian_logp(mean.to(z.dtype), logs.to(z.dtype), z)
    bpd = -objective if is_1d else -objective / (math.log(2.0) * chw)
    return outs, bpd


def glow_reverse(sd: SD, cfg: dict, z: Tensor, temperature: float = 0.0,
                 eps: Optional[Sequence[Tensor]] = None, y_onehot: Optional[Tensor] = None) -> List[Tensor]:
    """FlowNetGetAllOutputs.decode (models/kd_flows.py:55-73): all outputs of the inverse pass, last = x.
    `eps` supplies the N(0,1) draws of each Split2d in decode order (None -> zeros)."""
    plan = layer_plan(cfg)
    outs = []
    k = 0
    dummy = torch.zeros(z.shape[0], dtype=z.dtype)
    for i in reversed(range(len(plan))):
        kind = plan[i][0]
        pre = f"flow.layers.{i}."
        if kind == "squeeze":
            z = unsqueeze2d(z)
        elif kind == "step":
            z, _ = flowstep(z, sd, pre, dummy, True, y_onehot=y_onehot if cfg.get("y_condition") else None,
                            coupling=cfg.get("flow_coupling", "affine"), perm=step_perm(cfg, i))
        else:
            z = split2d_reverse(z, sd, pre, temperature, None if eps is None else eps[k])
            k += 1
        outs.append(z)
    return outs


# ------------------------------------------------------------------------------------------ KD step
def kd_indices(student_cfg: dict, teacher_cfg: dict) -> Tuple[List[int], List[int]]:
    """NFModel._get_kd_indices (pl_module.py:81-110): squeeze layers, every 2nd (student) / 4th (teacher) layer
    in 1-D, and the last layer."""
    def taps(cfg, every):
        plan = layer_plan(cfg)
        return [i for i, (kind, *_rest) in enumerate(plan)
                if kind == "squeeze" or (student_cfg.get("is_1d", False) and (i + 1) % every == 0)
                or i + 1 == len(plan)]
    return taps(student_cfg, 2), taps(teacher_cfg, 4)


def kd_loss(student_z: Sequence[Tensor], teacher_z: Sequence[Tensor], s_idx, t_idx) -> Tensor:
    """Per-sample mean-over-levels of per-level mean squared error (pl_module.py:266-282)."""
    total = None
    for si, ti in zip(s_idx, t_idx):
        part = ((student_z[si] - teacher_z[ti]) ** 2).flatten(1).mean(1)
        total = part if total is None else total + part
    return total / max(len(s_idx), 1)


def kd_step(student_sd: SD, student_cfg: dict, teacher_sd: SD, teacher_cfg: dict, x: Tensor,
            weights: dict, noise_s: Optional[Tensor] = None, noise_t: Optional[Tensor] = None,
            latent: Optional[Tensor] = None, y_onehot: Optional[Tensor] = None,
            sample_weights: Optional[Tensor] = None) -> dict:
    """NFModel.forward + loss (pl_module.py:198-320). The student adds dequantisation noise to x in place and the
    teacher then adds its own on top (pl_module.py:215-225 + models/utils.py:38), so the teacher sees
    x + noise_s + noise_t. The perceptual term is L1 between reverse passes at temperature 0.7 from `latent`."""
    is_1d = student_cfg.get("is_1d", False)
    xs = x if (is_1d or noise_s is None) else x + noise_s
    s_z, s_nll = glow_forward(student_sd, student_cfg, xs, y_onehot=y_onehot)
    out = {"nll": s_nll}
    s_idx, t_idx = kd_indices(student_cfg, teacher_cfg)
    if weights.get("kd", 0) > 0:
        xt = xs if (is_1d or noise_t is None) else xs + noise_t
        with torch.no_grad():
            t_z, _ = glow_forward(teacher_sd, teacher_cfg, xt, y_onehot=y_onehot)
        out["kd"] = kd_loss(s_z, t_z, s_idx, t_idx)
    else:
        out["kd"] = torch.zeros((), dtype=x.dtype)
    if weights.get("perceptual", 0) > 0:
        sx = glow_reverse(student_sd, student_cfg, latent, 0.7, y_onehot=y_onehot)[-1]
        with torch.no_grad():
            tx = glow_reverse(teacher_sd, teacher_cfg, latent, 0.7, y_onehot=y_onehot)[-1]
        perc = (sx - tx).abs().flatten(1).mean(1)
        out["perceptual"] = torch.where(torch.isnan(perc), torch.zeros_like(perc), perc)
    else:
        out["perceptual"] = torch.zeros((), dtype=x.dtype)
    result = weights.get("nll", 0) * out["nll"] + weights.get("kd", 0) * out["kd"] \
        + weights.get("perceptual", 0) * out["perceptual"]
    if sample_weights is not None:   # RICH: per-sample weights multiply the combined loss (pl_module.py:311-313)
        result = result * sample_weights
    return {"nll": out["nll"].mean(), "kd": out["kd"].mean(), "perceptual": out["perceptual"].mean(),
            "result_loss": result.mean(), "student_z": s_z}


# ------------------------------------------------------------------------------------------ synthetic weights
def random_state_dict(cfg: dict, seed: int, std: float = 0.05) -> SD:
    """A reference-format state_dict with seeded random weights of the reference's shapes, built WITHOUT any model
    class (bench.py's reference arm must not touch the product package): conv weights Xavier-normal like
    models/layers.py:209-214, invconv from the LU factors of a random orthogonal matrix like :336-352, and the
    tensors the reference zero-initialises (ActNorm bias/logs, Conv2dZeros, LinearZeros; SURVEY §0.5) drawn
    N(0, std^2) so that every coupling does real work. Timing input only — parity tests use fixtures / shared dicts."""
    g = torch.Generator().manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g)
    sd: SD = {}
    hid = cfg["hidden_channels"]
    is_1d = cfg.get("is_1d", False)
    cond = cfg["y_classes"] if cfg.get("y_condition", False) else 0
    for i, (kind, C, H, W) in enumerate(layer_plan(cfg)):
        pre = f"flow.layers.{i}."
        if kind == "step":
            shp = [1, C] if is_1d else [1, C, 1, 1]
            sd[pre + "actnorm.bias"], sd[pre + "actnorm.logs"] = rn(*shp) * std, rn(*shp) * std
            q = torch.linalg.qr(rn(C, C))[0]
            p_, lo, up = torch.lu_unpack(*torch.linalg.lu_factor(q))
            s_ = torch.diag(up)
            sd[pre + "invconv.p"], sd[pre + "invconv.sign_s"] = p_, torch.sign(s_)
            sd[pre + "invconv.lower"], sd[pre + "invconv.upper"] = lo, torch.triu(up, 1)
            sd[pre + "invconv.log_s"] = torch.log(torch.abs(s_))
            cin, cout = C // 2 + cond, (C - C // 2) * 2
            if is_1d:
                dims = [cin, hid, hid, hid, hid, hid, cout]
                for j, k in enumerate((0, 2, 4, 6, 8, 10)):
                    bound = 1.0 / math.sqrt(dims[j])
                    sd[f"{pre}block.{k}.weight"] = (torch.rand(dims[j + 1], dims[j], generator=g) * 2 - 1) * bound
                    sd[f"{pre}block.{k}.bias"] = (torch.rand(dims[j + 1], generator=g) * 2 - 1) * bound
            else:
                sd[pre + "block.0.conv.weight"] = rn(hid, cin, 3, 3) * math.sqrt(2.0 / (9 * (cin + hid)))
                sd[pre + "block.2.conv.weight"] = rn(hid, hid, 1, 1) * math.sqrt(2.0 / (2 * hid))
                for k in ("0", "2"):
                    sd[f"{pre}block.{k}.actnorm.bias"] = rn(1, hid, 1, 1) * std
                    sd[f"{pre}block.{k}.actnorm.logs"] = rn(1, hid, 1, 1) * std
                sd[pre + "block.4.conv.weight"] = rn(cout, hid, 3, 3) * std
                sd[pre + "block.4.conv.bias"] = rn(cout) * std
                sd[pre + "block.4.logs"] = rn(cout, 1, 1) * std
        elif kind == "split":
            sd[pre + "conv.conv.weight"] = rn(C, C // 2, 3, 3) * std
            sd[pre + "conv.conv.bias"] = rn(C) * std
            sd[pre + "conv.logs"] = rn(C, 1, 1) * std
    kind, C, H, W = layer_plan(cfg)[-1]
    sd["prior_h"] = torch.zeros([1, 2 * C] + ([] if is_1d else [H, W]))
    return sd
