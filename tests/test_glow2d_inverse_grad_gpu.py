"""Gradients through the 2-D inverse pass (the perceptual L1 term of pl_module.py:229-243,284-299, whose gradient reaches
the student through student(z, T=0.7, reverse=True)).

Oracle comparisons follow test_headline_parity_gpu.py: the CUDA path against oracle/glow_oracle.py with
`bf16_operands()` (the same tensors rounded at the same places), relative to max|.| of the compared tensor, and against
the plain fp32 oracle with the looser fp32 bounds.

The reference's Split2d samples z2 with torch.normal, whose derivative with respect to mean and std is zero (pinned by
the CPU test below). The oracle's split2d_reverse writes the sample as mean + exp(logs) * T * eps, which does carry a
gradient, so the inverse passes here use `glow_reverse_sampled`: the oracle's own layers with that sample detached.
"""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
dev = "cuda"

BOUND_OUT_BF16 = 2e-3      # CUDA vs bf16-operand oracle, relative to max|.|
BOUND_GRAD_BF16 = 6e-2
BOUND_OUT_F32 = 1e-2       # CUDA (bf16 operands) vs fp32 oracle
BOUND_LOGDET = 5e-4        # single step, relative to max|logdet| of that step


def rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-12)).item()


def images(B, H, g):
    return torch.floor(torch.rand(B, 3, H, H, generator=g) * 256) / 256 - 0.5


# ------------------------------------------------------------------------------------------------ oracle helpers
def split2d_reverse_sampled(z1, sd, pre, temperature, eps):
    """The reference's Split2d reverse under autograd: z2 = torch.normal(mean, exp(logs) * T) is a constant."""
    from oracle import glow_oracle as O
    h = O.conv_zeros(z1, sd, pre + "conv.")
    z2 = (h[:, 0::2] + torch.exp(h[:, 1::2]) * temperature * eps).detach()
    return torch.cat((z1, z2), 1)


def glow_reverse_sampled(sd, cfg, z, temperature, eps):
    """O.glow_reverse with the Split2d draws `eps` (decode order) taken as constants, like torch.normal's."""
    from oracle import glow_oracle as O
    plan = O.layer_plan(cfg)
    dummy = torch.zeros(z.shape[0], dtype=z.dtype)
    k = 0
    for i in reversed(range(len(plan))):
        kind, pre = plan[i][0], f"flow.layers.{i}."
        if kind == "squeeze":
            z = O.unsqueeze2d(z)
        elif kind == "step":
            z, _ = O.flowstep(z, sd, pre, dummy, True, coupling=cfg.get("flow_coupling", "affine"),
                              perm=O.step_perm(cfg, i))
        else:
            z = split2d_reverse_sampled(z, sd, pre, temperature, eps[k])
            k += 1
    return z


# ------------------------------------------------------------------------------------------------ one FlowStep
def make_step(C, hid, seed, coupling="affine", permutation="invconv", lu=True):
    from nf_distillation_b200.models.flows import FlowStep
    torch.manual_seed(seed)
    st = FlowStep(in_channels=C, hidden_channels=hid, actnorm_scale=1.0, flow_permutation=permutation,
                  flow_coupling=coupling, LU_decomposed=lu)
    for m in st.modules():
        if hasattr(m, "inited"):
            m.inited = True
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for p in st.parameters():
            if p.abs().max() == 0:
                p.copy_(torch.randn(p.shape, generator=g) * 0.05)
    sd = {k: v.clone() for k, v in st.state_dict().items()}
    perm = None if permutation == "invconv" else getattr(st, permutation).indices.clone()
    return st, sd, perm


def check_inverse_step(C, H, B, hid, seed, coupling="affine", permutation="invconv", lu=True):
    """Runs one FlowStep's inverse with grad on the GPU and through the oracle's autograd; returns the measured errors
    (vs the bf16-operand oracle) after asserting the bounds."""
    from oracle import glow_oracle as O
    st, sd, perm = make_step(C, hid, seed, coupling, permutation, lu)
    names = dict(st.named_parameters())
    g = torch.Generator().manual_seed(seed + 7)
    z = torch.randn(B, C, H, H, generator=g)
    ld0 = torch.randn(B, generator=g)
    wx, wl = torch.randn(B, C, H, H, generator=g), torch.randn(B, generator=g)

    def oracle(bf16):
        osd = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in sd.items()}
        zo, lo = z.clone().requires_grad_(True), ld0.clone().requires_grad_(True)
        with O.bf16_operands(bf16):
            x, ld = O.flowstep(zo, osd, "", lo, True, coupling=coupling, perm=perm)
            ((x * wx).sum() + (ld * wl).sum()).backward()
        return x.detach(), ld.detach(), zo.grad, lo.grad, {k: osd[k].grad for k in names}

    x32, ld32, dz32, _, g32 = oracle(False)
    x16, ld16, dz16, dld16, g16 = oracle(True)
    st = st.to(dev)
    with torch.no_grad():
        xi, ldi = st(z.to(dev), logdet=ld0.to(dev), reverse=True)
    zg, lg = z.to(dev).requires_grad_(True), ld0.to(dev).requires_grad_(True)
    xt, ldt = st(zg, logdet=lg, reverse=True)
    assert torch.equal(xt.detach(), xi), "training and inference inverse kernels must agree bit for bit"
    assert rel(ldt, ldi) < 1e-6      # (per-sample log-det partial sums meet in fp32 atomics: order is not fixed)
    ((xt * wx.to(dev)).sum() + (ldt * wl.to(dev)).sum()).backward()
    errs = {"x": rel(xt, x16), "ld": rel(ldt, ld16), "dz": rel(zg.grad, dz16)}
    assert errs["x"] < BOUND_OUT_BF16 and rel(xt, x32) < BOUND_OUT_F32, (errs, rel(xt, x32))
    assert errs["ld"] < BOUND_LOGDET and rel(ldt, ld32) < BOUND_LOGDET, (errs, rel(ldt, ld32))
    assert torch.equal(lg.grad.cpu(), dld16) and torch.equal(lg.grad.cpu(), wl)   # the log-det passes straight through
    assert errs["dz"] < BOUND_GRAD_BF16 and rel(zg.grad, dz32) < 0.1, (errs, rel(zg.grad, dz32))
    worst32 = 0.0
    for n_, p in st.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), n_
        e16, e32 = rel(p.grad, g16[n_]), rel(p.grad, g32[n_])
        errs[n_] = e16
        assert e16 < BOUND_GRAD_BF16, (n_, e16, e32)
        worst32 = max(worst32, e32)
    assert worst32 < 0.2, worst32     # (measured 0.11 / 0.12 at C=48 H=8 and C=96 H=4, below 0.1 elsewhere)
    print(f"\nC={C} H={H} B={B} hid={hid} {coupling}/{permutation}/lu={lu}: "
          + " ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("C,H,B,hid", [
    (12, 16, 40, 512),    # pconv_coupling<12>, fused conv kernels (M = 10240)
    (12, 16, 9, 64),      # pconv_coupling<12>, two GEMMs, ragged B
    (12, 32, 6, 64),      # 32x32 maps: banded coupling and banded coupling_inv_bwd
    (24, 8, 136, 512),    # pconv_coupling<24>, fused conv kernels (M = 8704)
    (48, 4, 520, 512),    # pconv_px<48>, fused conv kernels (M = 8320)
    (48, 8, 37, 256),     # per-tap GEMM + coupling_fwd fallback, ragged B
    (96, 4, 33, 64),      # pconv_px<96>
])
def test_flowstep_inverse_pass_gradients_match_oracle(C, H, B, hid):
    """One FlowStep's inverse pass with grad (FlowStep2dReverseFn: affine1x1_bwd without col2im -> coupling_inv_bwd ->
    the coupling net's backward -> col2im_add, then the batched inverse chain rule of the fused affine): x, log-det,
    the input gradient, the log-det gradient and every parameter gradient against the oracle's autograd through
    O.flowstep(reverse=True); the inference-mode inverse is bit-identical to the training-mode one.
    Measured vs the bf16-operand oracle: x 4e-7..2.1e-4, log-det 9e-8..1.6e-5, dz 2e-4..1.6e-2, parameter gradients
    <= 3.2e-2 (block.2.conv.weight, C=48 H=8), <= 9e-5 on the ActNorm / invconv tensors. Against the fp32 oracle the
    worst parameter gradient is 0.11-0.12 at C=48 H=8 and C=96 H=4 (bf16 operands through 1/s), below 0.1 elsewhere."""
    check_inverse_step(C, H, B, hid, 300 + C + H)


@pytest.mark.gpu
@pytest.mark.parametrize("coupling,permutation,lu", [
    ("additive", "invconv", True),
    ("affine", "shuffle", True),
    ("affine", "reverse", True),
    ("affine", "invconv", False),
])
def test_flowstep_inverse_pass_gradients_of_the_variants(coupling, permutation, lu):
    """Additive coupling (the affine kernels with the scale pinned to 1), the fixed shuffle / reverse permutations and
    the plain invconv weight (LU_decomposed=False), each against the oracle. Measured vs the bf16-operand oracle: x and
    log-det <= 6e-5, dz <= 3.4e-4, parameter gradients <= 5.3e-4."""
    check_inverse_step(12, 8, 24, 64, 500, coupling, permutation, lu)


# ------------------------------------------------------------------------------------------------ Split2d reverse
def test_torch_normal_has_zero_gradient_wrt_mean_and_std():
    """The semantics Split2dReverseFn follows: in torch, d normal(mean, std) / d(mean, std) = 0."""
    g = torch.Generator().manual_seed(0)
    mean = torch.randn(4, 5, generator=g).requires_grad_(True)
    std = (torch.rand(4, 5, generator=g) + 0.5).requires_grad_(True)
    out = torch.normal(mean, std, generator=g)
    (out * torch.randn(4, 5, generator=g)).sum().backward()
    for t_ in (mean, std):
        assert t_.grad is None or not t_.grad.any()


@pytest.mark.gpu
def test_split2d_reverse_passes_the_z1_half_and_gives_its_parameters_nothing():
    from nf_distillation_b200.models.layers import Split2d
    torch.manual_seed(3)
    sp = Split2d(num_channels=24).to(dev)
    with torch.no_grad():
        for p in sp.parameters():
            p.copy_(torch.randn_like(p) * 0.05)
    z1 = torch.randn(5, 12, 8, 8, device=dev).requires_grad_(True)
    out, _ = sp(z1, logdet=0, reverse=True, temperature=0.7)
    assert out.shape == (5, 24, 8, 8) and out.requires_grad
    assert torch.equal(out[:, :12].detach(), z1.detach())
    w = torch.randn_like(out)
    (out * w).sum().backward()
    assert torch.equal(z1.grad, w[:, :12])
    for p in sp.parameters():
        assert p.grad is None or not p.grad.any()


# ------------------------------------------------------------------------------------------------ the KD step
def kd_pair(perceptual, seed=0):
    from nf_distillation_b200.pl_module import NFModel
    from nf_distillation_b200.train import glow_cfg, kd_config, randomise_zero_params
    s_cfg, t_cfg = glow_cfg((32, 32, 3), 2, 3, 64), glow_cfg((32, 32, 3), 3, 3, 64)
    torch.manual_seed(seed)
    m = NFModel(kd_config(s_cfg, t_cfg, nll=0.9, kd=0.1, perceptual=perceptual))
    # std 0.01: with 0.05 the inverse passes of these untrained models reach |x| ~ 1e4 at T = 0.7, where a single
    # bf16 rounding of a coupling-net operand is amplified step after step and no two implementations agree
    randomise_zero_params(m.student, seed + 1, 0.01)
    randomise_zero_params(m.teacher, seed + 2, 0.01)
    s_sd = {k: v.clone() for k, v in m.student.state_dict().items()}
    t_sd = {k: v.clone() for k, v in m.teacher.state_dict().items()}
    return m, s_cfg, t_cfg, s_sd, t_sd


def oracle_kd(s_sd, s_cfg, t_sd, t_cfg, x, n1, n2, latent, eps_s, eps_t, w_perc, names):
    """O.kd_step's NLL + KD terms plus the perceptual L1 between the two inverse passes fed the given draws."""
    from oracle import glow_oracle as O
    sd = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in s_sd.items()}
    with O.bf16_operands():
        out = O.kd_step(sd, s_cfg, t_sd, t_cfg, x, {"nll": 0.9, "kd": 0.1, "perceptual": 0.0}, n1, n2)
        loss, perc = out["result_loss"], torch.zeros(())
        if w_perc > 0:
            sx = glow_reverse_sampled(sd, s_cfg, latent, 0.7, eps_s)
            with torch.no_grad():
                tx = glow_reverse_sampled(t_sd, t_cfg, latent, 0.7, eps_t)
            p = (sx - tx).abs().flatten(1).mean(1)
            perc = torch.where(torch.isnan(p), torch.zeros_like(p), p).mean()
            loss = loss + w_perc * perc
        loss.backward()
    scal = {"nll": out["nll"].item(), "kd": out["kd"].item(), "perceptual": perc.item(), "loss": loss.item()}
    return scal, {k: sd[k].grad for k in names}


@pytest.mark.gpu
def test_kd_step_with_perceptual_weight_matches_oracle_draw_for_draw(monkeypatch):
    """CIFAR-shaped pair (L=3, student K=2, teacher K=3, hidden 64), weights 0.9 / 0.1 / 0.1. Both models see the same
    dequantisation noise; the latent and the Split2d draws (student top level first, then the teacher) are regenerated
    by re-seeding the global generator and fed to the oracle. The four loss scalars and every student gradient are
    compared. The top level's share of the perceptual gradient arrives only through the Split2d pass-through, so the
    control compares (grad at weight 0.1) - (grad at weight 0) of the top-level parameters with the oracle's.
    Measured: nll / kd / perceptual / loss within 1e-6 relative; student gradients median 1.2e-3, worst 1.7e-2
    (flow.layers.5.block.0.conv.weight); top-level perceptual share worst 1.5e-2."""
    from nf_distillation_b200.models import utils as U
    B = 16
    g = torch.Generator().manual_seed(21)
    x = images(B, 32, g)
    n1, n2 = torch.rand(B, 3, 32, 32, generator=g) / 256, torch.rand(B, 3, 32, 32, generator=g) / 256
    grads, scal = {}, {}
    for wp in (0.1, 0.0):
        m, s_cfg, t_cfg, s_sd, t_sd = kd_pair(wp)
        names = set(dict(m.student.named_parameters()))
        m.to(dev)
        q = [n1.to(dev), n2.to(dev)]
        monkeypatch.setattr(U, "dequant_noise", lambda t_, n: q.pop(0))
        torch.manual_seed(1234)
        out = m.training_step([x.to(dev), None], 0)
        out["loss"].backward()
        torch.cuda.synchronize()
        scal[wp] = {k: v.item() for k, v in out.items()}
        grads[wp] = {n_: p.grad.detach().cpu().clone() for n_, p in m.student.named_parameters()}
        assert all(p.grad is None for p in m.teacher.parameters())
    # the same draws, in the reference's order: latent, student Split2d eps (top level first), teacher Split2d eps
    torch.manual_seed(1234)
    latent = torch.empty(B, 48, 4, 4, device=dev).normal_()      # prior mean 0, logs 0 (zero prior_h, no learn_top)
    eps_s = [torch.randn(B, 12, 8, 8, device=dev), torch.randn(B, 6, 16, 16, device=dev)]
    eps_t = [torch.randn(B, 12, 8, 8, device=dev), torch.randn(B, 6, 16, 16, device=dev)]
    cpu = lambda ts: [t_.cpu() for t_ in ts]
    o_scal, o_grads = {}, {}
    for wp in (0.1, 0.0):
        o_scal[wp], o_grads[wp] = oracle_kd(s_sd, s_cfg, t_sd, t_cfg, x, n1, n2, latent.cpu(), cpu(eps_s), cpu(eps_t),
                                            wp, names)
    p_, o_ = scal[0.1], o_scal[0.1]
    print("\nloss scalars (product, oracle):", {k: (p_[k], o_[k]) for k in o_})
    assert o_["perceptual"] > 0 and scal[0.0]["perceptual"] == 0.0
    assert abs(p_["nll"] - o_["nll"]) < 1e-4 * abs(o_["nll"])
    assert abs(p_["kd"] - o_["kd"]) < 1e-2 * abs(o_["kd"])
    assert abs(p_["perceptual"] - o_["perceptual"]) < 1e-2 * abs(o_["perceptual"])
    assert abs(p_["loss"] - o_["loss"]) < 1e-4 * abs(o_["loss"])
    errs = sorted((rel(grads[0.1][n_], o_grads[0.1][n_]), n_) for n_ in names)
    print("student gradients: median %.1e worst %.1e (%s)" % (errs[len(errs) // 2][0], errs[-1][0], errs[-1][1]))
    assert errs[len(errs) // 2][0] < 1e-2 and errs[-1][0] < 0.1, (errs[len(errs) // 2], errs[-3:])
    # control: the perceptual share of the top level's gradients (layers after the last Split2d)
    top = [n_ for n_ in names if n_.startswith(("flow.layers.9.", "flow.layers.10."))]
    assert top
    worst = 0.0
    for n_ in top:
        d_p, d_o = grads[0.1][n_] - grads[0.0][n_], o_grads[0.1][n_] - o_grads[0.0][n_]
        if d_o.abs().max() == 0:
            continue
        assert d_p.abs().max() > 0, f"{n_}: no perceptual gradient reached the top level"
        worst = max(worst, rel(d_p, d_o))
    print("top-level perceptual share: worst %.1e" % worst)
    assert worst < 0.1, worst


# ------------------------------------------------------------------------------------------------ KDTrainer
@pytest.mark.gpu
@pytest.mark.parametrize("use_graphs", [True, False])
def test_kd_trainer_trains_with_perceptual_weight(use_graphs):
    """KDTrainer captures (or runs eagerly) a step with perceptual > 0: three steps, finite losses, a non-zero
    perceptual term, and every student parameter tensor moves."""
    from nf_distillation_b200.train import KDTrainer, glow_cfg, kd_config
    s_cfg, t_cfg = glow_cfg((32, 32, 3), 2, 3, 64), glow_cfg((32, 32, 3), 3, 3, 64)
    B = 16
    tr = KDTrainer(kd_config(s_cfg, t_cfg, perceptual=0.1), (B, 3, 32, 32), torch.device(dev), use_graphs=use_graphs,
                   seed=5)
    assert not tr.pipelined
    tr.x.copy_(images(B, 32, torch.Generator().manual_seed(4)).to(dev))
    before = {n_: p.detach().clone() for n_, p in tr.module.student.named_parameters()}
    tr.warmup(iters=1)
    assert (tr.g_fb is not None) == use_graphs
    for _ in range(3):
        tr.step_device()
        losses = tr.losses.cpu()
        assert torch.isfinite(losses).all(), losses
        assert losses[2].item() > 0, "perceptual term must be non-zero"
    torch.cuda.synchronize()
    for n_, p in tr.module.student.named_parameters():
        assert not torch.equal(p.detach(), before[n_]), f"{n_} did not change"
