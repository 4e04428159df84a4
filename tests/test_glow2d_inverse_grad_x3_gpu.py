"""Gradients through the 2-D inverse pass in the fp32-class precision mode ("bf16x3": precise.FlowStep2dReverseX3Fn,
csrc/split3.cu coupling_inv_bwd_f32), against the plain fp32 oracle — the perceptual L1 term of
pl_module.py:229-243,284-299 trained at fp32 level. The bf16 mode of the same pass is checked in
test_glow2d_inverse_grad_gpu.py, whose helpers this file uses.

Bounds follow test_headline_parity_gpu.py's bf16x3 tests: a gradient that reaches the loss without passing a ReLU mask
of the step's coupling net is held at fp32 level; a gradient behind a mask is held in relative L2, because the few ReLU
units whose pre-activation lies within the mode's 5e-6 of zero take the other mask than the fp32 reference and each
moves its row of a weight gradient by O(1/sqrt(M)) (DESIGN §4).
"""
import os
import sys

import pytest
import torch

from test_glow2d_inverse_grad_gpu import glow_reverse_sampled, images, kd_pair, make_step, rel
from test_headline_parity_gpu import UNKINKED, StaticNoise, rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
dev = "cuda"

NFK_ERR_SHAPE, NFK_ERR_ARG = -1, -3


# ------------------------------------------------------------------------------------------------ C ABI (no device)
def test_coupling_inv_bwd_f32_argument_errors_without_gpu():
    """nfk_coupling_inv_bwd_f32 validates its arguments before any CUDA call: an unsupported channel count or an empty
    shape is NFK_ERR_SHAPE, a missing buffer NFK_ERR_ARG."""
    from nf_distillation_b200 import _lib
    f = _lib.LIB.nfk_coupling_inv_bwd_f32
    p = 256          # any non-null address: the checks fail before it is dereferenced
    bufs = [p] * 7
    for C in (10, 13, 16, 192, 0):
        assert f(*bufs, 4, C, 8, 8, None) == NFK_ERR_SHAPE, C
    for B, H, W in ((0, 8, 8), (4, 0, 8), (4, 8, -1)):
        assert f(*bufs, B, 12, H, W, None) == NFK_ERR_SHAPE, (B, H, W)
    for i in range(7):
        args = list(bufs)
        args[i] = None
        for C in (12, 24, 48, 96):
            assert f(*args, 4, C, 8, 8, None) == NFK_ERR_ARG, (i, C)


# ------------------------------------------------------------------------------------------------ one FlowStep
def kinked(name):
    """True for the gradients of a reverse step that pass a ReLU mask of its coupling net: everything of conv#1 and
    conv#2. The step's ActNorm / invconv act after the coupling in the inverse direction (x = Wf zc + bf), and the
    log-scale / zero-conv gradients weight every unit by its value (see UNKINKED)."""
    return name.startswith("block.") and name not in UNKINKED


def check_inverse_step_x3(C, H, B, hid, seed, coupling="affine", permutation="invconv", lu=True):
    """One FlowStep's inverse with grad in bf16x3 mode against the fp32 oracle's autograd through
    O.flowstep(reverse=True); returns the measured errors (relative to max|.|, and relative L2 for the kinked ones)."""
    from oracle import glow_oracle as O
    st, sd, perm = make_step(C, hid, seed, coupling, permutation, lu)
    st.precision = "bf16x3"
    names = dict(st.named_parameters())
    g = torch.Generator().manual_seed(seed + 7)
    z = torch.randn(B, C, H, H, generator=g)
    ld0 = torch.randn(B, generator=g)
    wx, wl = torch.randn(B, C, H, H, generator=g), torch.randn(B, generator=g)
    osd = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in sd.items()}
    zo = z.clone().requires_grad_(True)
    with O.bf16_operands(False):
        x32, ld32 = O.flowstep(zo, osd, "", ld0, True, coupling=coupling, perm=perm)
        ((x32 * wx).sum() + (ld32 * wl).sum()).backward()
    st = st.to(dev)
    with torch.no_grad():
        xi, ldi = st(z.to(dev), logdet=ld0.to(dev), reverse=True)
    zg, lg = z.to(dev).requires_grad_(True), ld0.to(dev).requires_grad_(True)
    xt, ldt = st(zg, logdet=lg, reverse=True)
    assert torch.equal(xt.detach(), xi), "training and inference inverse passes must agree bit for bit"
    assert rel(ldt, ldi) < 1e-6      # (per-sample log-det partial sums meet in fp32 atomics: order is not fixed)
    ((xt * wx.to(dev)).sum() + (ldt * wl.to(dev)).sum()).backward()
    assert torch.equal(lg.grad.cpu(), wl)           # the log-det passes straight through
    c1 = C // 2
    errs = {"x": rel(xt, x32), "ld": rel(ldt, ld32), "dz2": rel(zg.grad[:, c1:], zo.grad[:, c1:]),
            "dz": rel(zg.grad, zo.grad), "dz_l2": rel_l2(zg.grad, zo.grad)}
    for n_, p in st.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), n_
        errs[n_] = rel(p.grad, osd[n_].grad)
        if kinked(n_):
            errs[n_ + "_l2"] = rel_l2(p.grad, osd[n_].grad)
    print(f"\nC={C} H={H} B={B} hid={hid} {coupling}/{permutation}/lu={lu}: "
          + " ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    # x: measured 1.3e-6..3.8e-6, 8.2e-6 at C = 96 (the 96-channel inverse affine); log-det <= 1.1e-6
    assert errs["x"] < 2e-5 and errs["ld"] < 1e-5, errs
    # dz2 = dzc2 / s passes no ReLU mask (measured 2.5e-7..8.2e-6). dz1 = dzc1 + col2im(dcol) does: a flipped unit moves dz1
    # at the nine pixels its conv#1 taps reach, so dz is held like the forward x3 step's input gradient in relative L2
    # (measured 5e-6..1.2e-3) and in max-norm (measured 8e-6 where no unit flips, 9e-4..1.3e-2 where units do)
    assert errs["dz2"] < 1e-4 and errs["dz_l2"] < 5e-3 and errs["dz"] < 3e-2, errs
    M = B * H * H
    for n_ in names:
        if kinked(n_):
            # measured relative L2 <= 2.5e-3 at M >= 2304 pixels and 5.7e-3 (block.0.conv.weight) at M = 1280, max-norm
            # <= 1.9e-2 and 5.1e-2 at M = 1280: an entry of a weight-gradient row is a sum over M pixels, so one
            # flipped unit moves it by O(1/sqrt(M)) and a max-norm error counts the flips that land in one row
            assert errs[n_ + "_l2"] < 1e-2 and errs[n_] < max(3e-2, 3 * M ** -0.5), (n_, errs[n_], errs[n_ + "_l2"])
        else:       # measured <= 1.6e-5
            assert errs[n_] < 1e-4, (n_, errs[n_])
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("C,H,B,hid", [
    (12, 16, 40, 512),    # level 0 of the benched pair (M = 10240)
    (12, 16, 9, 64),      # ragged batch
    (12, 32, 6, 64),      # 32x32 maps (the banded launches of the bf16 mode)
    (24, 8, 20, 512),
    (48, 4, 37, 512),     # ragged batch
    (96, 4, 33, 64),
])
def test_flowstep_inverse_pass_gradients_in_bf16x3_match_the_fp32_oracle(C, H, B, hid):
    """FlowStep2dReverseX3Fn: affine1x1_bwd without col2im -> coupling_inv_bwd_f32 -> the split backward of the
    coupling net shared with FlowStep2dX3Fn -> col2im_add, then the batched inverse chain rule of the fused affine.
    x, log-det, dz and every parameter gradient against the fp32 oracle. Where no ReLU unit flips (C = 96 here) every
    tensor measures <= 1.5e-5; dz measures <= 1.2e-3 in relative L2 and <= 1.3e-2 in max-norm (the bf16 mode: < 0.1)."""
    check_inverse_step_x3(C, H, B, hid, 300 + C + H)


@pytest.mark.gpu
@pytest.mark.parametrize("coupling,permutation,lu", [
    ("additive", "invconv", True),
    ("affine", "shuffle", True),
    ("affine", "reverse", True),
    ("affine", "invconv", False),
])
def test_flowstep_inverse_pass_gradients_in_bf16x3_of_the_variants(coupling, permutation, lu):
    """Additive coupling (the affine arithmetic with the logit rows pinned at bias 30, so s == 1.0f), the fixed
    shuffle / reverse permutations and the plain invconv weight (LU_decomposed=False), against the fp32 oracle.
    Measured: x 1.3e-6..1.8e-6, log-det <= 1.1e-6, dz <= 1.9e-6, every parameter gradient <= 1.6e-5."""
    check_inverse_step_x3(12, 8, 24, 64, 500, coupling, permutation, lu)


@pytest.mark.gpu
@pytest.mark.parametrize("C,H,B", [(12, 16, 40), (48, 4, 37)])
def test_bf16x3_additive_flowstep_matches_the_fp32_oracle(C, H, B):
    """Additive coupling in bf16x3, forward with grad, at the bounds of
    test_bf16x3_precision_flowstep_matches_the_fp32_oracle except for the max-norm of the kinked gradients; the no-grad
    inverse undoes the forward. Measured: z <= 4.5e-6, log-det <= 1.1e-6, dx 6e-4 in relative L2, unkinked gradients
    <= 8.5e-6, kinked ones <= 3.7e-3 in relative L2 and <= 3.3e-2 in max-norm (block.0.conv.weight)."""
    from oracle import glow_oracle as O
    st, sd, _ = make_step(C, 512, 300 + C, coupling="additive")
    st.precision = "bf16x3"
    g = torch.Generator().manual_seed(C + 1)
    x = torch.randn(B, C, H, H, generator=g)
    ld0 = torch.randn(B, generator=g)
    wz, wl = torch.randn(B, C, H, H, generator=g), torch.randn(B, generator=g)
    names = dict(st.named_parameters())
    osd = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in sd.items()}
    xo = x.clone().requires_grad_(True)
    with O.bf16_operands(False):
        z32, ld32 = O.flowstep(xo, osd, "", ld0, False, coupling="additive")
        ((z32 * wz).sum() + (ld32 * wl).sum()).backward()
    st = st.to(dev)
    xg = x.to(dev).requires_grad_(True)
    zt, ldt = st(xg, logdet=ld0.to(dev), reverse=False)
    ((zt * wz.to(dev)).sum() + (ldt * wl.to(dev)).sum()).backward()
    errs = {"z": rel(zt, z32), "ld": rel(ldt, ld32), "dx": rel(xg.grad, xo.grad), "dx_l2": rel_l2(xg.grad, xo.grad)}
    for n_, p in st.named_parameters():
        errs[n_] = rel(p.grad, osd[n_].grad)
        errs[n_ + "_l2"] = rel_l2(p.grad, osd[n_].grad)
    print(f"\nadditive C={C} H={H} B={B}: " + " ".join(f"{k}={v:.1e}" for k, v in errs.items()))
    assert errs["z"] < 1e-4 and errs["ld"] < 1e-5, errs
    assert errs["dx_l2"] < 5e-3 and errs["dx"] < 1.5e-2, errs
    for n_ in names:
        if n_ in UNKINKED:
            assert errs[n_] < 5e-5, (n_, errs[n_])
        else:
            # the max-norm error of a weight-gradient row counts the flipped ReLU units that land in it, so it varies
            # with the draw more than the relative L2 does: 2.5e-2 / 3.3e-2 on block.0.conv.weight here against the
            # affine test's 1.5e-2 (its relative L2 bound holds unchanged)
            assert errs[n_] < max(5e-2, 3 * (B * H * H) ** -0.5) and errs[n_ + "_l2"] < 5e-3, (n_, errs[n_])
    with torch.no_grad():
        zi, ldi = st(x.to(dev), logdet=ld0.to(dev), reverse=False)
        back, ldb = st(zi, logdet=ldi, reverse=True)
    assert torch.equal(zi, zt.detach())
    assert rel(back, x) < 1e-4 and rel(ldb, ld0) < 1e-4


# ------------------------------------------------------------------------------------------------ the KD step
def oracle_kd_f32(s_sd, s_cfg, t_sd, t_cfg, x, n1, n2, latent, eps_s, eps_t, w_perc, names):
    """The reference's KD step in fp32 (NLL + KD + the perceptual L1 between the two inverse passes fed the given
    draws): loss scalars and the student's gradients."""
    from oracle import glow_oracle as O
    sd = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in s_sd.items()}
    with O.bf16_operands(False):
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
def test_bf16x3_kd_step_with_perceptual_weight_matches_the_fp32_oracle_draw_for_draw(monkeypatch):
    """The construction of test_kd_step_with_perceptual_weight_matches_oracle_draw_for_draw (CIFAR-shaped pair, L=3,
    student K=2, teacher K=3, hidden 64, weights 0.9 / 0.1 / 0.1, the same dequantisation noise, latent and Split2d
    draws) with both models in bf16x3, against the fp32 oracle: the four loss scalars and every student gradient at the
    bounds of test_bf16x3_precision_kd_step_taps_and_gradients_at_fp32_level. The perceptual share of each gradient,
    (grad at weight 0.1) - (grad at weight 0), is compared with the oracle's the same way, so an error in the inverse
    pass cannot hide under the NLL's larger gradient. Measured: loss scalars <= 1e-7 relative; student gradients median
    1.8e-5, worst 2.6e-3 (relative L2 1.9e-3); perceptual share median 7.6e-5, worst 9.1e-3 (relative L2 3.1e-3), both
    worst on flow.layers.1.block.0.conv.weight."""
    from nf_distillation_b200.models import utils as U
    B = 16
    g = torch.Generator().manual_seed(21)
    x = images(B, 32, g)
    n1, n2 = torch.rand(B, 3, 32, 32, generator=g) / 256, torch.rand(B, 3, 32, 32, generator=g) / 256
    grads, scal = {}, {}
    for wp in (0.1, 0.0):
        m, s_cfg, t_cfg, s_sd, t_sd = kd_pair(wp)
        m.student.set_precision("bf16x3")
        m.teacher.set_precision("bf16x3")
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
    torch.manual_seed(1234)
    latent = torch.empty(B, 48, 4, 4, device=dev).normal_()      # prior mean 0, logs 0 (zero prior_h, no learn_top)
    eps_s = [torch.randn(B, 12, 8, 8, device=dev), torch.randn(B, 6, 16, 16, device=dev)]
    eps_t = [torch.randn(B, 12, 8, 8, device=dev), torch.randn(B, 6, 16, 16, device=dev)]
    cpu = lambda ts: [t_.cpu() for t_ in ts]
    o_scal, o_grads = {}, {}
    for wp in (0.1, 0.0):
        o_scal[wp], o_grads[wp] = oracle_kd_f32(s_sd, s_cfg, t_sd, t_cfg, x, n1, n2, latent.cpu(), cpu(eps_s),
                                                cpu(eps_t), wp, names)
    p_, o_ = scal[0.1], o_scal[0.1]
    print("\nloss scalars (product, fp32 oracle):", {k: (p_[k], o_[k]) for k in o_})
    assert o_["perceptual"] > 0 and scal[0.0]["perceptual"] == 0.0
    for k in ("nll", "kd", "perceptual", "loss"):
        assert abs(p_[k] - o_[k]) <= 1e-5 * abs(o_[k]), (k, p_[k], o_[k])
    errs = sorted((rel(grads[0.1][n_], o_grads[0.1][n_]), rel_l2(grads[0.1][n_], o_grads[0.1][n_]), n_)
                  for n_ in names)
    print("student gradients: median %.1e worst %.1e (%s), worst rel L2 %.1e"
          % (errs[len(errs) // 2][0], errs[-1][0], errs[-1][2], max(e[1] for e in errs)))
    assert errs[-1][0] < 1.5e-2 and max(e[1] for e in errs) < 5e-3 and errs[len(errs) // 2][0] < 5e-4, errs[-3:]
    share = []
    for n_ in names:
        d_p, d_o = grads[0.1][n_] - grads[0.0][n_], o_grads[0.1][n_] - o_grads[0.0][n_]
        if d_o.abs().max() == 0:
            continue
        share.append((rel(d_p, d_o), rel_l2(d_p, d_o), n_))
    share.sort()
    print("perceptual share: %d tensors, median %.1e, worst %.1e (%s), worst rel L2 %.1e"
          % (len(share), share[len(share) // 2][0], share[-1][0], share[-1][2], max(e[1] for e in share)))
    # every tensor but the Split2d parameters (torch.normal's draw has no derivative) gets a perceptual share
    from nf_distillation_b200.models.layers import Split2d
    split = {f"flow.layers.{i}.{k}" for i, l in enumerate(m.student.flow.layers) if isinstance(l, Split2d)
             for k, _ in l.named_parameters()}
    assert names - {e[2] for e in share} == split and split
    assert share[-1][0] < 1.5e-2 and max(e[1] for e in share) < 5e-3, share[-3:]


# ------------------------------------------------------------------------------------------------ KDTrainer
@pytest.mark.gpu
def test_bf16x3_kd_trainer_with_perceptual_weight_makes_the_same_update_eager_and_graph_captured(monkeypatch):
    """KDTrainer with both models in bf16x3 and perceptual 0.1: one step from the same weights, batch, noise and
    latent / Split2d draws, run eagerly and replayed from a CUDA graph: the same loss scalars and the same gradient
    (fp32 atomics order aside), a finite update that moves every student tensor. Measured: losses equal to 1e-7
    relative, gradients to 3e-8 of max|g|."""
    from nf_distillation_b200.models import utils as U
    from nf_distillation_b200.train import KDTrainer, glow_cfg, kd_config
    s_cfg, t_cfg = glow_cfg((32, 32, 3), 2, 3, 64), glow_cfg((32, 32, 3), 3, 3, 64)
    B = 16
    g = torch.Generator().manual_seed(4)
    x = images(B, 32, g)
    n1, n2 = torch.rand(B, 3, 32, 32, generator=g) / 256, torch.rand(B, 3, 32, 32, generator=g) / 256
    res = {}
    for use_graphs in (False, True):
        noise = StaticNoise((B, 3, 32, 32))
        monkeypatch.setattr(U, "dequant_noise", noise)
        tr = KDTrainer(kd_config(s_cfg, t_cfg, perceptual=0.1), (B, 3, 32, 32), torch.device(dev),
                       use_graphs=use_graphs, seed=5)
        tr.module.student.set_precision("bf16x3")
        tr.module.teacher.set_precision("bf16x3")
        init = {k: v.detach().clone() for k, v in tr.module.student.state_dict().items()}
        tr.x.copy_(x.to(dev))
        noise.set(n1, n2)
        tr.warmup(iters=1)
        assert (tr.g_fb is not None) == use_graphs
        tr.reset_state(init)
        torch.manual_seed(99)            # the latent and Split2d draws of the step
        tr.step_device()
        torch.cuda.synchronize()
        res[use_graphs] = (tr.losses.cpu(), tr.flat_grad_view().detach().cpu().clone(),
                           {k: (v.detach().cpu() - init[k].cpu()) for k, v in tr.module.student.state_dict().items()
                            if v.dtype.is_floating_point})
    (le, ge, ue), (lg, gg, ug) = res[False], res[True]
    print("\nlosses eager", le.tolist(), "graph", lg.tolist(), "grad rel %.1e" % rel(gg, ge))
    assert torch.isfinite(le).all() and le[2].item() > 0, le
    assert torch.allclose(lg, le, rtol=1e-5, atol=0), (lg, le)
    assert torch.isfinite(ge).all() and rel(gg, ge) < 1e-4
    for k, d in ue.items():
        if not d.any() and not ug[k].any():
            continue      # buffers (prior_h) and frozen tensors
        assert torch.isfinite(d).all() and torch.isfinite(ug[k]).all(), k
        assert rel_l2(ug[k], d) < 1e-2, (k, rel_l2(ug[k], d))
    moved = [n_ for n_, p in tr.module.student.named_parameters() if ue[n_].abs().max() > 0]
    assert len(moved) == len(list(tr.module.student.parameters()))
