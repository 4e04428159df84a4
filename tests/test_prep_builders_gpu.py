"""GPU: the no-grad operand build of a FlowStep (FlowStep._consts, one launch per step) and the batched training build
(functional.PrepCtx) lay out and compute the same fused affine and coupling-net operands, bit for bit, in both
directions; and InvertibleConv1x1.get_weight is the fused affine of a step whose ActNorm is zero."""
import pytest
import torch

pytestmark = pytest.mark.gpu
dev = "cuda"

CASES = [(12, "invconv", "affine", True), (24, "invconv", "affine", True), (48, "invconv", "affine", True),
         (96, "invconv", "affine", True), (24, "invconv", "affine", False), (24, "shuffle", "affine", True),
         (24, "reverse", "affine", True), (24, "invconv", "additive", True)]


def make_step(C, perm, coupling, lu, is_1d=False, seed=0):
    from nf_distillation_b200.models import FlowStep
    torch.manual_seed(seed)
    step = FlowStep(C, 32 if is_1d else 64, 1.0, perm, coupling, lu, is_1d=is_1d).to(dev)
    with torch.no_grad():       # ActNorm and Conv2dZeros start at zero: give every parameter a value
        for p in step.parameters():
            p.add_(0.1 * torch.randn_like(p))
    return step


def batched(step, reverse):
    from nf_distillation_b200 import functional as Fn
    with torch.enable_grad():
        pctx = Fn.PrepCtx([step], reverse).build()
    return pctx.consts[0], pctx.cops[0]


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("C,perm,coupling,lu", CASES)
def test_consts_match_the_batched_build(C, perm, coupling, lu, reverse):
    step = make_step(C, perm, coupling, lu, seed=C)
    with torch.no_grad():
        k = step._consts(reverse)
    (Wf, bf, sl), (B1, B1T, B2, B2T, B3, B3T, bias1, bias2, bias3) = batched(step, reverse)
    torch.cuda.synchronize()
    for a, b in ((k.Wf, Wf), (k.bf, bf), (k.sl, sl), (k.B1, B1), (k.B2, B2), (k.B3, B3), (k.bias1, bias1),
                 (k.bias2, bias2), (k.bias3, bias3)):
        assert torch.equal(a, b)
    assert k.B1T is None and k.B2T is None and k.B3T is None      # the no-grad path has no dgrads to feed
    assert torch.equal(B1T, B1.T) and torch.equal(B2T, B2.T) and torch.equal(B3T, B3.T)


@pytest.mark.parametrize("reverse", [False, True])
def test_1d_consts_match_the_batched_build(reverse):
    step = make_step(6, "invconv", "affine", True, is_1d=True, seed=6)
    with torch.no_grad():
        k = step._consts(reverse)
    (Wf, bf, sl), cops = batched(step, reverse)
    assert cops is None
    assert torch.equal(k.Wf, Wf) and torch.equal(k.bf, bf) and torch.equal(k.sl, sl)


@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("lu", [True, False])
def test_get_weight_is_the_affine_of_a_step_with_zero_actnorm(lu, reverse):
    step = make_step(24, "invconv", "affine", lu, seed=3)
    with torch.no_grad():
        step.actnorm.bias.zero_()
        step.actnorm.logs.zero_()
        w, dlogdet = step.invconv.get_weight(torch.zeros(2, 24, 4, 8, device=dev), reverse)
    (Wf, _, sl), _ = batched(step, reverse)
    assert torch.equal(w.view(24, 24), Wf)
    assert torch.equal(dlogdet, (-sl[0] if reverse else sl[0]) * 32)
