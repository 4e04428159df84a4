"""GPU checks of the MAF / MADE path. PARITY UNPINNED: the reference ships no MAF code (README.md:7 only), so the
checker is this repo's own plain-PyTorch fp32 restatement of the paper (oracle/maf_oracle.py).

Tolerances (masked linears run on bf16 tensor-core tiles with fp32 accumulation; the affine transform and log-det
are fp32): outputs / nll 1e-3 relative to max, inverse round trip 1e-4 (the inverse evaluates the same bf16 network; the resident
kernel sums each pre-activation in a different order than the forward GEMM, so a hidden unit sitting on a bf16
rounding boundary may round the other way — the D-pass GEMM inverse, bit-consistent with the forward, holds 1e-5 and
the two inverses agree to 1e-4), input gradient 1e-2, parameter gradients: cosine similarity >= 0.999 and 0.1 of max|grad|
(0.99 / 0.2 for the 64-sample case, where bf16 rounding of the few summed terms dominates)."""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def rel(a, b):
    b = b.to(a.device)
    return ((a - b).abs().max() / (b.abs().max() + 1e-12)).item()


@pytest.mark.parametrize("D,H,K,B", [(6, 512, 5, 300), (63, 512, 3, 257), (63, 192, 2, 64), (63, 512, 2, 8229)])
def test_maf_forward_inverse_backward_vs_paper_restatement(D, H, K, B):
    from nf_distillation_b200.models.maf import create_maf_model
    from oracle import maf_oracle as MO
    torch.manual_seed(D + H)
    m = create_maf_model(dict(image_shape=[D], hidden_channels=H, K=K))
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    x = torch.randn(B, D) * 1.5 + 0.5
    o_outs, o_nll = MO.maf_forward(sd, D, K, x)
    m = m.cuda()
    with torch.no_grad():
        outs, nll, none = m(x.cuda(), None)
        assert none is None and len(outs) == K
        assert rel(nll, o_nll) < 1e-3
        for a, b in zip(outs, o_outs):
            assert rel(a, b) < 1e-3
        back = m(z=outs[-1], reverse=True)
        # x -> z -> x; fp32 cancellation in u*e^alpha + mu grows with the largest |mu| among B*D entries
        assert len(back) == K and rel(back[-1], x) < 1e-4
        # per-layer log-det antisymmetry
        z, ld = m.flow.layers[0](x.cuda(), logdet=torch.zeros(B, device="cuda"))
        xb, ld2 = m.flow.layers[0](z, logdet=ld, reverse=True)
        assert ld2.abs().max().item() < 1e-3 * (ld.abs().max().item() + 1) and rel(xb, x) < 1e-4
        # the resident one-launch inverse (both tile shapes) against the D-pass GEMM inverse it replaces
        lay = m.flow.layers[0]
        lay.resident_inverse = False
        x_dp, ld_dp = lay(z, logdet=ld, reverse=True)
        lay.resident_inverse = True
        assert rel(x_dp, x) < (1e-5 if B < 4096 else 1e-4)
        for push, mt in ((True, 0), (False, 1), (False, 2)):   # push kernel; pull kernel with 16 / 32 samples per warp
            lay.push_inverse, lay.resident_mtiles = push, mt
            # the push kernel needs degree changes on whole 8-unit tiles; with fewer tiles than degrees (H/8 < D-1)
            # the module keeps the standard per-unit MADE assignment and every request lands on the pull kernel
            aligned = H // 8 >= D - 1
            assert lay._inverse_jobs(z.device)[1] == (push and aligned)
            x_r, ld_r = lay(z, logdet=ld, reverse=True)
            assert rel(x_r, x_dp) < 1e-4, (push, mt)
            assert (ld_r - ld_dp).abs().max().item() < 1e-3 * (ld.abs().max().item() + 1), (push, mt)
        lay.push_inverse, lay.resident_mtiles = True, 0
    # autoregressive property: d z_i / d x_j = 0 for j > i  (layer 0, un-flipped view)
    with torch.no_grad():
        x2 = x.clone()
        x2[:, D - 1] += 1.0
        z1, _ = m.flow.layers[0](x.cuda(), logdet=None)
        z2, _ = m.flow.layers[0](x2.cuda(), logdet=None)
        un1, un2 = z1.flip(1), z2.flip(1)
        assert torch.equal(un1[:, : D - 1], un2[:, : D - 1])
    xs = x.clone().requires_grad_(True)
    sdg = {k: (v.clone().requires_grad_(True) if v.dtype.is_floating_point and k != "prior_h" else v)
           for k, v in sd.items()}
    MO.maf_forward(sdg, D, K, xs)[1].mean().backward()
    xg = x.cuda().requires_grad_(True)
    m(xg, None)[1].mean().backward()
    assert rel(xg.grad, xs.grad) < (1e-2 if B >= 256 else 3e-2)
    for n, p in m.named_parameters():
        ref = sdg[n].grad
        cs = torch.nn.functional.cosine_similarity(p.grad.flatten().cpu(), ref.flatten(), dim=0).item()
        assert cs > (0.999 if B >= 256 else 0.99) and rel(p.grad, ref) < (0.1 if B >= 256 else 0.2), (n, cs)


@pytest.mark.parametrize("D,H,B,flip", [(1, 64, 33, True), (2, 64, 16, False), (100, 64, 50, True), (17, 128, 1, True),
                                        (63, 512, 20000, True)])
def test_resident_inverse_matches_paper_restatement(D, H, B, flip):
    """One MADE layer, inverse only: the one-launch resident kernels (push: layer-2 tiles multiplied straight into
    running output sums; pull: h2 kept in shared memory) against the fp32 restatement's D-pass inverse
    (bf16 network vs fp32 network: 2e-3 of max|x|), at degenerate sizes (D = 1, D > H so some degrees own no hidden
    unit, a single sample, a ragged last tile) and at a batch that fills every SM several times."""
    from nf_distillation_b200.models.maf import MADE
    from oracle import maf_oracle as MO
    torch.manual_seed(D * 7 + H)
    made = MADE(D, H, flip=flip)
    with torch.no_grad():
        made.fc3.bias.normal_(0, 0.1)
    sd = {"l." + k: v.clone() for k, v in made.state_dict().items()}
    u = torch.randn(B, D)
    x_o, sum_alpha = MO.made_inverse(u, sd, "l.", D, flip=flip)
    made = made.cuda()
    with torch.no_grad():
        ld0 = torch.randn(B, device="cuda")
        for push, mt in ((True, 0), (False, 1), (False, 2)):
            made.push_inverse, made.resident_mtiles = push, mt
            assert made._inverse_jobs(ld0.device)[1] == (push and 2 * D <= 128)
            x, ld = made(u.cuda(), logdet=ld0, reverse=True)
            assert rel(x, x_o) < 2e-3, (push, mt)
            assert ((ld - ld0).cpu() - sum_alpha).abs().max().item() < 2e-3 * (sum_alpha.abs().max().item() + 1), (push, mt)
            x2, none = made(u.cuda(), logdet=None, reverse=True)
            assert none is None and torch.equal(x2, x)


def test_made_forward_with_a_512_wide_input_runs_the_gemm_pair_at_a_large_batch():
    """D = 500 pads to Dp = 512, deeper than the fused conv kernel takes (its A tile would leave shared memory for one
    weight slot), so at a batch >= 8192 the forward runs the two GEMMs, in inference and in training (h1 and the ReLU
    masks kept). Both against the fp32 restatement: u to 1e-3 of max; the log-det, a sum of 500 alphas computed by
    the bf16 network, to 2e-3 of (max + 1) as in the resident-inverse test."""
    from nf_distillation_b200 import ops
    from nf_distillation_b200.models.maf import MADE
    from oracle import maf_oracle as MO
    D, H, B = 500, 512, 8192
    torch.manual_seed(5)
    made = MADE(D, H, flip=True)
    with torch.no_grad():
        made.fc3.bias.normal_(0, 0.1)
    assert made.Dp == 512 and not ops.cnet_fused_supported(H, made.Dp)
    sd = {"l." + k: v.clone() for k, v in made.state_dict().items()}
    x = torch.randn(B, D)
    u_o, ld_o = MO.made_forward(x, sd, "l.", D)
    made = made.cuda()
    with torch.no_grad():
        u, ld = made(x.cuda(), logdet=torch.zeros(B, device="cuda"))
    ld_tol = 2e-3 * (ld_o.abs().max().item() + 1)
    assert rel(u, u_o) < 1e-3 and (ld.cpu() - ld_o).abs().max().item() < ld_tol
    u2, ld2 = made(x.cuda(), logdet=torch.zeros(B, device="cuda"))
    assert u2.requires_grad and rel(u2, u_o) < 1e-3 and (ld2.detach().cpu() - ld_o).abs().max().item() < ld_tol


def test_masked_tile_skipping_is_exact():
    """The ranged GEMM (structurally-zero k-blocks never loaded) equals the full GEMM on the masked weight, bit for bit."""
    from nf_distillation_b200 import ops
    from nf_distillation_b200.models.maf import MADE
    torch.manual_seed(0)
    made = MADE(63, 512, flip=True).cuda()
    ops_ = made._cached_operands()
    B2 = ops_[2]
    h1 = torch.relu(torch.randn(1000, 512, device="cuda")).bfloat16()
    bias = torch.randn(512, device="cuda")
    a = torch.empty(1000, 512, device="cuda", dtype=torch.bfloat16)
    b = torch.empty_like(a)
    kb0, kb1 = made._ranges
    assert sum(e - s for s, e in zip(kb0, kb1)) < len(kb0) * 8          # something is actually skipped
    ops.gemm_nt_ranged(h1, B2, 1000, 512, 512, ops.EPI_BIAS_RELU_BF16, a, made.bn, kb0, kb1, bias=bias)
    ops.gemm_nt_ranged(h1, B2, 1000, 512, 512, ops.EPI_BIAS_RELU_BF16, b, made.bn, [0] * len(kb0), [8] * len(kb0),
                       bias=bias)
    torch.cuda.synchronize()
    assert torch.equal(a, b)


def test_maf_kd_training_step_runs_through_nfmodel_contract():
    """teacher 10 MADE layers -> student 3 layers, D = 63 (BASELINE config 1) through the same loss code path."""
    from nf_distillation_b200 import functional as Fn
    from nf_distillation_b200.models.maf import create_maf_model
    torch.manual_seed(1)
    teacher = create_maf_model(dict(image_shape=[63], hidden_channels=512, K=10)).cuda()
    student = create_maf_model(dict(image_shape=[63], hidden_channels=512, K=3)).cuda()
    x = torch.randn(512, 63, device="cuda")
    s_z, s_nll, _ = student(x, None)
    with torch.no_grad():
        t_z, _, _ = teacher(x, None)
    kd = Fn.kd_mse([s_z[-1]], [t_z[-1]])
    loss = (0.9 * s_nll + 0.1 * kd).mean()
    loss.backward()
    assert torch.isfinite(loss) and all(p.grad is not None and torch.isfinite(p.grad).all()
                                        for p in student.parameters())
