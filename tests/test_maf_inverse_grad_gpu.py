"""GPU: gradients through the sequential MADE inverse (the perceptual L1 term of the KD loss for MAF students).

The checker is torch.autograd through the paper restatement's inverse (oracle/maf_oracle.py), fp32 on the CPU. The
product evaluates the network on bf16 tensor-core operands with fp32 accumulation and rounds dout, g2, g1 to bf16 as
the dgrad GEMM epilogues do. Input gradients hold 1e-2 of max as in test_maf_gpu.py (measured <= 1.7e-3). Parameter
gradients hold cosine >= 0.995 and 0.25 of max (measured worst: cosine 0.9977, 0.18 of max, fc2.weight at D = 6,
B = 300), looser than the forward MADE tests' 0.999 / 0.1. The cause is the upstream: random-sign g_x make a
parameter gradient a sum of B terms that largely cancel (~sqrt(B) x a term). The few hidden units whose
pre-activation sits within bf16 rounding of zero take the other ReLU branch in the bf16 network than in the fp32
restatement, and those whole terms do not cancel, so their share does not shrink with B (B = 20 000 measures the same
as B = 257). The coherent upstream of the forward tests sums to ~B x a term and hides them. The resident solve and the
D-pass solve carry the same operands and masks, and they agree to 1e-3 of max and cosine 0.99999 (measured: to 6
digits). That is the tight check of the new kernel."""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
dev = "cuda"


def rel(a, b):
    b = b.to(a.device)
    return ((a - b).abs().max() / (b.abs().max() + 1e-12)).item()


def cos(a, b):
    return torch.nn.functional.cosine_similarity(a.flatten().double().cpu(), b.flatten().double().cpu(), dim=0).item()


SHAPES = [(6, 512, 300, True), (63, 512, 257, True), (63, 192, 64, True), (63, 512, 20000, True),
          (1, 64, 33, True), (2, 64, 16, False), (100, 64, 50, True), (17, 128, 1, True), (63, 512, 257, False)]


def made_layer(D, H, flip):
    from nf_distillation_b200.models.maf import MADE
    torch.manual_seed(D * 7 + H)
    made = MADE(D, H, flip=flip)
    with torch.no_grad():
        made.fc3.bias.normal_(0, 0.1)
    return made


def inverse_grads(made, u, ld0, gx, gld):
    """(x, ld, g_u, g_ld_in, {param: grad}) of <x, gx> + <ld, gld> through made's inverse."""
    for p in made.parameters():
        p.grad = None
    uu, ll = u.clone().requires_grad_(True), ld0.clone().requires_grad_(True)
    x, ld = made(uu, logdet=ll, reverse=True)
    ((x * gx).sum() + (ld * gld).sum()).backward()
    return (x.detach(), ld.detach(), uu.grad, ll.grad,
            {n: p.grad.detach().clone() for n, p in made.named_parameters()})


def layer_case(D, H, B, flip, coherent=False):
    """Autograd through the restatement's inverse and both product solves for one layer: (made, no-grad x, no-grad
    ld, g_ld, oracle u (its .grad), oracle parameters (their .grad), {resident?: inverse_grads(...)}).
    coherent: g_x = g_ld = 1."""
    from oracle import maf_oracle as MO
    made = made_layer(D, H, flip)
    sd = {"l." + k: v.clone() for k, v in made.state_dict().items()}
    g = torch.Generator().manual_seed(B + D)
    u, gx, gld, ld0 = (torch.randn(B, D, generator=g), torch.randn(B, D, generator=g), torch.randn(B, generator=g),
                       torch.randn(B, generator=g))
    if coherent:
        gx, gld = torch.ones(B, D), torch.ones(B)
    uo = u.clone().requires_grad_(True)
    p = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    xo, sa = MO.made_inverse(uo, p, "l.", D, flip=flip)
    ((xo * gx).sum() + (sa * gld).sum()).backward()
    made = made.cuda()
    with torch.no_grad():
        x_ng, ld_ng = made(u.cuda(), logdet=ld0.cuda(), reverse=True)
    res = {}
    for resident in (True, False):
        made.resident_inverse = resident
        res[resident] = inverse_grads(made, u.cuda(), ld0.cuda(), gx.cuda(), gld.cuda())
    made.resident_inverse = True
    return made, x_ng, ld_ng, gld, uo, p, res


def error_table(uo, p, res):
    table = []
    for resident, (x, ld, g_u, g_ld, gp) in res.items():
        row = {"solve": "resident" if resident else "D-pass", "g_u": rel(g_u, uo.grad)}
        for n, v in gp.items():
            row[n] = (rel(v, p["l." + n].grad), cos(v, p["l." + n].grad))
        table.append(row)
    return table


@pytest.mark.parametrize("D,H,B,flip", SHAPES)
def test_inverse_layer_gradients_match_autograd(D, H, B, flip):
    """One MADE layer's inverse with g_x and g_ld: g_u, g_ld_in and every parameter gradient against autograd through
    the restatement, on the resident solve and on the D-pass solve; the two solves against each other; x from the
    gradient path bit-identical to the no-grad inverse."""
    made, x_ng, ld_ng, gld, uo, p, res = layer_case(D, H, B, flip)
    assert made._inverse_bwd_jobs(x_ng.device) is not None
    for resident, (x, ld, g_u, g_ld, gp) in res.items():
        if resident:
            assert torch.equal(x, x_ng) and torch.equal(ld, ld_ng)
        assert torch.equal(g_ld, gld.cuda())
    table = error_table(uo, p, res)
    print("\n(D, H, B, flip) =", (D, H, B, flip), *table, sep="\n  ")
    for row in table:
        assert row["g_u"] < 1e-2, row
        for n, v in row.items():
            if isinstance(v, tuple):
                ref = p["l." + n].grad
                if ref.abs().max() == 0:   # D = 1: nothing reaches the hidden weights
                    assert res[row["solve"] == "resident"][4][n].abs().max() == 0, n
                    continue
                assert v[0] < 0.25 and v[1] > 0.995, (row["solve"], n, v)
    # resident vs D-pass: the same bf16 operands and masks, another summation order
    a, b = res[True], res[False]
    assert rel(a[2], b[2]) < 1e-3
    for n in a[4]:
        if b[4][n].abs().max() > 0:
            assert cos(a[4][n], b[4][n]) > 0.99999 and rel(a[4][n], b[4][n]) < 1e-3, n


@pytest.mark.parametrize("D,H,B,flip", [(6, 512, 300, True), (63, 512, 257, True), (63, 512, 20000, True),
                                        (63, 512, 257, False)])
def test_coherent_upstream_holds_the_forward_tests_bound(D, H, B, flip):
    """With a coherent upstream (g_x = g_ld = 1, like the forward MADE tests' nll mean) the per-sample terms of a
    parameter gradient add instead of cancelling, and the bound of the forward MADE gradient tests holds: g_u 1e-2 of
    max, parameters cosine >= 0.999 and 0.1 of max. The looser parameter bound of the random-sign test above comes
    from cancellation alone."""
    _, _, _, _, uo, p, res = layer_case(D, H, B, flip, coherent=True)
    table = error_table(uo, p, res)
    print("\ncoherent upstream, (D, H, B, flip) =", (D, H, B, flip), *table, sep="\n  ")
    for row in table:
        assert row["g_u"] < 1e-2, row
        for n, v in row.items():
            if isinstance(v, tuple):
                assert v[0] < 0.1 and v[1] > 0.999, (row["solve"], n, v)


def test_trainable_inverse_reads_the_current_weights():
    """The gradient path of the inverse builds its operands from the parameters on every call: after the weights are
    written without a version bump (as FlatAdam's flat-buffer update does), its x equals the no-grad inverse of a
    module whose derived-operand caches were dropped, on the resident and on the D-pass inverse."""
    from nf_distillation_b200 import functional as Fn
    made = made_layer(63, 512, True).cuda()
    u = torch.randn(512, 63, device=dev, generator=torch.Generator(device=dev).manual_seed(2))
    for resident in (True, False):
        made.resident_inverse = resident
        x1, _ = made(u, reverse=True)
        assert x1.grad_fn is not None
        with torch.no_grad():
            for q in made.parameters():
                q.data.mul_(0.9)       # (.data: the parameter's version counter does not move)
        x2, _ = made(u, reverse=True)
        Fn.bump_param_epoch()
        with torch.no_grad():
            x_ref, _ = made(u, reverse=True)
        assert not torch.equal(x1, x_ref), resident
        assert torch.equal(x2.detach(), x_ref), resident


@pytest.mark.parametrize("resident", [True, False])
def test_solve_agrees_with_the_forward_chain(resident):
    """The identity of the reverse solve: the forward's parameter chain run from the solve's dout has the input
    gradient -g_x (its network part is c = mubar - g_x), and dout's padding columns are zero."""
    from nf_distillation_b200.models.maf import _made_grad_arena, _made_net_backward
    D, H, B = 63, 512, 4096
    made = made_layer(D, H, True).cuda()
    made.resident_inverse = resident
    g = torch.Generator(device=dev).manual_seed(3)
    u, gx, gld = (torch.randn(B, D, device=dev, generator=g), torch.randn(B, D, device=dev, generator=g),
                  torch.randn(B, device=dev, generator=g))
    with torch.no_grad():
        x, _ = made(u, reverse=True)
        params = made._params()
        ops_ = made._operands(params, True)
        xb = made._bf16_rows(x, None)
        h1, h2, out, m1, m2 = made._net(xb, B, ops_, params[1], params[3], keep=True)
        grads = _made_grad_arena(made, x.device)
        g_u, dout = torch.empty_like(x), torch.full((B, made.N3p), 7.0, device=dev, dtype=torch.bfloat16)
        made._inverse_solve(gx, gld, u, out, m1, m2, ops_, True, g_u, dout, grads[0])
        dxn, *_ = _made_net_backward(made, dout, xb, h1, h2, m1, m2, ops_[1], ops_[3], ops_[5], grads, True)
        torch.cuda.synchronize()
    assert torch.equal(dout[:, 2 * D:], torch.zeros_like(dout[:, 2 * D:]))
    mub = dout[:, :D].float()
    chain_dx = dxn[:, :D] - mub
    print("\nidentity: max|chain dx + g_x| / max|g_x| = %.2e" % rel(chain_dx, -gx))
    assert rel(chain_dx, -gx) < 2e-2
    assert rel(grads[0][:2 * D], dout[:, :2 * D].float().sum(0)) < 1e-2


def test_latent_without_grad_still_trains_the_student():
    """Silent-detach regression: a latent that does not require grad, trainable parameters -> x carries a grad_fn and
    x.sum().backward() reaches every MADE parameter."""
    from nf_distillation_b200.models.maf import create_maf_model
    torch.manual_seed(0)
    m = create_maf_model(dict(image_shape=[63], hidden_channels=512, K=3)).cuda()
    latent = torch.randn(512, 63, device=dev)
    assert not latent.requires_grad
    x = m(z=latent, reverse=True)[-1]
    assert x.grad_fn is not None
    x.sum().backward()
    for n, p in m.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all() and p.grad.abs().max() > 0, n


def maf_pair(perceptual, seed=0):
    from nf_distillation_b200.pl_module import NFModel
    from nf_distillation_b200.train import glow_cfg, kd_config
    s_cfg, t_cfg = glow_cfg((63,), 3, 1, 512, is_1d=True, y_classes=0), glow_cfg((63,), 10, 1, 512, is_1d=True, y_classes=0)
    s_cfg["architecture"] = t_cfg["architecture"] = "maf"
    torch.manual_seed(seed)
    return NFModel(kd_config(s_cfg, t_cfg, data="bsds300", nll=0.85, kd=0.05, perceptual=perceptual))


def test_kd_step_with_perceptual_weight_matches_oracle_draw_for_draw(monkeypatch):
    """MAF student (3 layers) and teacher (10), weights 0.85 / 0.05 / 0.1, both inverse passes fed one fixed latent
    (gaussian_sample monkeypatched). The nll / kd terms and the student gradients without the perceptual term are
    the MAF KD step other tests hold to the restatement; here the perceptual scalar is compared with the L1 between
    the restatement's two inverse passes, the loss with the weighted sum, and the perceptual share of every student
    gradient (grad at 0.1 minus grad at 0) with 0.1 x the restatement's autograd gradient of that L1."""
    from nf_distillation_b200 import pl_module
    from oracle import maf_oracle as MO
    B, D = 256, 63
    x = torch.randn(B, D, generator=torch.Generator().manual_seed(5))
    latent = torch.randn(B, D, generator=torch.Generator().manual_seed(6))
    monkeypatch.setattr(pl_module, "gaussian_sample", lambda mean, logs, t: latent.to(mean.device))
    scal, grads = {}, {}
    for wp in (0.1, 0.0):
        m = maf_pair(wp)
        s_sd = {k: v.clone() for k, v in m.student.state_dict().items()}
        t_sd = {k: v.clone() for k, v in m.teacher.state_dict().items()}
        m.to(dev)
        out = m.training_step([x.to(dev), None], 0)
        out["loss"].backward()
        torch.cuda.synchronize()
        scal[wp] = {k: v.item() for k, v in out.items()}
        grads[wp] = {n: p.grad.detach().cpu().clone() for n, p in m.student.named_parameters()}
        assert all(p.grad is None for p in m.teacher.parameters())
    sd = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and k != "prior_h" else v) for k, v in s_sd.items()}
    sx = MO.maf_inverse(sd, D, 3, latent)
    with torch.no_grad():
        tx = MO.maf_inverse(t_sd, D, 10, latent)
    perc = (sx - tx).abs().mean(1).mean()
    perc.backward()
    p_, p0 = scal[0.1], scal[0.0]
    print("\nproduct:", p_, "\noracle perceptual:", perc.item())
    assert p0["perceptual"] == 0.0 and perc.item() > 0
    assert abs(p_["perceptual"] - perc.item()) < 1e-2 * perc.item()
    for k in ("nll", "kd"):
        assert abs(p_[k] - p0[k]) <= 1e-5 * abs(p0[k]), k
    assert abs(p_["loss"] - p0["loss"] - 0.1 * p_["perceptual"]) < 1e-4 * abs(p_["loss"])
    errs = []
    for n in grads[0.1]:
        d_p, d_o = grads[0.1][n] - grads[0.0][n], 0.1 * sd[n].grad
        errs.append((rel(d_p, d_o), cos(d_p, d_o), n))
    errs.sort()
    print("perceptual share of the student gradients: worst", errs[-1], "median", errs[len(errs) // 2])
    assert all(c > 0.99 and r < 0.1 for r, c, _ in errs), errs[-3:]


def test_kd_trainer_trains_maf_with_perceptual_weight(monkeypatch):
    """KDTrainer with the MAF pair at perceptual 0.1, captured and eager, both after the default three eager warm-up
    steps (which change the weights before the capture): four steps from the same initial student. Finite losses, a
    non-zero perceptual term, every student parameter moves. Fed one fixed latent, the two trainers report the same
    losses at every step and end at the same parameters; a captured graph that reused operands derived from the
    warm-up weights would compute the student's sample, hence the perceptual term, from stale weights."""
    from nf_distillation_b200 import pl_module
    from nf_distillation_b200.train import KDTrainer, glow_cfg, kd_config
    s_cfg, t_cfg = glow_cfg((63,), 3, 1, 512, is_1d=True, y_classes=0), glow_cfg((63,), 10, 1, 512, is_1d=True, y_classes=0)
    s_cfg["architecture"] = t_cfg["architecture"] = "maf"
    B, steps = 1024, 4
    cfg = kd_config(s_cfg, t_cfg, data="bsds300", nll=0.85, kd=0.05, perceptual=0.1)
    xin = torch.randn(B, 63, generator=torch.Generator().manual_seed(4)).to(dev)
    latent = torch.randn(B, 63, generator=torch.Generator().manual_seed(6)).to(dev)
    monkeypatch.setattr(pl_module, "gaussian_sample", lambda mean, logs, t: latent)
    losses, moved = {}, {}
    for graphs in (True, False):
        tr = KDTrainer(cfg, (B, 63), torch.device(dev), use_graphs=graphs, seed=5, pipelined=False)
        tr.x.copy_(xin)
        p0 = tr.opt.p.detach().clone()
        tr.warmup()
        assert (tr.g_fb is not None) == graphs
        tr.opt.p.copy_(p0)
        tr.reset_state()
        before = {n: p.detach().clone() for n, p in tr.module.student.named_parameters()}
        losses[graphs] = []
        for _ in range(steps):
            tr.step_device()
            losses[graphs].append(tr.losses.cpu())
        torch.cuda.synchronize()
        for l_ in losses[graphs]:
            assert torch.isfinite(l_).all() and l_[2].item() > 0, l_
        for n, p in tr.module.student.named_parameters():
            assert not torch.equal(p.detach(), before[n]), f"{n} did not change"
        moved[graphs] = tr.opt.p.detach() - p0
    lg, le = torch.stack(losses[True]), torch.stack(losses[False])
    dl = ((lg - le).abs() / le.abs()).max(0).values
    print("\ngraphed vs eager over %d steps: losses (nll, kd, perceptual, loss) rel %s; parameters moved rel %.2e "
          "cos %.7f" % (steps, dl.tolist(), rel(moved[True], moved[False]), cos(moved[True], moved[False])))
    # measured 1.2e-7; operands derived from the warm-up weights put the perceptual term off by 2.3e-3
    assert dl.max().item() < 1e-5, dl
    # The parameters moved are compared by direction: Adam moves an element with a near-zero gradient by ~ +-lr, its
    # sign set by the order of the split-K atomics, so their max-norm difference (measured 0.27 of the largest move,
    # at cosine 0.9999991) is no measure of the trajectory; the per-step losses above are
    assert cos(moved[True], moved[False]) > 0.99999
