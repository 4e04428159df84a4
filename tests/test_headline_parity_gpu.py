"""GPU parity of what bench.py times, at the width it times it (hidden 512, every fused-kernel variant).

Three layers of evidence, from the strictest to the loosest:

 1. STAGE-EXACT: every kernel of a FlowStep's forward and backward sequence, fed with the CUDA path's OWN intermediate
    tensors, against plain torch fp32 arithmetic on those same inputs (tools/stage_check.py): fp32 outputs 5e-6, bf16
    outputs identical except for 1-ulp rounding flips on < 5e-4 of the elements (the fp32 value sits on a rounding
    boundary and the two summation orders fall on either side). This is what shows that no kernel hides a bug inside
    the "bf16 rounding" budget.
 2. END-TO-END vs the oracle with `bf16_operands()` (oracle/glow_oracle.py rounds the same tensors at the same places;
    tools/emulation on the CPU shows it IS the exact composition of the stage formulas). The two computations are NOT
    expected to agree to fp32 accuracy: every bf16 rounding turns a 1e-7 summation-order difference into +-1 ulp
    (4e-3) on a fraction of the elements, and the next GEMM spreads that over all its outputs, so rounding decisions
    decorrelate stage after stage (measured: outputs 2e-4..6e-4, gradients up to 1e-2..3e-2 of max|grad| on the
    tensors deepest in the backward chain, 5x below the distance to the fp32 oracle).
 3. END-TO-END vs the fp32 oracle (the reference's arithmetic): the stated tolerances of the bf16-operand mode,
    per-sample bpd / log-det 1e-4 (north_star), KD taps 1e-2, gradients median 1e-2 / worst 0.1 of max|grad|.

Reference: /root/reference/models/flows.py:25-34,142-171 (FlowStep), pl_module.py:198-320,348-382 (KD step, optimiser),
train.py:41-46 (seed, gradient_clip_val=30).
"""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
dev = "cuda"

BOUND_OUT_BF16 = 2e-3      # CUDA vs bf16-operand oracle, relative to max|.| (measured 2e-4 .. 6e-4)
BOUND_GRAD_BF16 = 6e-2     # (measured: <= 3e-2 on block.2 / block.0 weights, <= 2e-3 on everything else)
BOUND_OUT_F32 = 1e-2       # CUDA (bf16 operands) vs fp32 oracle (measured 1e-3 .. 2e-3)
BOUND_LOGDET = 5e-4        # single step, relative to max|logdet| of that step (measured 1e-4 .. 3e-4 vs fp32)


def rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).abs().max() / (b.abs().max() + 1e-12)).item()


def images(B, H, g):
    return torch.floor(torch.rand(B, 3, H, H, generator=g) * 256) / 256 - 0.5


def unpack_mask(m, N):
    """1-bit ReLU mask, word-major [ceil(N/32), M] int32 (ops.relu_mask_like) -> bool [M, N]."""
    words = m.to(torch.int64) & 0xFFFFFFFF
    bits = (words[:, :, None] >> torch.arange(32, device=m.device)[None, None, :]) & 1       # [W, M, 32]
    return bits.permute(1, 0, 2).reshape(m.shape[1], -1)[:, :N].bool()


# ------------------------------------------------------------------------------------------------ one FlowStep
def make_step(C, hid, seed):
    from nf_distillation_b200.models.flows import FlowStep
    torch.manual_seed(seed)
    st = FlowStep(in_channels=C, hidden_channels=hid, actnorm_scale=1.0, flow_permutation="invconv",
                  flow_coupling="affine", LU_decomposed=True)
    for m in st.modules():
        if hasattr(m, "inited"):
            m.inited = True
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for p in st.parameters():
            if p.abs().max() == 0:
                p.copy_(torch.randn(p.shape, generator=g) * 0.05)
    sd = {k: v.clone() for k, v in st.state_dict().items()}
    return st, sd


@pytest.mark.parametrize("C,H,B", [(12, 16, 40), (24, 8, 136), (48, 4, 520)])
def test_flowstep_hidden512_forward_backward_all_fused_variants(C, H, B):
    """One FlowStep at hidden 512 with M = B*H*W >= 8192 pixels, so the fused conv#1 -> conv#2 kernel runs (K1p = 64 /
    128 / 256 for C = 12 / 24 / 48: all three instantiations) in inference AND training mode: z, log-det, the saved
    h1 / h2 / 1-bit ReLU masks, and the gradients of the input and of all 14 parameter tensors (9 of them the coupling
    net's) against the oracle."""
    from oracle import glow_oracle as O
    from nf_distillation_b200 import functional as Fn
    from nf_distillation_b200 import ops
    hid = 512
    assert B * H * H >= 8192 and ops.cnet_fused_supported(hid, ops.round_up(9 * C // 2, 64))
    st, sd = make_step(C, hid, 100 + C)
    g = torch.Generator().manual_seed(C)
    x = torch.randn(B, C, H, H, generator=g)
    ld0 = torch.randn(B, generator=g)
    wz, wl = torch.randn(B, C, H, H, generator=g), torch.randn(B, generator=g)

    def oracle(bf16):
        osd = {k: (v.clone().requires_grad_(True) if v.dtype.is_floating_point and k in dict(st.named_parameters())
                   else v) for k, v in sd.items()}
        xo = x.clone().requires_grad_(True)
        with O.bf16_operands(bf16):
            z, ld = O.flowstep(xo, osd, "", ld0, False)
            ((z * wz).sum() + (ld * wl).sum()).backward()
        return z.detach(), ld.detach(), xo.grad, {k: v.grad for k, v in osd.items() if torch.is_tensor(v) and v.requires_grad}

    z32, ld32, dx32, g32 = oracle(False)
    z16, ld16, dx16, g16 = oracle(True)
    st = st.to(dev)
    # ---- inference mode (frozen-teacher path): fused kernel without h1 / masks
    with torch.no_grad():
        zi, ldi = st(x.to(dev), logdet=ld0.to(dev), reverse=False)
    assert rel(zi, z16) < BOUND_OUT_BF16 and rel(zi, z32) < BOUND_OUT_F32
    assert rel(ldi, ld32) < BOUND_LOGDET and rel(ldi, ld16) < BOUND_LOGDET
    # ---- training mode: the same kernel also stores h1 and the two ReLU masks
    xg = x.to(dev).requires_grad_(True)
    zt, ldt = st(xg, logdet=ld0.to(dev), reverse=False)
    assert torch.equal(zt.detach(), zi), "training and inference kernels must agree bit for bit"
    assert rel(ldt, ldi) < 1e-6      # (per-sample log-det partial sums meet in fp32 atomics: order is not fixed)
    ((zt * wz.to(dev)).sum() + (ldt * wl.to(dev)).sum()).backward()
    assert rel(xg.grad, dx16) < BOUND_GRAD_BF16 and rel(xg.grad, dx32) < 5e-2
    worst16 = worst32 = 0.0
    for n_, p in st.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), n_
        e16, e32 = rel(p.grad, g16[n_]), rel(p.grad, g32[n_])
        assert e16 < BOUND_GRAD_BF16, (n_, e16, e32)
        if not n_.startswith(("block.0.", "block.2.")):      # not behind two re-rounding stages: tight
            assert e16 < 5e-3, (n_, e16, e32)
        worst16, worst32 = max(worst16, e16), max(worst32, e32)
    assert worst32 < 0.1, worst32
    # ---- the saved activations themselves: h1, h2 (bf16) and the masks against the bf16-operand oracle
    with torch.no_grad():
        k = st._consts(False)
        y, _, (col, h1, h2, hsave, m1, m2) = Fn.flowstep2d_forward(x.to(dev), ld0.to(dev), k, hid, keep=True)
        with O.bf16_operands():
            yo, _ = O.actnorm(x, sd["actnorm.bias"], sd["actnorm.logs"], None, False)
            yo, _ = O.invconv(yo, sd, "invconv.", None, False)
            h1o = torch.relu(O.conv_actnorm(yo[:, :C // 2], sd, "block.0.")).to(torch.bfloat16)
            h2o = torch.relu(O.conv_actnorm(h1o.float(), sd, "block.2.")).to(torch.bfloat16)
        pix = lambda t: t.permute(0, 2, 3, 1).reshape(-1, t.shape[1])          # NCHW -> [M, channels]
        for name, a, b, lim in (("h1", h1, pix(h1o), 5e-4), ("h2", h2, pix(h2o), 3e-2)):
            a, b = a.float().cpu(), b.float()
            diff = (a - b).abs()
            # h1: rounding flips only. h2: a flipped h1 element moves all 512 pre-activations of its pixel by ~2e-4,
            # which flips a few per cent of that pixel's h2 roundings — still single ulps (4e-3 of the value)
            assert (diff > 0).float().mean().item() < lim, (name, (diff > 0).float().mean().item())
            assert diff.max().item() <= 1e-2 * b.abs().max().item(), name
        for m, h in ((m1, h1), (m2, h2)):
            assert torch.equal(unpack_mask(m, hid), h > 0), "mask bit <=> stored activation > 0"


@pytest.mark.parametrize("C,H,B", [(12, 16, 40), (24, 8, 136), (48, 4, 520)])
def test_every_kernel_of_a_flowstep_is_exact_on_its_own_inputs(C, H, B):
    """tools/stage_check.py: the 9 forward and 14 backward tensors of FlowStep2dFn at hidden 512 (M >= 8192: fused conv
    kernel, all three K1p variants; CTA-pair dgrads; split-K wgrads), each compared with torch fp32 arithmetic on the
    inputs THAT kernel received. fp32 results agree to summation order; bf16 results are identical except for 1-ulp
    flips on a small fraction of elements. A kernel with a wrong border, mask bit or operand would fail here, whatever
    the end-to-end rounding budget is."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import stage_check
    res = stage_check.run(C, H, B)
    names = [r[0] for r in res]
    for need in ("col", "h1", "h2", "hsave", "z2", "logdet", "dhcol", "dpre2", "dB3", "dpre1", "dB2", "dcol", "dB1",
                 "dx", "dWf", "dbf", "dbias1", "dbias2", "dbias3"):
        assert need in names, need
    for name, err, flips in res:
        if flips is None:
            assert err < 5e-6, (name, err)
        else:
            assert flips < 5e-4 and err < 1e-2, (name, err, flips)      # (err of a flipped element: 1 ulp = 4e-3)


@pytest.mark.parametrize("M,K1p", [(8192, 64), (8200, 128), (33000, 256), (65536, 64)])
def test_cnet_fused_kernel_is_bit_identical_to_the_two_gemms(M, K1p):
    """The fused conv kernel (csrc/cnet_ts.cu, h1 in tensor memory) against the two tcgen05 GEMMs it fuses
    (csrc/gemm_tc.cu): same bf16 products, same fp32 accumulation order per k-block -> h2 (both modes), h1 and both
    masks identical bit for bit; ragged M included."""
    from nf_distillation_b200 import ops
    hid = 512
    g = torch.Generator(device=dev).manual_seed(M + K1p)
    col = (torch.randn(M, K1p, device=dev, generator=g) * 0.5).bfloat16()
    B1 = (torch.randn(hid, K1p, device=dev, generator=g) * 0.1).bfloat16()
    B2 = (torch.randn(hid, hid, device=dev, generator=g) * 0.05).bfloat16()
    b1, b2 = torch.randn(hid, device=dev, generator=g) * 0.1, torch.randn(hid, device=dev, generator=g) * 0.1
    h1a = torch.empty(M, hid, device=dev, dtype=torch.bfloat16)
    h2a = torch.empty_like(h1a)
    m1a, m2a = ops.relu_mask_like(M, hid, dev), ops.relu_mask_like(M, hid, dev)
    ops.gemm_nt(col, B1, M, hid, K1p, ops.EPI_BIAS_RELU_BF16, h1a, bias=b1, aux=m1a)
    ops.gemm_nt(h1a, B2, M, hid, hid, ops.EPI_BIAS_RELU_BF16, h2a, bias=b2, aux=m2a)
    h1b, h2b, h2c = (torch.full_like(h1a, float("nan")) for _ in range(3))
    m1b, m2b = torch.zeros_like(m1a), torch.zeros_like(m2a)
    ops.cnet_fwd_fused(col, K1p, B1, B2, b1, b2, h2b, M, hid, h1=h1b, mask1=m1b, mask2=m2b)
    ops.cnet_fwd_fused(col, K1p, B1, B2, b1, b2, h2c, M, hid)
    assert torch.equal(h2a, h2b) and torch.equal(h2a, h2c) and torch.equal(h1a, h1b)
    assert torch.equal(m1a, m1b) and torch.equal(m2a, m2b)
    ref = torch.relu(col.float() @ B1.float().T + b1).bfloat16()
    assert rel(h1a, ref) < 1e-2


# ------------------------------------------------------------------------------------------------ the KD step
def kd_models(sK, tK, hid, seed=0):
    from nf_distillation_b200.pl_module import NFModel
    from nf_distillation_b200.train import glow_cfg, kd_config, randomise_zero_params
    s_cfg, t_cfg = glow_cfg((32, 32, 3), sK, 3, hid), glow_cfg((32, 32, 3), tK, 3, hid)
    torch.manual_seed(seed)
    m = NFModel(kd_config(s_cfg, t_cfg))
    randomise_zero_params(m.student, seed + 1)
    randomise_zero_params(m.teacher, seed + 2)
    s_sd = {k: v.clone() for k, v in m.student.state_dict().items()}
    t_sd = {k: v.clone() for k, v in m.teacher.state_dict().items()}
    return m, s_cfg, t_cfg, s_sd, t_sd


def oracle_kd_grads(s_sd, s_cfg, t_sd, t_cfg, x, n1, n2, names, bf16):
    from oracle import glow_oracle as O
    sd = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in s_sd.items()}
    with O.bf16_operands(bf16):
        out = O.kd_step(sd, s_cfg, t_sd, t_cfg, x, {"nll": 0.9, "kd": 0.1, "perceptual": 0.0}, n1, n2)
        out["result_loss"].backward()
    return {k: out[k].item() for k in ("nll", "kd", "result_loss")}, {k: sd[k].grad for k in names}, out["student_z"]


def test_kd_step_teacher_k32_student_k8_hidden512_gradients(monkeypatch):
    """BASELINE configs[3] at its real depth and width (teacher K=32, student K=8, L=3, hidden 512), B = 32 (M = 8192
    pixels at level 0: the fused conv kernel's path): loss terms, the student's KD taps and every student gradient
    against the oracle in both arithmetic modes."""
    from nf_distillation_b200.models import utils as U
    m, s_cfg, t_cfg, s_sd, t_sd = kd_models(8, 32, 512)
    names = set(dict(m.student.named_parameters()))
    g = torch.Generator().manual_seed(11)
    B = 32
    x = images(B, 32, g)
    n1, n2 = torch.rand(B, 3, 32, 32, generator=g) / 256, torch.rand(B, 3, 32, 32, generator=g) / 256
    l32, g32, z32 = oracle_kd_grads(s_sd, s_cfg, t_sd, t_cfg, x, n1, n2, names, False)
    l16, g16, z16 = oracle_kd_grads(s_sd, s_cfg, t_sd, t_cfg, x, n1, n2, names, True)
    m.to(dev)
    q = [n1.to(dev), n2.to(dev)]
    monkeypatch.setattr(U, "dequant_noise", lambda t_, n: q.pop(0))
    out = m.training_step([x.to(dev), None], 0)
    out["loss"].backward()
    for k_, r in (("nll", "nll"), ("loss", "result_loss")):
        assert abs(out[k_].item() - l32[r]) < 1e-4 * abs(l32[r]), (k_, out[k_].item(), l32[r])
    assert abs(out["kd"].item() - l32["kd"]) < 1e-2 * abs(l32["kd"])
    assert abs(out["kd"].item() - l16["kd"]) < 1e-3 * abs(l16["kd"])
    assert abs(out["nll"].item() - l16["nll"]) < 1e-5 * abs(l16["nll"])
    errs16, errs32 = [], []
    for n_, p in m.student.named_parameters():
        assert p.grad is not None, n_
        errs16.append((rel(p.grad, g16[n_]), n_))
        errs32.append((rel(p.grad, g32[n_]), n_))
    errs16.sort(); errs32.sort()
    # measured: vs bf16-operand oracle median 1.0e-3 / worst 8e-3; vs fp32 oracle median 2.5e-3 / worst 1.2e-2
    assert errs16[len(errs16) // 2][0] < 3e-3 and errs16[-1][0] < 2.5e-2, (errs16[len(errs16) // 2], errs16[-3:])
    assert errs32[len(errs32) // 2][0] < 1e-2 and errs32[-1][0] < 5e-2, (errs32[len(errs32) // 2], errs32[-1])


# ------------------------------------------------------------------------------------------------ KDTrainer
class StaticNoise:
    """Replaces models.utils.dequant_noise by reads of two static device buffers (student draw, teacher draw), so the
    noise of a CUDA-graph-replayed step can be set from the host before each replay."""

    def __init__(self, shape):
        self.bufs = [torch.zeros(shape, device=dev), torch.zeros(shape, device=dev)]
        self.i = 0

    def __call__(self, x, n_bins):
        b = self.bufs[self.i % 2]
        self.i += 1
        return b

    def set(self, n1, n2):
        self.bufs[0].copy_(n1)
        self.bufs[1].copy_(n2)


def oracle_adam_steps(s_sd, s_cfg, t_sd, t_cfg, xs, noises, names, bf16, lr=5e-4):
    """N reference training steps on the CPU: NFModel.forward/loss (pl_module.py:198-320) -> backward ->
    clip_grad_norm_(30) (train.py:46) -> Adam(lr) (pl_module.py:348-363)."""
    from oracle import glow_oracle as O
    sd = {k: (v.clone().requires_grad_(True) if k in names else v.clone()) for k, v in s_sd.items()}
    params = [sd[k] for k in sd if k in names]
    opt = torch.optim.Adam(params, lr=lr)
    traj = []
    for x, (n1, n2) in zip(xs, noises):
        opt.zero_grad(set_to_none=True)
        with O.bf16_operands(bf16):
            out = O.kd_step(sd, s_cfg, t_sd, t_cfg, x, {"nll": 0.9, "kd": 0.1, "perceptual": 0.0}, n1, n2)
            out["result_loss"].backward()
        torch.nn.utils.clip_grad_norm_(params, 30.0)
        opt.step()
        traj.append([out["nll"].item(), out["kd"].item(), 0.0, out["result_loss"].item()])
    return traj, {k: v.detach() for k, v in sd.items()}


@pytest.mark.parametrize("use_graphs", [True, False])
def test_kdtrainer_graph_replayed_steps_follow_the_oracle_optimiser_trajectory(use_graphs, monkeypatch):
    """train.KDTrainer is what bench.py times: CUDA-graph capture of forward/backward (teacher on a second stream),
    gradient clipping at 30 and Adam, replayed per step. Three steps on three different batches against three oracle
    steps (torch CPU Adam) from the same weights and noise, hidden 512: loss trajectory 1e-4 (kd: 1e-2 vs the fp32
    oracle, 1e-3 vs the bf16-operand oracle), every updated weight tensor within 1e-3 of max|w|, and the UPDATE
    (w_after - w_before) itself against the bf16-operand oracle: cosine >= 0.99 per tensor."""
    from nf_distillation_b200.models import utils as U
    from nf_distillation_b200.train import KDTrainer, glow_cfg, kd_config
    s_cfg, t_cfg = glow_cfg((32, 32, 3), 2, 3, 512), glow_cfg((32, 32, 3), 4, 3, 512)
    B, steps = 32, 3
    noise = StaticNoise((B, 3, 32, 32))
    monkeypatch.setattr(U, "dequant_noise", noise)
    tr = KDTrainer(kd_config(s_cfg, t_cfg), (B, 3, 32, 32), torch.device(dev), use_graphs=use_graphs, seed=42)
    names = set(dict(tr.module.student.named_parameters()))
    s_sd = {k: v.detach().cpu().clone() for k, v in tr.module.student.state_dict().items()}
    t_sd = {k: v.detach().cpu().clone() for k, v in tr.module.teacher.state_dict().items()}
    g = torch.Generator().manual_seed(5)
    xs = [images(B, 32, g) for _ in range(steps)]
    noises = [(torch.rand(B, 3, 32, 32, generator=g) / 256, torch.rand(B, 3, 32, 32, generator=g) / 256)
              for _ in range(steps)]
    traj32, w32 = oracle_adam_steps(s_sd, s_cfg, t_sd, t_cfg, xs, noises, names, False)
    traj16, w16 = oracle_adam_steps(s_sd, s_cfg, t_sd, t_cfg, xs, noises, names, True)
    # capture on a throw-away batch, then restore the initial state: warm-up steps must not count
    tr.x.copy_(xs[0].to(dev))
    noise.set(*noises[0])
    tr.warmup(iters=1)
    tr.reset_state(s_sd)
    got = []
    for x, n in zip(xs, noises):
        noise.set(*n)
        got.append(tr.step(x.pin_memory()).tolist())
    for i in range(steps):
        for j, (name, tol32, tol16) in enumerate((("nll", 1e-4, 1e-4), ("kd", 1e-2, 1e-3), ("perc", 0, 0),
                                                   ("loss", 1e-4, 1e-4))):
            if name == "perc":
                continue
            assert abs(got[i][j] - traj32[i][j]) <= tol32 * abs(traj32[i][j]), (i, name, got[i][j], traj32[i][j])
            assert abs(got[i][j] - traj16[i][j]) <= tol16 * abs(traj16[i][j]), (i, name, got[i][j], traj16[i][j])
    # Updated weights. Three Adam steps move an element by at most ~3 * lr * |m_hat / sqrt(v_hat)| ~ 2e-3, i.e. ~2 % of
    # max|w| of a Xavier conv weight, and elements whose gradient is smaller than its rounding noise take the step in
    # either direction, so "equal weights" is judged on the UPDATE d = w_after - w_before per tensor: relative L2
    # distance and cosine against the bf16-operand oracle's update (and the weights themselves within 2 % of max|w|).
    worst = {"cos": 1.0, "l2": 0.0}
    for n_, p in tr.module.student.named_parameters():
        w = p.detach().cpu()
        assert rel(w, w32[n_]) < 4e-2 and rel(w, w16[n_]) < 4e-2, n_
        du, do = (w - s_sd[n_]).flatten().double(), (w16[n_] - s_sd[n_]).flatten().double()
        assert du.abs().max() > 0, f"{n_} did not move"
        worst["cos"] = min(worst["cos"], (du @ do / (du.norm() * do.norm() + 1e-30)).item())
        worst["l2"] = max(worst["l2"], ((du - do).norm() / (do.norm() + 1e-30)).item())
    print("KDTrainer update vs bf16-operand oracle:", worst)
    assert worst["cos"] > 0.97 and worst["l2"] < 0.25, worst


def test_no_grad_student_calls_see_the_weights_of_graph_replayed_steps(monkeypatch):
    """A graph replay of the optimiser changes parameter VALUES without changing their version counter or storage; the
    cached no-grad operands (fused affine, folded bf16 weights) must not survive it: generate -> N replayed steps ->
    generate equals a freshly built model holding the updated weights."""
    from nf_distillation_b200.models import create_glow_model
    from nf_distillation_b200.train import KDTrainer, glow_cfg, kd_config
    s_cfg, t_cfg = glow_cfg((32, 32, 3), 2, 3, 64), glow_cfg((32, 32, 3), 2, 3, 64)
    B = 16
    tr = KDTrainer(kd_config(s_cfg, t_cfg), (B, 3, 32, 32), torch.device(dev), use_graphs=True, seed=1)
    g = torch.Generator().manual_seed(3)
    tr.x.copy_(images(B, 32, g).to(dev))
    z = torch.randn(4, 48, 4, 4, device=dev) * 0.7
    with torch.no_grad():
        before = tr.module.student(z=z, temperature=0.0, reverse=True)[-1].clone()   # fills the operand caches
        bpd_before = tr.module.student(tr.x.clone(), None)[1].clone()
    tr.warmup(iters=1)
    for _ in range(5):
        tr.step_device()
    torch.cuda.synchronize()
    with torch.no_grad():
        after = tr.module.student(z=z, temperature=0.0, reverse=True)[-1]
        bpd_after = tr.module.student(tr.x.clone(), None)[1]
    fresh = create_glow_model(s_cfg)
    fresh.load_state_dict(tr.module.student.state_dict())
    fresh = fresh.to(dev).eval()
    with torch.no_grad():
        ref = fresh(z=z, temperature=0.0, reverse=True)[-1]
    assert (after - before).abs().max().item() > 1e-4, "five optimiser steps must change the samples"
    assert torch.equal(after, ref), "stale cached operands: no-grad path does not see the replayed updates"
    assert (bpd_after - bpd_before).abs().max().item() > 0


# ------------------------------------------------------------------------------------------------ 1 rank vs N ranks
def _rank_worker(rank, world, port, q, s_sd_path):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from nf_distillation_b200.models import utils as U
    from nf_distillation_b200.train import KDTrainer, glow_cfg, init_distributed, kd_config, shard_batch
    rank, world, device = init_distributed()
    s_cfg, t_cfg = glow_cfg((32, 32, 3), 2, 3, 512), glow_cfg((32, 32, 3), 3, 3, 512)
    GB = 64
    g = torch.Generator().manual_seed(9)
    xg = images(GB, 32, g)
    n1g, n2g = torch.rand(GB, 3, 32, 32, generator=g) / 256, torch.rand(GB, 3, 32, 32, generator=g) / 256
    B = GB // world
    bufs = [shard_batch(n1g, rank, world).to(device), shard_batch(n2g, rank, world).to(device)]
    cnt = [0]

    def noise(x, n_bins):
        cnt[0] += 1
        return bufs[(cnt[0] - 1) % 2]
    U.dequant_noise = noise
    tr = KDTrainer(kd_config(s_cfg, t_cfg), (B, 3, 32, 32), device, use_graphs=True, seed=42)
    init = {k: v.detach().cpu().clone() for k, v in tr.module.student.state_dict().items()}
    tr.x.copy_(shard_batch(xg, rank, world).to(device))
    tr.warmup(iters=1)
    tr.reset_state(init)
    tr.x.copy_(shard_batch(xg, rank, world).to(device))
    tr.step_device()
    torch.cuda.synchronize()
    if rank == 0:
        torch.save({"w": {k: v.detach().cpu() for k, v in tr.module.student.state_dict().items()},
                    "g": tr.flat_grad_view().detach().cpu().clone(), "losses": tr.losses.cpu()}, s_sd_path)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    q.put((rank, "ok"))


def _run_world(world, path):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + (os.getpid() + world * 7) % 2000
    procs = [ctx.Process(target=_rank_worker, args=(r, world, port, q, path)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
        assert p.exitcode == 0
    return torch.load(path)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_one_rank_and_two_ranks_make_the_same_update_on_a_fixed_global_batch(tmp_path):
    """SURVEY §4 / §8e: batch-sharded data parallelism with ONE all-reduce (average) of the student gradients. The same
    global batch and noise on 1 GPU and sharded over 2 GPUs (NCCL): averaged gradient equal to 1e-5 of max|grad|,
    loss scalars 1e-6, and the Adam-updated weights equal to 1e-5 of max|w| (Adam's first step is lr * sign(g) for
    every |g| >> eps, so elements whose gradient is ~0 may differ by up to 2 lr; they are counted, not hidden)."""
    one = _run_world(1, str(tmp_path / "w1.pt"))
    two = _run_world(2, str(tmp_path / "w2.pt"))
    assert rel(two["g"], one["g"]) < 1e-5
    # rank 0's loss scalars are its shard's means; the global mean is checked through the gradient above
    bad = tot = 0
    for k, w1 in one["w"].items():
        if not w1.dtype.is_floating_point:
            continue
        d = (two["w"][k] - w1).abs()
        bad += (d > 1e-5 * (w1.abs().max() + 1e-12)).sum().item()
        tot += d.numel()
        assert d.max().item() <= 2.1 * 5e-4, k
    assert bad <= 1e-4 * tot, (bad, tot)


# ------------------------------------------------------------------------------------------------ fp32-class mode
def rel_l2(a, b):
    a, b = a.detach().double().cpu().flatten(), b.detach().double().cpu().flatten()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


# gradients that reach the loss WITHOUT passing a ReLU mask of this step's coupling net (everything else does)
UNKINKED = ("block.2.actnorm.logs", "block.4.logs", "block.4.conv.weight", "block.4.conv.bias")


@pytest.mark.parametrize("C,H,B", [(12, 16, 40), (24, 8, 20), (48, 4, 37)])
def test_bf16x3_precision_flowstep_matches_the_fp32_oracle(C, H, B):
    """precision="bf16x3" (nf_distillation_b200/precise.py, csrc/split3.cu): every coupling-net operand split into
    h + m bf16 parts, three partial products per GEMM, fp32 accumulation. Against the fp32 oracle (the reference's own
    arithmetic, /root/reference/models/layers.py:209-228): outputs 1e-4 of max|z| and log-det 1e-5 (measured 2e-6 /
    6e-7: fp32 level). Gradients: 5e-5 of max|grad| on every tensor that no ReLU mask separates from the loss; on the
    others a handful of the ~5 M ReLU units have |pre-activation| < 5e-6 and take the other mask than the reference,
    each moving its row of a weight gradient by O(1/sqrt(M)) — held to 5e-3 in relative L2 and 1.5e-2 in max-norm
    (measured 1e-3..3e-3 / 7e-3; the bf16 mode measures 2e-2 / 6e-2 on the same tensors)."""
    from oracle import glow_oracle as O
    st, sd = make_step(C, 512, 300 + C)
    st.precision = "bf16x3"
    g = torch.Generator().manual_seed(C + 1)
    x = torch.randn(B, C, H, H, generator=g)
    ld0 = torch.randn(B, generator=g)
    wz, wl = torch.randn(B, C, H, H, generator=g), torch.randn(B, generator=g)
    names = dict(st.named_parameters())
    osd = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in sd.items()}
    xo = x.clone().requires_grad_(True)
    z32, ld32 = O.flowstep(xo, osd, "", ld0, False)
    ((z32 * wz).sum() + (ld32 * wl).sum()).backward()
    st = st.to(dev)
    xg = x.to(dev).requires_grad_(True)
    zt, ldt = st(xg, logdet=ld0.to(dev), reverse=False)
    ((zt * wz.to(dev)).sum() + (ldt * wl.to(dev)).sum()).backward()
    assert rel(zt, z32) < 1e-4 and rel(ldt, ld32) < 1e-5
    assert rel_l2(xg.grad, xo.grad) < 5e-3 and rel(xg.grad, xo.grad) < 1.5e-2
    for n_, p in st.named_parameters():
        e, e2 = rel(p.grad, osd[n_].grad), rel_l2(p.grad, osd[n_].grad)
        if n_ in UNKINKED:
            assert e < 5e-5, (n_, e, e2)
        else:   # one flipped unit weighs 1/sqrt(M) of a gradient entry summed over M pixels
            assert e < max(1.5e-2, (B * H * H) ** -0.5) and e2 < 5e-3, (n_, e, e2)
    # inverse in the same mode undoes the forward (and the no-grad forward equals the training forward)
    with torch.no_grad():
        zi, ldi = st(x.to(dev), logdet=ld0.to(dev), reverse=False)
        back, ldb = st(zi, logdet=ldi, reverse=True)
    assert torch.equal(zi, zt.detach())
    assert rel(back, x) < 1e-4 and rel(ldb, ld0) < 1e-4


def test_bf16x3_precision_kd_step_taps_and_gradients_at_fp32_level(monkeypatch):
    """The KD training step (teacher K=4, student K=2, L=3, hidden 512, B=16) with both models in bf16x3 mode against
    the fp32 oracle: loss terms 1e-5, the student's KD taps 1e-4 of max|z| (the bf16 mode's bound is 1e-2), student
    gradients 5e-3 in relative L2 and 1.5e-2 in max-norm per tensor, median 5e-4 (ReLU-mask flips, see above; bf16
    mode: median 1e-2, worst 0.1 in max-norm)."""
    from nf_distillation_b200.models import utils as U
    m, s_cfg, t_cfg, s_sd, t_sd = kd_models(2, 4, 512, seed=3)
    m.student.set_precision("bf16x3")
    m.teacher.set_precision("bf16x3")
    names = set(dict(m.student.named_parameters()))
    g = torch.Generator().manual_seed(21)
    B = 16
    x = images(B, 32, g)
    n1, n2 = torch.rand(B, 3, 32, 32, generator=g) / 256, torch.rand(B, 3, 32, 32, generator=g) / 256
    l32, g32, z32 = oracle_kd_grads(s_sd, s_cfg, t_sd, t_cfg, x, n1, n2, names, False)
    m.to(dev)
    q = [n1.to(dev), n2.to(dev)]
    monkeypatch.setattr(U, "dequant_noise", lambda t_, n: q.pop(0))
    fw = m.forward([x.to(dev), None])
    for i in m.student_kd_indices:
        assert rel(fw["student_z"][i], z32[i]) < 1e-4, i
    losses = m.loss(fw)
    losses["result_loss"].backward()
    for k_, r in (("nll", "nll"), ("kd", "kd"), ("result_loss", "result_loss")):
        assert abs(losses[k_].item() - l32[r]) < 1e-5 * abs(l32[r]) + 1e-7, (k_, losses[k_].item(), l32[r])
    errs = sorted((rel(p.grad, g32[n_]), rel_l2(p.grad, g32[n_]), n_) for n_, p in m.student.named_parameters())
    assert errs[-1][0] < 1.5e-2 and max(e[1] for e in errs) < 5e-3 and errs[len(errs) // 2][0] < 5e-4, errs[-3:]


# ------------------------------------------------------------------------------------------------ teacher prefetch
@pytest.mark.parametrize("use_graphs", [True, False])
def test_pipelined_trainer_makes_the_same_updates_as_the_sequential_one(use_graphs, monkeypatch):
    """KDTrainer(pipelined=True) runs the frozen teacher's forward of batch t+1 beside the student's step on batch t.
    The teacher does not depend on the student, so the sequence of updates must be THE SAME as without pipelining:
    three steps on the same batches / noise from the same weights -> identical loss values (shifted by one call) and
    weights equal to fp32 atomics noise."""
    from nf_distillation_b200.models import utils as U
    from nf_distillation_b200.train import KDTrainer, glow_cfg, kd_config
    s_cfg, t_cfg = glow_cfg((32, 32, 3), 2, 3, 128), glow_cfg((32, 32, 3), 3, 3, 128)
    B, steps = 16, 3
    g = torch.Generator().manual_seed(8)
    xs = [images(B, 32, g) for _ in range(steps + 1)]
    noises = [(torch.rand(B, 3, 32, 32, generator=g) / 256, torch.rand(B, 3, 32, 32, generator=g) / 256)
              for _ in range(steps + 1)]
    results = {}
    for mode in ("plain", "pipelined"):
        noise = StaticNoise((B, 3, 32, 32))
        monkeypatch.setattr(U, "dequant_noise", noise)
        tr = KDTrainer(kd_config(s_cfg, t_cfg), (B, 3, 32, 32), torch.device(dev), use_graphs=use_graphs, seed=42,
                       pipelined=(mode == "pipelined"))
        assert tr.pipelined == (mode == "pipelined")
        init = {k: v.detach().cpu().clone() for k, v in tr.module.student.state_dict().items()}
        tr.x.copy_(xs[0].to(dev)); noise.set(*noises[0])
        tr.warmup(iters=1)
        tr.reset_state(init)
        losses, g1 = [], None
        if mode == "pipelined":
            tr.x.copy_(xs[0].to(dev)); noise.set(*noises[0]); noise.i = 0
            tr.prime()                                          # stage batch 0
        for t in range(steps):
            nxt = t + (mode == "pipelined")                     # pipelined: train on batch t while staging batch t + 1
            noise.set(*noises[nxt])
            losses.append(tr.step(xs[nxt].pin_memory()).tolist())
            if t == 0:
                g1 = tr.flat_grad_view().detach().cpu().clone()
        torch.cuda.synchronize()
        results[mode] = (losses, {k: v.detach().cpu().clone() for k, v in tr.module.student.state_dict().items()}, g1)
    # step 1 starts from identical weights: identical losses up to atomics order; later steps inherit the (Adam-
    # normalised) run-to-run noise of the earlier updates, measured at ~1e-5 of the kd term
    for i, (a, b) in enumerate(zip(results["plain"][0], results["pipelined"][0])):
        for u, v in zip(a, b):
            assert abs(u - v) <= (2e-6 if i == 0 else 1e-4) * abs(u) + 1e-8, (results["plain"][0], results["pipelined"][0])
    # first step: the same weights see the same batch -> the same gradient (fp32 atomics order aside)
    assert rel(results["pipelined"][2], results["plain"][2]) < 1e-5
    # after three Adam steps: Adam divides by sqrt(v), so an element whose gradient is small against the 1e-5 * max|g|
    # run-to-run noise of the fp32 atomics gets a visibly different normalised step (two runs of the SAME mode differ
    # the same way); the weights agree to a tenth of one step size on all but a handful of elements
    bad = tot = 0
    lr = 5e-4
    for k, w in results["plain"][1].items():
        if w.dtype.is_floating_point:
            d = (results["pipelined"][1][k] - w).abs()
            bad += (d > 0.1 * lr).sum().item()
            tot += d.numel()
            assert d.max().item() <= 2.1 * lr * steps, k
    assert bad <= 1e-2 * tot, (bad, tot)


@pytest.mark.parametrize("M,K3p", [(8192, 128), (8200, 256), (33000, 448), (65536, 128)])
def test_cnet_bwd_fused_kernel_matches_the_two_masked_gemms(M, K3p):
    """csrc/cnet_ts.cu in backward mode (both dgrads of the coupling net's chain in one kernel) against the two
    tcgen05 GEMMs with the ReLU-mask epilogue it replaces: same bf16 products, same k-block order -> dpre2 and dpre1
    identical bit for bit (ragged M included); the bias-gradient column sums agree to fp32 summation order."""
    from nf_distillation_b200 import ops
    hid = 512
    g = torch.Generator(device=dev).manual_seed(M + K3p)
    dhcol = (torch.randn(M, K3p, device=dev, generator=g) * 0.5).bfloat16()
    B3T = (torch.randn(hid, K3p, device=dev, generator=g) * 0.1).bfloat16()
    B2T = (torch.randn(hid, hid, device=dev, generator=g) * 0.05).bfloat16()
    m2 = torch.randint(-2 ** 31, 2 ** 31 - 1, (hid // 32, M), device=dev, generator=g, dtype=torch.int32)
    m1 = torch.randint(-2 ** 31, 2 ** 31 - 1, (hid // 32, M), device=dev, generator=g, dtype=torch.int32)
    d2a, d1a = torch.empty(M, hid, device=dev, dtype=torch.bfloat16), torch.empty(M, hid, device=dev, dtype=torch.bfloat16)
    b2a, b1a = torch.zeros(hid, device=dev), torch.zeros(hid, device=dev)
    ops.gemm_nt(dhcol, B3T, M, hid, K3p, ops.EPI_MASK_BF16, d2a, aux=m2, colsum=b2a)
    ops.gemm_nt(d2a, B2T, M, hid, hid, ops.EPI_MASK_BF16, d1a, aux=m1, colsum=b1a)
    d2b, d1b = torch.full_like(d2a, float("nan")), torch.full_like(d1a, float("nan"))
    b2b, b1b = torch.zeros(hid, device=dev), torch.zeros(hid, device=dev)
    ops.cnet_bwd_fused(dhcol, K3p, B3T, B2T, m2, m1, d2b, d1b, b2b, b1b, M, hid)
    assert torch.equal(d2a, d2b) and torch.equal(d1a, d1b)
    assert rel(b2b, b2a) < 1e-5 and rel(b1b, b1a) < 1e-5
    ref = (dhcol.float() @ B3T.float().T) * unpack_mask(m2, hid)
    assert rel(d2b, ref.bfloat16()) < 1e-2 and rel(b2b, d2b.float().sum(0)) < 1e-5
