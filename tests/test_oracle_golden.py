"""CPU: the oracle restatement (oracle/glow_oracle.py) must reproduce the vectors recorded from the unmodified
reference (tests/golden/, made by oracle/make_golden.py). fp32, tolerance 1e-5 relative on tensors, 1e-6 on bpd."""
import os
import sys

import pytest
import torch

from golden_util import cfg_of, load, state_dict_of, t

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import glow_oracle as O  # noqa: E402

FWD = ["glow2d_cifar_k2_h64", "glow2d_16_k1_h64", "glow1d_d6_k5_h32", "glow1d_d63_k5_h32",
       "glow2d_16_additive_shuffle_k2_h64", "glow2d_16_affine_reverse_k2_h64", "glow2d_16_learntop_k1_h64"]


def close(a, b, rtol=1e-5, atol=None):
    scale = b.abs().max().item() + 1e-12
    atol = atol if atol is not None else rtol * scale
    err = (a - b).abs().max().item()
    assert err <= atol, f"max err {err:.3e} > {atol:.3e} (scale {scale:.3e})"


@pytest.mark.parametrize("name", FWD)
def test_forward_matches_reference(name):
    d = load(name)
    cfg, sd = cfg_of(d), state_dict_of(d)
    x = t(d["x"])
    noise = None if cfg["is_1d"] else t(d["noise"])
    outs, bpd = O.glow_forward(sd, cfg, x, noise)
    n = sum(1 for k in d if k.startswith("out."))
    assert len(outs) == n
    for i, o in enumerate(outs):
        close(o, t(d[f"out.{i}"]))
    close(bpd, t(d["bpd"]), rtol=2e-6)


@pytest.mark.parametrize("name", FWD)
def test_reverse_matches_reference(name):
    d = load(name)
    cfg, sd = cfg_of(d), state_dict_of(d)
    n = sum(1 for k in d if k.startswith("out."))
    z = t(d[f"out.{n - 1}"])
    rev = O.glow_reverse(sd, cfg, z, temperature=0.0)
    assert len(rev) == int(d["rev_n"])
    close(rev[-1], t(d["rev_last"]), rtol=2e-4)


@pytest.mark.parametrize("name", FWD)
def test_step_logdets(name):
    d = load(name)
    cfg, sd = cfg_of(d), state_dict_of(d)
    x = t(d["x"]) if cfg["is_1d"] else t(d["x"]) + t(d["noise"])
    inp = x
    for i, (kind, C, H, W) in enumerate(O.layer_plan(cfg)):
        out = t(d[f"out.{i}"])
        if f"step.{i}.logdet_fwd" in d:
            B = x.shape[0]
            kw = dict(coupling=cfg.get("flow_coupling", "affine"), perm=O.step_perm(cfg, i))
            z, ld = O.flowstep(inp, sd, f"flow.layers.{i}.", torch.zeros(B), False, **kw)
            close(ld, t(d[f"step.{i}.logdet_fwd"]), rtol=1e-5)
            back, ld_r = O.flowstep(z, sd, f"flow.layers.{i}.", torch.zeros(B), True, **kw)
            close(ld_r, t(d[f"step.{i}.logdet_rev"]), rtol=1e-5)
            close(back, t(d[f"step.{i}.roundtrip"]), rtol=1e-4)
            close(ld + ld_r, torch.zeros(B), atol=1e-3 * (ld.abs().max().item() + 1))
        inp = out


@pytest.mark.parametrize("name", ["kd2d_cifar_t4_s2_h64", "kd1d_d63_t5_s3", "kd1d_rich_t2_s2"])
def test_kd_step_matches_reference(name):
    import json
    d = load(name)
    s_cfg, t_cfg = cfg_of(d, "s_cfg"), cfg_of(d, "t_cfg")
    s_sd, t_sd = state_dict_of(d, "s_sd."), state_dict_of(d, "t_sd.")
    weights = json.loads(str(d["weights"]))
    s_idx, t_idx = O.kd_indices(s_cfg, t_cfg)
    assert s_idx == list(d["s_idx"]) and t_idx == list(d["t_idx"])
    for v in s_sd.values():
        if v.dtype.is_floating_point:
            v.requires_grad_(True)
    latent = t(d["latent"]) if "latent" in d else None
    cond = t(d["cond"]) if "cond" in d else None             # RICH-shaped fixture: [x, cond, weights] batches
    sw = t(d["sample_w"]) if "sample_w" in d else None
    out = O.kd_step(s_sd, s_cfg, t_sd, t_cfg, t(d["x"]), weights, t(d["noise_s"]), t(d["noise_t"]), latent,
                    y_onehot=cond, sample_weights=sw)
    for key, ref in (("nll", "nll"), ("kd", "kd"), ("perceptual", "perceptual"), ("result_loss", "loss")):
        close(out[key].detach(), t(d[ref]), rtol=1e-5)
    for i in s_idx:
        close(out["student_z"][i].detach(), t(d[f"student_z.{i}"]))
    out["result_loss"].backward()
    checked = 0
    for k, v in s_sd.items():
        if v.requires_grad and ("grad." + k) in d:
            g = v.grad if v.grad is not None else torch.zeros_like(v)
            close(g, t(d["grad." + k]), rtol=2e-3, atol=2e-3 * (t(d["grad." + k]).abs().max().item() + 1e-8))
            checked += 1
    assert checked > 10


def test_bf16_operand_mode_rounds_only_the_coupling_gemm_operands():
    """oracle.glow_oracle.bf16_operands(): the mode the GPU tests use to separate operand rounding from bugs. It must
    (a) leave everything outside the 2-D coupling net untouched (1-D models, Split2d, prior: bit-identical to fp32),
    (b) stay within bf16 rounding of the fp32 mode on the golden fixture (outputs 1e-2, bpd 1e-4), and (c) round
    forward values only at the documented places: h1 / h2 of a FlowStep are exactly representable in bf16."""
    import torch.nn.functional as F  # noqa: F401
    d = load("glow2d_cifar_k2_h64")
    cfg, sd = cfg_of(d), state_dict_of(d)
    x, noise = t(d["x"]), t(d["noise"])
    o32, b32 = O.glow_forward(sd, cfg, x, noise)
    with O.bf16_operands():
        o16, b16 = O.glow_forward(sd, cfg, x, noise)
        z1 = o32[0][:, :6]
        h1 = torch.relu(O.conv_actnorm(z1, sd, "flow.layers.1.block.0."))
        h1q = O._q(h1)
    assert torch.equal(h1q, h1q.bfloat16().float()) and not torch.equal(h1, h1q)
    assert ((b16 - b32).abs() / b32.abs()).max() < 1e-4
    for a, b in zip(o16, o32):
        assert ((a - b).abs().max() / b.abs().max()).item() < 1e-2
    assert any(not torch.equal(a, b) for a, b in zip(o16, o32))
    # gradients flow through the rounding (straight-through) and stay close to the fp32 ones
    names = [k for k, v in sd.items() if v.dtype.is_floating_point and k != "prior_h" and not k.endswith(("invconv.p", "sign_s"))]
    g = {}
    for mode in (False, True):
        s2 = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in sd.items()}
        with O.bf16_operands(mode):
            O.glow_forward(s2, cfg, x, noise)[1].mean().backward()
        g[mode] = {k: s2[k].grad for k in names}
    errs = sorted(((g[True][k] - g[False][k]).abs().max() / (g[False][k].abs().max() + 1e-12)).item() for k in names)
    assert errs[len(errs) // 2] < 1e-2 and errs[-1] < 0.3
    # 1-D model: no tensor-core path, the mode must be a no-op
    d1 = load("glow1d_d6_k5_h32")
    cfg1, sd1 = cfg_of(d1), state_dict_of(d1)
    a = O.glow_forward(sd1, cfg1, t(d1["x"]))[1]
    with O.bf16_operands():
        b = O.glow_forward(sd1, cfg1, t(d1["x"]))[1]
    assert torch.equal(a, b)
