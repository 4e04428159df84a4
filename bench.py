#!/usr/bin/env python
"""Benchmark of the KD training hot path (BASELINE.json: "KD-train samples/sec (Glow 32x32x3, ...); logp delta").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B | --global-batch G] [--impl reference]
                    [--workload NAME] [--dump-outputs DIR]

One process per GPU (torchrun for N > 1). A step = one KD training step (student fwd, teacher fwd, multi-level
latent MSE, backward, clip 30, Adam) on one synthetic CIFAR-shaped batch per rank, from the seeded initial student.
Prints ONE JSON line.

--impl reference times the reference's CPU algorithm (oracle/ port; the reference is a Python script tree that does not
travel to the GPU box) and imports NOTHING from the product package.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: image shape, L, hidden, teacher K, student K, per-GPU batch, dtype = the arithmetic type of the GEMM operands
    # per-GPU batch 2048 (weak scaling). The reference's config uses 64 (conf/training/cifar.yaml:7) on its single
    # GPU (--batch 64 measures that point); throughput on synthetic data is quoted at a batch that fills a B200.
    "glow_cifar_kd_t32_s8": dict(image=(32, 32, 3), L=3, hidden=512, tK=32, sK=8, batch=2048, dtype="bf16"),
    # BASELINE configs[4]: Glow L=4 K=32 on CelebA-shaped 64x64x3, KD training (level-0 GEMM shape of batch 256 equals
    # CIFAR at batch 1024: 262 144 pixels)
    "glow_celeba_kd_t32_s8": dict(image=(64, 64, 3), L=4, hidden=512, tK=32, sK=8, batch=256, dtype="bf16"),
    # the reference's own CelebA pair (conf/teacher/celeba.yaml, conf/student/celeba.yaml): L=3, teacher K=32 hidden
    # 512, student K=16 hidden 256
    "glow_celeba_ref_kd_t32h512_s16h256": dict(image=(64, 64, 3), L=3, hidden=512, s_hidden=256, tK=32, sK=16,
                                               batch=256, dtype="bf16"),
    # BASELINE configs[2]: Glow L=3 K=32 hidden 512, forward + inverse + log-det (no gradients); metric = samples/s
    # through one x -> z (+ per-sample log-det / bpd) pass followed by one z -> x sampling pass
    "glow_cifar_fwd_inv_k32": dict(image=(32, 32, 3), L=3, hidden=512, tK=32, sK=32, batch=1024, mode="fwd_inv",
                                   dtype="bf16"),
    "glow_celeba_fwd_inv_k32": dict(image=(64, 64, 3), L=4, hidden=512, tK=32, sK=32, batch=256, mode="fwd_inv",
                                    dtype="bf16"),
    # MAF density evaluation + sampling: 10 MADE layers, D = 63, hidden 512; the z -> x pass is the shared-memory-
    # resident sequential inverse (csrc/maf_inverse.cu), one launch per layer
    "maf_bsds300_fwd_inv_k10": dict(image=(63,), L=1, hidden=512, tK=10, sK=10, batch=65536, is_1d=True, arch="maf",
                                    mode="fwd_inv", data="bsds300", dtype="bf16"),
    # secondary workloads (BASELINE configs[1]): BSDS300-shaped tabular KD, D = 63, reference batch 65 536
    # (conf/training/tabular.yaml: nll 0.85, kd 0.05, perceptual-L1 0.1 through the inverse pass); the 1-D path is fp32
    "glow1d_bsds300_kd_t5_s3": dict(image=(63,), L=1, hidden=32, s_hidden=16, tK=5, sK=3, batch=65536, is_1d=True,
                                    weights=(0.85, 0.05, 0.1), data="bsds300", dtype="f32"),
    # MAF teacher 10 MADE layers -> student 3 layers, hidden 512 (the reference names MAF but ships no code for it)
    "maf_bsds300_kd_t10_s3": dict(image=(63,), L=1, hidden=512, tK=10, sK=3, batch=65536, is_1d=True, arch="maf",
                                  weights=(0.9, 0.1, 0.0), data="bsds300", dtype="bf16"),
}
METRIC = "kd_train_samples_per_sec"


def glow_cfg(image_shape, K, L, hidden, is_1d=False, y_classes=10):
    """Constructor kwargs of the reference's GlowGetAllOutputs (conf/teacher/*.yaml minus `checkpoint`)."""
    return dict(image_shape=list(image_shape), hidden_channels=hidden, K=K, L=L, actnorm_scale=1.0,
                flow_permutation="invconv", flow_coupling="affine", LU_decomposed=True, y_classes=y_classes,
                learn_top=False, y_condition=False, is_1d=is_1d)


def synthetic_images(n, shape, seed):
    """floor(U[0,1)*256)/256 - 0.5, the value range produced by the reference's preprocess (data/src/utils.py:7-18)."""
    g = torch.Generator().manual_seed(seed)
    H, W, C = shape
    return torch.floor(torch.rand(n, C, H, W, generator=g) * 256.0) / 256.0 - 0.5


DUMP_BYTES = 64 << 20


def host_outputs(arrays):
    """The arrays --dump-outputs writes, copied to the host as float32 (float64 stays float64). An array larger than its
    share of DUMP_BYTES is replaced by a fixed sample of its flattened elements (seeded, sorted indices), so that two
    builds run with the same arguments can be compared element for element."""
    share = DUMP_BYTES // len(arrays)
    out = {}
    for name, a in arrays.items():
        a = a.detach()
        a = a.double() if a.dtype == torch.float64 else a.float()
        cap = share // a.element_size()
        if a.numel() > cap:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            a = a.flatten()[idx.to(a.device)]
        out[name] = a.cpu()
    return out


def dump_outputs(directory, arrays):
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a.numpy())


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


def profiled_traffic(kernel, M, K1p):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` at this exact shape, from the committed
    `ncu --set full` summaries (profiles/traffic.json, written by tools/ncu_traffic.py from the .ncu-rep of this
    round); (None, reason) when no capture of this shape exists — the number is never scaled from another shape."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None, "no profiles/traffic.json"
    for e in json.load(open(path)).get(kernel, []):
        if e.get("M") == M and e.get("K1p") == K1p:
            return e["dram_bytes"], e.get("src", "profiles/traffic.json")
    return None, f"no ncu capture at M={M}, K1p={K1p}"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        out = self.proc.communicate()[0]
        sm, mx, reasons = [], None, set()
        for line in out.strip().splitlines():
            f = [s.strip() for s in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------ dominant-kernel roofline
def time_graph(run, reps, nbuf):
    """Average device time of one call of run(i): `reps` calls captured in one CUDA graph (host launch overhead is not
    measured), rotating over `nbuf` buffer sets larger than L2, CUDA events on the launching stream."""
    for i in range(3):
        run(i % nbuf)
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for i in range(reps):
            run(i % nbuf)
    gr.replay()
    torch.cuda.synchronize()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    gr.replay()
    k1.record()
    torch.cuda.synchronize()
    return k0.elapsed_time(k1) / reps


def fused_kernel_name():
    """The fused conv kernel the library dispatches to: the tensor-memory variant (csrc/cnet_ts.cu) unless NFK_CNET_TS=0
    selects the shared-memory-panel one (csrc/cnet_fused.cu)."""
    return "cnet_fwd_fused_kernel" if os.environ.get("NFK_CNET_TS", "1").startswith("0") else "cnet_fwd_ts_kernel"


def cnet_roofline(B, H, W, C_img, hid, device):
    """Roofline of the dominant kernel of every 2-D Glow workload (profiles/r02_launches_*.txt): the fused
    conv3x3 -> ReLU -> conv1x1 -> ReLU of the coupling net at the level-0 shape, M = B*(H/2)*(W/2) pixels, timed alone.
    ALGORITHMIC FLOPs per launch = 2*M*hid*(9*C/2 + hid) with C = 4*C_img level-0 channels (the zero-padded K1p
    columns the kernel also multiplies are not counted), bytes = bf16 col + h2 + weights (DESIGN.md §3)."""
    from nf_distillation_b200 import ops
    pk = peaks()
    C = 4 * C_img
    M, K1, K1p = B * (H // 2) * (W // 2), 9 * C // 2, ops.round_up(9 * C // 2, 64)
    nbuf = 3
    cols = [(torch.randn(M, K1p, device=device) * 0.5).bfloat16() for _ in range(nbuf)]
    for c in cols:
        c[:, K1:] = 0
    outs_ = [torch.empty(M, hid, device=device, dtype=torch.bfloat16) for _ in range(nbuf)]
    W1 = (torch.randn(hid, K1p, device=device) * 0.1).bfloat16()
    W2 = (torch.randn(hid, hid, device=device) * 0.05).bfloat16()
    b1, b2 = torch.zeros(hid, device=device), torch.zeros(hid, device=device)
    fused = ops.cnet_fused_supported(hid, K1p) and M >= 8192

    def run(i):
        if fused:
            ops.cnet_fwd_fused(cols[i], K1p, W1, W2, b1, b2, outs_[i], M, hid)
        else:
            ops.gemm_nt(outs_[(i + 1) % nbuf], W2, M, hid, hid, ops.EPI_BIAS_RELU_BF16, outs_[i], bias=b2)
    kms = time_graph(run, 12, nbuf)
    flops = 2.0 * M * hid * ((K1 if fused else 0) + hid)
    ach = flops / (kms * 1e-3) / 1e12
    alg_bytes = 2.0 * (M * K1 + M * hid + hid * K1 + hid * hid)
    kname = fused_kernel_name() if fused else "gemm_nt_pair_kernel<1>"
    traffic, tsrc = profiled_traffic(kname, M, K1p) if fused else (None, "not captured")
    return {"bound": "tensor",
            "kernel": kname + (" (conv#1+conv#2 of the coupling net, level 0)" if fused else " (conv#2, level 0)"),
            "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"],
            "traffic": traffic, "traffic_src": tsrc,
            "peak_src": pk["src"] + " burst (kernel timed alone)", "us_per_launch": kms * 1e3,
            "flops_per_launch": flops, "algorithmic_bytes_per_launch": alg_bytes,
            "shape": {"M": M, "K1": K1, "K1p": K1p, "hid": hid}}


def kernel_table(B, H, W, C_img, hid, device):
    """Live roofline fractions of the OTHER kernels of the 2-D step at the level-0 shape of this run (the `roofline` key
    holds the dominant one): each timed alone like cnet_roofline, algorithmic bytes / FLOPs as in DESIGN.md §3, against
    the measured HBM copy bandwidth or bf16 burst peak."""
    from nf_distillation_b200 import ops
    pk = peaks()
    C = 4 * C_img
    Hs, Ws = H // 2, W // 2
    M = B * Hs * Ws
    K1p, K3p = ops.round_up(9 * C // 2, 64), ops.round_up(9 * C, 64)
    bf16, f32 = torch.bfloat16, torch.float32
    rows = []

    def add(name, bound, work, us):
        peak = pk["hbm_gbs"] if bound == "hbm" else pk["bf16_tflops"]
        ach = work / (us * 1e-6) / (1e9 if bound == "hbm" else 1e12)
        rows.append({"kernel": name, "bound": bound, "achieved": round(ach, 1), "peak": peak,
                     "unit": "GB/s" if bound == "hbm" else "TFLOP/s", "frac": round(ach / peak, 3),
                     "us_per_launch": round(us, 1)})

    nb = 2
    h2 = [(torch.randn(M, hid, device=device).clamp_min(0) * 0.5).to(bf16) for _ in range(nb)]
    ys = [torch.randn(B, C, Hs, Ws, device=device) for _ in range(nb)]
    xs = [torch.randn(B, C, Hs, Ws, device=device) for _ in range(nb)]
    ld = torch.zeros(B, device=device)
    B3 = (torch.randn(K3p, hid, device=device) * 0.02).to(bf16)
    b3 = torch.zeros(C, device=device)
    if ops.pconv_coupling_supported(C, Hs, Ws, hid):
        us = time_graph(lambda i: ops.pconv_coupling_fwd(h2[i], B3, K3p, b3, ys[i], None, ld, B, C, Hs, Ws, hid, False),
                        10, nb) * 1e3
        add(f"pconv_coupling_kernel<{C}> (Conv2dZeros + coupling, reads h2 once)", "hbm", 2.0 * M * hid + 4.0 * M * C, us)
    Wf, bfv, sl = torch.randn(C, C, device=device) * 0.3, torch.randn(C, device=device), torch.zeros(1, device=device)
    cols = [torch.empty(M, K1p, device=device, dtype=bf16) for _ in range(nb)]
    ld1 = torch.zeros(B, device=device)
    us = time_graph(lambda i: ops.affine1x1_fwd(xs[i], Wf, bfv, sl, ys[i], cols[i], K1p, ld, ld1, B, C, Hs, Ws), 10, nb) * 1e3
    add(f"affine1x1_fwd_kernel<{C}> (ActNorm o invconv + bf16 im2col)", "hbm", M * (8.0 * C + 2.0 * K1p), us)
    # backward kernels of the student
    dpre = [(torch.randn(M, hid, device=device) * 0.1).to(bf16) for _ in range(nb)]
    dW = torch.zeros(hid, hid, device=device)
    us = time_graph(lambda i: ops.gemm_tn(dpre[i], h2[i], hid, hid, M, dW), 10, nb) * 1e3
    add("gemm_tn_pair_kernel (conv#2 weight gradient, split-K over pixels, cta_group::2)", "tensor", 2.0 * M * hid * hid, us)
    W2T = (torch.randn(hid, hid, device=device) * 0.05).to(bf16)
    W3T = (torch.randn(hid, K3p, device=device) * 0.05).to(bf16)
    mask = ops.relu_mask_like(M, hid, device)
    mask.fill_(-1)
    cs, cs2 = torch.zeros(hid, device=device), torch.zeros(hid, device=device)
    outs = [torch.empty(M, hid, device=device, dtype=bf16) for _ in range(nb)]
    if ops.cnet_fused_supported(hid, K3p) and M >= 8192:
        dhc_ = [(torch.randn(M, K3p, device=device) * 0.1).to(bf16) for _ in range(nb)]
        us = time_graph(lambda i: ops.cnet_bwd_fused(dhc_[i], K3p, W3T, W2T, mask, mask, dpre[i], outs[i], cs, cs2, M,
                                                     hid), 10, nb) * 1e3
        add(fused_kernel_name().replace("fwd", "bwd") +
            " (Conv2dZeros dgrad -> ReLU mask -> conv1x1 dgrad -> ReLU mask + both bias gradients)",
            "tensor", 2.0 * M * hid * (9 * C + hid), us)
        del dhc_
    else:
        us = time_graph(lambda i: ops.gemm_nt(dpre[i], W2T, M, hid, hid, ops.EPI_MASK_BF16, outs[i], aux=mask,
                                              colsum=cs), 10, nb) * 1e3
        add("gemm_nt_pair_kernel<MASK_BF16> (conv#2 input gradient + ReLU mask + bias gradient)", "tensor",
            2.0 * M * hid * hid, us)
    del h2, dpre, outs, mask
    hsv = [torch.randn(M, C, device=device) for _ in range(nb)]
    dys = [torch.empty(B, C, Hs, Ws, device=device) for _ in range(nb)]
    dhc = [torch.empty(M, K3p, device=device, dtype=bf16) for _ in range(nb)]
    db3 = torch.zeros(C, device=device)
    us = time_graph(lambda i: ops.coupling_bwd(xs[i], ld, ys[i], hsv[i], dys[i], dhc[i], K3p, db3, B, C, Hs, Ws), 10, nb) * 1e3
    add(f"coupling_bwd_kernel<{C}> (coupling backward + bf16 im2col of dh)", "hbm", M * (14.0 * C + 2.0 * K3p), us)
    dcol = [torch.randn(M, K1p, device=device) * 0.1 for _ in range(nb)]
    dWf, dbf = torch.zeros(C, C, device=device), torch.zeros(C, device=device)
    us = time_graph(lambda i: ops.affine1x1_bwd(dys[i], dcol[i], K1p, xs[i], Wf, ys[i], dWf, dbf, B, C, Hs, Ws), 10, nb) * 1e3
    add(f"affine1x1_bwd_kernel<{C}> (col2im + W'^T dy + dW')", "hbm", M * (12.0 * C + 4.0 * K1p), us)
    return rows


def flow1d_roofline(B, D, hid, device):
    """1-D Glow: the fused FlowStep kernel (csrc/flow1d.cu) is fp32-FMA bound, its HBM side is 8*D bytes per sample;
    report the HBM fraction (the bound the tier's contract names for non-GEMM paths) of the inference kernel."""
    from nf_distillation_b200.models import create_glow_model
    pk = peaks()
    m = create_glow_model(glow_cfg([D], 1, 1, hid, is_1d=True, y_classes=0)).to(device).eval()
    for p in m.parameters():
        p.requires_grad_(False)
    step = m.flow.layers[0]
    xs = [torch.randn(B, D, device=device) for _ in range(3)]
    ld = torch.zeros(B, device=device)

    def run(i):
        with torch.no_grad():
            step(xs[i], logdet=ld, reverse=False)
    kms = time_graph(run, 12, 3)
    alg = 8.0 * D * B + 8.0 * B
    ach = alg / (kms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": f"flow1d_fwd_kernel (whole FlowStep, D={D}, hidden {hid})", "achieved": ach,
            "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"], "traffic": None,
            "traffic_src": "not captured", "peak_src": pk["src"], "us_per_launch": kms * 1e3,
            "algorithmic_bytes_per_launch": alg,
            "note": "fp32 FMA-pipe bound (6.6-11 k FMA per sample), not HBM bound: see DESIGN.md §3"}


def maf_roofline(B, D, H, device):
    """MAF: the fused two-GEMM masked-linear kernel (the coupling net's cnet_fwd_fused_kernel on [B, Dp] rows)."""
    from nf_distillation_b200 import ops
    pk = peaks()
    Dp = ops.round_up(D, 64)
    nbuf = 3
    xs = [(torch.randn(B, Dp, device=device) * 0.5).bfloat16() for _ in range(nbuf)]
    outs_ = [torch.empty(B, H, device=device, dtype=torch.bfloat16) for _ in range(nbuf)]
    W1 = (torch.randn(H, Dp, device=device) * 0.1).bfloat16()
    W2 = (torch.randn(H, H, device=device) * 0.05).bfloat16()
    b1, b2 = torch.zeros(H, device=device), torch.zeros(H, device=device)
    if not (ops.cnet_fused_supported(H, Dp) and B >= 8192):
        return None
    W2[:256, 256:] = 0      # the block-triangular mask of degree-sorted MADE units: skipped by the kernel (kb2_end_half0)
    kms = time_graph(lambda i: ops.cnet_fwd_fused(xs[i], Dp, W1, W2, b1, b2, outs_[i], B, H, kb2_end_half0=4), 12, nbuf)
    # algorithmic = the non-zero part of the masked products: layer 1 D x H, layer 2 ~ half of H x H (degree-sorted)
    flops = 2.0 * B * H * (D + H / 2.0)
    ach = flops / (kms * 1e-3) / 1e12
    traffic, tsrc = profiled_traffic(fused_kernel_name(), B, Dp)
    return {"bound": "tensor", "kernel": fused_kernel_name() + " (both masked linears of a MADE layer)",
            "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"],
            "traffic": traffic, "traffic_src": tsrc, "peak_src": pk["src"] + " burst (kernel timed alone)",
            "us_per_launch": kms * 1e3, "flops_per_launch": flops,
            "algorithmic_bytes_per_launch": 2.0 * (B * D + B * H + H * D + H * H / 2),
            "note": "masked FLOPs only; the kernel skips the zero k-blocks of the low-degree output half (4 of 16 B2 tiles) "
                    "and multiplies the zeros inside the remaining block-triangular tiles"}


def roofline_for(wl, B, device):
    if wl.get("arch") == "maf":
        return maf_roofline(B, wl["image"][0], wl["hidden"], device)
    if wl.get("is_1d", False):
        return flow1d_roofline(B, wl["image"][0], wl["hidden"], device)
    H, W, C = wl["image"]
    return cnet_roofline(B, H, W, C, wl["hidden"], device)


# ------------------------------------------------------------------------------------------ logp delta (vs the oracle)
def logp_delta(model, cfg, is_maf, wl, device, n=8):
    """BASELINE.json metric "...; logp delta": max relative error of the per-sample log-likelihood (bpd in 2-D, nll
    in nats in 1-D) and of the total log-det of the model under test against the CPU oracle (fp32 reference
    arithmetic) on a small batch of the same synthetic data, measured in this run. north_star bound: 1e-4."""
    from nf_distillation_b200.models import utils as U
    sd = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    if is_maf:
        from oracle import maf_oracle as MO
        D = wl["image"][0]
        x = torch.randn(n, D, generator=torch.Generator().manual_seed(77))
        with torch.no_grad():
            _, ref = MO.maf_forward(sd, D, len(model.flow.layers), x)
            _, got, _ = model(x.to(device), None)
        what = "oracle/maf_oracle.py"
    else:
        from oracle import glow_oracle as O
        if cfg.get("is_1d", False):
            x = torch.randn(n, cfg["image_shape"][0], generator=torch.Generator().manual_seed(77))
            noise = None
        else:
            x = synthetic_images(n, wl["image"], 77)
            noise = torch.rand(x.shape, generator=torch.Generator().manual_seed(78)) / 256
        with torch.no_grad():
            _, ref = O.glow_forward(sd, cfg, x, noise)
            orig = U.dequant_noise
            if noise is not None:
                U.dequant_noise = lambda t, nb: noise.to(device)
            try:
                _, got, _ = model(x.to(device), None)
            finally:
                U.dequant_noise = orig
        what = "oracle/glow_oracle.py"
    got = got.float().cpu()
    return {"max_rel_err_per_sample_logp": ((got - ref).abs() / ref.abs().clamp_min(1e-12)).max().item(),
            "samples": n, "oracle": what + " (torch CPU fp32)", "bound": 1e-4}


# ------------------------------------------------------------------------------------------ forward + inverse mode
def run_fwd_inv(args, wl, cfg_desc, warmup):
    """BASELINE configs[2]: one x -> z pass (all layer outputs, per-sample bpd) and one z -> x pass of the K=32 model,
    no gradients, captured in one CUDA graph. value = samples/s through the pair of passes."""
    from nf_distillation_b200 import ops
    from nf_distillation_b200.models import create_glow_model
    from nf_distillation_b200.train import init_distributed, randomise_zero_params
    import torch.distributed as dist
    rank, world, device = init_distributed()
    B = batch_per_gpu(args, wl, world)
    maf = wl.get("arch") == "maf"
    torch.manual_seed(42)
    n_pool = 4
    if maf:
        from nf_distillation_b200.models.maf import create_maf_model
        cfg = dict(image_shape=[wl["image"][0]], hidden_channels=wl["hidden"], K=wl["tK"])
        model = create_maf_model(cfg).to(device).eval()
        host_pool = [torch.randn(B, wl["image"][0], generator=torch.Generator().manual_seed(1000 + rank * 100 + i))
                     .pin_memory() for i in range(n_pool)]
        x = torch.empty(B, wl["image"][0], device=device)
    else:
        H, W, C = wl["image"]
        cfg = glow_cfg(wl["image"], wl["tK"], wl["L"], wl["hidden"])
        model = create_glow_model(cfg)
        randomise_zero_params(model, 43, std=0.01)
        model = model.to(device).eval()
        host_pool = [synthetic_images(B, wl["image"], 1000 + rank * 100 + i).pin_memory() for i in range(n_pool)]
        x = torch.empty(B, C, H, W, device=device)
    for p in model.parameters():        # inference workload: frozen weights keep their derived operands cached
        p.requires_grad_(False)
    dev_pool = [h.to(device) for h in host_pool]
    res = {}

    def passes():
        with torch.no_grad():
            outs, bpd, _ = model(x.clone(), None)
            rev = model(z=outs[-1], temperature=0.0, reverse=True)
            res["bpd"], res["z"], res["x"] = bpd, outs[-1], rev[-1]
            res["stat"] = torch.stack([bpd.mean(), rev[-1].abs().mean()])

    x.copy_(dev_pool[0])
    passes()
    torch.cuda.synchronize()
    c0 = ops.launch_count()
    passes()
    launches = ops.launch_count() - c0
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        passes()
        with torch.cuda.graph(gr):
            passes()
    torch.cuda.current_stream().wait_stream(side)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(warmup):
        x.copy_(dev_pool[i % n_pool]); gr.replay()
    sampler = ClockSampler(device.index or 0)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        x.copy_(dev_pool[i % n_pool]); gr.replay()
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / args.steps
    # the last timed step's per-sample bpd / nll, final latent and reconstruction
    outputs = host_outputs({k: res[k] for k in ("bpd", "z", "x")}) if args.dump_outputs and rank == 0 else None
    # end to end: pinned host batch -> H2D -> both passes -> D2H of (mean bpd, mean |x|)
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        x.copy_(host_pool[i % n_pool], non_blocking=True); gr.replay()
        stat = res["stat"].cpu()
    barrier()
    ms_e2e = (time.perf_counter() - t0) * 1e3 / args.steps
    t = torch.tensor([ms, ms_e2e], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()
    roof = roofline_for(wl, B, device) if rank == 0 else None
    cpu_base = delta = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        delta = logp_delta(model, cfg if not maf else None, maf, wl, device)
        v, cms, cores, sample = cpu_fwd_inv(wl, args.cpu_batch, 1)
        cpu_base = {"value": v, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample}
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if rank == 0:
        gb = B * world
        cfg_desc.update(per_gpu_batch=B, global_batch=gb, parallelism=f"dp{world}", cuda_graphs=True,
                        passes=("x->z (all layer outputs, nll) + z->x (sequential inverse of every MADE layer)" if maf else
                                "x->z (all outputs, bpd) + z->x (split parts at the prior mean, temperature 0)"),
                        l2="activations (~GBs per pass) exceed the 126 MB L2; inputs rotate over 4 batches")
        cfg_desc.pop("student", None); cfg_desc.pop("loss", None); cfg_desc.pop("optimizer", None)
        print(json.dumps({"metric": "fwd_inv_samples_per_sec", "value": gb / (ms * 1e-3), "unit": "samples/s",
                          "n_gpus": world, "steps": args.steps, "warmup": warmup, "ms_per_step": ms,
                          "higher_is_better": True, "scaling": scaling_kind(args), "vs_baseline": None,
                          "dtype": wl["dtype"], "data": "synthetic", "config": cfg_desc, "clocks": clocks,
                          "e2e": {"value": gb / (ms_e2e * 1e-3), "unit": "samples/s", "ms_per_step": ms_e2e,
                                  "h2d_bytes_per_step": host_pool[0].numel() * 4, "d2h_bytes_per_step": 8},
                          "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches,
                          "last": {"bpd_mean": float(stat[0]), "x_abs_mean": float(stat[1])},
                          "logp_delta": delta, "roofline": roof, "cpu_baseline": cpu_base}))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------ CPU arm (oracle port)
# Nothing below imports nf_distillation_b200: weights come from the oracles' own seeded initialisers.
def cpu_fwd_inv(wl, cb, n):
    """(samples/s, ms, threads, description) of n x (one x -> z pass + one z -> x pass) of `cb` samples on the host."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    if wl.get("arch") == "maf":
        from oracle import maf_oracle as MO
        D, cb = wl["image"][0], 4096
        sd = MO.random_state_dict(D, wl["hidden"], wl["tK"], 42)
        xc = torch.randn(cb, D, generator=torch.Generator().manual_seed(7))

        def once():
            outs, _ = MO.maf_forward(sd, D, wl["tK"], xc)
            MO.maf_inverse(sd, D, wl["tK"], outs[-1])
        what = "oracle/maf_oracle.py"
    else:
        from oracle import glow_oracle as O
        cfg = glow_cfg(wl["image"], wl["tK"], wl["L"], wl["hidden"])
        sd = O.random_state_dict(cfg, 42, std=0.01)
        xc = synthetic_images(cb, wl["image"], 7)

        def once():
            outs, _ = O.glow_forward(sd, cfg, xc)
            O.glow_reverse(sd, cfg, outs[-1], 0.0)
        what = "oracle/glow_oracle.py"
    with torch.no_grad():
        once()
        t0 = time.perf_counter()
        for _ in range(n):
            once()
        dt = (time.perf_counter() - t0) / n
    return cb / dt, dt * 1e3, cores, (f"{n} x (one forward + one inverse pass) of {cb} samples ({what}, torch CPU "
                                     f"fp32, {cores} threads)")


def cpu_kd_step_fn(wl, batch, seed=42):
    """The reference's CPU algorithm for this path, restated in oracle/ (the reference itself is a Python script tree
    with missing dependencies and does not travel to the GPU box): KD train step = fwd student + teacher, loss,
    backward, clip 30, Adam."""
    from oracle import glow_oracle as O
    is_1d = wl.get("is_1d", False)
    torch.manual_seed(seed)
    if wl.get("arch") == "maf":
        from oracle import maf_oracle as MO
        D = wl["image"][0]
        t_sd = MO.random_state_dict(D, wl["hidden"], wl["tK"], seed + 2)
        s_sd = {k: (v.requires_grad_(True) if v.dtype.is_floating_point else v)
                for k, v in MO.random_state_dict(D, wl["hidden"], wl["sK"], seed + 1).items()}
        params = [v for v in s_sd.values() if v.requires_grad]
        opt = torch.optim.Adam(params, lr=5e-4)
        x = torch.randn(batch, D)
        wn, wk, _ = wl["weights"]

        def step():
            opt.zero_grad(set_to_none=True)
            s_z, s_nll = MO.maf_forward(s_sd, D, wl["sK"], x)
            with torch.no_grad():
                t_z, _ = MO.maf_forward(t_sd, D, wl["tK"], x)
            kd = O.kd_loss(s_z, t_z, [1, 2], [3, 7])
            loss = (wn * s_nll + wk * kd).mean()
            loss.backward()
            torch.nn.utils.clip_grad_norm_(params, 30.0)
            opt.step()
            return float(loss.detach())
        return step
    yc = 0 if is_1d else 10
    s_cfg = glow_cfg(wl["image"], wl["sK"], wl["L"], wl.get("s_hidden", wl["hidden"]), is_1d=is_1d, y_classes=yc)
    t_cfg = glow_cfg(wl["image"], wl["tK"], wl["L"], wl["hidden"], is_1d=is_1d, y_classes=yc)
    t_sd = O.random_state_dict(t_cfg, seed + 2)
    s_sd = {k: (v.requires_grad_(True) if k != "prior_h" and not k.endswith((".p", ".sign_s")) else v)
            for k, v in O.random_state_dict(s_cfg, seed + 1).items()}
    params = [v for v in s_sd.values() if v.requires_grad]
    opt = torch.optim.Adam(params, lr=5e-4)
    if is_1d:
        x = torch.randn(batch, wl["image"][0])
        wn, wk, wp = wl["weights"]
        weights = {"nll": wn, "kd": wk, "perceptual": wp}
    else:
        x = synthetic_images(batch, wl["image"], seed)
        weights = {"nll": 0.9, "kd": 0.1, "perceptual": 0.0}

    def step():
        n1 = n2 = latent = None
        if is_1d:
            latent = torch.randn_like(x)
        else:
            n1, n2 = torch.rand_like(x) / 256, torch.rand_like(x) / 256
        opt.zero_grad(set_to_none=True)
        out = O.kd_step(s_sd, s_cfg, t_sd, t_cfg, x, weights, n1, n2, latent)
        out["result_loss"].backward()
        torch.nn.utils.clip_grad_norm_(params, 30.0)
        opt.step()
        return float(out["result_loss"].detach())
    return step


def run_cpu(wl, batch, steps, warmup):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step = cpu_kd_step_fn(wl, batch)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return batch / dt, dt * 1e3, cores


def cpu_batch_for(args, wl):
    if not wl.get("is_1d", False):
        return args.cpu_batch
    return 8192 if wl.get("arch") == "maf" else 65536


def run_reference_arm(args, wl, cfg_desc):
    """bench.py --impl reference: the reference's CPU algorithm for this workload (oracle/ port) on the box's host
    cores, bounded sample per step; rank 0 only. No product code is imported on this path."""
    n = args.steps
    if wl.get("mode") == "fwd_inv":
        metric = "fwd_inv_samples_per_sec"
        value, ms, cores, sample = cpu_fwd_inv(wl, args.cpu_batch, n)
        cb = 4096 if wl.get("arch") == "maf" else args.cpu_batch
        for k in ("student", "loss", "optimizer"):
            cfg_desc.pop(k, None)
    else:
        metric = METRIC
        cb = cpu_batch_for(args, wl)
        value, ms, cores = run_cpu(wl, cb, n, 1)
        sample = (f"{cb}-sample KD train steps of the same workload (oracle/ port of the reference, torch CPU fp32, "
                  f"{cores} threads)")
    cfg_desc.update(per_gpu_batch=cb, global_batch=cb, parallelism="cpu")
    print(json.dumps({
        "impl": "reference", "metric": metric, "value": value, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": n, "warmup": 1, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg_desc,
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
    assert not any(m.startswith("nf_distillation_b200") for m in sys.modules), "reference arm must not load the product"


def batch_per_gpu(args, wl, world):
    if args.global_batch:
        assert args.global_batch % world == 0, "--global-batch must divide evenly over the ranks"
        return args.global_batch // world
    return args.batch or wl["batch"]


def scaling_kind(args):
    return "strong" if args.global_batch else "weak"


# ------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: workload's); weak scaling")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="STRONG scaling: total batch fixed, each rank takes global/N (overrides --batch)")
    ap.add_argument("--workload", default="glow_cifar_kd_t32_s8", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-table", action="store_true",
                    help="skip the live roofline table of the non-dominant kernels (key `kernels`)")
    ap.add_argument("--cpu-batch", type=int, default=32)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "bf16x3"],
                    help="arithmetic of the 2-D coupling-net GEMMs: bf16 operands (default) or the fp32-class "
                         "3-term split (models.flows.Glow.set_precision)")
    ap.add_argument("--no-pipeline", action="store_true",
                    help="2-D KD workloads: do NOT prefetch the frozen teacher's forward of the next batch beside the "
                         "student's step (train.KDTrainer(pipelined=...)); default is pipelined")
    ap.add_argument("--u8-input", action="store_true",
                    help="image workloads: feed raw uint8 pixels (a quarter of the H2D bytes); preprocess + noise + first "
                         "squeeze run as the step's first kernel")
    ap.add_argument("--ncu-step", action="store_true",
                    help="profiling aid: warm up, then run ONE eager step between cudaProfilerStart/Stop and exit "
                         "(use with ncu --profile-from-start off); prints no bench value")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy "
                         "(float32, at most 64 MB; a seeded sample of an array too large for its share)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "native" or args.ncu_step):
        ap.error("--dump-outputs applies to the timed native path")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    warmup = max(args.warmup, 3) if args.impl == "native" else max(args.warmup, 1)
    arch = wl.get("arch", "glow")
    cfg_desc = {"workload": args.workload, "teacher": f"{arch} K={wl['tK']} L={wl['L']} hidden={wl['hidden']}",
                "student": f"{arch} K={wl['sK']} L={wl['L']} hidden={wl.get('s_hidden', wl['hidden'])}",
                "image": list(wl["image"]),
                "loss": "0.9 nll + 0.1 kd(mse, 4 levels)" if "weights" not in wl else
                        "%.2f nll + %.2f kd(mse) + %.2f perceptual(l1, inverse pass)" % wl["weights"],
                "optimizer": "adam 5e-4, clip 30"}

    if args.impl == "reference":
        if rank != 0:
            return
        return run_reference_arm(args, wl, cfg_desc)

    if wl.get("mode") == "fwd_inv":
        return run_fwd_inv(args, wl, cfg_desc, warmup)
    import torch.distributed as dist
    from nf_distillation_b200 import ops
    from nf_distillation_b200.train import KDTrainer, init_distributed, kd_config
    rank, world, device = init_distributed()
    B = batch_per_gpu(args, wl, world)
    is_1d = wl.get("is_1d", False)
    if is_1d:
        D = wl["image"][0]
        s_cfg = glow_cfg(wl["image"], wl["sK"], wl["L"], wl.get("s_hidden", wl["hidden"]), is_1d=True, y_classes=0)
        t_cfg = glow_cfg(wl["image"], wl["tK"], wl["L"], wl["hidden"], is_1d=True, y_classes=0)
        if wl.get("arch") == "maf":
            s_cfg["architecture"] = t_cfg["architecture"] = "maf"
        wn, wk, wp = wl["weights"]
        config = kd_config(s_cfg, t_cfg, data=wl["data"], nll=wn, kd=wk, perceptual=wp)
        shape = (B, D)
    else:
        H, W, C = wl["image"]
        s_cfg = glow_cfg(wl["image"], wl["sK"], wl["L"], wl.get("s_hidden", wl["hidden"]))
        config = kd_config(s_cfg, glow_cfg(wl["image"], wl["tK"], wl["L"], wl["hidden"]))
        shape = (B, C, H, W)
    u8 = args.u8_input and not is_1d
    trainer = KDTrainer(config, shape, device, use_graphs=not args.no_graphs,
                        input_dtype=torch.uint8 if u8 else torch.float32, pipelined=not args.no_pipeline)
    dtype = wl["dtype"]
    if args.precision != "bf16":
        if is_1d:
            raise SystemExit("--precision applies to the 2-D Glow workloads (the 1-D path is fp32 already)")
        trainer.module.student.set_precision(args.precision)
        trainer.module.teacher.set_precision(args.precision)
        dtype = "bf16x3 (fp32-class: hi+lo split bf16 operands, 3 partial products, fp32 accumulate)"
    n_pool = 4

    def synth(i):
        if is_1d:   # z-scored tabular features (data/src/power.py:42-52): N(0, 1)
            g = torch.Generator().manual_seed(1000 + rank * 100 + i)
            return torch.randn(B, wl["image"][0], generator=g)
        img = synthetic_images(B, wl["image"], 1000 + rank * 100 + i)
        return ((img + 0.5) * 256.0).round().to(torch.uint8) if u8 else img      # the same pixels, raw
    host_pool = [synth(i).pin_memory() for i in range(n_pool)]
    dev_pool = [h.to(device) for h in host_pool]
    trainer.x.copy_(dev_pool[0])
    if args.ncu_step:
        trainer.use_graphs = False
        trainer.warmup(iters=3)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        trainer.step_device()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        print(json.dumps({"ncu_step": True, "batch": B, "losses": trainer.losses.cpu().tolist()}))
        return
    # Every warm-up and timed step trains the seeded initial student with fresh optimiser state. The kernels reduce with
    # float atomics, so a step's results vary from run to run in the last bits; a step that continued from the previous
    # step's weights would take that variation as input, and Adam's early updates (about lr * sign(g)) move a weight
    # whose gradient is within rounding of zero by up to 2 lr. Restarting keeps the inputs of every step identical from
    # run to run, and its results equal up to rounding; the work of a step is unchanged. The restart (one copy of the
    # flat parameters, memsets of the optimiser state) is timed with the step: 47 us of a 38 ms step of the default
    # workload (B200, 1000 W).
    p0 = trainer.opt.p.clone()

    def restart():
        trainer.opt.p.copy_(p0)
        trainer.reset_state()

    # logp delta of the student as initialised, before any step (rank 0, single GPU, with the CPU legs)
    delta = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        trainer.module.student.eval()
        delta = logp_delta(trainer.module.student, None if wl.get("arch") == "maf" else s_cfg,
                           wl.get("arch") == "maf", wl, device)
        trainer.module.student.train()
    # count kernels of ONE step: an eager step (forward, backward, clip + Adam) outside the graphs
    trainer.warmup(iters=1)                      # eager step(s) + graph capture
    c0 = ops.launch_count()
    trainer._forward_backward()
    trainer._clip_and_update()
    launches_per_step = ops.launch_count() - c0
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing (value)
    for i in range(warmup):
        trainer.x.copy_(dev_pool[i % n_pool])
        restart()
        trainer.step_device()
    sampler = ClockSampler(device.index or 0)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        trainer.x.copy_(dev_pool[i % n_pool])
        restart()
        trainer.step_device()
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / args.steps
    losses = trainer.losses.cpu().tolist()
    # the last timed step's loss scalars (nll, kd, perceptual, loss) and the student's averaged gradient before clipping,
    # flat in student.parameters() order. The updated weights are left out: Adam's first update is about lr * sign(g),
    # not a result that agrees up to rounding.
    outputs = None
    if args.dump_outputs and rank == 0:
        outputs = host_outputs({"losses": trainer.losses,
                                "student_grads": torch.cat([g.flatten() for g in trainer.opt.g_views])})

    # ---- end-to-end timing through the public API: pinned host batch -> H2D -> step -> D2H of the loss scalars
    for i in range(2):
        trainer.step(host_pool[i % n_pool])
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        last = trainer.step(host_pool[i % n_pool])
    barrier()
    ms_e2e = (time.perf_counter() - t0) * 1e3 / args.steps

    t = torch.tensor([ms, ms_e2e], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()

    roof = roofline_for(wl, B, device) if rank == 0 and args.precision == "bf16" else None
    ktable = None
    pipelined = trainer.pipelined
    if rank == 0 and world == 1 and not is_1d and args.precision == "bf16" and not args.no_kernel_table:
        del trainer, dev_pool
        torch.cuda.empty_cache()
        ktable = kernel_table(B, H, W, C, wl["hidden"], device)

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = cpu_batch_for(args, wl)
        v, cms, cores = run_cpu(wl, cb, 2, 1)
        cpu_base = {"value": v, "unit": "samples/s", "cores": cores, "kind": "port",
                    "sample": f"2 KD train steps of {cb} samples, same model/config "
                              f"(oracle/ on torch CPU fp32, {cores} threads), {cms:.0f} ms/step"}

    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if rank == 0:
        gb = B * world
        cfg_desc.update(per_gpu_batch=B, global_batch=gb, parallelism=f"dp{world}",
                        cuda_graphs=not args.no_graphs, input="uint8 pixels" if u8 else "fp32 (preprocessed)",
                        teacher_prefetch=("1 batch: the frozen teacher's forward of batch t+1 runs beside the student's "
                                          "step on batch t (same updates; one batch consumed and one update made per "
                                          "step)") if pipelined else "off",
                        l2="per-step working set (activations ~GBs) exceeds the 126 MB L2; inputs rotate over 4 batches",
                        step_start="every warm-up and timed step starts from the seeded initial student and fresh Adam "
                                   "state; the restart (parameter copy + optimiser-state memsets) is timed with it")
        out = {"metric": METRIC, "value": gb / (ms * 1e-3), "unit": "samples/s", "n_gpus": world,
               "steps": args.steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
               "scaling": scaling_kind(args), "vs_baseline": None, "dtype": dtype,
               "data": "synthetic", "config": cfg_desc, "clocks": clocks,
               "e2e": {"value": gb / (ms_e2e * 1e-3), "unit": "samples/s", "ms_per_step": ms_e2e,
                       "h2d_bytes_per_step": host_pool[0].numel() * host_pool[0].element_size(),
                       "d2h_bytes_per_step": 16},
               "gpu_launches": launches_per_step * args.steps, "gpu_launches_per_step": launches_per_step,
               "losses_last_step": dict(zip(("nll", "kd", "perceptual", "loss"), losses)),
               "logp_delta": delta, "roofline": roof, "kernels": ktable, "cpu_baseline": cpu_base}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
