"""Cost of the perceptual L1 term (gradients through the student's 2-D inverse pass) on the headline KD pair.

glow_cifar_kd_t32_s8 (teacher K=32, student K=8, L=3, hidden 512, CIFAR 32x32x3) trained by KDTrainer with loss weights
nll 0.9 / kd 0.1 and perceptual 0 vs 0.1, at B = 2048 and B = 64. The two arms of a batch size live in one process and
their timed windows alternate, so drift of the shared machine hits both. Each step restarts from the seeded initial
student with fresh optimiser state (as bench.py does), so every step does the same work.

Also times the two kernels only the inverse pass's backward runs, coupling_inv_bwd and col2im_add, at the level-0 shape
(C = 12, 16x16 maps) with CUDA events over graph-captured launches that rotate over buffer sets larger than L2.

Prints one JSON line (and writes it to --out when given).
usage: python tools/perceptual_bench.py [--batches 2048,64] [--steps 10] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

HBM_DATASHEET_GBS = 7700.0    # HGX B200 data sheet, one GPU (1000 W card)


def gpu_info():
    q = {"name": torch.cuda.get_device_name(), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        name, pl = [s.strip() for s in out.strip().splitlines()[0].split(",")]
        q.update(name=name, power_limit_w=float(pl))
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        pass
    return q


def images(B, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.floor(torch.rand(B, 3, 32, 32, generator=g) * 256.0) / 256.0 - 0.5


def make_trainer(B, perceptual, device):
    from nf_distillation_b200.train import KDTrainer, glow_cfg, kd_config
    s_cfg, t_cfg = glow_cfg((32, 32, 3), 8, 3, 512), glow_cfg((32, 32, 3), 32, 3, 512)
    tr = KDTrainer(kd_config(s_cfg, t_cfg, nll=0.9, kd=0.1, perceptual=perceptual), (B, 3, 32, 32), device,
                   use_graphs=True, pipelined=True)
    tr.x.copy_(images(B, 1000).to(device))
    return tr


def launches_per_step(tr):
    from nf_distillation_b200 import ops
    c0 = ops.launch_count()
    tr._forward_backward()
    tr._clip_and_update()
    torch.cuda.synchronize()
    return ops.launch_count() - c0


def time_steps(tr, p0, steps):
    def restart():
        tr.opt.p.copy_(p0)
        tr.reset_state()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        restart()
        tr.step_device()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def time_graph(run, reps, nbuf):
    """Device time of one run(i): `reps` calls in one CUDA graph, rotating over `nbuf` buffer sets."""
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


def kernel_times(B, device):
    """coupling_inv_bwd and col2im_add at the level-0 shape of batch B (C = 12, 16x16)."""
    from nf_distillation_b200 import ops
    C, H, W = 12, 16, 16
    CH, M = C // 2, B * H * W
    K1p, K3p = ops.round_up(9 * CH, 64), ops.round_up(9 * C, 64)
    per_set = M * (4 * C * 4 + 2 * K3p + 4 * K1p)
    nbuf = max(2, int(400e6 / per_set) + 1)                  # > 3x the 126 MB L2
    mk = lambda *s, dt=torch.float32: [torch.randn(*s, device=device).to(dt) for _ in range(nbuf)]
    g_zc, zc, dz = mk(B, C, H, W), mk(B, C, H, W), mk(B, C, H, W)
    hsave = [t * 0.3 for t in mk(M, C)]
    dhcol, dcol = mk(M, K3p, dt=torch.bfloat16), mk(M, K1p)
    g_ld, db3 = torch.randn(B, device=device), torch.zeros(C, device=device)
    out = {}
    us = time_graph(lambda i: ops.coupling_inv_bwd(g_zc[i], g_ld, zc[i], hsave[i], dz[i], dhcol[i], K3p, db3, B, C, H,
                                                   W), 20, nbuf) * 1e3
    by = M * (14.0 * C + 2.0 * K3p)
    out["coupling_inv_bwd"] = {"us": round(us, 2), "alg_bytes": int(by), "bytes_formula": "M*(14*C + 2*K3p)",
                               "gbs": round(by / us * 1e-3, 1),
                               "frac_hbm_datasheet": round(by / us * 1e-3 / HBM_DATASHEET_GBS, 3)}
    us = time_graph(lambda i: ops.col2im_add(dcol[i], K1p, dz[i], B, C, H, W), 20, nbuf) * 1e3
    by = M * (4.0 * 9 * CH + 8.0 * CH)
    out["col2im_add"] = {"us": round(us, 2), "alg_bytes": int(by), "bytes_formula": "M*(4*9*C/2 + 8*C/2)",
                         "gbs": round(by / us * 1e-3, 1),
                         "frac_hbm_datasheet": round(by / us * 1e-3 / HBM_DATASHEET_GBS, 3)}
    out.update(M=M, C=C, H=H, W=W, K1p=K1p, K3p=K3p)
    return out


def bench_batch(B, steps, rounds, warmup, device):
    arms = {}
    for wp in (0.0, 0.1):
        tr = make_trainer(B, wp, device)
        p0 = tr.opt.p.clone()                    # the seeded initial student: every timed step restarts from it
        tr.warmup(iters=1)
        n = launches_per_step(tr)
        time_steps(tr, p0, warmup)
        arms[wp] = {"tr": tr, "p0": p0, "launches": n, "ms": []}
    for _ in range(rounds):
        for wp, a in arms.items():
            a["ms"].append(time_steps(a["tr"], a["p0"], steps))
    res = {}
    for wp, a in arms.items():
        ms = sorted(a["ms"])[len(a["ms"]) // 2]
        losses = a["tr"].losses.cpu().tolist()
        res[f"perceptual_{wp}"] = {"ms_per_step": round(ms, 3), "samples_per_s": round(B / ms * 1e3, 1),
                                   "ms_per_round": [round(v, 3) for v in a["ms"]], "launches_per_step": a["launches"],
                                   "pipelined_teacher": a["tr"].pipelined, "losses": [round(v, 5) for v in losses],
                                   "grad_finite": bool(torch.isfinite(a["tr"].opt.g).all())}
    res["perceptual_overhead"] = round(res["perceptual_0.1"]["ms_per_step"] / res["perceptual_0.0"]["ms_per_step"], 3)
    for a in arms.values():
        del a["tr"]
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="2048,64")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("perceptual_bench needs a CUDA device")
    device = torch.device("cuda", torch.cuda.current_device())
    batches = [int(b) for b in args.batches.split(",")]
    result = {"workload": "glow_cifar_kd_t32_s8", "weights": {"nll": 0.9, "kd": 0.1, "perceptual": [0.0, 0.1]},
              "gpu": gpu_info(), "steps": args.steps, "rounds": args.rounds,
              "timing": "CUDA events over `steps` graph-replayed steps per round, median of the rounds; arms alternate",
              "hbm_peak_gbs": HBM_DATASHEET_GBS, "hbm_peak_src": "HGX B200 data sheet, one GPU"}
    for B in batches:
        result[f"B{B}"] = bench_batch(B, args.steps, args.rounds, args.warmup, device)
    result["kernels_level0"] = kernel_times(batches[0], device)
    result["gpu_after"] = gpu_info()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
