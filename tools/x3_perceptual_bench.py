"""Cost of training through the 2-D inverse pass in the fp32-class precision mode ("bf16x3") against the bf16 mode.

glow_cifar_kd_t32_s8 (teacher K=32, student K=8, L=3, hidden 512, CIFAR 32x32x3) trained by KDTrainer (one CUDA graph
per step) with loss weights nll 0.9 / kd 0.1 / perceptual 0.1, both models in bf16 or both in bf16x3, at B = 64 and
512. The two arms of a batch size live in one process and their timed windows alternate; each step restarts from the
seeded initial student with fresh optimiser state, so every step does the same work.

At this pair's randomised initialisation the 32-step teacher's inverse at T = 0.7 overflows fp32, so the perceptual
term is replaced by 0 (the reference's NaN guard, DESIGN §3) and the gradient is not finite: these runs time the
kernels, they do not train. The output says so ("trains": false) whenever it happens.

Prints one JSON line (and writes it to --out when given).
usage: python tools/x3_perceptual_bench.py [--batches 64,512] [--steps 5] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import torch  # noqa: E402

from perceptual_bench import gpu_info, images, launches_per_step, time_steps  # noqa: E402

PERCEPTUAL = 0.1


def make_trainer(B, precision, device):
    from nf_distillation_b200.train import KDTrainer, glow_cfg, kd_config
    s_cfg, t_cfg = glow_cfg((32, 32, 3), 8, 3, 512), glow_cfg((32, 32, 3), 32, 3, 512)
    tr = KDTrainer(kd_config(s_cfg, t_cfg, nll=0.9, kd=0.1, perceptual=PERCEPTUAL), (B, 3, 32, 32), device,
                   use_graphs=True)
    tr.module.student.set_precision(precision)
    tr.module.teacher.set_precision(precision)
    tr.x.copy_(images(B, 1000).to(device))
    return tr


def bench_batch(B, steps, rounds, warmup, device):
    arms = {}
    for prec in ("bf16", "bf16x3"):
        tr = make_trainer(B, prec, device)
        p0 = tr.opt.p.clone()                    # the seeded initial student: every timed step restarts from it
        tr.warmup(iters=1)
        n = launches_per_step(tr)
        time_steps(tr, p0, warmup)
        arms[prec] = {"tr": tr, "p0": p0, "launches": n, "ms": []}
    for _ in range(rounds):
        for a in arms.values():
            a["ms"].append(time_steps(a["tr"], a["p0"], steps))
    res = {}
    for prec, a in arms.items():
        ms = sorted(a["ms"])[len(a["ms"]) // 2]
        losses = a["tr"].losses.cpu().tolist()
        finite = bool(torch.isfinite(a["tr"].opt.g).all())
        res[prec] = {"ms_per_step": round(ms, 3), "samples_per_s": round(B / ms * 1e3, 1),
                     "ms_per_round": [round(v, 3) for v in a["ms"]], "launches_per_step": a["launches"],
                     "losses_nll_kd_perc_loss": [round(v, 5) for v in losses], "grad_finite": finite,
                     "trains": finite and losses[2] > 0}
    res["x3_over_bf16"] = round(res["bf16x3"]["ms_per_step"] / res["bf16"]["ms_per_step"], 3)
    for a in arms.values():
        del a["tr"]
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="64,512")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("x3_perceptual_bench needs a CUDA device")
    device = torch.device("cuda", torch.cuda.current_device())
    result = {"workload": "glow_cifar_kd_t32_s8", "weights": {"nll": 0.9, "kd": 0.1, "perceptual": PERCEPTUAL},
              "arms": "both models bf16 vs both models bf16x3", "gpu": gpu_info(), "steps": args.steps,
              "rounds": args.rounds,
              "timing": "CUDA events over `steps` graph-replayed steps per round, median of the rounds; arms alternate"}
    batches = [int(b) for b in args.batches.split(",")]
    for B in batches:
        result[f"B{B}"] = bench_batch(B, args.steps, args.rounds, args.warmup, device)
    trains = all(result[f"B{B}"][prec]["trains"] for B in batches for prec in ("bf16", "bf16x3"))
    result["note"] = ("every arm trains" if trains else
                      "the teacher's inverse at T = 0.7 overflows fp32 at this initialisation: the perceptual term is "
                      "replaced by 0 and the gradient is not finite, so these runs time the kernels and do not train")
    result["gpu_after"] = gpu_info()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
