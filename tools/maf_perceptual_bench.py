"""Cost of the perceptual L1 term for MAF students (gradients through the sequential MADE inverse).

maf_bsds300_kd_t10_s3 (D = 63, hidden 512, teacher 10 MADE layers, student 3, B = 65 536) trained by KDTrainer with
loss weights nll 0.9 / kd 0.1 and perceptual 0 vs 0.1. The two arms live in one process and their timed windows
alternate; each step restarts from the seeded initial student with fresh optimiser state, so every step does the
same work.

Per MADE layer (D = 63, H = 512, B = 65 536), CUDA events over graph-captured launches: the forward resident inverse,
the resident reverse solve, the D-pass reverse solve, and the whole inverse-layer backward (forward recomputed at x,
reverse solve, parameter chain). Prints one JSON line and writes it to --out.
usage: python tools/maf_perceptual_bench.py [--batch 65536] [--steps 5] [--rounds 3] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from perceptual_bench import gpu_info, launches_per_step, time_graph, time_steps  # noqa: E402


def make_trainer(B, perceptual, device):
    from nf_distillation_b200.train import KDTrainer, glow_cfg, kd_config
    s_cfg = glow_cfg((63,), 3, 1, 512, is_1d=True, y_classes=0)
    t_cfg = glow_cfg((63,), 10, 1, 512, is_1d=True, y_classes=0)
    s_cfg["architecture"] = t_cfg["architecture"] = "maf"
    tr = KDTrainer(kd_config(s_cfg, t_cfg, data="bsds300", nll=0.9, kd=0.1, perceptual=perceptual), (B, 63), device,
                   use_graphs=True, pipelined=True)
    tr.x.copy_(torch.randn(B, 63, generator=torch.Generator().manual_seed(1000)).to(device))
    return tr


def layer_times(B, device, reps=10):
    from nf_distillation_b200.models.maf import MADE, _made_grad_arena, _made_net_backward
    D, H = 63, 512
    torch.manual_seed(0)
    made = MADE(D, H, flip=True).to(device)
    u, gx, gld = torch.randn(B, D, device=device), torch.randn(B, D, device=device), torch.randn(B, device=device)
    with torch.no_grad():
        x, _ = made(u, reverse=True)
        params = made._params()
        ops_ = made._operands(params, True)
        xb = made._bf16_rows(x, None)
        h1, h2, out, m1, m2 = made._net(xb, B, ops_, params[1], params[3], keep=True)
        g_u = torch.empty_like(x)
        dout = torch.empty(B, made.N3p, device=device, dtype=torch.bfloat16)
        db3 = torch.zeros(2 * D, device=device)

        def solve(resident):
            made.resident_inverse = resident
            made._inverse_solve(gx, gld, u, out, m1, m2, ops_, True, g_u, dout, db3)
            made.resident_inverse = True

        def whole(_):
            ops2 = made._operands(params, True)
            xb2 = made._bf16_rows(x, None)
            a1, a2, o2, k1, k2 = made._net(xb2, B, ops2, params[1], params[3], keep=True)
            grads = _made_grad_arena(made, device)
            made._inverse_solve(gx, gld, u, o2, k1, k2, ops2, True, g_u, dout, grads[0])
            _made_net_backward(made, dout, xb2, a1, a2, k1, k2, ops2[1], ops2[3], ops2[5], grads, False)

        res = {"D": D, "H": H, "B": B, "inputs": "one buffer set (activations 65536 x 512 bf16 exceed the 126 MB L2)"}
        res["forward_resident_inverse_ms"] = time_graph(lambda _: made(u, reverse=True), reps, 1)
        res["reverse_solve_resident_ms"] = time_graph(lambda _: solve(True), reps, 1)
        res["reverse_solve_dpass_ms"] = time_graph(lambda _: solve(False), 2, 1)
        res["inverse_layer_backward_ms"] = time_graph(whole, reps, 1)
    return {k: (round(v, 4) if isinstance(v, float) else v) for k, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_maf_perceptual_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    device = torch.device("cuda", 0)
    B = args.batch
    result = {"gpu": gpu_info(), "workload": "maf_bsds300_kd_t10_s3", "batch": B,
              "weights": "nll 0.9 / kd 0.1 / perceptual 0 vs 0.1"}
    result["per_layer"] = layer_times(B, device)
    arms = {}
    for wp in (0.0, 0.1):
        tr = make_trainer(B, wp, device)
        p0 = tr.opt.p.clone()
        tr.warmup(iters=1)
        n = launches_per_step(tr)
        time_steps(tr, p0, args.warmup)
        arms[wp] = {"tr": tr, "p0": p0, "launches": n, "ms": []}
    for _ in range(args.rounds):
        for a in arms.values():
            a["ms"].append(time_steps(a["tr"], a["p0"], args.steps))
    for wp, a in arms.items():
        result[f"perceptual_{wp}"] = {"step_ms_median": round(sorted(a["ms"])[len(a["ms"]) // 2], 3),
                                      "step_ms_all": [round(v, 3) for v in a["ms"]], "launches_per_step": a["launches"],
                                      "losses": [round(v, 6) for v in a["tr"].losses.cpu().tolist()]}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
