"""Time the coupling net's first-conv input gradient + affine1x1_bwd at the three level shapes of glow_cifar_kd_t32_s8.

Per level (C, H x W) and batch size, two arms:
  pair   gemm_nt (EPI_F32) -> dcol [M, K1p] fp32, then affine1x1_bwd (col2im, dx = W'^T dy, dW', db')
  fused  conv1_dgrad_affine_bwd (csrc/dgrad_col2im.cu): the same result, dcol never leaves the SM
Each arm is graph-replayed over buffer sets larger than L2 (bench.py::time_graph), CUDA events on the stream.

Algorithmic bytes: pair = dpre1 read + dcol write (GEMM) + dcol, dy, x read + dx write (affine1x1_bwd); fused = dpre1,
dy, x read + dx write. The share of peak is those bytes over the time, against the HGX B200 data sheet's 7.7 TB/s.
Prints one JSON line and writes it to --out (default profiles/r05_dgrad1_bench.json).
usage: python tools/dgrad1_bench.py [--batches 2048,64] [--reps 40] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from bench import time_graph  # noqa: E402
from perceptual_bench import gpu_info  # noqa: E402

HBM_DATASHEET_GBS = 7700.0
L2_BYTES = 126 << 20
LEVELS = [(12, 16), (24, 8), (48, 4)]    # (C, H = W) of the student's three levels on CIFAR 32x32x3


def bench_level(C, H, B, hid, reps):
    from nf_distillation_b200 import ops
    dev = torch.device("cuda")
    W, CH = H, C // 2
    M, K1p = B * H * W, ops.round_up(9 * CH, 64)
    set_bytes = M * hid * 2 + 3 * M * C * 4 + M * K1p * 4
    nbuf = max(2, -(-2 * L2_BYTES // set_bytes))
    g = torch.Generator(device=dev).manual_seed(C + B)
    dpre1 = [torch.randn(M, hid, device=dev, generator=g).bfloat16() for _ in range(nbuf)]
    dys = [torch.randn(B, C, H, W, device=dev, generator=g) for _ in range(nbuf)]
    xs = [torch.randn(B, C, H, W, device=dev, generator=g) for _ in range(nbuf)]
    dxs = [torch.empty(B, C, H, W, device=dev) for _ in range(nbuf)]
    dcols = [torch.empty(M, K1p, device=dev) for _ in range(nbuf)]
    B1T = torch.zeros(K1p, hid, device=dev, dtype=torch.bfloat16)
    B1T[:9 * CH] = (torch.randn(9 * CH, hid, device=dev, generator=g) * 0.03).bfloat16()
    Wf = torch.randn(C, C, device=dev, generator=g) * 0.3
    dWf, dbf = torch.zeros(C, C, device=dev), torch.zeros(C, device=dev)

    def pair(i):
        ops.gemm_nt(dpre1[i], B1T, M, K1p, hid, ops.EPI_F32, dcols[i])
        ops.affine1x1_bwd(dys[i], dcols[i], K1p, xs[i], Wf, dxs[i], dWf, dbf, B, C, H, W)

    def gemm(i):
        ops.gemm_nt(dpre1[i], B1T, M, K1p, hid, ops.EPI_F32, dcols[i])

    def aff(i):
        ops.affine1x1_bwd(dys[i], dcols[i], K1p, xs[i], Wf, dxs[i], dWf, dbf, B, C, H, W)

    def fused(i):
        ops.conv1_dgrad_affine_bwd(dpre1[i], B1T, K1p, dys[i], xs[i], Wf, dxs[i], dWf, dbf, B, C, H, W, hid)

    zc = M * hid * 2
    bytes_gemm = zc + M * K1p * 4
    bytes_aff = M * K1p * 4 + 3 * M * C * 4
    bytes_fused = zc + 3 * M * C * 4
    us = {}
    for name, fn in (("pair", pair), ("fused", fused), ("gemm", gemm), ("affine1x1_bwd", aff), ("fused_again", fused)):
        us[name] = time_graph(fn, reps, nbuf) * 1e3
    us["fused"] = min(us["fused"], us.pop("fused_again"))   # two windows around the pair's: drift shows as a spread

    def row(t, by):
        return {"us": round(t, 2), "bytes_mb": round(by / 1e6, 1),
                "frac_7p7": round(by / (t * 1e-6) / (HBM_DATASHEET_GBS * 1e9), 3)}

    return {"C": C, "H": H, "W": W, "B": B, "M": M, "hid": hid, "nbuf": nbuf,
            "pair": row(us["pair"], bytes_gemm + bytes_aff), "gemm_nt_f32": row(us["gemm"], bytes_gemm),
            "affine1x1_bwd": row(us["affine1x1_bwd"], bytes_aff), "fused": row(us["fused"], bytes_fused),
            "speedup": round(us["pair"] / us["fused"], 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="2048,64")
    ap.add_argument("--reps", type=int, default=40)
    ap.add_argument("--hid", type=int, default=512)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_dgrad1_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dgrad1_bench needs a CUDA device")
    res = {"gpu": gpu_info(), "levels": []}
    for B in (int(b) for b in a.batches.split(",")):
        for C, H in LEVELS:
            r = bench_level(C, H, B, a.hid, a.reps)
            res["levels"].append(r)
            print(f"B={B:5d} C={C:2d} {H}x{H}: pair {r['pair']['us']:7.1f} us (gemm {r['gemm_nt_f32']['us']:6.1f} + "
                  f"affine1x1_bwd {r['affine1x1_bwd']['us']:6.1f})  fused {r['fused']['us']:7.1f} us "
                  f"{r['fused']['bytes_mb']:6.1f} MB {r['fused']['frac_7p7']:.2f} of 7.7 TB/s  x{r['speedup']}",
                  file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
