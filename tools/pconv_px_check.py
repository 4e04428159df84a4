"""The pixel-major Conv2dZeros + coupling kernel of the 4x4-map level (csrc/pconv_px.cu) against pconv_coupling_kernel<48>
(NFK_PCONV_PX=0, run in a child process): outputs, saved conv outputs and log-dets must be bit-identical; then timing."""
import os, subprocess, sys, tempfile
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from nf_distillation_b200 import ops

CASES = [(2048, False, True), (70, False, False), (3, True, True), (257, True, False)]


def run(B, reverse, keep):
    dev = "cuda"
    C, H, W, hid = 48, 4, 4, 512
    M, K3p = B * H * W, ops.round_up(9 * C, 64)
    g = torch.Generator(device=dev).manual_seed(B)
    h2 = (torch.randn(M, hid, device=dev, generator=g).clamp_min(0) * 0.5).bfloat16()
    B3 = (torch.randn(K3p, hid, device=dev, generator=g) * 0.02).bfloat16()
    b3 = torch.randn(C, device=dev, generator=g) * 0.1
    y = torch.randn(B, C, H, W, device=dev, generator=g)
    ld = torch.zeros(B, device=dev)
    hs = torch.zeros(M, C, device=dev) if keep else None
    ops.pconv_coupling_fwd(h2, B3, K3p, b3, y, hs, ld, B, C, H, W, hid, reverse)
    torch.cuda.synchronize()
    return y.cpu(), ld.cpu(), (hs.cpu() if keep else None)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "child":
        torch.save([run(*c) for c in CASES], sys.argv[2])
        sys.exit(0)
    mine = [run(*c) for c in CASES]
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "pconv_px_ref.pt")
        subprocess.run([sys.executable, os.path.abspath(__file__), "child", path],
                       env=dict(os.environ, NFK_PCONV_PX="0"), check=True, timeout=300)
        ref = torch.load(path)
    ok = True
    for c, a, b in zip(CASES, mine, ref):
        eq_y = torch.equal(a[0], b[0])
        dl = (a[1] - b[1]).abs().max().item() / (b[1].abs().max().item() + 1e-12)   # log-det partial sums meet in atomics
        eq_h = a[2] is None or torch.equal(a[2], b[2])
        print(f"B={c[0]} reverse={c[1]} keep={c[2]}: y identical {eq_y}, hsave identical {eq_h}, logdet rel diff {dl:.2e}")
        ok = ok and eq_y and eq_h and dl < 1e-5
    print("OK" if ok else "MISMATCH")
    sys.exit(0 if ok else 1)
