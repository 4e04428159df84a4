"""CPU: the host planner of the MADE inverse's reverse solve (nfk_made_inverse_bwd_jobs) and its error codes.

The math: for one MADE layer with forward u_d = (x_d - mu_d(x_<d)) e^{-alpha_d(x_<d)}, the inverse returns x and
ld_in + sum alpha(x). Given g_x and g_ld, one sweep d = D-1 .. 0 gives every gradient:
    c_d = sum_{k > d} (dmu_k/dx_d mubar_k + dalpha_k/dx_d alphabar_k),   mubar_d = g_x,d + c_d,
    v_d = e^{alpha_d} mubar_d,   alphabar_d = v_d u_d + g_ld;   g_u = v (output order),   g_ld_in = g_ld,
and the parameter gradients are the forward network's VJP at x from [mubar | alphabar]. The first test checks this
against torch.autograd through the paper restatement in fp64; the second replays the planner's job stream in fp32
torch, job by job as the CUDA kernel runs it, against that fp64 reference."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _layer(D, H, aligned, dtype, seed):
    from oracle import maf_oracle as MO
    g = torch.Generator().manual_seed(seed)
    if aligned:
        deg = MO.hidden_degrees(D, H).to(torch.int32)
    else:   # the per-unit assignment (degree changes inside 8-unit tiles)
        deg = (torch.arange(H) * max(D - 1, 1) // H + 1).to(torch.int32) if D > 1 else torch.ones(H, dtype=torch.int32)
    r = lambda *s: torch.randn(*s, generator=g, dtype=dtype)
    return {"l.deg1": deg, "l.deg2": deg.clone(),
            "l.fc1.weight": r(H, D) * 0.3, "l.fc1.bias": r(H) * 0.1, "l.fc2.weight": r(H, H) * 0.1,
            "l.fc2.bias": r(H) * 0.1, "l.fc3.weight": r(2 * D, H) * 0.05, "l.fc3.bias": r(2 * D) * 0.1}


def _autograd_reference(sd, D, flip, u, gx, gld):
    """fp64 gradients of <x, gx> + <sum alpha, gld> through the sequential inverse: (g_u, {param: grad})."""
    from oracle import maf_oracle as MO
    u = u.clone().requires_grad_(True)
    p = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    x, sa = MO.made_inverse(u, p, "l.", D, flip=flip)
    ((x * gx).sum() + (sa * gld).sum()).backward()
    return x.detach(), u.grad, {k: v.grad for k, v in p.items() if v.is_floating_point()}


def _param_vjp(sd, D, x, mub, alb):
    """Parameter gradients of sum(mu mubar + alpha alphabar) at fixed x (the forward network's VJP)."""
    from oracle import maf_oracle as MO
    p = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    xr = x.clone().requires_grad_(True)
    mu, al = MO.made_net(xr, p, "l.", D)
    ((mu * mub).sum() + (al * alb).sum()).backward()
    return xr.grad, {k: v.grad for k, v in p.items() if v.is_floating_point()}


@pytest.mark.parametrize("flip", [False, True])
def test_reverse_sweep_equals_autograd_in_fp64(flip):
    """The sweep above, with c_d from the network's VJP of the rows already final, against autograd through the
    restatement's inverse: g_u, every parameter gradient, and the identity (the forward chain's input gradient at x,
    from ubar = -v and ld-bar = -g_ld, equals -g_x)."""
    from oracle import maf_oracle as MO
    D, H, B = 7, 64, 5
    sd = _layer(D, H, True, torch.float64, 0)
    u, gx, gld = torch.randn(B, D, dtype=torch.float64), torch.randn(B, D, dtype=torch.float64), torch.randn(B, dtype=torch.float64)
    x, gu_ref, gp_ref = _autograd_reference(sd, D, flip, u, gx, gld)
    mu, al = MO.made_net(x, sd, "l.", D)
    uu = (x - mu) * torch.exp(-al)
    mub, alb, v = (torch.zeros(B, D, dtype=torch.float64) for _ in range(3))
    for d in reversed(range(D)):
        c, _ = _param_vjp(sd, D, x, mub, alb)
        mub[:, d] = gx[:, d] + c[:, d]
        v[:, d] = torch.exp(al[:, d]) * mub[:, d]
        alb[:, d] = v[:, d] * uu[:, d] + gld
    g_u = v.flip(1) if flip else v
    assert (g_u - gu_ref).abs().max().item() < 1e-12
    c, gp = _param_vjp(sd, D, x, mub, alb)
    for k in gp:
        assert (gp[k] - gp_ref[k]).abs().max().item() < 1e-12, k
    assert (c - mub + gx).abs().max().item() < 1e-12   # chain dx = c - mubar = -g_x


def _replay(jobs, sd, D, H, x, u_out, gx, gld, flip):
    """Run the planner's job stream in fp32 torch: (g_u, mubar, alphabar). Straddling tiles and k-ranges that start
    below the first final unit hold scratch / zero values that must only meet masked-zero weights."""
    from oracle import maf_oracle as MO
    deg = sd["l.deg1"].long()
    m1, m2, m3 = MO.masks(D, deg, sd["l.deg2"].long())
    W1, W2, W3 = sd["l.fc1.weight"] * m1, sd["l.fc2.weight"] * m2, sd["l.fc3.weight"] * m3
    h1 = torch.relu(x @ W1.T + sd["l.fc1.bias"])
    h2 = torch.relu(h1 @ W2.T + sd["l.fc2.bias"])
    out = h2 @ W3.T + sd["l.fc3.bias"]
    r1, r2 = (h1 > 0).float(), (h2 > 0).float()
    B = x.shape[0]
    N3p = (2 * D + 63) // 64 * 64
    B3T = torch.zeros(H, N3p)
    B3T[:, :2 * D] = W3.T
    B2T, B1T = W2.T.contiguous(), W1.T.contiguous()      # [H (layer 1), H (layer 2)], [D, H]
    u = u_out.flip(1) if flip else u_out                   # input order
    ds, g2, g1 = torch.zeros(B, N3p), torch.zeros(B, H), torch.zeros(B, H)
    g_u = torch.full((B, D), float("nan"))
    order = []
    for q in jobs.tolist():
        phase, two, kch, row0, k0 = q[0] & 3, (q[0] >> 2) & 1, q[0] >> 3, q[1], q[6]
        k = slice(k0 * 16, (k0 + kch) * 16)
        o = slice(row0, min(row0 + (16 if two else 8), H))
        if phase == 1:
            g2[:, o] = r2[:, o] * (ds[:, k] @ B3T[o, k].T)
        elif phase == 0:
            g1[:, o] = r1[:, o] * (g2[:, k] @ B2T[o, k].T)
        else:
            d = row0
            order.append(d)
            c = g1[:, k] @ B1T[d, k]
            mub = gx[:, d] + c
            v = torch.exp(out[:, D + d]) * mub
            ds[:, d], ds[:, D + d] = mub, v * u[:, d] + gld
            g_u[:, D - 1 - d if flip else d] = v
    assert order == list(reversed(range(D)))
    return g_u, ds[:, :D], ds[:, D:2 * D]


@pytest.mark.parametrize("D", [1, 2, 6, 17, 63, 100])
@pytest.mark.parametrize("H", [64, 512])
def test_reverse_job_table_reproduces_the_fp64_sweep(D, H):
    """nfk_made_inverse_bwd_jobs is host code: replay its job stream (layer-2 tile pairs from the finished dout rows,
    layer-1 tile pairs, then c_d and row d) in fp32 and compare with fp64 autograd through the restatement's inverse,
    for tile-aligned and per-unit degrees and both flips; the ring plan keeps every job's bytes alive until it is used."""
    from nf_distillation_b200 import ops
    N3p = (2 * D + 63) // 64 * 64
    B = 6
    for aligned in (True, False):
        sd64 = _layer(D, H, aligned, torch.float64, D * 31 + H)
        deg = sd64["l.deg1"].long()
        cnt = (deg[None, :] <= torch.arange(D + 1)[:, None]).sum(1)
        jobs = ops.made_inverse_bwd_jobs(cnt, cnt, D, H, N3p)
        assert jobs.shape[1] == 8 and ((jobs[:, 0] & 3) == 2).sum().item() == D
        size = lambda q: 0 if (q[0] >> 3) == 0 else \
            ((1 if (q[0] & 3) == 2 else (16 if q[0] & 4 else 8)) * ((q[0] >> 3) * 32 + 16) + 127) // 128 * 128
        jl = jobs.tolist()
        soff = 0
        for j, q in enumerate(jl):
            assert q[4] * 16 == soff and q[5] * 16 == size(q) and q[3] >= 1
            assert q[6] * 16 + (q[0] >> 3) * 16 <= (N3p if (q[0] & 3) == 1 else H)
            soff += size(q)
            for b in range(1, min(q[3], len(jl)) if size(q) else 0):
                o = jl[(j - b) % len(jl)]
                assert not (q[2] < o[2] + size(o) and o[2] < q[2] + size(q)), (D, H, j, b)
        for flip in (False, True):
            g = torch.Generator().manual_seed(D + H + flip)
            u = torch.randn(B, D, generator=g, dtype=torch.float64)
            gx = torch.randn(B, D, generator=g, dtype=torch.float64)
            gld = torch.randn(B, generator=g, dtype=torch.float64)
            x, gu_ref, gp_ref = _autograd_reference(sd64, D, flip, u, gx, gld)
            sd32 = {k: (v.float() if v.is_floating_point() else v) for k, v in sd64.items()}
            g_u, mub, alb = _replay(jobs, sd32, D, H, x.float(), u.float(), gx.float(), gld.float(), flip)
            tol = lambda ref: 1e-4 * (ref.abs().max().item() + 1e-3)
            assert (g_u.double() - gu_ref).abs().max().item() < tol(gu_ref), (aligned, flip)
            _, gp = _param_vjp(sd64, D, x, mub.double(), alb.double())
            for k in gp:
                assert (gp[k] - gp_ref[k]).abs().max().item() < tol(gp_ref[k]), (aligned, flip, k)


def test_reverse_solve_error_codes():
    """Host entry points of the reverse solve: bad arguments and unsupported shapes come back as error codes before
    any CUDA call."""
    from nf_distillation_b200 import _lib
    L = _lib.LIB
    D, H, N3p = 6, 64, 64
    good = torch.tensor([0, 16, 24, 40, 48, 64, 64], dtype=torch.int32)
    falling = torch.tensor([0, 16, 8, 40, 48, 64, 64], dtype=torch.int32)
    assert L.nfk_made_inverse_bwd_supported(D, H, N3p) == 1
    assert L.nfk_made_inverse_bwd_supported(D, 100, N3p) == 0          # H % 64
    assert L.nfk_made_inverse_bwd_supported(40, H, 64) == 0            # N3p < 2D
    assert L.nfk_made_inverse_bwd_jobs(good.data_ptr(), good.data_ptr(), D, H, N3p, None, 0) > 0
    assert L.nfk_made_inverse_bwd_jobs(falling.data_ptr(), falling.data_ptr(), D, H, N3p, None, 0) == -3
    assert L.nfk_made_inverse_bwd_jobs(None, None, D, H, N3p, None, 0) == -3
    assert L.nfk_made_inverse_bwd_jobs(good.data_ptr(), good.data_ptr(), D, 100, N3p, None, 0) == -1
    assert L.nfk_made_inverse_bwd_pack(None, 1, None, None, None, D, H, N3p, None, None) == -3
    assert L.nfk_made_inverse_bwd_pack(None, 1, None, None, None, D, 100, N3p, None, None) == -1
    assert L.nfk_made_inverse_bwd_resident(None, None, None, None, None, None, None, None, 1, None, None, None, 4, D, H,
                                           N3p, 1, 0, None) == -3
    assert L.nfk_made_inverse_bwd_resident(None, None, None, None, None, None, None, None, 1, None, None, None, 4, D,
                                           100, N3p, 1, 0, None) == -1
    assert L.nfk_made_inv_bwd_update(None, 0, None, None, None, N3p, None, None, None, None, 4, D, 0, 1, None) == -3
    assert L.nfk_made_inv_bwd_update(None, 0, None, None, None, N3p, None, None, None, None, 4, D, D, 1, None) == -1
