"""CPU: the C-ABI library loads and exports every symbol include/nfk.h declares; host-side logic that needs no GPU."""
import ctypes
import os
import re
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "nfk.h")).read()
    return sorted(set(re.findall(r"\bint\s+(nfk_\w+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from nf_distillation_b200 import _lib
    syms = declared_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(_lib.LIB, s), f"{s} declared in include/nfk.h but not exported by libnfk.so"
    assert set(_lib.SIGNATURES) == set(syms), "ctypes signatures and header diverge"
    assert _lib.LIB.nfk_version() >= 1


def test_argument_errors_without_gpu():
    """Shape / argument validation happens before any CUDA call, so it is testable on the CPU."""
    from nf_distillation_b200 import _lib
    L = _lib.LIB
    assert L.nfk_gemm_nt_bf16(None, 64, None, 64, 128, 100, 64, 0, None, 64, None, None, 0, None, None) == -1
    assert L.nfk_gemm_nt_bf16(None, 64, None, 64, 128, 64, 60, 0, None, 64, None, None, 0, None, None) == -1
    assert L.nfk_invconv_prep(None, None, None, None, None, None, None, None, 12, 0, 0, None, None, None, None) == -3
    assert L.nfk_affine1x1_fwd(None, None, None, None, None, None, 0, None, None, 0, 12, 4, 4, None) == -1
    assert L.nfk_kd_mse_fwd(None, None, 4, 16, 1.0, None, None) == -3


def test_fused_conv_kernel_shape_limits():
    """nfk_cnet_fused_supported is the one statement of the fused conv kernel's shapes: hidden width 512 and a
    first-GEMM depth K that is a multiple of 64 and leaves shared memory for two weight slots (K <= 448). The entry
    points refuse K = 512 with NFK_ERR_SHAPE before any CUDA call, so callers take the two-GEMM path instead."""
    from nf_distillation_b200 import _lib, ops
    L = _lib.LIB
    for K in (64, 128, 256, 448):
        assert L.nfk_cnet_fused_supported(512, K) == 1 and ops.cnet_fused_supported(512, K), K
    for hid, K in ((512, 512), (512, 100), (256, 128), (512, 0), (512, 1 << 30)):
        assert L.nfk_cnet_fused_supported(hid, K) == 0 and not ops.cnet_fused_supported(hid, K), (hid, K)
    M = 8192
    assert L.nfk_cnet_fwd_fused(None, 512, None, None, None, None, None, None, None, None, M, M, 512, None) == -1
    assert L.nfk_cnet_fwd_fused_ranged(None, 512, None, None, None, None, None, None, None, None, M, M, 512, 8,
                                       None) == -1
    assert L.nfk_cnet_bwd_fused(None, 512, None, None, None, None, M, None, None, None, None, M, 512, None) == -1
    # a supported shape gets past the shape check to the argument checks (still no CUDA call)
    assert L.nfk_cnet_fwd_fused(None, 448, None, None, None, None, None, None, None, None, M, M, 512, None) == -3
    assert L.nfk_cnet_bwd_fused(None, 448, None, None, None, None, M, None, None, None, None, M, 512, None) == -3


def test_state_dict_keys_and_module_tree():
    from nf_distillation_b200.models import FlowStep, SqueezeLayer, create_glow_model
    cfg = dict(image_shape=[32, 32, 3], hidden_channels=64, K=2, L=3, actnorm_scale=1.0,
               flow_permutation="invconv", flow_coupling="affine", LU_decomposed=True, y_classes=10,
               learn_top=False, y_condition=False, is_1d=False)
    m = create_glow_model(cfg)
    sd = m.state_dict()
    for k in ("prior_h", "flow.layers.1.actnorm.bias", "flow.layers.1.invconv.lower", "flow.layers.1.invconv.p",
              "flow.layers.1.invconv.sign_s", "flow.layers.1.block.0.conv.weight",
              "flow.layers.1.block.0.actnorm.logs", "flow.layers.1.block.4.logs", "flow.layers.1.block.4.conv.bias",
              "flow.layers.3.conv.logs", "flow.layers.3.conv.conv.weight"):
        assert k in sd, k
    assert isinstance(m.flow.layers[0], SqueezeLayer) and isinstance(m.flow.layers[1], FlowStep)
    assert len(m.flow.layers) == 3 * (2 + 1) + 2
    assert m.flow.output_shapes[0] == [-1, 12, 16, 16] and m.flow.output_shapes[-1] == [-1, 48, 4, 4]
    assert all(mod.inited for mod in m.modules() if hasattr(mod, "inited"))
    mean, logs = m.prior(None)
    assert mean.shape == (32, 48, 4, 4) and logs.shape == (32, 48, 4, 4)
    with pytest.raises(RuntimeError):
        m(torch.zeros(2, 3, 32, 32), None)      # no CPU path: must fail loudly


# the torch seed each golden fixture was recorded with (oracle/make_golden.py main())
GOLDEN_SEEDS = {"glow2d_cifar_k2_h64": 42, "glow2d_16_k1_h64": 7, "glow2d_16_additive_shuffle_k2_h64": 17,
                "glow2d_16_affine_reverse_k2_h64": 19, "glow2d_16_learntop_k1_h64": 29, "glow1d_d6_k5_h32": 11,
                "glow1d_d63_k5_h32": 13, "kd2d_cifar_t4_s2_h64": 21, "kd1d_d63_t5_s3": 23, "kd1d_rich_t2_s2": 31}


def test_seeded_init_matches_reference_bit_for_bit():
    """Every golden fixture stores the state dict the unmodified reference built under torch.manual_seed(seed), after
    oracle/make_golden.py re-drew its zero-initialised tensors from Generator(seed + 1). The same seeds, create_glow_model
    and the same re-draw reproduce it key for key and bit for bit (student before teacher in the KD fixtures), and the
    fixed permutations of the variant fixtures index for index. The re-draw overwrites the zero-initialised tensors
    (ActNorm, Conv2dZeros, LinearZeros), so their zero initialisation is checked before it."""
    import warnings
    warnings.filterwarnings("ignore")
    from golden_util import cfg_of, load, state_dict_of
    from nf_distillation_b200.models import create_glow_model
    from nf_distillation_b200.models.layers import ActNorm1d, ActNorm2d, Conv2dZeros, LinearZeros
    from oracle.make_golden import randomise
    zero_init = (ActNorm1d, ActNorm2d, Conv2dZeros, LinearZeros)
    for name, seed in GOLDEN_SEEDS.items():
        d = load(name)
        keys = [("cfg", "sd.")] if "cfg" in d else [("s_cfg", "s_sd."), ("t_cfg", "t_sd.")]
        cfgs = [cfg_of(d, k) for k, _ in keys]
        torch.manual_seed(seed)
        gen = torch.Generator().manual_seed(seed + 1)
        models = [create_glow_model({k: v for k, v in c.items() if k != "perm_indices"}) for c in cfgs]
        for m in models:
            zeros = [p for mod in m.modules() if isinstance(mod, zero_init) for p in mod.parameters()]
            assert zeros and not any(p.any() for p in zeros), name
            randomise(m, gen)
        for (_, prefix), cfg, m in zip(keys, cfgs, models):
            ref, mine = state_dict_of(d, prefix), m.state_dict()
            assert set(ref) == set(mine), name
            assert all(torch.equal(ref[k], mine[k]) for k in ref), name
            for i, idx in cfg.get("perm_indices", {}).items():
                assert getattr(m.flow.layers[int(i)], cfg["flow_permutation"]).indices.tolist() == idx, (name, i)


def test_kd_indices_match_reference_rule():
    sys.path.insert(0, ROOT)
    from oracle import glow_oracle as O
    from nf_distillation_b200.pl_module import NFModel
    base = dict(actnorm_scale=1.0, flow_permutation="invconv", flow_coupling="affine", LU_decomposed=True,
                learn_top=False, y_condition=False)
    s = dict(base, image_shape=[32, 32, 3], hidden_channels=64, K=8, L=3, is_1d=False, y_classes=10)
    tch = dict(s, K=32)
    cfg = {"data": {"name": "cifar"}, "student": s, "teacher": tch,
           "loss": {"nll": {"weight": 0.9}, "kd": {"weight": 0.1, "name": "mse"},
                    "perceptual": {"weight": 0.0, "name": "l1"}},
           "optimizer": "adam", "learning_rate": 5e-4, "weight_decay": 0.0}
    m = NFModel(cfg)
    assert (m.student_kd_indices, m.teacher_kd_indices) == ([0, 10, 20, 28], [0, 34, 68, 100])   # SURVEY §3.2 probe
    assert (m.student_kd_indices, m.teacher_kd_indices) == O.kd_indices(s, tch)
    s1 = dict(base, image_shape=[63], hidden_channels=16, K=3, L=1, is_1d=True, y_classes=0)
    t1 = dict(s1, hidden_channels=32, K=5)
    cfg1 = dict(cfg, data={"name": "bsds300"}, student=s1, teacher=t1)
    m1 = NFModel(cfg1)
    assert (m1.student_kd_indices, m1.teacher_kd_indices) == ([1, 2], [3, 4])
    assert isinstance(m.configure_optimizers(), torch.optim.Adam)


def test_checkpoints_in_both_reference_formats_load(tmp_path):
    """pl_module.py:112-129: a raw state_dict, or a Lightning checkpoint whose keys carry the `student.` prefix (other
    entries, e.g. `teacher.*`, are ignored), load into the drop-in module unchanged."""
    import torch
    from nf_distillation_b200.pl_module import NFModel
    from nf_distillation_b200.models import create_glow_model
    from nf_distillation_b200.train import glow_cfg, kd_config
    cfg = glow_cfg((32, 32, 3), 2, 2, 64)
    torch.manual_seed(1)
    src = create_glow_model(cfg)
    with torch.no_grad():
        for p in src.parameters():
            p.add_(torch.randn_like(p) * 0.01)
    raw, lightning = tmp_path / "raw.ckpt", tmp_path / "pl.ckpt"
    torch.save(src.state_dict(), raw)
    torch.save({"epoch": 3, "state_dict": {**{"student." + k: v for k, v in src.state_dict().items()},
                                           "teacher.flow.layers.1.actnorm.bias": torch.zeros(1)}}, lightning)
    for path in (raw, lightning):
        s_cfg = dict(cfg, checkpoint=str(path))
        m = NFModel(kd_config(s_cfg, glow_cfg((32, 32, 3), 2, 2, 64), kd=0.0))   # kd = perceptual = 0: no teacher
        assert m.teacher is None
        got = m.student.state_dict()
        assert got.keys() == src.state_dict().keys()
        assert all(torch.equal(got[k].cpu(), v) for k, v in src.state_dict().items())


def test_pre_and_postprocess_match_the_reference_helpers():
    import torch
    from nf_distillation_b200 import data_utils as U
    g = torch.Generator().manual_seed(0)
    img = torch.randint(0, 256, (4, 3, 8, 8), generator=g).float() / 255.0
    x = U.preprocess(img)
    assert x.min() >= -0.5 and x.max() < 0.5
    assert torch.allclose(x, torch.round(img * 255) / 256 - 0.5, atol=1e-6)
    back = U.postprocess(x.clone())
    # (the reference scales by 1/256 on the way in and by 255 on the way out, so the round trip truncates: k*255/256)
    assert back.dtype == torch.uint8 and torch.equal(back, ((x + 0.5) * 255).byte())


def test_resident_inverse_job_table_reproduces_the_sequential_inverse():
    """nfk_made_inverse_jobs is host code: replay its job stream in fp32 torch (each job = one 8/16-unit tile of a
    hidden layer over the k-chunks it names, or the (mu_d, alpha_d) row pair) and compare with the paper
    restatement's D-pass inverse — the schedule the CUDA kernel executes finalises every unit exactly when its
    inputs are final, including degrees that own no unit (D > H) and tiles straddling two degrees."""
    import torch
    from nf_distillation_b200 import ops
    from nf_distillation_b200.models.maf import hidden_degrees
    from oracle import maf_oracle as MO
    for D, H in [(6, 512), (63, 512), (63, 192), (1, 64), (2, 64), (100, 64), (17, 128)]:
        torch.manual_seed(D)
        deg = hidden_degrees(D, H)
        pre = "l."
        sd = {pre + "deg1": deg, pre + "deg2": deg.clone(),
              pre + "fc1.weight": torch.randn(H, D) * 0.1, pre + "fc1.bias": torch.randn(H) * 0.1,
              pre + "fc2.weight": torch.randn(H, H) * 0.05, pre + "fc2.bias": torch.randn(H) * 0.1,
              pre + "fc3.weight": torch.randn(2 * D, H) * 0.02, pre + "fc3.bias": torch.randn(2 * D) * 0.1}
        m1, m2, m3 = MO.masks(D, deg.long(), deg.long())
        W1, W2, W3 = sd[pre + "fc1.weight"] * m1, sd[pre + "fc2.weight"] * m2, sd[pre + "fc3.weight"] * m3
        Dp = (D + 63) // 64 * 64
        W1p = torch.zeros(H, Dp)
        W1p[:, :D] = W1
        edges = torch.arange(D + 1)
        cnt = (deg.long()[None, :] <= edges[:, None]).sum(1)
        N3p = (2 * D + 63) // 64 * 64
        size_rows = lambda rows, kch: (rows * (kch * 32 + 16) + 127) // 128 * 128
        for push in (False, True):
            jobs = ops.made_inverse_jobs(cnt, cnt, D, H, Dp, N3p, push=push)
            aligned = all(int(i + 1) % 8 == 0 for i in (deg[1:] != deg[:-1]).nonzero().flatten())
            if push and (2 * D > 128 or not aligned):
                # more than 16 output tiles, or degrees that change inside an 8-unit tile (hidden_degrees keeps the
                # standard per-unit MADE assignment when there are fewer tiles than degrees): pull kernel only
                assert jobs is None
                continue
            # every x_d is finished exactly once: by a (mu, alpha) job of its own, or (push) by the step's last layer-2 job
            assert jobs.shape[1] == 8
            assert ((jobs[:, 0] & 3) == 2).sum().item() + (jobs[:, 7] != 0).sum().item() == D
            assert push or not (jobs[:, 7] != 0).any()

            def size(q):
                phase, kch, rows = q[0] & 3, q[0] >> 3, (2 if (q[0] & 3) == 2 else (16 if q[0] & 4 else 8))
                if not push:
                    return size_rows(rows, kch) if kch else 0
                return 0 if phase == 2 else (size_rows(rows, kch) if phase == 0 else size_rows(16, kch) + 2 * N3p * 16)
            # ring plan: 16-byte aligned ranges; a job never overwrites bytes of the `back - 1` jobs before it
            jl = jobs.tolist()
            soff = 0
            for j, q in enumerate(jl):
                assert q[2] % 16 == 0 and q[3] >= 1
                assert q[4] * 16 == soff and q[5] * 16 == size(q)      # packed stream: job after job
                soff += size(q)
                for b in range(1, min(q[3], len(jl)) if size(q) else 0):
                    o = jl[(j - b) % len(jl)]
                    assert not (q[2] < o[2] + size(o) and o[2] < q[2] + size(q)), (D, H, j, b)
            # replay: pull = h2 kept, (mu, alpha) recomputed from it per step; push = outputs accumulated as tiles finish
            u = torch.randn(19, D)
            uf = u.flip(1)
            xb, h1, h2 = torch.zeros(19, Dp), torch.zeros(19, H), torch.zeros(19, H)
            out = torch.zeros(19, 2 * D)
            x, ld = torch.zeros(19, D), torch.zeros(19)
            def finish(d, k):
                if push:
                    mu, al = out[:, d] + sd[pre + "fc3.bias"][d], out[:, D + d] + sd[pre + "fc3.bias"][D + d]
                else:
                    mu = h2[:, :k] @ W3[d, :k] + sd[pre + "fc3.bias"][d]
                    al = h2[:, :k] @ W3[D + d, :k] + sd[pre + "fc3.bias"][D + d]
                x[:, d] = uf[:, d] * torch.exp(al) + mu
                xb[:, d] = x[:, d]
                ld.add_(al)

            order = []
            for q in jl:
                desc, row0, fin = q[0], q[1], q[7]
                phase, two, kch = desc & 3, desc & 4, desc >> 3
                k = kch * 16
                o = slice(row0, row0 + (16 if two else 8))
                if phase == 0:
                    h1[:, o] = torch.relu(xb[:, :k] @ W1p[o, :k].T + sd[pre + "fc1.bias"][o])
                elif phase == 1:
                    h2[:, o] = torch.relu(h1[:, :k] @ W2[o, :k].T + sd[pre + "fc2.bias"][o])
                    if push:
                        out += h2[:, o] @ W3[:, o].T
                        if fin:
                            order.append(fin - 1)
                            finish(fin - 1, 0)
                else:
                    assert not push or kch == 0
                    order.append(row0)
                    finish(row0, k)
            assert order == list(range(D))
            x_o, a_o = MO.made_inverse(u, sd, pre, D)
            assert (x - x_o).abs().max().item() < 1e-5 * (x_o.abs().max().item() + 1), (D, H, push)
            assert (ld - a_o).abs().max().item() < 1e-5 * (a_o.abs().max().item() + 1), (D, H, push)
        continue
        x_o, a_o = MO.made_inverse(u, sd, pre, D)
        assert (x - x_o).abs().max().item() < 1e-5 * (x_o.abs().max().item() + 1), (D, H)
        assert (ld - a_o).abs().max().item() < 1e-5 * (a_o.abs().max().item() + 1), (D, H)


def test_resident_inverse_planner_error_codes():
    """Host entry points of the resident MADE inverse: bad arguments and unsupported shapes come back as error codes
    (no GPU touched); push planning refuses degrees that do not change on whole 8-unit tiles."""
    import ctypes
    import torch
    from nf_distillation_b200 import _lib, ops
    L = _lib.LIB
    D, H, Dp, N3p = 6, 64, 64, 64
    good = torch.tensor([0, 16, 24, 40, 48, 64, 64], dtype=torch.int32)          # tile-aligned, non-decreasing
    ragged = torch.tensor([0, 13, 26, 39, 52, 64, 64], dtype=torch.int32)        # sorted but not tile-aligned
    falling = torch.tensor([0, 16, 8, 40, 48, 64, 64], dtype=torch.int32)
    call = lambda c, push: L.nfk_made_inverse_jobs(c.data_ptr(), c.data_ptr(), D, H, Dp, N3p, push, None, 0)
    assert call(good, 0) > 0 and call(good, 1) > 0
    assert call(ragged, 0) > 0 and call(ragged, 1) == -1                         # NFK_ERR_SHAPE: pull kernel only
    assert call(falling, 0) == -3                                                # NFK_ERR_ARG
    assert L.nfk_made_inverse_jobs(None, None, D, H, Dp, N3p, 0, None, 0) == -3
    assert L.nfk_made_inverse_jobs(good.data_ptr(), good.data_ptr(), D, 100, Dp, N3p, 0, None, 0) == -1   # H % 64
    assert ops.made_inverse_jobs(ragged, ragged, D, H, Dp, N3p, push=True) is None
    assert L.nfk_made_inverse_resident_supported(D, H, Dp) == 1 and L.nfk_made_inverse_push_supported(D, H, Dp, N3p) == 1
    assert L.nfk_made_inverse_push_supported(100, 64, 128, 256) == 0             # 2D > 128: more than 16 output tiles
    # launch-side argument checks happen before any CUDA call
    assert L.nfk_made_inverse_resident(None, None, None, None, None, None, 1, 0, N3p, None, None, None, 4, D, H, Dp,
                                       1, 0, None) == -3
    assert L.nfk_made_inverse_pack(None, 1, None, None, None, N3p, D, H, Dp, 0, None, None) == -3


def test_reference_arm_of_the_bench_never_loads_the_product():
    """`bench.py --impl reference` times the reference's CPU algorithm (oracle port) with weights from the oracle's own
    seeded initialiser and must not touch the product: bench.py asserts, after the run, that no nf_distillation_b200
    module was imported into the process (so libnfk.so cannot have been mapped). Here: the arm runs, exits 0 (the
    assertion held) and prints one JSON line with the contract's keys."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "bench.py")).read()
    assert 'assert not any(m.startswith("nf_distillation_b200") for m in sys.modules)' in src
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--workload", "glow1d_bsds300_kd_t5_s3"], capture_output=True, text=True, timeout=300,
                         cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "port" and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["dtype"] == "f32"
