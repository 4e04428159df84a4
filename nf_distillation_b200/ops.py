"""Tensor-level wrappers over the libnfk C-ABI (include/nfk.h): shape/dtype checks, pointer extraction, error
codes -> exceptions. No arithmetic happens here and there is no fallback path: every call lands in a CUDA kernel.
"""
from __future__ import annotations

import ctypes

import torch

from ._lib import LIB, check

EPI_F32, EPI_BIAS_RELU_BF16, EPI_MASK_BF16 = 0, 1, 2

_LAUNCHES = 0  # kernels launched through this module (bench.py reports it as gpu_launches)


def launch_count() -> int:
    return _LAUNCHES


def _p(t):
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "libnfk needs contiguous CUDA tensors"
    return t.data_ptr()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _count(n=1):
    global _LAUNCHES
    _LAUNCHES += n


def round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def relu_mask_like(M, N, device):
    """Storage for the 1-bit ReLU mask of an [M, N] activation: int32 words, word-major [ceil(N/32), M] so that the
    32 rows a warp owns are contiguous (coalesced writes in the forward epilogue, coalesced reads in the dgrad's)."""
    return torch.empty((N + 31) // 32, M, device=device, dtype=torch.int32)


def gemm_nt(A, B, M, N, K, epi, out, bias=None, aux=None, colsum=None):
    """out[M,N] = A[M,K] @ B[N,K]^T on tcgen05 (bf16 operands, fp32 TMEM accumulate) with a fused epilogue.
    aux = 1-bit ReLU mask (relu_mask_like): written by EPI_BIAS_RELU_BF16 (optional), read by EPI_MASK_BF16."""
    assert A.dtype == torch.bfloat16 and B.dtype == torch.bfloat16
    assert aux is None or aux.dtype == torch.int32
    _count()
    check(LIB.nfk_gemm_nt_bf16(_p(A), A.stride(0), _p(B), B.stride(0), M, N, K, epi, _p(out), out.stride(0),
                               _p(bias), _p(aux), 0 if aux is None else aux.stride(0), _p(colsum), _st()),
          "nfk_gemm_nt_bf16")


def gemm_tn(A, B, Mo, No, Kpix, out):
    """out[Mo,No] += A[Kpix,Mo]^T @ B[Kpix,No] (split-K over pixels, fp32 red.add); out must be zeroed."""
    assert A.dtype == torch.bfloat16 and B.dtype == torch.bfloat16 and out.dtype == torch.float32
    _count()
    check(LIB.nfk_gemm_tn_bf16(_p(A), A.stride(0), _p(B), B.stride(0), Mo, No, Kpix, _p(out), out.stride(0),
                               sm_count(), _st()), "nfk_gemm_tn_bf16")


_SM = {}


def sm_count() -> int:
    d = torch.cuda.current_device()
    if d not in _SM:
        _SM[d] = torch.cuda.get_device_properties(d).multi_processor_count
    return _SM[d]


def invconv_item(an_bias, an_logs, lower, upper, log_s, p, sign_s, weight, C, reverse, transpose, outW, outb, out_sl):
    """One nfk_invconv_item (include/nfk.h) for invconv_prep_batch."""
    from ._lib import InvconvItem
    return InvconvItem(_p(an_bias), _p(an_logs), _p(lower), _p(upper), _p(log_s), _p(p), _p(sign_s), _p(weight), C,
                       int(reverse), int(transpose), _p(outW), _p(outb), _p(out_sl))


def invconv_prep_batch(items):
    """Fused ActNorm o invconv matrices of many FlowSteps in one launch (one CTA per step)."""
    from ._lib import InvconvItem
    n = len(items)
    if not n:
        return
    arr = (InvconvItem * n)(*items)
    _count((n + 23) // 24)
    check(LIB.nfk_invconv_prep_batch(n, ctypes.addressof(arr), _st()), "nfk_invconv_prep_batch")


def invconv_bwd_item(fwd_item, dWf_ptr, dWf_ld, dbf, g_ld, B, pixels, d_bias, d_logs, d_lower, d_upper, d_log_s,
                     d_weight=None):
    from ._lib import InvconvBwdItem
    return InvconvBwdItem(fwd_item, dWf_ptr, dWf_ld, _p(dbf), _p(g_ld), B, float(pixels), _p(d_bias), _p(d_logs),
                          _p(d_lower), _p(d_upper), _p(d_log_s), _p(d_weight))


def invconv_prep_bwd_batch(items):
    from ._lib import InvconvBwdItem
    n = len(items)
    if not n:
        return
    arr = (InvconvBwdItem * n)(*items)
    _count((n + 23) // 24)
    check(LIB.nfk_invconv_prep_bwd_batch(n, ctypes.addressof(arr), _st()), "nfk_invconv_prep_bwd_batch")


def coupling_item(cw, cin, hid, cout, K1p, K3p, with_t, B1, B1T, B2, B2T, B3, B3T, bias1, bias2, bias3):
    from ._lib import CouplingItem
    return CouplingItem(*[_p(t) for t in cw], cin, hid, cout, K1p, K3p, int(with_t), _p(B1), _p(B1T), _p(B2), _p(B2T),
                        _p(B3), _p(B3T), _p(bias1), _p(bias2), _p(bias3))


def coupling_prep_batch(items):
    """bf16 GEMM operands of the coupling nets of many FlowSteps in one launch."""
    from ._lib import CouplingItem
    n = len(items)
    if not n:
        return
    arr = (CouplingItem * n)(*items)
    _count((n + 15) // 16)
    check(LIB.nfk_coupling_prep_batch(n, ctypes.addressof(arr), _st()), "nfk_coupling_prep_batch")


def coupling_bwd_item(fwd_item, gin, gout):
    from ._lib import CouplingBwdItem
    return CouplingBwdItem(fwd_item, *[_p(t) for t in gin], *[_p(t) for t in gout])


def coupling_prep_bwd_batch(items):
    from ._lib import CouplingBwdItem
    n = len(items)
    if not n:
        return
    arr = (CouplingBwdItem * n)(*items)
    _count((n + 11) // 12)
    check(LIB.nfk_coupling_prep_bwd_batch(n, ctypes.addressof(arr), _st()), "nfk_coupling_prep_bwd_batch")


def affine1x1_fwd(x, Wf, bf, sl, y, col, K1p, ld_in, ld_out, B, C, H, W):
    _count()
    check(LIB.nfk_affine1x1_fwd(_p(x), _p(Wf), _p(bf), _p(sl), _p(y), _p(col), K1p, _p(ld_in), _p(ld_out), B, C, H,
                                W, _st()), "nfk_affine1x1_fwd")


def coupling_fwd(P, K3p, bias3, y, hsave, ld, B, C, H, W, reverse):
    _count()
    check(LIB.nfk_coupling_fwd(_p(P), K3p, _p(bias3), _p(y), _p(hsave), _p(ld), B, C, H, W, int(reverse), _st()),
          "nfk_coupling_fwd")


def coupling_bwd(g_out, g_ld, z_out, hsave, dy, dhcol, K3p, dbias3, B, C, H, W):
    _count()
    check(LIB.nfk_coupling_bwd(_p(g_out), _p(g_ld), _p(z_out), _p(hsave), _p(dy), _p(dhcol), K3p, _p(dbias3), B, C,
                               H, W, _st()), "nfk_coupling_bwd")


def affine1x1_bwd(dy, dcol, K1p, x, Wf, dx, dWf, dbf, B, C, H, W):
    _count()
    check(LIB.nfk_affine1x1_bwd(_p(dy), _p(dcol), K1p, _p(x), _p(Wf), _p(dx), _p(dWf), _p(dbf), B, C, H, W, _st()),
          "nfk_affine1x1_bwd")


def coupling_inv_bwd(g_zc, g_ld, zc, hsave, dz, dhcol, K3p, dbias3, B, C, H, W):
    """Backward of the inverse affine coupling (include/nfk.h: nfk_coupling_inv_bwd)."""
    _count()
    check(LIB.nfk_coupling_inv_bwd(_p(g_zc), _p(g_ld), _p(zc), _p(hsave), _p(dz), _p(dhcol), K3p, _p(dbias3), B, C,
                                   H, W, _st()), "nfk_coupling_inv_bwd")


def col2im_add(dcol, K1p, dz, B, C, H, W):
    """dz[:, :C/2] += col2im(dcol) in place (include/nfk.h: nfk_col2im_add)."""
    _count()
    check(LIB.nfk_col2im_add(_p(dcol), K1p, _p(dz), B, C, H, W, _st()), "nfk_col2im_add")


def split2d_fwd(x, w, bias, logs, z1_out, ld, B, C, H, W, z1_sq=None):
    """z1_sq (optional): the squeezed copy of z1 written in the same pass (the next level's input)."""
    _count()
    check(LIB.nfk_split2d_squeeze_fwd(_p(x), _p(w), _p(bias), _p(logs), _p(z1_out), _p(z1_sq), _p(ld), B, C, H, W,
                                      _st()), "nfk_split2d_squeeze_fwd")


def dequant_squeeze(src, noise, x_out, sq_out, n_bits=8):
    """preprocess (uint8 src) + dequantisation noise + first squeeze in one pass (csrc/preproc.cu)."""
    _count()
    B, C, H, W = src.shape
    check(LIB.nfk_dequant_squeeze(_p(src), int(src.dtype == torch.uint8), n_bits, _p(noise), _p(x_out), _p(sq_out),
                                  B, C, H, W, _st()), "nfk_dequant_squeeze")


def split2d_rev(z1, w, bias, logs, eps, temperature, out, B, C, H, W):
    _count()
    check(LIB.nfk_split2d_rev(_p(z1), _p(w), _p(bias), _p(logs), _p(eps), float(temperature), _p(out), B, C, H, W,
                              _st()), "nfk_split2d_rev")


def split2d_bwd(x, w, bias, logs, g_z1, g_ld, dx, dw, dbias, dlogs, B, C, H, W, g_z1_sq=None):
    _count()
    check(LIB.nfk_split2d_squeeze_bwd(_p(x), _p(w), _p(bias), _p(logs), _p(g_z1), _p(g_z1_sq), _p(g_ld), _p(dx),
                                      _p(dw), _p(dbias), _p(dlogs), B, C, H, W, _st()), "nfk_split2d_squeeze_bwd")


def prior_bpd_fwd(z, mean, logs, logdet, B, n, scale, out):
    _count()
    check(LIB.nfk_prior_bpd_fwd(_p(z), _p(mean), _p(logs), _p(logdet), B, n, float(scale), _p(out), _st()),
          "nfk_prior_bpd_fwd")


def prior_bpd_bwd(z, mean, logs, g_bpd, B, n, scale, dz, dlogdet):
    _count()
    check(LIB.nfk_prior_bpd_bwd(_p(z), _p(mean), _p(logs), _p(g_bpd), B, n, float(scale), _p(dz), _p(dlogdet),
                                _st()), "nfk_prior_bpd_bwd")


def kd_mse_fwd(s, t, B, n, scale, acc):
    _count()
    check(LIB.nfk_kd_mse_fwd(_p(s), _p(t), B, n, float(scale), _p(acc), _st()), "nfk_kd_mse_fwd")


def kd_mse_bwd(s, t, g, B, n, scale, ds, accumulate=False):
    _count()
    check(LIB.nfk_kd_mse_bwd(_p(s), _p(t), _p(g), B, n, float(scale), _p(ds), int(accumulate), _st()),
          "nfk_kd_mse_bwd")


def pconv_coupling_supported(C, H, W, hid):
    return bool(LIB.nfk_pconv_coupling_supported(C, H, W, hid))


def pconv_coupling_fwd(h2, B3, K3p, bias3, y, hsave, ld, B, C, H, W, hid, reverse):
    """Conv2dZeros (per-tap tcgen05 products + col2im) fused with the affine coupling; y / ld updated in place."""
    _count()
    check(LIB.nfk_pconv_coupling_fwd(_p(h2), _p(B3), K3p, _p(bias3), _p(y), _p(hsave), _p(ld), B, C, H, W, hid,
                                     int(reverse), _st()), "nfk_pconv_coupling_fwd")


def conv1_dgrad_affine_bwd_supported(C, H, W, hid):
    return bool(LIB.nfk_conv1_dgrad_affine_bwd_supported(C, H, W, hid))


def conv1_dgrad_affine_bwd(dpre1, B1T, K1p, dy, x, Wf, dx, dWf, dbf, B, C, H, W, hid):
    """First conv's input gradient (per-tap tcgen05 products + col2im) fused with affine1x1_bwd; dWf / dbf accumulate."""
    assert dpre1.dtype == torch.bfloat16 and B1T.dtype == torch.bfloat16
    _count()
    check(LIB.nfk_conv1_dgrad_affine_bwd(_p(dpre1), _p(B1T), K1p, _p(dy), _p(x), _p(Wf), _p(dx), _p(dWf), _p(dbf), B,
                                         C, H, W, hid, _st()), "nfk_conv1_dgrad_affine_bwd")


def flow1d_supported(D, Cc, hid, training=False):
    return bool(LIB.nfk_flow1d_supported(D, Cc, hid, int(training)))


def flow1d_sizes(D, Cc, hid):
    """(total_fwd, total_bwd, total_grad, n_act, per-layer [(offG, offGB, ninp, noutp)] * 7)."""
    import ctypes
    vals = [ctypes.c_int() for _ in range(4)]
    offs = (ctypes.c_int * 28)()
    check(LIB.nfk_flow1d_sizes(D, Cc, hid, *[ctypes.addressof(v) for v in vals], ctypes.addressof(offs)),
          "nfk_flow1d_sizes")
    return (*[v.value for v in vals], [tuple(offs[4 * l:4 * l + 4]) for l in range(7)])


def flow1d_pack(Wf, bf, ws, bs, D, Cc, hid, PF, PB):
    import ctypes
    _count()
    wa = (ctypes.c_void_p * 6)(*[_p(t) for t in ws])
    ba = (ctypes.c_void_p * 6)(*[_p(t) for t in bs])
    check(LIB.nfk_flow1d_pack(_p(Wf), _p(bf), ctypes.addressof(wa), ctypes.addressof(ba), D, Cc, hid, _p(PF), _p(PB),
                              _st()), "nfk_flow1d_pack")


def flow1d_fwd(x, cond, PF, sl, y, ld_in, ld_out, acts, B, D, Cc, hid, reverse):
    _count()
    check(LIB.nfk_flow1d_fwd(_p(x), _p(cond), _p(PF), _p(sl), _p(y), _p(ld_in), _p(ld_out), _p(acts), B, D, Cc, hid,
                             int(reverse), _st()), "nfk_flow1d_fwd")


def flow1d_bwd(x_in, cond, acts, PB, y_out, g_out, g_ld, dx, G, B, D, Cc, hid, reverse):
    _count()
    check(LIB.nfk_flow1d_bwd(_p(x_in), _p(cond), _p(acts), _p(PB), _p(y_out), _p(g_out), _p(g_ld), _p(dx), _p(G), B, D,
                             Cc, hid, int(reverse), _st()), "nfk_flow1d_bwd")


def affine_rows(x, Wf, bf, sl, y, ld_in, ld_out, B, D, pixels):
    _count()
    check(LIB.nfk_affine_rows(_p(x), _p(Wf), _p(bf), _p(sl), _p(y), _p(ld_in), _p(ld_out), B, D, float(pixels),
                              _st()), "nfk_affine_rows")


def gemm_nt_ranged(A, B, M, N, K, epi, out, bn, kb_begin, kb_end, bias=None, aux=None, colsum=None):
    """gemm_nt with tile width bn and per-n-tile k-block ranges (structurally-zero mask tiles are never loaded)."""
    import ctypes
    _count()
    n = len(kb_begin)
    kb0 = (ctypes.c_int * n)(*kb_begin)
    kb1 = (ctypes.c_int * n)(*kb_end)
    check(LIB.nfk_gemm_nt_bf16_ranged(_p(A), A.stride(0), _p(B), B.stride(0), M, N, K, epi, _p(out), out.stride(0),
                                      _p(bias), _p(aux), 0 if aux is None else aux.stride(0), _p(colsum), bn,
                                      ctypes.addressof(kb0), ctypes.addressof(kb1), _st()), "nfk_gemm_nt_bf16_ranged")


def made_prep(w1, w2, w3, deg1, deg2, D, H, Dp, N3p, B1, B1T, B2, B2T, B3, B3T, with_t):
    _count()
    check(LIB.nfk_made_prep(_p(w1), _p(w2), _p(w3), _p(deg1), _p(deg2), D, H, Dp, N3p, _p(B1), _p(B1T), _p(B2),
                            _p(B2T), _p(B3), _p(B3T), int(with_t), _st()), "nfk_made_prep")


def made_prep_bwd(dB1, dB2, dB3, deg1, deg2, D, H, Dp, dw1, dw2, dw3):
    _count()
    check(LIB.nfk_made_prep_bwd(_p(dB1), _p(dB2), _p(dB3), _p(deg1), _p(deg2), D, H, Dp, _p(dw1), _p(dw2), _p(dw3),
                                _st()), "nfk_made_prep_bwd")


def rows_to_bf16(x, B, D, Dp, xb):
    _count()
    check(LIB.nfk_rows_to_bf16(_p(x), B, D, Dp, _p(xb), _st()), "nfk_rows_to_bf16")


def made_affine_fwd(x, out, N3p, u, ub, Dp, ld_in, ld_out, B, D, flip):
    _count()
    check(LIB.nfk_made_affine_fwd(_p(x), _p(out), N3p, _p(u), _p(ub), Dp, _p(ld_in), _p(ld_out), B, D, int(flip),
                                  _st()), "nfk_made_affine_fwd")


def made_affine_bwd(x, out, N3p, g_u, g_ld, dx, dout, db3, B, D, flip):
    _count()
    check(LIB.nfk_made_affine_bwd(_p(x), _p(out), N3p, _p(g_u), _p(g_ld), _p(dx), _p(dout), _p(db3), B, D, int(flip),
                                  _st()), "nfk_made_affine_bwd")


def made_inv_update(x, xb, Dp, u_in, out, N3p, ld_in, ld_out, B, D, i, flip, last):
    _count()
    check(LIB.nfk_made_inv_update(_p(x), _p(xb), Dp, _p(u_in), _p(out), N3p, _p(ld_in), _p(ld_out), B, D, i,
                                  int(flip), int(last), _st()), "nfk_made_inv_update")


def made_inverse_resident_supported(D, H, Dp) -> bool:
    return bool(LIB.nfk_made_inverse_resident_supported(D, H, Dp))


def made_inverse_push_supported(D, H, Dp, N3p) -> bool:
    return bool(LIB.nfk_made_inverse_push_supported(D, H, Dp, N3p))


def made_inverse_jobs(cnt1, cnt2, D, H, Dp, N3p=0, push=False):
    """Host-side job table of the resident inverse from the degree counts (CPU int32 tensors [D+1]) -> [njobs, 8]:
    (phase | two << 2 | k-chunks << 3, first row, weight-ring byte offset, jobs back to the ring bytes' last user,
    packed-stream offset / 16, bytes / 16, 0, 0). Returns None when push=True and the degrees do not change on whole
    8-unit tiles (or the shape does not fit the push kernel)."""
    import torch
    cnt1 = cnt1.to(torch.int32).contiguous().cpu()
    cnt2 = cnt2.to(torch.int32).contiguous().cpu()
    n = LIB.nfk_made_inverse_jobs(cnt1.data_ptr(), cnt2.data_ptr(), D, H, Dp, N3p, int(push), None, 0)
    if push and n == -1:     # NFK_ERR_SHAPE: not tile-aligned / not supported -> caller uses the pull kernel
        return None
    if n <= 0:
        check(n if n < 0 else -1, "nfk_made_inverse_jobs")
    jobs = torch.empty(n, 8, dtype=torch.int32)
    check(0 if LIB.nfk_made_inverse_jobs(cnt1.data_ptr(), cnt2.data_ptr(), D, H, Dp, N3p, int(push), jobs.data_ptr(),
                                         n) == n else -1, "nfk_made_inverse_jobs")
    return jobs


def made_inverse_pack(jobs_dev, B1, B2, B3, N3p, D, H, Dp, push, wstream):
    """Weights of every job, packed job after job in the shared-memory layout the inverse kernel copies in one piece."""
    _count()
    check(LIB.nfk_made_inverse_pack(_p(jobs_dev), jobs_dev.shape[0], _p(B1), _p(B2), _p(B3), N3p, D, H, Dp, int(push),
                                    _p(wstream), _st()), "nfk_made_inverse_pack")


def made_inverse_resident(u_in, wstream, b1, b2, b3, jobs, push, N3p, x, ld_in, ld_out, B, D, H, Dp, flip, mtiles=0):
    """The whole sequential inverse of one MADE layer in one launch (activations resident in shared memory)."""
    _count()
    check(LIB.nfk_made_inverse_resident(_p(u_in), _p(wstream), _p(b1), _p(b2), _p(b3), _p(jobs), jobs.shape[0],
                                        int(push), N3p, _p(x), _p(ld_in), _p(ld_out), B, D, H, Dp, int(flip),
                                        int(mtiles), _st()), "nfk_made_inverse_resident")


def made_inv_bwd_update(c, ldc, g_x, g_ld, out, N3p, u_in, g_u, dout, db3, B, D, d, flip):
    """Pass d of the D-pass reverse solve (gradients of the sequential inverse); c = None at d = D-1."""
    _count()
    check(LIB.nfk_made_inv_bwd_update(_p(c), ldc, _p(g_x), _p(g_ld), _p(out), N3p, _p(u_in), _p(g_u), _p(dout),
                                      _p(db3), B, D, d, int(flip), _st()), "nfk_made_inv_bwd_update")


def made_inverse_bwd_supported(D, H, N3p) -> bool:
    return bool(LIB.nfk_made_inverse_bwd_supported(D, H, N3p))


def made_inverse_bwd_jobs(cnt1, cnt2, D, H, N3p):
    """Host-side job table of the one-launch reverse solve (same counts and layout as made_inverse_jobs; column 6 =
    first k-chunk of the job), steps D-1 .. 0."""
    import torch
    cnt1 = cnt1.to(torch.int32).contiguous().cpu()
    cnt2 = cnt2.to(torch.int32).contiguous().cpu()
    n = LIB.nfk_made_inverse_bwd_jobs(cnt1.data_ptr(), cnt2.data_ptr(), D, H, N3p, None, 0)
    if n <= 0:
        check(n if n < 0 else -1, "nfk_made_inverse_bwd_jobs")
    jobs = torch.empty(n, 8, dtype=torch.int32)
    check(0 if LIB.nfk_made_inverse_bwd_jobs(cnt1.data_ptr(), cnt2.data_ptr(), D, H, N3p, jobs.data_ptr(), n) == n
          else -1, "nfk_made_inverse_bwd_jobs")
    return jobs


def made_inverse_bwd_pack(jobs_dev, B1T, B2T, B3T, D, H, N3p, wstream):
    """Transposed weights of every reverse-solve job, packed job after job in shared-memory layout."""
    _count()
    check(LIB.nfk_made_inverse_bwd_pack(_p(jobs_dev), jobs_dev.shape[0], _p(B1T), _p(B2T), _p(B3T), D, H, N3p,
                                        _p(wstream), _st()), "nfk_made_inverse_bwd_pack")


def made_inverse_bwd_resident(g_x, g_ld, out, m1, m2, u_in, wstream, jobs, g_u, dout, db3, B, D, H, N3p, flip,
                              mtiles=0):
    """The whole reverse solve of one MADE layer's inverse in one launch (include/nfk.h)."""
    _count()
    check(LIB.nfk_made_inverse_bwd_resident(_p(g_x), _p(g_ld), _p(out), _p(m1), _p(m2), _p(u_in), _p(wstream),
                                            _p(jobs), jobs.shape[0], _p(g_u), _p(dout), _p(db3), B, D, H, N3p,
                                            int(flip), int(mtiles), _st()), "nfk_made_inverse_bwd_resident")


def cnet_fused_supported(hid, K, M=None) -> bool:
    """Whether the coupling net (or MADE's two masked linears) on M rows of depth K at hidden width `hid` runs as the
    fused conv#1 -> conv#2 kernel rather than two GEMMs: the kernel takes the shape (nfk_cnet_fused_supported) and
    M >= 8192. M=None asks about the shape alone."""
    return (M is None or M >= 8192) and bool(LIB.nfk_cnet_fused_supported(hid, K))


def cnet_fwd_fused(col, K1p, B1, B2, bias1, bias2, h2, M, hid, h1=None, mask1=None, mask2=None, kb2_end_half0=8):
    """conv3x3 -> ReLU -> conv1x1 -> ReLU in one kernel: h1 never leaves the SM (training also stores it + masks).
    kb2_end_half0 < 8: the k-blocks of B2 beyond it are structurally zero for output channels [0, 256) and are skipped
    (MADE's block-triangular hidden mask)."""
    _count()
    ldm = 0 if mask1 is None else mask1.stride(0)
    check(LIB.nfk_cnet_fwd_fused_ranged(_p(col), K1p, _p(B1), _p(B2), _p(bias1), _p(bias2), _p(h1), _p(h2), _p(mask1),
                                        _p(mask2), ldm, M, hid, int(kb2_end_half0), _st()), "nfk_cnet_fwd_fused_ranged")


def _loss_levels(s_list, t_list, ds_list=None):
    from ._lib import NFK_LOSS_MAX_LEVELS, LossLevels
    L = len(s_list)
    if L > NFK_LOSS_MAX_LEVELS:
        raise ValueError(f"at most {NFK_LOSS_MAX_LEVELS} KD levels per launch")
    lv = LossLevels()
    lv.L = L
    for k in range(L):
        lv.s[k], lv.t[k] = _p(s_list[k]), _p(t_list[k])
        lv.ds[k] = None if ds_list is None or ds_list[k] is None else _p(ds_list[k])
        lv.n[k] = s_list[k][0].numel()
    return lv


def kd_nll_loss_fwd(s_list, t_list, z_last, prior_mean, prior_logs, logdet, nll_scale, nll_in, perc, sample_w, w_nll,
                    w_kd, w_perc, B, nll_out, kd_out, means):
    """NFModel.loss in one launch (include/nfk.h: nfk_kd_nll_loss_fwd)."""
    _count()
    lv = _loss_levels(s_list, t_list)
    scratch = torch.empty(LIB.nfk_kd_nll_loss_scratch_floats(B), device=means.device, dtype=torch.float32)
    nz = 0 if z_last is None else z_last[0].numel()
    check(LIB.nfk_kd_nll_loss_fwd(ctypes.addressof(lv), _p(z_last), nz, _p(prior_mean), _p(prior_logs), _p(logdet),
                                  float(nll_scale), _p(nll_in), _p(perc), _p(sample_w), float(w_nll), float(w_kd),
                                  float(w_perc), B, _p(nll_out), _p(kd_out), _p(means), _p(scratch), _st()),
          "nfk_kd_nll_loss_fwd")


def kd_nll_loss_bwd(s_list, t_list, ds_list, z_last, prior_mean, prior_logs, nll_scale, sample_w, w_nll, w_kd, w_perc,
                    B, g_means, g_nll, g_kd, dz_last, dlogdet, dnll_in, dperc):
    _count()
    lv = _loss_levels(s_list, t_list, ds_list)
    nz = 0 if z_last is None else z_last[0].numel()
    check(LIB.nfk_kd_nll_loss_bwd(ctypes.addressof(lv), _p(z_last), nz, _p(prior_mean), _p(prior_logs),
                                  float(nll_scale), _p(sample_w), float(w_nll), float(w_kd), float(w_perc), B,
                                  _p(g_means), _p(g_nll), _p(g_kd), _p(dz_last), _p(dlogdet), _p(dnll_in), _p(dperc),
                                  _st()), "nfk_kd_nll_loss_bwd")


def optim_partials() -> int:
    return int(LIB.nfk_optim_partials())


def grad_sqnorm(g, partials, step=None):
    _count()
    check(LIB.nfk_grad_sqnorm(_p(g), g.numel(), _p(partials), _p(step), _st()), "nfk_grad_sqnorm")


def adam_step(p, g, m, v, partials, step, max_norm, lr, beta1, beta2, eps, weight_decay, adamax, norm_out=None):
    _count()
    check(LIB.nfk_adam_step(_p(p), _p(g), _p(m), _p(v), p.numel(), _p(partials), _p(step), float(max_norm), float(lr),
                            float(beta1), float(beta2), float(eps), float(weight_decay), int(adamax), _p(norm_out),
                            _st()), "nfk_adam_step")


def cnet_bwd_fused(dhcol, K3p, B3T, B2T, mask_h2, mask_h1, dpre2, dpre1, dbias2, dbias1, M, hid):
    """Both dgrads of the coupling net's backward chain in one kernel (include/nfk.h: nfk_cnet_bwd_fused)."""
    _count()
    check(LIB.nfk_cnet_bwd_fused(_p(dhcol), K3p, _p(B3T), _p(B2T), _p(mask_h2), _p(mask_h1), mask_h2.stride(0),
                                 _p(dpre2), _p(dpre1), _p(dbias2), _p(dbias1), M, hid, _st()), "nfk_cnet_bwd_fused")
