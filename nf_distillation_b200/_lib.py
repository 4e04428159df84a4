"""ctypes binding of libnfk.so (see include/nfk.h). There is no fallback: if the library is missing and cannot
be built, importing this module raises."""
from __future__ import annotations

import ctypes
import os

from . import build as _build

_c = ctypes
_vp, _i, _ll, _f = _c.c_void_p, _c.c_int, _c.c_longlong, _c.c_float

ERRORS = {
    -1: "NFK_ERR_SHAPE (unsupported / inconsistent sizes)",
    -2: "NFK_ERR_ALIGN (pointer or leading dimension not 16-byte aligned)",
    -3: "NFK_ERR_ARG (missing / invalid argument)",
    -4: "NFK_ERR_LAUNCH (CUDA launch failure)",
    -5: "NFK_ERR_DRIVER (tensor-map encode failure)",
}



class InvconvItem(_c.Structure):
    """nfk_invconv_item (include/nfk.h)."""
    _fields_ = [(n, _vp) for n in ("an_bias", "an_logs", "lower", "upper", "log_s", "p", "sign_s", "weight")] + \
               [("C", _i), ("reverse", _i), ("transpose", _i)] + \
               [(n, _vp) for n in ("outW", "outb", "out_sl")]


class InvconvBwdItem(_c.Structure):
    """nfk_invconv_bwd_item (include/nfk.h)."""
    _fields_ = [("fwd", InvconvItem), ("dWf", _vp), ("dWf_ld", _i), ("dbf", _vp), ("g_ld", _vp), ("B", _i),
                ("pixels", _f)] + \
               [(n, _vp) for n in ("d_bias", "d_logs", "d_lower", "d_upper", "d_log_s", "d_weight")]


class CouplingItem(_c.Structure):
    """nfk_coupling_item (include/nfk.h)."""
    _fields_ = [(n, _vp) for n in ("w1", "b1", "l1", "w2", "b2", "l2", "w3", "b3", "l3")] + \
               [(n, _i) for n in ("cin", "hid", "cout", "K1p", "K3p", "with_transposed")] + \
               [(n, _vp) for n in ("B1", "B1T", "B2", "B2T", "B3", "B3T", "bias1", "bias2", "bias3")]


class CouplingBwdItem(_c.Structure):
    """nfk_coupling_bwd_item (include/nfk.h)."""
    _fields_ = [("fwd", CouplingItem)] + \
               [(n, _vp) for n in ("dB1", "dbias1", "dB2", "dbias2", "dB3", "dbias3")] + \
               [(n, _vp) for n in ("dw1", "db1", "dl1", "dw2", "db2", "dl2", "dw3", "db3", "dl3")]


NFK_LOSS_MAX_LEVELS = 8


class LossLevels(_c.Structure):
    """nfk_loss_levels (include/nfk.h)."""
    _fields_ = [("s", _vp * NFK_LOSS_MAX_LEVELS), ("t", _vp * NFK_LOSS_MAX_LEVELS), ("ds", _vp * NFK_LOSS_MAX_LEVELS),
                ("n", _i * NFK_LOSS_MAX_LEVELS), ("L", _i)]


# name -> argtypes; every function returns int. Keep in the same order as include/nfk.h.
SIGNATURES: dict[str, list] = {
    "nfk_version": [],
    "nfk_gemm_nt_bf16": [_vp, _ll, _vp, _ll, _i, _i, _i, _i, _vp, _ll, _vp, _vp, _ll, _vp, _vp],
    "nfk_gemm_set_prof": [_vp],
    "nfk_gemm_tn_bf16": [_vp, _ll, _vp, _ll, _i, _i, _i, _vp, _ll, _i, _vp],
    "nfk_invconv_prep_batch": [_i, _vp, _vp],
    "nfk_invconv_prep_bwd_batch": [_i, _vp, _vp],
    "nfk_coupling_prep_batch": [_i, _vp, _vp],
    "nfk_coupling_prep_bwd_batch": [_i, _vp, _vp],
    "nfk_affine1x1_fwd": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _vp],
    "nfk_coupling_fwd": [_vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "nfk_coupling_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp],
    "nfk_affine1x1_bwd": [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "nfk_coupling_inv_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp],
    "nfk_col2im_add": [_vp, _i, _vp, _i, _i, _i, _i, _vp],
    "nfk_split2d_fwd": [_vp] * 6 + [_i] * 4 + [_vp],
    "nfk_split2d_rev": [_vp] * 5 + [_f, _vp] + [_i] * 4 + [_vp],
    "nfk_split2d_bwd": [_vp] * 10 + [_i] * 4 + [_vp],
    "nfk_split2d_squeeze_fwd": [_vp] * 7 + [_i] * 4 + [_vp],
    "nfk_split2d_squeeze_bwd": [_vp] * 11 + [_i] * 4 + [_vp],
    "nfk_dequant_squeeze": [_vp, _i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "nfk_prior_bpd_fwd": [_vp] * 4 + [_i, _i, _f, _vp, _vp],
    "nfk_prior_bpd_bwd": [_vp] * 4 + [_i, _i, _f, _vp, _vp, _vp],
    "nfk_kd_mse_fwd": [_vp, _vp, _i, _i, _f, _vp, _vp],
    "nfk_kd_mse_bwd": [_vp, _vp, _vp, _i, _i, _f, _vp, _i, _vp],
    "nfk_flow1d_supported": [_i, _i, _i, _i],
    "nfk_flow1d_sizes": [_i, _i, _i, _vp, _vp, _vp, _vp, _vp],
    "nfk_flow1d_pack": [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp],
    "nfk_flow1d_fwd": [_vp] * 8 + [_i] * 5 + [_vp],
    "nfk_flow1d_bwd": [_vp] * 9 + [_i] * 5 + [_vp],
    "nfk_affine_rows": [_vp] * 7 + [_i, _i, _f, _vp],
    "nfk_gemm_nt_bf16_ranged": [_vp, _ll, _vp, _ll, _i, _i, _i, _i, _vp, _ll, _vp, _vp, _ll, _vp, _i, _vp, _vp, _vp],
    "nfk_cnet_fused_supported": [_i, _i],
    "nfk_cnet_set_prof": [_vp],
    "nfk_cnet_fwd_fused": [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i, _vp],
    "nfk_cnet_bwd_fused": [_vp, _i, _vp, _vp, _vp, _vp, _ll, _vp, _vp, _vp, _vp, _i, _i, _vp],
    "nfk_cnet_fwd_fused_ranged": [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _i, _i, _vp],
    "nfk_pconv_coupling_supported": [_i, _i, _i, _i],
    "nfk_pconv_coupling_fwd": [_vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "nfk_conv1_dgrad_affine_bwd_supported": [_i, _i, _i, _i],
    "nfk_conv1_dgrad_affine_bwd": [_vp] * 9 + [_i] * 5 + [_vp],
    "nfk_made_prep": [_vp] * 5 + [_i] * 4 + [_vp] * 6 + [_i, _vp],
    "nfk_made_prep_bwd": [_vp] * 5 + [_i] * 3 + [_vp] * 3 + [_vp],
    "nfk_rows_to_bf16": [_vp, _i, _i, _i, _vp, _vp],
    "nfk_made_affine_fwd": [_vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _vp],
    "nfk_made_affine_bwd": [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp],
    "nfk_made_inv_update": [_vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "nfk_made_inverse_resident_supported": [_i, _i, _i],
    "nfk_made_inverse_push_supported": [_i, _i, _i, _i],
    "nfk_made_inverse_jobs": [_vp, _vp, _i, _i, _i, _i, _i, _vp, _i],
    "nfk_made_inverse_pack": [_vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp],
    "nfk_made_inverse_resident": [_vp] * 6 + [_i] * 3 + [_vp] * 3 + [_i] * 6 + [_vp],
    "nfk_made_inv_bwd_update": [_vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "nfk_made_inverse_bwd_supported": [_i, _i, _i],
    "nfk_made_inverse_bwd_jobs": [_vp, _vp, _i, _i, _i, _vp, _i],
    "nfk_made_inverse_bwd_pack": [_vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp],
    "nfk_made_inverse_bwd_resident": [_vp] * 8 + [_i] + [_vp] * 3 + [_i] * 6 + [_vp],
    "nfk_kd_nll_loss_scratch_floats": [_i],
    "nfk_kd_nll_loss_fwd": [_vp, _vp, _i, _vp, _vp, _vp, _f, _vp, _vp, _vp, _f, _f, _f, _i, _vp, _vp, _vp, _vp, _vp],
    "nfk_kd_nll_loss_bwd": [_vp, _vp, _i, _vp, _vp, _f, _vp, _f, _f, _f, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    "nfk_optim_partials": [],
    "nfk_grad_sqnorm": [_vp, _ll, _vp, _vp, _vp],
    "nfk_adam_step": [_vp, _vp, _vp, _vp, _ll, _vp, _vp, _f, _f, _f, _f, _f, _f, _i, _vp, _vp],
    "nfk_split3_rows": [_vp, _ll, _ll, _i, _i, _i, _vp, _vp],
    "nfk_im2col3x3_split3": [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp],
    "nfk_act_split3": [_vp, _ll, _i, _i, _vp, _ll, _i, _vp, _vp, _vp],
    "nfk_coupling_bwd_f32": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "nfk_coupling_inv_bwd_f32": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
}


class NfkError(RuntimeError):
    pass


def _load() -> ctypes.CDLL:
    path = _build.LIB_PATH
    if _build.needs_build():
        try:
            _build.build()
        except Exception as e:  # stale .so + no nvcc on this machine
            if not os.path.exists(path):
                raise ImportError(
                    f"libnfk.so is not built and cannot be built here ({e}); there is no CPU fallback") from e
    lib = ctypes.CDLL(path)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library diverge
        fn.argtypes = argtypes
        fn.restype = _c.c_int
    return lib


LIB = _load()


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise NfkError(f"{what} failed: {ERRORS.get(rc, rc)}")


def ptr(t) -> int | None:
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
