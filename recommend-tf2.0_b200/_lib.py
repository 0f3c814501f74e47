"""ctypes binding of librtf_b200.so (the C-ABI declared in include/rtf_b200.h).

There is no CPU fallback and no alternative backend: if the shared library is
missing, or a kernel is requested without a CUDA device, this module raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librtf_b200.so")
CSRC_DIR = os.path.join(_HERE, "csrc")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "rtf_b200.h")

POOL_NONE, POOL_SUM, POOL_MEAN = 0, 1, 2
OPT_NONE, OPT_SGD, OPT_ADAGRAD, OPT_ADAM = 0, 1, 2, 3
SEG_CHUNK = 64
MAX_FIELDS = 64


class RtfError(RuntimeError):
    pass


class rtf_opt(C.Structure):
    _fields_ = [("kind", C.c_int32), ("lr", C.c_float), ("beta1", C.c_float),
                ("beta2", C.c_float), ("eps", C.c_float), ("l2", C.c_float),
                ("lr_dev", C.c_void_p)]


_p = C.c_void_p
_i64 = C.c_int64
_int = C.c_int

# name -> argtypes; every symbol include/rtf_b200.h declares must be listed here
SIGNATURES = {
    "rtf_version": [C.POINTER(C.c_int)],
    "rtf_embed_fwd": [_p, _p, _p, _int, _p, _int, _i64, _int, _i64, _i64, _i64, _int, _p, _i64,
                      _p, _p],
    "rtf_embed_bwd_workspace": [_i64, _int, C.POINTER(C.c_size_t)],
    "rtf_embed_bwd": [_p, _p, _p, _p, _p, _int, _p, _int, _p, _int, _i64, _int, _i64, _i64,
                      _i64, _int, _p, _i64, C.POINTER(rtf_opt), _p, _p, _p,
                      C.POINTER(C.c_int), _p, C.c_size_t, _p],
    "rtf_embed_bwd_prepare": [_p, _p, _int, _p, _int, _p, _int, _i64, _int, _i64, _i64, _i64, _p,
                              C.POINTER(C.c_int), _p, C.c_size_t, _p],
    "rtf_embed_bwd_apply": [_p, _p, _p, _p, _p, _int, _p, _int, _i64, _int, _int, _p, _i64,
                            C.POINTER(rtf_opt), _p, _p, _p, C.c_size_t, _p],
    "rtf_dot_interact_fwd": [_p, _i64, _int, _int, _p, _i64, _int, _p],
    "rtf_dot_interact_bwd": [_p, _p, _i64, _i64, _int, _int, _p, _p],
    "rtf_dot_rows_fwd": [_p, _p, _int, _int, _i64, _p, _i64, _int, _p, _i64, _p],
    "rtf_dot_rows_bwd": [_p, _p, _int, _int, _i64, _p, _i64, _p, _p, _p],
    "rtf_embed_dot_fwd": [_p, _p, _int, _int, _p, _int, _i64, _i64, _i64, _p, _i64, _p, _i64,
                          _int, _p, _p],
    "rtf_embed_dot_bwd": [_p, _p, _int, _int, _p, _int, _i64, _i64, _i64, _p, _i64, _p, _i64,
                          _p, _i64, _p, _i64, _p],
    "rtf_embed_dot_peer_fwd": [_p, _p, _i64, _int, C.c_uint64, _p, _int, _int, _p, _int, _i64, _i64, _i64, _p,
                               _i64, _p, _i64, _int, _p, _i64, _p, _p],
    "rtf_embed_dot_peer_bwd": [_p, _i64, _p, _int, _int, _p, _int, _i64, _i64, _i64, _p, _i64, _p,
                               _i64, _p, _i64, _p, _p, _int, C.c_uint64, _i64, _p],
    "rtf_colsum_workspace": [_i64, _int, C.POINTER(C.c_size_t)],
    "rtf_colsum": [_p, _i64, _p, _i64, _int, _p, _p, _p],
    "rtf_bn_workspace": [_i64, _int, C.POINTER(C.c_size_t)],
    "rtf_bn_fwd": [_p, _i64, _i64, _int, _p, _p, C.c_float, C.c_float, _p, _i64, _p, _p, _p, _p, _p,
                   C.c_size_t, _p],
    "rtf_bn_bwd": [_p, _i64, _p, _i64, _i64, _int, _p, _p, _p, _p, _i64, _p, _p, _p, C.c_size_t, _p],
    "rtf_layernorm_workspace": [_i64, _int, C.POINTER(C.c_size_t)],
    "rtf_layernorm_fwd": [_p, _i64, _int, _p, _p, C.c_float, _p, _p, _p, _p],
    "rtf_layernorm_bwd": [_p, _p, _p, _p, _p, _i64, _int, _p, _p, _p, _p, C.c_size_t, _p],
    "rtf_bce_workspace": [_i64, C.POINTER(C.c_size_t)],
    "rtf_bce_fwd": [_p, _p, _i64, _p, _p, _p, _p],
    "rtf_auc_update": [_p, _p, _i64, _int, _p, _p, _p],
    "rtf_auc_result": [_p, _int, _p, _p],
    "rtf_relu_bwd_colsum_workspace": [_i64, _int, C.POINTER(C.c_size_t)],
    "rtf_relu_bwd_colsum": [_p, _p, _i64, _int, _p, _p, _p, _p],
    "rtf_autoint_layer_supported": [_int, _int, _int, _int],
    "rtf_autoint_layer_workspace": [_i64, _int, _int, C.POINTER(C.c_size_t)],
    "rtf_autoint_layer_fwd": [_p, _i64, _int, _int, _p, _p, _p, _p, _int, _int, _int, C.c_float, _p, _p],
    "rtf_autoint_layer_bwd": [_p, _i64, _int, _int, _p, _p, _p, _p, _int, _int, _int, C.c_float, _p, _p,
                              _p, _p, _p, C.c_size_t, _p],
    "rtf_sasrec_score_fwd": [_p, _i64, _p, _i64, _p, _i64, _p, _p, _int, _i64, _i64, _int, _int, _p, _p, _p, _p],
    "rtf_sasrec_score_bwd": [_p, _i64, _p, _i64, _p, _i64, _p, _p, _int, _i64, _i64, _int, _int, _p, _p, _p,
                             _p, _p, _p],
    "rtf_topk_ip_workspace": [_i64, _i64, _int, _int, C.POINTER(C.c_size_t)],
    "rtf_topk_ip": [_p, _i64, _i64, _p, _i64, _i64, _int, _int, _p, _p, _p, _p, C.c_size_t, _p],
    "rtf_peer_pull_rows": [_p, _p, _i64, _int, C.c_uint64, _p, _int, _int, _p, _int, _i64, _i64, _i64, _p,
                           _i64, _p, _p],
    "rtf_ssm_gather": [_p, _p, _p, _p, _i64, _int, _int, _p, _p, _p, _p],
    "rtf_ssm_logits_fwd": [_p, _i64, _p, _i64, _p, _p, _p, _p, _p, _p, _i64, _i64, _int, _int, _int, _p, _p,
                           _p, _p],
    "rtf_ssm_logits_bwd": [_p, _i64, _p, _i64, _p, _p, _p, _p, _p, _p, _i64, _i64, _int, _int, _int, _p, _p,
                           _p, _p, _i64, _p],
    "rtf_ssm_true_gx": [_p, _p, _p, _i64, _i64, _int, _p, _i64, _p],
    "rtf_dense_adam": [_p, _p, _p, _p, _i64, C.POINTER(rtf_opt), _p],
    "rtf_rows_apply_dense": [_p, _p, _p, _p, _p, _i64, _int, C.POINTER(rtf_opt), _p],
    "rtf_dense_gemm_nn_workspace": [_int, _int, _int, _int, C.POINTER(C.c_size_t)],
    "rtf_dense_gemm_nt_workspace": [_int, _int, _int, _int, C.POINTER(C.c_size_t)],
    "rtf_dense_gemm_tn_workspace": [_int, _int, _int, _int, C.POINTER(C.c_size_t)],
    "rtf_dense_gemm_nn": [_p, _i64, _i64, _p, _i64, _i64, _p, _int, _p, _i64, _i64, _int, _int, _int,
                          _int, _p, C.c_size_t, _p],
    "rtf_dense_gemm_nt": [_p, _i64, _i64, _p, _i64, _i64, _p, _int, _p, _i64, _i64, _int, _int, _int,
                          _int, _p, C.c_size_t, _p],
    "rtf_dense_gemm_tn": [_p, _i64, _i64, _p, _i64, _i64, _p, _int, _p, _i64, _i64, _int, _int, _int,
                          _int, _p, C.c_size_t, _p],
    "rtf_split_bf16x3": [_p, _i64, _int, _i64, _p, _i64, _i64, _p],
    "rtf_dense_gemm_nn_planes_workspace": [_int, _int, _int, _int, C.POINTER(C.c_size_t)],
    "rtf_dense_gemm_nt_planes_workspace": [_int, _int, _int, _int, C.POINTER(C.c_size_t)],
    "rtf_dense_gemm_tn_planes_workspace": [_int, _int, _int, _int, C.POINTER(C.c_size_t)],
    "rtf_dense_gemm_nn_planes": [_p, _i64, _i64, _i64, _p, _i64, _i64, _i64, _p, _int, _p, _i64, _i64,
                                 _int, _int, _int, _int, _p, C.c_size_t, _p],
    "rtf_dense_gemm_nt_planes": [_p, _i64, _i64, _i64, _p, _i64, _i64, _i64, _p, _int, _p, _i64, _i64,
                                 _int, _int, _int, _int, _p, C.c_size_t, _p],
    "rtf_dense_gemm_tn_planes": [_p, _i64, _i64, _i64, _p, _i64, _i64, _i64, _p, _int, _p, _i64, _i64,
                                 _int, _int, _int, _int, _p, C.c_size_t, _p],
    "rtf_fm_layer_workspace": [_i64, _int, C.POINTER(C.c_size_t)],
    "rtf_fm_layer_fwd": [_p, _i64, _p, _int, _p, _i64, _int, _int, _i64, _int, _int, _p, _p, _p],
    "rtf_fm_layer_bwd": [_p, _i64, _p, _int, _p, _i64, _int, _int, _i64, _int, _int, _p, _p,
                         _i64, _p, _p, _i64, _p, _p],
    "rtf_fm_gather_fwd": [_p, _p, _int, _int, _int, _p, _int, _p, _i64, _p, _int, _i64, _i64,
                          _i64, _p, _p, _p, _p, _p],
    "rtf_fm_gather_bwd": [_p, _p, _int, _int, _int, _p, _int, _p, _i64, _p, _int, _i64, _i64,
                          _i64, _p, _p, _p, _p, _p, _p, _p],
    "rtf_attn_fwd": [_p, _i64, _i64, _p, _i64, _i64, _p, _i64, _i64, _p, _i64, _p, _i64, _int,
                     _int, _int, _int, _int, _int, C.c_float, _p, _i64, _i64, _p, _p, _p],
    "rtf_attn_bwd": [_p, _i64, _i64, _p, _i64, _i64, _p, _i64, _i64, _p, _i64, _p, _i64, _int,
                     _int, _int, _int, _int, _int, C.c_float, _p, _i64, _i64, _p, _p, _p, _i64,
                     _i64, _p, _p, _i64, _i64, _p, _i64, _i64, _p, _i64, _i64, _p],
    "rtf_din_attn_fwd": [_p, _i64, _p, _i64, _p, _i64, _p, _i64, _p, _p, _int, _i64, _int, _int,
                         _p, _i64, _p],
    "rtf_din_attn_bwd": [_p, _i64, _p, _i64, _p, _i64, _p, _i64, _p, _p, _int, _i64, _int, _int,
                         _p, _i64, _p, _i64, _p, _i64, _p, _i64, _p, _p],
    "rtf_log_uniform_workspace": [_int, C.POINTER(C.c_size_t)],
    "rtf_log_uniform_sample": [C.c_uint64, _int, _i64, _p, _p, _p, _p],
    "rtf_log_uniform_sample_dseed": [_p, _int, _i64, _p, _p, _p, _p],
    "rtf_log_uniform_expected": [_p, _i64, _i64, _p, _p, _p],
    "rtf_sampled_softmax_workspace": [_int, _int, C.POINTER(C.c_size_t)],
    "rtf_sampled_softmax_fwd": [_p, _i64, _p, _p, _p, _p, _p, _p, _i64, _i64, _int, _int, _int,
                                _p, _p, _p, _p, _p],
    "rtf_sampled_softmax_bwd": [_p, _i64, _p, _p, _p, _p, _p, _p, _i64, _i64, _int, _int, _int,
                                _p, _p, _p, _i64, _p, _p, _p],
}

_lib = None


def build(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into librtf_b200.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC_DIR, "-j", str(min(8, os.cpu_count() or 1))]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout)
    if res.returncode != 0:
        raise RtfError("building librtf_b200.so failed (see make output above)")
    return LIB_PATH


def lib() -> C.CDLL:
    """Load the library once; raises (never falls back) when it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RtfError(
                f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or make -C recommend-tf2.0_b200/csrc). There is no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is missing
            fn.argtypes = argtypes
            fn.restype = C.c_int
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    if rc < 0:
        names = {-1: "RTF_E_ARG", -2: "RTF_E_ALIGN", -3: "RTF_E_RANGE", -4: "RTF_E_WORKSPACE"}
        raise RtfError(f"{what}: {names.get(rc, rc)}")
    raise RtfError(f"{what}: cudaError_t {rc}")


def require_cuda(t, what: str):
    if not t.is_cuda:
        raise RtfError(f"{what}: tensor is on {t.device}; the recommend-tf2.0_b200 kernels run "
                       "on CUDA (sm_100a) only and have no CPU fallback")


def current_stream_ptr() -> int:
    """Raw cudaStream_t of torch's current stream (the C call, not the Stream object: this runs
    ~60 times per training step and the host must stay ahead of the GPU)."""
    import torch
    try:
        return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())
    except AttributeError:      # private API moved: the public, slower route
        return torch.cuda.current_stream().cuda_stream


def host_array(ctype, values):
    arr = (ctype * len(values))(*values)
    return arr
