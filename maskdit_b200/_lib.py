"""ctypes binding of `libmaskdit_b200.so` (the C ABI declared in include/maskdit_b200.h).

There is NO fallback: if the CUDA library is missing or a kernel returns a non-zero status this module raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int64, c_longlong, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# MDT_LIB_PATH: development A/B of two builds inside one GPU session (default: the in-tree library)
LIB_PATH = os.environ.get("MDT_LIB_PATH") or os.path.join(_HERE, "libmaskdit_b200.so")


class MdtError(RuntimeError):
    pass


class GemmArgs(Structure):
    _fields_ = [
        ("A", c_void_p), ("B", c_void_p),
        ("M", c_int), ("N", c_int), ("K", c_int),
        ("lda", c_int), ("ldb", c_int),
        ("a_mn", c_int), ("b_mn", c_int),
        ("epi", c_int), ("act", c_int),
        ("out", c_void_p), ("ldo", c_int), ("out_fp32", c_int),
        ("bias", c_void_p),
        ("aux", c_void_p), ("ld_aux", c_int),
        ("resid", c_void_p), ("ld_resid", c_int),
        ("gate", c_void_p), ("ld_gate", c_int),
        ("rows_per_group", c_int),
        ("block_n", c_int),
        ("colsum", c_void_p),
    ]


class ModelCfg(Structure):
    """mdt_model_cfg (include/maskdit_b200.h)."""
    _fields_ = [
        ("img_resolution", c_int), ("img_channels", c_int), ("patch_size", c_int), ("num_classes", c_int),
        ("hidden", c_int), ("depth", c_int), ("heads", c_int), ("mlp_hidden", c_int),
        ("dec_hidden", c_int), ("dec_depth", c_int), ("dec_heads", c_int), ("dec_mlp_hidden", c_int),
        ("has_mask_token", c_int), ("sigma_data", c_float),
    ]


GRAD_READY_FN = ctypes.CFUNCTYPE(None, c_void_p, c_longlong, c_longlong)

EPI_STORE, EPI_GELU, EPI_GATE_RESID, EPI_DGELU, EPI_ATOMIC = range(5)
ACT_NONE, ACT_SILU = 0, 1

_lib = None

# name -> argtypes  (every function returns int status; last arg is the stream)
_P, _I, _F, _LL, _D = c_void_p, c_int, c_float, c_longlong, c_double
_SIGS = {
    "mdt_gemm_bf16": [POINTER(GemmArgs), _P],
    "mdt_gemm_plan": [POINTER(GemmArgs), _P],
    "mdt_gemm_profile_enable": [_I],
    "mdt_gemm_profile_read": [_P, _P, _I],
    "mdt_mask_indices": [_P, _I, _I, _I, _P, _P, _P, _P],
    "mdt_patch_embed": [_P, _P, _F, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "mdt_patch_embed_bwd": [_P, _P, _F, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "mdt_timestep_freq": [_P, _I, _I, _P, _P],
    "mdt_silu": [_P, _P, _P, _P, _LL, _P],
    "mdt_silu_bwd": [_P, _P, _P, _P, _LL, _P],
    "mdt_cast_f32_bf16": [_P, _P, _LL, _P],
    "mdt_colsum_bf16": [_P, _I, _I, _I, _P, _P],
    "mdt_colsum_f32": [_P, _I, _I, _I, _P, _P],
    "mdt_ln_modulate": [_P, _P, _P, _I, _I, _P, _P, _P, _I, _I, _F, _P],
    "mdt_ln_modulate_bwd": [_P, _P, _P, _P, _P, _I, _I, _P, _I, _P, _P, _I, _I, _I, _P],
    "mdt_gate_bwd": [_P, _P, _P, _I, _I, _P, _P, _I, _P, _I, _I, _P],
    "mdt_ln_modulate_bwd_gate": [_P, _P, _P, _P, _P, _I, _I, _P, _I, _P, _P, _I, _P, _P, _I, _P, _P, _I, _P, _I, _I, _P],
    "mdt_attention_fwd": [_P, _P, _P, _I, _I, _I, _I, _P],
    "mdt_attention_bwd": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "mdt_attention_last_impl": [_I],
    "mdt_attention_impl_log": [_P, _I],
    "mdt_gemm_configs_seen": [_I],
    "mdt_gemm_last_config": [],
    "mdt_unmask_tokens": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "mdt_unmask_tokens_bwd": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "mdt_edm_loss": [_P, _P, _P, _P, _P, _P, _F, _F, _P, _P, _P, _I, _I, _I, _I, _P],
    "mdt_step_front": [_P, _P, _P, _P, _P, _F, _F, _F, _F, _P, _P, _P, _P, _I, _I, _I, _I, _P],
    "mdt_edm_precond_out": [_P, _P, _P, _F, _P, _I, _I, _I, _I, _P],
    "mdt_edm_precond_out_bwd": [_P, _P, _F, _P, _I, _I, _I, _I, _P],
    "mdt_cfg_precond_out": [_P, _P, _P, _F, _F, _P, _I, _I, _I, _I, _P],
    "mdt_heun_update": [_I, _P, _P, _P, _P, _P, _D, _D, _LL, _P],
    "mdt_lincomb_f64": [_D, _P, _D, _P, _D, _P, _P, _P, _D, _LL, _P],
    "mdt_to_uint8_nhwc": [_P, _P, _I, _I, _I, _I, _P],
    # step driver (csrc/driver.cu)
    "mdt_model_create": [POINTER(ModelCfg), POINTER(c_void_p)],
    "mdt_model_num_tensors": [_P],
    "mdt_model_param_info": [_P, _I, c_char_p, _I, POINTER(c_longlong), POINTER(c_longlong)],
    "mdt_model_mod_width": [_P],
    "mdt_forward": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P, _LL, _P, _P],
    "mdt_backward": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _P, _LL, GRAD_READY_FN, _P, _P],
    "mdt_nccl_unique_id": [_P],
    "mdt_nccl_comm_create": [_P, _I, _I, _I, POINTER(c_void_p)],
    "mdt_nccl_comm_destroy": [_P],
    "mdt_allreduce_grads": [_P, _P, _LL, _I, _P],
    "mdt_vae_post_quant": [_P, _P, _P, _F, _P, _I, _I, _I, _P],
    "mdt_vae_gn_stats": [_P, _P, _P, _I, _I, _I, _P],
    "mdt_vae_im2col": [_P, _P, _P, _P, _I, _I, _I, _P, _I, _I, _I, _I, _I, _P],
    "mdt_vae_softmax_rows": [_P, _F, _P, _I, _I, _P],
    "mdt_vae_softmax_rows_ld": [_P, _F, _P, _I, _I, _I, _P],
    "mdt_vae_im2col_down": [_P, _P, _I, _I, _I, _I, _I, _P],
    "mdt_vae_image_to_rows": [_P, _P, _I, _I, _I, _I, _P],
    "mdt_vae_quant_out": [_P, _I, _P, _P, _P, _I, _I, _I, _P],
    "mdt_vae_rows_to_nchw": [_P, _P, _I, _I, _I, _I, _P],
    "mdt_adamw_ema_g16": [_P, _P, _P, _P, _P, _P, _LL, _F, _F, _F, _F, _F, _I, _F, _F, _I, _P],
    "mdt_set_sm_budget": [_I],
    "mdt_get_sm_budget": [],
    "mdt_adamw_ema": [_P, _P, _P, _P, _P, _P, _LL, _F, _F, _F, _F, _F, _I, _F, _F, _I, _P],
}


def lib():
    """Load the CUDA library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MdtError(
                f"{LIB_PATH} not found: build it with `python -m maskdit_b200.build` "
                "(there is no CPU / PyTorch fallback for the MaskDiT hot path)")
        L = ctypes.CDLL(LIB_PATH)
        L.mdt_status_string.restype = c_char_p
        L.mdt_status_string.argtypes = [c_int]
        L.mdt_abi_version.restype = c_int
        L.mdt_model_destroy.restype = None
        L.mdt_model_destroy.argtypes = [c_void_p]
        L.mdt_model_param_count.restype = c_longlong
        L.mdt_model_param_count.argtypes = [c_void_p, c_int]
        L.mdt_workspace_bytes.restype = c_longlong
        L.mdt_workspace_bytes.argtypes = [c_void_p, c_int, c_int, c_int]
        for name, sig in _SIGS.items():
            if not hasattr(L, name) and os.environ.get("MDT_ALLOW_PARTIAL_LIB") == "1":
                continue  # development only: probing a partially built library
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol -> loud
            fn.restype = c_int
            fn.argtypes = sig
        _lib = L
    return _lib


def exported_symbols():
    return ["mdt_status_string", "mdt_abi_version", "mdt_model_destroy", "mdt_model_param_count",
            "mdt_workspace_bytes", *_SIGS.keys()]


LAUNCHES = 0  # kernels launched through the C ABI (bench.py reports it as gpu_launches)
GEMM_PROFILE = None  # when a list: gemm() appends (flops, start_event, end_event, shape key) per launch (bench.py roofline)


def check(status: int, what: str, n_kernels: int = 1):
    global LAUNCHES
    LAUNCHES += n_kernels
    if status != 0:
        msg = lib().mdt_status_string(status).decode()
        raise MdtError(f"{what} failed: {msg} (status {status})")


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    return 0 if t is None else t.data_ptr()


def _req_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise MdtError("maskdit_b200 kernels need CUDA tensors (no CPU fallback)")


PLAN_FIELDS = ("block_n", "cg", "splits", "pair_halves", "narrow_last", "num_m_tiles", "num_n_tiles", "num_kb", "units",
               "grid")


def gemm_plan(M, N, K, *, a_mn=False, b_mn=False, epi=EPI_STORE, block_n=0):
    """The host-side decisions `mdt_gemm_bf16` takes for this problem (tile width, SM pairs, k-slices, unit order,
    grid), without a launch or a device: `mdt_gemm_plan`.  Operand pointers are dummies (checked for alignment only)."""
    a = GemmArgs()
    a.A = a.B = a.out = a.aux = a.resid = a.gate = 4096
    a.M, a.N, a.K = M, N, K
    a.lda, a.ldb, a.ldo = (M if a_mn else K), (N if b_mn else K), N
    a.a_mn, a.b_mn, a.epi, a.act = int(a_mn), int(b_mn), epi, ACT_NONE
    a.out_fp32 = int(epi in (EPI_ATOMIC, EPI_GATE_RESID))
    a.ld_aux = a.ld_resid = a.ld_gate = N
    a.rows_per_group, a.block_n = 1, block_n
    out = (c_longlong * 10)()
    st = lib().mdt_gemm_plan(ctypes.byref(a), out)
    if st != 0:
        raise MdtError(f"mdt_gemm_plan failed: {lib().mdt_status_string(st).decode()} (status {st})")
    return dict(zip(PLAN_FIELDS, (int(v) for v in out)))


def gemm(A, B, M, N, K, *, lda=None, ldb=None, a_mn=False, b_mn=False, epi=EPI_STORE, act=ACT_NONE, out=None,
         ldo=None, bias=None, aux=None, ld_aux=0, resid=None, ld_resid=0, gate=None, ld_gate=0, rows_per_group=1,
         block_n=0, colsum=None):
    """out[M,N] (+)= sum_k A[m,k] B[n,k].  `out` dtype (bf16/fp32) selects the store type."""
    _req_cuda(A, B, out)
    assert A.dtype == torch.bfloat16 and B.dtype == torch.bfloat16
    assert out is not None and out.dtype in (torch.bfloat16, torch.float32)
    a = GemmArgs()
    a.A, a.B = A.data_ptr(), B.data_ptr()
    a.M, a.N, a.K = M, N, K
    a.lda = lda if lda is not None else (M if a_mn else K)
    a.ldb = ldb if ldb is not None else (N if b_mn else K)
    a.a_mn, a.b_mn = int(a_mn), int(b_mn)
    a.epi, a.act = epi, act
    a.out, a.ldo, a.out_fp32 = out.data_ptr(), (ldo if ldo is not None else N), int(out.dtype == torch.float32)
    a.bias = ptr(bias)
    a.aux, a.ld_aux = ptr(aux), ld_aux
    a.resid, a.ld_resid = ptr(resid), ld_resid
    a.gate, a.ld_gate = ptr(gate), ld_gate
    a.rows_per_group = rows_per_group
    a.block_n = block_n
    a.colsum = ptr(colsum)
    if GEMM_PROFILE is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(lib().mdt_gemm_bf16(ctypes.byref(a), stream_ptr()), "mdt_gemm_bf16")
        e1.record()
        GEMM_PROFILE.append((2.0 * M * N * K, e0, e1, (M, N, K, int(a_mn), int(b_mn), epi, a.out_fp32)))
        return out
    check(lib().mdt_gemm_bf16(ctypes.byref(a), stream_ptr()), "mdt_gemm_bf16")
    return out
