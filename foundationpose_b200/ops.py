"""Thin torch-tensor front end over the single-operator C-ABI hooks (`fp_op_*`).

Used by the parity tests to check each CUDA kernel against the oracle in isolation.  torch is only
the owner of device memory and streams here; all compute happens inside libfpose.so.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import lib


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.FposeError("libfpose operators need CUDA tensors (there is no CPU path)")


def gemm_layer(kind, x, w_packed, bias, *, n_img, Hin, Win, Cin, Cout, out=None, out_ld=None, out_split=0,
               res=None, res_ld=0, post_add=None, relu=False):
    """Run one implicit-GEMM layer.  `x`: fp16 activation tensor in the layout the kind expects."""
    _require_cuda(x, w_packed, bias, res, post_add, out)
    assert x.dtype == torch.float16 and w_packed.dtype == torch.float16 and bias.dtype == torch.float32
    if kind == _lib.LAYER_LINEAR:
        Ho, Wo = 1, Win
    elif kind == _lib.LAYER_CONV3_S1:
        Ho, Wo = Hin, Win
    else:
        Ho, Wo = Hin // 2, Win // 2
    if out is None:
        out_ld = Cout
        out = torch.empty(n_img, Ho, Wo, Cout, dtype=torch.float16, device=x.device)
    L = _lib.GemmLayer(kind, n_img, Hin, Win, Cin, Cout, _ptr(x), _ptr(w_packed), _ptr(bias), _ptr(res),
                       res_ld, _ptr(out), out_ld, out_split, _ptr(post_add), 1 if relu else 0)
    _lib.check(lib.fp_op_gemm_layer(C.byref(L), _stream()), "fp_op_gemm_layer")
    return out


lib.fp_op_attention.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
lib.fp_op_attention.restype = C.c_int


def attention(qkv, impl=1):
    """qkv fp16 [B*400, 1536] -> fp16 [B*400, 512]; impl 1 = tcgen05, 0 = mma.sync."""
    _require_cuda(qkv)
    assert qkv.dtype == torch.float16 and qkv.shape[1] == 1536 and qkv.shape[0] % 400 == 0
    B = qkv.shape[0] // 400
    out = torch.empty(qkv.shape[0], 512, dtype=torch.float16, device=qkv.device)
    _lib.check(lib.fp_op_attention(_ptr(qkv), _ptr(out), B, impl, _stream()), "fp_op_attention")
    return out


lib.fp_op_attention_grouped.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
lib.fp_op_attention_grouped.restype = C.c_int


def attention_grouped(qkv, n_groups):
    """The product's attention launch: n_groups = 1 (scorer) qkv fp16 [B*400, 1536] -> [B*400, 512];
    n_groups = 2 (refiner, both heads) qkv fp16 [B*400, 3072] -> [2, B*400, 512]."""
    _require_cuda(qkv)
    assert n_groups in (1, 2)
    assert qkv.dtype == torch.float16 and qkv.shape[1] == 1536 * n_groups and qkv.shape[0] % 400 == 0
    assert qkv.is_contiguous()
    B = qkv.shape[0] // 400
    out = torch.empty(n_groups, qkv.shape[0], 512, dtype=torch.float16, device=qkv.device)
    _lib.check(lib.fp_op_attention_grouped(_ptr(qkv), _ptr(out), B, n_groups, _stream()), "fp_op_attention_grouped")
    return out if n_groups == 2 else out[0]


GEMM_PLAN_FIELDS = ("kernel", "bn", "cg", "slabs", "patch", "grid", "work_tiles", "bw", "bh", "bimg", "m_tiles",
                    "n_tiles")
GEMM_KERNELS = ("tile", "swap", "swap_patch", "stem")
lib.fp_op_gemm_last_plan.argtypes = [C.POINTER(C.c_int), C.c_int]
lib.fp_op_gemm_last_plan.restype = C.c_int


def gemm_last_plan():
    """What the last GEMM launch on this thread chose (include/fpose.h fp_op_gemm_last_plan), as a dict; `kernel` is
    one of GEMM_KERNELS."""
    buf = (C.c_int * len(GEMM_PLAN_FIELDS))()
    _lib.check(lib.fp_op_gemm_last_plan(buf, len(GEMM_PLAN_FIELDS)), "fp_op_gemm_last_plan")
    plan = dict(zip(GEMM_PLAN_FIELDS, list(buf)))
    plan["kernel"] = GEMM_KERNELS[plan["kernel"]]
    return plan
