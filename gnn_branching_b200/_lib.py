"""ctypes binding of libgnnb.so (include/gnnb.h).  No CPU fallback: a missing library is a hard error."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('GNNB_LIB') or os.path.join(_HERE, 'libgnnb.so')   # GNNB_LIB: debug builds (phase tracing)

GNNB_OK, GNNB_ERR_INVALID, GNNB_ERR_CUDA, GNNB_ERR_STATE, GNNB_ERR_NAN, GNNB_ERR_UNSUPPORTED = range(6)
LAYER_CONV, LAYER_LINEAR = 0, 1
MEM_DEVICE, MEM_HOST = 0, 1
MATH_TC_FP16X3, MATH_SIMT_FP32 = 0, 1
TOPK_MAX = 64                                      # GNNB_TOPK_MAX
KERNEL_CLASSES = ['relax', 'update_fwd', 'update_bwd', 'update_bwd_score', 'input_embed', 'input_update', 'prop_fwd',
                  'prop_bwd', 'output', 'argmax', 'layer_fwd', 'layer_bwd', 'layer_bwd_score']

EXPORTS = ['gnnb_create', 'gnnb_destroy', 'gnnb_set_gnn_weights', 'gnnb_set_network', 'gnnb_set_option',
           'gnnb_get_option', 'gnnb_score', 'gnnb_score_winners', 'gnnb_score_topk', 'gnnb_topk', 'gnnb_check', 'gnnb_launch_count', 'gnnb_last_error',
           'gnnb_debug_snapshot', 'gnnb_abi_version', 'gnnb_profile_read', 'gnnb_profile_reset', 'gnnb_babsr',
           'gnnb_score_grad', 'gnnb_get_gradients', 'gnnb_get_gnn_weights', 'gnnb_adam_step', 'gnnb_adam_reset',
           'gnnb_kw_bounds', 'gnnb_child_bounds', 'gnnb_root_bounds', 'gnnb_queue_create', 'gnnb_queue_destroy', 'gnnb_queue_add', 'gnnb_queue_pick', 'gnnb_queue_prune', 'gnnb_queue_stats']

_fp = C.POINTER(C.c_float)
_fpp = C.POINTER(_fp)


class LayerDesc(C.Structure):
    _fields_ = [('kind', C.c_int32), ('c_in', C.c_int32), ('h_in', C.c_int32), ('w_in', C.c_int32),
                ('c_out', C.c_int32), ('h_out', C.c_int32), ('w_out', C.c_int32),
                ('ksize', C.c_int32), ('stride', C.c_int32), ('pad', C.c_int32),
                ('weight', _fp), ('bias', _fp)]


class FrontierDesc(C.Structure):
    _fields_ = [('B', C.c_int32), ('mem', C.c_int32),
                ('lb', _fpp), ('ub', _fpp), ('dual', _fpp), ('prim_pre', _fpp), ('prim_post', _fpp),
                ('prim_out', _fp), ('primal_input', _fp), ('wp', _fp), ('bp', _fp), ('mask', _fp)]


class DomainsDesc(C.Structure):
    _fields_ = [('B', C.c_int32), ('mem', C.c_int32), ('lower_bound', _fp), ('upper_bound', _fp), ('lb', _fpp), ('ub', _fpp),
                ('mask', C.POINTER(C.c_int8)), ('decision', C.POINTER(C.c_int32))]


class GnnbError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f'libgnnb status {status}: {message}')
        self.status = status


_lib = None


def load() -> C.CDLL:
    """Load libgnnb.so from the package directory (built by ``__graft_entry__.build()``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                          '(there is no CPU or PyTorch fallback for the scoring path)')
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.gnnb_abi_version.restype = C.c_int
    lib.gnnb_create.argtypes = [C.POINTER(vp), C.c_int]
    lib.gnnb_destroy.argtypes = [vp]
    lib.gnnb_destroy.restype = None
    lib.gnnb_set_gnn_weights.argtypes = [vp, _fpp, C.POINTER(C.c_int64), C.c_int, C.c_int, C.c_int]
    lib.gnnb_set_network.argtypes = [vp, C.POINTER(LayerDesc), C.c_int, C.c_int, C.c_int, C.c_int]
    lib.gnnb_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
    lib.gnnb_get_option.argtypes = [vp, C.c_char_p]
    lib.gnnb_get_option.restype = C.c_int64
    lib.gnnb_score.argtypes = [vp, C.POINTER(FrontierDesc), _fp, C.POINTER(C.c_int32), _fp, vp]
    lib.gnnb_score_winners.argtypes = [vp, C.POINTER(FrontierDesc), vp, _fp, vp]
    _ip = C.POINTER(C.c_int32)
    lib.gnnb_score_topk.argtypes = [vp, C.POINTER(FrontierDesc), C.c_int32, _fp, _ip, _fp, vp]
    lib.gnnb_topk.argtypes = [vp, C.c_int32, C.c_int32, _fp, _fp, C.c_int32, _fp, _ip, vp]
    lib.gnnb_babsr.argtypes = [vp, C.POINTER(FrontierDesc), C.c_int32, C.c_float, _ip, _ip, _ip, _ip, _ip, _fp, vp]
    lib.gnnb_score_grad.argtypes = [vp, C.POINTER(FrontierDesc), C.c_int32, _ip, _ip, _fp, _fp, vp]
    lib.gnnb_get_gradients.argtypes = [vp, _fpp, C.POINTER(C.c_int64), C.c_int]
    lib.gnnb_get_gnn_weights.argtypes = [vp, _fpp, C.POINTER(C.c_int64), C.c_int]
    lib.gnnb_adam_step.argtypes = [vp, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, vp]
    lib.gnnb_adam_reset.argtypes = [vp]
    lib.gnnb_kw_bounds.argtypes = [vp, C.c_int32, _fp, C.c_float, _fp, _fp, _fpp, _fpp, _fpp, _fpp, vp]
    lib.gnnb_child_bounds.argtypes = [vp, C.c_int32, _fp, C.c_float, _fp, _fp, _fpp, _fpp, _ip, _ip, _ip, _fpp, _fpp,
                                      C.POINTER(C.POINTER(C.c_int8)), _ip, vp]
    lib.gnnb_root_bounds.argtypes = [vp, C.c_int32, _fp, C.c_float, _fp, _fp, _fpp, _fpp, C.POINTER(C.POINTER(C.c_int8)), _ip, vp]
    lib.gnnb_queue_create.argtypes = [vp, C.c_int64, C.POINTER(vp)]
    lib.gnnb_queue_destroy.argtypes = [vp]
    lib.gnnb_queue_destroy.restype = None
    lib.gnnb_queue_add.argtypes = [vp, C.POINTER(DomainsDesc), C.POINTER(C.c_uint8), _ip, vp]
    lib.gnnb_queue_pick.argtypes = [vp, C.c_float, C.c_int32, C.POINTER(DomainsDesc), _ip, vp]
    lib.gnnb_queue_prune.argtypes = [vp, C.c_float, vp]
    lib.gnnb_queue_stats.argtypes = [vp, C.POINTER(C.c_int64), _fp, vp]
    lib.gnnb_check.argtypes = [vp, vp, C.POINTER(C.c_int64)]
    lib.gnnb_launch_count.argtypes = [vp]
    lib.gnnb_launch_count.restype = C.c_int64
    lib.gnnb_last_error.argtypes = [vp, C.c_char_p, C.c_int]
    lib.gnnb_debug_snapshot.argtypes = [vp, C.c_char_p, _fp, C.c_int64, C.POINTER(C.c_int64)]
    lib.gnnb_profile_read.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.gnnb_profile_reset.argtypes = [vp]
    for name in EXPORTS:
        getattr(lib, name)
    _lib = lib
    return lib


def fptr(t) -> '_fp':
    """float* of a contiguous fp32 torch tensor (host or device)."""
    return C.cast(t.data_ptr(), _fp)


def fptr_array(tensors) -> '_fpp':
    arr = (_fp * len(tensors))(*[fptr(t) for t in tensors])
    return C.cast(arr, _fpp), arr
