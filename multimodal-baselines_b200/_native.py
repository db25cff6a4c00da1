"""ctypes binding of libmmb_b200.so (the C ABI in include/mmb_b200.h).

There is no CPU fallback: if the shared library is missing or cannot be loaded, importing
this module raises, and every entry point raises if no CUDA device is present.
PyTorch is used only for device memory, streams and torch.distributed.
"""
import ctypes as C
import os

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libmmb_b200.so')

MMB_OK, MMB_E_INVALID, MMB_E_CUDA, MMB_E_UNSUPPORTED, MMB_E_INDEX, MMB_E_COMM = 0, 1, 2, 3, 4, 5
STATUS_BAD_INDEX, STATUS_NONFINITE, STATUS_COMM_TIMEOUT = 1, 2, 4
GRAM_AUTO, GRAM_FP32, GRAM_TF32X3 = 0, 1, 2

if not os.path.exists(LIB_PATH):
    raise ImportError(
        'libmmb_b200.so is not built (expected at %s). Build it with '
        '`python multimodal-baselines_b200/build.py` or `python -c "import __graft_entry__ as g; '
        'g.build()"`. There is no CPU fallback for this path.' % LIB_PATH)

lib = C.CDLL(LIB_PATH)

_p, _i, _i64, _sz, _f = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_float

# name -> (restype, argtypes); mirrors include/mmb_b200.h line by line.
SIGNATURES = {
    'mmb_version': (_i, []),
    'mmb_last_error': (C.c_char_p, []),
    'mmb_device_info': (_i, [C.POINTER(_i)] * 3),
    'mmb_set_option': (_i, [C.c_char_p, _i]),
    'mmb_launch_count': (C.c_ulonglong, []),
    'mmb_last_kernel': (C.c_char_p, [_i]),
    'mmb_host_alloc': (_i, [C.POINTER(_p), _sz]),
    'mmb_host_alloc_wc': (_i, [C.POINTER(_p), _sz]),
    'mmb_host_free': (_i, [_p]),
    'mmb_seq2weight': (_i, [_p, _p, _p, _i64, _i64, _i64, _p, _p, _p]),
    'mmb_weighted_average': (_i, [_p, _i64, _i, _p, _p, _i64, _i64, _p, _p, _p]),
    'mmb_sif_embed': (_i, [_p, _i64, _i, _p, _p, _i64, _i64, _p, _p, _p]),
    'mmb_sif_embed_workspace_bytes': (_sz, [_i64, _i, _i64, _i64]),
    'mmb_sif_embed_ws': (_i, [_p, _i64, _i, _p, _p, _i64, _i64, _p, _p, _p, _sz, _p]),
    'mmb_sif_embed_multi_workspace_bytes': (_sz, [_i64, _i]),
    'mmb_sif_embed_multi': (_i, [_p, _i64, _i, _p, _i, _p, _i64, _i64, _p, _p, _p, _sz, _p]),
    'mmb_sif_embed_gram_workspace_bytes': (_sz, [_i64, _i, _i64, _i64, _i]),
    'mmb_sif_embed_gram': (_i, [_p, _i64, _i, _p, _p, _i64, _i64, _p, _p, _p, _p, _sz, _i, _p]),
    'mmb_sif_embed_ragged': (_i, [_p, _i64, _i, _p, _p, _p, _i64, _i64, _i64, _p, _p, _p]),
    'mmb_ids_lengths': (_i, [_p, _i64, _i64, _i64, _p, _p, _p]),
    'mmb_ids_compact': (_i, [_p, _i64, _i64, _p, _p, _p]),
    'mmb_token_mask': (_i, [_p, _i64, _p, _p]),
    'mmb_step_mask': (_i, [_p, _i64, _i, _p, _p]),
    'mmb_gram_workspace_bytes': (_sz, [_i64, _i, _i]),
    'mmb_gram': (_i, [_p, _i64, _i, _p, _p, _sz, _i, _p]),
    'mmb_pc_workspace_bytes': (_sz, [_i, _i]),
    'mmb_pc_from_gram': (_i, [_p, _i, _p, _i, _i, _i, _i, _p, _p, _sz, _p]),
    'mmb_start_block_xt': (_i, [_p, _i64, _i, _p, _i, _p, _p]),
    'mmb_remove_pc': (_i, [_p, _i64, _i, _p, _i, _p, _p]),
    'mmb_sif_workspace_bytes': (_sz, [_i64, _i, _i]),
    'mmb_sif_embedding': (_i, [_p, _i64, _i, _p, _p, _i64, _i64, _i, _p, _p, _p, _p, _p, _sz, _i, _p, _p]),
    'mmb_sif_embedding_host': (_i, [_p, _i64, _i, _p, _p, _i64, _i64, _i, _p, _p, _i, _p, _i, _i64]),
    'mmb_sif_embedding_host_peer': (_i, [_p, _i64, _i, _p, _p, _i64, _i64, _i, _p, _p, _i, _p, _i, _i64, _i64, _i, _i,
                                         _p, C.c_uint64]),
    'mmb_host_pipeline_trim': (_i, [_sz]),
    'mmb_comm_abort': (_i, [_i, _i, _p, C.c_uint64, _p]),
    'mmb_comm_bytes': (_sz, []),
    'mmb_comm_alloc': (_i, [C.POINTER(_p)]),
    'mmb_comm_free': (_i, [_p]),
    'mmb_comm_export': (_i, [_p, _p]),
    'mmb_comm_open': (_i, [_p, C.POINTER(_p)]),
    'mmb_comm_close': (_i, [_p]),
    'mmb_allreduce_peer': (_i, [_p, _i64, _i, _i, _i, _p, C.c_uint64, _p, _p]),
    'mmb_gram_allreduce_peer': (_i, [_p, _i64, _i, _p, _p, _sz, _i, _i, _i, _p, C.c_uint64, _p, _p]),
    'mmb_heads_forward': (_i, [_p, _i, _i, _i, _p, _p, _p, _p, _p, _p]),
    'mmb_heads_backward_workspace_bytes': (_sz, [_i, _i, _i, _p]),
    'mmb_heads_backward': (_i, [_p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    'mmb_scale_multi': (_i, [_i, _i, _p, _p, _p, _p, _p, _p]),
    'mmb_combine_lp': (_i, [_p, _p, _i, _i, _f, _f, _p, _p, _p, _p]),
    'mmb_combine_lp_backward': (_i, [_p, _i, _i, _f, _f, _p, _p, _p, _p, _p]),
    'mmb_gather_multi': (_i, [_i, _i, _p, _p, _p, _p, _p]),
    'mmb_gauss_ll': (_i, [_i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    'mmb_closed_form_stats': (_i, [_i, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    'mmb_closed_form_finish': (_i, [_i, _i, _i, _p, _p, _p, _p, _i, _p, _p]),
    'mmb_feature_minmax_workspace_bytes': (_sz, [_i64, _i]),
    'mmb_feature_minmax': (_i, [_p, _i64, _i, _p, _p, _p, _sz, _p]),
    'mmb_prep_features': (_i, [_p, _i64, _i, _i, _p, _i, _i, _p, _p, _p, _p, _p]),
    'mmb_row_inv_norm': (_i, [_p, _i64, _i, _p, _p]),
    'mmb_word_ll_workspace_bytes': (_sz, [_i, _i64, _i]),
    'mmb_word_ll': (_i, [_p, _i, _i, _p, _p, _i64, _p, _i64, _i64, _p, _p, _i64, _i64, _i, _f, _p, _p,
                         _p, _sz, _p, _p]),
    'mmb_gauss_moments': (_i, [_p, _p, _i64, _i, _i, _p, _p]),
    'mmb_gauss_ll_stats': (_i, [_i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    'mmb_word_ll_ids_workspace_bytes': (_sz, [_i, _i64, _i]),
    'mmb_word_ll_ids': (_i, [_p, _i, _i, _p, _p, _i64, _p, _i64, _p, _p, _i64, _i64, _i, _f, _p, _p,
                             _p, _sz, _p, _p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)   # AttributeError here = header and library disagree
    _fn.restype = _res
    _fn.argtypes = _args


class MMBError(RuntimeError):
    pass


def last_error():
    return (lib.mmb_last_error() or b'').decode('utf-8', 'replace')


def check(rc):
    """Turn a non-zero return code into the exception the reference would raise."""
    if rc == MMB_OK:
        return
    msg = last_error()
    if rc == MMB_E_INDEX:
        raise IndexError(msg)
    if rc == MMB_E_INVALID:
        raise ValueError(msg)
    if rc == MMB_E_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise MMBError('libmmb_b200 rc=%d: %s' % (rc, msg))


def require_cuda():
    if not torch.cuda.is_available():
        raise MMBError('libmmb_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
    return torch.device('cuda', torch.cuda.current_device())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device (or pinned-host) pointer of a contiguous torch tensor; None -> NULL."""
    if t is None:
        return C.c_void_p(0)
    assert t.is_contiguous(), 'libmmb_b200 takes dense row-major buffers'
    return C.c_void_p(t.data_ptr())


def np_ptr(a):
    if a is None:
        return C.c_void_p(0)
    assert a.flags['C_CONTIGUOUS']
    return C.c_void_p(a.ctypes.data)


def to_device(a, dtype, device=None):
    """NumPy array / torch tensor -> contiguous CUDA tensor of `dtype` (no copy if already so)."""
    device = device or require_cuda()
    if isinstance(a, torch.Tensor):
        return a.to(device=device, dtype=dtype).contiguous()
    a = np.asarray(a)
    if a.dtype == np.float64 and dtype == torch.float32:
        a = a.astype(np.float32)          # same rounding as NumPy's own float64 -> float32 cast
    return torch.as_tensor(np.ascontiguousarray(a)).to(device=device, dtype=dtype).contiguous()


def raise_on_status(status_tensor, V=None):
    """Read a device status word (synchronises) and raise like the reference would."""
    s = int(status_tensor.item())
    if s & STATUS_BAD_INDEX:
        raise IndexError('index out of bounds for axis 0 with size %s' % (V if V is not None else '?'))
    return s


class PinnedArray:
    """A NumPy array backed by cudaHostAlloc memory (full PCIe rate for the *_host calls)."""

    def __init__(self, shape, dtype, write_combined=False):
        self.dtype = np.dtype(dtype)
        self.shape = tuple(int(s) for s in np.atleast_1d(shape))
        nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self._ptr = C.c_void_p()
        check((lib.mmb_host_alloc_wc if write_combined else lib.mmb_host_alloc)(C.byref(self._ptr), nbytes))
        buf = (C.c_char * max(nbytes, 1)).from_address(self._ptr.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def free(self):
        if self._ptr is not None and self._ptr.value:
            self.array = None
            lib.mmb_host_free(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
