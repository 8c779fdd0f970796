"""ctypes binding of libagcf.so (include/agcf.h).

The product path has NO CPU fallback: if the shared library is missing or a
call returns an error, an exception is raised.  Device pointers come from torch
tensors (``tensor.data_ptr()``); torch is plumbing for memory and streams only.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int32, c_int64, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# ARLIB_B200_LIB selects another BUILD of the same library (kernel tuning experiments); never a fallback
LIB_PATH = os.environ.get("ARLIB_B200_LIB") or os.path.join(_HERE, "libagcf.so")

AGCF_OK = 0
_ERR = {-1: "AGCF_EINVAL", -2: "AGCF_EUNSUPPORTED", -3: "AGCF_ECUDA", -4: "AGCF_EWORKSPACE"}

P = c_void_p        # every device pointer / stream
I32, I64, U64, F32 = c_int32, c_int64, c_uint64, c_float



class SpmmArgs(ctypes.Structure):
    """struct agcf_spmm_args (include/agcf.h), field for field"""
    _fields_ = [
        ("vrows", P), ("vpart", P), ("n_vrows", I32), ("n_vrows_dev", P),
        ("col", P), ("val", P), ("partial", P), ("tickets", P),
        ("X", P), ("Y", P), ("addend", P),
        ("acc_in", P), ("acc_out", P), ("acc_div", F32),
        ("noise", P), ("eps", F32),
        ("noise_seed", U64), ("noise_stream", ctypes.c_uint32), ("noise_step", P), ("noise_main", I32),
        ("aux_Y", P * 2), ("aux_noise", P * 2), ("aux_stream", ctypes.c_uint32 * 2),
        ("row_mask", P), ("col_mask", P),
        ("peer_Y_host", P), ("peer_acc_host", P), ("n_peers", I32),
        ("mc_Y", P), ("mc_acc", P),
        ("adam_p", P), ("adam_m", P), ("adam_v", P), ("adam_coefs", P),
        ("adam_beta1", F32), ("adam_beta2", F32), ("adam_eps", F32),
        ("zero_acc_in", I32),
        ("sched", P),
        ("d", I32),
        ("flags", I32),
        ("mask_bits", I32),
        ("acc_terms", P * 8), ("n_acc_terms", I32),
        ("addend_mask", P),
    ]


# name -> (restype, argtypes); mirrors include/agcf.h one to one
SIGNATURES = {
    "agcf_abi_version": (c_int32, []),
    "agcf_strerror": (c_char_p, [c_int32]),
    "agcf_last_cuda_error": (c_int32, []),
    "agcf_last_cuda_error_where": (c_char_p, []),
    "agcf_device_sm_count": (c_int32, []),
    "agcf_norm_adj_csr": (c_int32, [P, P, P, P, P, P, I32, I64, P]),
    "agcf_csr_expand_rows": (c_int32, [P, P, I32, I64, P]),
    "agcf_spmm_csr_f32": (c_int32, [P, P, I32, P, P, P, P, P, P, P, P, P, F32, P, F32, P, P, P, P, I32, P, P, I32, P]),
    "agcf_spmm_csr_f32_ex": (c_int32, [ctypes.POINTER(SpmmArgs), P]),
    "agcf_spmm_batch_worklists": (c_int32, [P, P, I32, I32, P, I32, I32, I32, I32, P, P, P, I32, P]),
    "agcf_adam_coefs": (c_int32, [P, I32, F32, F32, F32, P, P]),
    "agcf_sddmm_csr_f32": (c_int32, [P, P, P, P, P, I32, P, I32, I32, P]),
    "agcf_concat_rows_f32": (c_int32, [P, I64, P, I64, P, I32, P]),
    "agcf_bpr_sample_epoch": (c_int32, [P, P, I32, P, P, I32, U64, U64, P, P, P, P]),
    "agcf_bpr_group_batches": (c_int32, [P, P, P, I32, I32, I32, P, P, P, P, I32, P, P]),
    "agcf_bpr_cl_ids": (c_int32, [P, P, P, P, I32, I32, I32, P, P, P, P]),
    "agcf_bpr_ws_bytes": (c_int64, [I32]),
    "agcf_bpr_forward": (c_int32, [P, P, P, P, I32, I32, I32, F32, P, P, P, P]),
    "agcf_bpr_xchg_bytes": (c_int64, [I32]),
    "agcf_bpr_partial": (c_int32, [P, P, P, P, I32, I32, I32, I32, I32, P, P, I32, P]),
    "agcf_bpr_finish": (c_int32, [P, I32, I32, I32, F32, P, P, P, P, P]),
    "agcf_bpr_backward": (c_int32, [P, P, P, P, I32, I32, I32, F32, F32, P, P, P, P, P, P, P, P]),
    "agcf_zero_rows": (c_int32, [P, P, I32, P, I32, P]),
    "agcf_infonce_ws_bytes": (c_int64, [I32, I32]),
    "agcf_infonce_forward": (c_int32, [P, P, P, I32, P, I32, F32, P, P, I64, P]),
    "agcf_infonce_backward": (c_int32, [I32, P, I32, F32, P, F32, P, I64, P, P, I32, P, P, I32, P]),
    "agcf_ngcf_dense_forward": (c_int32, [P, P, P, P, P, P, F32, I32, I32, P]),
    "agcf_ngcf_dense_backward": (c_int32, [P, P, P, P, P, P, P, P, I32, I32, I32, P]),
    "agcf_ngcf_reduce_wgrad": (c_int32, [P, I32, P, I32, P]),
    "agcf_ngcf_dense_forward_peers": (c_int32, [P, P, P, P, P, P, F32, I32, I32, P, P, I32, P, P, P]),
    "agcf_ngcf_dense_backward_peers": (c_int32, [P, P, P, P, P, P, P, P, I32, I32, I32, P, I32, P, P]),
    "agcf_ngcf_reduce_wgrad_peers": (c_int32, [P, I32, P, I32, P, I32, P, P]),
    "agcf_adam_step_f32": (c_int32, [P, P, P, P, I64, F32, F32, F32, F32, I32, P, P, I32, P, P]),
    "agcf_increment_i32": (c_int32, [P, P]),
    "agcf_group_handoff": (c_int32, [P, P, I32, I32, P, P, P]),
    "agcf_score_topk_ws_bytes": (c_int64, [I32, I32, I32, I32]),
    "agcf_score_topk": (c_int32, [P, P, I32, P, I32, I32, P, P, I32, I32, I32, P, P, P, P, I64, P]),
    "agcf_score_group_max": (c_int32, [P, P, I32, P, I32, I32, P, P, I32, I32, P, P, I64, P]),
    "agcf_topk_merge": (c_int32, [P, P, I32, I32, I32, P, P, P]),
    "agcf_score_rows": (c_int32, [P, P, I32, P, I32, I32, P, P]),
    "agcf_rank_metrics": (c_int32, [P, I32, P, P, P, I32, P, I32, P, P, P]),
}


class AgcfError(RuntimeError):
    pass


_lib = None


def load():
    """Load libagcf.so (once).  Raises if it has not been built: there is no
    fallback implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise AgcfError(
            "libagcf.so not found at %s -- build it with `make -C arlib_b200/csrc` "
            "(or python -c 'import __graft_entry__ as g; g.build()'); arlib_b200 has no CPU fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc == AGCF_OK:
        return
    lib = load()
    msg = "%s failed: %s (%s)" % (what or "agcf call", _ERR.get(rc, rc), lib.agcf_strerror(rc).decode())
    if rc == -3:
        msg += " cudaError=%d: %s" % (lib.agcf_last_cuda_error(), lib.agcf_last_cuda_error_where().decode())
    raise AgcfError(msg)


def ptr(t):
    """device pointer of a torch tensor (or None -> NULL)"""
    if t is None:
        return None
    return t.data_ptr()


def ptr_array(ptrs):
    """host array of device pointers (void* const*) for the peer arguments"""
    if not ptrs:
        return None, 0
    arr = (c_void_p * len(ptrs))(*[int(x) for x in ptrs])
    return arr, len(ptrs)


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream
