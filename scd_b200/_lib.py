"""ctypes binding of ``libscd_b200.so`` (the C ABI in ``include/scd_b200.h``).

There is no fallback of any kind: if the library is missing, cannot be loaded, or a call fails, a
``RuntimeError`` is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, 'libscd_b200.so')

_i64, _int, _f32, _sz, _vp = C.c_int64, C.c_int, C.c_float, C.c_size_t, C.c_void_p

# name -> (restype, argtypes); every symbol include/scd_b200.h declares
SIGNATURES = {
    'scd_version': (_int, []),
    'scd_last_error': (C.c_char_p, []),
    'scd_debug_set_name_profile': (None, [_vp]),
    'scd_pairwise_distance': (_int, [_vp, _i64, _int, _vp, _int, _vp, _vp, _vp]),
    'scd_estep_workspace_bytes': (_sz, [_int, _int]),
    'scd_estep_uses_tensor_cores': (_int, [_i64, _int, _int]),
    'scd_estep': (_int, [_vp, _i64, _int, _vp, _int, _vp, _vp, _vp, _int, _vp, _sz, _vp]),
    'scd_kpp_workspace_bytes': (_sz, [_i64]),
    'scd_kpp_update': (_int, [_vp, _i64, _int, _vp, _vp, _int, _vp, _vp, _vp, _sz, _vp]),
    'scd_kpp_select': (_int, [_vp, _i64, _int, C.c_double, _vp, _vp, _vp, _sz, _vp]),
    'scd_labelled_inertia': (_int, [_vp, _vp, _i64, _int, _vp, _int, _vp, _vp]),
    'scd_mstep_workspace_bytes': (_sz, [_i64, _int]),
    'scd_mstep_sums': (_int, [_vp, _vp, _i64, _int, _int, _vp, _vp, _vp, _sz, _vp]),
    'scd_pack_counts_inertia': (_int, [_vp, _vp, _int, _vp, _vp]),
    'scd_finalize_centers': (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _int, _int, _vp, _sz, _vp, _sz, _vp]),
    'scd_vocab_prepare': (_int, [_vp, _int, _int, _i64, _i64, _vp, _vp]),
    'scd_cast_bf16': (_int, [_vp, _i64, _vp, _vp]),
    'scd_gather_rows_bf16': (_int, [_vp, _vp, _int, _int, _i64, _vp, _vp]),
    'scd_name_topk_workspace_bytes': (_sz, [_i64, _i64, _int]),
    'scd_name_topk_plan': (_int, [_i64, _i64, _int, _vp]),
    'scd_name_topk_plan_pair': (_int, [_i64, _i64, _int, _int, _vp, _int]),
    'scd_name_topk': (_int, [_vp, _i64, _int, _vp, _i64, _f32, _int, _int, _i64, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'scd_topk_merge': (_int, [_vp, _vp, _vp, _vp, _int, _i64, _int, _f32, _int, _vp, _vp, _vp]),
    'scd_vote_workspace_bytes': (_sz, [_i64, _int]),
    'scd_vote_spill_bytes': (_sz, [_i64, _int]),
    'scd_vote': (_int, [_vp, _int, _int, _vp, _i64, _int, _vp, _int, _int, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    'scd_vote_presorted': (_int, [_vp, _int, _int, _vp, _i64, _int, _vp, _int, _int, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'scd_pack_vote_records': (_int, [_vp, _vp, _int, _int, _i64, _vp, _vp]),
    'scd_vote_records': (_int, [_vp, _int, _i64, _int, _vp, _int, _int, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp]),
    'scd_peer_flag_bytes': (_sz, []),
    'scd_peer_mstep_bytes': (_sz, [_int, _int]),
    'scd_peer_barrier': (_int, [_vp, _int, _int, _int, _vp]),
    'scd_finalize_centers_peer': (_int, [_vp, _vp, _int, _int, _int, _sz, _vp, _vp, _vp, _vp, _vp, _int, _int, _vp, _sz, _vp]),
    'scd_pack_vote_records_peer': (_int, [_vp, _int, _int, _sz, _vp, _vp, _int, _int, _i64, _i64, _vp]),
    'scd_pack_sorted_records_peer': (_int, [_vp, _int, _int, _sz, _sz, _vp, _int, _int, _i64, _i64, _vp, _int, _vp]),
    'scd_vote_segments': (_int, [_vp, _int, _i64, _i64, _int, _vp, _int, _vp, _int, _int, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'scd_label_histogram': (_int, [_vp, _i64, _int, _vp, _vp]),
    'scd_constrained_assign': (_int, [_vp, _i64, _int, _i64, _i64, _vp, C.POINTER(_i64), C.POINTER(_i64)]),
    'scd_contingency': (_int, [_vp, _int, _vp, _int, _i64, _int, _vp, _vp, _vp, _vp, _vp, _vp]),
    'scd_linear_assignment': (_int, [_vp, _int, _int, _vp, C.POINTER(_int)]),
}

ESTEP_EXACT, ESTEP_PLANES_READY = 1, 2          # scd_estep flags (include/scd_b200.h)

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f'{LIB_PATH} is missing - build it with `python -m scd_b200.build` '
                           '(scd_b200 has no CPU or library fallback)')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().scd_last_error()
        raise RuntimeError(f'{what} failed: {msg.decode() if msg else "unknown error"}')


def ptr(t) -> int | None:
    """Device (or host) address of a torch tensor, None for None."""
    return None if t is None else t.data_ptr()


_UPLOAD_STREAMS = {}


def upload_stream(device=None):
    """The one side stream per device that host -> device feature uploads are issued on (``naming.score_topk`` and
    ``kmeans.assign_from_host`` on host inputs).  Staging and destination buffers of those uploads are ALLOCATED under this
    stream, so an upload never has to wait for the work queued on the caller's stream (the caching allocator hands a
    block back only to the stream it was allocated on), and successive uploads queue behind each other on the wire."""
    import torch
    idx = torch.cuda.current_device() if device is None else torch.device(device).index
    if idx is None:
        idx = torch.cuda.current_device()
    st = _UPLOAD_STREAMS.get(idx)
    if st is None:
        st = _UPLOAD_STREAMS[idx] = torch.cuda.Stream(device=idx)
    return st
