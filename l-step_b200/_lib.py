"""ctypes binding of liblstep_b200.so — the thin C-ABI layer between the PyTorch host and the
sm_100a kernels (include/lstep_b200.h). PyTorch is used for device memory and streams only;
every argument crosses the boundary as a raw device pointer.

There is no CPU implementation behind this module: if the library is missing or no B200-class
device is present, the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

from . import build as _build

_LIB = None
_LOCK = threading.Lock()

i64, i32, f32p, vp = C.c_int64, C.c_int, C.c_void_p, C.c_void_p
sz = C.c_size_t


class CSR(C.Structure):
    """struct lstep_csr"""
    _fields_ = [("indptr", vp), ("nbr", vp), ("eid", vp), ("t", vp), ("num_rows", i64), ("nnz", i64)]


class PEStreamDesc(C.Structure):
    """struct lstep_pe_stream"""
    _fields_ = [("src", vp), ("dst", vp), ("t", vp), ("ring", vp), ("cur", vp), ("V1", i64), ("T", i32), ("d", i32), ("row_cap", i64)]


class ChangeLog(C.Structure):
    """struct lstep_changelog"""
    _fields_ = [("base", vp), ("ev_node", vp), ("ev_row", vp), ("ev_cnt", vp), ("ev_hash", vp), ("ev_mask", vp), ("rows", i64),
                ("T", i32), ("cap", i32), ("H", i32), ("d", i32), ("row_mul", i64), ("row_add", i64)]


class PeerGroup(C.Structure):
    """struct lstep_peer_group"""
    _fields_ = [("rank", i32), ("world", i32), ("table", vp * 16), ("new_rows", vp * 16), ("filt", vp * 16), ("inbox", vp * 16),
                ("flags", vp * 16), ("cap", i64)]


class PEMLP(C.Structure):
    """struct lstep_pe_mlp"""
    _fields_ = [("w1", vp), ("b1", vp), ("w2", vp), ("b2", vp), ("ws", vp), ("bs", vp), ("tw", vp), ("d", i32), ("t", i32),
                ("w1_tc", vp), ("w2_tc", vp), ("ws_tc", vp)]


_SIGS = {
    "lstep_strerror": (C.c_char_p, [i32]),
    "lstep_last_cuda_error": (C.c_char_p, []),
    "lstep_abi_version": (i32, []),
    "lstep_device_ok": (i32, []),
    "lstep_csr_build_workspace_bytes": (sz, [i64, i64]),
    "lstep_csr_build_from_edges": (i32, [vp, vp, vp, vp, i64, i64, vp, vp, vp, vp, vp, sz, vp, vp]),
    "lstep_csr_build_from_entries": (i32, [vp, vp, vp, vp, i64, i64, vp, vp, vp, vp, vp, sz, vp, vp]),
    "lstep_csr_relayout": (i32, [C.POINTER(CSR), vp, vp, vp, vp, vp, vp, vp, vp]),
    "lstep_csr_ingest": (i32, [C.POINTER(CSR), vp, vp, vp, vp, i64, vp, i64, vp, vp]),
    "lstep_csr_relayout_rows": (i32, [C.POINTER(CSR), vp, i64, i64, vp, i64, vp, vp, vp, vp, vp, vp]),
    "lstep_csr_add_rows": (i32, [C.POINTER(CSR), vp, i64, vp, vp]),
    "lstep_sample_recent": (i32, [C.POINTER(CSR), vp, vp, i64, i64, i32, vp, vp, vp, vp, vp]),
    "lstep_sample_recent_compact": (i32, [C.POINTER(CSR), vp, vp, i64, i64, i32, vp, vp, vp, vp]),
    "lstep_dft_collapse": (i32, [vp, vp, i32, i32, i32, vp, vp]),
    "lstep_dft_filter": (i32, [vp, i64, i64, i32, i32, i32, i32, vp, i64, vp, vp, i64, vp]),
    "lstep_dft_filter_bwd": (i32, [vp, i64, i64, i32, i32, i32, i32, vp, i64, vp, vp, vp]),
    "lstep_packed_ld": (i32, [i32]),
    "lstep_packed_rows": (i32, [i32]),
    "lstep_pack_linear": (i32, [vp, vp, i32, i32, vp, vp, vp]),
    "lstep_packed_tc_floats": (sz, [i32, i32]),
    "lstep_pack_linear_tc": (i32, [vp, i32, i32, vp, vp]),
    "lstep_time_features": (i32, [vp, i64, vp, i32, vp, vp]),
    "lstep_feature_aggregate": (i32, [C.POINTER(CSR), vp, vp, i64, i64, i32, vp, i64, i32, vp, i32, vp, vp, vp, vp]),
    "lstep_nbr_aggregate": (i32, [vp, i64, vp, vp, vp, i64, i32, vp, i32, i32, vp, vp]),
    "lstep_nbr_lookup_aggregate": (i32, [C.POINTER(CSR), vp, vp, i64, i32, vp, i64, vp, i32, i32, vp, vp, vp]),
    "lstep_nbr_aggregate_bwd": (i32, [vp, vp, i64, i32, i32, i32, vp, i64, vp]),
    "lstep_neighborhood_pe": (i32, [vp, i64, vp, vp, vp, vp, i64, i32, C.POINTER(PEMLP), vp, vp, sz, vp]),
    "lstep_pe_mlp_apply": (i32, [vp, vp, vp, i64, C.POINTER(PEMLP), vp, i64, vp, vp]),
    "lstep_update_pe_workspace_bytes": (sz, [i64, i64, i32, i32, i32, i64]),
    "lstep_update_pe": (i32, [vp, i64, C.POINTER(CSR), vp, i64, vp, vp, vp, i64, C.c_double, i32, C.POINTER(PEMLP), vp, sz,
                              vp, vp]),
    "lstep_update_pe_workspace_init": (i32, [vp, sz, i64, vp]),
    "lstep_update_pe_phase_a": (i32, [vp, i64, vp, i64, vp, vp, vp, i64, C.c_double, i32, C.POINTER(PEMLP), vp, sz, vp]),
    "lstep_update_pe_phase_b_partial": (i32, [vp, i64, C.POINTER(CSR), vp, vp, i64, vp, i64, i64, C.c_double, i32, C.POINTER(PEMLP),
                                              vp, sz, vp, vp]),
    "lstep_update_pe_workspace_layout": (i32, [i64, i64, i32, i32, i32, i64, C.POINTER(i64)]),
    "lstep_segment_sum_rows": (i32, [vp, i64, vp, i64, i32, vp, i64, vp]),
    "lstep_dft_filter_scatter": (i32, [vp, i64, i64, i32, i32, i32, i32, vp, vp, i64, vp, vp, i64, vp]),
    "lstep_ring_copy_rows": (i32, [vp, vp, i64, i32, i32, i32, i64, i64, i32, vp]),
    "lstep_pe_step_workspace_bytes": (sz, [i64, i64, i32, i32, i32, i32, i64]),
    "lstep_ring_load": (i32, [vp, vp, i64, i32, i32, i32, vp]),
    "lstep_pe_rows_init": (i32, [vp, vp, i32, i32, vp, i64, i64, i64, i64, vp, i64, vp]),
    "lstep_pe_step": (i32, [C.POINTER(PEStreamDesc), C.POINTER(CSR), i64, i64, vp, i64, C.c_double, i32, i32, i32, vp,
                            C.POINTER(C.c_void_p), i32, vp, i32, C.POINTER(PEMLP), C.POINTER(PEMLP), vp, sz, vp, vp]),
    "lstep_pe_steps": (i32, [C.POINTER(PEStreamDesc), C.POINTER(CSR), i64, vp, vp, vp, vp, vp, C.POINTER(i32), C.POINTER(i32), vp,
                             C.POINTER(C.c_void_p), vp, i32, vp, i64, i32, C.POINTER(PEMLP), C.POINTER(PEMLP), vp, sz, vp, vp]),
    "lstep_pe_step_sharded": (i32, [C.POINTER(PEStreamDesc), C.POINTER(CSR), i64, i64, vp, i64, C.c_double, C.POINTER(C.c_void_p), i32, i64, i64,
                                    vp, i32, C.POINTER(PEMLP), C.POINTER(PEMLP), vp, sz, vp, vp]),
    "lstep_changelog_filter": (i32, [C.POINTER(ChangeLog), i32, i32, vp, i64, vp, vp, i64, vp, vp]),
    "lstep_changelog_append": (i32, [C.POINTER(ChangeLog), i32, i32, vp, vp, vp, i64, vp, i64, vp, i32, i32, vp, vp]),
    "lstep_pe_step_changelog": (i32, [C.POINTER(PEStreamDesc), C.POINTER(ChangeLog), C.POINTER(CSR), i64, i64, vp, i64, C.c_double, i32, i32, vp,
                                      C.POINTER(C.c_void_p), i32, i64, i64, vp, i32, C.POINTER(PEMLP), C.POINTER(PEMLP), vp, sz, vp, vp, i32]),
    "lstep_peer_inbox_bytes": (sz, [i32, i64, i32]),
    "lstep_ipc_alloc": (i32, [sz, C.POINTER(C.c_void_p)]),
    "lstep_ipc_free": (i32, [vp]),
    "lstep_ipc_export": (i32, [vp, C.POINTER(C.c_ubyte)]),
    "lstep_ipc_open": (i32, [C.POINTER(C.c_ubyte), C.POINTER(C.c_void_p)]),
    "lstep_ipc_close": (i32, [vp]),
    "lstep_peer_rows_bcast": (i32, [vp, i64, i32, vp, C.POINTER(PeerGroup), i32, C.c_uint32, vp]),
    "lstep_peer_signal": (i32, [C.POINTER(PeerGroup), C.c_uint32, vp]),
    "lstep_peer_sync_tables": (i32, [C.POINTER(PeerGroup), C.c_uint32, i32, vp, i32, i64, vp]),
    "lstep_peer_wait": (i32, [C.POINTER(PeerGroup), C.c_uint32, i32, vp, vp]),
    "lstep_pe_step_peer": (i32, [C.POINTER(PEStreamDesc), C.POINTER(ChangeLog), C.POINTER(CSR), C.POINTER(PeerGroup), i64, i64, vp, i64, vp, vp, i64,
                                 C.c_double, i32, i32, vp, C.POINTER(C.c_void_p), i32, i64, i64, vp, i32, C.POINTER(PEMLP), C.POINTER(PEMLP), vp, sz,
                                 vp, C.c_uint32, i32, i32, vp]),
    "lstep_pe_steps_peer": (i32, [C.POINTER(PEStreamDesc), C.POINTER(ChangeLog), C.POINTER(CSR), C.POINTER(PeerGroup), i64, vp, vp, vp, vp, vp, vp, vp,
                                  vp, C.POINTER(i32), vp, C.POINTER(C.c_void_p), vp, i32, vp, i64, i32, C.POINTER(PEMLP), C.POINTER(PEMLP), vp, sz,
                                  vp, C.POINTER(C.c_uint32), i32, vp]),
    "lstep_set_option": (i32, [C.c_char_p, i32]),
    "lstep_get_option": (i32, [C.c_char_p, C.POINTER(i32)]),
    "lstep_step_profile": (i32, [i32]),
    "lstep_step_profile_read": (i32, [C.POINTER(C.c_float)]),
    "lstep_step_profile_read_all": (i32, [C.POINTER(C.c_float), i32]),
    "lstep_host_stepper_create": (i32, [i32, i64, i32, i32, C.POINTER(C.c_void_p)]),
    "lstep_host_stepper_destroy": (None, [vp]),
    "lstep_pe_step_host": (i32, [vp, C.POINTER(PEStreamDesc), C.POINTER(CSR), i64, vp, vp, vp, vp, i64, i32, i32, i32, vp,
                                 C.POINTER(C.c_void_p), i32, vp, i32, C.POINTER(PEMLP), C.POINTER(PEMLP), vp, sz, vp, vp,
                                 C.POINTER(i64)]),
    "lstep_pe_steps_host": (i32, [vp, C.POINTER(PEStreamDesc), C.POINTER(CSR), i64, i64, vp, vp, vp, C.POINTER(C.c_void_p), i32,
                                  C.POINTER(i32), C.POINTER(i32), vp, i32, C.POINTER(PEMLP), C.POINTER(PEMLP), vp, sz, vp, vp, vp,
                                  C.POINTER(i64)]),
    "lstep_pe_step_changelog_host": (i32, [vp, C.POINTER(PEStreamDesc), C.POINTER(ChangeLog), C.POINTER(CSR), i64, vp, vp, vp, vp, i64, i32,
                                           i32, vp, C.POINTER(C.c_void_p), i32, vp, i32, C.POINTER(PEMLP), C.POINTER(PEMLP), vp, sz, vp, vp,
                                           C.POINTER(i64)]),
    "lstep_pe_steps_changelog_host": (i32, [vp, C.POINTER(PEStreamDesc), C.POINTER(ChangeLog), C.POINTER(CSR), i64, i64, vp, vp, vp,
                                            C.POINTER(C.c_void_p), i32, C.POINTER(i32), C.POINTER(i32), vp, i32, C.POINTER(PEMLP),
                                            C.POINTER(PEMLP), vp, sz, vp, vp, vp, C.POINTER(i64)]),
    "lstep_pe_step_peer_host": (i32, [vp, C.POINTER(PEStreamDesc), C.POINTER(ChangeLog), C.POINTER(CSR), C.POINTER(PeerGroup), i64, vp, vp, vp, vp,
                                      i64, i32, i32, vp, C.POINTER(C.c_void_p), i32, vp, i32, C.POINTER(PEMLP), C.POINTER(PEMLP), vp, sz, vp,
                                      C.c_uint32, i32, i32, vp, C.POINTER(i64)]),
    "lstep_pe_steps_peer_host": (i32, [vp, C.POINTER(PEStreamDesc), C.POINTER(ChangeLog), C.POINTER(CSR), C.POINTER(PeerGroup), i64, i64, vp, vp,
                                       vp, C.POINTER(C.c_void_p), i32, C.POINTER(i32), C.POINTER(i32), vp, i32, C.POINTER(PEMLP),
                                       C.POINTER(PEMLP), vp, sz, vp, C.POINTER(C.c_uint32), i32, vp, vp, C.POINTER(i64)]),
    "lstep_host_stepper_set_ingest": (i32, [vp, vp, i64, C.c_double]),
    "lstep_host_step_result": (i32, [vp, i64, C.POINTER(C.POINTER(C.c_float)), C.POINTER(i64)]),
    "lstep_host_stepper_bytes": (None, [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
}

EXPORTS = tuple(_SIGS)


class LstepError(RuntimeError):
    pass


def library_path() -> str:
    return _build.LIB


def load(require_device: bool = True):
    """Load (building first if the sources changed and nvcc is present) the CUDA library."""
    global _LIB
    with _LOCK:
        if _LIB is None:
            try:
                _build.build()
            except Exception:
                if not os.path.exists(_build.LIB):
                    raise
            if not os.path.exists(_build.LIB):
                raise LstepError(f"{_build.LIB} is missing: build it with `python -m lstep_b200.build` "
                                 "(lstep_b200 has no CPU path)")
            lib = C.CDLL(_build.LIB)
            for name, (res, args) in _SIGS.items():
                fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
                fn.restype, fn.argtypes = res, args
            if lib.lstep_abi_version() != 2:
                raise LstepError("liblstep_b200.so ABI version mismatch; rebuild")
            _LIB = lib
    if require_device:
        if not torch.cuda.is_available():
            raise LstepError("lstep_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return _LIB


def check(status: int, what: str = ""):
    if status == 0:
        return
    lib = load(False)
    msg = lib.lstep_strerror(status).decode()
    if status == 4:
        msg += ": " + lib.lstep_last_cuda_error().decode()
    if status == 1:
        raise ValueError(f"{what}: {msg}")
    if status == 5:  # the reference raises IndexError for a node id outside its tables
        raise IndexError(f"{what}: index out of range ({msg})")
    raise LstepError(f"{what}: {msg}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


FLAG_NODE_OUT_OF_RANGE = 1
FLAG_UNSORTED_STREAM = 2
FLAG_CHANGELOG_FULL = 4
FLAG_PEER_TIMEOUT = 8
FLAG_CSR_FULL = 16
FLAG_FIXED_POINT_RANGE = 32


def fixed_point_bound(n_ids: int, K: int) -> float:
    """The magnitude phase B's 32.32 fixed-point sums take: 2^31 / (n_ids*K + 1), rounded toward zero to fp32
    (fixed_point_bound() in csrc/common.cuh). A contribution x is in range when |x| < bound."""
    import numpy as np
    b = 2.0 ** 31 / (float(n_ids) * int(K) + 1.0)
    f = np.float32(b)
    if float(f) > b:
        f = np.nextafter(f, np.float32(0))
    return float(f)
