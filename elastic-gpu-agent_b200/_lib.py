"""ctypes binding of the C ABI declared in include/egpu_alloc.h.

The library is built in-tree by __graft_entry__.build() (nvcc, sm_100a) as
elastic-gpu-agent_b200/lib/libegpu_alloc.so.  Importing this module without it
raises: there is no Python or CPU fallback for the allocation path.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# EGPU_LIB_PATH: experiments only (an alternative build of the same sources)
LIB_PATH = os.environ.get("EGPU_LIB_PATH") or os.path.join(_HERE, "lib", "libegpu_alloc.so")

i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)

OK = 0
ERR_INVALID = -1
ERR_NO_DEVICE = -2
ERR_CUDA = -3
ERR_NOMEM = -4
ERR_NO_TABLE = -5
ERR_STATE = -6
ERR_PARSE = -7
ERR_UNSAT = -8

VARIANT_AUTO = 0
VARIANT_GRID = 1
VARIANT_SORTED = 2
VARIANT_LUT = 3

F_COMMIT = 1
F_INPUTS_READY = 2
F_PREFIX_COMMIT = 4
F_APPLY = 8
IDX_DEFERRED = -2

EV_ALLOC = 0
EV_FREE = 1


MAX_BATCHES = 64


class Batch(C.Structure):
    """egpu_batch of include/egpu_alloc.h"""
    _fields_ = [("d_req_core", C.c_void_p), ("d_req_mem", C.c_void_p), ("R", C.c_int64), ("d_out_idx", C.c_void_p),
                ("d_delta", C.c_void_p), ("d_table_out", C.c_void_p)]


class EgpuError(RuntimeError):
    def __init__(self, code: int, what: str, detail: str = ""):
        self.code = code
        msg = f"{what}: {strerror(code)} ({code})"
        if detail:
            msg += f" [{detail}]"
        super().__init__(msg)


_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    sigs = {
        "egpu_abi_version": (C.c_int, []),
        "egpu_strerror": (C.c_char_p, [C.c_int]),
        "egpu_ctx_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
        "egpu_ctx_destroy": (None, [vp]),
        "egpu_last_error": (C.c_char_p, [vp]),
        "egpu_backend": (C.c_int, [vp]),
        "egpu_launch_count": (C.c_int64, [vp]),
        "egpu_set_variant": (C.c_int, [vp, C.c_int]),
        "egpu_table_set": (C.c_int, [vp, i32p, i32p, C.c_int32]),
        "egpu_table_get": (C.c_int, [vp, i32p, i32p, i32p]),
        "egpu_table_size": (C.c_int, [vp]),
        "egpu_bestfit_batch": (C.c_int, [vp, vp, vp, C.c_int64, vp, vp, vp, C.c_int]),
        "egpu_bestfit_batch_rounds": (C.c_int, [vp, vp, vp, C.c_int64, vp, vp, vp, C.c_int32, C.POINTER(C.c_int32),
                                                C.POINTER(C.c_int64)]),
        "egpu_bestfit_batch_rounds_dev": (C.c_int, [vp, vp, vp, C.c_int64, vp, vp, C.c_int32, C.POINTER(C.c_int32),
                                                    C.POINTER(C.c_int64), vp]),
        "egpu_bestfit_batch_packed": (C.c_int, [vp, vp, C.c_int64, vp, vp, vp, C.c_int]),
        "egpu_bestfit_batch_packed_dev": (C.c_int, [vp, vp, C.c_int64, vp, vp, vp, C.c_int, vp]),
        "egpu_host_alloc": (C.c_int, [vp, C.POINTER(vp), C.c_int64]),
        "egpu_host_free": (None, [vp, vp]),
        "egpu_host_register": (C.c_int, [vp, vp, C.c_int64]),
        "egpu_host_unregister": (C.c_int, [vp, vp]),
        "egpu_bestfit_batch_dev": (C.c_int, [vp, vp, vp, C.c_int64, vp, vp, vp, C.c_int, vp]),
        "egpu_table_apply_deltas_dev": (C.c_int, [vp, vp, C.c_int, vp, C.c_int, vp]),
        "egpu_synth_requests_dev": (C.c_int, [vp, C.c_int, C.c_uint64, C.c_int64, C.c_int64, vp, vp, vp]),
        "egpu_replay": (C.c_int, [vp, vp, vp, vp, C.c_int64, vp]),
        "egpu_bestfit_cards": (C.c_int, [vp, vp, vp, C.c_int64, vp, vp, vp, vp, C.c_int]),
        "egpu_bestfit_cards_dev": (C.c_int, [vp, vp, vp, C.c_int64, vp, vp, vp, vp, C.c_int, vp]),
        "egpu_replay_cards": (C.c_int, [vp, vp, vp, vp, C.c_int64, vp, vp]),
        "egpu_peer_export": (C.c_int, [vp, vp]),
        "egpu_peer_attach": (C.c_int, [vp, C.c_int, C.c_int, vp]),
        "egpu_peer_detach": (C.c_int, [vp]),
        "egpu_bestfit_batch_shard_dev": (C.c_int, [vp, vp, vp, C.c_int64, vp, vp, C.c_int, C.c_uint64, vp]),
        "egpu_bestfit_batch_shard_prefix_dev": (C.c_int, [vp, vp, vp, C.c_int64, vp, vp, vp, C.c_int, C.c_uint64, vp]),
        "egpu_bestfit_batch_shard_lag_dev": (C.c_int, [vp, vp, vp, C.c_int64, vp, vp, C.c_int, C.c_uint64, C.c_int, vp, vp]),
        "egpu_table_apply_peers_dev": (C.c_int, [vp, C.c_uint64, vp, C.c_int, vp]),
        "egpu_table_apply_peers_multi_dev": (C.c_int, [vp, C.c_uint64, C.c_int, vp, C.c_int, vp]),
        "egpu_peer_last_timeout": (C.c_int64, [vp]),
        "egpu_bestfit_batches_dev": (C.c_int, [vp, vp, C.c_int32, C.c_int, vp]),
        "egpu_bestfit_batches_shard_dev": (C.c_int, [vp, vp, C.c_int32, C.c_int, C.c_uint64, vp]),
        "egpu_peer_gate_dev": (C.c_int, [vp, vp]),
        "egpu_peer_gate_open": (C.c_int, [vp]),
        "egpu_peer_gate_timeouts": (C.c_int64, [vp]),
        "egpu_bestfit_query": (C.c_int, [vp, i32p, i32p, C.c_int32, vp, vp, C.c_int64, vp]),
        "egpu_device_hash_batch": (C.c_int, [vp, vp, vp, C.c_int64, vp, C.c_int64, vp, vp]),
        "egpu_device_hash": (C.c_int, [vp, vp, C.c_int64, vp]),
        "egpu_device_locate": (C.c_int, [vp, vp, vp, C.c_int64, vp, C.c_int64, C.POINTER(C.c_int64)]),
        "egpu_device_id_format": (C.c_int, [C.c_int32, C.c_int64, C.c_char_p, C.c_int64]),
        "egpu_device_id_parse": (C.c_int, [C.c_char_p, C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
        "egpu_preferred_allocation": (C.c_int, [vp, vp, C.c_int64, vp, C.c_int64, C.c_int32, C.c_int, vp, C.POINTER(C.c_int32)]),
        "egpu_table_restore_flat": (C.c_int, [vp, vp, vp, C.c_int64, vp, C.c_int64, vp, vp, vp, vp, vp, vp, C.c_int32, C.c_int,
                                              vp, vp]),
        "egpu_table_restore": (C.c_int, [vp, vp, vp, vp, vp, C.c_int64, vp, vp, C.c_int64, vp, vp, C.c_int32, C.c_int, vp, vp,
                                         vp]),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)  # AttributeError = header/library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def strerror(code: int) -> str:
    return load().egpu_strerror(code).decode()
