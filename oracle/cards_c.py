"""ctypes loader for oracle/libcards_oracle.so, the C oracle of whole-card requests
(oracle/cards_oracle.c, DESIGN.md §2.8).  TEST INFRASTRUCTURE ONLY.

build() compiles it next to this file (__graft_entry__.build() calls it); load() builds it when
it is missing.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(_HERE, "cards_oracle.c")
LIB_PATH = os.path.join(_HERE, "libcards_oracle.so")
_lib = None


def build() -> None:
    if os.path.exists(LIB_PATH) and os.path.getmtime(LIB_PATH) >= os.path.getmtime(SRC):
        return
    # the system gcc, no -march=native: the library travels to machines whose CPU may differ
    subprocess.run(["/usr/bin/gcc", "-O2", "-fPIC", "-Wall", "-Wextra", "-std=c11", "-shared", "-o", LIB_PATH, SRC],
                   check=True)


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            build()
        lib = C.CDLL(LIB_PATH)
        vp = C.c_void_p
        lib.oracle_bestfit_cards_snapshot.restype = C.c_int
        lib.oracle_bestfit_cards_snapshot.argtypes = [vp, vp, C.c_int32, vp, vp, C.c_int64, vp, vp, vp, vp, vp]
        lib.oracle_replay_cards.restype = C.c_int
        lib.oracle_replay_cards.argtypes = [vp, vp, C.c_int32, vp, vp, vp, C.c_int64, vp, vp]
        _lib = lib
    return _lib


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _p(a):
    return C.c_void_p(a.ctypes.data)


def bestfit_cards_snapshot(free_core, free_mem, req_core, req_mem):
    """(idx, cards uint64[R], delta_core, delta_mem, table_out[3D]) per spec §2.8 (snapshot)."""
    fc, fm, rc, rm = _i32(free_core), _i32(free_mem), _i32(req_core), _i32(req_mem)
    D, R = fc.size, rc.size
    idx = np.empty(R, dtype=np.int32)
    cards = np.empty(R, dtype=np.uint64)
    dc = np.zeros(D, dtype=np.int64)
    dm = np.zeros(D, dtype=np.int64)
    tab = np.zeros(3 * D, dtype=np.int32)
    r = load().oracle_bestfit_cards_snapshot(_p(fc), _p(fm), D, _p(rc), _p(rm), R, _p(idx), _p(cards), _p(dc), _p(dm),
                                             _p(tab))
    if r != 0:
        raise ValueError(f"oracle_bestfit_cards_snapshot failed: {r}")
    return idx, cards, dc, dm, tab


def replay_cards(free_core, free_mem, kind, a, b):
    """(idx, cards uint64[E], free_core', free_mem') per spec §2.8 (sequential)."""
    fc, fm = _i32(free_core).copy(), _i32(free_mem).copy()
    k, a_, b_ = _i32(kind), _i32(a), _i32(b)
    out = np.empty(k.size, dtype=np.int32)
    cards = np.empty(k.size, dtype=np.uint64)
    r = load().oracle_replay_cards(_p(fc), _p(fm), fc.size, _p(k), _p(a_), _p(b_), k.size, _p(out), _p(cards))
    if r != 0:
        raise ValueError(f"oracle_replay_cards failed: {r}")
    return out, cards, fc, fm
