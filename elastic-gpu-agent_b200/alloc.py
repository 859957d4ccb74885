"""Host-side wrapper of the best-fit allocation path (one context per GPU).

Mirrors the slot the path occupies in the reference: a plugin owns one
allocator (constructed with the plugin, pkg/plugins/base.go:208-233), commits
are serialised by a lock (pkg/plugins/gpushare.go:114,239; the lock lives inside
the C library), errors surface as exceptions the way the Go handlers return
`error` (pkg/plugins/gpushare.go:41-43).

All compute happens in the CUDA library behind include/egpu_alloc.h; numpy
arrays here are only the caller-owned host buffers of that C ABI.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L


def _i32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.int32)


def _ptr(a: np.ndarray):
    return C.c_void_p(a.ctypes.data)


def _stream(stream):
    """cudaStream_t for the C ABI.  None -> NULL = the context's own stream.  An integer is a
    stream handle as torch reports it (`torch.cuda.Stream.cuda_stream`); torch reports the
    legacy default stream as 0, which the C ABI would read as NULL, so 0 is translated to
    cudaStreamLegacy (0x1)."""
    if stream is None:
        return C.c_void_p(None)
    return C.c_void_p(1 if int(stream) == 0 else int(stream))


class BestFitAllocator:
    """Best-fit device choice over a node-local capacity table on one B200."""

    def __init__(self, cuda_device: int = 0):
        self._lib = L.load()
        h = C.c_void_p()
        rc = self._lib.egpu_ctx_create(int(cuda_device), C.byref(h))
        if rc != L.OK:
            raise L.EgpuError(rc, "egpu_ctx_create")
        self._h = h
        self.cuda_device = int(cuda_device)

    # -- lifetime -----------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.egpu_ctx_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self) -> C.c_void_p:
        return self._h

    def _check(self, rc: int, what: str):
        if rc != L.OK:
            raise L.EgpuError(rc, what, self._lib.egpu_last_error(self._h).decode())

    @property
    def launch_count(self) -> int:
        return int(self._lib.egpu_launch_count(self._h))

    def set_variant(self, variant: int):
        self._check(self._lib.egpu_set_variant(self._h, int(variant)), "egpu_set_variant")

    # -- capacity table -----------------------------------------------------
    def set_table(self, free_core, free_mem):
        fc, fm = _i32(free_core), _i32(free_mem)
        if fc.shape != fm.shape or fc.ndim != 1:
            raise L.EgpuError(L.ERR_INVALID, "set_table")
        rc = self._lib.egpu_table_set(self._h, fc.ctypes.data_as(L.i32p), fm.ctypes.data_as(L.i32p), fc.size)
        self._check(rc, "egpu_table_set")

    def table(self):
        D = self._lib.egpu_table_size(self._h)
        if D < 0:
            raise L.EgpuError(D, "egpu_table_size")
        fc = np.empty(D, dtype=np.int32)
        fm = np.empty(D, dtype=np.int32)
        ov = np.empty(D, dtype=np.int32)
        rc = self._lib.egpu_table_get(self._h, fc.ctypes.data_as(L.i32p), fm.ctypes.data_as(L.i32p),
                                      ov.ctypes.data_as(L.i32p))
        self._check(rc, "egpu_table_get")
        return fc, fm, ov

    # -- snapshot mode, host buffers -----------------------------------------
    def bestfit(self, req_core, req_mem, commit: bool = False, out_idx: np.ndarray | None = None,
                prefix_commit: bool = False):
        """Returns (idx int32[R], delta_core int64[D], delta_mem int64[D]).  prefix_commit:
        spec 2.5 - requests beyond a device's capacity come back as -2 (DEFERRED)."""
        rc_, rm_ = _i32(req_core), _i32(req_mem)
        if rc_.shape != rm_.shape or rc_.ndim != 1:
            raise L.EgpuError(L.ERR_INVALID, "bestfit")
        D = self._lib.egpu_table_size(self._h)
        if D < 0:
            raise L.EgpuError(D, "egpu_table_size")
        R = rc_.size
        idx = out_idx if out_idx is not None else np.empty(R, dtype=np.int32)
        dc = np.zeros(D, dtype=np.int64)
        dm = np.zeros(D, dtype=np.int64)
        rc = self._lib.egpu_bestfit_batch(self._h, _ptr(rc_), _ptr(rm_), R, _ptr(idx), _ptr(dc), _ptr(dm),
                                          (L.F_COMMIT if commit else 0) | (L.F_PREFIX_COMMIT if prefix_commit else 0))
        self._check(rc, "egpu_bestfit_batch")
        return idx, dc, dm

    def bestfit_rounds(self, req_core, req_mem, max_rounds: int = 1 << 20):
        """egpu_bestfit_batch_rounds: committing prefix-commit rounds until nothing is deferred.
        Returns (idx, delta_core, delta_mem, rounds, still_deferred)."""
        rc_, rm_ = _i32(req_core), _i32(req_mem)
        if rc_.shape != rm_.shape or rc_.ndim != 1:
            raise L.EgpuError(L.ERR_INVALID, "bestfit_rounds")
        D = self._lib.egpu_table_size(self._h)
        if D < 0:
            raise L.EgpuError(D, "egpu_table_size")
        R = rc_.size
        idx = np.empty(R, dtype=np.int32)
        dc = np.zeros(D, dtype=np.int64)
        dm = np.zeros(D, dtype=np.int64)
        rounds, left = C.c_int32(0), C.c_int64(0)
        rc = self._lib.egpu_bestfit_batch_rounds(self._h, _ptr(rc_), _ptr(rm_), R, _ptr(idx), _ptr(dc), _ptr(dm),
                                                 int(max_rounds), C.byref(rounds), C.byref(left))
        self._check(rc, "egpu_bestfit_batch_rounds")
        return idx, dc, dm, int(rounds.value), int(left.value)

    def bestfit_rounds_dev(self, d_core: int, d_mem: int, R: int, d_idx: int, max_rounds: int = 1 << 20,
                           stream: int | None = None):
        """Device-array form; returns (delta int64[2*D], rounds, still_deferred)."""
        D = self._lib.egpu_table_size(self._h)
        if D < 0:
            raise L.EgpuError(D, "egpu_table_size")
        delta = np.zeros(2 * D, dtype=np.int64)
        rounds, left = C.c_int32(0), C.c_int64(0)
        rc = self._lib.egpu_bestfit_batch_rounds_dev(self._h, C.c_void_p(d_core), C.c_void_p(d_mem), int(R), C.c_void_p(d_idx),
                                                     _ptr(delta), int(max_rounds), C.byref(rounds), C.byref(left), _stream(stream))
        self._check(rc, "egpu_bestfit_batch_rounds_dev")
        return delta, int(rounds.value), int(left.value)

    def bestfit_raw(self, p_core: int, p_mem: int, R: int, p_idx: int, p_dc: int, p_dm: int, commit: bool = False):
        """Same call on raw host addresses (e.g. pinned buffers from host_alloc)."""
        rc = self._lib.egpu_bestfit_batch(self._h, C.c_void_p(p_core), C.c_void_p(p_mem), R, C.c_void_p(p_idx),
                                          C.c_void_p(p_dc), C.c_void_p(p_dm), 1 if commit else 0)
        self._check(rc, "egpu_bestfit_batch")

    # -- packed wire format ----------------------------------------------------
    @staticmethod
    def pack_requests(req_core, req_mem) -> np.ndarray:
        """EGPU_PACK_REQUEST over arrays; out-of-domain rows become EGPU_PACKED_INVALID."""
        c = np.asarray(req_core, dtype=np.int64)
        m = np.asarray(req_mem, dtype=np.int64)
        ok = (c >= 0) & (c <= 127) & (m >= 0) & (m < (1 << 18))
        return np.where(ok, (c << 18) | m, 0xFFFFFFFF).astype(np.uint32)

    def bestfit_packed(self, req_packed, commit: bool = False):
        """Returns (idx int8[R], delta_core int64[D], delta_mem int64[D])."""
        p = np.ascontiguousarray(req_packed, dtype=np.uint32)
        D = self._lib.egpu_table_size(self._h)
        if D < 0:
            raise L.EgpuError(D, "egpu_table_size")
        idx = np.empty(p.size, dtype=np.int8)
        dc = np.zeros(D, dtype=np.int64)
        dm = np.zeros(D, dtype=np.int64)
        rc = self._lib.egpu_bestfit_batch_packed(self._h, _ptr(p), p.size, _ptr(idx), _ptr(dc), _ptr(dm), 1 if commit else 0)
        self._check(rc, "egpu_bestfit_batch_packed")
        return idx, dc, dm

    def bestfit_packed_raw(self, p_req: int, R: int, p_idx8: int, p_dc: int, p_dm: int, commit: bool = False):
        rc = self._lib.egpu_bestfit_batch_packed(self._h, C.c_void_p(p_req), int(R), C.c_void_p(p_idx8), C.c_void_p(p_dc),
                                                 C.c_void_p(p_dm), 1 if commit else 0)
        self._check(rc, "egpu_bestfit_batch_packed")

    def bestfit_packed_dev(self, d_req: int, R: int, d_idx8: int, d_delta: int = 0, d_table_out: int = 0,
                           commit: bool = False, stream: int | None = None):
        """egpu_bestfit_batch_packed_dev: packed words and int8 indices in device memory (16-byte aligned);
        d_delta int64[2*D] and d_table_out int32[3*D] may be 0."""
        rc = self._lib.egpu_bestfit_batch_packed_dev(self._h, C.c_void_p(d_req), int(R), C.c_void_p(d_idx8),
                                                     C.c_void_p(d_delta or None), C.c_void_p(d_table_out or None),
                                                     L.F_COMMIT if commit else 0, _stream(stream))
        self._check(rc, "egpu_bestfit_batch_packed_dev")

    def host_alloc(self, nbytes: int) -> int:
        p = C.c_void_p()
        self._check(self._lib.egpu_host_alloc(self._h, C.byref(p), int(nbytes)), "egpu_host_alloc")
        return int(p.value)

    def host_free(self, addr: int):
        self._lib.egpu_host_free(self._h, C.c_void_p(addr))

    def host_register(self, arr: np.ndarray):
        """egpu_host_register on a caller-owned numpy array (stays pinned until host_unregister)."""
        self._check(self._lib.egpu_host_register(self._h, C.c_void_p(arr.ctypes.data), int(arr.nbytes)), "egpu_host_register")

    def host_unregister(self, arr: np.ndarray):
        self._check(self._lib.egpu_host_unregister(self._h, C.c_void_p(arr.ctypes.data)), "egpu_host_unregister")

    def pinned_array(self, n: int, dtype=np.int32) -> np.ndarray:
        """numpy view over pinned host memory owned by the context (freed with it
        only if the caller calls host_free(arr.ctypes.data))."""
        dt = np.dtype(dtype)
        addr = self.host_alloc(max(1, n) * dt.itemsize)
        buf = (C.c_char * (max(1, n) * dt.itemsize)).from_address(addr)
        return np.frombuffer(buf, dtype=dt, count=n)

    # -- whole-card requests (core = 100 * k asks for k whole cards) -------------
    def bestfit_cards(self, req_core, req_mem, commit: bool = False, cards: bool = True):
        """egpu_bestfit_cards.  Returns (idx int32[R], cards uint64[R] or None, delta_core int64[D],
        delta_mem int64[D]); cards=False asks for no masks."""
        rc_, rm_ = _i32(req_core), _i32(req_mem)
        if rc_.shape != rm_.shape or rc_.ndim != 1:
            raise L.EgpuError(L.ERR_INVALID, "bestfit_cards")
        D = self._lib.egpu_table_size(self._h)
        if D < 0:
            raise L.EgpuError(D, "egpu_table_size")
        R = rc_.size
        idx = np.empty(R, dtype=np.int32)
        masks = np.empty(R, dtype=np.uint64) if cards else None
        dc = np.zeros(D, dtype=np.int64)
        dm = np.zeros(D, dtype=np.int64)
        rc = self._lib.egpu_bestfit_cards(self._h, _ptr(rc_), _ptr(rm_), R, _ptr(idx),
                                          _ptr(masks) if cards else C.c_void_p(None), _ptr(dc), _ptr(dm),
                                          L.F_COMMIT if commit else 0)
        self._check(rc, "egpu_bestfit_cards")
        return idx, masks, dc, dm

    def bestfit_cards_dev(self, d_core: int, d_mem: int, R: int, d_idx: int, d_cards: int = 0, d_delta: int = 0,
                          d_table_out: int = 0, commit: bool = False, stream: int | None = None, inputs_ready: bool = False):
        """egpu_bestfit_cards_dev: device arrays (16-byte aligned); d_cards uint64[R], d_delta int64[2*D] and
        d_table_out int32[3*D] may be 0."""
        flags = (L.F_COMMIT if commit else 0) | (L.F_INPUTS_READY if inputs_ready else 0)
        rc = self._lib.egpu_bestfit_cards_dev(self._h, C.c_void_p(d_core), C.c_void_p(d_mem), int(R), C.c_void_p(d_idx),
                                              C.c_void_p(d_cards or None), C.c_void_p(d_delta or None),
                                              C.c_void_p(d_table_out or None), flags, _stream(stream))
        self._check(rc, "egpu_bestfit_cards_dev")

    # -- snapshot mode, device buffers ---------------------------------------
    def bestfit_dev(self, d_core: int, d_mem: int, R: int, d_idx: int, d_delta: int = 0, d_table_out: int = 0,
                    commit: bool = False, stream: int | None = None, inputs_ready: bool = False, prefix_commit: bool = False):
        flags = (L.F_COMMIT if commit else 0) | (L.F_INPUTS_READY if inputs_ready else 0) | \
                (L.F_PREFIX_COMMIT if prefix_commit else 0)
        rc = self._lib.egpu_bestfit_batch_dev(self._h, C.c_void_p(d_core), C.c_void_p(d_mem), int(R),
                                              C.c_void_p(d_idx), C.c_void_p(d_delta or None),
                                              C.c_void_p(d_table_out or None), flags,
                                              _stream(stream))
        self._check(rc, "egpu_bestfit_batch_dev")

    @staticmethod
    def make_batches(batches):
        """(d_core, d_mem, R, d_idx, d_delta, d_table_out) tuples -> the egpu_batch array of the C ABI
        (build it once and pass it to bestfit_batches_dev / bestfit_batches_shard_dev)."""
        arr = (L.Batch * len(batches))()
        for k, (c, m, R, i, dl, to) in enumerate(batches):
            arr[k] = L.Batch(c or None, m or None, int(R), i or None, dl or None, to or None)
        return arr

    def bestfit_batches_dev(self, batches, stream: int | None = None, inputs_ready: bool = False):
        """egpu_bestfit_batches_dev: up to 64 batches scored against the current table in one launch."""
        arr = batches if isinstance(batches, C.Array) else self.make_batches(batches)
        rc = self._lib.egpu_bestfit_batches_dev(self._h, arr, len(arr), L.F_INPUTS_READY if inputs_ready else 0, _stream(stream))
        self._check(rc, "egpu_bestfit_batches_dev")

    def bestfit_batches_shard_dev(self, batches, first_step: int, stream: int | None = None, inputs_ready: bool = False,
                                  apply: bool = False):
        """K sharded steps in one launch: batch k = exchange step first_step + k.  apply: the CTAs that complete a
        batch's sums also apply that step (EGPU_F_APPLY) - table' lands in the batch's d_table_out, no apply call."""
        arr = batches if isinstance(batches, C.Array) else self.make_batches(batches)
        rc = self._lib.egpu_bestfit_batches_shard_dev(self._h, arr, len(arr),
                                                      (L.F_INPUTS_READY if inputs_ready else 0) | (L.F_APPLY if apply else 0),
                                                      int(first_step), _stream(stream))
        self._check(rc, "egpu_bestfit_batches_shard_dev")

    def query(self, free_core, free_mem, req_core, req_mem) -> np.ndarray:
        """egpu_bestfit_query: score against the table given here; the context's own table is untouched."""
        fc, fm, rc_, rm_ = _i32(free_core), _i32(free_mem), _i32(req_core), _i32(req_mem)
        if fc.shape != fm.shape or fc.ndim != 1 or rc_.shape != rm_.shape or rc_.ndim != 1:
            raise L.EgpuError(L.ERR_INVALID, "query")
        idx = np.empty(rc_.size, dtype=np.int32)
        rc = self._lib.egpu_bestfit_query(self._h, fc.ctypes.data_as(L.i32p), fm.ctypes.data_as(L.i32p), fc.size,
                                          _ptr(rc_), _ptr(rm_), rc_.size, _ptr(idx))
        self._check(rc, "egpu_bestfit_query")
        return idx

    def gate_dev(self, stream: int | None = None):
        self._check(self._lib.egpu_peer_gate_dev(self._h, _stream(stream)), "egpu_peer_gate_dev")

    def gate_open(self):
        self._check(self._lib.egpu_peer_gate_open(self._h), "egpu_peer_gate_open")

    @property
    def gate_timeouts(self) -> int:
        return int(self._lib.egpu_peer_gate_timeouts(self._h))

    def apply_deltas_dev(self, d_deltas: int, G: int, d_table_out: int = 0, commit: bool = True, stream: int | None = None):
        rc = self._lib.egpu_table_apply_deltas_dev(self._h, C.c_void_p(d_deltas), int(G),
                                                   C.c_void_p(d_table_out or None), 1 if commit else 0,
                                                   _stream(stream))
        self._check(rc, "egpu_table_apply_deltas_dev")

    def synth_requests_dev(self, dist: int, seed: int, first_row: int, R: int, d_core: int, d_mem: int,
                           stream: int | None = None):
        rc = self._lib.egpu_synth_requests_dev(self._h, int(dist), int(seed), int(first_row), int(R),
                                               C.c_void_p(d_core), C.c_void_p(d_mem), _stream(stream))
        self._check(rc, "egpu_synth_requests_dev")

    # -- multi-GPU: peer-memory exchange ----------------------------------------
    def peer_export(self) -> bytes:
        buf = C.create_string_buffer(64)
        self._check(self._lib.egpu_peer_export(self._h, buf), "egpu_peer_export")
        return buf.raw

    def peer_attach(self, rank: int, world: int, handles: list[bytes]):
        blob = b"".join(handles)
        if len(blob) != 64 * world:
            raise L.EgpuError(L.ERR_INVALID, "peer_attach")
        self._check(self._lib.egpu_peer_attach(self._h, int(rank), int(world), C.c_char_p(blob)), "egpu_peer_attach")

    def peer_detach(self):
        self._check(self._lib.egpu_peer_detach(self._h), "egpu_peer_detach")

    def bestfit_shard_dev(self, d_core: int, d_mem: int, R: int, d_idx: int, d_delta: int, step: int, stream: int | None = None,
                          inputs_ready: bool = False):
        rc = self._lib.egpu_bestfit_batch_shard_dev(self._h, C.c_void_p(d_core), C.c_void_p(d_mem), int(R),
                                                    C.c_void_p(d_idx), C.c_void_p(d_delta or None),
                                                    L.F_INPUTS_READY if inputs_ready else 0, int(step),
                                                    _stream(stream))
        self._check(rc, "egpu_bestfit_batch_shard_dev")

    def bestfit_shard_prefix_dev(self, d_core: int, d_mem: int, R: int, d_idx: int, d_delta: int, d_table_out: int, step: int,
                                 commit: bool = False, stream: int | None = None):
        """Prefix-commit over row shards (rank-major order); consumes exchange steps `step` and `step + 1`."""
        rc = self._lib.egpu_bestfit_batch_shard_prefix_dev(self._h, C.c_void_p(d_core), C.c_void_p(d_mem), int(R),
                                                           C.c_void_p(d_idx), C.c_void_p(d_delta or None),
                                                           C.c_void_p(d_table_out or None),
                                                           L.F_PREFIX_COMMIT | (L.F_COMMIT if commit else 0), int(step),
                                                           _stream(stream))
        self._check(rc, "egpu_bestfit_batch_shard_prefix_dev")

    def bestfit_shard_lag_dev(self, d_core: int, d_mem: int, R: int, d_idx: int, d_delta: int, step: int, lag: int,
                              d_table_out_lagged: int = 0, stream: int | None = None, inputs_ready: bool = False):
        rc = self._lib.egpu_bestfit_batch_shard_lag_dev(self._h, C.c_void_p(d_core), C.c_void_p(d_mem), int(R),
                                                        C.c_void_p(d_idx), C.c_void_p(d_delta or None),
                                                        L.F_INPUTS_READY if inputs_ready else 0, int(step), int(lag),
                                                        C.c_void_p(d_table_out_lagged or None), _stream(stream))
        self._check(rc, "egpu_bestfit_batch_shard_lag_dev")

    def apply_peers_dev(self, step: int, d_table_out: int = 0, commit: bool = False, stream: int | None = None):
        rc = self._lib.egpu_table_apply_peers_dev(self._h, int(step), C.c_void_p(d_table_out or None),
                                                  1 if commit else 0, _stream(stream))
        self._check(rc, "egpu_table_apply_peers_dev")

    def apply_peers_multi_dev(self, first_step: int, d_table_outs: list[int], commit: bool = False, stream: int | None = None):
        n = len(d_table_outs)
        arr = (C.c_void_p * n)(*[C.c_void_p(p or None) for p in d_table_outs])
        rc = self._lib.egpu_table_apply_peers_multi_dev(self._h, int(first_step), n, arr, 1 if commit else 0,
                                                        _stream(stream))
        self._check(rc, "egpu_table_apply_peers_multi_dev")

    @property
    def peer_last_timeout(self) -> int:
        return int(self._lib.egpu_peer_last_timeout(self._h))

    # -- sequential mode ------------------------------------------------------
    def replay(self, kind, a, b):
        k, a_, b_ = _i32(kind), _i32(a), _i32(b)
        if not (k.shape == a_.shape == b_.shape) or k.ndim != 1:
            raise L.EgpuError(L.ERR_INVALID, "replay")
        out = np.empty(k.size, dtype=np.int32)
        rc = self._lib.egpu_replay(self._h, _ptr(k), _ptr(a_), _ptr(b_), k.size, _ptr(out))
        self._check(rc, "egpu_replay")
        return out

    def replay_cards(self, kind, a, b, cards: bool = True):
        """egpu_replay_cards: replay with whole-card ALLOCs.  Returns (idx int32[E], cards uint64[E] or None)."""
        k, a_, b_ = _i32(kind), _i32(a), _i32(b)
        if not (k.shape == a_.shape == b_.shape) or k.ndim != 1:
            raise L.EgpuError(L.ERR_INVALID, "replay_cards")
        out = np.empty(k.size, dtype=np.int32)
        masks = np.empty(k.size, dtype=np.uint64) if cards else None
        rc = self._lib.egpu_replay_cards(self._h, _ptr(k), _ptr(a_), _ptr(b_), k.size, _ptr(out),
                                         _ptr(masks) if cards else C.c_void_p(None))
        self._check(rc, "egpu_replay_cards")
        return out, masks
