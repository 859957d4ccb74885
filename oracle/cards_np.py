"""oracle/cards_np.py — numpy restatement of whole-card requests (DESIGN.md §2.8).

TEST INFRASTRUCTURE ONLY, like oracle/bestfit_np.py, whose domain checks and table' it reuses.
Written a different way from oracle/cards_oracle.c: a row gets the k feasible devices with the
smallest packed keys of Appendix A.3 (one sort per row), not k sequential picks; neither uses
the run property the CUDA scan relies on.
"""
from __future__ import annotations

import numpy as np

from .bestfit_np import CORE_MAX, INT32_MAX, MAX_DEVICES, apply_delta, table_valid


def cards_k(req_core):
    """Spec §2.8: (k, per-card core) per request.  k = 1 for core <= 100 (spec §2.3 unchanged),
    k = core / 100 for core = 100*k with 2 <= k <= 64, k = 0 (infeasible) for any other core."""
    c = np.asarray(req_core, dtype=np.int64)
    whole = (c > CORE_MAX) & (c % 100 == 0) & (c // 100 <= MAX_DEVICES)
    k = np.where(c <= CORE_MAX, 1, np.where(whole, c // 100, 0))
    return k, np.where(whole, CORE_MAX, c)


def pick_cards_grid(free_core, free_mem, req_core, req_mem):
    """Spec §2.8 by the packed-key order: a row gets the k feasible devices with the smallest
    keys (lc, lm, d) of Appendix A.3, or nothing when fewer than k are feasible.  Returns
    (idx = the smallest key's device or -1, cards uint64 mask, take bool[R, D] by device)."""
    fc = np.asarray(free_core, dtype=np.int64)[None, :]
    fm = np.asarray(free_mem, dtype=np.int64)[None, :]
    k, per = cards_k(req_core)
    rc = per[:, None]
    rm = np.asarray(req_mem, dtype=np.int64)[:, None]
    D = fc.shape[1]
    R = rc.shape[0]
    d = np.arange(D, dtype=np.int64)[None, :]
    lc = fc - rc
    lm = fm - rm
    feasible = (rc >= 0) & (rm >= 0) & (lc >= 0) & (lm >= 0)
    key = np.sort(np.where(feasible, (lc << 24) | (lm << 6) | d, INT32_MAX), axis=1)
    kth = np.take_along_axis(key, np.clip(k - 1, 0, D - 1)[:, None], axis=1)[:, 0]
    ok = (k >= 1) & (k <= D) & (kth != INT32_MAX)
    taken_sorted = (np.arange(D)[None, :] < k[:, None]) & ok[:, None]
    devs = key & 63
    take = np.zeros((R, D), dtype=bool)
    rows = np.broadcast_to(np.arange(R)[:, None], (R, D))
    take[rows[taken_sorted], devs[taken_sorted]] = True
    cards = (take.astype(np.uint64) << np.arange(D, dtype=np.uint64)[None, :]).sum(axis=1, dtype=np.uint64)
    idx = np.where(ok, devs[:, 0] if D else -1, -1).astype(np.int32)
    return idx, cards, take


def cards_snapshot(free_core, free_mem, req_core, req_mem, chunk: int = 1 << 15):
    """Spec §2.4 extended by §2.8.  Returns (idx int32[R], cards uint64[R], delta_core int64[D],
    delta_mem int64[D], table_out int32[3*D])."""
    assert table_valid(free_core, free_mem)
    fc = np.asarray(free_core, dtype=np.int64)
    fm = np.asarray(free_mem, dtype=np.int64)
    rc = np.asarray(req_core, dtype=np.int32)
    rm = np.asarray(req_mem, dtype=np.int32)
    D = fc.size
    R = rc.size
    idx = np.empty(R, dtype=np.int32)
    cards = np.empty(R, dtype=np.uint64)
    dc = np.zeros(D, dtype=np.int64)
    dm = np.zeros(D, dtype=np.int64)
    for s in range(0, R, chunk):
        i, c, take = pick_cards_grid(fc, fm, rc[s:s + chunk], rm[s:s + chunk])
        idx[s:s + chunk] = i
        cards[s:s + chunk] = c
        _, per = cards_k(rc[s:s + chunk])
        dc += (take * per[:, None]).sum(axis=0)
        dm += (take * rm[s:s + chunk].astype(np.int64)[:, None]).sum(axis=0)
    return idx, cards, dc, dm, apply_delta(fc, fm, dc, dm)


def replay_cards(free_core, free_mem, kind, a, b):
    """Spec §2.6 extended by §2.8, pure-Python loop (small cases only).  Returns
    (idx int32[E], cards uint64[E], free_core', free_mem')."""
    assert table_valid(free_core, free_mem)
    fc = [int(x) for x in free_core]
    fm = [int(x) for x in free_mem]
    D = len(fc)
    E = len(kind)
    out = np.full(E, -1, dtype=np.int32)
    cards = np.zeros(E, dtype=np.uint64)
    live = {}  # ALLOC event -> (devices, per-card core, mem)
    for i in range(E):
        if int(kind[i]) == 0:
            c, m = int(a[i]), int(b[i])
            (k,), (per,) = cards_k([c])
            keys = sorted((fc[d] - per, fm[d] - m, d) for d in range(D)
                          if per >= 0 and m >= 0 and fc[d] >= per and fm[d] >= m)
            if 1 <= k <= len(keys):
                devs = [key[2] for key in keys[:int(k)]]
                for d in devs:
                    fc[d] -= int(per)
                    fm[d] -= m
                live[i] = (devs, int(per), m)
                out[i] = devs[0]
                cards[i] = sum(1 << d for d in devs)
        else:
            t = int(a[i])
            if int(kind[i]) == 1 and 0 <= t < i and t in live:
                devs, per, m = live.pop(t)
                for d in devs:
                    fc[d] += per
                    fm[d] += m
                out[i] = devs[0]
                cards[i] = sum(1 << d for d in devs)
    return out, cards, np.array(fc, dtype=np.int32), np.array(fm, dtype=np.int32)
