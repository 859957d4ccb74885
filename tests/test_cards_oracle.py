"""CPU tests (no GPU) of whole-card requests (DESIGN.md 2.8): the hand-derived known answers in
both oracles, the two oracles against each other on edge and random tables, the run property the
CUDA scan relies on (by brute force), agreement with the single-card oracles when no row asks
for more than one card, and argument checks of the new entry points that need no device."""
import itertools
import json
import os

import numpy as np
import pytest

import edge_cases as ec
from oracle import cards_c, cards_np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KAT = json.load(open(os.path.join(ROOT, "tests", "golden", "bestfit_cards_kat.json")))


def full_cards_table(D: int, seed: int = 0):
    """'many full cards': most rows (100, m) with few distinct m, so whole-card requests have
    ties, runs that end exactly at D, and runs one card too long"""
    rng = np.random.default_rng([D, seed, 7])
    fc = np.where(rng.random(D) < 0.8, 100, rng.integers(0, 100, D)).astype(np.int32)
    fm = rng.choice([0, 1, 4096, 4097, ec.MEM_MAX], D).astype(np.int32)
    return fc, fm


def card_requests(fc, fm, n_random: int, rng):
    """k = 1 .. D + 1 (and 64, 65) at every memory threshold of the table, non-multiples of 100,
    int32 extremes, plus random rows"""
    D = fc.size
    ks = sorted(set(range(1, D + 2)) | {64, 65})
    mems = sorted(set(np.unique(fm).tolist()) | {int(m) + 1 for m in np.unique(fm)} | {0})
    cores, rmem = [], []
    for k in ks:
        for m in mems:
            cores.append(100 * k)
            rmem.append(m)
    for c in (101, 150, 199, 201, 250, 6401, 6499, 6500, 6600, ec.I32_MAX, ec.I32_MIN, -100, -200):
        cores += [c, c]
        rmem += [0, int(fm.min())]
    for m in ec.BAD_MEMS:
        cores += [200, 100]
        rmem += [m, m]
    rc, rm = ec.random_requests(rng, n_random)
    whole = rng.random(n_random) < 0.3
    rc[whole] = 100 * rng.integers(2, D + 2, int(whole.sum()))
    return (np.concatenate([np.array(cores, np.int64).astype(np.int32), rc]),
            np.concatenate([np.array(rmem, np.int64).astype(np.int32), rm]))


def tables():
    for D in ec.D_VALUES:
        for fam in ec.TABLE_FAMILIES:
            t = ec.make_table(fam, D)
            yield f"{fam}-{D}", t.fc, t.fm
        fc, fm = full_cards_table(D)
        yield f"full_cards-{D}", fc, fm


# ---- known answers ---------------------------------------------------------------------------

@pytest.mark.parametrize("case", KAT["snapshot"], ids=lambda c: c["name"])
def test_snapshot_kat_both_oracles(case):
    for fn in (cards_c.bestfit_cards_snapshot, cards_np.cards_snapshot):
        idx, cards, dc, dm, tab = fn(case["free_core"], case["free_mem"], case["req_core"], case["req_mem"])
        assert idx.tolist() == case["idx"] and cards.tolist() == case["cards"]
        assert dc.tolist() == case["delta_core"] and dm.tolist() == case["delta_mem"]
        assert tab.tolist() == case["table_out"]


@pytest.mark.parametrize("case", KAT["sequential"], ids=lambda c: c["name"])
def test_sequential_kat_both_oracles(case):
    for fn in (cards_c.replay_cards, cards_np.replay_cards):
        idx, cards, fc, fm = fn(case["free_core"], case["free_mem"], case["kind"], case["a"], case["b"])
        assert idx.tolist() == case["idx"] and cards.tolist() == case["cards"]
        assert fc.tolist() == case["free_core_after"] and fm.tolist() == case["free_mem_after"]


# ---- the two oracles agree -------------------------------------------------------------------

@pytest.mark.parametrize("name,fc,fm", list(tables()), ids=lambda x: x if isinstance(x, str) else "")
def test_oracles_agree_on_edge_tables(name, fc, fm):
    rng = np.random.default_rng(abs(hash(name)) % (1 << 32))
    rc, rm = card_requests(fc, fm, 600, rng)
    a = cards_c.bestfit_cards_snapshot(fc, fm, rc, rm)
    b = cards_np.cards_snapshot(fc, fm, rc, rm)
    for x, y in zip(a, b):
        assert np.array_equal(x, y), name


@pytest.mark.parametrize("D", [1, 2, 8, 9, 33, 64])
def test_oracles_agree_on_churn(D, egpu):
    kind, a, b = egpu.synth.churn_events(5, 3000)
    rng = np.random.default_rng(D)
    whole = (kind == 0) & (rng.random(kind.size) < 0.1)
    a = a.copy()
    a[whole] = 100 * rng.integers(2, max(3, D // 2 + 2), int(whole.sum()))
    fc, fm = np.full(D, 100, np.int32), np.full(D, 40000, np.int32)
    x = cards_c.replay_cards(fc, fm, kind, a, b)
    y = cards_np.replay_cards(fc, fm, kind, a, b)
    for u, v in zip(x, y):
        assert np.array_equal(u, v)
    assert (x[1][kind == 0] != 0).sum() > 0
    assert D <= 2 or np.any([bin(int(c)).count("1") > 1 for c in x[1]]), "no whole-card ALLOC was placed"


# ---- the run property the CUDA scan uses -------------------------------------------------------

def test_run_property_by_brute_force():
    """The k best whole cards are sorted positions [p, p + k) with p the first feasible position
    for (100, mem), feasible iff p + k <= D; and they are the k-subset of feasible cards whose
    sorted keys are lexicographically smallest (brute force over subsets for D <= 7)."""
    rng = np.random.default_rng(20_000)
    checked = 0
    for trial in range(20_000):
        D = int(rng.integers(1, 65)) if trial % 4 else int(rng.integers(1, 8))
        fc = rng.choice([100, 100, 100, 99, 0, int(rng.integers(0, 101))], D).astype(np.int32)
        fm = rng.choice([0, 1, 2, 300, 301, int(rng.integers(0, 1 << 18))], D).astype(np.int32)
        k = int(rng.integers(2, D + 2))
        mem = int(rng.choice([0, 1, 2, 300, 301, 302]))
        idx, cards, *_ = cards_c.bestfit_cards_snapshot(fc, fm, [100 * k], [mem])
        rows = ec.sorted_rows(fc, fm)
        p = next((j for j, (c, m, _) in enumerate(rows) if c >= 100 and m >= mem), D)
        run = [d for _, _, d in rows[p:p + k]]
        if p + k <= D:
            assert idx[0] == run[0] and int(cards[0]) == sum(1 << d for d in run)
        else:
            assert idx[0] == -1 and cards[0] == 0
        if D <= 7:
            feas = [d for d in range(D) if fc[d] >= 100 and fm[d] >= mem]
            key = {d: (int(fc[d]) - 100, int(fm[d]) - mem, d) for d in feas}
            best = min((sorted(key[d] for d in s) for s in itertools.combinations(feas, k)), default=None)
            if best is None:
                assert idx[0] == -1
            else:
                assert int(cards[0]) == sum(1 << t[2] for t in best) and idx[0] == best[0][2]
        checked += 1
    assert checked == 20_000


# ---- single-card batches: exactly the existing oracles ---------------------------------------------

@pytest.mark.parametrize("name,fc,fm", list(tables())[::3], ids=lambda x: x if isinstance(x, str) else "")
def test_single_card_batches_equal_the_existing_oracles(name, fc, fm, oracle_c):
    rc, rm = ec.edge_requests(ec.EdgeTable("x", fc, fm, {}), 1027)
    rc = np.where(rc > 100, -1, rc).astype(np.int32)  # no row asks for more than one card
    idx, cards, dc, dm, tab = cards_c.bestfit_cards_snapshot(fc, fm, rc, rm)
    e_idx, e_dc, e_dm, e_tab = oracle_c.snapshot(fc, fm, rc, rm)
    assert np.array_equal(idx, e_idx) and np.array_equal(dc, e_dc) and np.array_equal(dm, e_dm) and np.array_equal(tab, e_tab)
    assert np.array_equal(cards, np.where(idx >= 0, np.left_shift(1, idx.astype(np.uint64) % 64).astype(np.uint64), 0))
    n_idx, _, n_dc, n_dm, _ = cards_np.cards_snapshot(fc, fm, rc, rm)
    assert np.array_equal(n_idx, e_idx) and np.array_equal(n_dc, e_dc) and np.array_equal(n_dm, e_dm)


def test_single_card_replay_equals_the_existing_oracle(oracle_c, egpu):
    kind, a, b = egpu.synth.churn_events(5, 5000)
    fc, fm = egpu.synth.table_full(8)
    idx, cards, cfc, cfm = cards_c.replay_cards(fc, fm, kind, a, b)
    e_idx, efc, efm = oracle_c.replay(fc, fm, kind, a, b)
    assert np.array_equal(idx, e_idx) and np.array_equal(cfc, efc) and np.array_equal(cfm, efm)
    assert np.array_equal(cards != 0, idx >= 0)


# ---- the C ABI without a device ------------------------------------------------------------------

def test_new_entry_points_reject_bad_arguments_without_a_device(egpu):
    import ctypes as C
    from elastic_gpu_agent_b200 import _lib as L
    lib = egpu.load()
    assert lib.egpu_abi_version() == 1005
    assert lib.egpu_bestfit_cards(None, None, None, 0, None, None, None, None, 0) == L.ERR_INVALID
    assert lib.egpu_bestfit_cards_dev(None, None, None, 0, None, None, None, None, 0, None) == L.ERR_INVALID
    assert lib.egpu_replay_cards(None, None, None, None, 0, None, None) == L.ERR_INVALID
    # a bogus (never dereferenced) context: argument checks come before the context is used
    bogus = C.c_void_p(16)
    assert lib.egpu_bestfit_cards_dev(bogus, None, None, -1, None, None, None, None, 0, None) == L.ERR_INVALID
    assert lib.egpu_bestfit_cards_dev(bogus, None, None, 1 << 31, None, None, None, None, 0, None) == L.ERR_INVALID
    assert lib.egpu_bestfit_cards_dev(bogus, None, None, 0, None, None, None, None, L.F_PREFIX_COMMIT, None) == L.ERR_INVALID
    assert lib.egpu_bestfit_cards_dev(bogus, None, None, 0, None, None, None, None, 64, None) == L.ERR_INVALID
    assert lib.egpu_bestfit_cards_dev(bogus, None, None, 4, None, None, None, None, 0, None) == L.ERR_INVALID
    assert lib.egpu_bestfit_cards_dev(bogus, C.c_void_p(16), C.c_void_p(16), 4, C.c_void_p(16), C.c_void_p(24), None, None, 0,
                                      None) == L.ERR_INVALID
    assert lib.egpu_bestfit_cards_dev(bogus, C.c_void_p(16), C.c_void_p(16), 4, C.c_void_p(16), None, C.c_void_p(8), None, 0,
                                      None) == L.ERR_INVALID
    assert lib.egpu_bestfit_cards_dev(bogus, C.c_void_p(16), C.c_void_p(20), 4, C.c_void_p(16), None, None, None, 0,
                                      None) == L.ERR_INVALID
    assert lib.egpu_bestfit_cards(bogus, None, None, 1 << 31, None, None, None, None, 0) == L.ERR_INVALID
    assert lib.egpu_bestfit_cards(bogus, None, None, 0, None, None, None, None, L.F_PREFIX_COMMIT) == L.ERR_INVALID
    assert lib.egpu_bestfit_cards(bogus, None, None, 3, None, None, None, None, 0) == L.ERR_INVALID
    assert lib.egpu_replay_cards(bogus, None, None, None, -1, None, None) == L.ERR_INVALID
    assert lib.egpu_replay_cards(bogus, None, None, None, 5, None, None) == L.ERR_INVALID
    assert lib.egpu_replay_cards(bogus, None, None, None, 1 << 31, None, None) == L.ERR_INVALID
