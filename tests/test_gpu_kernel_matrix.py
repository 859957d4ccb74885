"""Every scan kernel against the oracle, on every output, at the inputs where integer bit tricks fail.

The library has 23 scan instantiations (five register-scan forms for each of the four D buckets,
and three lookup-table scans) behind eight entry points.  Here each of them is compared with
oracle_c on the indices, both demand sums, all 3 D words of table', the committed table and the
sticky oversubscription flags:

  * the matrix: D x table family (tests/edge_cases.py) x entry point, every kernel variant a path has;
  * the epilogue outputs: saturated table' in memory and in core, and oversubscription in one
    dimension only, on every launch form that writes table';
  * two full turns of both epilogue-slot rings with changing flag patterns;
  * the row limit EGPU_MAX_ROWS (2^31 - 1) at full size, and its rejection one row above;
  * kernel coverage: every scan instantiation is seen launching under torch.profiler.
"""
import functools
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import edge_cases as E  # noqa: E402

pytestmark = pytest.mark.gpu

GRID, SORTED, LUT = 1, 2, 3
ENTRY_POINTS = ("host", "dev_lone", "dev_ready", "batches", "packed", "query", "prefix", "rounds", "chain")


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def _stream(torch):
    return torch.cuda.current_stream().cuda_stream


def _dev(torch, a):
    """device copy of a host array (an empty array gets a 4-element buffer: a valid pointer)"""
    a = np.ascontiguousarray(a)
    if a.size == 0:
        return torch.empty(4, dtype=torch.int32, device="cuda")
    return torch.from_numpy(a).cuda()


def _eq(got, exp, what):
    got, exp = np.asarray(got), np.asarray(exp)
    assert got.shape == exp.shape, f"{what}: shape {got.shape} != {exp.shape}"
    bad = np.flatnonzero(got != exp)
    assert bad.size == 0, f"{what}: {bad.size} mismatches, first at {bad[:4].tolist()}: {got[bad[:4]].tolist()} != {exp[bad[:4]].tolist()}"


def committed(tab, D):
    """what a commit installs: table' with negative leftovers clamped to 0"""
    return np.maximum(tab[:D], 0), np.maximum(tab[D:2 * D], 0), tab[2 * D:]


@functools.lru_cache(maxsize=None)
def _case(family, D, R, seed=0):
    """table, edge requests and the oracle's snapshot answer"""
    from oracle import oracle_c
    t = E.make_table(family, D)
    E.check_claims(t)
    rc, rm = E.edge_requests(t, R, seed)
    return t, rc, rm, oracle_c.snapshot(t.fc, t.fm, rc, rm, 4)


def _check_snapshot(what, D, got, exp, table_out=True):
    idx, delta, tab = got
    o_idx, o_dc, o_dm, o_tab = exp
    _eq(idx, o_idx, f"{what}: idx")
    if delta is not None:
        _eq(delta, np.concatenate([o_dc, o_dm]), f"{what}: delta")
    if table_out:
        _eq(tab, o_tab, f"{what}: table'")


# ---------------------------------------------------------------------------------------------
# The matrix
# ---------------------------------------------------------------------------------------------

def _host(alloc, D):
    for family in E.TABLE_FAMILIES:
        for variant in (GRID, SORTED, LUT):
            alloc.set_variant(variant)
            for R in E.SIZES:
                t, rc, rm, exp = _case(family, D, R)
                alloc.set_table(t.fc, t.fm)
                idx, dc, dm = alloc.bestfit(rc, rm)
                _check_snapshot((family, variant, R), D, (idx, np.concatenate([dc, dm]), None), exp, table_out=False)
            fc, fm, ov = alloc.table()
            _eq(fc, t.fc, "table untouched")
            _eq(fm, t.fm, "table untouched")
            assert not ov.any()


def _dev_single(alloc, D, torch, ready):
    s = _stream(torch)
    for family in E.TABLE_FAMILIES:
        t = _case(family, D, 1)[0]
        for variant in (GRID, SORTED, LUT):
            alloc.set_variant(variant)
            alloc.set_table(t.fc, t.fm)
            runs = []
            for R in E.SIZES:
                _, rc, rm, exp = _case(family, D, R)
                runs.append((R, exp, _dev(torch, rc), _dev(torch, rm), torch.full((R + 4,), -9, dtype=torch.int32, device="cuda"),
                             torch.full((2 * D,), -1, dtype=torch.int64, device="cuda"),
                             torch.full((3 * D,), -7, dtype=torch.int32, device="cuda")))
            torch.cuda.synchronize()  # inputs complete: with inputs_ready the launches below may overlap
            for R, exp, c, m, idx, delta, tab in runs:
                alloc.bestfit_dev(c.data_ptr(), m.data_ptr(), R, idx.data_ptr(), delta.data_ptr(), tab.data_ptr(), False, s,
                                  inputs_ready=ready)
                if not ready:
                    torch.cuda.synchronize()
            torch.cuda.synchronize()
            for R, exp, c, m, idx, delta, tab in runs:
                got = idx.cpu().numpy()
                assert (got[R:] == -9).all(), "wrote past R"
                _check_snapshot((family, variant, R, ready), D, (got[:R], delta.cpu().numpy(), tab.cpu().numpy()), exp)


def _batches(alloc, D, torch):
    """K = 5 ragged batches in one launch, one of them empty and one with a single row"""
    s = _stream(torch)
    rows = (70_001, 0, 1, 1027, 5)
    for family in E.TABLE_FAMILIES:
        t = _case(family, D, 1)[0]
        for variant in (SORTED, LUT):
            alloc.set_variant(variant)
            alloc.set_table(t.fc, t.fm)
            keep, tup = [], []
            for k, R in enumerate(rows):
                rc, rm = _case(family, D, R, seed=k)[1:3] if R else (np.zeros(0, np.int32), np.zeros(0, np.int32))
                c, m = _dev(torch, rc), _dev(torch, rm)
                idx = torch.full((R + 4,), -9, dtype=torch.int32, device="cuda")
                delta = torch.full((2 * D,), -1, dtype=torch.int64, device="cuda")
                tab = torch.full((3 * D,), -7, dtype=torch.int32, device="cuda")
                keep.append((R, rc, rm, c, m, idx, delta, tab))
                tup.append((c.data_ptr(), m.data_ptr(), R, idx.data_ptr(), delta.data_ptr(), tab.data_ptr()))
            torch.cuda.synchronize()
            alloc.bestfit_batches_dev(tup, s)
            torch.cuda.synchronize()
            from oracle import oracle_c
            for k, (R, rc, rm, c, m, idx, delta, tab) in enumerate(keep):
                exp = oracle_c.snapshot(t.fc, t.fm, rc, rm, 4)
                got = idx.cpu().numpy()
                assert (got[R:] == -9).all(), "wrote past R"
                _check_snapshot((family, variant, "batch", k, R), D, (got[:R], delta.cpu().numpy(), tab.cpu().numpy()), exp)
            fc, fm, ov = alloc.table()
            _eq(fc, t.fc, "a multi-batch launch never commits")
            _eq(fm, t.fm, "a multi-batch launch never commits")


def _packed(alloc, D, torch, egpu, oracle_c):
    s = _stream(torch)
    rng = np.random.default_rng(D)
    for family in E.TABLE_FAMILIES:
        t = _case(family, D, 1)[0]
        alloc.set_table(t.fc, t.fm)
        for R in E.SIZES:
            _, rc, rm, exp = _case(family, D, R)
            idx, dc, dm = alloc.bestfit_packed(egpu.BestFitAllocator.pack_requests(rc, rm))
            _check_snapshot((family, "packed", R), D, (idx.astype(np.int32), np.concatenate([dc, dm]), None), exp, False)
        # raw words, against the oracle on the requests they decode to; device buffers with table'
        for R in (5, 1027):
            words = E.raw_packed_words(rng)
            words = np.concatenate([words, egpu.BestFitAllocator.pack_requests(*E.thresholds(t.fc, t.fm))])
            if words.size < R:
                words = np.concatenate([words, rng.integers(0, 1 << 32, R - words.size, dtype=np.int64).astype(np.uint32)])
            words = np.ascontiguousarray(words[rng.permutation(words.size)][:R])
            uc, um = E.unpack_words(words)
            exp = oracle_c.snapshot(t.fc, t.fm, uc, um, 4)
            idx, dc, dm = alloc.bestfit_packed(words)
            _check_snapshot((family, "packed raw", R), D, (idx.astype(np.int32), np.concatenate([dc, dm]), None), exp, False)
            w = torch.from_numpy(words.view(np.int32)).cuda()
            idx8 = torch.full((R + 16,), 77, dtype=torch.int8, device="cuda")
            delta = torch.full((2 * D,), -1, dtype=torch.int64, device="cuda")
            tab = torch.full((3 * D,), -7, dtype=torch.int32, device="cuda")
            alloc.bestfit_packed_dev(w.data_ptr(), R, idx8.data_ptr(), delta.data_ptr(), tab.data_ptr(), stream=s)
            torch.cuda.synchronize()
            got = idx8.cpu().numpy()
            assert (got[R:] == 77).all(), "wrote past R"
            _check_snapshot((family, "packed_dev", R), D, (got[:R].astype(np.int32), delta.cpu().numpy(), tab.cpu().numpy()), exp)


def _query(alloc, D):
    other = E.make_table("random", D, seed=5)
    alloc.set_table(other.fc, other.fm)
    for family in E.TABLE_FAMILIES:
        for R in E.SIZES:
            t, rc, rm, exp = _case(family, D, R)
            _eq(alloc.query(t.fc, t.fm, rc, rm), exp[0], (family, "query", R))
    fc, fm, ov = alloc.table()
    _eq(fc, other.fc, "query leaves the context's table alone")
    _eq(fm, other.fm, "query leaves the context's table alone")


def _prefix(alloc, D, torch, oracle_c):
    s = _stream(torch)
    for family in E.TABLE_FAMILIES:
        for variant in (SORTED, LUT):
            alloc.set_variant(variant)
            for R in E.SIZES:
                t, rc, rm, _ = _case(family, D, R)
                o_idx, o_dc, o_dm, o_tab = oracle_c.prefix_commit(t.fc, t.fm, rc, rm)
                alloc.set_table(t.fc, t.fm)
                c, m = _dev(torch, rc), _dev(torch, rm)
                idx = torch.full((R + 4,), -9, dtype=torch.int32, device="cuda")
                delta = torch.full((2 * D,), -1, dtype=torch.int64, device="cuda")
                tab = torch.full((3 * D,), -7, dtype=torch.int32, device="cuda")
                alloc.bestfit_dev(c.data_ptr(), m.data_ptr(), R, idx.data_ptr(), delta.data_ptr(), tab.data_ptr(), True, s,
                                  prefix_commit=True)
                torch.cuda.synchronize()
                what = (family, variant, "prefix", R)
                _check_snapshot(what, D, (idx.cpu().numpy()[:R], delta.cpu().numpy(), tab.cpu().numpy()), (o_idx, o_dc, o_dm, o_tab))
                fc, fm, ov = alloc.table()
                _eq(fc, o_tab[:D], f"{what}: committed core")
                _eq(fm, o_tab[D:2 * D], f"{what}: committed mem")
                assert not ov.any()


def _rounds(alloc, D, oracle_c):
    for family in E.TABLE_FAMILIES:
        for variant in (SORTED, LUT):
            alloc.set_variant(variant)
            for R in E.SIZES:
                cap = 6 if R > 1027 else 1 << 20
                t, rc, rm, _ = _case(family, D, R)
                alloc.set_table(t.fc, t.fm)
                idx, dc, dm, rounds, left = alloc.bestfit_rounds(rc, rm, cap)
                o_idx, o_dc, o_dm, o_fc, o_fm, o_rounds, o_left = oracle_c.rounds(t.fc, t.fm, rc, rm, cap)
                what = (family, variant, "rounds", R)
                assert (rounds, left) == (o_rounds, o_left), what
                _eq(idx, o_idx, f"{what}: idx")
                _eq(np.concatenate([dc, dm]), np.concatenate([o_dc, o_dm]), f"{what}: delta")
                fc, fm, ov = alloc.table()
                _eq(fc, o_fc, f"{what}: table core")
                _eq(fm, o_fm, f"{what}: table mem")
                assert not ov.any()


def _chain(alloc, D, torch, oracle_c):
    """Four committing batches (edge_cases.chain_requests), checked step by step.  Emptied devices
    pile up as identical (0, 0) rows, and from D = 33 on they straddle sorted position 32 in the
    view the device re-sorted after the commit.  The scans after a commit read that view (register
    scans) or the lookup tables rebuilt from it."""
    s = _stream(torch)
    for family in E.TABLE_FAMILIES:
        t = _case(family, D, 1)[0]
        for variant in (GRID, SORTED, LUT):
            alloc.set_variant(variant)
            alloc.set_table(t.fc, t.fm)
            cur_c, cur_m, sticky = t.fc.copy(), t.fm.copy(), np.zeros(D, np.int32)
            rng = np.random.default_rng(D)  # the chain test_oracle_edges checks for the tie across position 32
            straddled = False
            for step in range(4):
                rc, rm = E.chain_requests(cur_c, cur_m, step, rng)
                R = rc.size
                o_idx, o_dc, o_dm, o_tab = oracle_c.snapshot(cur_c, cur_m, rc, rm)
                c, m = _dev(torch, rc), _dev(torch, rm)
                idx = torch.full((R + 4,), -9, dtype=torch.int32, device="cuda")
                delta = torch.full((2 * D,), -1, dtype=torch.int64, device="cuda")
                tab = torch.full((3 * D,), -7, dtype=torch.int32, device="cuda")
                alloc.bestfit_dev(c.data_ptr(), m.data_ptr(), R, idx.data_ptr(), delta.data_ptr(), tab.data_ptr(), True, s)
                torch.cuda.synchronize()
                what = (family, variant, "chain step", step)
                _check_snapshot(what, D, (idx.cpu().numpy()[:R], delta.cpu().numpy(), tab.cpu().numpy()), (o_idx, o_dc, o_dm, o_tab))
                cur_c, cur_m, ov = committed(o_tab, D)
                sticky |= ov
                fc, fm, gov = alloc.table()
                _eq(fc, cur_c, f"{what}: committed core")
                _eq(fm, cur_m, f"{what}: committed mem")
                _eq(gov, sticky, f"{what}: sticky oversubscription")
                if step < 3:  # a later step scans this table
                    straddled |= E.tie_across_32(cur_c, cur_m)
            if D >= 33:
                assert straddled, (family, variant, "no tie across sorted position 32 after a commit")


@pytest.mark.parametrize("entry", ENTRY_POINTS)
@pytest.mark.parametrize("D", E.D_VALUES)
def test_kernel_matrix(D, entry, alloc, oracle_c, egpu, torch):
    if entry == "host":
        _host(alloc, D)
    elif entry in ("dev_lone", "dev_ready"):
        _dev_single(alloc, D, torch, ready=entry == "dev_ready")
    elif entry == "batches":
        _batches(alloc, D, torch)
    elif entry == "packed":
        _packed(alloc, D, torch, egpu, oracle_c)
    elif entry == "query":
        _query(alloc, D)
    elif entry == "prefix":
        _prefix(alloc, D, torch, oracle_c)
    elif entry == "rounds":
        _rounds(alloc, D, oracle_c)
    else:
        _chain(alloc, D, torch, oracle_c)


# ---------------------------------------------------------------------------------------------
# Epilogue outputs: saturated table', oversubscription in one dimension
# ---------------------------------------------------------------------------------------------

EPI_D = (4, 16, 33, 64)


@functools.lru_cache(maxsize=None)
def _epi_scenarios(D):
    """(name, fc, fm, rc, rm, roles, oracle answer) of the three epilogue scenarios on D devices"""
    from oracle import oracle_c
    rng = np.random.default_rng(D)
    out = []
    # memory: about 20 000 rows of (0, 2^18-1) on one device; table' mem saturates at INT32_MIN
    fc = np.full(D, 100, np.int32)
    fm = rng.integers(0, 1000, D).astype(np.int32)
    tgt = D // 3
    fc[tgt], fm[tgt] = 0, E.MEM_MAX
    out.append(("mem_saturates", fc, fm, np.zeros(20_003, np.int32), np.full(20_003, E.MEM_MAX, np.int32), None))
    # core: 2^25 rows of core 100 on one device; table' core saturates at INT32_MIN
    fc = rng.integers(0, 100, D).astype(np.int32)
    fm = rng.integers(0, E.MEM_MAX, D).astype(np.int32)
    tgt = D - 1 - D // 4
    fc[tgt], fm[tgt] = 100, 7
    R = (1 << 25) + 1
    out.append(("core_saturates", fc, fm, np.full(R, 100, np.int32), np.zeros(R, np.int32), None))
    # one device over in core only, one in memory only, one in both, one untouched
    fc, fm = E.role_table(D)
    roles = E.spread_roles(D)
    rc, rm = E.role_requests(D, roles, 20_011, rng)
    out.append(("one_dimension", fc, fm, rc, rm, roles))
    res = []
    for name, fc, fm, rc, rm, roles in out:
        exp = oracle_c.snapshot(fc, fm, rc, rm, 4)
        tab = exp[3]
        if name == "mem_saturates":
            assert tab[D + D // 3] == E.I32_MIN
        elif name == "core_saturates":
            assert tab[D - 1 - D // 4] == E.I32_MIN
        else:
            E.check_roles(roles, fc, fm, tab)
        res.append((name, fc, fm, rc, rm, roles, exp))
    return res


@pytest.mark.parametrize("path", ["lone", "pipelined", "commit", "multi", "packed_dev"])
@pytest.mark.parametrize("D", EPI_D)
def test_epilogue_outputs(D, path, alloc, oracle_c, egpu, torch):
    s = _stream(torch)
    scen = _epi_scenarios(D)
    dev = [(_dev(torch, sc[3]), _dev(torch, sc[4])) for sc in scen]

    def outs(R, idx_dtype=None):
        return (torch.full((R + 16,), -9, dtype=idx_dtype or torch.int32, device="cuda"),
                torch.full((2 * D,), -1, dtype=torch.int64, device="cuda"),
                torch.full((3 * D,), -7, dtype=torch.int32, device="cuda"))

    def check(what, R, exp, o, roles=None, fc=None, fm=None):
        idx = o[0].cpu().numpy()
        assert (idx[R:] == -9).all(), f"{what}: wrote past R"
        tab = o[2].cpu().numpy()
        _check_snapshot(what, D, (idx[:R].astype(np.int32), o[1].cpu().numpy(), tab), exp)
        if roles is not None:
            E.check_roles(roles, fc, fm, tab)

    def check_table(what, exp, commit, fc, fm):
        g_c, g_m, g_ov = alloc.table()
        e_c, e_m, e_ov = committed(exp[3], D) if commit else (fc, fm, np.zeros(D, np.int32))
        _eq(g_c, e_c, f"{what}: table core")
        _eq(g_m, e_m, f"{what}: table mem")
        _eq(g_ov, e_ov, f"{what}: sticky oversubscription")

    if path in ("lone", "commit"):
        for variant in (GRID, SORTED, LUT):
            alloc.set_variant(variant)
            for (name, fc, fm, rc, rm, roles, exp), (c, m) in zip(scen, dev):
                alloc.set_table(fc, fm)
                o = outs(rc.size)
                alloc.bestfit_dev(c.data_ptr(), m.data_ptr(), rc.size, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(),
                                  path == "commit", s)
                torch.cuda.synchronize()
                check((name, variant, path), rc.size, exp, o, roles, fc, fm)
                check_table((name, variant, path), exp, path == "commit", fc, fm)
    elif path == "pipelined":
        for variant in (SORTED, LUT):
            alloc.set_variant(variant)
            for (name, fc, fm, rc, rm, roles, exp), (c, m) in zip(scen, dev):
                alloc.set_table(fc, fm)
                os_ = [outs(rc.size) for _ in range(3)]
                torch.cuda.synchronize()
                for o in os_:  # three pipelined launches of the same batch
                    alloc.bestfit_dev(c.data_ptr(), m.data_ptr(), rc.size, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(),
                                      False, s, inputs_ready=True)
                torch.cuda.synchronize()
                for k, o in enumerate(os_):
                    check((name, variant, path, k), rc.size, exp, o, roles, fc, fm)
    elif path == "multi":
        # one launch, one table: the role table with device D - 1 able to take both saturating batches
        # (spread_roles leaves D - 1 untouched, and role_requests pads with rows no table can take)
        fc, fm = E.role_table(D)
        fc[D - 1], fm[D - 1] = 100, E.MEM_MAX
        roles = E.spread_roles(D)
        assert roles[D - 1] == "none"
        for variant in (SORTED, LUT):
            alloc.set_variant(variant)
            alloc.set_table(fc, fm)
            batches, keep = [], []
            empty = np.zeros(0, np.int32)
            for rc, rm, c, m in [(sc[3], sc[4], c, m) for sc, (c, m) in zip(scen, dev)] + [(empty, empty, dev[0][0], dev[0][1])]:
                o = outs(rc.size)
                keep.append((rc, rm, c, m, o))
                batches.append((c.data_ptr(), m.data_ptr(), rc.size, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr()))
            torch.cuda.synchronize()
            alloc.bestfit_batches_dev(batches, s)
            torch.cuda.synchronize()
            for k, (rc, rm, c, m, o) in enumerate(keep):
                exp = oracle_c.snapshot(fc, fm, rc, rm, 4)
                if k == 0:
                    assert exp[3][D + D - 1] == E.I32_MIN
                elif k == 1:
                    assert exp[3][D - 1] == E.I32_MIN
                check((variant, "multi batch", k), rc.size, exp, o, roles if k == 2 else None, fc, fm)
            check_table((variant, "multi"), None, False, fc, fm)
    else:  # packed_dev
        for (name, fc, fm, rc, rm, roles, exp) in scen:
            w = torch.from_numpy(egpu.BestFitAllocator.pack_requests(rc, rm).view(np.int32)).cuda()
            for commit in (False, True):
                alloc.set_table(fc, fm)
                o = outs(rc.size, torch.int8)
                alloc.bestfit_packed_dev(w.data_ptr(), rc.size, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), commit, s)
                torch.cuda.synchronize()
                check((name, "packed_dev", commit), rc.size, exp, o, roles, fc, fm)
                check_table((name, "packed_dev", commit), exp, commit, fc, fm)


# ---------------------------------------------------------------------------------------------
# Slot hygiene: two full turns of both epilogue rings
# ---------------------------------------------------------------------------------------------

SINGLE_SLOTS, MULTI_SLOTS = 32, 128


@pytest.mark.parametrize("D", [8, 64])
def test_epilogue_slot_rings_two_full_turns(D, alloc, oracle_c, torch):
    """Every launch takes the next slot of a ring (32 slots for single launches, 128 for the
    batches of multi-batch launches) and must leave it clean for the launch that uses it next.
    The oversubscription pattern changes on every launch, and some launches pass no table'."""
    s = _stream(torch)
    fc, fm = E.role_table(D)
    rng = np.random.default_rng(D)
    alloc.set_table(fc, fm)

    def new_batch(i, R):
        roles = [E.ROLES[j] for j in rng.integers(0, 4, D)]
        rc, rm = E.role_requests(D, roles, R, rng)
        exp = oracle_c.snapshot(fc, fm, rc, rm)
        with_tab = i % 5 != 3
        o = (torch.full((R + 4,), -9, dtype=torch.int32, device="cuda"), torch.full((2 * D,), -1, dtype=torch.int64, device="cuda"),
             torch.full((3 * D,), -7, dtype=torch.int32, device="cuda") if with_tab else None)
        return (roles, rc, rm, _dev(torch, rc), _dev(torch, rm), exp, o)

    def check(what, b):
        roles, rc, rm, c, m, exp, o = b
        R = rc.size
        _eq(o[0].cpu().numpy()[:R], exp[0], f"{what}: idx")
        _eq(o[1].cpu().numpy(), np.concatenate([exp[1], exp[2]]), f"{what}: delta")
        if o[2] is not None:
            tab = o[2].cpu().numpy()
            _eq(tab, exp[3], f"{what}: table'")
            E.check_roles(roles, fc, fm, tab)

    for variant in (SORTED, LUT):
        alloc.set_variant(variant)
        # single ring: 2 turns + 6, lone and pipelined launches mixed
        singles = [new_batch(i, 20_011 if i % 2 else 4_099) for i in range(2 * SINGLE_SLOTS + 6)]
        torch.cuda.synchronize()
        for i, b in enumerate(singles):
            o = b[6]
            alloc.bestfit_dev(b[3].data_ptr(), b[4].data_ptr(), b[1].size, o[0].data_ptr(), o[1].data_ptr(),
                              o[2].data_ptr() if o[2] is not None else 0, False, s, inputs_ready=(i // 7) % 2 == 1)
        torch.cuda.synchronize()
        for i, b in enumerate(singles):
            check((variant, "single launch", i), b)
        # multi ring: 2 turns + 14 batches in launches of 1..45 batches
        sizes = [45, 1, 40, 45, 30, 45, 44, 20]
        assert sum(sizes) > 2 * MULTI_SLOTS
        launches = [[new_batch(i * 100 + k, 4_099 if k % 3 else 9_001) for k in range(K)] for i, K in enumerate(sizes)]
        torch.cuda.synchronize()
        for i, bs in enumerate(launches):
            tup = [(b[3].data_ptr(), b[4].data_ptr(), b[1].size, b[6][0].data_ptr(), b[6][1].data_ptr(),
                    b[6][2].data_ptr() if b[6][2] is not None else 0) for b in bs]
            alloc.bestfit_batches_dev(tup, s, inputs_ready=i % 2 == 1)
        torch.cuda.synchronize()
        for i, bs in enumerate(launches):
            for k, b in enumerate(bs):
                check((variant, "multi launch", i, "batch", k), b)


# ---------------------------------------------------------------------------------------------
# Row limit: EGPU_MAX_ROWS at full size
# ---------------------------------------------------------------------------------------------

def _free_gib(torch):
    free, _ = torch.cuda.mem_get_info()
    return free / (1 << 30)


def _host_free_gib():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) / (1 << 20)
    except OSError:
        pass
    return 0.0


def test_row_limit_full_size(egpu, oracle_c, torch):
    """R = EGPU_MAX_ROWS rows of (100, 2^18-1) on one device: the demand sums are exact, table' is
    saturated, every scan form agrees, and the epilogue slots are clean afterwards.  One row more
    is rejected by every device entry point without launching anything."""
    need = 40
    if _free_gib(torch) < need:
        msg = f"needs {need} GiB of free device memory, {_free_gib(torch):.1f} GiB free"
        print(msg)
        pytest.skip(msg)
    N = 1 << 31  # EGPU_MAX_ROWS + 1 rows, real buffers
    R = E.MAX_ROWS
    word = (100 << 18) | E.MEM_MAX
    fc, fm = np.array([100, 99], np.int32), np.array([E.MEM_MAX, E.MEM_MAX], np.int32)
    exp_delta = [R * 100, 0, R * E.MEM_MAX, 0]
    assert exp_delta[2] == 562_947_805_675_521 and exp_delta[0] == 214_748_364_700
    exp_tab = [E.I32_MIN, 99, E.I32_MIN, E.MEM_MAX, 1, 0]
    s = _stream(torch)
    c = torch.full((N,), 100, dtype=torch.int32, device="cuda")
    m = torch.full((N,), E.MEM_MAX, dtype=torch.int32, device="cuda")
    idx = torch.empty((N,), dtype=torch.int32, device="cuda")
    delta = torch.empty(4, dtype=torch.int64, device="cuda")
    tab = torch.empty(6, dtype=torch.int32, device="cuda")
    rng = np.random.default_rng(1)
    with egpu.BestFitAllocator(0) as a:
        a.set_table(fc, fm)

        def small_launches(n):
            rf, rmm = E.role_table(2)
            a.set_table(rf, rmm)
            for i in range(n):
                roles = [E.ROLES[j] for j in rng.integers(0, 4, 2)]
                rc, rm = E.role_requests(2, roles, 4099, rng)
                exp = oracle_c.snapshot(rf, rmm, rc, rm)
                o = torch.empty(4100, dtype=torch.int32, device="cuda")
                dc_, dm_ = _dev(torch, rc), _dev(torch, rm)
                a.bestfit_dev(dc_.data_ptr(), dm_.data_ptr(), rc.size, o.data_ptr(), delta.data_ptr(), tab.data_ptr(), False, s)
                torch.cuda.synchronize()
                _eq(o.cpu().numpy()[:rc.size], exp[0], ("small launch", i))
                _eq(delta.cpu().numpy(), np.concatenate([exp[1], exp[2]]), ("small launch", i, "delta"))
                _eq(tab.cpu().numpy(), exp[3], ("small launch", i, "table'"))
            a.set_table(fc, fm)

        for variant in (SORTED, LUT, GRID):
            a.set_variant(variant)
            idx[:16].fill_(-9)
            idx[R - 16:].fill_(-9)
            a.bestfit_dev(c.data_ptr(), m.data_ptr(), R, idx.data_ptr(), delta.data_ptr(), tab.data_ptr(), False, s)
            torch.cuda.synchronize()
            assert delta.cpu().tolist() == exp_delta, variant
            assert tab.cpu().tolist() == exp_tab, variant
            assert (idx[:16] == 0).all() and (idx[R - 16:R] == 0).all(), variant
            small_launches(40)
        a.set_variant(SORTED)
        del c, m, idx
        torch.cuda.empty_cache()
        # the packed entry point, same batch
        words = torch.full((N,), word, dtype=torch.int32, device="cuda")
        idx8 = torch.full((N,), 77, dtype=torch.int8, device="cuda")
        a.bestfit_packed_dev(words.data_ptr(), R, idx8.data_ptr(), delta.data_ptr(), tab.data_ptr(), stream=s)
        torch.cuda.synchronize()
        assert delta.cpu().tolist() == exp_delta and tab.cpu().tolist() == exp_tab
        assert (idx8[:R] == 0).all() and int(idx8[R]) == 77
        small_launches(40)

        # one row more: rejected, nothing launched
        n0 = a.launch_count
        delta.fill_(-1)
        for call in ("packed_dev", "batch_dev", "batches_dev"):
            with pytest.raises(egpu.EgpuError) as ei:
                if call == "packed_dev":
                    a.bestfit_packed_dev(words.data_ptr(), N, idx8.data_ptr(), delta.data_ptr(), tab.data_ptr(), stream=s)
                elif call == "batch_dev":
                    a.bestfit_dev(words.data_ptr(), words.data_ptr(), N, words.data_ptr(), delta.data_ptr(), tab.data_ptr(), False, s)
                else:
                    a.bestfit_batches_dev([(words.data_ptr(), words.data_ptr(), N, words.data_ptr(), delta.data_ptr(), tab.data_ptr())], s)
            assert ei.value.code == -1, call
        torch.cuda.synchronize()
        assert a.launch_count == n0 and delta.cpu().tolist() == [-1] * 4
        del words, idx8
        torch.cuda.empty_cache()
        # the host packed call: needs about 10 GiB of host memory for real buffers of that size
        if _host_free_gib() < 12:
            print(f"host packed call at EGPU_MAX_ROWS + 1 rows skipped: {_host_free_gib():.1f} GiB of host memory available, needs 12")
        else:
            hw = np.full(N, word, np.uint32)
            hi = np.full(N, 77, np.int8)
            with pytest.raises(egpu.EgpuError) as ei:
                a.bestfit_packed_raw(hw.ctypes.data, N, hi.ctypes.data, 0, 0)
            assert ei.value.code == -1 and a.launch_count == n0
            del hw, hi


# ---------------------------------------------------------------------------------------------
# Kernel coverage
# ---------------------------------------------------------------------------------------------

OTHER_KERNELS = ("lut_build_kernel", "prefix_cut_kernel", "prefix_apply_kernel", "prefix_finalize_kernel",
                 "deferred_count_kernel", "deferred_scan_kernel", "deferred_scatter_kernel", "round_writeback_kernel")


def test_every_scan_kernel_launches(alloc, oracle_c, egpu, torch):
    """One small case of every form in every D bucket, under torch.profiler: each of the 23 scan
    instantiations (and the lookup-table build, prefix-commit and rounds kernels) must launch."""
    from torch.profiler import ProfilerActivity, profile
    s = _stream(torch)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        x = torch.ones(1024, device="cuda")
        (x * 2).sum().item()
        for D in E.BUCKET_D.values():
            t, rc, rm, exp = _case("random", D, 1027)
            c, m = _dev(torch, rc), _dev(torch, rm)
            idx = torch.empty(1032, dtype=torch.int32, device="cuda")
            for variant in (GRID, SORTED, LUT):
                alloc.set_variant(variant)
                alloc.set_table(t.fc, t.fm)
                _eq(alloc.bestfit(rc, rm)[0], exp[0], (D, variant))
                if variant != GRID:
                    alloc.bestfit(rc, rm, prefix_commit=True)
                    alloc.bestfit_batches_dev([(c.data_ptr(), m.data_ptr(), rc.size, idx.data_ptr(), 0, 0)], s)
                    torch.cuda.synchronize()
                    _eq(idx.cpu().numpy()[:rc.size], exp[0], (D, variant, "multi"))
            _eq(alloc.bestfit_packed(egpu.BestFitAllocator.pack_requests(rc, rm))[0].astype(np.int32), exp[0], (D, "packed"))
        # rounds: the later rounds gather the deferred rows and write their answers back
        w = egpu.synth.workload("cfg3")
        alloc.set_variant(SORTED)
        alloc.set_table(w["free_core"], w["free_mem"])
        rc, rm = egpu.synth.requests(3, 5, 20_001)
        rc, rm = np.minimum(rc, 5).astype(np.int32), np.minimum(rm, 2048).astype(np.int32)
        rounds = alloc.bestfit_rounds(rc, rm)[3]
        assert rounds > 2
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    if not names:
        pytest.skip("torch.profiler recorded no CUDA kernels at all (not even a torch op's)")
    launched = {E.canonical_kernel(n) for n in names} - {None}
    missing = sorted(set(E.SCAN_KERNELS) - launched)
    print(f"scan kernels launched: {len(set(E.SCAN_KERNELS) & launched)}/{len(E.SCAN_KERNELS)}")
    assert not missing, missing
    for k in OTHER_KERNELS:
        assert any(k in n for n in names), k
