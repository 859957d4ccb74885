"""GPU parity tests: the CUDA path, called through the C ABI, must be bit-exact
against the CPU oracle (oracle/) on the same inputs.

"Bit-exact" is against the builder-defined oracle: the reference has no best-fit
path to compare with (SURVEY.md §0) — parity unpinned."""
import hashlib
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
KAT = json.load(open(os.path.join(HERE, "golden", "bestfit_kat.json")))
SYN = json.load(open(os.path.join(HERE, "golden", "bestfit_synth.json")))
VARIANTS = [1, 2, 3]  # EGPU_VARIANT_GRID, EGPU_VARIANT_SORTED, EGPU_VARIANT_LUT


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def committed(tab, D):
    """what commit installs: table' with negative leftovers clamped to 0"""
    return np.maximum(tab[:D], 0), np.maximum(tab[D:2 * D], 0), tab[2 * D:]


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("case", KAT["snapshot"], ids=lambda c: c["name"])
def test_snapshot_kat(case, variant, alloc):
    alloc.set_variant(variant)
    alloc.set_table(case["free_core"], case["free_mem"])
    idx, dc, dm = alloc.bestfit(case["req_core"], case["req_mem"], commit=True)
    assert idx.tolist() == case["idx"]
    assert dc.tolist() == case["delta_core"] and dm.tolist() == case["delta_mem"]
    fc, fm, ov = alloc.table()
    assert fc.tolist() == [max(v, 0) for v in case["table_core"]]
    assert fm.tolist() == [max(v, 0) for v in case["table_mem"]]
    assert ov.tolist() == case["oversub"]


@pytest.mark.parametrize("case", KAT["sequential"], ids=lambda c: c["name"])
def test_sequential_kat(case, alloc):
    alloc.set_table(case["free_core"], case["free_mem"])
    idx = alloc.replay(case["kind"], case["a"], case["b"])
    assert idx.tolist() == case["idx"]
    fc, fm, _ = alloc.table()
    assert fc.tolist() == case["table_core"] and fm.tolist() == case["table_mem"]


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("name", ["cfg2", "cfg3", "cfg3_1m", "cfg4"])
def test_configs_bit_exact_vs_oracle_and_golden(name, variant, alloc, oracle_c, egpu):
    w = egpu.synth.workload(name)
    rc, rm = egpu.synth.requests(w["dist"], w["seed"], w["R"])
    alloc.set_variant(variant)
    alloc.set_table(w["free_core"], w["free_mem"])
    idx, dc, dm = alloc.bestfit(rc, rm, commit=True)
    o_idx, o_dc, o_dm, o_tab = oracle_c.snapshot(w["free_core"], w["free_mem"], rc, rm, 4)
    assert np.array_equal(idx, o_idx)
    assert np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)
    g = SYN["snapshot"][name]
    assert digest(idx) == g["idx_sha256"]
    assert dc.tolist() == g["delta_core"] and dm.tolist() == g["delta_mem"]
    fc, fm, ov = alloc.table()
    efc, efm, eov = committed(o_tab, w["D"])
    assert np.array_equal(fc, efc) and np.array_equal(fm, efm) and np.array_equal(ov, eov)


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("D", [1, 2, 7, 8, 9, 16, 17, 31, 32, 33, 63, 64])
def test_random_tables_every_device_count(D, variant, alloc, oracle_c, egpu):
    rng = np.random.default_rng(1000 + D)
    fc = rng.integers(0, 101, D).astype(np.int32)
    fm = rng.integers(0, 1 << 18, D).astype(np.int32)
    R = 40_003  # ragged: not a multiple of 4
    rc = rng.integers(-1, 104, R).astype(np.int32)
    rm = rng.integers(-1, (1 << 18) + 2, R).astype(np.int32)
    rm[::3] = rng.integers(0, 4096, rm[::3].size)  # plenty of feasible rows
    alloc.set_variant(variant)
    alloc.set_table(fc, fm)
    idx, dc, dm = alloc.bestfit(rc, rm)
    o_idx, o_dc, o_dm, _ = oracle_c.snapshot(fc, fm, rc, rm, 4)
    assert np.array_equal(idx, o_idx)
    assert np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)
    # commit=False leaves the table alone
    fc2, fm2, ov2 = alloc.table()
    assert np.array_equal(fc2, fc) and np.array_equal(fm2, fm) and not ov2.any()


@pytest.mark.parametrize("R", [0, 1, 2, 3, 4, 5, 255, 1023, 1024, 1025, 2049])
def test_empty_and_ragged_batches(R, alloc, oracle_c, egpu):
    w = egpu.synth.workload("cfg3")
    rc, rm = egpu.synth.requests(3, 77, R)
    alloc.set_table(w["free_core"], w["free_mem"])
    for variant in VARIANTS:
        alloc.set_variant(variant)
        idx, dc, dm = alloc.bestfit(rc, rm)
        o_idx, o_dc, o_dm, _ = oracle_c.snapshot(w["free_core"], w["free_mem"], rc, rm)
        assert np.array_equal(idx, o_idx) and np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)


@pytest.mark.parametrize("D,dist", [(8, 3), (64, 4)])
def test_zero_copy_pinned_buffers(D, dist, alloc, oracle_c, egpu):
    """Pinned caller buffers take the zero-copy path (the scan reads/writes host memory
    across PCIe); a misaligned pinned slice must fall back to staging.  Same answers."""
    w = egpu.synth.workload("cfg3" if D == 8 else "cfg4")
    R = 300_001
    rc, rm = egpu.synth.requests(dist, 55, R)
    pc, pm, pi = alloc.pinned_array(R + 8), alloc.pinned_array(R + 8), alloc.pinned_array(R + 8)
    dc, dm = alloc.pinned_array(D, np.int64), alloc.pinned_array(D, np.int64)
    o_idx, o_dc, o_dm, _ = oracle_c.snapshot(w["free_core"], w["free_mem"], rc, rm, 4)
    alloc.set_table(w["free_core"], w["free_mem"])
    for off in (0, 1, 4):  # element offsets: 0 and 4 are 16-byte aligned, 1 is not
        pc[off:off + R] = rc
        pm[off:off + R] = rm
        pi[:] = -9
        n0 = alloc.launch_count
        alloc.bestfit_raw(pc.ctypes.data + 4 * off, pm.ctypes.data + 4 * off, R, pi.ctypes.data + 4 * off,
                          dc.ctypes.data, dm.ctypes.data)
        assert alloc.launch_count in (n0 + 1, n0 + 2)  # one scan (+ one lookup-table build after set_table)
        assert np.array_equal(pi[off:off + R], o_idx)
        assert (pi[:off] == -9).all() and (pi[off + R:] == -9).all()
        assert np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)
    for a in (pc, pm, pi, dc, dm):
        alloc.host_free(a.ctypes.data)


@pytest.mark.parametrize("D", [1, 8, 9, 33, 64])
def test_packed_wire_format(D, alloc, oracle_c, egpu):
    """5-byte-per-decision format: same decisions as the int32 arrays, staged and zero-copy."""
    rng = np.random.default_rng(2000 + D)
    fc = rng.integers(0, 101, D).astype(np.int32)
    fm = rng.integers(0, 1 << 18, D).astype(np.int32)
    for R in (0, 1, 15, 16, 17, 70_001):
        rc = rng.integers(-1, 130, R).astype(np.int32)
        rm = rng.integers(-1, (1 << 18) + 2, R).astype(np.int32)
        rm[::2] = rng.integers(0, 8192, rm[::2].size)
        packed = alloc.pack_requests(rc, rm)
        # what the packed format can express: out-of-domain rows are "invalid" = infeasible, as in the spec
        o_idx, o_dc, o_dm, _ = oracle_c.snapshot(fc, fm, rc, rm, 4)
        alloc.set_table(fc, fm)
        idx, dc, dm = alloc.bestfit_packed(packed)
        assert np.array_equal(idx.astype(np.int32), o_idx) and np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)
        if R:
            pr = alloc.pinned_array(R, np.uint32)
            pi = alloc.pinned_array(R + 16, np.int8)
            hdc, hdm = alloc.pinned_array(D, np.int64), alloc.pinned_array(D, np.int64)
            pr[:] = packed
            pi[:] = 55
            alloc.bestfit_packed_raw(pr.ctypes.data, R, pi.ctypes.data, hdc.ctypes.data, hdm.ctypes.data)
            assert np.array_equal(pi[:R].astype(np.int32), o_idx) and (pi[R:] == 55).all()
            assert np.array_equal(hdc, o_dc) and np.array_equal(hdm, o_dm)
            for a in (pr, pi, hdc, hdm):
                alloc.host_free(a.ctypes.data)


@pytest.mark.parametrize("case", KAT["prefix_commit"], ids=lambda c: c["name"])
def test_prefix_commit_kat(case, alloc):
    for variant in (2, 3):
        alloc.set_variant(variant)
        alloc.set_table(case["free_core"], case["free_mem"])
        idx, dc, dm = alloc.bestfit(case["req_core"], case["req_mem"], commit=True, prefix_commit=True)
        assert idx.tolist() == case["idx"]
        assert dc.tolist() == case["delta_core"] and dm.tolist() == case["delta_mem"]
        fc, fm, ov = alloc.table()
        assert fc.tolist() == case["table_core"] and fm.tolist() == case["table_mem"] and not ov.any()


@pytest.mark.parametrize("case", KAT["rounds"], ids=lambda c: c["name"])
def test_rounds_kat(case, alloc):
    for variant in (2, 3):
        alloc.set_variant(variant)
        alloc.set_table(case["free_core"], case["free_mem"])
        idx, dc, dm, rounds, left = alloc.bestfit_rounds(case["req_core"], case["req_mem"], case["max_rounds"])
        assert idx.tolist() == case["idx"]
        assert dc.tolist() == case["delta_core"] and dm.tolist() == case["delta_mem"]
        assert (rounds, left) == (case["rounds"], case["left"])
        fc, fm, ov = alloc.table()
        assert fc.tolist() == case["table_core"] and fm.tolist() == case["table_mem"] and not ov.any()


@pytest.mark.parametrize("D,R,dist", [(8, 5_000, 3), (8, 300_001, 2), (64, 100_003, 4), (16, 2_049, 3), (3, 1_023, 2)])
def test_rounds_match_oracle(D, R, dist, alloc, oracle_c, egpu):
    """egpu_bestfit_batch_rounds to the fixed point: indices, total committed demand, final table,
    number of rounds - all bit-exact against the oracle; then capped at 2 rounds."""
    w = egpu.synth.workload("cfg4" if D == 64 else "cfg3")
    rng = np.random.default_rng(D * 1000 + R)
    fc = w["free_core"][:D] if D <= len(w["free_core"]) else rng.integers(0, 101, D).astype(np.int32)
    fm = w["free_mem"][:D] if D <= len(w["free_mem"]) else rng.integers(0, 100000, D).astype(np.int32)
    rc, rm = egpu.synth.requests(dist, 11, R)
    rm = np.minimum(rm, 4096).astype(np.int32)      # small memory asks: many rows fit, many rounds
    rc = np.minimum(rc, 7).astype(np.int32)
    for cap in (1 << 20, 2):
        alloc.set_table(fc, fm)
        idx, dc, dm, rounds, left = alloc.bestfit_rounds(rc, rm, cap)
        o_idx, o_dc, o_dm, o_fc, o_fm, o_rounds, o_left = oracle_c.rounds(fc, fm, rc, rm, cap)
        assert (rounds, left) == (o_rounds, o_left)
        assert np.array_equal(idx, o_idx)
        assert np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)
        g_fc, g_fm, ov = alloc.table()
        assert np.array_equal(g_fc, o_fc) and np.array_equal(g_fm, o_fm) and not ov.any()
    assert o_rounds == 2


def test_rounds_dev_form(alloc, oracle_c, egpu):
    import torch
    w = egpu.synth.workload("cfg3")
    R = 70_001
    rc, rm = egpu.synth.requests(3, 5, R)
    rc, rm = np.minimum(rc, 5).astype(np.int32), np.minimum(rm, 2048).astype(np.int32)
    c, m = torch.from_numpy(rc).cuda(), torch.from_numpy(rm).cuda()
    idx = torch.empty(R, dtype=torch.int32, device="cuda")
    alloc.set_table(w["free_core"], w["free_mem"])
    delta, rounds, left = alloc.bestfit_rounds_dev(c.data_ptr(), m.data_ptr(), R, idx.data_ptr(),
                                                   stream=torch.cuda.current_stream().cuda_stream)
    o_idx, o_dc, o_dm, o_fc, o_fm, o_rounds, o_left = oracle_c.rounds(w["free_core"], w["free_mem"], rc, rm)
    assert (rounds, left) == (o_rounds, o_left) and o_rounds > 2
    assert np.array_equal(idx.cpu().numpy(), o_idx) and np.array_equal(delta, np.concatenate([o_dc, o_dm]))


@pytest.mark.parametrize("variant", [2, 3])
@pytest.mark.parametrize("D,R", [(1, 5), (8, 1000), (8, 70_003), (9, 40_001), (64, 70_003), (64, 1_000_003), (8, 4_000_001)])
def test_prefix_commit_matches_oracle(D, R, variant, alloc, oracle_c):
    rng = np.random.default_rng(31 * D + R)
    fc = rng.integers(0, 101, D).astype(np.int32)
    fm = rng.integers(0, 1 << 18, D).astype(np.int32)
    # small requests, so that the cut of each device falls somewhere inside the batch
    rc = rng.integers(0, 3, R).astype(np.int32)
    rm = rng.integers(0, 300, R).astype(np.int32)
    rc[rng.integers(0, R, max(1, R // 50))] = rng.integers(-1, 120, max(1, R // 50))
    alloc.set_variant(variant)
    alloc.set_table(fc, fm)
    idx, dc, dm = alloc.bestfit(rc, rm, prefix_commit=True)
    o_idx, o_dc, o_dm, o_tab = oracle_c.prefix_commit(fc, fm, rc, rm)
    assert np.array_equal(idx, o_idx)
    assert np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)
    g_c, g_m, _ = alloc.table()
    assert np.array_equal(g_c, fc) and np.array_equal(g_m, fm)  # no commit asked


def test_prefix_commit_retry_rounds_fill_the_node(alloc, oracle_c, egpu):
    """The caller's loop of spec 2.5: commit what fits, re-score the deferred rows against the
    new table, until nothing is deferred.  Every round must match the oracle and the table must
    never go negative."""
    import torch
    fc, fm = egpu.synth.table_full(8)
    rc, rm = egpu.synth.requests(2, 123, 3000)   # cfg2 sizes: 5..100 % core
    alloc.set_table(fc, fm)
    cur_c, cur_m = fc.copy(), fm.copy()
    pend = np.arange(rc.size)
    placed = np.full(rc.size, -9, dtype=np.int32)
    for rounds in range(1, 50):
        idx, dc, dm = alloc.bestfit(rc[pend], rm[pend], commit=True, prefix_commit=True)
        o_idx, o_dc, o_dm, o_tab = oracle_c.prefix_commit(cur_c, cur_m, rc[pend], rm[pend])
        assert np.array_equal(idx, o_idx) and np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)
        cur_c, cur_m = o_tab[:8].copy(), o_tab[8:16].copy()
        g_c, g_m, ov = alloc.table()
        assert np.array_equal(g_c, cur_c) and np.array_equal(g_m, cur_m) and not ov.any() and (g_c >= 0).all()
        placed[pend[idx != -2]] = idx[idx != -2]
        pend = pend[idx == -2]
        if pend.size == 0:
            break
    assert pend.size == 0 and rounds < 49
    # the node ends up (nearly) full of core: whatever is left cannot hold the smallest request that failed
    assert (placed >= -1).all()


def test_prefix_commit_not_with_grid_variant(alloc, egpu):
    alloc.set_variant(1)
    alloc.set_table([10], [10])
    with pytest.raises(egpu.EgpuError) as ei:
        alloc.bestfit([1], [1], prefix_commit=True)
    assert ei.value.code == -6


def test_ties_pick_lowest_index_everywhere(alloc):
    for D in (8, 64):
        alloc.set_table([100] * D, [1000] * D)
        idx, dc, _ = alloc.bestfit(np.full(4099, 1, np.int32), np.full(4099, 1, np.int32))
        assert (idx == 0).all() and dc[0] == 4099 and not dc[1:].any()


def test_int64_demand_sums_do_not_overflow(alloc, oracle_c):
    """10^6 rows x 200000 MiB overflows int32; deltas are int64 (spec §2.4)."""
    R = 1_000_000
    rc = np.ones(R, np.int32)
    rm = np.full(R, 200_000, np.int32)
    alloc.set_table([100, 50], [250_000, 1000])
    idx, dc, dm = alloc.bestfit(rc, rm, commit=True)
    assert (idx == 0).all() and dc[0] == R and dm[0] == 200_000 * R
    fc, fm, ov = alloc.table()
    assert fc.tolist() == [0, 50] and fm.tolist() == [0, 1000] and ov.tolist() == [1, 0]


def test_commit_chain_matches_oracle(alloc, oracle_c, egpu):
    """commit=1 over several small batches == oracle applied batch by batch."""
    fc, fm = egpu.synth.table_full(8)
    alloc.set_table(fc, fm)
    cur_c, cur_m = fc.copy(), fm.copy()
    for k in range(6):
        rc, rm = egpu.synth.requests(2, 100 + k, 7)
        idx, dc, dm = alloc.bestfit(rc, rm, commit=True)
        o_idx, o_dc, o_dm, o_tab = oracle_c.snapshot(cur_c, cur_m, rc, rm)
        assert np.array_equal(idx, o_idx) and np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)
        cur_c, cur_m, _ = committed(o_tab, 8)
        g_c, g_m, _ = alloc.table()
        assert np.array_equal(g_c, cur_c) and np.array_equal(g_m, cur_m)


def test_churn_replay_cfg5_final_state(alloc, oracle_c, egpu):
    w = egpu.synth.workload("cfg5")
    kind, a, b = egpu.synth.churn_events(w["seed"], w["R"])
    alloc.set_table(w["free_core"], w["free_mem"])
    idx = alloc.replay(kind, a, b)
    o_idx, o_fc, o_fm = oracle_c.replay(w["free_core"], w["free_mem"], kind, a, b)
    assert np.array_equal(idx, o_idx)
    fc, fm, _ = alloc.table()
    assert np.array_equal(fc, o_fc) and np.array_equal(fm, o_fm)
    g = SYN["sequential"]["cfg5_head20000"]
    assert digest(idx[:g["E"]]) == g["idx_sha256"]


@pytest.mark.parametrize("D,E", [(8, 1), (8, 31), (8, 33), (33, 5000), (64, 5000), (8, 300_000)])
def test_replay_random(D, E, alloc, oracle_c):
    rng = np.random.default_rng(D * 7919 + E)
    fc = rng.integers(0, 101, D).astype(np.int32)
    fm = rng.integers(0, 1 << 18, D).astype(np.int32)
    kind = (rng.random(E) < 0.45).astype(np.int32)
    a = np.where(kind == 0, rng.integers(0, 40, E), (rng.random(E) * np.arange(E)).astype(np.int64) - 1).astype(np.int32)
    b = rng.integers(0, 30000, E).astype(np.int32)
    kind[rng.integers(0, E, max(1, E // 50))] = 2  # unknown kinds are no-ops
    alloc.set_table(fc, fm)
    idx = alloc.replay(kind, a, b)
    o_idx, o_fc, o_fm = oracle_c.replay(fc, fm, kind, a, b)
    assert np.array_equal(idx, o_idx)
    g_c, g_m, _ = alloc.table()
    assert np.array_equal(g_c, o_fc) and np.array_equal(g_m, o_fm)


def test_replay_all_kernels_agree(oracle_c, egpu):
    """Every replay kernel on churn streams with the odd cases sprinkled in (double frees, frees of non-ALLOC
    events, frees of later events, unknown kinds), against the oracle.  The input picks the kernel: the two-warp
    kernel for D <= 32 while the events fit shared memory (E <= 200 Ki), else the one-warp kernels - table in
    registers for D <= 8, lane = device above - with `live` in HBM past 200 Ki events."""
    def odd_stream(E):
        kind, a, b = egpu.synth.churn_events(9, E)
        kind, a, b = kind.copy(), a.copy(), b.copy()
        rng = np.random.default_rng(3)
        for i in rng.integers(10, kind.size, 400):     # sprinkle the odd cases in
            r = rng.integers(0, 5)
            if r == 0:
                kind[i], a[i] = 1, a[i - 1] if kind[i - 1] == 1 else i - 1        # free right after / double free
            elif r == 1:
                kind[i], a[i] = 1, i + 5                                           # target in the future
            elif r == 2:
                kind[i], a[i] = 1, -3
            elif r == 3:
                kind[i] = 7                                                        # unknown kind
            else:
                kind[i], a[i], b[i] = 0, 101, 5                                    # infeasible ALLOC (then possibly freed later)
        return kind, a, b

    for E, Ds in ((50_000, (1, 3, 8, 9, 32, 33)), (200 * 1024 + 1, (1, 8, 9, 32, 33))):
        kind, a, b = odd_stream(E)
        for D in Ds:
            fc, fm = egpu.synth.table_fragmented(40 + D, D)
            fc = np.maximum(fc, 30)
            o_idx, o_fc, o_fm = oracle_c.replay(fc, fm, kind, a, b)
            with egpu.BestFitAllocator(0) as al:
                al.set_table(fc, fm)
                idx = al.replay(kind, a, b)
                g_c, g_m, _ = al.table()
            assert np.array_equal(idx, o_idx), (E, D)
            assert np.array_equal(g_c, o_fc) and np.array_equal(g_m, o_fm), (E, D)
    # sizes around the 256-event ring chunks
    fc, fm = egpu.synth.table_full(8)
    for E in (1, 2, 255, 256, 257, 511, 512, 513, 1000):
        k2, a2, b2 = egpu.synth.churn_events(5, E)
        o_idx, o_fc, o_fm = oracle_c.replay(fc, fm, k2, a2, b2)
        with egpu.BestFitAllocator(0) as al:
            al.set_table(fc, fm)
            assert np.array_equal(al.replay(k2, a2, b2), o_idx), E
            g_c, g_m, _ = al.table()
        assert np.array_equal(g_c, o_fc) and np.array_equal(g_m, o_fm)


def test_device_synth_matches_numpy(alloc, egpu):
    import torch
    R = 100_003
    for dist in (2, 3, 4):
        c = torch.empty(R, dtype=torch.int32, device="cuda")
        m = torch.empty(R, dtype=torch.int32, device="cuda")
        alloc.synth_requests_dev(dist, 9, 12345, R, c.data_ptr(), m.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        rc, rm = egpu.synth.requests(dist, 9, R, first_row=12345)
        assert np.array_equal(c.cpu().numpy(), rc) and np.array_equal(m.cpu().numpy(), rm)


def test_device_buffer_entry_point_and_table_out(alloc, oracle_c, egpu):
    import torch
    w = egpu.synth.workload("cfg4")
    R = 262_147
    rc, rm = egpu.synth.requests(4, 21, R)
    s = torch.cuda.current_stream().cuda_stream
    c = torch.from_numpy(rc).cuda()
    m = torch.from_numpy(rm).cuda()
    idx = torch.empty(R, dtype=torch.int32, device="cuda")
    delta = torch.empty(2 * 64, dtype=torch.int64, device="cuda")
    tab = torch.empty(3 * 64, dtype=torch.int32, device="cuda")
    alloc.set_table(w["free_core"], w["free_mem"])
    alloc.bestfit_dev(c.data_ptr(), m.data_ptr(), R, idx.data_ptr(), delta.data_ptr(), tab.data_ptr(), False, s)
    torch.cuda.synchronize()
    o_idx, o_dc, o_dm, o_tab = oracle_c.snapshot(w["free_core"], w["free_mem"], rc, rm, 4)
    assert np.array_equal(idx.cpu().numpy(), o_idx)
    assert np.array_equal(delta.cpu().numpy(), np.concatenate([o_dc, o_dm]))
    assert np.array_equal(tab.cpu().numpy(), o_tab)


@pytest.mark.parametrize("D", [8, 64])
def test_pipelined_launches_overlap_safely(D, alloc, oracle_c, egpu):
    """EGPU_F_INPUTS_READY lets consecutive scans overlap (programmatic dependent
    launch).  A chain of 24 batches over a ring of buffers, with a commit in the
    middle and one launch that reuses the previous output buffer, must equal the
    oracle applied batch by batch."""
    import torch
    rng = np.random.default_rng(D)
    fc = rng.integers(20, 101, D).astype(np.int32)
    fm = rng.integers(1 << 15, 1 << 18, D).astype(np.int32)
    s = torch.cuda.current_stream().cuda_stream
    R = 60_001
    nb = 6
    host = [egpu.synth.requests(4, 300 + b, R) for b in range(nb)]
    dev = [(torch.from_numpy(c).cuda(), torch.from_numpy(m).cuda()) for c, m in host]
    outs = [torch.empty(R + 3, dtype=torch.int32, device="cuda") for _ in range(nb)]
    deltas = [torch.empty(2 * D, dtype=torch.int64, device="cuda") for _ in range(24)]
    torch.cuda.synchronize()
    alloc.set_table(fc, fm)
    plan = []
    for i in range(24):
        b = i % nb
        ob = b if i != 13 else (i - 1) % nb      # launch 13 writes where launch 12 wrote
        commit = i in (7, 8, 20)
        plan.append((b, ob, commit))
        alloc.bestfit_dev(dev[b][0].data_ptr(), dev[b][1].data_ptr(), R, outs[ob].data_ptr(), deltas[i].data_ptr(), 0,
                          commit, s, inputs_ready=True)
    torch.cuda.synchronize()
    # replay on the oracle; only the LAST writer of each output buffer is checkable
    cur_c, cur_m = fc.copy(), fm.copy()
    last_writer = {}
    expect = []
    for i, (b, ob, commit) in enumerate(plan):
        o_idx, o_dc, o_dm, o_tab = oracle_c.snapshot(cur_c, cur_m, host[b][0], host[b][1], 4)
        expect.append((o_idx, np.concatenate([o_dc, o_dm])))
        last_writer[ob] = i
        if commit:
            cur_c, cur_m, _ = committed(o_tab, D)
    for i in range(24):
        assert np.array_equal(deltas[i].cpu().numpy(), expect[i][1]), f"delta of launch {i}"
    for ob, i in last_writer.items():
        assert np.array_equal(outs[ob][:R].cpu().numpy(), expect[i][0]), f"indices of launch {i}"
    g_c, g_m, _ = alloc.table()
    assert np.array_equal(g_c, cur_c) and np.array_equal(g_m, cur_m)


def test_pipelined_launches_many_small_batches(alloc, oracle_c, egpu):
    """Hundreds of tiny batches back to back (each one CTA): many launches could be in
    flight at once; the launch groups bound that and results stay exact.  Also a run
    where every launch shares ONE demand-sum buffer (must fall back to ordered launches:
    the buffer ends up holding the last launch's sums)."""
    import torch
    w = egpu.synth.workload("cfg3")
    s = torch.cuda.current_stream().cuda_stream
    n, R = 300, 513
    rc, rm = egpu.synth.requests(3, 41, n * R)
    c = torch.from_numpy(rc).cuda()
    m = torch.from_numpy(rm).cuda()
    stride = 516  # 513 rows * 4 B is not a multiple of 16: batch k sits at a 16-byte aligned offset
    idx = torch.full((n * stride,), -7, dtype=torch.int32, device="cuda")
    deltas = torch.zeros(n, 16, dtype=torch.int64, device="cuda")
    shared = torch.zeros(16, dtype=torch.int64, device="cuda")
    alloc.set_table(w["free_core"], w["free_mem"])
    torch.cuda.synchronize()
    idx2 = torch.full((n * stride,), -7, dtype=torch.int32, device="cuda")
    c2 = torch.zeros(n * stride, dtype=torch.int32, device="cuda")
    m2 = torch.zeros(n * stride, dtype=torch.int32, device="cuda")
    for k in range(n):
        c2[k * stride:k * stride + R] = c[k * R:(k + 1) * R]
        m2[k * stride:k * stride + R] = m[k * R:(k + 1) * R]
    torch.cuda.synchronize()
    for k in range(n):
        o = 4 * k * stride
        alloc.bestfit_dev(c2.data_ptr() + o, m2.data_ptr() + o, R, idx2.data_ptr() + o, deltas[k].data_ptr(), 0, False, s,
                          inputs_ready=True)
    for k in range(n):
        o = 4 * k * stride
        alloc.bestfit_dev(c2.data_ptr() + o, m2.data_ptr() + o, R, idx.data_ptr() + o, shared.data_ptr(), 0, False, s,
                          inputs_ready=True)
    torch.cuda.synchronize()
    got = idx2.cpu().numpy().reshape(n, stride)
    got_b = idx.cpu().numpy().reshape(n, stride)
    dl = deltas.cpu().numpy()
    for k in range(n):
        o_idx, o_dc, o_dm, _ = oracle_c.snapshot(w["free_core"], w["free_mem"], rc[k * R:(k + 1) * R], rm[k * R:(k + 1) * R])
        assert np.array_equal(got[k, :R], o_idx) and (got[k, R:] == -7).all()
        assert np.array_equal(got_b[k, :R], o_idx)
        assert np.array_equal(dl[k], np.concatenate([o_dc, o_dm]))
    assert np.array_equal(shared.cpu().numpy(), dl[n - 1])


def test_events_after_launches_see_completed_scans(alloc, egpu):
    """Stream semantics: an event recorded after scans (plain or pipelined with
    inputs_ready=True, which trigger their successors early) must not complete before the
    indices are written — checked from another stream that waits only for the event."""
    import torch
    w = egpu.synth.workload("cfg3")
    alloc.set_table(w["free_core"], w["free_mem"])
    R = 32 << 20
    st = torch.cuda.Stream()
    side = torch.cuda.Stream()
    sh = st.cuda_stream
    with torch.cuda.stream(st):
        c = torch.empty(R, dtype=torch.int32, device="cuda")
        m = torch.empty_like(c)
        alloc.synth_requests_dev(3, 7, 0, R, c.data_ptr(), m.data_ptr(), sh)
        outs = [torch.empty(R, dtype=torch.int32, device="cuda") for _ in range(3)]
        dls = [torch.zeros(16, dtype=torch.int64, device="cuda") for _ in range(3)]
    torch.cuda.synchronize()
    for ready in (False, True):
        with torch.cuda.stream(st):
            for o in outs:
                o.fill_(-9)
        torch.cuda.synchronize()
        ev = torch.cuda.Event()
        for i in range(6):
            alloc.bestfit_dev(c.data_ptr(), m.data_ptr(), R, outs[i % 3].data_ptr(), dls[i % 3].data_ptr(), 0, False, sh,
                              inputs_ready=ready)
        ev.record(st)
        side.wait_event(ev)
        with torch.cuda.stream(side):
            unwritten = (outs[2] == -9).sum() + (outs[0] == -9).sum() + (outs[1] == -9).sum()
        torch.cuda.synchronize()
        assert int(unwritten) == 0, (ready, int(unwritten))


def test_full_size_properties_64mi(alloc, egpu):
    """BASELINE full size and beyond, checked through size-independent properties:
    forced-infeasible rows are -1, every chosen device is feasible, the demand
    sums equal a torch recomputation, and the two kernel variants agree."""
    import torch
    w = egpu.synth.workload("cfg3")
    R = 16 << 20
    s = torch.cuda.current_stream().cuda_stream
    c = torch.empty(R, dtype=torch.int32, device="cuda")
    m = torch.empty(R, dtype=torch.int32, device="cuda")
    alloc.synth_requests_dev(3, 7, 0, R, c.data_ptr(), m.data_ptr(), s)
    alloc.set_table(w["free_core"], w["free_mem"])
    outs = []
    for variant in VARIANTS:
        alloc.set_variant(variant)
        idx = torch.empty(R, dtype=torch.int32, device="cuda")
        delta = torch.empty(16, dtype=torch.int64, device="cuda")
        alloc.bestfit_dev(c.data_ptr(), m.data_ptr(), R, idx.data_ptr(), delta.data_ptr(), 0, False, s)
        torch.cuda.synchronize()
        outs.append((idx, delta))
    for o in outs[1:]:
        assert torch.equal(outs[0][0], o[0]) and torch.equal(outs[0][1], o[1])
    idx, delta = outs[1]
    assert bool((idx[15::16] == -1).all())
    fc = torch.tensor(w["free_core"], device="cuda")
    fm = torch.tensor(w["free_mem"], device="cuda")
    ok = idx >= 0
    sel = idx[ok].long()
    assert bool((fc[sel] >= c[ok]).all()) and bool((fm[sel] >= m[ok]).all())
    # rows marked infeasible really fit nowhere
    bad = ~ok
    fits = ((fc[None, :] >= c[bad][:, None]) & (fm[None, :] >= m[bad][:, None])).any(dim=1)
    assert not bool(fits.any())
    dc = torch.zeros(8, dtype=torch.int64, device="cuda").index_add_(0, sel, c[ok].long())
    dm = torch.zeros(8, dtype=torch.int64, device="cuda").index_add_(0, sel, m[ok].long())
    assert torch.equal(delta, torch.cat([dc, dm]))


def test_concurrent_callers_share_one_context(alloc, oracle_c, egpu):
    """grpc-go runs every RPC on its own goroutine, goroutines migrate between OS threads, and
    the reference serialises commits with one mutex per plugin (pkg/plugins/gpushare.go:114).
    Here: 6 OS threads hammer ONE context (ctypes drops the GIL); every answer must be exact."""
    import threading
    w = egpu.synth.workload("cfg3")
    alloc.set_table(w["free_core"], w["free_mem"])
    errors = []

    def worker(k):
        try:
            for i in range(25):
                R = 1000 + 37 * k + i
                rc, rm = egpu.synth.requests(3, 1000 * k + i, R)
                idx, dc, dm = alloc.bestfit(rc, rm)
                o_idx, o_dc, o_dm, _ = oracle_c.snapshot(w["free_core"], w["free_mem"], rc, rm)
                if not (np.array_equal(idx, o_idx) and np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)):
                    errors.append((k, i))
        except Exception as ex:  # noqa: BLE001
            errors.append((k, repr(ex)))

    threads = [threading.Thread(target=worker, args=(k,)) for k in range(6)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors[:3]


def test_misaligned_device_pointers_are_rejected(alloc, egpu):
    import torch
    alloc.set_table([10], [10])
    c = torch.zeros(64, dtype=torch.int32, device="cuda")
    m = torch.zeros(64, dtype=torch.int32, device="cuda")
    o = torch.zeros(64, dtype=torch.int32, device="cuda")
    for bad in ((4, 0, 0), (0, 8, 0), (0, 0, 12)):
        with pytest.raises(egpu.EgpuError) as ei:
            alloc.bestfit_dev(c.data_ptr() + bad[0], m.data_ptr() + bad[1], 8, o.data_ptr() + bad[2])
        assert ei.value.code == -1
    alloc.bestfit_dev(c.data_ptr() + 16, m.data_ptr() + 32, 8, o.data_ptr() + 48)  # 16-byte aligned offsets are fine
    torch.cuda.synchronize()


def test_error_paths(alloc, egpu):
    with pytest.raises(egpu.EgpuError) as ei:
        alloc.bestfit([1], [1])
    assert ei.value.code == -5  # no table
    for bad in ([[101], [1]], [[-1], [1]], [[1], [1 << 18]], [[1] * 65, [1] * 65]):
        with pytest.raises(egpu.EgpuError) as ei:
            alloc.set_table(*bad)
        assert ei.value.code == -1
    assert alloc.launch_count == 0
    alloc.set_table([1], [1])
    alloc.bestfit([1], [1])
    assert alloc.launch_count == 1
