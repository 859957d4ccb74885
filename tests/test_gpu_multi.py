"""GPU tests of the round-2 entry points: multi-batch launches (egpu_bestfit_batches_dev),
the stateless query (egpu_bestfit_query), the start gate, the all-gather form of the
multi-GPU step (egpu_table_apply_deltas_dev + sharding.sharded_step) and the two launch-order
cases the round-1 review found.  Expected values come from the CPU oracle ("bit-exact" =
CUDA == builder-defined oracle; the reference has no best-fit path, SURVEY.md §0)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _dev_batches(torch, egpu, dist, seeds, rows, D, with_table=True):
    """device arrays + the tuples BestFitAllocator.make_batches wants; returns (host inputs, tensors, tuples)"""
    host, tens, tup = [], [], []
    for seed, R in zip(seeds, rows):
        rc, rm = egpu.synth.requests(dist, seed, R)
        c = torch.from_numpy(rc).cuda() if R else torch.empty(4, dtype=torch.int32, device="cuda")
        m = torch.from_numpy(rm).cuda() if R else torch.empty(4, dtype=torch.int32, device="cuda")
        idx = torch.full((R + 4,), -9, dtype=torch.int32, device="cuda")
        dl = torch.full((2 * D,), -1, dtype=torch.int64, device="cuda")
        to = torch.full((3 * D,), -7, dtype=torch.int32, device="cuda") if with_table else None
        host.append((rc, rm))
        tens.append((c, m, idx, dl, to))
        tup.append((c.data_ptr(), m.data_ptr(), R, idx.data_ptr(), dl.data_ptr(), to.data_ptr() if with_table else 0))
    return host, tens, tup


def _check_batches(oracle_c, w, host, tens, rows, D, table=True):
    for (rc, rm), (c, m, idx, dl, to), R in zip(host, tens, rows):
        o_idx, o_dc, o_dm, o_tab = oracle_c.snapshot(w["free_core"], w["free_mem"], rc, rm, 4)
        assert np.array_equal(idx[:R].cpu().numpy(), o_idx)
        assert (idx[R:].cpu().numpy() == -9).all()
        assert np.array_equal(dl.cpu().numpy(), np.concatenate([o_dc, o_dm]))
        if table:
            assert np.array_equal(to.cpu().numpy(), o_tab)


@pytest.mark.parametrize("name,variant", [("cfg3", 2), ("cfg4", 3), ("cfg4", 2), ("cfg3", 3)])
@pytest.mark.parametrize("K", [1, 3, 20, 64])
def test_multi_batch_launch_equals_separate_calls(name, variant, K, alloc, oracle_c, egpu):
    import torch
    w = egpu.synth.workload(name)
    D = int(w["D"])
    alloc.set_variant(variant)
    alloc.set_table(w["free_core"], w["free_mem"])
    rng = np.random.default_rng(K)
    rows = [int(r) for r in rng.choice([0, 1, 3, 4, 5, 1023, 4096, 20_001, 70_003], K)]
    rows[0] = 70_003
    host, tens, tup = _dev_batches(torch, egpu, w["dist"], range(300, 300 + K), rows, D)
    s = torch.cuda.current_stream().cuda_stream
    n0 = alloc.launch_count
    alloc.bestfit_batches_dev(tup, s)
    torch.cuda.synchronize()
    assert alloc.launch_count - n0 in (1, 2)  # one scan launch (+ one lookup-table build after set_table)
    _check_batches(oracle_c, w, host, tens, rows, D)
    # the table is untouched: a multi-batch launch never commits
    fc, fm, ov = alloc.table()
    assert np.array_equal(fc, w["free_core"]) and np.array_equal(fm, w["free_mem"]) and not ov.any()


@pytest.mark.parametrize("name", ["cfg3", "cfg4"])
def test_multi_batch_launches_pipelined_on_one_stream(name, alloc, oracle_c, egpu):
    """Seven launches of 1..64 batches back to back with EGPU_F_INPUTS_READY: they overlap
    (late wait), cross a group boundary (more than 64 batches in flight) and reuse the ring of
    epilogue slots; one launch rewrites outputs of an earlier one and must be ordered after it."""
    import torch
    w = egpu.synth.workload(name)
    D = int(w["D"])
    alloc.set_table(w["free_core"], w["free_mem"])
    st = torch.cuda.Stream()
    sizes = [20, 64, 7, 64, 33, 1, 50]
    with torch.cuda.stream(st):
        groups = []
        for g, K in enumerate(sizes):
            rows = [30_001 + 4 * k for k in range(K)]
            groups.append((rows,) + _dev_batches(torch, egpu, w["dist"], range(1000 * g, 1000 * g + K), rows, D))
    torch.cuda.synchronize()
    for rows, host, tens, tup in groups:
        alloc.bestfit_batches_dev(tup, st.cuda_stream, inputs_ready=True)
    # same outputs as group 0, other inputs: must land AFTER group 0's results
    rows0, host0, tens0, tup0 = groups[0]
    host_b, tens_b, tup_b = _dev_batches(torch, egpu, w["dist"], range(9000, 9000 + len(rows0)), rows0, D)
    tup_b = [(t[0], t[1], t[2], o[3], o[4], o[5]) for t, o in zip(tup_b, tup0)]
    alloc.bestfit_batches_dev(tup_b, st.cuda_stream, inputs_ready=True)
    torch.cuda.synchronize()
    for rows, host, tens, tup in groups[1:]:
        _check_batches(oracle_c, w, host, tens, rows, D)
    _check_batches(oracle_c, w, host_b, tens0, rows0, D)


def test_multi_batch_rejects_bad_arguments(alloc, egpu):
    import torch
    w = egpu.synth.workload("cfg3")
    alloc.set_table(w["free_core"], w["free_mem"])
    host, tens, tup = _dev_batches(torch, egpu, 3, [1, 2], [1000, 1000], 8)
    with pytest.raises(egpu.EgpuError) as ei:  # two batches write the same index array
        alloc.bestfit_batches_dev([tup[0], (tup[1][0], tup[1][1], 1000, tup[0][3], tup[1][4], tup[1][5])])
    assert ei.value.code == -1
    with pytest.raises(egpu.EgpuError) as ei:
        alloc.bestfit_batches_dev([tup[0]] * 65)
    assert ei.value.code == -1
    with pytest.raises(egpu.EgpuError) as ei:  # misaligned request array
        alloc.bestfit_batches_dev([(tup[0][0] + 4,) + tup[0][1:]])
    assert ei.value.code == -1
    alloc.set_variant(1)
    with pytest.raises(egpu.EgpuError) as ei:  # the literal grid variant has no multi-batch form
        alloc.bestfit_batches_dev(tup)
    assert ei.value.code == -6
    torch.cuda.synchronize()


def test_lookup_scan_with_clustered_memory_values(alloc, oracle_c, egpu):
    """Many distinct free_mem values inside one 64 MiB bucket: the rare walk of the lookup scan."""
    rng = np.random.default_rng(5)
    D = 64
    fc = rng.integers(0, 101, D).astype(np.int32)
    fm = (1000 + rng.permutation(200)[:D]).astype(np.int32)  # 64 distinct values within four buckets
    fm[:5] = [0, 63, 64, 127, (1 << 18) - 1]
    R = 100_003
    rc = rng.integers(0, 101, R).astype(np.int32)
    rm = rng.integers(900, 1300, R).astype(np.int32)
    rm[::7] = rng.integers(-1, (1 << 18) + 2, rm[::7].size)
    for variant in (3, 2):
        alloc.set_variant(variant)
        alloc.set_table(fc, fm)
        idx, dc, dm = alloc.bestfit(rc, rm)
        o_idx, o_dc, o_dm, _ = oracle_c.snapshot(fc, fm, rc, rm, 4)
        assert np.array_equal(idx, o_idx) and np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)


def test_lookup_scan_sums_survive_many_trips(alloc, egpu):
    """Every request lands on one device with the largest addends: the 32-bit shared-memory words
    of the lookup scan must be folded before any field overflows.  A lone lookup launch at
    R >= 16 Mi holds at most 148 x 8 x 2 CTAs of 256 threads, so at R = 2^28 each thread scans
    >= 442 rows = >= 55 trips of 8; without the fold every 32 trips the 12-bit field of a copy
    (<= 3 per add, 4 lanes x 8 rows per trip) would overflow after 42 trips.  3 GiB of HBM."""
    import torch
    D = 64
    fc = np.full(D, 100, dtype=np.int32)
    fm = np.full(D, (1 << 18) - 1, dtype=np.int32)
    fc[1:] = np.arange(1, D) % 100  # device 0 is the only one that takes core = 100
    fc[0] = 100
    fc[1:] = np.minimum(fc[1:], 99)
    R = 1 << 28
    c = torch.full((R,), 100, dtype=torch.int32, device="cuda")
    m = torch.full((R,), (1 << 18) - 1, dtype=torch.int32, device="cuda")
    idx = torch.full((R,), -9, dtype=torch.int32, device="cuda")
    dl = torch.zeros(2 * D, dtype=torch.int64, device="cuda")
    alloc.set_variant(3)
    alloc.set_table(fc, fm)
    alloc.bestfit_dev(c.data_ptr(), m.data_ptr(), R, idx.data_ptr(), dl.data_ptr(), 0, False,
                      torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert bool((idx == 0).all())
    dc, dm = dl[:D].cpu().numpy(), dl[D:].cpu().numpy()
    assert dc[0] == 100 * R and dm[0] == ((1 << 18) - 1) * R and not dc[1:].any() and not dm[1:].any()


def test_query_leaves_the_context_table_alone(alloc, oracle_c, egpu):
    w = egpu.synth.workload("cfg3")
    alloc.set_table(w["free_core"], w["free_mem"])
    rc, rm = egpu.synth.requests(3, 9, 10_001)
    for D in (1, 8, 13, 32, 64):
        rng = np.random.default_rng(D)
        fc = rng.integers(0, 101, D).astype(np.int32)
        fm = rng.integers(0, 1 << 18, D).astype(np.int32)
        got = alloc.query(fc, fm, rc, rm)
        exp, *_ = oracle_c.snapshot(fc, fm, rc, rm, 4)
        assert np.array_equal(got, exp)
    t_fc, t_fm, t_ov = alloc.table()
    assert np.array_equal(t_fc, w["free_core"]) and np.array_equal(t_fm, w["free_mem"]) and not t_ov.any()
    idx, *_ = alloc.bestfit(rc, rm)  # and the context still answers from its own table
    exp, *_ = oracle_c.snapshot(w["free_core"], w["free_mem"], rc, rm, 4)
    assert np.array_equal(idx, exp)


def test_preferred_allocation_does_not_clobber_the_tracked_table(alloc, egpu):
    """The round-1 review: one context that tracks the node's committed table must survive
    GetPreferredAllocation calls (INTEGRATION.md uses a single context)."""
    from elastic_gpu_agent_b200 import plugin
    fc = np.array([100, 40, 75, 10], dtype=np.int32)
    fm = np.array([183359, 9000, 50000, 123], dtype=np.int32)
    alloc.set_table(fc, fm)
    available = ["%d-%02d" % (0, u) for u in range(40, 100)] + ["%d-%02d" % (2, u) for u in range(75, 100)]
    ids, gpu = plugin.preferred_allocation(alloc, available, [], 25, plugin.RESOURCE_CORE)
    assert gpu == 2 and len(ids) == 25
    t_fc, t_fm, t_ov = alloc.table()
    assert np.array_equal(t_fc, fc) and np.array_equal(t_fm, fm) and not t_ov.any()
    assert alloc._lib.egpu_table_size(alloc.handle) == 4


def test_commit_after_a_pipelined_launch_with_table_out(alloc, oracle_c, egpu):
    """A committing launch must not overtake the epilogue of the launch before it: that launch's
    table' is computed from the table as it was (round-1 advisor finding)."""
    import torch
    w = egpu.synth.workload("cfg3")
    D, R = 8, 1 << 20
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        bufs = []
        for k in range(6):
            rc, rm = egpu.synth.requests(3, 40 + k, R)
            rc = np.minimum(rc, 2).astype(np.int32)   # small demands: the committed table stays interesting
            rm = np.minimum(rm, 3).astype(np.int32)
            bufs.append((rc, rm, torch.from_numpy(rc).cuda(), torch.from_numpy(rm).cuda(),
                         torch.empty(R, dtype=torch.int32, device="cuda"), torch.zeros(2 * D, dtype=torch.int64, device="cuda"),
                         torch.full((3 * D,), -7, dtype=torch.int32, device="cuda")))
    torch.cuda.synchronize()
    for trial in range(5):
        alloc.set_table(w["free_core"], w["free_mem"])
        cur_c, cur_m = w["free_core"].copy(), w["free_mem"].copy()
        expect = []
        for k, (rc, rm, c, m, idx, dl, to) in enumerate(bufs):
            commit = k in (2, 4)
            alloc.bestfit_dev(c.data_ptr(), m.data_ptr(), R, idx.data_ptr(), dl.data_ptr(), to.data_ptr(), commit, st.cuda_stream,
                              inputs_ready=True)
            o_idx, o_dc, o_dm, o_tab = oracle_c.snapshot(cur_c, cur_m, rc, rm, 4)
            expect.append((o_idx, o_tab))
            if commit:
                cur_c, cur_m = np.maximum(o_tab[:D], 0), np.maximum(o_tab[D:2 * D], 0)
        torch.cuda.synchronize()
        for (o_idx, o_tab), (_, _, _, _, idx, _, to) in zip(expect, bufs):
            assert np.array_equal(idx.cpu().numpy(), o_idx)
            assert np.array_equal(to.cpu().numpy(), o_tab)


def test_prefix_commit_cut_in_the_ragged_tail_of_a_capped_grid(alloc, oracle_c, egpu):
    """R = 4 * 303105 + 2: with the grid capped, ceil(nvec / tiles) * (tiles - 1) can exceed nvec
    and the last tile holds only the R % 4 tail rows; the capacity crossing is put there."""
    R = 4 * 303105 + 2
    fc = np.array([100, 0, 0, 0, 0, 0, 0, 0], dtype=np.int32)
    fm = np.array([1000, 0, 0, 0, 0, 0, 0, 0], dtype=np.int32)
    rc = np.zeros(R, dtype=np.int32)
    rm = np.zeros(R, dtype=np.int32)
    rm[-2:] = 600  # the second-to-last row fits (600 <= 1000), the last one crosses (1200 > 1000)
    for rpt in (None,):
        alloc.set_table(fc, fm)
        idx, dc, dm = alloc.bestfit(rc, rm, commit=True, prefix_commit=True)
        o_idx, o_dc, o_dm, o_tab = oracle_c.prefix_commit(fc, fm, rc, rm)
        assert np.array_equal(idx, o_idx) and idx[-1] == -2 and idx[-2] == 0
        assert np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)
        t_fc, t_fm, t_ov = alloc.table()
        assert np.array_equal(np.concatenate([t_fc, t_fm, t_ov]), o_tab)


def test_shard_dev_validates_step_and_flags(alloc, egpu):
    import torch
    alloc.set_table([1], [1])
    alloc.peer_attach(0, 1, [alloc.peer_export()])
    c = torch.zeros(8, dtype=torch.int32, device="cuda")
    import ctypes as C
    lib = egpu.load()
    vp = C.c_void_p
    rc = lib.egpu_bestfit_batch_shard_dev(alloc.handle, vp(c.data_ptr()), vp(c.data_ptr()), 4, vp(c.data_ptr()), None, 0,
                                          C.c_uint64(1 << 47), None)
    assert rc == -1
    rc = lib.egpu_bestfit_batch_shard_dev(alloc.handle, vp(c.data_ptr()), vp(c.data_ptr()), 4, vp(c.data_ptr()), None, 4,
                                          C.c_uint64(0), None)  # EGPU_F_PREFIX_COMMIT: use the _prefix entry point
    assert rc == -1
    alloc.peer_detach()


# ---- the all-gather form of the multi-GPU step (what north_star literally names) ----------

@pytest.mark.parametrize("name", ["cfg3", "cfg4"])
@pytest.mark.parametrize("G", [1, 2, 8])
def test_apply_deltas_on_gathered_vectors(name, G, alloc, oracle_c, egpu):
    """egpu_table_apply_deltas_dev on G synthetic gathered demand vectors: table' with and
    without commit, oversubscription flags, against sharding.combine_demands and the oracle."""
    import torch
    from elastic_gpu_agent_b200 import sharding
    w = egpu.synth.workload(name)
    D = int(w["D"])
    R = 20_000
    vecs = []
    tot_c, tot_m = np.zeros(D, np.int64), np.zeros(D, np.int64)
    for g in range(G):
        rc, rm = egpu.synth.requests(w["dist"], 600 + g, R)
        _, dc, dm, _ = oracle_c.snapshot(w["free_core"], w["free_mem"], rc, rm, 4)
        vecs.append(np.concatenate([dc, dm]))
        tot_c += dc
        tot_m += dm
    gathered = np.stack(vecs)
    exp = sharding.combine_demands(w["free_core"], w["free_mem"], gathered)
    assert exp[2 * D:].any()  # the batch oversubscribes some device: the flag path is exercised
    assert np.array_equal(exp[:D], np.clip(w["free_core"].astype(np.int64) - tot_c, -2**31, 2**31 - 1))
    s = torch.cuda.current_stream().cuda_stream
    d_g = torch.from_numpy(gathered.reshape(-1)).cuda()
    tab = torch.full((3 * D,), -7, dtype=torch.int32, device="cuda")
    alloc.set_table(w["free_core"], w["free_mem"])
    alloc.apply_deltas_dev(d_g.data_ptr(), G, tab.data_ptr(), False, s)
    torch.cuda.synchronize()
    assert np.array_equal(tab.cpu().numpy(), exp)
    fc, fm, ov = alloc.table()
    assert np.array_equal(fc, w["free_core"]) and np.array_equal(fm, w["free_mem"]) and not ov.any()
    tab.fill_(-7)
    alloc.apply_deltas_dev(d_g.data_ptr(), G, tab.data_ptr(), True, s)
    torch.cuda.synchronize()
    assert np.array_equal(tab.cpu().numpy(), exp)
    fc, fm, ov = alloc.table()
    assert np.array_equal(fc, np.maximum(exp[:D], 0)) and np.array_equal(fm, np.maximum(exp[D:2 * D], 0))
    assert np.array_equal(ov, exp[2 * D:])
    # the committed table is the one the next scan scores against (sorted view / lookup tables rebuilt)
    rc, rm = egpu.synth.requests(w["dist"], 77, 10_003)
    idx, *_ = alloc.bestfit(rc, rm)
    o_idx, *_ = oracle_c.snapshot(np.maximum(exp[:D], 0), np.maximum(exp[D:2 * D], 0), rc, rm, 4)
    assert np.array_equal(idx, o_idx)


@pytest.mark.parametrize("name", ["cfg3", "cfg4"])
def test_sharded_step_world1_equals_snapshot(name, alloc, oracle_c, egpu):
    """sharding.sharded_step (scan -> all-gather -> apply_deltas) at world = 1, three committing
    steps in a row."""
    import torch
    from elastic_gpu_agent_b200 import sharding
    w = egpu.synth.workload(name)
    D, R = int(w["D"]), 50_003
    alloc.set_table(w["free_core"], w["free_mem"])
    s = torch.cuda.current_stream().cuda_stream
    cur_c, cur_m = w["free_core"].copy(), w["free_mem"].copy()
    for step in range(3):
        rc, rm = egpu.synth.requests(w["dist"], 800 + step, R)
        rc, rm = np.minimum(rc, 3).astype(np.int32), np.minimum(rm, 5).astype(np.int32)
        c, m = torch.from_numpy(rc).cuda(), torch.from_numpy(rm).cuda()
        idx = torch.empty(R + 1, dtype=torch.int32, device="cuda")
        delta = torch.zeros(2 * D, dtype=torch.int64, device="cuda")
        gathered = torch.zeros(2 * D, dtype=torch.int64, device="cuda")
        tab = torch.zeros(3 * D, dtype=torch.int32, device="cuda")
        sharding.sharded_step(alloc, c.data_ptr(), m.data_ptr(), R, idx.data_ptr(), delta, gathered, tab, 1, s, commit=True)
        torch.cuda.synchronize()
        o_idx, o_dc, o_dm, o_tab = oracle_c.snapshot(cur_c, cur_m, rc, rm, 4)
        assert np.array_equal(idx[:R].cpu().numpy(), o_idx)
        assert np.array_equal(gathered.cpu().numpy(), np.concatenate([o_dc, o_dm]))
        assert np.array_equal(tab.cpu().numpy(), o_tab)
        assert np.array_equal(tab.cpu().numpy(), sharding.combine_demands(cur_c, cur_m, gathered.cpu().numpy()[None, :]))
        cur_c, cur_m = np.maximum(o_tab[:D], 0), np.maximum(o_tab[D:2 * D], 0)
    fc, fm, _ = alloc.table()
    assert np.array_equal(fc, cur_c) and np.array_equal(fm, cur_m)


# ---- sharded multi-batch launches + start gate, world = 1 (world = 2: test_gpu_peer_exchange.py) ----

@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("name", ["cfg3", "cfg4"])
def test_world1_sharded_multi_batch_and_gate(name, fused, alloc, oracle_c, egpu):
    """fused = EGPU_F_APPLY: the batch's own last CTA applies its exchange step; otherwise one apply launch."""
    import torch
    w = egpu.synth.workload(name)
    D = int(w["D"])
    alloc.set_table(w["free_core"], w["free_mem"])
    alloc.peer_attach(0, 1, [alloc.peer_export()])
    st, ap = torch.cuda.Stream(), torch.cuda.Stream()
    K, first = 40, 250  # crosses the wrap of the 256 exchange slots
    rows = [25_001 + k for k in range(K)]
    with torch.cuda.stream(st):
        host, tens, tup = _dev_batches(torch, egpu, w["dist"], range(50, 50 + K), rows, D)
    torch.cuda.synchronize()
    # compute-sanitizer makes kernel launches blocking: a gate kernel would wait for a host that is stuck in its launch
    gated = not os.environ.get("EGPU_UNDER_SANITIZER")
    for rep in range(2):  # the second pass reuses the same exchange steps: the first must have consumed its flags
        if gated:
            alloc.gate_dev(st.cuda_stream)
        alloc.bestfit_batches_shard_dev(tup, first, st.cuda_stream, inputs_ready=True, apply=fused)
        if not fused:
            alloc.apply_peers_multi_dev(first, [t[4].data_ptr() for t in tens], False, ap.cuda_stream)
        if gated:
            alloc.gate_open()
        torch.cuda.synchronize()
        assert alloc.peer_last_timeout == 0
        _check_batches(oracle_c, w, host, tens, rows, D)
        for t in tens:
            t[4].fill_(-7)
        torch.cuda.synchronize()
    alloc.peer_detach()


def test_gate_unattached_waits_for_the_host(alloc, egpu):
    import time
    import torch
    alloc.set_table([1], [1])
    st = torch.cuda.Stream()
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    alloc.gate_dev(st.cuda_stream)
    with torch.cuda.stream(st):
        flag.fill_(1)
    time.sleep(0.05)
    assert not st.query()          # still behind the gate
    alloc.gate_open()
    st.synchronize()
    assert int(flag.item()) == 1 and alloc.peer_last_timeout == 0 and alloc.gate_timeouts == 0


def test_gate_that_is_never_opened_gives_up(alloc, egpu):
    """A gate whose host never opens it (what happens when launches are blocking) lets the stream go on after
    ~2 s and is counted; the next gate works again."""
    import time
    import torch
    alloc.set_table([1], [1])
    st = torch.cuda.Stream()
    t0 = time.perf_counter()
    alloc.gate_dev(st.cuda_stream)
    st.synchronize()
    dt = time.perf_counter() - t0
    assert 0.5 < dt < 10 and alloc.gate_timeouts == 1
    alloc.gate_open()                  # the late open belongs to the gate that gave up
    alloc.gate_dev(st.cuda_stream)
    alloc.gate_open()
    st.synchronize()
    assert alloc.gate_timeouts == 1


def test_registered_caller_memory_takes_the_zero_copy_path(alloc, oracle_c, egpu):
    """egpu_host_register: plain caller memory pinned in place; the same call then runs as one launch that
    reads and writes it across PCIe (no staging copies), and the answers are the same."""
    w = egpu.synth.workload("cfg3")
    R = 200_003
    rc, rm = egpu.synth.requests(3, 21, R)
    # page-aligned caller buffers (what C.malloc / mmap give a cgo caller for a large slice)
    def aligned(n):
        raw = np.empty(n * 4 + 4096, dtype=np.uint8)
        off = (-raw.ctypes.data) % 4096
        return raw[off:off + n * 4].view(np.int32), raw
    c, _k1 = aligned(R)
    m, _k2 = aligned(R)
    i, _k3 = aligned(R)
    c[:], m[:] = rc, rm
    o_idx, o_dc, o_dm, _ = oracle_c.snapshot(w["free_core"], w["free_mem"], rc, rm, 4)
    alloc.set_table(w["free_core"], w["free_mem"])
    dc, dm = np.zeros(8, np.int64), np.zeros(8, np.int64)
    alloc.bestfit_raw(c.ctypes.data, m.ctypes.data, R, i.ctypes.data, dc.ctypes.data, dm.ctypes.data)   # pageable: staged
    assert np.array_equal(i, o_idx)
    for a in (c, m, i):
        alloc.host_register(a)
    i[:] = -9
    alloc.bestfit_raw(c.ctypes.data, m.ctypes.data, R, i.ctypes.data, dc.ctypes.data, dm.ctypes.data)   # registered: in place
    assert np.array_equal(i, o_idx) and np.array_equal(dc, o_dc) and np.array_equal(dm, o_dm)
    for a in (c, m, i):
        alloc.host_unregister(a)
    i[:] = -9
    alloc.bestfit_raw(c.ctypes.data, m.ctypes.data, R, i.ctypes.data, dc.ctypes.data, dm.ctypes.data)   # staged again
    assert np.array_equal(i, o_idx)
