"""GPU tests of whole-card requests (DESIGN.md 2.8): egpu_bestfit_cards[_dev] and egpu_replay_cards
against oracle_c on idx, card masks, both demand sums, all 3*D words of table', the committed
table and the sticky oversubscription flag; bit-identity with the single-card entry points when no
row asks for more than one card; restore of what a whole-card churn left placed; and a profiler
run in which every new kernel launches."""
import numpy as np
import pytest

import edge_cases as ec
from oracle import cards_c
from test_cards_oracle import card_requests, full_cards_table

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    return torch


def dev(a, dtype=None):
    torch = _torch()
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return t if dtype is None else t.to(dtype)


def empty(n, dtype):
    torch = _torch()
    return torch.zeros(max(n, 4), dtype=dtype, device="cuda")


def u64(t, n):
    return t[:n].cpu().numpy().view(np.uint64)


def tables(D):
    t = [("full_cards", *full_cards_table(D))]
    for fam in ("ties", "random", "extremes"):
        e = ec.make_table(fam, D)
        t.append((fam, e.fc, e.fm))
    return t


def requests(fc, fm, R, seed):
    rng = np.random.default_rng([fc.size, R, seed])
    rc, rm = card_requests(fc, fm, 256, rng)
    return ec.shape(rc, rm, R, rng)


def expect_commit(cur_fc, cur_fm, cur_ov, tab):
    D = cur_fc.size
    return (np.maximum(tab[:D], 0).astype(np.int32), np.maximum(tab[D:2 * D], 0).astype(np.int32),
            (cur_ov | tab[2 * D:]).astype(np.int32))


@pytest.mark.parametrize("D", ec.D_VALUES)
def test_host_and_lone_device_calls(alloc, D):
    torch = _torch()
    for name, fc, fm in tables(D):
        for R in ec.SIZES:
            rc, rm = requests(fc, fm, R, 1)
            e_idx, e_cards, e_dc, e_dm, e_tab = cards_c.bestfit_cards_snapshot(fc, fm, rc, rm)
            alloc.set_table(fc, fm)
            for want_cards in (True, False):
                idx, cards, dc, dm = alloc.bestfit_cards(rc, rm, cards=want_cards)
                assert np.array_equal(idx, e_idx), (name, R)
                assert not want_cards or np.array_equal(cards, e_cards), (name, R)
                assert np.array_equal(dc, e_dc) and np.array_equal(dm, e_dm), (name, R)
            drc, drm = dev(rc), dev(rm)
            for want_cards in (True, False):
                didx, dcards = empty(R, torch.int32), empty(R, torch.int64)
                ddelta, dtab = empty(2 * D, torch.int64), empty(3 * D, torch.int32)
                alloc.bestfit_cards_dev(drc.data_ptr(), drm.data_ptr(), R, didx.data_ptr(), dcards.data_ptr() if want_cards else 0,
                                        ddelta.data_ptr(), dtab.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
                torch.cuda.synchronize()
                assert np.array_equal(didx[:R].cpu().numpy(), e_idx), (name, R)
                if want_cards:
                    assert np.array_equal(u64(dcards, R), e_cards), (name, R)
                else:
                    assert not dcards.any().item()
                assert np.array_equal(ddelta[:2 * D].cpu().numpy(), np.concatenate([e_dc, e_dm])), (name, R)
                assert np.array_equal(dtab[:3 * D].cpu().numpy(), e_tab), (name, R)
            gfc, gfm, gov = alloc.table()
            assert np.array_equal(gfc, fc) and np.array_equal(gfm, fm) and not gov.any()  # nothing committed


@pytest.mark.parametrize("D", ec.D_VALUES)
def test_pipelined_and_committing_chains(alloc, D):
    torch = _torch()
    stream = torch.cuda.Stream()
    fc, fm = full_cards_table(D, seed=3)
    alloc.set_table(fc, fm)
    # pipelined: INPUTS_READY launches on one stream, each with its own outputs, half without masks
    batches = []
    for k, R in enumerate((1027, 70_001, 5, 1027, 3, 70_001, 1)):
        rc, rm = requests(fc, fm, R, 10 + k)
        batches.append((rc, rm, dev(rc), dev(rm), empty(R, torch.int32), empty(R, torch.int64), empty(2 * D, torch.int64),
                        empty(3 * D, torch.int32)))
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        for k, (rc, rm, drc, drm, didx, dcards, ddelta, dtab) in enumerate(batches):
            alloc.bestfit_cards_dev(drc.data_ptr(), drm.data_ptr(), rc.size, didx.data_ptr(), dcards.data_ptr() if k % 2 else 0,
                                    ddelta.data_ptr(), dtab.data_ptr(), stream=stream.cuda_stream, inputs_ready=True)
    stream.synchronize()
    for k, (rc, rm, drc, drm, didx, dcards, ddelta, dtab) in enumerate(batches):
        e_idx, e_cards, e_dc, e_dm, e_tab = cards_c.bestfit_cards_snapshot(fc, fm, rc, rm)
        assert np.array_equal(didx[:rc.size].cpu().numpy(), e_idx), k
        if k % 2:
            assert np.array_equal(u64(dcards, rc.size), e_cards), k
        assert np.array_equal(ddelta[:2 * D].cpu().numpy(), np.concatenate([e_dc, e_dm])), k
        assert np.array_equal(dtab[:3 * D].cpu().numpy(), e_tab), k
    # committing chain: device and host calls alternate; the committed table and the sticky flag follow the oracle
    cur_fc, cur_fm, cur_ov = fc.copy(), fm.copy(), np.zeros(D, np.int32)
    for step in range(4):
        rc, rm = requests(cur_fc, cur_fm, (1027, 70_001, 5, 3)[step], 20 + step)
        e_idx, e_cards, e_dc, e_dm, e_tab = cards_c.bestfit_cards_snapshot(cur_fc, cur_fm, rc, rm)
        if step % 2 == 0:
            drc, drm = dev(rc), dev(rm)
            didx, dcards = empty(rc.size, torch.int32), empty(rc.size, torch.int64)
            ddelta, dtab = empty(2 * D, torch.int64), empty(3 * D, torch.int32)
            torch.cuda.synchronize()  # inputs and zeroed outputs were made on torch's stream
            with torch.cuda.stream(stream):
                alloc.bestfit_cards_dev(drc.data_ptr(), drm.data_ptr(), rc.size, didx.data_ptr(), dcards.data_ptr(), ddelta.data_ptr(),
                                        dtab.data_ptr(), commit=True, stream=stream.cuda_stream, inputs_ready=True)
            stream.synchronize()
            idx, cards = didx[:rc.size].cpu().numpy(), u64(dcards, rc.size)
            assert np.array_equal(ddelta[:2 * D].cpu().numpy(), np.concatenate([e_dc, e_dm])) and np.array_equal(
                dtab[:3 * D].cpu().numpy(), e_tab), step
        else:
            idx, cards, dc, dm = alloc.bestfit_cards(rc, rm, commit=True)
            assert np.array_equal(dc, e_dc) and np.array_equal(dm, e_dm), step
        assert np.array_equal(idx, e_idx) and np.array_equal(cards, e_cards), step
        cur_fc, cur_fm, cur_ov = expect_commit(cur_fc, cur_fm, cur_ov, e_tab)
        gfc, gfm, gov = alloc.table()
        assert np.array_equal(gfc, cur_fc) and np.array_equal(gfm, cur_fm) and np.array_equal(gov, cur_ov), step


@pytest.mark.parametrize("D", [1, 8, 9, 17, 33, 64])
def test_single_card_batches_are_bit_identical_to_bestfit_batch(alloc, D):
    torch = _torch()
    e = ec.make_table("ties", D)
    rc, rm = ec.edge_requests(e, 70_001)
    rc = np.where(rc > 100, 127, rc).astype(np.int32)
    alloc.set_table(e.fc, e.fm)
    drc, drm = dev(rc), dev(rm)
    outs = []
    for cards_call in (False, True):
        didx, ddelta, dtab = empty(rc.size, torch.int32), empty(2 * D, torch.int64), empty(3 * D, torch.int32)
        sh = torch.cuda.current_stream().cuda_stream
        if cards_call:
            alloc.bestfit_cards_dev(drc.data_ptr(), drm.data_ptr(), rc.size, didx.data_ptr(), 0, ddelta.data_ptr(), dtab.data_ptr(),
                                    stream=sh)
        else:
            alloc.bestfit_dev(drc.data_ptr(), drm.data_ptr(), rc.size, didx.data_ptr(), ddelta.data_ptr(), dtab.data_ptr(), stream=sh)
        torch.cuda.synchronize()
        outs.append((didx.cpu().numpy(), ddelta.cpu().numpy(), dtab.cpu().numpy()))
    for x, y in zip(*outs):
        assert np.array_equal(x, y)
    h1 = alloc.bestfit(rc, rm)
    h2 = alloc.bestfit_cards(rc, rm, cards=False)
    assert np.array_equal(h1[0], h2[0]) and np.array_equal(h1[1], h2[2]) and np.array_equal(h1[2], h2[3])
    kind, a, b = ec_churn(D, 0.0, 20_000)
    fc, fm = np.full(D, 100, np.int32), np.full(D, 40_000, np.int32)
    alloc.set_table(fc, fm)
    r1 = alloc.replay(kind, a, b)
    t1 = alloc.table()
    alloc.set_table(fc, fm)
    r2, _ = alloc.replay_cards(kind, a, b)
    t2 = alloc.table()
    assert np.array_equal(r1, r2) and all(np.array_equal(x, y) for x, y in zip(t1, t2))


def ec_churn(D, whole_share, E, seed=5):
    """cfg5 churn with a share of its ALLOCs turned into whole-card requests of 2..min(D, 8) cards, mem 0"""
    from elastic_gpu_agent_b200 import synth
    kind, a, b = synth.churn_events(seed, E)
    rng = np.random.default_rng([D, E, seed])
    whole = (kind == 0) & (rng.random(E) < whole_share)
    a, b = a.copy(), b.copy()
    a[whole] = 100 * rng.integers(2, max(3, min(D, 8) + 1), int(whole.sum()))
    b[whole] = 0
    return kind, a.astype(np.int32), b.astype(np.int32)


@pytest.mark.parametrize("E", [50_000, 204_801])
@pytest.mark.parametrize("D", [1, 8, 9, 32, 33, 64])
def test_replay_cards_matches_oracle(alloc, D, E):
    kind, a, b = ec_churn(D, 0.05, E)
    fc, fm = np.full(D, 100, np.int32), np.full(D, 183_359, np.int32)
    alloc.set_table(fc, fm)
    got, cards = alloc.replay_cards(kind, a, b)
    e_idx, e_cards, efc, efm = cards_c.replay_cards(fc, fm, kind, a, b)
    assert np.array_equal(got, e_idx) and np.array_equal(cards, e_cards)
    gfc, gfm, _ = alloc.table()
    assert np.array_equal(gfc, efc) and np.array_equal(gfm, efm)
    if D >= 8:
        assert any(bin(int(c)).count("1") > 1 for c in e_cards), "no whole-card ALLOC was placed"
    # the table it leaves is sorted again: a scan right after sees it
    rc, rm = np.array([200, 100, 50], np.int32), np.array([0, 10, 10], np.int32)
    idx, _, dc, dm = alloc.bestfit_cards(rc, rm)
    x = cards_c.bestfit_cards_snapshot(efc, efm, rc, rm)
    assert np.array_equal(idx, x[0]) and np.array_equal(dc, x[2]) and np.array_equal(dm, x[3])


def test_restore_after_whole_card_churn_equals_live_table(alloc):
    """cfg5-style churn with whole-card ALLOCs (mem 0) through egpu_replay_cards; the persisted state of
    what is still placed (a whole-card ALLOC = one core record of 100*k IDs with k links) is restored on a
    fresh table and must equal the live table."""
    from elastic_gpu_agent_b200 import restore
    from oracle import restore_py as RP
    D, mem_cap = 8, 4096
    kind, a, b = ec_churn(D, 0.1, 3000, seed=7)
    b = np.minimum(b, mem_cap // 4).astype(np.int32)
    # then every ALLOC the churn left issued is freed and a few whole-card and single-card pods arrive,
    # so that whole-card ALLOCs are held at the end whatever the churn did
    freed = set(a[kind == 1].tolist())
    issued = [i for i in range(kind.size) if kind[i] == 0 and i not in freed]
    tail = [(1, i, 0) for i in issued] + [(0, 300, 0), (0, 30, 100), (0, 200, 0), (0, 50, 200)]
    kind = np.concatenate([kind, np.array([t[0] for t in tail], np.int32)])
    a = np.concatenate([a, np.array([t[1] for t in tail], np.int32)])
    b = np.concatenate([b, np.array([t[2] for t in tail], np.int32)])
    cap_core, cap_mem = np.full(D, 100, np.int32), np.full(D, mem_cap, np.int32)
    alloc.set_table(cap_core, cap_mem)
    out, cards = alloc.replay_cards(kind, a, b)
    live_fc, live_fm, _ = alloc.table()
    live = {}
    for i in range(kind.size):
        if kind[i] == 0 and out[i] >= 0:
            live[i] = i
        elif kind[i] == 1 and out[i] >= 0:
            live.pop(int(a[i]), None)
    held = [i for i in sorted(live)]
    assert any(a[i] > 100 for i in held), "churn left no whole-card ALLOC placed"
    rng = np.random.default_rng(3)
    core_pool, mem_pool = rng.permutation(D * 100), rng.permutation(D * mem_cap)
    cp = mp = 0
    records, links = [], []
    for n, i in enumerate(held):
        gpus = [d for d in range(D) if (int(cards[i]) >> d) & 1]
        gpus.sort(key=lambda d: d != out[i])  # link 0 = the first card
        containers = {}
        take = core_pool[cp:cp + a[i]]
        cp += a[i]
        ids = ["%d-%02d" % (int(t) // 100, int(t) % 100) for t in take]
        containers["core"] = (ids, RP.CORE)
        links += [("elastic-gpu-%s-%d" % (RP.device_hash(ids), j), "/dev/nvidia%d" % g) for j, g in enumerate(gpus)]
        if b[i] > 0:
            take = mem_pool[mp:mp + b[i]]
            mp += b[i]
            ids = ["%d-%02d" % (int(t) // mem_cap, int(t) % mem_cap) for t in take]
            containers["mem"] = (ids, RP.MEM)
            links.append(("elastic-gpu-%s-0" % RP.device_hash(ids), "/dev/nvidia%d" % out[i]))
        records.append(RP.marshal_record("default", "pod-%d" % n, containers))
    fc, fm, ov, counts, _ = restore.restore_table(alloc, records, links, cap_core, cap_mem)
    assert counts[1:].sum() == 0
    assert np.array_equal(fc, live_fc) and np.array_equal(fm, live_fm) and not ov.any()


def test_profiler_sees_every_new_kernel(alloc, tmp_path):
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for D in (8, 16, 32, 64):
            fc, fm = full_cards_table(D)
            alloc.set_table(fc, fm)
            alloc.bestfit_cards(*requests(fc, fm, 1027, 0))
        alloc.replay_cards(*ec_churn(8, 0.1, 500))
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    for DT, T in ((8, 256), (16, 256), (32, 256), (64, 128)):
        assert any(f"cards_scan_kernel<{DT}, {T}>" in n for n in names), (DT, sorted(names))
    assert any("replay_cards_kernel" in n for n in names), sorted(names)
