"""CPU tests: the generators of tests/edge_cases.py keep the properties they are named after, and
the two oracle restatements agree on every edge case the kernel tests feed them (indices, demand
sums and table', saturated table' and int32-extreme requests included).  This checks the
reference before the GPU is compared with it."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import edge_cases as E  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("family", E.TABLE_FAMILIES)
@pytest.mark.parametrize("D", E.D_VALUES)
def test_table_families_keep_their_property(family, D):
    t = E.make_table(family, D)
    assert t.fc.shape == t.fm.shape == (D,)
    E.check_claims(t)


def test_lut_overflow_layouts_reach_capacity():
    """two thresholds in each of 32 buckets is the most DevLut::ovf can hold; 64 in one bucket is
    the densest block"""
    t = E.make_table("lut_blocks", 64)
    assert E.lut_multi_buckets(t.fm) == E.LUT_OVF_BLOCKS
    v = np.unique(t.fm)
    assert (np.bincount(v >> 6)[np.unique(v >> 6)] == 2).all()
    t = E.make_table("lut_one_bucket", 64)
    assert np.unique(t.fm >> 6).size == 1 and np.unique(t.fm).size == 64


@pytest.mark.parametrize("D", E.D_VALUES)
def test_request_families_cover_their_edges(D):
    rng = np.random.default_rng(D)
    t = E.make_table("random", D)
    tc, tm = E.thresholds(t.fc, t.fm)
    pairs = set(zip(tc.tolist(), tm.tolist()))
    for c, m in zip(t.fc.tolist(), t.fm.tolist()):
        assert {(c, m), (c, m + 1), (c + 1, m), (0, 0), (c, 0), (0, m)} <= pairs
        assert {(0, m & ~63), (0, m | 63), (0, (m | 63) + 1)} <= pairs
    oc, om = E.out_of_domain(rng)
    got = set(zip(oc.tolist(), om.tolist()))
    assert {(c, m) for c in E.BAD_CORES for m in E.BAD_MEMS} <= got
    for R in E.SIZES:
        rc, rm = E.edge_requests(t, R)
        assert rc.shape == rm.shape == (R,) and rc.dtype == rm.dtype == np.int32
        if R >= 1027:  # every edge row is in, shuffled
            assert pairs | {(c, m) for c in E.BAD_CORES for m in E.BAD_MEMS} <= set(zip(rc.tolist(), rm.tolist()))


def _agree(oracle_c, oracle_np, fc, fm, rc, rm, what):
    a = oracle_c.snapshot(fc, fm, rc, rm, 4)
    b = oracle_np.snapshot(fc, fm, rc, rm)
    for name, x, y in zip(("idx", "delta_core", "delta_mem", "table'"), a, b):
        assert np.array_equal(x, y), f"{what}: {name}"
    return a


@pytest.mark.parametrize("D", E.D_VALUES)
def test_oracles_agree_on_edge_cases(D, oracle_c, oracle_np):
    for family in E.TABLE_FAMILIES:
        t = E.make_table(family, D)
        for R in E.SIZES:
            rc, rm = E.edge_requests(t, R)
            _agree(oracle_c, oracle_np, t.fc, t.fm, rc, rm, (family, R))
            if R <= 1027:
                a = oracle_c.prefix_commit(t.fc, t.fm, rc, rm)
                b = oracle_np.prefix_commit(t.fc, t.fm, rc, rm)
                assert all(np.array_equal(x, y) for x, y in zip(a, b)), (family, R, "prefix-commit")


def test_oracles_agree_on_saturated_table(oracle_c, oracle_np):
    """table' = table - demand saturates to int32 in both restatements"""
    # memory: 20 000 rows of (0, 2^18-1) on one device
    fc, fm = np.array([100, 0, 50], np.int32), np.array([5, E.MEM_MAX, 7], np.int32)
    rc = np.zeros(20_000, np.int32)
    rm = np.full(20_000, E.MEM_MAX, np.int32)
    idx, dc, dm, tab = _agree(oracle_c, oracle_np, fc, fm, rc, rm, "mem")
    assert (idx == 1).all() and dm[1] == 20_000 * E.MEM_MAX
    assert tab.tolist() == [100, 0, 50, 5, E.I32_MIN, 7, 0, 1, 0]
    # core: 2^25 rows of core 100
    R = 1 << 25
    fc, fm = np.array([99, 100], np.int32), np.array([E.MEM_MAX, 7], np.int32)
    idx, dc, dm, tab = _agree(oracle_c, oracle_np, fc, fm, np.full(R, 100, np.int32), np.zeros(R, np.int32), "core")
    assert dc.tolist() == [0, 100 * R] and tab.tolist() == [99, E.I32_MIN, E.MEM_MAX, 7, 0, 1]


@pytest.mark.parametrize("D", [4, 9, 33, 64])
def test_oracles_agree_on_one_dimension_oversubscription(D, oracle_c, oracle_np):
    fc, fm = E.role_table(D)
    rng = np.random.default_rng(D)
    for turn in range(4):
        roles = [E.ROLES[(d + turn) % 4] for d in range(D)]
        rc, rm = E.role_requests(D, roles, 4099, rng)
        _, _, _, tab = _agree(oracle_c, oracle_np, fc, fm, rc, rm, turn)
        E.check_roles(roles, fc, fm, tab)


def test_packed_words_decode_to_the_requests_they_pack(egpu):
    rng = np.random.default_rng(7)
    rc, rm = E.random_requests(rng, 10_000)
    oc, om = E.out_of_domain(rng)
    rc, rm = np.concatenate([rc, oc]), np.concatenate([rm, om])
    uc, um = E.unpack_words(egpu.BestFitAllocator.pack_requests(rc, rm))
    inside = (rc >= 0) & (rc <= 127) & (rm >= 0) & (rm <= E.MEM_MAX)
    assert np.array_equal(uc[inside], rc[inside]) and np.array_equal(um[inside], rm[inside])
    assert (uc[~inside] == -1).all() and (um[~inside] == -1).all()
    uc, um = E.unpack_words(E.raw_packed_words(rng))
    assert (uc[:5].tolist(), um[:5].tolist()) == ([0, 127, -1, 101, -1], [0, E.MEM_MAX, -1, 0, -1])
    assert (uc[7:] == -1).all()


def test_scan_kernel_list_matches_the_library():
    """the 23 scan instantiations the GPU coverage test expects are exactly the library's"""
    lib = os.path.join(ROOT, "elastic-gpu-agent_b200", "lib", "libegpu_alloc.so")
    tool = shutil.which("cuobjdump") or (os.path.exists("/usr/local/cuda/bin/cuobjdump") and "/usr/local/cuda/bin/cuobjdump")
    if not os.path.exists(lib) or not tool:
        pytest.skip("needs the built library and cuobjdump")
    out = subprocess.run([tool, "-symbols", lib], check=True, capture_output=True, text=True).stdout
    names = {E.canonical_kernel(tok) for tok in out.split() if tok.startswith("_ZN4egpu")}
    names.discard(None)
    assert len(E.SCAN_KERNELS) == 23 and names == set(E.SCAN_KERNELS)


@pytest.mark.parametrize("family", E.TABLE_FAMILIES)
@pytest.mark.parametrize("D", [d for d in E.D_VALUES if d >= 33])
def test_commit_chain_ties_across_32(family, D, oracle_c):
    """The commit chain of the kernel tests leaves identical rows on both sides of sorted position
    32 in a table that a later step of the chain scans."""
    cur_c, cur_m = E.make_table(family, D)[1:3]
    rng = np.random.default_rng(D)
    straddled = False
    for step in range(3):
        rc, rm = E.chain_requests(cur_c, cur_m, step, rng)
        assert rc.size % 4
        tab = oracle_c.snapshot(cur_c, cur_m, rc, rm)[3]
        cur_c, cur_m = np.maximum(tab[:D], 0), np.maximum(tab[D:2 * D], 0)
        straddled |= E.tie_across_32(cur_c, cur_m)
    assert straddled
