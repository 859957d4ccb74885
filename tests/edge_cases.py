"""Edge-case generators shared by the oracle and kernel tests (not a test module).

Tables come in families, each built for any D in 1..64.  Every family returns its table with
the property it was built for (`EdgeTable.claims`), and the tests assert those claims, so a
family cannot quietly stop exercising what it is named after:

  ties            fc in {0, 1, 99, 100}, fm in {0, 1, 63, 64, 65, 2^18-1}: duplicate rows; for
                  D >= 33 identical rows sit on both sides of sorted position 32, where the
                  register scan splits its 64 rows into two halves of 32
  lut_blocks      distinct fm values two per 64 MiB bucket: every used bucket needs a block of
                  the lookup table's overflow area (DevLut::ovf); D = 64 fills all 32 blocks
  lut_one_bucket  up to 64 distinct fm values in ONE bucket (one block, every rank in it)
  extremes        (0, 0), (100, 2^18-1), (100, 0), (0, 2^18-1), then random rows
  random          uniform rows

Request families for a table: `thresholds` (requests exactly at, and one past, every row's
capacity, and the bucket edges around every fm), `out_of_domain` (int32 extremes and values
just outside the domain, which go through the unsigned clamps of the kernels), and `shape`,
which shuffles rows and pads them with random ones to a given (ragged) batch size.
"""
from __future__ import annotations

import re
import zlib
from typing import NamedTuple

import numpy as np

CORE_MAX = 100
MEM_MAX = (1 << 18) - 1
I32_MIN = -(1 << 31)
I32_MAX = (1 << 31) - 1
MAX_ROWS = I32_MAX  # EGPU_MAX_ROWS

D_VALUES = (1, 2, 8, 9, 16, 17, 31, 32, 33, 63, 64)
TABLE_FAMILIES = ("ties", "lut_blocks", "lut_one_bucket", "extremes", "random")
SIZES = (1, 3, 5, 1027, 70_001)  # ragged: none is a multiple of 4

TIE_CORES = (0, 1, 99, 100)
TIE_MEMS = (0, 1, 63, 64, 65, MEM_MAX)
BAD_CORES = (I32_MIN, -1, 101, 127, 128, I32_MAX)
BAD_MEMS = (I32_MIN, -1, 1 << 18, 1 << 25, I32_MAX)
LUT_OVF_BLOCKS = 32  # DevLut::ovf holds (kMaxD / 2) blocks of 64 ranks


class EdgeTable(NamedTuple):
    family: str
    fc: np.ndarray  # int32[D]
    fm: np.ndarray  # int32[D]
    claims: dict


def _rng(*key) -> np.random.Generator:
    """a generator seeded by the key (strings by CRC: stable across processes, unlike hash())"""
    return np.random.default_rng([zlib.crc32(k.encode()) if isinstance(k, str) else int(k) for k in key])


def sorted_rows(fc, fm) -> list[tuple[int, int, int]]:
    """rows in the scans' order: by (free_core, free_mem, device)"""
    return sorted((int(c), int(m), d) for d, (c, m) in enumerate(zip(fc, fm)))


def has_duplicates(fc, fm) -> bool:
    return len(set(zip(np.asarray(fc).tolist(), np.asarray(fm).tolist()))) < len(fc)


def tie_across_32(fc, fm) -> bool:
    """identical rows at sorted positions 31 and 32"""
    rows = sorted_rows(fc, fm)
    return len(rows) >= 33 and rows[31][:2] == rows[32][:2]


def lut_multi_buckets(fm) -> int:
    """Buckets (fm >> 6) that hold two or more distinct fm values: each takes one block of
    DevLut::ovf.  Counted the way lut_build_kernel counts them."""
    v = np.unique(np.asarray(fm, dtype=np.int64))
    _, n = np.unique(v >> 6, return_counts=True)
    return int((n >= 2).sum())


def _ties(D: int, rng) -> tuple[np.ndarray, np.ndarray]:
    pairs = [(c, m) for c in TIE_CORES for m in TIE_MEMS]
    if D < 33:
        pick = rng.integers(0, len(pairs), D)
        if D >= 2:
            pick[-1] = pick[0]  # at least one duplicate
        rows = [pairs[i] for i in pick]
    else:
        # 30 rows below p, copies of p on sorted positions 30..33 (31 and 32 among them), the rest above
        p = (99, 64)
        below = [q for q in pairs if q < p]
        above = [q for q in pairs if q > p]
        n_p = min(4, D - 30)
        rows = [below[i] for i in rng.integers(0, len(below), 30)] + [p] * n_p
        rows += [above[i] for i in rng.integers(0, len(above), D - 30 - n_p)]
    rows = [rows[i] for i in rng.permutation(D)]
    return np.array([r[0] for r in rows], np.int32), np.array([r[1] for r in rows], np.int32)


def _lut_blocks(D: int, rng) -> np.ndarray:
    # D // 2 buckets with two distinct values each (+ one bucket with one when D is odd); the
    # first and the last in-domain bucket are always among them
    nb = (D + 1) // 2
    buckets = rng.choice(np.arange(1, MEM_MAX >> 6), size=nb, replace=False)
    if nb >= 2:
        buckets[0], buckets[1] = 0, MEM_MAX >> 6
    vals = []
    for k, b in enumerate(buckets):
        offs = rng.choice(64, size=2, replace=False)
        if k == 0:
            offs = np.array([0, 63])  # both edges of a bucket
        vals += [int(b) * 64 + int(o) for o in offs]
    return rng.permutation(np.array(vals[:D], np.int32))


def make_table(family: str, D: int, seed: int = 0) -> EdgeTable:
    rng = _rng(family, D, seed)
    fc = rng.integers(0, CORE_MAX + 1, D).astype(np.int32)
    if family == "ties":
        fc, fm = _ties(D, rng)
        claims = {"duplicates": D >= 2, "tie_across_32": D >= 33}
    elif family == "lut_blocks":
        fm = _lut_blocks(D, rng)
        claims = {"distinct_fm": D, "multi_buckets": D // 2}
    elif family == "lut_one_bucket":
        b = int(rng.integers(0, (MEM_MAX >> 6) + 1))
        fm = (b * 64 + rng.permutation(64)[:D]).astype(np.int32)
        claims = {"distinct_fm": D, "multi_buckets": 1 if D >= 2 else 0}
    elif family == "extremes":
        fm = rng.integers(0, MEM_MAX + 1, D).astype(np.int32)
        ext = [(0, 0), (CORE_MAX, MEM_MAX), (CORE_MAX, 0), (0, MEM_MAX)]
        for d, (c, m) in enumerate(ext[:D]):
            fc[d], fm[d] = c, m
        claims = {"extreme_rows": min(D, 4)}
    elif family == "random":
        fm = rng.integers(0, MEM_MAX + 1, D).astype(np.int32)
        claims = {}
    else:
        raise ValueError(family)
    return EdgeTable(family, fc.astype(np.int32), fm.astype(np.int32), claims)


def check_claims(t: EdgeTable) -> None:
    """the property each family is built for (raises AssertionError)"""
    fc, fm, D = t.fc, t.fm, t.fc.size
    assert ((fc >= 0) & (fc <= CORE_MAX) & (fm >= 0) & (fm <= MEM_MAX)).all(), "table outside the domain"
    c = t.claims
    if t.family == "ties":
        assert set(fc.tolist()) <= set(TIE_CORES) and set(fm.tolist()) <= set(TIE_MEMS)
        assert has_duplicates(fc, fm) == c["duplicates"]
        if c["tie_across_32"]:
            assert tie_across_32(fc, fm)
    if "distinct_fm" in c:
        assert np.unique(fm).size == c["distinct_fm"]
    if "multi_buckets" in c:
        assert lut_multi_buckets(fm) == c["multi_buckets"] <= LUT_OVF_BLOCKS
    if "extreme_rows" in c:
        ext = [(0, 0), (CORE_MAX, MEM_MAX), (CORE_MAX, 0), (0, MEM_MAX)]
        assert list(zip(fc[:c["extreme_rows"]].tolist(), fm[:c["extreme_rows"]].tolist())) == ext[:c["extreme_rows"]]


# ---- requests -------------------------------------------------------------------------------

def thresholds(fc, fm) -> tuple[np.ndarray, np.ndarray]:
    """Per row: (fc, fm), (fc, fm + 1), (fc + 1, fm), (0, 0), (fc, 0), (0, fm).  Per distinct fm:
    the first and last value of its 64 MiB bucket and the values just outside it."""
    fc = np.asarray(fc, np.int64)
    fm = np.asarray(fm, np.int64)
    z = np.zeros_like(fc)
    cores = [fc, fc, fc + 1, z, fc, z]
    mems = [fm, fm + 1, fm, z, z, fm]
    v = np.unique(fm)
    lo, hi = v & ~63, v | 63
    for m in (lo, hi, lo - 1, hi + 1):
        cores.append(np.zeros_like(m))
        mems.append(m)
    rc, rm = np.concatenate(cores), np.concatenate(mems)
    ok = rm >= 0
    return rc[ok].astype(np.int32), rm[ok].astype(np.int32)


def out_of_domain(rng, n_valid: int = 32) -> tuple[np.ndarray, np.ndarray]:
    """every bad core with every bad mem, each bad value next to an in-domain one, and in-domain rows"""
    cores, mems = [], []
    for c in BAD_CORES:
        for m in BAD_MEMS:
            cores.append(c)
            mems.append(m)
        cores += [c, c]
        mems += [0, int(rng.integers(0, MEM_MAX + 1))]
    for m in BAD_MEMS:
        cores += [0, int(rng.integers(0, CORE_MAX + 1))]
        mems += [m, m]
    cores += rng.integers(0, CORE_MAX + 1, n_valid).tolist()
    mems += rng.integers(0, 1 << 12, n_valid).tolist()
    return np.array(cores, np.int64).astype(np.int32), np.array(mems, np.int64).astype(np.int32)


def random_requests(rng, n: int) -> tuple[np.ndarray, np.ndarray]:
    """mostly in-domain, many small enough to fit, a few just outside"""
    rc = rng.integers(-1, CORE_MAX + 3, n).astype(np.int32)
    rm = rng.integers(-1, (1 << 18) + 2, n).astype(np.int32)
    small = rng.random(n) < 0.5
    rm[small] = rng.integers(0, 1 << 12, int(small.sum()))
    return rc, rm


def shape(rc, rm, R: int, rng) -> tuple[np.ndarray, np.ndarray]:
    """the rows shuffled, padded with random rows (or subsampled) to exactly R rows"""
    n = rc.size
    if n >= R:
        keep = rng.choice(n, size=R, replace=False)
        return rc[keep].copy(), rm[keep].copy()
    pc, pm = random_requests(rng, R - n)
    c, m = np.concatenate([rc, pc]), np.concatenate([rm, pm])
    p = rng.permutation(R)
    return c[p].astype(np.int32), m[p].astype(np.int32)


def edge_requests(t: EdgeTable, R: int, seed: int = 0) -> tuple[np.ndarray, np.ndarray]:
    """thresholds of the table + out-of-domain rows, shaped to R rows"""
    rng = _rng("req", t.family, t.fc.size, R, seed)
    tc, tm = thresholds(t.fc, t.fm)
    oc, om = out_of_domain(rng)
    return shape(np.concatenate([tc, oc]), np.concatenate([tm, om]), R, rng)


# ---- oversubscription patterns -----------------------------------------------------------------

ROLES = ("none", "core", "mem", "both")


def role_table(D: int) -> tuple[np.ndarray, np.ndarray]:
    """Device d has fc = d + 2 and fm = 2000 + 1000 d: both grow with d, so a request
    (fc_d, m <= fm_d) and a request (1, fm_d) both have device d as their best fit."""
    d = np.arange(D)
    return (d + 2).astype(np.int32), (2000 + 1000 * d).astype(np.int32)


def role_requests(D: int, roles, R: int, rng) -> tuple[np.ndarray, np.ndarray]:
    """Requests that oversubscribe device d in core only, in memory only, in both or not at all
    (roles[d]), shuffled among infeasible rows up to R rows.  For role_table(D)."""
    fc, fm = role_table(D)
    cores, mems = [], []
    for d, role in enumerate(roles):
        c, m = int(fc[d]), int(fm[d])
        pair = {"none": [], "core": [(c, 1), (c, 1)], "mem": [(1, m), (1, m)], "both": [(c, m), (c, m)]}[role]
        for q in pair:
            cores.append(q[0])
            mems.append(q[1])
    n = R - len(cores)
    assert n >= 0
    bad = rng.integers(0, 3, n)  # infeasible on any table: core or mem just outside the domain, or negative
    cores += np.where(bad == 0, CORE_MAX + 1, np.where(bad == 1, 0, -1)).tolist()
    mems += np.where(bad == 1, MEM_MAX + 1, 0).tolist()
    p = rng.permutation(R)
    return np.array(cores, np.int32)[p], np.array(mems, np.int32)[p]


def spread_roles(D: int) -> list[str]:
    """one device over in core only, one in memory only, one in both, one untouched (never device D - 1)"""
    roles = ["none"] * D
    for k, role in enumerate(("core", "mem", "both", "none")):
        roles[(k * (D // 4) + D // 8) % D] = role
    return roles


def chain_requests(cur_c, cur_m, step: int, rng) -> tuple[np.ndarray, np.ndarray]:
    """Batch `step` of a commit chain: the exact rows of the next third of the devices in sorted
    order, which empties them, and out-of-domain rows; a ragged number of rows.  Emptied devices
    pile up as identical (0, 0) rows; from D = 33 on they come to straddle sorted position 32."""
    D = len(cur_c)
    order = [r[2] for r in sorted_rows(cur_c, cur_m)]
    third = -(-D // 3)
    pick = order[(step * third) % D:][:third]
    oc, om = out_of_domain(rng, n_valid=8)
    rc = np.concatenate([np.asarray(cur_c)[pick], oc]).astype(np.int32)
    rm = np.concatenate([np.asarray(cur_m)[pick], om]).astype(np.int32)
    n = rc.size + 1 if (rc.size + 1) % 4 else rc.size + 2
    return shape(rc, rm, n, rng)


def check_roles(roles, fc, fm, table_out) -> None:
    """table' (int32[3D]) shows exactly the oversubscription each device's role asks for"""
    D = len(roles)
    c, m, ov = table_out[:D], table_out[D:2 * D], table_out[2 * D:]
    for d, role in enumerate(roles):
        assert (c[d] < 0) == (role in ("core", "both")) and (m[d] < 0) == (role in ("mem", "both")), (d, role)
        assert ov[d] == (role != "none"), (d, role)


# ---- packed wire format ----------------------------------------------------------------------

def raw_packed_words(rng, n_random: int = 64) -> np.ndarray:
    """edge words of EGPU_PACK_REQUEST's format: 0, the largest in-format word, the first word out of
    format, core 101, EGPU_PACKED_INVALID and random out-of-format words"""
    w = [0, (1 << 25) - 1, 1 << 25, 101 << 18, 0xFFFFFFFF, (100 << 18) | MEM_MAX, (100 << 18) | (MEM_MAX + 1 - 64)]
    w += rng.integers(1 << 25, 1 << 32, n_random, dtype=np.int64).tolist()
    return np.array(w, np.uint32)


def unpack_words(words) -> tuple[np.ndarray, np.ndarray]:
    """the request a packed word stands for: (core, mem), or (-1, -1) for words >= 2^25"""
    w = np.asarray(words, np.int64)
    ok = w < (1 << 25)
    return np.where(ok, w >> 18, -1).astype(np.int32), np.where(ok, w & 0x3FFFF, -1).astype(np.int32)


# ---- the scan kernels of the library -----------------------------------------------------------

# Every scan instantiation: five register-scan forms (sorted, grid, sorted CONTIG, sorted
# multi-batch, packed) for each D bucket (8 / 16 / 32 / 64 rows; 128 threads at 64), and the
# lookup-table scan (single, CONTIG, multi-batch).
_BUCKETS = ((8, 256), (16, 256), (32, 256), (64, 128))
SCAN_KERNELS = tuple(
    [f"bestfit_sorted_kernel<{d},{t},false>" for d, t in _BUCKETS]
    + [f"bestfit_grid_kernel<{d},{t}>" for d, t in _BUCKETS]
    + [f"bestfit_sorted_kernel<{d},{t},true>" for d, t in _BUCKETS]
    + [f"bestfit_sorted_multi_kernel<{d},{t}>" for d, t in _BUCKETS]
    + [f"bestfit_sorted_packed_kernel<{d},{t}>" for d, t in _BUCKETS]
    + ["bestfit_lut_kernel<256,false>", "bestfit_lut_kernel<256,true>", "bestfit_lut_multi_kernel<256>"])
BUCKET_D = {8: 8, 16: 16, 32: 32, 64: 64}  # a D that selects each bucket

_BOOL = {"false": "false", "true": "true", "(bool)0": "false", "(bool)1": "true", "0": "false", "1": "true"}


def canonical_kernel(name: str) -> str | None:
    """'void egpu::bestfit_sorted_kernel<8, 256, false>(egpu::DevState*, ...)' or the mangled symbol
    -> 'bestfit_sorted_kernel<8,256,false>'; None when the name is not a scan kernel"""
    m = re.search(r"_ZN4egpu\d+(bestfit_\w+?_kernel)I((?:L[ib]\d+E)+)E", name)
    if m:
        args = []
        for kind, val in re.findall(r"L([ib])(\d+)E", m.group(2)):
            args.append(val if kind == "i" else ("true" if val == "1" else "false"))
        return f"{m.group(1)}<{','.join(args)}>"
    m = re.search(r"(bestfit_\w+?_kernel)<([^>]*)>", name)
    if not m:
        return None
    args = [a.strip() for a in m.group(2).split(",")]
    args = [_BOOL.get(a, a.rstrip("uU")) for a in args]
    return f"{m.group(1)}<{','.join(args)}>"
