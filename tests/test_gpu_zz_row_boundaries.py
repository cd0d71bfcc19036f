"""`-m gpu`: one call past 2^31 and 2^32 rows, against answers computed exactly in Python (no oracle).

A fragment is a row count plus column pointers, so many fragments may point at the same device buffers.  Each case
builds one or two PHYSICAL fragments (2^24 + 17 rows: not a multiple of any scan chunk), references them `m` times and
adds a prefix view (same pointers, fewer rows, truthful chunk stats) to land on an exact total such as 2^32 - 1 or
2^32.  The expected answer is the physical fragment's own, scaled by `m` with Python integers:

  * COUNT / integer SUM per group: sort by key, np.add.reduceat over int64, times m; SUM wraps to int64 (agg_sum);
  * a COUNT read from a 4-byte slot: the low 32 bits as a signed int32 (ResultSetBufferAccessors.h:246-253);
  * MIN / MAX: the physical fragment's; DOUBLE SUM / AVG: math.fsum times m, within 1e-6 relative.

Which layout the planner picked (kernel, slot widths, keyless) is asserted alongside the rows.  Physical data stays
under 1 GB of device memory; the calls scan between 3e9 and 1e10 rows each.
"""
from __future__ import annotations

import math
import os
import subprocess
import sys

import numpy as np
import pytest

import sqlmini
from heavydb_b200 import abi, executor

pytestmark = pytest.mark.gpu

PHYS = 2**24 + 17
U32_MAX = 2**32 - 1


def _need_device_memory(gb=4):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < gb * 2**30:
        pytest.skip(f"needs about {gb} GB of free device memory, {free / 2**30:.1f} GB free")


def wrap64(x):
    return ((x + 2**63) % 2**64) - 2**63


def wrap32(x):
    return ((x + 2**31) % 2**32) - 2**31


def views(total, phys=PHYS):
    """[(rows, multiplicity)]: full references to a physical fragment plus one prefix view summing to `total`."""
    m, r = divmod(total, phys)
    return [(phys, m)] + ([(r, 1)] if r else [])


class Physical:
    """One physical fragment: host numpy columns and their device copies (`dev`: columns already on the device, None for
    the ones to upload; upload=False keeps the fragment host-only)."""

    def __init__(self, col_types, cols, dev=None, upload=True):
        self.col_types = col_types
        self.host = [np.ascontiguousarray(c) for c in cols]
        self.dev = list(dev) if dev is not None else [None] * len(cols)
        self._stats = {}
        if upload:
            import torch
            self.dev = [d if d is not None else torch.from_numpy(c.view(np.uint8).copy()).cuda() for c, d in zip(self.host, self.dev)]
            torch.cuda.synchronize()

    def stats(self, n):
        """Chunk stats of the first n rows (what a prefix view advertises)."""
        if n not in self._stats:
            self._stats[n] = [abi.chunk_stats(c[:n], t, nn) for c, (t, nn) in zip(self.host, self.col_types)]
        return self._stats[n]

    def table(self, total, device=True):
        """The aliased table of `total` rows: device pointers, or (device=False) the same host arrays again and again."""
        t = abi.Table(self.col_types)
        for n, mult in views(total, len(self.host[0])):
            st = self.stats(n)
            for _ in range(mult):
                fid = len(t.fragments)
                if device:
                    t.add_device_fragment(n, [d.data_ptr() for d in self.dev], st, fragment_id=fid)
                else:
                    t.fragments.append(abi.Fragment(n, host_cols=[c[:n] for c in self.host], stats=list(st), fragment_id=fid))
        assert t.total_tuples() == total
        return t


def grouped(keys, vals, mask, total):
    """{key: [count, sum(vals[0]), ...]} over the aliased table of `total` rows, as exact Python integers (no wrap)."""
    out = {}
    for n, mult in views(total, keys.size):
        sel = mask[:n]
        k = keys[:n][sel]
        order = np.argsort(k, kind="stable")
        ks = k[order]
        if ks.size == 0:
            continue
        starts = np.flatnonzero(np.r_[True, ks[1:] != ks[:-1]])
        counts = np.diff(np.r_[starts, ks.size])
        sums = [np.add.reduceat(v[:n][sel][order].astype(np.int64), starts) for v in vals]
        for i, s in enumerate(starts):
            acc = out.setdefault(int(ks[s]), [0] * (1 + len(vals)))
            acc[0] += int(counts[i]) * mult
            for j, sm in enumerate(sums):
                acc[1 + j] += int(sm[i]) * mult
    return out


def check_plan(rs, kernel, widths, keyless=None):
    p = rs.getQueryMemDesc()
    assert p.kernel == kernel, ("kernel", p.kernel, kernel)
    assert list(p.slot_padded_width[: p.num_slots]) == widths, ("slot widths", list(p.slot_padded_width[: p.num_slots]), widths)
    if keyless is not None:
        assert p.keyless_hash == keyless, ("keyless_hash", p.keyless_hash, keyless)
    return p


def rows_equal(got, want, fp_cols=()):
    """Unordered rows against {key: row}; columns in fp_cols within 1e-6 relative, the rest exact."""
    assert len(got) == len(want), (len(got), len(want), got[:5])
    for row in got:
        exp = want[row[0]]
        assert len(row) == len(exp), (row, exp)
        for c, (a, b) in enumerate(zip(row, exp)):
            if c in fp_cols:
                assert abs(a - b) <= 1e-6 * abs(b), (c, row, exp)
            else:
                assert a == b, (c, row, exp)


def run(table, sql, names, device=True, **kw):
    unit = sqlmini.parse(sql, table, names, bigint_count=kw.pop("bigint_count", False), inner=kw.pop("inner", None))
    eo = executor.execution_options(bigint_count=kw.pop("bigint_count_eo", False), force_kernel=kw.pop("force_kernel", 0))
    guess, card = kw.pop("guess", 0), kw.pop("has_card", False)
    assert not kw
    return executor.Executor().executeWorkUnit(guess, True, table, unit, eo=eo, has_cardinality_estimation=card,
                                               memory_level=abi.GPU_LEVEL if device else abi.CPU_LEVEL)


# ---- the main physical fragment ----------------------------------------------------------------------------------------
# k   TINYINT NOT NULL  : 124/128 of the rows in group 0, 2/128 in group 1, 1/128 each in groups 2 and 3
# t8  TINYINT           : [-100, 100], every 11th row NULL
# i32 INT NOT NULL      : [2^31 - 2^20, 2^31): a sum over 4e9 of them wraps int64, every add carries out of 32 bits
# b64 BIGINT NOT NULL   : [-2^40, 2^40]
# d   DOUBLE NOT NULL   : [0, 1)
NAMES = ["k", "t8", "i32", "b64", "d"]
TYPES = [(abi.kTINYINT, True), (abi.kTINYINT, False), (abi.kINT, True), (abi.kBIGINT, True), (abi.kDOUBLE, True)]
T_BIG = 4_500_000_000          # one group above 2^32 rows
T_MID = 3_000_000_000          # between 2^31 and 2^32


@pytest.fixture(scope="module")
def main_phys():
    _need_device_memory()
    rng = np.random.default_rng(2**31 + 1)
    i = np.arange(PHYS)
    r = i % 128
    k = np.where(r < 124, 0, np.where(r < 126, 1, r - 124)).astype(np.int8)
    t8 = rng.integers(-100, 101, PHYS).astype(np.int8)
    t8[i % 11 == 5] = abi.NULL_TINYINT
    i32 = rng.integers(2**31 - 2**20, 2**31, PHYS).astype(np.int32)
    b64 = rng.integers(-2**40, 2**40 + 1, PHYS).astype(np.int64)
    d = rng.random(PHYS)
    return Physical(TYPES, [k, t8, i32, b64, d])


def _non_grouped_expected(ph, total):
    """NON_GROUPED_SQL's row: 64-bit counts and integer sums, fsum for the DOUBLE column."""
    k, t8, i32, b64, d = ph.host
    cnt = cnt8 = s8 = s32 = 0
    sd = 0.0
    for n, mult in views(total, PHYS):
        sel = d[:n] < 0.97
        nn = sel & (t8[:n] != abi.NULL_TINYINT)
        cnt += int(sel.sum()) * mult
        cnt8 += int(nn.sum()) * mult
        s8 += int(t8[:n][nn].astype(np.int64).sum()) * mult
        s32 += int(i32[:n][sel].astype(np.int64).sum()) * mult
        sd += math.fsum(d[:n][sel]) * mult
    sel = d < 0.97
    nn = sel & (t8 != abi.NULL_TINYINT)
    return (cnt, cnt8, wrap64(s8), int(t8[nn].min()), int(t8[nn].max()), s8 / cnt8,
            wrap64(s32), int(i32[sel].min()), int(i32[sel].max()),
            sd, float(d[sel].min()), float(d[sel].max()), sd / cnt)


NON_GROUPED_SQL = ("SELECT COUNT(*), COUNT(t8), SUM(t8), MIN(t8), MAX(t8), AVG(t8), SUM(i32), MIN(i32), MAX(i32), "
                   "SUM(d), MIN(d), MAX(d), AVG(d) FROM t WHERE d < 0.97;")
NON_GROUPED_FP = (5, 9, 12)


def test_a_non_grouped_past_2_32_rows(main_phys):
    t = main_phys.table(T_BIG)
    rs = run(t, NON_GROUPED_SQL, NAMES)
    check_plan(rs, abi.KERNEL_NON_GROUPED, [8] * 15)
    got = rs.rows()
    want = _non_grouped_expected(main_phys, T_BIG)
    assert want[0] > 2**32 and want[6] < 0              # 64-bit count past 2^32; SUM(i32) of positive values wrapped
    assert len(got) == 1
    rows_equal([(0,) + got[0]], {0: (0,) + want}, fp_cols=tuple(c + 1 for c in NON_GROUPED_FP))


def _grouped_expected(ph, total):
    k, t8, i32, b64, d = ph.host
    g = grouped(k, [i32, b64], np.ones(PHYS, bool), total)
    return {key: (key, c, wrap64(s32), wrap64(s64)) for key, (c, s32, s64) in g.items()}


GROUPED_SQL = "SELECT k, COUNT(*), SUM(i32), SUM(b64) FROM t GROUP BY k;"


@pytest.mark.parametrize("force", [0, abi.KERNEL_PERFECT_GLOBAL], ids=["smem", "forced_global"])
def test_bc_grouped_tinyint_key_group_above_2_32(main_phys, force):
    """(b) the shared-memory table: 32-bit low words in shared memory, carries to HBM; (c) forced onto the HBM/L2 table:
    split lo / hi accumulators.  COUNT(*) alone gets its 8-byte slot from the tuple count (more than UINT32_MAX)."""
    t = main_phys.table(T_BIG)
    rs = run(t, GROUPED_SQL, NAMES, force_kernel=force)
    check_plan(rs, force or abi.KERNEL_PERFECT_SMEM, [8, 8, 8, 8], keyless=1)
    want = _grouped_expected(main_phys, T_BIG)
    assert want[0][1] > 2**32
    assert sum(int(v) for v in main_phys.host[2][main_phys.host[0] == 0]) * (T_BIG // PHYS) >= 2**63   # SUM(i32) of group 0 wraps
    rows_equal(rs.rows(), want)
    rs = run(t, "SELECT k, COUNT(*) FROM t GROUP BY k;", NAMES, force_kernel=force)
    check_plan(rs, force or abi.KERNEL_PERFECT_SMEM, [8, 8])
    rows_equal(rs.rows(), {key: row[:2] for key, row in want.items()})


def test_f_order_by_8_byte_counts(main_phys):
    """ORDER BY COUNT(*) DESC where group 0 (> 2^32 rows) truncated to 32 bits would sort below group 1."""
    t = main_phys.table(T_BIG)
    rs = run(t, "SELECT k, COUNT(*) FROM t GROUP BY k ORDER BY 2 DESC, 1 LIMIT 3;", NAMES)
    check_plan(rs, abi.KERNEL_PERFECT_SMEM, [8, 8])
    g = _grouped_expected(main_phys, T_BIG)
    want = sorted(((key, row[1]) for key, row in g.items()), key=lambda r: (-r[1], r[0]))[:3]
    trunc = sorted(((key, row[1] % 2**32) for key, row in g.items()), key=lambda r: (-r[1], r[0]))[:3]
    assert [r[0] for r in trunc] != [r[0] for r in want]        # the premise of the case
    assert rs.rows() == want


@pytest.mark.parametrize("total,bigint_count,width", [
    (T_MID, False, 4), (U32_MAX, False, 4), (U32_MAX + 1, False, 8), (U32_MAX, True, 8)],
    ids=["3e9", "2^32-1", "2^32", "2^32-1-bigint_count"])
def test_h_count_slot_width_flips_at_2_32(main_phys, total, bigint_count, width):
    """Up to UINT32_MAX tuples COUNT(*) gets a 4-byte slot, which reads back as the reference's signed int32: group 0
    (more than 2^31 rows) comes back negative.  From 2^32 tuples on, or under bigint_count, the slot is 8 bytes."""
    t = main_phys.table(total)
    rs = run(t, "SELECT k, COUNT(*) FROM t GROUP BY k;", NAMES, bigint_count=bigint_count, bigint_count_eo=bigint_count)
    check_plan(rs, abi.KERNEL_PERFECT_SMEM, [width, width])
    g = grouped(main_phys.host[0], [], np.ones(PHYS, bool), total)
    assert g[0][0] > 2**31
    want = {key: (key, wrap32(c[0]) if width == 4 else c[0]) for key, c in g.items()}
    if width == 4:
        assert want[0][1] < 0
    rows_equal(rs.rows(), want)


def test_g_host_columns(main_phys):
    """(a) and (b) with host columns: the same 1-byte numpy arrays appended again and again, staged slice by slice."""
    ph = Physical(TYPES[:2], main_phys.host[:2], upload=False)
    t = ph.table(T_BIG, device=False)
    names = NAMES[:2]
    k, t8 = ph.host
    rs = run(t, "SELECT COUNT(*), COUNT(t8), SUM(t8), MIN(t8), MAX(t8), AVG(t8) FROM t WHERE k < 3;", names, device=False)
    check_plan(rs, abi.KERNEL_NON_GROUPED, [8] * 7)
    cnt = cnt8 = s8 = 0
    for n, mult in views(T_BIG, PHYS):
        sel = k[:n] < 3
        nn = sel & (t8[:n] != abi.NULL_TINYINT)
        cnt, cnt8, s8 = cnt + int(sel.sum()) * mult, cnt8 + int(nn.sum()) * mult, s8 + int(t8[:n][nn].astype(np.int64).sum()) * mult
    nn = (k < 3) & (t8 != abi.NULL_TINYINT)
    assert cnt > 2**32
    rows_equal([(0,) + rs.rows()[0]], {0: (0, cnt, cnt8, s8, int(t8[nn].min()), int(t8[nn].max()), s8 / cnt8)}, fp_cols=(6,))
    rs = run(t, "SELECT k, COUNT(*), SUM(t8) FROM t WHERE t8 IS NOT NULL GROUP BY k;", names, device=False)
    check_plan(rs, abi.KERNEL_PERFECT_SMEM, [8, 8, 8])
    g = grouped(k, [t8], t8 != abi.NULL_TINYINT, T_BIG)
    assert max(c[0] for c in g.values()) > 2**32 * 0.9
    rows_equal(rs.rows(), {key: (key, c, s) for key, (c, s) in g.items()})


# ---- (d) a group whose values in [1, 2^31) sum to exactly 2^64 --------------------------------------------------------
HOT_ROWS = 2**24 + 2**16          # x 512 copies: ~8.6e9 rows of values just under 2^31
D_COPIES = 512


@pytest.fixture(scope="module")
def wrap_phys():
    _need_device_memory()
    target = 2**64 // D_COPIES                   # what one physical copy of the hot group must sum to
    v0, rem = divmod(target, HOT_ROWS)
    hot = np.full(HOT_ROWS, v0, dtype=np.int64)
    hot[:rem] += 1
    assert 1 <= hot.min() and hot.max() < 2**31 and int(hot.sum()) * D_COPIES == 2**64
    rng = np.random.default_rng(64)
    other = 2**20
    k_other = rng.integers(1, 50, other)
    v_other = rng.integers(-3, 4, other)
    v_other[k_other == 7] = 0                    # a group of zeros
    k = np.concatenate([np.zeros(HOT_ROWS, np.int64), k_other])
    v = np.concatenate([hot, v_other]).astype(np.int64)
    perm = rng.permutation(k.size)
    return Physical([(abi.kBIGINT, True), (abi.kBIGINT, True)], [k[perm], v[perm]])


def test_d_hbm_table_group_summing_to_2_64(wrap_phys):
    """The HBM-table kernels' touched flag: group 0's SUM is 0 mod 2^64 yet the group is present.  With plain int64 words
    (B2Q_GLOBAL_SPLIT=0, see the next test) the flag rests on "a value in [1, 2^31) cannot sum to zero under 2^32 rows",
    so past 2^32 rows the executor must keep the split layout."""
    ph = wrap_phys
    total = ph.host[0].size * D_COPIES
    t = ph.table(total)
    rs = run(t, "SELECT k, SUM(v) FROM t GROUP BY k;", ["k", "v"], force_kernel=abi.KERNEL_PERFECT_GLOBAL)
    check_plan(rs, abi.KERNEL_PERFECT_GLOBAL, [8, 8], keyless=0)
    g = grouped(ph.host[0], [ph.host[1]], np.ones(ph.host[0].size, bool), total)
    assert g[0][1] == 2**64 and g[7][1] == 0
    want = {key: (key, wrap64(s)) for key, (c, s) in g.items()}
    assert want[0] == (0, 0)
    rows_equal(rs.rows(), want)


def test_d_plain_word_layout_keeps_the_group_past_2_32_rows():
    """The same query in a process whose HBM-table kernels default to plain int64 words (read once per process)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, B2Q_GLOBAL_SPLIT="0")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu",
                        "tests/test_gpu_zz_row_boundaries.py::test_d_hbm_table_group_summing_to_2_64"],
                       cwd=root, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]


# ---- (e) sparse BIGINT keys: baseline hash -------------------------------------------------------------------------
@pytest.mark.parametrize("force", [0, abi.KERNEL_BASELINE_PROBE], ids=["radix", "probe"])
def test_e_baseline_hash_sparse_keys(main_phys, force):
    """Sparse keys: the baseline hash, through the radix passes (whose scratch runs in batches of fewer than 2^32 tuples,
    the last one short) or forced onto the per-row probe kernel."""
    ndv = 1000
    dense = (np.arange(PHYS) * 7919) % ndv
    key = ((dense.astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)) >> np.uint64(1)).astype(np.int64)
    v = main_phys.host[3]
    ph = Physical([(abi.kBIGINT, True), (abi.kBIGINT, True)], [key, v], dev=[None, main_phys.dev[3]])
    total = T_BIG + 12345
    t = ph.table(total)
    rs = run(t, "SELECT key, COUNT(*), SUM(v) FROM t GROUP BY key;", ["key", "v"], guess=2 * ndv, has_card=True, force_kernel=force)
    check_plan(rs, abi.KERNEL_BASELINE_GLOBAL, [0, 8, 8])      # the probe kernel is an execution choice of the same plan
    g = grouped(key, [v], np.ones(PHYS, bool), total)
    assert len(g) == ndv and sum(c[0] for c in g.values()) == total
    rows_equal(rs.rows(), {kk: (kk, c, wrap64(s)) for kk, (c, s) in g.items()})


# ---- (i) a join whose tables together pass UINT32_MAX rows ------------------------------------------------------------
def test_i_join_count_slot_counts_the_inner_table(main_phys):
    """Outer 2^32 - 2^20 rows (aliased), inner 2^21: the reference sums the tuples of both tables (query_infos), so COUNT(*)
    gets an 8-byte slot and group 0 (> 2^31 rows) comes back positive."""
    inner_rows = 2**21
    d_id = np.arange(inner_rows, dtype=np.int32)
    d_attr = (d_id >> 18).astype(np.int32)              # 8 groups of 2^18 ids
    dim = abi.Table([(abi.kINT, True), (abi.kINT, True)])
    dim.add_host_fragment([d_id, d_attr])
    rng = np.random.default_rng(21)
    i = np.arange(PHYS)
    fk = np.where(i % 10 < 7, rng.integers(0, 2**18, PHYS), rng.integers(0, inner_rows, PHYS)).astype(np.int32)
    ph = Physical([(abi.kINT, True)], [fk])
    total = 2**32 - 2**20
    t = ph.table(total)
    rs = run(t, "SELECT d.attr, COUNT(*) FROM t JOIN d ON t.fk = d.id GROUP BY d.attr;", ["fk"], inner=(dim, ["id", "attr"]))
    check_plan(rs, abi.KERNEL_PERFECT_SMEM, [8, 8])
    g = grouped(d_attr[fk], [], np.ones(PHYS, bool), total)
    assert g[0][0] > 2**31
    rows_equal(rs.rows(), {a: (a, c[0]) for a, c in g.items()})
