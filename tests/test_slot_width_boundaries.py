"""The tuple-count boundary of the COUNT(*) slot width, pinned by hand.

pick_target_compact_width (QueryMemoryDescriptor.cpp:826-833) sums `qi.info.getNumTuples()` over every table in
query_infos and gives a single-column GROUP BY whose targets are COUNT(*) and narrow integer projections 4-byte slots
when that sum is at most UINT32_MAX = 2^32 - 1, 8-byte slots otherwise.  With a join level query_infos holds the outer
AND the inner table.  A 4-byte COUNT slot reads back as a signed int32 (ResultSetBufferAccessors.h:246-253), so the
width decides whether a group of more than 2^31 rows comes back negative.

Stats-only tables: the planners read row counts and chunk statistics, no data.  The expected widths below are read off
the reference's rule, not taken from either planner; both planners are asserted on their own, then against each other.
"""
import numpy as np
import pytest

import oracle_lib
import sqlmini
from heavydb_b200 import abi, executor

U32_MAX = 2**32 - 1
NARROW, WIDE = [4, 4], [8, 8]


def _stats(lo, hi):
    s = abi.ChunkStats()
    s.int_min, s.int_max, s.has_nulls = lo, hi, 0
    return s


def _outer(fragment_tuples):
    """t(x INT NOT NULL in [0, 9], fk INT NOT NULL in [0, 999]) as chunk stats only, one fragment per entry."""
    t = abi.Table([(abi.kINT, True), (abi.kINT, True)])
    for i, n in enumerate(fragment_tuples):
        t.add_remote_fragment(n, [_stats(0, 9), _stats(0, 999)], fragment_id=i)
    return t


def _dimension(rows):
    """d(id INT NOT NULL = row, attr INT NOT NULL = id % 7): the inner table of a hash join needs its columns."""
    d = abi.Table([(abi.kINT, True), (abi.kINT, True)])
    d.add_host_fragment([np.arange(rows, dtype=np.int32), (np.arange(rows) % 7).astype(np.int32)])
    return d


def _widths(unit, table, bigint_count=False):
    """(oracle widths, product widths), each asserted by the caller, and the two full plans."""
    o = oracle_lib.plan(unit, table, bigint_count=bigint_count)
    p = executor.Executor().plan(unit, table, eo=executor.execution_options(bigint_count=bigint_count))
    return list(o.slot_padded_width[: o.num_slots]), list(p.slot_padded_width[: p.num_slots]), o, p


# total tuples -> widths, by QueryMemoryDescriptor.cpp:830: `total_tuples <= UINT32_MAX ? 4 : crt_min_byte_width (8)`
SINGLE_TABLE = [
    ([U32_MAX], NARROW),                                   # exactly at the line
    ([U32_MAX + 1], WIDE),                                 # one past it
    ([2**31, 2**31 - 1], NARROW),                          # two fragments summing to UINT32_MAX
    ([2**31, 2**31], WIDE),                                # ... and to 2^32
    ([2**30] * 3 + [2**30 - 1], NARROW),                   # four fragments, none near the line on its own
    ([2**30] * 4, WIDE),
    ([1_000_003] * 4294 + [U32_MAX - 1_000_003 * 4294], NARROW),   # many fragments, ragged last one
    ([1_000_003] * 4294 + [U32_MAX - 1_000_003 * 4294 + 1], WIDE),
    ([U32_MAX, 0], NARROW),                                # an empty fragment adds nothing
    ([2**40], WIDE),
]


@pytest.mark.parametrize("fragments,widths", SINGLE_TABLE, ids=[f"{len(f)}frags-{sum(f)}" for f, _ in SINGLE_TABLE])
def test_count_slot_width_at_the_uint32_line(fragments, widths):
    t = _outer(fragments)
    for sql in ("SELECT x, COUNT(*) FROM t GROUP BY x;", "SELECT COUNT(*), x FROM t GROUP BY x;"):
        unit = sqlmini.parse(sql, t, ["x", "fk"])
        ow, pw, o, p = _widths(unit, t)
        assert ow == widths, ("oracle", sql, sum(fragments))
        assert pw == widths, ("product", sql, sum(fragments))
        assert p.as_dict() == o.as_dict()


@pytest.mark.parametrize("total", [U32_MAX, U32_MAX + 1])
def test_bigint_count_keeps_8_bytes_on_both_sides_of_the_line(total):
    """g_bigint_count short-circuits the rule (QueryMemoryDescriptor.cpp:752-754): 8 bytes whatever the tuple count."""
    t = _outer([total])
    unit = sqlmini.parse("SELECT x, COUNT(*) FROM t GROUP BY x;", t, ["x", "fk"], bigint_count=True)
    ow, pw, o, p = _widths(unit, t, bigint_count=True)
    assert ow == WIDE and pw == WIDE and p.as_dict() == o.as_dict()


JOIN_SQL = "SELECT d.attr, COUNT(*) FROM t JOIN d ON t.fk = d.id GROUP BY d.attr;"
# (outer fragments, inner rows, widths): outer + inner tuples against UINT32_MAX (QueryMemoryDescriptor.cpp:827-830 loops
# over query_infos, which holds both tables of the join)
JOIN_CASES = [
    ([U32_MAX - 1000], 1000, NARROW),                      # outer + inner == UINT32_MAX
    ([U32_MAX - 999], 1000, WIDE),                         # outer + inner == 2^32, the outer alone is below the line
    ([2**31, 2**31 - 1 - 1000], 1000, NARROW),
    ([2**31, 2**31 - 1000], 1000, WIDE),
    ([2**32 - 2**20], 2**21, WIDE),                        # the shape of the device test: 2^32 + 2^20 tuples in all
    ([2**32 - 2**20], 2**20 - 1, NARROW),
    ([U32_MAX + 1], 1000, WIDE),                           # the outer alone past the line
]


@pytest.mark.parametrize("fragments,inner_rows,widths", JOIN_CASES,
                         ids=[f"{len(f)}frags-{sum(f)}+{n}" for f, n, _ in JOIN_CASES])
def test_join_counts_the_inner_table_toward_the_line(fragments, inner_rows, widths):
    t = _outer(fragments)
    d = _dimension(inner_rows)
    unit = sqlmini.parse(JOIN_SQL, t, ["x", "fk"], inner=(d, ["id", "attr"]))
    ow, pw, o, p = _widths(unit, t)
    assert ow == widths, ("oracle", sum(fragments) + inner_rows)
    assert pw == widths, ("product", sum(fragments) + inner_rows)
    assert p.as_dict() == o.as_dict()
    assert o.query_desc_type == abi.GroupByPerfectHash and o.join_entry_count == inner_rows
