"""Pins the oracle's hash + probe against the reference's OWN runtime (QueryEngine/MurmurHash.cpp + QueryEngine/GroupByRuntime.cpp +
QueryEngine/DecodersImpl.h, see oracle/ref_shim.cpp), and against the probe constants recorded in SURVEY.md §8c.  What the reference's
runtime answered on the inputs below is stored in tests/golden/ref_runtime.npz (made by tools/ref_runtime_golden.py), so these tests
need neither the reference's sources nor a build of them."""
import hashlib
import os

import numpy as np
import pytest

import oracle_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_runtime.npz")

GGV_CASES = [(8, 97, 60), (8, 64, 64), (4, 101, 80), (8, 16, 40)]     # (key_width, entry_count, nkeys)
FAST_CASES = [(5, 0, 0), (17, 3, 0), (40, 10, 2)]                       # (key, min, bucket)
DECODED_COLUMNS = [("dd", "days"), ("dd16", "days"), ("ts", "fixed"), ("s8", "unsigned"), ("s16", "unsigned")]
DAY_QUERIES = ["SELECT dt, COUNT(*) FROM s WHERE dt > 1555286410 GROUP BY dt;", "SELECT dd, COUNT(*) FROM s WHERE dd >= 1555372801 GROUP BY dd;"]
JOIN_SQL = "SELECT COUNT(*), SUM(d.big) FROM t JOIN d ON t.fk32 = d.id32;"


def fresh_ggv_buffer(key_width, entry_count, row_size_quad=3):
    """An empty baseline-hash buffer of rows [key 8][slot][slot]."""
    b = np.zeros(entry_count * row_size_quad, dtype=np.int64)
    if key_width == 8:
        b.reshape(entry_count, row_size_quad)[:, 0] = np.iinfo(np.int64).max
    else:
        b.view(np.int32).reshape(entry_count, 2 * row_size_quad)[:, 0] = np.iinfo(np.int32).max
    return b


def decoder_table():
    import str_tables as stt
    return stt.str_table(3000, seed=21, frag_rows=700)


def day_table():
    import str_tables as stt
    return stt.str_table(3000, seed=22, frag_rows=700)


def join_tables():
    import join_tables as jt
    return jt.dim_table(), jt.fact_table(5000, seed=9, frag_rows=1300)


def chunk_digest(*tables_and_columns):
    """sha256 over the chunks of the given (table, column indices) pairs: ties a stored answer to the exact input it was computed on."""
    h = hashlib.sha256()
    for table, cols in tables_and_columns:
        for f in table.fragments:
            for c in cols:
                h.update(np.ascontiguousarray(f.host_cols[c]).tobytes())
    return h.digest()


def test_murmur3_known_answers():
    L = oracle_lib.lib()
    k64 = np.array([12345], dtype=np.int64)
    k32 = np.array([7], dtype=np.int32)
    assert L.oracle_murmur3(k64.ctypes.data, 8, 0) == 342635441
    assert L.oracle_murmur3(k32.ctypes.data, 4, 0) == 1343918321


@pytest.fixture(scope="module")
def golden():
    with np.load(GOLDEN) as z:
        return {k: z[k] for k in z.files}


def test_murmur3_matches_reference(golden):
    L = oracle_lib.lib()
    data = np.ascontiguousarray(golden["murmur_data"])
    for length in range(0, 33):
        for j, seed in enumerate(golden["murmur_seeds"]):
            assert L.oracle_murmur3(data.ctypes.data, length, int(seed)) == golden["murmur_data_hash"][length, j]
    keys = np.ascontiguousarray(golden["murmur_keys"])
    for i in range(keys.size):
        assert L.oracle_murmur3(keys[i:i + 1].ctypes.data, 8, 0) == golden["murmur_keys_hash"][i]


@pytest.mark.parametrize("key_width,entry_count,nkeys", GGV_CASES)
def test_get_group_value_matches_reference(golden, key_width, entry_count, nkeys):
    """Same insert sequence into two tables -> identical slot addresses, identical key placement, and the same
    'table full' answer (NULL) once entry_count distinct keys are in (GroupByRuntime.cpp:25-48)."""
    L = oracle_lib.lib()
    tag = f"ggv_{key_width}_{entry_count}_{nkeys}"
    keys, want_off = golden[tag + "_keys"], golden[tag + "_off"]
    ours = fresh_ggv_buffer(key_width, entry_count)
    for k, r_off in zip(keys, want_off):
        kb = np.zeros(1, dtype=np.int64)
        if key_width == 8:
            kb[0] = k
        else:
            kb.view(np.int32)[0] = k
        o = L.oracle_get_group_value(ours.ctypes.data, entry_count, kb.ctypes.data, 1, key_width, 3)
        assert o == r_off
        if o >= 0:
            ours[o] += 1
    assert np.array_equal(ours, golden[tag + "_buf"])


def test_get_group_value_fast_reference(golden):
    """Perfect-hash direct index: off = (key - min) / bucket * row_size_quad, key written on first touch
    (GroupByRuntime.cpp:194-209) — the formula the oracle's run_fragment and the CUDA kernels use."""
    row_size_quad = 3
    buf = golden["fast_buf"]
    for (key, mn, bucket), r_off in zip(FAST_CASES, golden["fast_off"]):
        d = key - mn
        if bucket:
            d //= bucket
        assert r_off == d * row_size_quad + 1
        assert buf[d * row_size_quad] == key


def test_chunk_decoders_match_reference(golden):
    """The oracle reads ENCODING FIXED, DICT(8|16) and DATE ENCODING DAYS chunks exactly like the reference's
    decoders: per column, MIN / MAX / COUNT over the values the REFERENCE decodes == the oracle's answer."""
    import sqlmini
    import str_tables as stt
    table = decoder_table()
    names = stt.STR_NAMES
    assert chunk_digest((table, [names.index(c) for c, _ in DECODED_COLUMNS])) == golden["dec_digest"].tobytes()
    for (col, kind), (mn, mx, count) in zip(DECODED_COLUMNS, golden["dec_min_max_count"].tolist()):
        agg = "COUNT({0})" if kind == "unsigned" else "MIN({0}), MAX({0}), COUNT({0})"
        res = oracle_lib.execute(sqlmini.parse(f"SELECT {agg.format(col)}, COUNT(*) FROM s;", table, names), table).rows()[0]
        if kind == "unsigned":
            assert res == (count, 3000)
        else:
            assert res == (mn, mx, count, 3000), col


def test_day_bucket_index_matches_reference(golden):
    """DATE keys: entry = (key - min) / 86400 with min possibly off the day grid (a simple qual narrowed it) — every
    non-empty entry of the oracle's buffer sits where the reference's get_group_value_fast puts its key."""
    import sqlmini
    import str_tables as stt
    table = day_table()
    for q, sql in enumerate(DAY_QUERIES):
        res = oracle_lib.execute(sqlmini.parse(sql, table, stt.STR_NAMES), table)
        p = res.plan
        assert p.bucket == 86400 and p.min_val % 86400 != 0 and not p.keyless_hash
        row_quad = p.row_size // 8
        assert [p.min_val, p.bucket, row_quad, p.entry_count] == golden[f"day{q}_plan"].tolist(), sql
        ref_off = dict(zip(golden[f"day{q}_keys"].tolist(), golden[f"day{q}_off"].tolist()))
        buf = res.buffer().view(np.int64).reshape(p.entry_count, row_quad)
        seen = 0
        for i in range(p.entry_count):
            key = int(buf[i, 0])
            if key == np.iinfo(np.int64).max:
                continue
            assert ref_off.get(key) == i * row_quad + 1, (sql, i, key)
            seen += 1
        assert seen == len(ref_off) == res.row_count() > 5


def test_one_to_one_join_table_matches_reference(golden):
    """fill_one_to_one_hashtable + get_hash_slot + hash_join_idx[_nullable] (JoinHashImpl.h, GroupByRuntime.cpp:283-316),
    the reference's own code, drove a Python join over these tables; the oracle's joined aggregates must agree."""
    import join_tables as jt
    import sqlmini
    dim, fact = join_tables()
    assert chunk_digest((dim, range(len(jt.DIM_NAMES))), (fact, range(len(jt.FACT_NAMES)))) == golden["join_digest"].tobytes()
    matches, total = golden["join_matches_sum"].tolist()
    unit = sqlmini.parse(JOIN_SQL, fact, jt.FACT_NAMES, inner=(dim, jt.DIM_NAMES))
    assert oracle_lib.execute(unit, fact).rows() == [(matches, total)]
    assert 0 < matches < 5000
