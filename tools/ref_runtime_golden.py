#!/usr/bin/env python
"""TEST INFRASTRUCTURE (fixture generator; never imported by the product, tests, smoke() or bench.py — it is the committed script that
made tests/golden/ref_runtime.npz).  Runs the reference's own hash / probe / decoder runtime (oracle/_ref/libref_groupby.so, built by
`make -C oracle ref` where the reference tree exists, see oracle/ref_shim.cpp) on the inputs of tests/test_oracle_ref.py and stores
what it answered, so that the oracle is pinned against the reference on machines that never see the reference's sources.

    python tools/ref_runtime_golden.py          # writes tests/golden/ref_runtime.npz

Stored per test (inputs that are not a seeded test table are stored too):
  murmur_*   MurmurHash3 of every prefix (0..32 bytes) of 64 random bytes under three seeds, and of 2000 int64 keys
  ggv_*      get_group_value: the key sequence, the slot offset of each insert (-1 = table full) and the final buffer
  fast_*     get_group_value_fast: returned offsets and the buffer after three inserts
  dec_*      chunk decoders: MIN / MAX / COUNT over the values the reference decodes, per column, and a digest of the chunks
  day_*      DATE bucket index: for the keys of two queries, where get_group_value_fast puts each key
  join_*     one-to-one join table built and probed by the reference: matches and SUM over the fact table
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle_lib  # noqa: E402
import sqlmini  # noqa: E402
import join_tables as jt  # noqa: E402
import str_tables as stt  # noqa: E402
from heavydb_b200 import abi  # noqa: E402
from test_oracle_ref import (DAY_QUERIES, DECODED_COLUMNS, FAST_CASES, GGV_CASES, chunk_digest, day_table,  # noqa: E402
                             decoder_table, fresh_ggv_buffer, join_tables)

REF_SO = os.path.join(ROOT, "oracle", "_ref", "libref_groupby.so")
OUT = os.path.join(ROOT, "tests", "golden", "ref_runtime.npz")


def load_ref():
    R = C.CDLL(REF_SO)
    R.MurmurHash3.restype = C.c_uint32
    R.MurmurHash3.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
    R.get_group_value.restype = C.c_void_p
    R.get_group_value.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]
    R.get_group_value_fast.restype = C.c_void_p
    R.get_group_value_fast.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_uint32]
    for name in ("fixed_width_int_decode", "fixed_width_unsigned_decode"):
        getattr(R, name).restype = C.c_int64
        getattr(R, name).argtypes = [C.c_void_p, C.c_int32, C.c_int64]
    R.fixed_width_small_date_decode.restype = C.c_int64
    R.fixed_width_small_date_decode.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64]
    R.fill_one_to_one_hashtable.restype = C.c_int
    R.fill_one_to_one_hashtable.argtypes = [C.c_size_t, C.c_void_p, C.c_int32]
    R.get_hash_slot.restype = C.c_void_p
    R.get_hash_slot.argtypes = [C.c_void_p, C.c_int64, C.c_int64]
    R.hash_join_idx_nullable.restype = C.c_int64
    R.hash_join_idx_nullable.argtypes = [C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64]
    return R


def murmur(R, g):
    rng = np.random.default_rng(7)
    data = rng.integers(0, 256, size=64, dtype=np.uint8)
    seeds = np.array([0, 1, 0x9747B28C], dtype=np.uint32)
    g["murmur_data"], g["murmur_seeds"] = data, seeds
    g["murmur_data_hash"] = np.array([[R.MurmurHash3(data.ctypes.data, n, int(s)) for s in seeds] for n in range(33)], dtype=np.uint32)
    keys = rng.integers(-2**62, 2**62, size=2000, dtype=np.int64)
    g["murmur_keys"] = keys
    g["murmur_keys_hash"] = np.array([R.MurmurHash3(keys[i:i + 1].ctypes.data, 8, 0) for i in range(keys.size)], dtype=np.uint32)


def get_group_value(R, g):
    for kw, ec, nk in GGV_CASES:
        keys = np.random.default_rng(ec).integers(1, 50 if ec == 16 else 10**6, size=nk)
        keys = np.concatenate([keys, keys[: nk // 2]])  # revisit
        buf = fresh_ggv_buffer(kw, ec)
        offs = []
        for k in keys:
            kb = np.zeros(1, dtype=np.int64)
            if kw == 8:
                kb[0] = k
            else:
                kb.view(np.int32)[0] = k
            r = R.get_group_value(buf.ctypes.data, ec, kb.ctypes.data, 1, kw, 3)
            off = -1 if not r else (r - buf.ctypes.data) // 8
            if off >= 0:
                buf[off] += 1
            offs.append(off)
        tag = f"ggv_{kw}_{ec}_{nk}"
        g[tag + "_keys"], g[tag + "_off"], g[tag + "_buf"] = keys, np.array(offs, dtype=np.int64), buf


def get_group_value_fast(R, g):
    row_size_quad, n = 3, 20
    buf = np.full(n * row_size_quad, np.iinfo(np.int64).max, dtype=np.int64)
    g["fast_off"] = np.array([(R.get_group_value_fast(buf.ctypes.data, k, mn, b, row_size_quad) - buf.ctypes.data) // 8
                              for k, mn, b in FAST_CASES], dtype=np.int64)
    g["fast_buf"] = buf


def decoders(R, g):
    table = decoder_table()
    names = stt.STR_NAMES
    null64 = abi.NULL_BIGINT
    g["dec_digest"] = np.frombuffer(chunk_digest((table, [names.index(c) for c, _ in DECODED_COLUMNS])), dtype=np.uint8)
    agg = []
    for col, kind in DECODED_COLUMNS:
        c = names.index(col)
        width = np.dtype(table.physical_dtype(c)).itemsize
        vals = []
        for f in table.fragments:
            a = f.host_cols[c]
            for pos in range(a.size):
                if kind == "days":
                    v = R.fixed_width_small_date_decode(a.ctypes.data, width, table.physical_null(c), null64, pos)
                    if v != null64:
                        vals.append(v)
                elif kind == "fixed":
                    v = R.fixed_width_int_decode(a.ctypes.data, width, pos)
                    if v != table.physical_null(c):     # codgenAdjustFixedEncNull maps it to the logical NULL
                        vals.append(v)
                else:
                    v = R.fixed_width_unsigned_decode(a.ctypes.data, width, pos)
                    if stt.STR_COLS[c][2] or v != table.physical_null(c):
                        vals.append(v)
        agg.append((min(vals), max(vals), len(vals)))
    g["dec_min_max_count"] = np.array(agg, dtype=np.int64)


def day_buckets(R, g):
    table = day_table()
    for q, sql in enumerate(DAY_QUERIES):
        res = oracle_lib.execute(sqlmini.parse(sql, table, stt.STR_NAMES), table)
        p = res.plan
        row_quad = p.row_size // 8
        buf = res.buffer().view(np.int64).reshape(p.entry_count, row_quad)
        keys = np.array(sorted(int(k) for k in buf[:, 0] if k != np.iinfo(np.int64).max), dtype=np.int64)
        offs = []
        for key in keys:
            scratch = np.full(p.entry_count * row_quad, np.iinfo(np.int64).max, dtype=np.int64)
            offs.append((R.get_group_value_fast(scratch.ctypes.data, int(key), p.min_val, p.bucket, row_quad) - scratch.ctypes.data) // 8)
        g[f"day{q}_plan"] = np.array([p.min_val, p.bucket, row_quad, p.entry_count], dtype=np.int64)
        g[f"day{q}_keys"], g[f"day{q}_off"] = keys, np.array(offs, dtype=np.int64)


def join(R, g):
    dim, fact = join_tables()
    g["join_digest"] = np.frombuffer(chunk_digest((dim, range(len(jt.DIM_NAMES))), (fact, range(len(jt.FACT_NAMES)))), dtype=np.uint8)
    ids = dim.fragments[0].host_cols[jt.DIM_NAMES.index("id32")]
    big = dim.fragments[0].host_cols[jt.DIM_NAMES.index("big")]
    mn, mx = int(ids.min()), int(ids.max())
    buff = np.full(mx - mn + 1, -1, dtype=np.int32)
    for row, k in enumerate(ids):
        assert R.fill_one_to_one_hashtable(row, R.get_hash_slot(buff.ctypes.data, int(k), mn), -1) == 0
    matches, total = 0, 0
    for f in fact.fragments:
        for k in f.host_cols[jt.FACT_NAMES.index("fk32")]:
            idx = R.hash_join_idx_nullable(buff.ctypes.data, int(k), mn, mx, abi.NULL_INT)
            if idx >= 0:
                matches += 1
                total += int(big[idx])
    g["join_matches_sum"] = np.array([matches, total], dtype=np.int64)


def main():
    if not os.path.exists(REF_SO):
        raise SystemExit(f"{REF_SO} is missing: run `make -C oracle ref` where the reference tree exists")
    R = load_ref()
    g = {}
    for step in (murmur, get_group_value, get_group_value_fast, decoders, day_buckets, join):
        step(R, g)
    np.savez_compressed(OUT, **g)
    print(OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
