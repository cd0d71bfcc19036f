#!/usr/bin/env python
"""bench.py — rows/s and achieved HBM GB/s of the scan -> filter -> group-by/aggregate path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--rows R] [--config c2|c2all|c3|c4] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input (BASELINE.json configs[1] at N = 1):
    1e9 rows, c0/c1 int64 ~U[0,1e6), g int32 ~U[0,1e4):  SELECT g, SUM(c1), COUNT(*) FROM t WHERE c0 < 500000 GROUP BY g
    30 fragments of 32 Mi rows (reference default fragment size, Fragmenter/FragmentDefaultValues.h:19).

`value`     whole-job rows/s with the columns already resident in HBM (timed region = the full C-ABI call:
            table init + scan + merge of CTA tables + materialise + D2H of the result buffer).
`roofline`  algorithmic bytes (20 B/row) / mean scan-kernel time (CUDA events on the launching stream, measured
            inside libb2q around the kernel) against MEASURED_PEAKS.json's HBM copy bandwidth.
`e2e`       the same query through the C ABI with HOST (pinned) column buffers: H2D copies of every referenced column
            inside the timed region, result read back to the host.
`cpu_baseline`  the oracle (CPU restatement of the reference's executor) on a bounded sample, all host threads.

N > 1 (torchrun): fragments are sharded over ranks (weak scaling: every rank scans `rows` rows of its own
fragments, fragment ids are global), partial aggregate tables are merged with NCCL all-reduce (one per dense array),
time = max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

_JSON_OUT = sys.stdout   # main() re-points it at the real stdout and sends fd 1 to stderr

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SEED = 0x5EED
FRAG_ROWS = 1 << 25  # 32 Mi rows

CONFIGS = {
    # name: (columns [(name, type, lo, span)], sql template, algorithmic bytes/row, workload string)
    "c2": ([("c0", "i64", 0, 10**6), ("c1", "i64", 0, 10**6), ("g", "i32", 0, 10**4)],
           "SELECT g, SUM(c1), COUNT(*) FROM t WHERE c0 < 500000 GROUP BY g;", 20,
           "configs[1]: filter c0<k (50%) + GROUP BY int32 g (1e4 groups) SUM(int64)/COUNT, 3 of the 4 int64 columns unused by the minimal query are not read"),
    "c2all": ([("c0", "i64", 0, 10**6), ("c1", "i64", 0, 10**6), ("c2", "i64", 0, 10**6), ("c3", "i64", 0, 10**6), ("g", "i32", 0, 10**4)],
              "SELECT g, SUM(c1), SUM(c2), SUM(c3), COUNT(*) FROM t WHERE c0 < 500000 GROUP BY g;", 36,
              "configs[1] all-columns variant: 4 x int64 + int32 key, SUM x3 + COUNT"),
    "c3": ([("f", "i64", 0, 10**6), ("g", "i32", 0, 256), ("v", "f64", 0, 1)],
           "SELECT g, AVG(v) FROM t WHERE f < 500000 GROUP BY g;", 20, "configs[2]: 256 groups AVG(double)"),
    "c4": ([("key", "i64", 0, 10**7), ("v", "i64", 0, 10**6)],
           "SELECT key, SUM(v) FROM t GROUP BY key;", 16, "configs[3]: 1e7 dense int64 keys SUM (HBM/L2 table)"),
    # sparse keys (key = U[0,1e7) * 900000000007): the range is too wide for a perfect hash => baseline hash,
    # open addressing in HBM, entry_count = NDV * 1.5 like RelAlgExecutor's estimator path
    "c4s": ([("key", "i64", 0, 10**7, 900_000_000_007), ("v", "i64", 0, 10**6)],
            "SELECT key, SUM(v) FROM t GROUP BY key;", 16, "configs[3] sparse variant: 1e7 sparse int64 keys SUM (global-memory hash table, MurmurHash3 + CAS)"),
}
CONFIGS["c2enc"] = (
    # the same table declared with the reference's fixed-width encodings (BIGINT ENCODING FIXED(32), INT ENCODING
    # FIXED(16)): 10 B/row instead of 20 — SURVEY.md §8f-2 "lets the kernels read real HeavyDB chunks"
    [("c0", "i64", 0, 10**6, 1, 4), ("c1", "i64", 0, 10**6, 1, 4), ("g", "i32", 0, 10**4, 1, 2)],
    CONFIGS["c2"][1], 10, "configs[1] with ENCODING FIXED chunks: c0,c1 BIGINT FIXED(32), g INT FIXED(16)")
# SURVEY §8f-1: the same aggregations ending in ORDER BY ... LIMIT (top-k on the device: only the kept rows are copied back)
CONFIGS["c2top"] = (CONFIGS["c2"][0], "SELECT g, SUM(c1), COUNT(*) FROM t WHERE c0 < 500000 GROUP BY g ORDER BY 2 DESC, 1 LIMIT 10;", 20,
                    "configs[1] + ORDER BY SUM DESC LIMIT 10 (device compaction + radix sort + gather)")
CONFIGS["c4top"] = (CONFIGS["c4"][0], "SELECT key, SUM(v) FROM t GROUP BY key ORDER BY 2 DESC, 1 LIMIT 10;", 16,
                    "configs[3] + ORDER BY SUM DESC LIMIT 10 over 1e7 groups (device compaction + radix sort + gather)")
# SURVEY §8f-3: star join — the fact table probes a 1e5-row dimension through a one-to-one perfect join table and
# groups by a dimension attribute (the dimension is generated on the host: id = row, attr = splitmix64(row) % 1000)
CONFIGS["c2join"] = ([("c0", "i64", 0, 10**6), ("c1", "i64", 0, 10**6), ("fk", "i32", 0, 10**5)],
                     "SELECT d.attr, SUM(t.c1), COUNT(*) FROM t JOIN d ON t.fk = d.id WHERE t.c0 < 500000 GROUP BY d.attr;", 20,
                     "configs[1] shape through a star join: filter c0<k (50%), INNER JOIN dim(1e5 rows) ON fk = id, GROUP BY dim.attr (1000 groups), SUM/COUNT")
CONFIGS["c2joins"] = ([("c0", "i64", 0, 10**6), ("c1", "i64", 0, 10**6), ("fk", "i32", 0, 10**4)],
                      CONFIGS["c2join"][1], 20,
                      "star join with a 1e4-row dimension: the (packed) join table is TMA-staged into shared memory")
# the cardinality-estimation query that precedes c4s in the reference's flow (CardinalityEstimationRequired ->
# RelAlgExecutor::getNDVEstimation): NDVEstimator over the sparse key, 8 B/row
CONFIGS["c4sndv"] = ([("key", "i64", 0, 10**7, 900_000_000_007)], "ESTIMATOR NDV(key)", 8,
                     "NDV estimator query over 1e7 sparse int64 keys (linear_probabilistic_count into a 1 MiB bitmap)")
ENTRY_GUESS = {"c4s": 15_000_000}


def make_unit(cfg, sql, table, names):
    """The execution unit of a config: parsed SQL, or the estimator unit (no SQL form: RelAlgExecutor synthesises it)."""
    from heavydb_b200 import abi, sqlmini
    if sql.startswith("ESTIMATOR"):
        b = abi.UnitBuilder(table)
        b.estimator([names.index("key")])
        return b.build()
    return sqlmini.parse(sql, table, names, inner=join_inner(cfg))


def join_inner(cfg):
    """(inner abi.Table, names) for the join configs, else None.  Built on the host; the library copies it per query."""
    if cfg not in ("c2join", "c2joins"):
        return None
    from heavydb_b200 import abi
    n = 10**5 if cfg == "c2join" else 10**4
    ids = np.arange(n, dtype=np.int32)
    x = ids.astype(np.uint64) + np.uint64(0x9E3779B97F4A7C15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    attr = ((x ^ (x >> np.uint64(31))) % np.uint64(1000)).astype(np.int32)
    t = abi.Table([(abi.kINT, True), (abi.kINT, True)])
    t.add_host_fragment([ids, attr])
    return t, ["id", "attr"]


def col_enc(col):
    return col[5] if len(col) > 5 else 0


def col_stride(col):
    return col[4] if len(col) > 4 else 1


def phys_type(col):
    """sql type of the PHYSICAL chunk elements (what the generator must write)."""
    from heavydb_b200 import abi
    e = col_enc(col)
    return {0: np_type(col[1]), 1: abi.kTINYINT, 2: abi.kSMALLINT, 4: abi.kINT}[e]


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.load_start = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0=None, t1=None):
        """Samples inside [t0, t1] (the timed region); if the region is shorter than the sampling period, the
        samples of the whole loaded window (warm-up + timed steps) are used and the fact is reported."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        inside = [r for ts, r in self.rows if t0 is not None and t0 <= ts <= t1]
        window = "timed region"
        if len(inside) < 3:
            inside = [r for ts, r in self.rows if self.load_start is not None and self.load_start <= ts <= (t1 or ts)]
            window = "warm-up + timed region (timed region shorter than 3 sampling periods)"
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in inside:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


def np_type(t):
    from heavydb_b200 import abi
    return {"i64": abi.kBIGINT, "i32": abi.kINT, "f64": abi.kDOUBLE}[t]


METRIC = "rows/sec and HBM GB/s on 1e9-row filter+groupby"   # BASELINE.json's metric; both arms print the same string


def gen_specs(cols):
    """[(physical sql type, col_tag, lo, span, stride)] — what the device generator and the oracle's generator are both given."""
    return [(phys_type(c), tag, c[2], c[3], col_stride(c)) for tag, c in enumerate(cols)]


def chunk_stats(col):
    from heavydb_b200 import abi
    st = abi.ChunkStats()
    if col[1] == "f64":
        st.fp_min, st.fp_max = 0.0, 1.0
    else:
        st.int_min, st.int_max = col[2], col[2] + (col[3] - 1) * col_stride(col)
    return st


def rank_fragments(rows, rank, world, ring=0):
    """[(fragment_id, rows, alias_id)] of one rank: ceil(rows / FRAG_ROWS) fragments with ids rank, rank + world, ...
    (fragment_id % num_devices == device, InsertOrderFragmenter.cpp:435-443).  ring > 0: only `ring` physical fragments exist
    per rank; logical fragment k re-reads physical fragment k % ring (its generator rows are those of alias_id)."""
    out, remaining, k = [], rows, 0
    while remaining > 0:
        m = min(FRAG_ROWS, remaining)
        fid = rank + k * world
        alias = rank + (k % ring) * world if ring else fid
        out.append((fid, m, alias))
        remaining -= m
        k += 1
    return out


def build_device_table(cfg, frags, torch, remote=()):
    """This rank's fragments generated directly in HBM with the counter-based generator (global row = alias_id * FRAG_ROWS + i),
    plus the other ranks' fragments as chunk stats only (every rank then plans over the same table)."""
    from heavydb_b200 import abi, executor
    cols = CONFIGS[cfg][0]
    table = abi.Table([(np_type(c[1]), True) for c in cols], encoded_sizes=[col_enc(c) for c in cols])
    keep, phys = [], {}
    stats = [chunk_stats(c) for c in cols]
    for fid, m, alias in frags:
        if alias not in phys or phys[alias][0] < m:
            ptrs = []
            for tag, col in enumerate(cols):
                ty = phys_type(col)
                buf = torch.empty(m * abi.SIZE_OF[ty], dtype=torch.uint8, device="cuda")
                executor.gen_column_device(buf.data_ptr(), ty, SEED, tag, alias * FRAG_ROWS, m, col[2], col[3], stride=col_stride(col))
                keep.append(buf)
                ptrs.append(buf.data_ptr())
            phys[alias] = (m, ptrs)
        table.add_device_fragment(m, phys[alias][1], stats, fragment_id=fid)
    for fid, m, _ in remote:
        table.add_remote_fragment(m, stats, fid)
    torch.cuda.synchronize()
    return table, keep


def stats_only_table(cfg, frags):
    """The whole table as the oracle's generated-table executor wants it: sizes, ids (the ALIAS id: it names the generator rows)
    and chunk stats, no buffers."""
    from heavydb_b200 import abi
    cols = CONFIGS[cfg][0]
    t = abi.Table([(np_type(c[1]), True) for c in cols], encoded_sizes=[col_enc(c) for c in cols])
    stats = [chunk_stats(c) for c in cols]
    for _, m, alias in frags:
        t.add_remote_fragment(m, stats, alias)
    return t


def oracle_threads_for(plan):
    """One output buffer per oracle worker: as many workers as cores, bounded by 24 GB of buffers."""
    n = os.cpu_count() or 1
    per = max(int(plan.buffer_size), 1)
    return max(1, min(n, (24 << 30) // per))


def parity_check(cfg, unit, rs, all_frags, guess):
    """Bit-exact check of the TIMED result against the oracle over the FULL input (every fragment of every rank, regenerated on
    the host slab by slab): integer / bit-pattern slots identical, floating-point SUM within 1e-6 relative."""
    import gpu_util as gu
    import oracle_lib
    from heavydb_b200 import abi
    t0 = time.perf_counter()
    cols = CONFIGS[cfg][0]
    table = stats_only_table(cfg, all_frags)
    gplan = rs.getQueryMemDesc()
    threads = oracle_threads_for(gplan)
    rows = sum(m for _, m, _ in all_frags)
    out = {"rows": rows, "ok": False, "oracle_threads": threads, "checker": "oracle/ (CPU restatement of the reference's executor) over the same generated rows"}
    try:
        ref = oracle_lib.execute_generated(unit, table, gen_specs(cols), SEED, FRAG_ROWS, entry_guess=guess, has_card=guess > 0, num_threads=threads)
        if unit.unit.has_estimator:
            ok = np.array_equal(rs.getHostEstimatorBuffer(), ref.buffer().view(np.uint8))
            out.update(ok=bool(ok), compared="estimator bitmap, bit for bit")
        else:
            oplan = ref.plan
            assert gplan.as_dict() == oplan.as_dict(), "plan differs from the oracle's"
            g, w = rs.getStorageBuffer(), ref.buffer()
            if gplan.query_desc_type == abi.GroupByBaselineHash:
                # a key may sit in different slots of the two tables (insertion order): compare the rows, sorted by key
                q = gplan.row_size // 8
                gm, wm = g.view(np.int64).reshape(-1, q), w.view(np.int64).reshape(-1, q)
                gm, wm = gm[gm[:, 0] != abi.EMPTY_KEY_64], wm[wm[:, 0] != abi.EMPTY_KEY_64]
                assert gm.shape == wm.shape, f"{gm.shape[0]} groups, oracle {wm.shape[0]}"
                gm, wm = gm[np.argsort(gm[:, 0], kind="stable")], wm[np.argsort(wm[:, 0], kind="stable")]
                fp = {gplan.slot_offset[t.first_slot] // 8 for t in gplan.targets[:gplan.num_targets]
                      if t.is_agg and t.agg_kind in (abi.kSUM, abi.kAVG) and t.agg_arg_type.type == abi.kDOUBLE}
                for c in range(q):
                    if c in fp:
                        a, b = gm[:, c].view(np.float64), wm[:, c].view(np.float64)
                        assert ((a == b) | (np.abs(a - b) <= gu.FP_RTOL * np.abs(b))).all(), f"fp SUM word {c}"
                    else:
                        assert np.array_equal(gm[:, c], wm[:, c]), f"row word {c} differs"
                out["compared"] = f"{gm.shape[0]} (key, slots) rows sorted by key, bit for bit (fp SUM within 1e-6)"
            else:
                gu.buffers_equal(g, w, gplan)
                out["compared"] = f"raw {gplan.buffer_size}-byte output buffer, bit for bit (fp SUM within 1e-6)"
            assert rs.rowCount() == ref.row_count()
            out["ok"] = True
    except AssertionError as e:
        out["error"] = str(e)[:300]
    except Exception as e:  # the check must never take the bench line down with it
        out["error"] = f"{type(e).__name__}: {e}"[:300]
    out["seconds"] = round(time.perf_counter() - t0, 2)
    return out


def host_table_for_reference(cfg, rows, threads):
    """The reference arm's table: `threads` fragments of rows/threads rows, each generated (first touch) by the pinned worker
    that later scans it."""
    import oracle_lib
    from heavydb_b200 import abi
    cols = CONFIGS[cfg][0]
    nfrag = threads
    per = [rows // nfrag + (1 if f < rows % nfrag else 0) for f in range(nfrag)]
    row0 = [sum(per[:f]) for f in range(nfrag)]
    arrays = [[np.empty(per[f], dtype=abi.NUMPY_OF[phys_type(c)]) for c in cols] for f in range(nfrag)]
    oracle_lib.gen_fragments(arrays, gen_specs(cols), per, row0, SEED, threads)
    table = abi.Table([(np_type(c[1]), True) for c in cols], encoded_sizes=[col_enc(c) for c in cols])
    stats = [chunk_stats(c) for c in cols]
    for f in range(nfrag):
        fr = abi.Fragment(per[f], host_cols=arrays[f], stats=list(stats), fragment_id=f)
        table.fragments.append(fr)
    return table


def workload_config(cfg, rows, world, scaling):
    cols, sql, bpr, workload = CONFIGS[cfg]
    return {"workload": workload, "query": sql, "rows_per_gpu": rows, "rows_total": rows * world, "algorithmic_bytes_per_row": bpr,
            "generator": f"counter-based splitmix64 columns, seed {SEED:#x}", "scaling": scaling}


def run_reference(args):
    """--impl reference: the reference's CPU algorithm for this path (the oracle port) on the box's host cores, over the SAME
    workload as the GPU arm (rows_per_gpu rows; the rate is per row, so N GPUs' worth is not repeated N times), one
    NUMA-pinned thread per fragment, fragments first-touched by the thread that scans them."""
    import oracle_lib
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "all"])
    cols, sql, bpr, workload = CONFIGS[args.config]
    threads = os.cpu_count() or 1
    rows = args.rows
    oracle_lib.set_thread_pinning(True)
    table = host_table_for_reference(args.config, rows, threads)
    names = [c[0] for c in cols]
    unit = make_unit(args.config, sql, table, names)
    guess = ENTRY_GUESS.get(args.config, 0)
    times = []
    n_out = 0
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        res = oracle_lib.execute(unit, table, entry_guess=guess, has_card=guess > 0, num_threads=threads)
        n_out = res.row_count()
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
        del res
    ms = 1e3 * sum(times) / len(times)
    value = rows / (ms / 1e3)
    sample = (f"{rows} rows of the same workload in {threads} host fragments (one pinned thread per fragment, first-touch local), "
              f"per-fragment buffers + host reduce (KernelPerFragment); N > 1 arms scan N x as many rows at the same per-row rate")
    cfgd = workload_config(args.config, rows, int(os.environ.get("WORLD_SIZE", "1")), "weak")
    cfgd.update({"groups_out": int(n_out), "rows_per_step": rows})
    out = {
        "impl": "reference", "metric": METRIC,
        "note": "the reference's CPU algorithm for this path (restated in oracle/, validated against the reference's own tests) on the host cores",
        "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
        "data": "synthetic", "config": cfgd,
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), file=_JSON_OUT, flush=True)
    return 0


def cpu_baseline_sample(cfg, budget_s=12.0):
    """The reported CPU baseline inside the GPU arm's line: the oracle on a bounded sample (2^29 rows) of the same workload."""
    import oracle_lib
    cols, sql, _, _ = CONFIGS[cfg]
    threads = os.cpu_count() or 1
    rows = 1 << 29
    oracle_lib.set_thread_pinning(True)
    try:
        table = host_table_for_reference(cfg, rows, threads)
        unit = make_unit(cfg, sql, table, [c[0] for c in cols])
        guess = ENTRY_GUESS.get(cfg, 0)
        oracle_lib.execute(unit, table, entry_guess=guess, has_card=guess > 0, num_threads=threads)  # warm
        t0 = time.perf_counter()
        reps = 0
        while reps < 3 or (time.perf_counter() - t0 < budget_s and reps < 30):
            oracle_lib.execute(unit, table, entry_guess=guess, has_card=guess > 0, num_threads=threads)
            reps += 1
        dt = (time.perf_counter() - t0) / reps
    finally:
        oracle_lib.set_thread_pinning(False)
    return {"value": rows / dt, "unit": "rows/s", "cores": threads, "kind": "port",
            "sample": f"{rows} rows of the same workload in {threads} host fragments, one pinned thread per fragment + host reduce, {reps} reps"}


class Runner:
    """One configuration on this rank's GPU: table in HBM, the unit, and `step()` = one pass of the hot path through the C ABI
    (scan -> cross-GPU merge inside libb2q when world > 1 -> materialise -> D2H of the result buffer)."""

    def __init__(self, cfg, rows, rank, world, comm, torch, force_kernel=0, ring=0):
        from heavydb_b200 import abi, executor
        self.cfg, self.rows, self.rank, self.world, self.comm = cfg, rows, rank, world, comm
        self.abi, self.executor = abi, executor
        cols, sql, self.bytes_per_row, self.workload = CONFIGS[cfg]
        self.sql, self.names = sql, [c[0] for c in cols]
        self.frags = [rank_fragments(rows, r, world, ring) for r in range(world)]
        remote = [f for r in range(world) if r != rank for f in self.frags[r]]
        self.table, self.keep = build_device_table(cfg, self.frags[rank], torch, remote)
        self.unit = make_unit(cfg, sql, self.table, self.names)
        self.ex = executor.Executor()
        self.eo = executor.execution_options(force_kernel=force_kernel)
        # the C structs the entry point takes (B2QTableInfo: this rank's fragments + every other rank's as chunk stats), built ONCE: a
        # native caller holds them as such; re-marshalling O(all fragments) Python objects per step is not part of the query
        self.bt = self.table.build(abi.GPU_LEVEL)
        self.guess = ENTRY_GUESS.get(cfg, 0)

    def all_frags(self):
        return [f for r in range(self.world) for f in self.frags[r]]

    def step(self):
        abi, executor = self.abi, self.executor
        if self.comm is not None:
            return executor.execute_work_unit_dist(self.comm, self.ex, self.guess, True, self.bt, self.unit, eo=self.eo,
                                                   has_cardinality_estimation=self.guess > 0)
        return self.ex.executeWorkUnit(self.guess, True, self.bt, self.unit, eo=self.eo, has_cardinality_estimation=self.guess > 0,
                                       memory_level=abi.GPU_LEVEL)

    def free(self, torch):
        self.keep.clear()
        self.table = None
        self.bt = None
        torch.cuda.empty_cache()


def timed_steps(runner, steps, warmup, torch, dist, sampler=None):
    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
    scan_ms, step_ms = [], []
    t_begin = t_end = None
    rs = None
    for i in range(warmup + steps):
        rs = None
        barrier()
        if i == warmup:
            t_begin = time.time()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rs = runner.step()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1), rs.kernel_ms()], device="cuda", dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if i >= warmup:
            step_ms.append(float(t[0].item()))
            scan_ms.append(float(t[1].item()))
        t_end = time.time()
    return rs, float(np.mean(step_ms)), float(np.mean(scan_ms)), t_begin, t_end


DUMP_MAX_BYTES = 60_000_000   # array bytes written by --dump-outputs: under 64 MB with the .npy headers


def target_names(sql):
    """File-name-safe names of the SELECT list: "g, SUM(c1), COUNT(*)" -> ["g", "sum_c1", "count"]."""
    body = sql[len("SELECT "):sql.index(" FROM ")]
    names, depth, cur = [], 0, ""
    for ch in body:
        depth += (ch == "(") - (ch == ")")
        if ch == "," and depth == 0:
            names.append(cur)
            cur = ""
        else:
            cur += ch
    names.append(cur)
    return ["_".join("".join(c if c.isalnum() else " " for c in n.lower()).split()) for n in names]


def dump_outputs(out_dir, rs, sql, ordered):
    """Writes what the caller of the timed path received in the last step, one float64 array per target as
    out_dir/col<i>_<target>.npy (NULLs are the target type's inline sentinel), or for the estimator query its NDV estimate
    and bitmap.  Rows of a GROUP BY without ORDER BY come in hash-table order, which another build may change, so they
    are sorted by all columns, keys first: two builds then compare row for row.  Beyond DUMP_MAX_BYTES a fixed, seeded
    sample of the sorted rows is written."""
    os.makedirs(out_dir, exist_ok=True)
    if sql.startswith("ESTIMATOR"):
        arrays = {"ndv_estimate": np.array([rs.getNDVEstimator()], dtype=np.float64),
                  "estimator_bitmap": rs.getHostEstimatorBuffer().astype(np.float32)}
    else:
        cols = [a for _, _, a in rs.columnarResults()]
        n = cols[0].size
        order = np.arange(n) if ordered else np.lexsort(cols[::-1])
        keep = DUMP_MAX_BYTES // (8 * len(cols))
        if n > keep:
            order = order[np.sort(np.random.default_rng(SEED).choice(n, size=keep, replace=False))]
        arrays = {f"col{i}_{name}": a[order].astype(np.float64) for i, (name, a) in enumerate(zip(target_names(sql), cols))}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return sorted(arrays)


def config_block(cfg, rows, torch, steps=3, warmup=1):
    """kernel_ms / ms_per_step / roofline fraction / full-size parity of one more BASELINE configuration (N = 1)."""
    peak, _ = measured_peak()
    try:
        r = Runner(cfg, rows, 0, 1, None, torch)
        rs, ms, k_ms, _, _ = timed_steps(r, steps, warmup, torch, None)
        achieved = rows * r.bytes_per_row / (k_ms / 1e3) / 1e9
        out = {"workload": r.workload, "query": r.sql, "rows": rows, "steps": steps, "ms_per_step": ms, "kernel_ms": k_ms,
               "rows_per_s": rows / (ms / 1e3), "achieved_gbs": achieved, "frac": achieved / peak,
               "algorithmic_bytes_per_row": r.bytes_per_row, "kernel": int(rs.getQueryMemDesc().kernel),
               "entry_count": int(rs.getQueryMemDesc().entry_count), "launches_per_step": int(rs.stats()["kernel_launches"]),
               "groups_out": int(rs.rowCount()) if not r.sql.startswith("ESTIMATOR") else int(rs.getNDVEstimator())}
        out["parity_check"] = parity_check(cfg, r.unit, rs, r.all_frags(), r.guess)
        del rs
        r.free(torch)
        return out
    except Exception as e:
        torch.cuda.empty_cache()
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--rows", type=int, default=1_000_000_000, help="rows per GPU (weak scaling)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="strong: --total-rows rows in total (BASELINE configs[4]: 8e9), split over the GPUs")
    ap.add_argument("--total-rows", type=int, default=8_000_000_000)
    ap.add_argument("--configs", default="auto", help="extra BASELINE configurations measured + parity-checked into the line's `configs` "
                    "block: comma list, 'none', or 'auto' (= c2all,c3,c4,c4s at N = 1, none at N > 1)")
    ap.add_argument("--e2e-rows", type=int, default=0, help="rows of the host-buffer end-to-end leg (0 = auto)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--force-kernel", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result columns of the last timed step to DIR/<name>.npy "
                    "(float64, at most 64 MB: a seeded row sample beyond that), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's result; the reference arm has none")
    # the contract is ONE JSON line on stdout: whatever libraries print there (NCCL's version banner, for one) goes to stderr
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    from heavydb_b200 import abi, build, executor
    build.build()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the path has no CPU fallback")
    torch.cuda.set_device(local)
    dist, comm = None, None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        # torch.distributed is plumbing (rendezvous, barriers, max-over-ranks of the timings); the data-path merge is
        # libb2q's own NCCL communicator, whose 128-byte id travels over the process group
        box = [executor.Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        comm = executor.Comm.init_rank(box[0], world, rank, device=local)
    rows, ring = args.rows, 0
    if args.scaling == "strong":
        rows = args.total_rows // world
        bytes_per_row = sum(abi.SIZE_OF[phys_type(c)] for c in CONFIGS[args.config][0])
        free_b, _ = torch.cuda.mem_get_info()
        if rows * bytes_per_row > 0.7 * free_b:   # N = 1 of configs[4] is 160 GB: scan a ring of resident fragments instead
            ring = max(1, int(0.5 * free_b // (FRAG_ROWS * bytes_per_row)))
    runner = Runner(args.config, rows, rank, world, comm, torch, force_kernel=args.force_kernel, ring=ring)
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)  # let nvidia-smi come up so that samples exist for a millisecond-scale timed region
    sampler.load_start = time.time()
    rs, ms, k_ms, t_begin, t_end = timed_steps(runner, args.steps, args.warmup, torch, dist)
    clocks = sampler.stop(t_begin, t_end)
    sql, bytes_per_row = runner.sql, runner.bytes_per_row
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = dump_outputs(args.dump_outputs, rs, sql, ordered=runner.unit.unit.num_order_entries > 0)
    launches_per_step = rs.stats()["kernel_launches"]
    sort_us = rs.stats()["sort_us"]
    result_rows = rs.rowCount() if not sql.startswith("ESTIMATOR") else rs.getNDVEstimator()
    plan_kernel, plan_entries = int(rs.getQueryMemDesc().kernel), int(rs.getQueryMemDesc().entry_count)
    total_rows = rows * world
    value = total_rows / (ms / 1e3)
    peak, peak_src = measured_peak()
    achieved = rows * bytes_per_row / (k_ms / 1e3) / 1e9
    traffic, traffic_src = None, None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json"))).get(args.config)
        if tr:
            traffic = (tr["dram_read_bytes"] + tr["dram_write_bytes"]) * (rows / tr["rows"])
            traffic_src = f"{tr['source']} (ncu --set full at commit {tr.get('commit', '?')}, {tr['rows']} rows/launch, scaled to {rows})"
    except Exception:
        pass
    cfgd = workload_config(args.config, rows, world, args.scaling)
    cfgd.update({"fragments_per_gpu": len(runner.frags[rank]), "fragment_rows": FRAG_ROWS, "kernel": plan_kernel, "entry_count": plan_entries,
                 "groups_out": int(result_rows), "l2": "inputs larger than L2",
                 "merge": "none (1 GPU)" if world == 1 else "NCCL inside libb2q on the scan stream (b2q_execute_work_unit_dist)"})
    if ring:
        cfgd["hbm_ring"] = f"{ring} resident fragments re-read round-robin ({rows * bytes_per_row / 1e9:.0f} GB of columns do not fit one GPU)"
    if sort_us:
        cfgd["sort_ms"] = sort_us / 1e3
    out = {
        "metric": METRIC,
        "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "int64",
        "data": "synthetic (counter-based splitmix64 columns generated in HBM; inputs 20 GB/GPU >> 126 MB L2, no flush needed)",
        "config": cfgd,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes": rows * bytes_per_row,
                     "peak_source": peak_src, "kernel": "b2q_k_scan", "kernel_ms": k_ms,
                     "algorithmic_bytes_per_row": bytes_per_row},
        "clocks": clocks,
        "gpu_launches": int(launches_per_step) * args.steps,  # per step: b2q_k_init, the scan / radix passes, b2q_k_materialize (+ NCCL's own)
    }
    if dumped:
        out["dumped_outputs"] = dumped
    # the timed result, checked bit for bit against the oracle over the full input of ALL ranks
    if not args.no_parity:
        if rank == 0:
            subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "all"])
            out["parity_check"] = parity_check(args.config, runner.unit, rs, runner.all_frags(), runner.guess)
        if dist is not None:
            dist.barrier()
    main_buf = rs.getStorageBuffer().copy() if world == 1 and not sql.startswith("ESTIMATOR") else None
    del rs
    runner.free(torch)
    if not args.no_e2e:
        e2e = e2e_leg(args, torch, dist, rank, world, comm, args.config, rows if args.scaling == "weak" else min(rows, 10**9), main_buf)
        if world == 1 and args.config == "c2":   # the same table declared with the reference's fixed-width encodings: half the bytes per row
            e2e["c2enc"] = e2e_leg(args, torch, dist, rank, world, comm, "c2enc", rows, None)
        out["e2e"] = e2e
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "all"])
            out["cpu_baseline"] = cpu_baseline_sample(args.config)
        except Exception as e:  # the oracle is only a reported baseline
            out["cpu_baseline"] = {"value": None, "unit": "rows/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
    extra = args.configs
    if extra == "auto":
        extra = "c2all,c3,c4,c4s" if (world == 1 and args.config == "c2" and args.scaling == "weak" and not args.no_parity) else "none"
    if extra != "none" and world == 1:
        out["configs"] = {c: config_block(c, rows, torch) for c in extra.split(",") if c in CONFIGS}
    if rank == 0:
        print(json.dumps(out), file=_JSON_OUT, flush=True)
    if comm is not None:
        comm.destroy()
    if dist is not None:
        dist.destroy_process_group()
    return 0


def gpu_numa_cpus(torch):
    """CPUs of the NUMA node the GPU hangs off (so pinned host buffers are allocated next to its PCIe root)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None, node
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        return cpus, node
    except Exception as e:  # noqa
        return None, str(e)


def e2e_leg(args, torch, dist, rank, world, comm, cfg, rows_req, main_buf):
    """Host (pinned) buffers -> C ABI -> host result, on every rank at once: each rank streams ITS fragments from pinned host memory
    on its GPU's NUMA node over its own PCIe link; H2D of every referenced column and the D2H of the result are inside the timed
    region; time = max over ranks, value = all ranks' rows / that time."""
    import psutil
    from heavydb_b200 import abi, executor
    cols, sql, _, _ = CONFIGS[cfg]
    names = [c[0] for c in cols]
    cpus, node = gpu_numa_cpus(torch)
    old_aff = None
    if cpus:
        try:
            old_aff = os.sched_getaffinity(0)
            os.sched_setaffinity(0, cpus & old_aff or cpus)
        except Exception:
            old_aff = None
    bytes_per_row = sum(abi.SIZE_OF[phys_type(c)] for c in cols)
    guess = ENTRY_GUESS.get(cfg, 0)
    avail = psutil.virtual_memory().available
    rows = args.e2e_rows or rows_req
    cap = int(avail * 0.4 / max(world, 1) // bytes_per_row)
    rows = max(FRAG_ROWS, min(rows, cap))
    if dist is not None:   # every rank the same share
        t = torch.tensor([rows], device="cuda", dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        rows = int(t.item())
    frags = [rank_fragments(rows, r, world) for r in range(world)]
    table = abi.Table([(np_type(c[1]), True) for c in cols], encoded_sizes=[col_enc(c) for c in cols])
    stats = [chunk_stats(c) for c in cols]
    keep = []
    for fid, m, _ in frags[rank]:
        harrs = []
        for tag, col in enumerate(cols):
            ty = phys_type(col)
            dev = torch.empty(m * abi.SIZE_OF[ty], dtype=torch.uint8, device="cuda")
            executor.gen_column_device(dev.data_ptr(), ty, SEED, tag, fid * FRAG_ROWS, m, col[2], col[3], stride=col_stride(col))
            host = torch.empty(m * abi.SIZE_OF[ty], dtype=torch.uint8, pin_memory=True)
            host.copy_(dev)
            keep.append(host)
            harrs.append(host.numpy().view(abi.NUMPY_OF[ty]))
            del dev
        table.fragments.append(abi.Fragment(m, host_cols=harrs, stats=list(stats), fragment_id=fid))
    for r in range(world):
        if r != rank:
            for fid, m, _ in frags[r]:
                table.add_remote_fragment(m, stats, fid)
    torch.cuda.synchronize()
    if old_aff:
        os.sched_setaffinity(0, old_aff)
    unit = make_unit(cfg, sql, table, names)
    ex = executor.Executor()
    eo = executor.execution_options(force_kernel=args.force_kernel)
    bt = table.build(abi.CPU_LEVEL)
    # what this box's PCIe link delivers for plain copies out of the very same pinned buffers (no kernels, one stream):
    # the ceiling the end-to-end leg can reach — boxes of the pool differ by almost 2x here
    raw_gbs = None
    try:
        probe = [h for h in keep if h.numel() >= (64 << 20)]
        if probe:
            scratch = torch.empty(max(h.numel() for h in probe), dtype=torch.uint8, device="cuda")
            scratch[:probe[0].numel()].copy_(probe[0], non_blocking=True)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for h in probe:
                scratch[:h.numel()].copy_(h, non_blocking=True)
            e1.record()
            torch.cuda.synchronize()
            raw_gbs = sum(h.numel() for h in probe) / (e0.elapsed_time(e1) / 1e3) / 1e9
            del scratch
    except Exception:  # the probe is informational
        raw_gbs = None
    times, d2h, n, phases, same = [], 0, 0, {}, None
    for i in range(2 + 3):
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        if comm is not None:
            rs = executor.execute_work_unit_dist(comm, ex, guess, True, bt, unit, eo=eo, has_cardinality_estimation=guess > 0, memory_level=abi.CPU_LEVEL)
        else:
            rs = ex.executeWorkUnit(guess, True, bt, unit, eo=eo, has_cardinality_estimation=guess > 0, memory_level=abi.CPU_LEVEL)
        n = rs.rowCount()
        dt = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        d2h = int(rs.getQueryMemDesc().buffer_size)
        phases = rs.stats()
        if i >= 2:
            times.append(dt)
        if i == 4 and main_buf is not None and rows == rows_req:
            same = bool(np.array_equal(rs.getStorageBuffer(), main_buf))
        del rs
    dt = float(np.mean(times))
    total = rows * world
    out = {"value": total / dt, "unit": "rows/s", "h2d_bytes_per_step": int(total * bytes_per_row), "d2h_bytes_per_step": d2h * world,
           "rows": total, "rows_per_gpu": rows, "ms_per_step": dt * 1e3,
           "host_memory": f"pinned, allocated on each GPU's NUMA node (rank 0: node {node})", "h2d_gbs": total * bytes_per_row / dt / 1e9,
           "h2d_raw_gbs_same_buffers_rank0": raw_gbs, "groups_out": int(n),
           "host_phases_ms": {k[5:-3]: phases[k] / 1e3 for k in ("host_setup_us", "host_stream_us", "host_teardown_us")}}
    if same is not None:
        out["same_bytes_as_the_hbm_resident_result"] = same
    keep.clear()
    return out


if __name__ == "__main__":
    sys.exit(main())
