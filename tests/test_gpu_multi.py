"""Multi-device execution with the merge inside libb2q (NCCL): `b2q_execute_work_unit_multi` — one call, one host thread per
device (Execute.cpp:3055-3101) — against the oracle over the whole table, on however many devices the box has (1 device:
the same code path with a one-rank communicator); and, on boxes with >= 2 GPUs, the one-process-per-GPU form
(`b2q_execute_work_unit_dist` under torchrun, tools/multigpu_check.py)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import gpu_util as gu
import oracle_lib
import order_queries as oq
import sqlmini
from heavydb_b200 import abi, executor
from test_gpu_parity import RAND_NAMES, RAND_QUERIES, random_table

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def device_views(table, ndev):
    """Per device: its fragments (fragment_id % ndev, InsertOrderFragmenter.cpp:435-443) resident in that device's HBM plus
    the other devices' fragments as chunk stats only."""
    import torch
    views, keep = [], []
    for d in range(ndev):
        v = abi.Table(table.col_types, encoded_sizes=table.encoded_sizes, deleted_column=table.deleted_column)
        for f in table.fragments:
            if f.fragment_id % ndev == d:
                ptrs = []
                for a in f.host_cols:
                    t = torch.from_numpy(a.view(np.uint8).copy()).cuda(d)
                    keep.append(t)
                    ptrs.append(t.data_ptr())
                v.add_device_fragment(f.num_tuples, ptrs, f.stats, fragment_id=f.fragment_id, device_id=d)
            else:
                v.add_remote_fragment(f.num_tuples, f.stats, f.fragment_id)
        views.append(v)
    for d in range(ndev):
        torch.cuda.synchronize(d)
    return views, keep


def test_work_unit_multi_matches_oracle():
    ndev = min(executor.lib().b2q_device_count(), 4)
    comms = executor.Comm.init_all(list(range(ndev)))
    try:
        table = random_table(120000, seed=23, frag_rows=10000)    # 12 fragments
        views, _keep = device_views(table, ndev)
        ex = executor.Executor()
        for sql in RAND_QUERIES + oq.RAND_ORDER_QUERIES:
            unit = sqlmini.parse(sql, table, RAND_NAMES)
            rs = executor.execute_work_unit_multi(comms, ex, 4000, True, views, unit, has_cardinality_estimation=True)
            ref = oracle_lib.execute(unit, table, entry_guess=4000, has_card=True, num_threads=4)
            if unit.unit.num_order_entries:
                gu.rows_equal_ordered(rs.rows(), ref.rows())
            else:
                gu.rows_equal(rs.rows(), ref.rows(), col_tol=gu.column_tolerances(ref.plan, 120000))
            assert rs.rowCount() == ref.row_count(), sql
            if not unit.unit.num_order_entries and not unit.unit.has_limit:
                assert rs.getQueryMemDesc().as_dict() == ref.plan.as_dict()
        for cols in (["k32"], ["k16", "nn32"], ["sparse"]):    # estimator bitmaps: all-gather + OR
            b = abi.UnitBuilder(table)
            b.estimator([RAND_NAMES.index(c) for c in cols])
            unit = b.build()
            rs = executor.execute_work_unit_multi(comms, ex, 1, True, views, unit)
            ref = oracle_lib.execute(unit, table, num_threads=4)
            assert np.array_equal(rs.getHostEstimatorBuffer(), ref.buffer().view(np.uint8)), cols
    finally:
        for c in comms:
            c.destroy()


def test_multi_reports_the_same_error_on_every_device():
    ndev = min(executor.lib().b2q_device_count(), 2)
    comms = executor.Comm.init_all(list(range(ndev)))
    try:
        table = random_table(20000, seed=9, frag_rows=2500)
        views, _keep = device_views(table, ndev)
        unit = sqlmini.parse("SELECT sparse, COUNT(*) FROM r GROUP BY sparse;", table, RAND_NAMES)
        with pytest.raises(executor.QueryExecutionError) as ei:   # fewer entries than distinct keys
            executor.execute_work_unit_multi(comms, executor.Executor(), 100, True, views, unit, has_cardinality_estimation=True)
        assert ei.value.code == abi.ERR_OUT_OF_SLOTS
    finally:
        for c in comms:
            c.destroy()


def test_dist_two_ranks_under_torchrun():
    if executor.lib().b2q_device_count() < 2:
        pytest.skip("needs 2 GPUs (one process per GPU under torchrun)")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29517", os.path.join(ROOT, "tools", "multigpu_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "multigpu_check ok" in out.stdout
