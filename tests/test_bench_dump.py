"""bench.py --dump-outputs: the files hold what the last timed step returned to its caller — the scan's PosList and the join's
RowID pairs at the seeded sample positions, their chunk / partition offsets and the whole Q1 result — each equal to the
oracle on the same generated tables."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as orc
from bench import Q1_AGGREGATES, Q1_GROUPBY, Q1_PREDICATES, SCAN_PREDICATE, dump_positions, row_id_columns
from hyrise_b200 import capi
from hyrise_b200.tpch import L_ORDERKEY, O_ORDERKEY, TpchTables

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SF = 0.2   # 1.2 M lineitem rows: more join pairs than the dump keeps, so the sampled form is what gets checked


@pytest.mark.gpu
def test_dump_outputs_are_the_timed_results(tmp_path):
    command = [sys.executable, os.path.join(REPO, "bench.py"), "--sf", str(SF), "--steps", "2", "--warmup", "0",
               "--no-cpu-baseline", "--no-e2e", "--no-verify", "--dump-outputs", str(tmp_path)]
    run = subprocess.run(command, capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stdout[-2000:] + run.stderr[-2000:]
    dumped = {name[:-len(".npy")]: np.load(tmp_path / name) for name in os.listdir(tmp_path)}
    assert all(array.dtype == np.float64 for array in dumped.values())
    assert sum(array.nbytes for array in dumped.values()) <= 64 << 20

    tables = TpchTables(SF, seed=42)
    threads = os.cpu_count() or 1
    scan = orc.table_scan(tables.lineitem, SCAN_PREDICATE, threads=threads)
    positions = dump_positions(len(scan.row_ids))
    assert np.array_equal(dumped["scan_positions"], positions)
    assert np.array_equal(dumped["scan_row_ids"], row_id_columns(scan.row_ids[positions]))
    assert np.array_equal(dumped["scan_chunk_offsets"], scan.chunk_offsets)

    join = orc.join_hash(tables.orders, O_ORDERKEY, tables.lineitem, L_ORDERKEY, capi.JOIN_INNER, -1, threads=threads)
    positions = dump_positions(join.pair_count)
    assert len(positions) < join.pair_count
    assert np.array_equal(dumped["join_positions"], positions)
    assert np.array_equal(dumped["join_build_row_ids"], row_id_columns(join.build[positions]))
    assert np.array_equal(dumped["join_probe_row_ids"], row_id_columns(join.probe[positions]))
    assert np.array_equal(dumped["join_partition_offsets"], join.partition_offsets)

    q1 = orc.aggregate_hash(tables.lineitem, Q1_GROUPBY, Q1_AGGREGATES, predicates=Q1_PREDICATES, threads=threads)
    assert np.array_equal(dumped["aggregate_row_ids"], row_id_columns(q1.row_ids))
    assert np.array_equal(dumped["aggregate_nulls"], np.stack(q1.nulls, axis=1))
    np.testing.assert_allclose(dumped["aggregate_values"], np.stack([v.astype(np.float64) for v in q1.values], axis=1),
                               rtol=1e-6, atol=0)
    tables.close()
