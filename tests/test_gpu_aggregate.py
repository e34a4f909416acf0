"""AggregateHash parity: the CUDA path (through the C-ABI) against the oracle. Group order and representative RowIDs
bit-exact, counts / integer sums exact, floating-point SUM / AVG within 1e-6 relative (BASELINE.json north_star)."""
import numpy as np
import pytest

import oracle_lib as orc
from aggregate_cases import CASES
from helpers import ENCODINGS, assert_aggregate_outputs_equal, random_table, tbl, tpch
from hyrise_b200 import capi
from hyrise_b200.device import Aggregate, Expression, Predicate
from test_oracle_aggregate import (Q1_AGGREGATES, Q1_PREDICATES, Q6_AGGREGATES, Q6_PREDICATES, lineitem_table,
                                   make_aggregates)

pytestmark = pytest.mark.gpu


def check_aggregate(device, table, device_table, groupby, aggregates, predicates=(), filters=None):
    expected = orc.aggregate_hash(table, groupby, aggregates, predicates=predicates,
                                  input_filter=filters[1] if filters else None)
    got = device.aggregate_hash(device_table, groupby, aggregates, predicates=predicates,
                                input_filter=filters[0] if filters else None)
    assert_aggregate_outputs_equal(got, expected)
    return got


@pytest.mark.parametrize("case", CASES, ids=[f"{c[0]}@{c[1]}" for c in CASES])
def test_reference_cases(device, case):
    name, line, input_file, chunk_size, dictionary, definitions, groupby, expected_file, on_reference_table = case
    for encoding in (["Dictionary"] if dictionary else ENCODINGS):
        table = tbl(input_file, chunk_size).encode(encoding)
        device_table = device.upload(table)
        aggregates = make_aggregates(definitions)
        check_aggregate(device, table, device_table, groupby, aggregates)
        if on_reference_table and table.column_definitions[0].data_type != capi.TYPE_STRING:
            predicate = Predicate(0, capi.PRED_GREATER_THAN, 0)
            filters = (device.table_scan(device_table, predicate), orc.table_scan(table, predicate))
            check_aggregate(device, table, device_table, groupby, aggregates, filters=filters)
            check_aggregate(device, table, device_table, groupby, aggregates, predicates=[predicate])  # fused form
        device_table.drop()


@pytest.mark.parametrize("encoding", ENCODINGS)
def test_random_tables(device, encoding):
    rng = np.random.default_rng(77)
    table = random_table(rng, 40_000, 4_999).encode(encoding)
    device_table = device.upload(table)
    column = Expression.column
    all_functions = [Aggregate(capi.AGG_SUM, column(0)), Aggregate(capi.AGG_AVG, column(1)), Aggregate(capi.AGG_MIN, column(2)),
                     Aggregate(capi.AGG_MAX, column(3)), Aggregate(capi.AGG_COUNT, column(0)), Aggregate(capi.AGG_COUNT_STAR),
                     Aggregate(capi.AGG_MIN, column(1)), Aggregate(capi.AGG_MAX, column(0)), Aggregate(capi.AGG_SUM, column(2)),
                     Aggregate(capi.AGG_AVG, column(3))]
    sums_only = [Aggregate(capi.AGG_SUM, column(2)), Aggregate(capi.AGG_AVG, column(2)), Aggregate(capi.AGG_COUNT, column(2)),
                 Aggregate(capi.AGG_COUNT_STAR)]
    for groupby in ([], [4], [0], [4, 0], [1], [2], [3, 4], [0, 1, 4]):
        check_aggregate(device, table, device_table, groupby, all_functions)
        check_aggregate(device, table, device_table, groupby, sums_only)
        check_aggregate(device, table, device_table, groupby, sums_only, predicates=[Predicate(4, capi.PRED_LESS_THAN, 100)])
    check_aggregate(device, table, device_table, [4], [])                       # DISTINCT (no aggregate functions)
    check_aggregate(device, table, device_table, [], [Aggregate(capi.AGG_COUNT_STAR)])
    device_table.drop()


def test_few_groups_fast_path(device):
    # <= 4 and <= 8 groups with the product-chain expressions of TPC-H; more than 8 groups falls back transparently
    rng = np.random.default_rng(3)
    rows = 100_000
    from hyrise_b200.storage import ColumnDefinition, Table
    definitions = [ColumnDefinition("g", capi.TYPE_INT32), ColumnDefinition("a", capi.TYPE_FLOAT32),
                   ColumnDefinition("b", capi.TYPE_FLOAT32, True), ColumnDefinition("c", capi.TYPE_FLOAT32),
                   ColumnDefinition("d", capi.TYPE_FLOAT64), ColumnDefinition("i", capi.TYPE_INT64, True)]
    for group_count in (1, 3, 4, 7, 8, 9, 40):
        columns = [rng.integers(100, 100 + group_count, rows, dtype=np.int32),
                   (rng.integers(90_000, 10_000_000, rows) / 100).astype(np.float32),
                   (rng.integers(0, 11, rows) / 100).astype(np.float32), (rng.integers(0, 9, rows) / 100).astype(np.float32),
                   rng.normal(0, 1e3, rows), rng.integers(-10 ** 9, 10 ** 9, rows, dtype=np.int64)]
        nulls = [None, None, rng.random(rows) < 0.05, None, None, rng.random(rows) < 0.05]
        table = Table.from_columns(definitions, columns, nulls, chunk_size=9_973).encode("Dictionary")
        device_table = device.upload(table)
        one = ("lit", capi.TYPE_INT32, 1)
        chain = [Aggregate(capi.AGG_SUM, Expression.column(1)),
                 Aggregate(capi.AGG_SUM, Expression([("col", 1), one, ("col", 2), "-", "*"])),
                 Aggregate(capi.AGG_SUM, Expression([("col", 1), one, ("col", 2), "-", "*", one, ("col", 3), "+", "*"])),
                 Aggregate(capi.AGG_AVG, Expression.column(2)), Aggregate(capi.AGG_COUNT, Expression.column(2)),
                 Aggregate(capi.AGG_COUNT_STAR)]
        check_aggregate(device, table, device_table, [0], chain)
        check_aggregate(device, table, device_table, [0], chain, predicates=[Predicate(3, capi.PRED_GREATER_THAN, 0.02)])
        check_aggregate(device, table, device_table, [0], [Aggregate(capi.AGG_SUM, Expression.column(4)),
                                                           Aggregate(capi.AGG_AVG, Expression.column(4))])
        check_aggregate(device, table, device_table, [0], [Aggregate(capi.AGG_SUM, Expression.column(5)),
                                                           Aggregate(capi.AGG_AVG, Expression.column(5)),
                                                           Aggregate(capi.AGG_COUNT, Expression.column(5))])
        # arithmetic outside the product-chain family -> general kernel (RPN interpreter)
        check_aggregate(device, table, device_table, [0], [Aggregate(capi.AGG_SUM, Expression(
            [("col", 1), ("col", 3), "+", ("lit", capi.TYPE_FLOAT64, 2.5), "/"]))])
        device_table.drop()


def test_tpch_q1_q6_real_data(device):
    # tpch_queries.cpp Q1 / Q6 on dbgen sf-0.01 with the reference's default encodings (FoR + dictionaries)
    table, _ = lineitem_table()
    device_table = device.upload(table)
    q1 = check_aggregate(device, table, device_table, [5, 6], Q1_AGGREGATES, predicates=Q1_PREDICATES)
    assert q1.group_count == 4
    check_aggregate(device, table, device_table, [], Q6_AGGREGATES, predicates=Q6_PREDICATES)
    # the unfused plan: chained TableScans feeding the aggregate through PosLists
    device_filter, oracle_filter = None, None
    for predicate in Q6_PREDICATES:
        device_filter = device.table_scan(device_table, predicate, device_filter)
        oracle_filter = orc.table_scan(table, predicate, oracle_filter)
    check_aggregate(device, table, device_table, [], Q6_AGGREGATES, filters=(device_filter, oracle_filter))
    device_table.drop()


def test_q1_non_finite_values_stay_in_their_group(device):
    """The streaming kernel adds every row to every group through a 0 / 1 mask (one DFMA instead of DADD + two selects); a
    step that holds inf / NaN / an overflowing product must take the select form, or 0 * inf = NaN would leak into the other
    groups. Poisoned rows sit in single groups; the others must still match the oracle to 1e-6."""
    from hyrise_b200.storage import ColumnDefinition, Table

    data = dict(tpch("sf-0.01_lineitem.npz"))
    names = ["l_orderkey", "l_quantity", "l_extendedprice", "l_discount", "l_tax", "l_returnflag", "l_linestatus", "l_shipdate"]
    types = [capi.TYPE_INT32] + [capi.TYPE_FLOAT32] * 4 + [capi.TYPE_STRING] * 3
    definitions = [ColumnDefinition(name, data_type) for name, data_type in zip(names, types)]
    flags, status = data["l_returnflag"], data["l_linestatus"]
    group_rows = {key: np.flatnonzero((flags == key[0]) & (status == key[1])) for key in ((b"A", b"F"), (b"R", b"F"), (b"N", b"O"))}
    overflowing = np.flatnonzero((flags == b"N") & (status == b"O") & (data["l_discount"] == 0) & (data["l_tax"] >= 0.02))[0]
    cases = [
        {"l_extendedprice": [(group_rows[(b"A", b"F")][5], np.inf)]},                       # +inf in one group
        {"l_quantity": [(group_rows[(b"R", b"F")][77], np.nan)]},                            # NaN in a raw-only column
        {"l_extendedprice": [(overflowing, 3.4e38)]},                                        # finite, price * 1 * (1 + tax) is not
        {"l_extendedprice": [(group_rows[(b"A", b"F")][9], np.inf), (group_rows[(b"A", b"F")][20_000 % 5_000], -np.inf)]},
    ]
    for poison in cases:
        columns = {name: np.array(data[name]) for name in names}
        for name, edits in poison.items():
            for row, value in edits:
                columns[name][row] = value
        table = Table.from_columns(definitions, [columns[name] for name in names], chunk_size=10_000).encode("Automatic")
        device_table = device.upload(table)
        got = check_aggregate(device, table, device_table, [5, 6], Q1_AGGREGATES, predicates=Q1_PREDICATES)
        assert got.group_count == 4
        poisoned = np.zeros(4, dtype=bool)
        for values in got.values:
            poisoned |= ~np.isfinite(values.astype(np.float64))
        assert poisoned.sum() == 1, got.values  # exactly one group is poisoned
        device_table.drop()


def test_generated_q1_sf1(device):
    """Q1 on the generated SF 1 lineitem (6 M rows, 65 535-row chunks) against the oracle on the same segments."""
    from hyrise_b200.tpch import TpchTables

    tables = TpchTables(1.0, seed=42)
    device_table = device.upload(tables.lineitem)
    predicates = [Predicate(7, capi.PRED_LESS_THAN_EQUALS, "1998-09-02")]
    expected = orc.aggregate_hash(tables.lineitem, [5, 6], Q1_AGGREGATES, predicates=predicates)
    got = device.aggregate_hash(device_table, [5, 6], Q1_AGGREGATES, predicates=predicates)
    assert_aggregate_outputs_equal(got, expected)
    assert got.group_count == 4 and int(got.values[7].sum()) > 5_800_000
    device_table.drop()
    tables.close()
