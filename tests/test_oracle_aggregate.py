"""Pins the oracle's AggregateHash restatement to the reference's golden result tables
(src/test/lib/operators/aggregate_test.cpp -> resources/test_data/tbl/aggregateoperator/**) and to SQLite for the
TPC-H Q1 / Q6 shapes on real dbgen data (the reference's own --verify oracle, benchmark_sql_executor.cpp:106). CPU only."""
import sqlite3

import numpy as np
import pytest

import oracle_lib as orc
from aggregate_cases import CASES
from helpers import aggregate_rows, assert_rows_match_unordered, expected_rows, tbl, tpch
from hyrise_b200 import capi
from hyrise_b200.device import Aggregate, Expression, Predicate
from hyrise_b200.storage import ColumnDefinition, Table


def make_aggregates(definitions):
    return [Aggregate(function, None if column is None else Expression.column(column)) for column, function in definitions]


@pytest.mark.parametrize("case", CASES, ids=[f"{c[0]}@{c[1]}" for c in CASES])
def test_reference_golden_tables(case):
    name, line, input_file, chunk_size, dictionary, definitions, groupby, expected_file, on_reference_table = case
    table = tbl(input_file, chunk_size)
    if dictionary:
        table.encode("Dictionary")
    want = expected_rows(tbl(expected_file))
    output = orc.aggregate_hash(table, groupby, make_aggregates(definitions))
    assert_rows_match_unordered(aggregate_rows(table, groupby, output), want)
    if on_reference_table:
        # test_output's second half: the same aggregate on a TableScan(column 0 > 0) output (aggregate_test.cpp:67-76)
        scan = orc.table_scan(table, Predicate(0, capi.PRED_GREATER_THAN, 0)) \
            if table.column_definitions[0].data_type != capi.TYPE_STRING else None
        if scan is not None:
            output = orc.aggregate_hash(table, groupby, make_aggregates(definitions), input_filter=scan)
            assert_rows_match_unordered(aggregate_rows(table, groupby, output), want)


def test_empty_input_without_groupby():
    # aggregate_hash.cpp:1395-1405: no rows and no GROUP BY -> one row, NULL for SUM/MIN/MAX/AVG and 0 for COUNT
    table = tbl("aggregateoperator/groupby_int_1gb_1agg/input.tbl", 2)
    nothing = orc.table_scan(table, Predicate(0, capi.PRED_GREATER_THAN, 10 ** 9))
    output = orc.aggregate_hash(table, [], make_aggregates([(1, capi.AGG_MAX), (1, capi.AGG_COUNT), (None, capi.AGG_COUNT_STAR)]),
                                input_filter=nothing)
    assert output.group_count == 1
    assert output.nulls[0][0] and output.values[1][0] == 0 and output.values[2][0] == 0
    output = orc.aggregate_hash(table, [0], make_aggregates([(1, capi.AGG_MAX)]), input_filter=nothing)
    assert output.group_count == 0


def test_group_order_and_immediate_keys():
    # first-appearance order (get_or_add_result, aggregate_hash.cpp:317-403) vs the immediate key shortcut (:781-804)
    definitions = [ColumnDefinition("k", capi.TYPE_INT32, True), ColumnDefinition("v", capi.TYPE_INT32)]
    keys = np.array([7, 3, 7, 5, 3, 9, 0, 5], dtype=np.int32)
    nulls = np.array([0, 0, 0, 0, 0, 0, 1, 0], dtype=bool)
    table = Table.from_columns(definitions, [keys, np.arange(8, dtype=np.int32)], [nulls, None], chunk_size=3)
    output = orc.aggregate_hash(table, [0], make_aggregates([(1, capi.AGG_SUM)]))
    assert output.used_immediate_keys                       # key range 3..9 < 1.2 * 8 rows
    assert [None if n else v for v, n in zip(output.values[0].tolist(), output.nulls[0].tolist())] == [6, 1 + 4, 3 + 7, 0 + 2, 5]
    # representative row = last row of the group in immediate mode (:367)
    assert [(int(r["chunk_id"]), int(r["chunk_offset"])) for r in output.row_ids] == [(2, 0), (1, 1), (2, 1), (0, 2), (1, 2)]
    wide = keys.copy()
    wide[0] = 1000                                           # range too wide -> hash path, first-appearance order
    table = Table.from_columns(definitions, [wide, np.arange(8, dtype=np.int32)], [nulls, None], chunk_size=3)
    output = orc.aggregate_hash(table, [0], make_aggregates([(1, capi.AGG_SUM)]))
    assert not output.used_immediate_keys
    assert output.values[0].tolist() == [0, 1 + 4, 2, 3 + 7, 5, 6]
    assert [(int(r["chunk_id"]), int(r["chunk_offset"])) for r in output.row_ids] == [(0, 0), (0, 1), (0, 2), (1, 0), (1, 2), (2, 0)]


def lineitem_table(scale="sf-0.01", chunk_size=10_000):
    data = tpch(f"{scale}_lineitem.npz")
    names = ["l_orderkey", "l_quantity", "l_extendedprice", "l_discount", "l_tax", "l_returnflag", "l_linestatus", "l_shipdate"]
    types = [capi.TYPE_INT32] + [capi.TYPE_FLOAT32] * 4 + [capi.TYPE_STRING] * 3
    definitions = [ColumnDefinition(name, data_type) for name, data_type in zip(names, types)]
    table = Table.from_columns(definitions, [data[name] for name in names], chunk_size=chunk_size).encode("Automatic")
    return table, data


Q1_AGGREGATES = [
    Aggregate(capi.AGG_SUM, Expression.column(1)),
    Aggregate(capi.AGG_SUM, Expression.column(2)),
    Aggregate(capi.AGG_SUM, Expression([("col", 2), ("lit", capi.TYPE_INT32, 1), ("col", 3), "-", "*"])),
    Aggregate(capi.AGG_SUM, Expression([("col", 2), ("lit", capi.TYPE_INT32, 1), ("col", 3), "-", "*",
                                        ("lit", capi.TYPE_INT32, 1), ("col", 4), "+", "*"])),
    Aggregate(capi.AGG_AVG, Expression.column(1)),
    Aggregate(capi.AGG_AVG, Expression.column(2)),
    Aggregate(capi.AGG_AVG, Expression.column(3)),
    Aggregate(capi.AGG_COUNT_STAR),
]
Q1_PREDICATES = [Predicate(7, capi.PRED_LESS_THAN_EQUALS, b"1998-09-02")]
# l_discount BETWEEN 0.05 AND 0.07001 / l_quantity < 24 after lossless_predicate_cast to float (tpch_queries.cpp:206-210)
def next_float_towards(value: float, towards: float) -> np.float32:
    """utils/lossless_predicate_cast.cpp:18-38: the float to compare a float column with instead of a double literal."""
    casted = np.float32(value)
    if (float(casted) < value and towards < value) or (float(casted) > value and towards > value):
        return casted
    return np.nextafter(casted, np.float32(towards), dtype=np.float32)


Q6_PREDICATES = [
    Predicate(7, capi.PRED_BETWEEN_UPPER_EXCLUSIVE, b"1994-01-01", b"1995-01-01"),
    # x >= 0.05 <=> x >= next(0.05); x <= 0.07001 <=> x <= prev(0.07001)   (lossless_predicate_cast.hpp:36-56)
    Predicate(3, capi.PRED_BETWEEN_INCLUSIVE, next_float_towards(0.05, float("inf")), next_float_towards(0.07001, float("-inf"))),
    Predicate(1, capi.PRED_LESS_THAN, 24.0),
]
Q6_AGGREGATES = [Aggregate(capi.AGG_SUM, Expression([("col", 2), ("col", 3), "*"]))]


def sqlite_lineitem(data):
    connection = sqlite3.connect(":memory:")
    connection.execute("create table lineitem (l_quantity real, l_extendedprice real, l_discount real, l_tax real, "
                       "l_returnflag text, l_linestatus text, l_shipdate text)")
    rows = zip(data["l_quantity"].astype(float).tolist(), data["l_extendedprice"].astype(float).tolist(),
               data["l_discount"].astype(float).tolist(), data["l_tax"].astype(float).tolist(),
               [v.decode() for v in data["l_returnflag"]], [v.decode() for v in data["l_linestatus"]],
               [v.decode() for v in data["l_shipdate"]])
    connection.executemany("insert into lineitem values (?,?,?,?,?,?,?)", rows)
    return connection


def test_tpch_q1_against_sqlite():
    # tpch_queries.cpp:38-46 on resources/test_data/tbl/tpch/sf-0.01; SQLite computes in double, the reference computes
    # the products in float (expression_utils.cpp:172-205), hence the check_table_equal-style relative tolerance.
    table, data = lineitem_table()
    output = orc.aggregate_hash(table, [5, 6], Q1_AGGREGATES, predicates=Q1_PREDICATES)
    connection = sqlite_lineitem(data)
    want = connection.execute(
        "select l_returnflag, l_linestatus, sum(l_quantity), sum(l_extendedprice), sum(l_extendedprice*(1-l_discount)), "
        "sum(l_extendedprice*(1-l_discount)*(1+l_tax)), avg(l_quantity), avg(l_extendedprice), avg(l_discount), count(*) "
        "from lineitem where l_shipdate <= '1998-09-02' group by l_returnflag, l_linestatus").fetchall()
    want = [tuple(v.encode() if isinstance(v, str) else v for v in row) for row in want]
    assert output.group_count == 4
    assert_rows_match_unordered(aggregate_rows(table, [5, 6], output), want, rel=1e-4)


def test_tpch_q6_against_sqlite():
    table, data = lineitem_table()
    output = orc.aggregate_hash(table, [], Q6_AGGREGATES, predicates=Q6_PREDICATES)
    connection = sqlite_lineitem(data)
    want = connection.execute(
        "select sum(l_extendedprice*l_discount) from lineitem where l_shipdate >= '1994-01-01' and "
        "l_shipdate < '1995-01-01' and l_discount between 0.05 and 0.07001 and l_quantity < 24").fetchall()
    assert_rows_match_unordered(aggregate_rows(table, [], output), want, rel=1e-4)


def test_chunk_parallel_phases_do_not_change_the_result():
    """The CPU arm runs the Projection and the group-key partitioning as one job per chunk (like the reference's JobTasks)
    and the aggregation phase on one thread: the output must be identical to the fully sequential run, bit for bit."""
    from helpers import random_table
    from hyrise_b200.tpch import TpchTables, L_DISCOUNT, L_EXTENDEDPRICE, L_LINESTATUS, L_QUANTITY, L_RETURNFLAG, L_SHIPDATE, L_TAX
    tables = TpchTables(0.05, seed=7)
    one = ("lit", capi.TYPE_INT32, 1)
    aggregates = [Aggregate(capi.AGG_SUM, Expression.column(L_QUANTITY)),
                  Aggregate(capi.AGG_SUM, Expression([("col", L_EXTENDEDPRICE), one, ("col", L_DISCOUNT), "-", "*", one,
                                                      ("col", L_TAX), "+", "*"])),
                  Aggregate(capi.AGG_AVG, Expression.column(L_DISCOUNT)), Aggregate(capi.AGG_COUNT_STAR)]
    predicates = [Predicate(L_SHIPDATE, capi.PRED_LESS_THAN_EQUALS, "1998-09-02")]
    sequential = orc.aggregate_hash(tables.lineitem, [L_RETURNFLAG, L_LINESTATUS], aggregates, predicates=predicates, threads=1)
    parallel = orc.aggregate_hash(tables.lineitem, [L_RETURNFLAG, L_LINESTATUS], aggregates, predicates=predicates, threads=6)
    assert sequential.group_count == parallel.group_count == 4
    assert np.array_equal(sequential.row_ids, parallel.row_ids)
    for a, b in zip(sequential.values, parallel.values):
        assert np.array_equal(a, b)
    rng = np.random.default_rng(9)
    table = random_table(rng, 30_000, 1_999).encode("Dictionary")
    mixed = [Aggregate(capi.AGG_SUM, Expression.column(2)), Aggregate(capi.AGG_MIN, Expression.column(1)),
             Aggregate(capi.AGG_AVG, Expression.column(3)), Aggregate(capi.AGG_COUNT, Expression.column(0))]
    for groupby in ([4], [0, 4], []):
        sequential = orc.aggregate_hash(table, groupby, mixed, threads=1)
        parallel = orc.aggregate_hash(table, groupby, mixed, threads=5)
        assert np.array_equal(sequential.row_ids, parallel.row_ids)
        for a, b, na, nb in zip(sequential.values, parallel.values, sequential.nulls, parallel.nulls):
            assert np.array_equal(na, nb) and np.array_equal(a[~na], b[~nb])
