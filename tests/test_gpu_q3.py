"""TPC-H Q3 composed from the device operators (SURVEY.md 8f-3): scans feeding joins, a join's output feeding the next join
(PosLists in result order referencing many chunks), a high-cardinality group-by over a join's output, ORDER BY revenue DESC
LIMIT 10 — on dbgen sf-0.01 against SQLite running the reference's query text (tpch_queries.cpp:92-109), which is how the
reference verifies itself (benchmark_sql_executor.cpp:106-, --verify)."""
import sqlite3

import numpy as np
import pytest

import oracle_lib as orc
from helpers import row_ids_equal, tpch
from hyrise_b200 import capi
from hyrise_b200.device import Aggregate, Expression, Predicate
from hyrise_b200.storage import ColumnDefinition, Table

pytestmark = pytest.mark.gpu

Q3_SQL = """SELECT l_orderkey, SUM(l_extendedprice*(1.0-l_discount)) as revenue, o_orderdate, o_shippriority
      FROM customer, orders, lineitem
      WHERE c_mktsegment = 'BUILDING' AND c_custkey = o_custkey AND l_orderkey = o_orderkey
      AND o_orderdate < '1995-03-15' AND l_shipdate > '1995-03-15'
      GROUP BY l_orderkey, o_orderdate, o_shippriority ORDER BY revenue DESC, o_orderdate LIMIT 10"""


def load(name, columns, chunk_size, encoding="Automatic"):
    data = tpch(f"sf-0.01_{name}.npz")
    definitions, arrays = [], []
    for column in columns:
        values = data[column]
        if values.dtype.kind == "S":
            definitions.append(ColumnDefinition(column, capi.TYPE_STRING))
            arrays.append(values)
        elif values.dtype == np.float32:
            definitions.append(ColumnDefinition(column, capi.TYPE_FLOAT32))
            arrays.append(values)
        else:
            definitions.append(ColumnDefinition(column, capi.TYPE_INT32))
            arrays.append(values)
    return Table.from_columns(definitions, arrays, chunk_size=chunk_size).encode(encoding), data


@pytest.mark.parametrize("radix_bits", [0, 3])
def test_q3_against_sqlite(device, radix_bits):
    customer, customer_data = load("customer", ["c_custkey", "c_mktsegment"], 400)
    orders, orders_data = load("orders", ["o_orderkey", "o_custkey", "o_orderdate", "o_shippriority"], 4_000)
    lineitem, lineitem_data = load("lineitem", ["l_orderkey", "l_extendedprice", "l_discount", "l_shipdate"], 16_000)
    customer_dev, orders_dev, lineitem_dev = device.upload(customer), device.upload(orders), device.upload(lineitem)

    # sigma(customer), sigma(orders), sigma(lineitem)
    building = device.table_scan(customer_dev, Predicate(1, capi.PRED_EQUALS, b"BUILDING"))
    early_orders = device.table_scan(orders_dev, Predicate(2, capi.PRED_LESS_THAN, b"1995-03-15"))
    late_lines = device.table_scan(lineitem_dev, Predicate(3, capi.PRED_GREATER_THAN, b"1995-03-15"))
    # customer |x| orders on custkey; its orders side (a PosList in result order over many chunks) feeds the next join
    first = device.join_hash(customer_dev, 0, orders_dev, 1, capi.JOIN_INNER, radix_bits, build_filter=building,
                             probe_filter=early_orders)
    expected_first = orc.join_hash(customer, 0, orders, 1, capi.JOIN_INNER, radix_bits,
                                   build_filter=orc.table_scan(customer, Predicate(1, capi.PRED_EQUALS, b"BUILDING")),
                                   probe_filter=orc.table_scan(orders, Predicate(2, capi.PRED_LESS_THAN, b"1995-03-15")))
    assert first.info()[0] == expected_first.pair_count
    if radix_bits > 0:
        # (with radix_bits == 0 the reference's probe "partitions" are the input chunks, join_hash.cpp:294: it cuts the
        # result per probe input chunk; the device result is one partition — DESIGN.md)
        chunks = first.output_chunks()
        assert np.array_equal(chunks, expected_first.output_chunk_offsets), "write_output_chunks slicing differs"
    qualifying_orders = first.pos_list(1)
    total, chunk_count = qualifying_orders.info()
    assert total == expected_first.pair_count and chunk_count == 1
    assert row_ids_equal(qualifying_orders.to_host(), expected_first.probe)
    # (customer |x| orders) |x| lineitem on orderkey
    second = device.join_hash(orders_dev, 0, lineitem_dev, 0, capi.JOIN_INNER, radix_bits, build_filter=qualifying_orders,
                              probe_filter=late_lines)
    joined_lines = second.pos_list(1)
    # GROUP BY l_orderkey (o_orderdate and o_shippriority depend on it) over the join's output, SUM(price * (1 - discount))
    revenue = Aggregate(capi.AGG_SUM, Expression([("col", 1), ("lit", capi.TYPE_FLOAT64, 1.0), ("col", 2), "-", "*"]))
    output = device.aggregate_hash(lineitem_dev, [0], [revenue], input_filter=joined_lines, keep_result=True)
    top = device.aggregate_top_k(output.result_handle, 0, 10, descending=True)
    device.free_aggregate_result(output.result_handle)

    # --- SQLite on the same data, the reference's query text
    connection = sqlite3.connect(":memory:")
    connection.execute("CREATE TABLE customer (c_custkey INT, c_mktsegment TEXT)")
    connection.execute("CREATE TABLE orders (o_orderkey INT, o_custkey INT, o_orderdate TEXT, o_shippriority INT)")
    connection.execute("CREATE TABLE lineitem (l_orderkey INT, l_extendedprice REAL, l_discount REAL, l_shipdate TEXT)")
    connection.executemany("INSERT INTO customer VALUES (?, ?)",
                           zip(customer_data["c_custkey"].tolist(), [s.decode() for s in customer_data["c_mktsegment"]]))
    connection.executemany("INSERT INTO orders VALUES (?, ?, ?, ?)",
                           zip(orders_data["o_orderkey"].tolist(), orders_data["o_custkey"].tolist(),
                               [s.decode() for s in orders_data["o_orderdate"]], orders_data["o_shippriority"].tolist()))
    connection.executemany("INSERT INTO lineitem VALUES (?, ?, ?, ?)",
                           zip(lineitem_data["l_orderkey"].tolist(), lineitem_data["l_extendedprice"].astype(np.float64).tolist(),
                               lineitem_data["l_discount"].astype(np.float64).tolist(), [s.decode() for s in lineitem_data["l_shipdate"]]))
    expected_rows = connection.execute(Q3_SQL).fetchall()
    all_groups = connection.execute(Q3_SQL.split("ORDER BY")[0]).fetchall()
    assert output.group_count == len(all_groups)
    assert len(top) == len(expected_rows) == 10

    order_keys = lineitem_data["l_orderkey"]
    lines_per_chunk = 16_000
    order_date = dict(zip(orders_data["o_orderkey"].tolist(), [s.decode() for s in orders_data["o_orderdate"]]))
    for rank, group in enumerate(top):
        row = output.row_ids[group]
        key = int(order_keys[int(row["chunk_id"]) * lines_per_chunk + int(row["chunk_offset"])])
        want_key, want_revenue, want_date, _ = expected_rows[rank]
        assert key == want_key, (rank, key, want_key)
        assert abs(output.values[0][group] - want_revenue) <= 1e-5 * abs(want_revenue), (rank, output.values[0][group], want_revenue)
        assert order_date[key] == want_date
    for handle in (building, early_orders, late_lines, qualifying_orders, joined_lines):
        handle.free()
    first.free()
    second.free()
    for table in (customer_dev, orders_dev, lineitem_dev):
        table.drop()
