"""Pins the oracle's JoinHash restatement to the reference's known answers (join_hash_steps_test.cpp,
join_hash_test.cpp) and to JoinVerification semantics on the join_test_runner inputs. CPU only."""
import itertools

import numpy as np
import pytest

import oracle_lib as orc
from helpers import join_result_rows, rows_with_keys, tbl, tpch, verification_join
from hyrise_b200 import capi
from hyrise_b200.storage import ColumnDefinition, Table

MODES = [capi.JOIN_INNER, capi.JOIN_LEFT, capi.JOIN_SEMI, capi.JOIN_ANTI_NULL_AS_TRUE, capi.JOIN_ANTI_NULL_AS_FALSE]


def test_radix_bit_calculation():
    # join_hash_test.cpp:122-129 + the config-3 value derived in SURVEY.md §8a (15 M build rows -> 7 bits)
    lib = orc.load()
    assert lib.orc_calculate_radix_bits(1, 0) == 0
    assert lib.orc_calculate_radix_bits(0, 1) == 0
    assert lib.orc_calculate_radix_bits(0, 0) == 0
    assert lib.orc_calculate_radix_bits(1, 1) == 0
    assert lib.orc_calculate_radix_bits(2 ** 64 - 1, 2 ** 64 - 1) > 0
    assert lib.orc_calculate_radix_bits(15_000_000, 59_986_052) == 7
    assert lib.orc_calculate_radix_bits(150_000_000, 600_037_902) == 8


def test_materialize_output_bloom_filter():
    # join_hash_steps_test.cpp:169-188: std::hash<int> is the identity -> slots 0, 6, 7, 9, 13, 18
    table = tbl("int_int4_with_null.tbl", 10)
    _, _, _, _, bloom = orc.debug_materialize(table, 0, False, 1)
    assert bloom.tolist() == [0, 6, 7, 9, 13, 18]


def test_materialize_input_bloom_filter():
    # join_hash_steps_test.cpp:190-220
    table = tbl("int_int4_with_null.tbl", 10)
    values, row_ids, _, _, _ = orc.debug_materialize(table, 0, False, 1, input_bloom_slots=[6, 7, 9])
    assert values.tolist() == [7, 7, 9, 6, 9, 7]
    assert row_ids["chunk_offset"].tolist() == [1, 2, 3, 4, 8, 9]


def test_materialize_keep_nulls():
    # join_hash_steps_test.cpp:106-167
    table = tbl("int_int4_with_null.tbl", 10)
    with_nulls = orc.debug_materialize(table, 0, True, 0)
    without_nulls = orc.debug_materialize(table, 0, False, 0)
    assert len(with_nulls[0]) == table.row_count
    assert len(without_nulls[0]) < table.row_count
    assert without_nulls[0][6] == 9
    assert with_nulls[0][6] == 13
    _, nulls = table.column_values(0)
    assert with_nulls[2].tolist() == nulls.tolist()


def test_materialize_histograms():
    # join_hash_steps_test.cpp:222-263: 0/1 table, chunk size 10
    table = Table.from_columns([ColumnDefinition("a", capi.TYPE_INT32)], [np.arange(1000, dtype=np.int32) % 2],
                               chunk_size=10)
    histograms = orc.debug_materialize(table, 0, False, 1)[3]
    assert histograms.shape == (100, 2) and (histograms == 5).all()
    histograms = orc.debug_materialize(table, 0, False, 2)[3]
    assert ((histograms == 5) | (histograms == 0)).all() and int((histograms == 0).sum()) == 200


def int_column_pairs():
    # l_int, l_int_null, l_long, l_long_null columns are 0, 1, 6, 7
    return [(0, 0), (1, 1), (0, 1), (6, 6), (7, 7), (0, 6), (7, 1)]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("radix_bits", [0, 1, 2, 5])                 # join_test_runner.cpp radix bit choices
@pytest.mark.parametrize("sizes", [(10, 15), (15, 10), (0, 10), (10, 0), (0, 0), (15, 15)])
@pytest.mark.parametrize("chunk_size", [10, 3, 1])
def test_join_test_runner_inputs(mode, radix_bits, sizes, chunk_size):
    # join_test_runner.cpp:184-543 configurations over the int/long key columns, compared against nested-loop semantics
    left = tbl(f"join_test_runner/input_table_left_{sizes[0]}.tbl", chunk_size)
    right = tbl(f"join_test_runner/input_table_right_{sizes[1]}.tbl", chunk_size)
    for left_column, right_column in int_column_pairs():
        # JoinHash::_on_execute side selection (join_hash.cpp:139-155): probe = left for Semi/Anti/Left; for Inner the
        # smaller table is the build side.
        if mode == capi.JOIN_INNER and left.row_count <= right.row_count:
            build, build_column, probe, probe_column = left, left_column, right, right_column
        else:
            build, build_column, probe, probe_column = right, right_column, left, left_column
        result = orc.join_hash(build, build_column, probe, probe_column, mode, radix_bits)
        got = join_result_rows(result.build, result.probe)
        want = verification_join(rows_with_keys(build, build_column), rows_with_keys(probe, probe_column), mode)
        assert sorted(got) == sorted(want), (mode, radix_bits, sizes, left_column, right_column)
        assert result.partition_offsets[-1] == len(got)


def test_tpch_sf0001_join():
    # join_hash_test.cpp:26-46, 70-82: orders x lineitem on orderkey, chunk size 10, 10 radix bits -> use the maximum 8
    lineitem = tpch("sf-0.001_lineitem.npz")
    orders = tpch("sf-0.001_orders.npz")
    orders_table = Table.from_columns([ColumnDefinition("o_orderkey", capi.TYPE_INT32)], [orders["o_orderkey"]],
                                      chunk_size=10)
    lineitem_table = Table.from_columns([ColumnDefinition("l_orderkey", capi.TYPE_INT32)], [lineitem["l_orderkey"]],
                                        chunk_size=10)
    result = orc.join_hash(orders_table, 0, lineitem_table, 0, capi.JOIN_INNER, 8)
    assert result.pair_count == len(lineitem["l_orderkey"])  # every lineitem has exactly one order
    # output chunks after write_output_chunks merging never exceed the input chunk count (the ChunkCount test)
    assert len(result.output_chunk_offsets) - 1 <= max(orders_table.chunk_count, lineitem_table.chunk_count)
    keys = orders["o_orderkey"]
    build_index = result.build["chunk_id"].astype(np.int64) * 10 + result.build["chunk_offset"]
    probe_index = result.probe["chunk_id"].astype(np.int64) * 10 + result.probe["chunk_offset"]
    assert (keys[build_index] == lineitem["l_orderkey"][probe_index]).all()
    # order: partition-major, probe order inside a partition
    partitions = lineitem["l_orderkey"][probe_index] & 255
    assert (np.diff(partitions) >= 0).all()
    for partition in np.unique(partitions):
        assert (np.diff(probe_index[partitions == partition]) > 0).all()
