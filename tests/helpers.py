"""Shared helpers for the parity tests."""
from __future__ import annotations

import os

import numpy as np

from hyrise_b200 import capi
from hyrise_b200.device import ROW_ID_DTYPE, Predicate
from hyrise_b200.storage import ColumnDefinition, Table, load_table

HERE = os.path.dirname(os.path.abspath(__file__))
TBL = os.path.join(HERE, "golden", "tbl")
TPCH = os.path.join(HERE, "golden", "tpch")

ENCODINGS = ["Unencoded", "Dictionary", "FrameOfReference"]  # table_scan_test.cpp:267-270 minus RunLength


def tbl(name: str, chunk_size: int = capi.DEFAULT_CHUNK_SIZE) -> Table:
    return load_table(os.path.join(TBL, name), chunk_size)


def tpch(name: str):
    return np.load(os.path.join(TPCH, name))


def column_values_at(table: Table, column_id: int, row_ids: np.ndarray):
    """Dereference RowIDs like a ReferenceSegment (reference_segment.hpp): list of python values, None for NULL."""
    out = []
    cache = {}
    for row in row_ids:
        chunk_id, offset = int(row["chunk_id"]), int(row["chunk_offset"])
        if chunk_id not in cache:
            segment = table.chunks[chunk_id].segments[column_id]
            cache[chunk_id] = (segment.decode(), segment.null_mask())
        values, nulls = cache[chunk_id]
        out.append(None if nulls[offset] else values[offset].item())
    return out


def row_ids_equal(a: np.ndarray, b: np.ndarray) -> bool:
    a = np.ascontiguousarray(a, dtype=ROW_ID_DTYPE)
    b = np.ascontiguousarray(b, dtype=ROW_ID_DTYPE)
    return a.shape == b.shape and bool(np.array_equal(a.view(np.uint64), b.view(np.uint64)))


def assert_pos_lists_equal(device_rows, device_offsets, oracle_list) -> None:
    assert np.array_equal(np.asarray(device_offsets, dtype=np.uint64), oracle_list.chunk_offsets), \
        "per-chunk PosList boundaries differ"
    assert row_ids_equal(device_rows, oracle_list.row_ids), "RowIDs differ"


def random_table(rng: np.random.Generator, rows: int, chunk_size: int, with_nulls: bool = True) -> Table:
    """Five-type table (int, long, float, double + a low-cardinality int) for randomized parity runs."""
    definitions = [
        ColumnDefinition("i", capi.TYPE_INT32, with_nulls),
        ColumnDefinition("l", capi.TYPE_INT64, with_nulls),
        ColumnDefinition("f", capi.TYPE_FLOAT32, with_nulls),
        ColumnDefinition("d", capi.TYPE_FLOAT64, with_nulls),
        ColumnDefinition("k", capi.TYPE_INT32, False),
    ]
    columns = [
        rng.integers(-1000, 1000, rows, dtype=np.int32),
        rng.integers(-(10 ** 12), 10 ** 12, rows, dtype=np.int64),
        (rng.integers(0, 2000, rows) / 8).astype(np.float32),
        rng.normal(0, 100, rows).astype(np.float64),
        rng.integers(0, 300, rows, dtype=np.int32),
    ]
    nulls = [(rng.random(rows) < 0.1) if (with_nulls and d.nullable) else None for d in definitions]
    return Table.from_columns(definitions, columns, nulls, chunk_size)


# ---------------------------------------------------------------------------------------------------------------------
# JoinVerification (src/lib/operators/join_verification.cpp:50-213): nested-loop semantics, used unordered.
# ---------------------------------------------------------------------------------------------------------------------
def rows_with_keys(table: Table, column_id: int, filter_list=None):
    """[(RowID tuple, key or None)] in table order (or filter order)."""
    out = []
    if filter_list is not None:
        cache = {}
        for row in filter_list.row_ids:
            chunk_id, offset = int(row["chunk_id"]), int(row["chunk_offset"])
            if chunk_id not in cache:
                segment = table.chunks[chunk_id].segments[column_id]
                cache[chunk_id] = (segment.decode(), segment.null_mask())
            values, nulls = cache[chunk_id]
            out.append(((chunk_id, offset), None if nulls[offset] else values[offset].item()))
        return out
    for chunk_id, chunk in enumerate(table.chunks):
        segment = chunk.segments[column_id]
        values, nulls = segment.decode(), segment.null_mask()
        for offset in range(segment.row_count):
            out.append(((chunk_id, offset), None if nulls[offset] else values[offset].item()))
    return out


NULL_ROW = (0xFFFFFFFF, 0xFFFFFFFF)


def verification_join(build_rows, probe_rows, mode):
    """Multiset of output rows: (build RowID, probe RowID) pairs, or probe RowIDs for Semi/Anti."""
    out = []
    build_has_null = any(key is None for _, key in build_rows)
    build_keys = {}
    for row_id, key in build_rows:
        if key is not None:
            build_keys.setdefault(key, []).append(row_id)
    for probe_id, key in probe_rows:
        matches = build_keys.get(key, []) if key is not None else []
        if mode == capi.JOIN_INNER:
            out.extend((b, probe_id) for b in matches)
        elif mode in (capi.JOIN_LEFT, capi.JOIN_RIGHT):
            if matches:
                out.extend((b, probe_id) for b in matches)
            else:
                out.append((NULL_ROW, probe_id))
        elif mode == capi.JOIN_SEMI:
            if matches:
                out.append(probe_id)
        elif mode == capi.JOIN_ANTI_NULL_AS_FALSE:
            if not matches:
                out.append(probe_id)
        elif mode == capi.JOIN_ANTI_NULL_AS_TRUE:
            if not build_rows:
                out.append(probe_id)
            elif key is not None and not matches and not build_has_null:
                out.append(probe_id)
    return out


def reference_join_order(build_rows, probe_rows, mode, radix_bits):
    """The exact output sequence of JoinHashImpl (join_hash_steps.hpp:509-922): grouped by key & (2^bits - 1) (std::hash
    of an int is the identity; NULL probe rows hash their placeholder value), inside a partition in probe order, for
    one probe row in build order."""
    mask = (1 << radix_bits) - 1
    build_has_null = any(key is None for _, key in build_rows)
    if mode == capi.JOIN_ANTI_NULL_AS_TRUE and build_has_null:
        return []
    build_keys = {}
    for row_id, key in build_rows:
        if key is not None:
            build_keys.setdefault(key, []).append(row_id)
    partitions = [[] for _ in range(mask + 1)]
    for probe_id, key, null_placeholder in probe_rows:
        value = null_placeholder if key is None else key
        partitions[value & mask].append((probe_id, key))
    out = []
    for rows in partitions:
        for probe_id, key in rows:
            matches = build_keys.get(key, []) if key is not None else []
            if mode == capi.JOIN_INNER:
                out.extend((b, probe_id) for b in matches)
            elif mode in (capi.JOIN_LEFT, capi.JOIN_RIGHT):
                out.extend((b, probe_id) for b in matches) if matches else out.append((NULL_ROW, probe_id))
            elif mode == capi.JOIN_SEMI:
                if matches:
                    out.append(probe_id)
            elif mode == capi.JOIN_ANTI_NULL_AS_FALSE:
                if not matches:
                    out.append(probe_id)
            elif mode == capi.JOIN_ANTI_NULL_AS_TRUE:
                if (not build_rows) or (key is not None and not matches):
                    out.append(probe_id)
    return out


def join_result_rows(build_rows_array, probe_rows_array):
    probe = [(int(r["chunk_id"]), int(r["chunk_offset"])) for r in probe_rows_array]
    if build_rows_array is None:
        return probe
    build = [(int(r["chunk_id"]), int(r["chunk_offset"])) for r in build_rows_array]
    return list(zip(build, probe))


# ---------------------------------------------------------------------------------------------------------------------
# Aggregate result comparison (check_table_equal.cpp:34,109-116: unordered rows, relative float tolerance)
# ---------------------------------------------------------------------------------------------------------------------
def aggregate_rows(table: Table, groupby_column_ids, output) -> list[tuple]:
    """Result rows (group-by values dereferenced through the representative RowIDs, then the aggregate values)."""
    rows = []
    group_values = [column_values_at(table, column_id, output.row_ids) if output.group_count else []
                    for column_id in groupby_column_ids]
    for g in range(output.group_count):
        row = [values[g] for values in group_values]
        for values, nulls in zip(output.values, output.nulls):
            row.append(None if nulls[g] else values[g].item())
        rows.append(tuple(row))
    return rows


def expected_rows(table: Table) -> list[tuple]:
    columns = []
    for column_id in range(table.column_count):
        values, nulls = table.column_values(column_id)
        columns.append([None if null else (bytes(v) if isinstance(v, bytes) else v.item())
                        for v, null in zip(values, nulls)])
    return list(zip(*columns)) if columns and len(columns[0]) else []


def _cell_close(a, b, rel=1e-6) -> bool:
    if a is None or b is None:
        return a is None and b is None
    if isinstance(a, bytes) or isinstance(b, bytes):
        return a == b
    if isinstance(a, float) or isinstance(b, float):
        return abs(float(a) - float(b)) <= rel * max(1.0, abs(float(a)), abs(float(b)))
    return a == b


def assert_rows_match_unordered(got: list[tuple], want: list[tuple], rel=1e-6) -> None:
    assert len(got) == len(want), f"row count {len(got)} != {len(want)}\n got {got}\nwant {want}"
    remaining = list(want)
    for row in got:
        for index, candidate in enumerate(remaining):
            if len(candidate) == len(row) and all(_cell_close(a, b, rel) for a, b in zip(row, candidate)):
                remaining.pop(index)
                break
        else:
            raise AssertionError(f"row {row} not expected; remaining {remaining}")


def assert_aggregate_outputs_equal(device_output, oracle_output, rel=1e-6) -> None:
    """Device vs oracle: same groups in the same order, same representative rows, integers exact, floats within rel."""
    assert device_output.group_count == oracle_output.group_count
    assert device_output.used_immediate_keys == oracle_output.used_immediate_keys
    assert row_ids_equal(device_output.row_ids, oracle_output.row_ids), \
        f"representative RowIDs differ:\n{device_output.row_ids}\n{oracle_output.row_ids}"
    assert device_output.value_types == oracle_output.value_types
    for index, (got, want) in enumerate(zip(device_output.values, oracle_output.values)):
        assert np.array_equal(device_output.nulls[index], oracle_output.nulls[index]), f"aggregate {index}: NULLs differ"
        valid = ~oracle_output.nulls[index]
        if got.dtype.kind in "iu":
            assert np.array_equal(got[valid], want[valid]), f"aggregate {index}: {got} != {want}"
        else:
            assert np.allclose(got[valid], want[valid], rtol=rel, atol=0.0, equal_nan=True), f"aggregate {index}: {got} != {want}"


# ---- table_scan_between_test.cpp: the parameterised fixture (:43-96) and the literal expectations (:194-243) ------------
BETWEEN_CASES = {
    "BetweenInclusive": [
        (12.25, 16.25, [1, 2, 3]), (12.0, 16.25, [1, 2, 3]), (12.25, 16.75, [1, 2, 3]), (12.0, 16.75, [1, 2, 3]),
        (0.0, 16.75, [0, 1, 2, 3]), (16.0, 50.75, [3, 4, 5, 6, 7, 8, 9, 10]), (13.0, 16.25, [2, 3]), (12.25, 15.0, [1, 2]),
        (0.25, 50.75, [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10]), (0.25, 0.75, []),
    ],
    "BetweenLowerExclusive": [(11.0, 16.25, [1, 2, 3]), (12.25, 16.25, [2, 3]), (13.0, 16.25, [2, 3])],
    "BetweenUpperExclusive": [(12.25, 17.0, [1, 2, 3]), (12.25, 16.25, [1, 2]), (12.25, 15.0, [1, 2])],
    "BetweenExclusive": [(12.25, 16.25, [2]), (11.0, 16.25, [1, 2]), (12.25, 17.0, [2, 3]), (11.0, 17.0, [1, 2, 3]),
                         (13.0, 16.25, [2]), (12.25, 15.0, [2]), (13.0, 15.0, [2])],
}
BETWEEN_CONDITIONS = {"BetweenInclusive": capi.PRED_BETWEEN_INCLUSIVE, "BetweenLowerExclusive": capi.PRED_BETWEEN_LOWER_EXCLUSIVE,
                      "BetweenUpperExclusive": capi.PRED_BETWEEN_UPPER_EXCLUSIVE, "BetweenExclusive": capi.PRED_BETWEEN_EXCLUSIVE}


def between_fixture(data_type: int, encoding: str, sort_mode: str | None, nullable: bool) -> Table:
    """SetUp (:43-96): column a = static_cast<Type>(10.25 + 2 i) (30.25 - 2 i when descending), column b = row index; with a
    sort mode three NULL rows are prepended, without one every third value is NULL; chunk size 6, the two full chunks
    encoded, the open one left unencoded."""
    numpy_type = {capi.TYPE_INT32: np.int32, capi.TYPE_INT64: np.int64, capi.TYPE_FLOAT32: np.float32,
                  capi.TYPE_FLOAT64: np.float64}[data_type]
    number_of_nulls = 3 if (nullable and sort_mode) else 0
    values, nulls, index = [], [], []
    for i in range(number_of_nulls):
        values.append(0)
        nulls.append(True)
        index.append(i)
    for i in range(11):
        double_value = 30.25 - i * 2.0 if sort_mode == "descending" else 10.25 + i * 2.0
        is_null = nullable and not sort_mode and i % 3 == 2
        values.append(0 if is_null else (int(double_value) if data_type in (capi.TYPE_INT32, capi.TYPE_INT64) else double_value))
        nulls.append(is_null)
        index.append(i + number_of_nulls)
    definitions = [ColumnDefinition("a", data_type, nullable), ColumnDefinition("b", capi.TYPE_INT32, nullable)]
    null_arrays = [np.array(nulls, dtype=bool), np.zeros(len(values), dtype=bool)] if nullable else None
    table = Table.from_columns(definitions, [np.array(values, dtype=numpy_type), np.array(index, dtype=np.int32)], null_arrays,
                               chunk_size=6)
    full_chunks = [chunk for chunk in range(table.chunk_count) if table.get_chunk(chunk).size == 6][:2]
    table.encode([encoding, "Unencoded"], full_chunks)
    return table


def between_expected(expected_with_null: list[int], sort_mode: str | None, nullable: bool) -> list[int]:
    """The index transformation of _test_between_scan (:155-186)."""
    number_of_nulls = 3 if (nullable and sort_mode) else 0
    expected = list(expected_with_null)
    if sort_mode == "descending":
        expected = sorted((10 + number_of_nulls) - e for e in expected)
    if sort_mode == "ascending":
        expected = [e + number_of_nulls for e in expected]
    if nullable and not sort_mode:
        expected = [e for e in expected if e % 3 != 2]
    return expected


def between_bounds(data_type: int, left: float, right: float):
    """static_cast<ColumnDataType>(double) of both bounds (:133-134)."""
    if data_type in (capi.TYPE_INT32, capi.TYPE_INT64):
        return int(left), int(right)
    return left, right
