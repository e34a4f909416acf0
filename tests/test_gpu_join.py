"""JoinHash parity: the CUDA path (through the C-ABI) against the oracle — PosList pairs bit-exact, in reference order."""
import numpy as np
import pytest

import oracle_lib as orc
from helpers import ENCODINGS, random_table, row_ids_equal, rows_with_keys, tbl, tpch
from hyrise_b200 import capi
from hyrise_b200.device import Predicate
from hyrise_b200.storage import ColumnDefinition, Table

pytestmark = pytest.mark.gpu



# Every case runs with the library's own choice (rank table + span kernels where they apply), with the open-addressing
# table forced, with the direct-address table forced (span kernels, then the 4096-row tile kernels) and with MATCH.ANY
# ranking instead of ballots (hyb_context_set_option): all must reproduce the reference order. The oracle result is
# computed once per case.
TABLE_KINDS = {"auto": ("auto", "1", "ballot"), "hash": ("hash", "1", "ballot"), "direct": ("direct", "1", "ballot"),
               "direct-tiles": ("direct", "0", "ballot"), "rank-match": ("rank", "1", "match")}


def select_table_kind(device, kind):
    table, span, rank = TABLE_KINDS[kind]
    device.set_option("join_table", table)
    device.set_option("join_span", span)
    device.set_option("join_rank", rank)


@pytest.fixture(autouse=True)
def restore_table_kind(device):
    yield
    select_table_kind(device, "auto")


MODES = [capi.JOIN_INNER, capi.JOIN_LEFT, capi.JOIN_SEMI, capi.JOIN_ANTI_NULL_AS_TRUE, capi.JOIN_ANTI_NULL_AS_FALSE]


def check_join(device, build, build_dev, build_column, probe, probe_dev, probe_column, mode, radix_bits,
               build_filter=None, probe_filter=None):
    """build_filter / probe_filter: (DevicePosList, HostPosList) pairs."""
    expected = orc.join_hash(build, build_column, probe, probe_column, mode, radix_bits,
                             build_filter=build_filter[1] if build_filter else None,
                             probe_filter=probe_filter[1] if probe_filter else None)
    for kind in TABLE_KINDS:
        select_table_kind(device, kind)
        result = device.join_hash(build_dev, build_column, probe_dev, probe_column, mode, radix_bits,
                                  build_filter=build_filter[0] if build_filter else None,
                                  probe_filter=probe_filter[0] if probe_filter else None)
        try:
            pairs, partitions, bits = result.info()
            context = (kind, mode, radix_bits, build_column, probe_column)
            assert pairs == expected.pair_count, context
            assert bits == expected.radix_bits, context
            assert np.array_equal(result.partition_offsets(), expected.partition_offsets), context
            got_build, got_probe = result.to_host()
            assert row_ids_equal(got_probe, expected.probe), context
            if expected.build is not None:
                assert row_ids_equal(got_build, expected.build), context
        finally:
            result.free()
    select_table_kind(device, "auto")
    return expected


@pytest.mark.parametrize("encoding", ENCODINGS)
@pytest.mark.parametrize("chunk_size", [10, 3])
def test_join_test_runner_inputs(device, encoding, chunk_size):
    # join_test_runner.cpp:184-543: modes x radix bits x table sizes x key columns (int / int_null / long / long_null)
    tables = {}
    for side in ("left", "right"):
        for size in (0, 10, 15):
            table = tbl(f"join_test_runner/input_table_{side}_{size}.tbl", chunk_size).encode(encoding)
            tables[(side, size)] = (table, device.upload(table) if table.chunk_count else None)
    pairs = [(0, 0), (1, 1), (0, 1), (6, 6), (7, 7), (0, 6), (7, 1)]
    for mode in MODES:
        for radix_bits in (0, 1, 2, 5):
            for left_size, right_size in [(10, 15), (15, 10), (15, 15)]:
                left, left_dev = tables[("left", left_size)]
                right, right_dev = tables[("right", right_size)]
                for left_column, right_column in pairs:
                    if mode == capi.JOIN_INNER and left.row_count <= right.row_count:
                        check_join(device, left, left_dev, left_column, right, right_dev, right_column, mode, radix_bits)
                    else:
                        check_join(device, right, right_dev, right_column, left, left_dev, left_column, mode, radix_bits)
    for table, device_table in tables.values():
        if device_table:
            device_table.drop()


@pytest.mark.parametrize("mode", MODES)
def test_empty_sides(device, mode):
    # an empty build side (no chunks at all is not uploadable: use a one-row table filtered to nothing)
    left = tbl("join_test_runner/input_table_left_10.tbl", 4)
    right = tbl("join_test_runner/input_table_right_15.tbl", 4)
    left_dev, right_dev = device.upload(left), device.upload(right)
    nothing = Predicate(0, capi.PRED_GREATER_THAN, 10 ** 9)
    left_none = (device.table_scan(left_dev, nothing), orc.table_scan(left, nothing))
    right_none = (device.table_scan(right_dev, nothing), orc.table_scan(right, nothing))
    for radix_bits in (0, 2):
        check_join(device, right, right_dev, 1, left, left_dev, 1, mode, radix_bits, build_filter=right_none)
        check_join(device, right, right_dev, 1, left, left_dev, 1, mode, radix_bits, probe_filter=left_none)
        check_join(device, right, right_dev, 1, left, left_dev, 1, mode, radix_bits, build_filter=right_none,
                   probe_filter=left_none)
    left_dev.drop()
    right_dev.drop()


@pytest.mark.parametrize("encoding", ENCODINGS)
@pytest.mark.parametrize("mode", MODES)
def test_random_duplicates_and_nulls(device, encoding, mode):
    # many-to-many keys (duplicate build keys -> position lists in build-row order), NULLs on both sides, negative keys
    rng = np.random.default_rng(2024 + mode)
    build = random_table(rng, 6_000, 1_000).encode(encoding)
    probe = random_table(rng, 20_000, 2_047).encode(encoding)
    build_dev, probe_dev = device.upload(build), device.upload(probe)
    for radix_bits in (0, 3, 8):
        check_join(device, build, build_dev, 4, probe, probe_dev, 4, mode, radix_bits)   # non-nullable, ~20 dups/key
        check_join(device, build, build_dev, 0, probe, probe_dev, 0, mode, radix_bits)   # nullable int32, negatives
    check_join(device, build, build_dev, 1, probe, probe_dev, 1, mode, 2)                # int64 keys
    check_join(device, build, build_dev, 4, probe, probe_dev, 1, mode, 2)                # int32 build, int64 probe
    build_dev.drop()
    probe_dev.drop()


def test_filtered_inputs(device):
    # reference-table inputs: both sides pre-filtered by a TableScan (join_hash_test.cpp:52-66 uses scanned inputs)
    rng = np.random.default_rng(5)
    build = random_table(rng, 5_000, 512).encode("Dictionary")
    probe = random_table(rng, 30_000, 4_096).encode("FrameOfReference")
    build_dev, probe_dev = device.upload(build), device.upload(probe)
    build_predicate = Predicate(4, capi.PRED_LESS_THAN, 150)
    probe_predicate = Predicate(0, capi.PRED_GREATER_THAN_EQUALS, -200)
    build_filter = (device.table_scan(build_dev, build_predicate), orc.table_scan(build, build_predicate))
    probe_filter = (device.table_scan(probe_dev, probe_predicate), orc.table_scan(probe, probe_predicate))
    for mode in MODES:
        check_join(device, build, build_dev, 4, probe, probe_dev, 4, mode, 4, build_filter, probe_filter)
        check_join(device, build, build_dev, 4, probe, probe_dev, 4, mode, 0, None, probe_filter)
    build_dev.drop()
    probe_dev.drop()


def test_tpch_sf001_orders_lineitem(device):
    # join_hash_test.cpp:26-46 shape on real dbgen data (sf-0.01: 15 000 orders x 60 175 lineitems), reference encodings
    lineitem = tpch("sf-0.01_lineitem.npz")
    orders = tpch("sf-0.01_orders.npz")
    orders_table = Table.from_columns([ColumnDefinition("o_orderkey", capi.TYPE_INT32)], [orders["o_orderkey"]],
                                      chunk_size=4_000).encode("Unencoded")
    lineitem_table = Table.from_columns([ColumnDefinition("l_orderkey", capi.TYPE_INT32)], [lineitem["l_orderkey"]],
                                        chunk_size=16_000).encode("FrameOfReference")
    orders_dev, lineitem_dev = device.upload(orders_table), device.upload(lineitem_table)
    for radix_bits in (-1, 0, 7):
        expected = check_join(device, orders_table, orders_dev, 0, lineitem_table, lineitem_dev, 0, capi.JOIN_INNER,
                              radix_bits)
        assert expected.pair_count == len(lineitem["l_orderkey"])
    check_join(device, orders_table, orders_dev, 0, lineitem_table, lineitem_dev, 0, capi.JOIN_SEMI, 7)
    # the other direction: lineitem as build side -> duplicate build keys
    check_join(device, lineitem_table, lineitem_dev, 0, orders_table, orders_dev, 0, capi.JOIN_INNER, 3)
    orders_dev.drop()
    lineitem_dev.drop()


def test_generated_sf1_properties(device):
    """orders x lineitem at SF 1 (6 M probe rows, 65 535-row chunks, FoR keys): size-independent properties."""
    from hyrise_b200.tpch import TpchTables, L_ORDERKEY, O_ORDERKEY

    tables = TpchTables(1.0, seed=42)
    orders_dev, lineitem_dev = device.upload(tables.orders), device.upload(tables.lineitem)
    result = device.join_hash(orders_dev, O_ORDERKEY, lineitem_dev, L_ORDERKEY, capi.JOIN_INNER, -1)
    pairs, partitions, bits = result.info()
    assert bits == 4 and partitions == 16             # calculate_radix_bits(1.5 M) = 4
    assert pairs == tables.lineitem.row_count           # PK-FK: every lineitem finds exactly one order
    build_rows, probe_rows = result.to_host()
    probe_index = probe_rows["chunk_id"].astype(np.int64) * capi.DEFAULT_CHUNK_SIZE + probe_rows["chunk_offset"]
    build_index = build_rows["chunk_id"].astype(np.int64) * capi.DEFAULT_CHUNK_SIZE + build_rows["chunk_offset"]
    assert np.array_equal(np.sort(probe_index), np.arange(pairs))      # a permutation of the probe rows
    order_keys = ((build_index + 1) >> 3 << 5) | ((build_index + 1) & 7)  # dbgen sparse key of order index + 1
    offsets = result.partition_offsets()
    for partition in range(partitions):
        begin, end = int(offsets[partition]), int(offsets[partition + 1])
        assert (order_keys[begin:end] & (partitions - 1) == partition).all()
        assert (np.diff(probe_index[begin:end]) > 0).all()             # probe order inside the partition
    # the matched order really is the lineitem's order: lineitem rows are generated order by order
    assert (np.diff(build_index[np.argsort(probe_index)]) >= 0).all()
    result.free()
    orders_dev.drop()
    lineitem_dev.drop()
    tables.close()


@pytest.mark.parametrize("partition_count", [1, 2, 8])
def test_partition_for_exchange(device, partition_count):
    """hyb_join_partition: stable split of the non-NULL {key, RowID} tuples by key & (partition_count - 1)."""
    import ctypes as C

    import torch
    rng = np.random.default_rng(11)
    table = random_table(rng, 30_000, 4_099).encode("Automatic")
    device_table = device.upload(table)
    torch_device = torch.device("cuda", 0)
    for column, filtered in ((0, False), (1, False), (4, True)):
        scan = device.table_scan(device_table, Predicate(4, capi.PRED_LESS_THAN, 200)) if filtered else None
        host_filter = orc.table_scan(table, Predicate(4, capi.PRED_LESS_THAN, 200)) if filtered else None
        side = capi.JoinSide(device_table.handle, column, scan.handle if scan else 0)
        positions = C.c_uint64()
        capi.check(device.lib.hyb_join_side_positions(device.ptr, C.byref(side), C.byref(positions)))
        keys = torch.zeros(positions.value + 8, dtype=torch.int64, device=torch_device)
        row_ids = torch.zeros(positions.value + 8, dtype=torch.int64, device=torch_device)
        torch.cuda.synchronize()
        offsets = (C.c_uint64 * (partition_count + 1))()
        capi.check(device.lib.hyb_join_partition(device.ptr, C.byref(side), partition_count, 1000, keys.data_ptr(),
                                                 row_ids.data_ptr(), offsets))
        offsets = np.array(offsets[:], dtype=np.int64)
        # expectation from the host copy of the table: rows in order, NULL keys dropped, stable split by the low key bits
        rows = rows_with_keys(table, column, host_filter)
        want_keys = np.array([key for _, key in rows if key is not None], dtype=np.int64)
        want_rows = np.array([(chunk_id + 1000) | (offset << 32) for (chunk_id, offset), key in rows if key is not None],
                             dtype=np.int64)
        owner = want_keys & (partition_count - 1)
        order = np.argsort(owner, kind="stable")
        assert offsets[-1] == len(want_keys)
        assert np.array_equal(np.diff(offsets), np.bincount(owner, minlength=partition_count))
        assert np.array_equal(keys[:offsets[-1]].cpu().numpy(), want_keys[order])
        assert np.array_equal(row_ids[:offsets[-1]].cpu().numpy(), want_rows[order])
        if scan:
            scan.free()
    device_table.drop()


@pytest.mark.parametrize("shift_bits", [0, 2, 3])
def test_int64_keys_with_common_low_bits(device, shift_bits):
    """What one rank joins after a radix exchange: non-NULL int64 keys that agree in their low bits (direct table indexed
    by (key - min) >> shift), unique and duplicated build sides, probe keys with other low bits mixed in."""
    rng = np.random.default_rng(31 + shift_bits)
    step = 1 << shift_bits
    base = 5_000_000_000
    unique_keys = base + 3 % step + step * rng.permutation(40_000)[:12_000].astype(np.int64)
    for build_keys in (unique_keys, np.concatenate([unique_keys[:3_000], unique_keys[:1_000]])):
        probe_keys = base + rng.integers(-500, 45_000 * step, 50_000).astype(np.int64)
        build = Table.from_columns([ColumnDefinition("k", capi.TYPE_INT64)], [build_keys], chunk_size=5_000).encode("Unencoded")
        probe = Table.from_columns([ColumnDefinition("k", capi.TYPE_INT64)], [probe_keys], chunk_size=8_191).encode("Unencoded")
        build_dev, probe_dev = device.upload(build), device.upload(probe)
        for mode in (capi.JOIN_INNER, capi.JOIN_SEMI, capi.JOIN_LEFT):
            for radix_bits in (0, 4):
                check_join(device, build, build_dev, 0, probe, probe_dev, 0, mode, radix_bits)
        build_dev.drop()
        probe_dev.drop()


@pytest.mark.parametrize("partition_count", [1, 2, 8])
def test_partition_push_addressing(device, partition_count):
    """hyb_join_partition_push with all "peers" in local memory: every group must arrive, in order, at the destination the
    exchange callback names — the same bytes hyb_join_partition writes into its grouped local buffers."""
    import ctypes as C

    import torch
    rng = np.random.default_rng(12)
    table = random_table(rng, 60_000, 8_191).encode("Automatic")
    device_table = device.upload(table)
    torch_device = torch.device("cuda", 0)
    for column in (0, 1, 4):
        side = capi.JoinSide(device_table.handle, column, 0)
        positions = C.c_uint64()
        capi.check(device.lib.hyb_join_side_positions(device.ptr, C.byref(side), C.byref(positions)))
        keys = torch.zeros(positions.value + 8, dtype=torch.int64, device=torch_device)
        row_ids = torch.zeros(positions.value + 8, dtype=torch.int64, device=torch_device)
        torch.cuda.synchronize()
        offsets = (C.c_uint64 * (partition_count + 1))()
        capi.check(device.lib.hyb_join_partition(device.ptr, C.byref(side), partition_count, 77, keys.data_ptr(),
                                                 row_ids.data_ptr(), offsets))
        offsets = [int(v) for v in offsets]
        received = {}

        def exchange(_user, counts, dest_keys, dest_rows):
            for p in range(partition_count):
                assert int(counts[p]) == offsets[p + 1] - offsets[p]
                # 1000 int64 of slack in front: a store at a wrong (smaller) index would land there and be caught
                received[p] = (torch.full((int(counts[p]) + 2000,), -7, dtype=torch.int64, device=torch_device),
                               torch.full((int(counts[p]) + 2000,), -7, dtype=torch.int64, device=torch_device))
                dest_keys[p] = received[p][0].data_ptr() + 8000
                dest_rows[p] = received[p][1].data_ptr() + 8000
            torch.cuda.synchronize()
            return 0

        callback = capi.EXCHANGE_FN(exchange)
        capi.check(device.lib.hyb_join_partition_push(device.ptr, C.byref(side), partition_count, 77, callback, None))
        for p in range(partition_count):
            count = offsets[p + 1] - offsets[p]
            for got, want in ((received[p][0], keys), (received[p][1], row_ids)):
                got = got.cpu().numpy()
                assert np.all(got[:1000] == -7) and np.all(got[1000 + count:] == -7), (column, p)
                assert np.array_equal(got[1000:1000 + count], want[offsets[p]:offsets[p + 1]].cpu().numpy()), (column, p)
    device_table.drop()


@pytest.mark.parametrize("probe_encoding", ["Unencoded", "FrameOfReference"])
@pytest.mark.parametrize("key_step", [1, 3, 200])
def test_sorted_unique_build_span_path(device, probe_encoding, key_step):
    """The PK-FK shape the span kernels and the rank table are built for: a strictly increasing build key column, probe
    keys with hits and misses, FoR offsets of 1 / 2 / 4 bytes (key_step widens the blocks' value range), partial spans at
    chunk ends, every radix width, plus a build side behind an (order-preserving) scan."""
    rng = np.random.default_rng(77 + key_step)
    build_keys = (1_000 + key_step * np.arange(30_000) + (np.arange(30_000) // 8) * 24 * key_step).astype(np.int32)
    probe_keys = np.sort(rng.integers(900, int(build_keys[-1]) + 200, 70_000)).astype(np.int32)
    if key_step == 3:
        probe_keys = rng.permutation(probe_keys)  # unsorted probe side: ranks must still follow probe order
    build = Table.from_columns([ColumnDefinition("k", capi.TYPE_INT32)], [build_keys], chunk_size=7_000).encode("Unencoded")
    probe = Table.from_columns([ColumnDefinition("k", capi.TYPE_INT32)], [probe_keys], chunk_size=20_000).encode(probe_encoding)
    build_dev, probe_dev = device.upload(build), device.upload(probe)
    for radix_bits in (0, 1, 5, 8):
        expected = check_join(device, build, build_dev, 0, probe, probe_dev, 0, capi.JOIN_INNER, radix_bits)
        assert 0 < expected.pair_count < len(probe_keys)
    check_join(device, build, build_dev, 0, probe, probe_dev, 0, capi.JOIN_SEMI, 4)
    check_join(device, build, build_dev, 0, probe, probe_dev, 0, capi.JOIN_LEFT, 4)
    predicate = Predicate(0, capi.PRED_GREATER_THAN, int(build_keys[9_000]))
    build_filter = (device.table_scan(build_dev, predicate), orc.table_scan(build, predicate))
    check_join(device, build, build_dev, 0, probe, probe_dev, 0, capi.JOIN_INNER, 3, build_filter=build_filter)
    build_filter[0].free()
    build_dev.drop()
    probe_dev.drop()


def test_peer_group_single_rank(device):
    """The native multi-GPU path with a world of one: counts published through the control block, device-side flag waits,
    the fused split + push kernel storing into this rank's own arena, the local join over the received tuples and the
    translation back to (global) RowIDs — and the partial-group exchange of the aggregate. (tests/gpu_distributed_worker.py
    runs the same calls on >= 2 GPUs.)"""
    from hyrise_b200 import distributed as hd
    from hyrise_b200.tpch import L_LINESTATUS, L_ORDERKEY, L_RETURNFLAG, L_SHIPDATE, O_ORDERKEY, TpchTables
    from test_oracle_aggregate import Q1_AGGREGATES

    tables = TpchTables(0.05, seed=11)
    lineitem, orders = device.upload(tables.lineitem), device.upload(tables.orders)
    group = hd.connect_peer_group(device, 4 * tables.lineitem.row_count + 4096)   # room for the partitioned aggregate's records
    for colocated in ("0", "1"):  # a world of one is trivially co-located: force the exchange path first, then the shortcut
        device.set_option("join_colocated", colocated)
        for radix_bits in (3, 0, 3):  # repeated calls reuse the arena, the received tables and the epoch flags
            expected = orc.join_hash(tables.orders, O_ORDERKEY, tables.lineitem, L_ORDERKEY, capi.JOIN_INNER, radix_bits)
            result = group.join_hash(orders, O_ORDERKEY, lineitem, L_ORDERKEY, 0, 0, radix_bits)
            got_build, got_probe = result.to_host()
            assert result.info()[0] == expected.pair_count
            assert np.array_equal(result.partition_offsets(), expected.partition_offsets)
            assert row_ids_equal(got_probe, expected.probe) and row_ids_equal(got_build, expected.build)
            result.free()
        stats = group.stats()
        assert stats.colocated == int(colocated) and stats.tuples_sent == 0
        if colocated == "0":
            assert stats.tuples_received == tables.lineitem.row_count + tables.orders.row_count
    # global RowIDs of the co-located path: chunk bases are added to the emitted RowIDs of both sides
    expected = orc.join_hash(tables.orders, O_ORDERKEY, tables.lineitem, L_ORDERKEY, capi.JOIN_INNER, 3)
    result = group.join_hash(orders, O_ORDERKEY, lineitem, L_ORDERKEY, 1000, 70_000, 3)
    got_build, got_probe = result.to_host()
    assert np.array_equal(got_build["chunk_id"], expected.build["chunk_id"] + 1000)
    assert np.array_equal(got_probe["chunk_id"], expected.probe["chunk_id"] + 70_000)
    assert np.array_equal(got_build["chunk_offset"], expected.build["chunk_offset"])
    assert np.array_equal(got_probe["chunk_offset"], expected.probe["chunk_offset"])
    result.free()
    predicates = [Predicate(L_SHIPDATE, capi.PRED_LESS_THAN_EQUALS, "1998-09-02")]
    got = group.aggregate_hash(lineitem, [L_RETURNFLAG, L_LINESTATUS], Q1_AGGREGATES, predicates, 0, 0)
    want = orc.aggregate_hash(tables.lineitem, [L_RETURNFLAG, L_LINESTATUS], Q1_AGGREGATES, predicates=predicates)
    from helpers import assert_aggregate_outputs_equal
    assert_aggregate_outputs_equal(got, want)
    # high cardinality: the partial groups do not fit the 32 KB block -> partitioned exchange (with a world of one, through
    # this rank's own tuple regions), result identical to the local operator's
    from hyrise_b200.device import Aggregate, Expression
    wide = [Aggregate(capi.AGG_SUM, Expression.column(1)), Aggregate(capi.AGG_MIN, Expression.column(2)), Aggregate(capi.AGG_COUNT_STAR)]
    got = group.aggregate_hash(lineitem, [L_ORDERKEY, L_LINESTATUS], wide, [], 0, 0)
    assert group.stats().aggregate_partitioned == 1
    want = orc.aggregate_hash(tables.lineitem, [L_ORDERKEY, L_LINESTATUS], wide)
    assert_aggregate_outputs_equal(got, want)
    got = group.aggregate_hash(lineitem, [L_ORDERKEY], wide, [], 0, 0)   # single int32 column: immediate-key order
    want = orc.aggregate_hash(tables.lineitem, [L_ORDERKEY], wide)
    assert_aggregate_outputs_equal(got, want)
    group.destroy()
    lineitem.drop()
    orders.drop()
    tables.close()
