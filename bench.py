#!/usr/bin/env python
"""bench.py — the hot path of BASELINE.json on synthetic TPC-H-shaped tables.

One *step* = one pass of the three operators over the resident lineitem / orders tables of TPC-H scale factor --sf
(default 100 = the configuration BASELINE.json's metric is quoted on; with N ranks every rank owns 1/N of it — strong
scaling):
  1. TableScan   l_shipdate < '1995-01-01' on lineitem (DictionarySegment<string>, u16 value-IDs)  -> RowIDPosList
  2. JoinHash    orders (ValueSegment<int32>) x lineitem (FrameOfReference u16) on orderkey, Inner -> two PosLists
  3. AggregateHash  TPC-H Q1: l_shipdate <= '1998-09-02' fused, GROUP BY l_returnflag, l_linestatus, 4 SUM 3 AVG COUNT(*)
`value` = rows processed per second = (rows scanned + probe rows joined + rows aggregated) / step time, all ranks.

    python bench.py --gpus N --steps K --warmup W            our arm (one process per GPU under torchrun for N > 1)
    python bench.py --impl reference ...                     the CPU arm: the oracle restatement of the reference's
                                                             operators on the host cores, on a bounded sample
    python bench.py ... --dump-outputs DIR                   also write the last timed step's results to DIR/*.npy, so
                                                             that two builds can be compared output for output

Prints ONE JSON line (see DESIGN.md "Measurement" for every field).
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

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

from hyrise_b200 import capi  # noqa: E402
from hyrise_b200.device import Aggregate, DeviceContext, Expression, Predicate, ROW_ID_DTYPE  # noqa: E402
from hyrise_b200.tpch import (L_DISCOUNT, L_EXTENDEDPRICE, L_LINESTATUS, L_ORDERKEY, L_QUANTITY, L_RETURNFLAG,  # noqa: E402
                              L_SHIPDATE, L_TAX, O_ORDERKEY, TpchTables)

SCAN_PREDICATE = Predicate(L_SHIPDATE, capi.PRED_LESS_THAN, "1995-01-01")
Q1_PREDICATES = [Predicate(L_SHIPDATE, capi.PRED_LESS_THAN_EQUALS, "1998-09-02")]
_ONE = ("lit", capi.TYPE_INT32, 1)
Q1_AGGREGATES = [
    Aggregate(capi.AGG_SUM, Expression.column(L_QUANTITY)),
    Aggregate(capi.AGG_SUM, Expression.column(L_EXTENDEDPRICE)),
    Aggregate(capi.AGG_SUM, Expression([("col", L_EXTENDEDPRICE), _ONE, ("col", L_DISCOUNT), "-", "*"])),
    Aggregate(capi.AGG_SUM, Expression([("col", L_EXTENDEDPRICE), _ONE, ("col", L_DISCOUNT), "-", "*", _ONE,
                                        ("col", L_TAX), "+", "*"])),
    Aggregate(capi.AGG_AVG, Expression.column(L_QUANTITY)),
    Aggregate(capi.AGG_AVG, Expression.column(L_EXTENDEDPRICE)),
    Aggregate(capi.AGG_AVG, Expression.column(L_DISCOUNT)),
    Aggregate(capi.AGG_COUNT_STAR),
]
Q1_GROUPBY = [L_RETURNFLAG, L_LINESTATUS]


def measured_peak_gbs() -> tuple[float, str]:
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as handle:
            return float(json.load(handle)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clocks and throttle reasons with nvidia-smi while the timed region runs."""

    QUERY = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.device_index = device_index
        self.samples: list[list[str]] = []
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._run, daemon=True)

    def _run(self) -> None:
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.device_index}", f"--query-gpu={self.QUERY}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                fields = [field.strip() for field in out.strip().split(",")]
                if len(fields) >= 6:
                    self.samples.append(fields)
            except Exception:  # noqa: BLE001 - best effort
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join(timeout=5)

    def summary(self) -> dict:
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        clocks = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        maxima = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [name for index, name in enumerate(names) if any(s[2 + index].lower() == "active" for s in self.samples)]
        return {"sm_mhz": clocks[len(clocks) // 2] if clocks else None, "sm_max_mhz": max(maxima) if maxima else None,
                "reasons": reasons, "samples": len(self.samples)}


class SlicedTable:
    """The first `chunks` chunks of a generated table (shares the segment buffers): the bounded CPU sample."""

    def __init__(self, table, chunks: int):
        self._table = table
        self.chunk_count = min(chunks, table.chunk_count)
        self.column_count = table.column_count
        self.column_definitions = table.column_definitions
        self._view = capi.TableView(self.chunk_count, table.column_count, table._view.segments)
        self.row_count = sum(table.segment_desc(chunk, 0).row_count for chunk in range(self.chunk_count))

    def view(self):
        from hyrise_b200.tpch import _ViewHolder
        return _ViewHolder(self._view)

    def string_value_id_bounds(self, predicate):
        return self._table.string_value_id_bounds(predicate)[: self.chunk_count]


def cpu_arm(tables: TpchTables, sample_lineitem_chunks: int, steps: int, warmup: int) -> dict:
    """The reference's operators on the host cores: the oracle restatement (oracle/liboracle.so), chunk-parallel where the
    reference spawns JobTasks, sequential where the reference is (AggregateHash's aggregation phase)."""
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import oracle_lib as orc

    cores = os.cpu_count() or 1
    lineitem = SlicedTable(tables.lineitem, sample_lineitem_chunks)
    # the orders that own those lineitem rows (1..7 lines per order, mean 4) plus slack
    orders_chunks = max(1, min(tables.orders.chunk_count, int(np.ceil(lineitem.row_count / 3.9 / capi.DEFAULT_CHUNK_SIZE)) + 1))
    orders = SlicedTable(tables.orders, orders_chunks)
    times = []
    detail = {}
    for step in range(warmup + steps):
        begin = time.perf_counter()
        t0 = time.perf_counter()
        scan = orc.table_scan(lineitem, SCAN_PREDICATE, threads=cores)
        t1 = time.perf_counter()
        join = orc.join_hash(orders, O_ORDERKEY, lineitem, L_ORDERKEY, capi.JOIN_INNER, -1, threads=cores)
        t2 = time.perf_counter()
        aggregate = orc.aggregate_hash(lineitem, Q1_GROUPBY, Q1_AGGREGATES, predicates=Q1_PREDICATES, threads=cores)
        t3 = time.perf_counter()
        if step >= warmup:
            times.append(t3 - begin)
            detail = {"scan_ms": (t1 - t0) * 1e3, "join_ms": (t2 - t1) * 1e3, "aggregate_ms": (t3 - t2) * 1e3,
                      "scan_matches": int(len(scan.row_ids)), "join_pairs": int(join.pair_count),
                      "groups": int(aggregate.group_count)}
    rows_per_step = 3 * lineitem.row_count
    seconds = float(np.mean(times))
    return {"value": rows_per_step / seconds, "ms_per_step": seconds * 1e3, "cores": cores, "rows_per_step": rows_per_step,
            "sample": f"first {lineitem.chunk_count} lineitem chunks ({lineitem.row_count} rows) + first {orders.chunk_count} "
                      f"orders chunks of the same generated tables", "detail": detail}


def ncu_traffic(kernels, sf, world):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant operator's kernels, from the committed
    `ncu --set full` capture of this workload (profiles/traffic.json, written by tools/make_profiles.py). None when the
    capture was taken on another workload."""
    path = os.path.join(REPO, "profiles", "traffic.json")
    if not os.path.exists(path) or world != 1:
        return None
    capture = json.load(open(path))
    if abs(capture.get("sf", -1) - sf) > 1e-9:
        return None
    total = 0.0
    for kernel in kernels:
        matches = [value for name, value in capture["kernels"].items() if name.split("<")[0] == kernel]
        if not matches:
            return None
        total += matches[0]["dram_bytes_per_launch"]
    return total


def verify_results(device, tables, lineitem, orders, outputs, distributed, rank, world) -> dict:
    """Checks the timed operators' results on THIS rank's shard (outside the timed region):
      scan    the match count against a numpy count over the host value-IDs (every row), a PosList sample bit-exact;
      join    (1 GPU) pair count = lineitem rows (PK-FK), per-partition probe order, and on a sample of pairs the build
              and probe keys decoded on the host are equal and fall into the pair's radix partition;
      Q1      the CUDA aggregate of the first chunks against the CPU oracle on the same chunks (<= 1e-6 relative)."""
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import ctypes as C

    import oracle_lib as orc
    from helpers import assert_aggregate_outputs_equal

    report = {"ok": True, "checks": []}

    def check(name, condition, detail=""):
        report["checks"].append({"name": name, "ok": bool(condition), "detail": detail})
        report["ok"] = report["ok"] and bool(condition)

    host = tables.lineitem
    # ---- scan: full count on the host (value-ID < per-chunk bound; u16 value-IDs)
    bounds = host.string_value_id_bounds(SCAN_PREDICATE)
    expected = 0
    sample_chunk = min(3, host.chunk_count - 1)
    sample_offsets = None
    for chunk in range(host.chunk_count):
        desc = host.segment_desc(chunk, L_SHIPDATE)
        dtype = {capi.VEC_FIXED_1B: np.uint8, capi.VEC_FIXED_2B: np.uint16, capi.VEC_FIXED_4B: np.uint32}[desc.vector_type]
        ids = np.ctypeslib.as_array(C.cast(desc.attribute_vector, C.POINTER(np.ctypeslib.as_ctypes_type(dtype))), shape=(desc.row_count,))
        hits = ids < bounds[chunk, 0]
        expected += int(hits.sum())
        if chunk == sample_chunk:
            sample_offsets = np.flatnonzero(hits).astype(np.uint32)
    scan = device.table_scan(lineitem, SCAN_PREDICATE)
    total, _ = scan.info()
    check("scan count", total == expected, f"{total} vs {expected}")
    offsets = scan.chunk_offsets()
    begin, end = int(offsets[sample_chunk]), int(offsets[sample_chunk + 1])
    got = np.empty(end - begin, dtype=ROW_ID_DTYPE)
    capi.check(device.lib.hyb_pos_list_copy(device.ptr, scan.handle, begin, end - begin, got.ctypes.data))
    check("scan PosList sample", len(got) == len(sample_offsets) and bool((got["chunk_id"] == sample_chunk).all())
          and np.array_equal(got["chunk_offset"], sample_offsets), f"chunk {sample_chunk}: {len(got)} RowIDs")
    scan.free()
    check("timed scan count", distributed or int(outputs[0]) == expected, f"{outputs[0]}")

    # ---- join (single GPU: the local join is the whole join)
    if not distributed:
        join = device.join_hash(orders, O_ORDERKEY, lineitem, L_ORDERKEY, capi.JOIN_INNER, -1)
        pairs, partitions, bits = join.info()
        check("join pair count", pairs == host.row_count == int(outputs[1]), f"{pairs} pairs, {host.row_count} lineitem rows")
        part_offsets = join.partition_offsets().astype(np.int64)
        rng = np.random.default_rng(7)
        sample = 200_000
        good = True
        for partition in rng.choice(partitions, size=min(partitions, 6), replace=False):
            begin, end = int(part_offsets[partition]), int(part_offsets[partition + 1])
            count = min(sample, end - begin)
            if count == 0:
                continue
            build_rows = np.empty(count, dtype=ROW_ID_DTYPE)
            probe_rows = np.empty(count, dtype=ROW_ID_DTYPE)
            capi.check(device.lib.hyb_join_result_copy(device.ptr, join.handle, begin, count, build_rows.ctypes.data,
                                                       probe_rows.ctypes.data))
            probe_position = probe_rows["chunk_id"].astype(np.int64) * capi.DEFAULT_CHUNK_SIZE + probe_rows["chunk_offset"]
            good = good and bool((np.diff(probe_position) > 0).all())                    # probe order inside the partition
            build_keys = host_keys(tables.orders, O_ORDERKEY, build_rows)
            probe_keys = host_keys(host, L_ORDERKEY, probe_rows)
            good = good and np.array_equal(build_keys, probe_keys)                        # the pair really joins
            good = good and bool(((probe_keys & (partitions - 1)) == partition).all())    # and sits in its radix partition
        check("join pairs sample (keys equal, radix partition, probe order)", good, f"radix_bits {bits}")
        join.free()

    # ---- Q1 on the first chunks against the oracle
    chunks = min(host.chunk_count, 24)
    sliced = SlicedTable(host, chunks)
    device_slice = device.upload(sliced)
    got = device.aggregate_hash(device_slice, Q1_GROUPBY, Q1_AGGREGATES, predicates=Q1_PREDICATES)
    want = orc.aggregate_hash(sliced, Q1_GROUPBY, Q1_AGGREGATES, predicates=Q1_PREDICATES, threads=os.cpu_count() or 1)
    try:
        assert_aggregate_outputs_equal(got, want)
        check("Q1 vs oracle on the first chunks", True, f"{chunks} chunks, {got.group_count} groups")
    except AssertionError as error:
        check("Q1 vs oracle on the first chunks", False, str(error)[:300])
    device_slice.drop()
    return report


def host_keys(table, column_id: int, row_ids: np.ndarray) -> np.ndarray:
    """int32 keys at the given RowIDs, decoded on the host from the generator's segments (ValueSegment / FoR)."""
    import ctypes as C

    keys = np.empty(len(row_ids), dtype=np.int64)
    for chunk in np.unique(row_ids["chunk_id"]):
        select = row_ids["chunk_id"] == chunk
        offsets = row_ids["chunk_offset"][select].astype(np.int64)
        desc = table.segment_desc(int(chunk), column_id)
        if desc.encoding == capi.ENC_UNENCODED:
            values = np.ctypeslib.as_array(C.cast(desc.values, C.POINTER(C.c_int32)), shape=(desc.row_count,))
            keys[select] = values[offsets]
        else:
            dtype = {capi.VEC_FIXED_1B: C.c_uint8, capi.VEC_FIXED_2B: C.c_uint16, capi.VEC_FIXED_4B: C.c_uint32}[desc.vector_type]
            codes = np.ctypeslib.as_array(C.cast(desc.attribute_vector, C.POINTER(dtype)), shape=(desc.row_count,))
            blocks = (desc.row_count + capi.FOR_BLOCK_SIZE - 1) // capi.FOR_BLOCK_SIZE
            minima = np.ctypeslib.as_array(C.cast(desc.values, C.POINTER(C.c_int32)), shape=(blocks,))
            keys[select] = minima[offsets // capi.FOR_BLOCK_SIZE].astype(np.int64) + codes[offsets].astype(np.int64)
    return keys


DUMP_SAMPLE_ROWS = 1 << 19   # per RowID output: the five sampled arrays below come to about 32 MB at any scale factor
DUMP_RUN_ROWS = 1 << 10


def dump_positions(total: int) -> np.ndarray:
    """Positions of a RowID output that --dump-outputs writes: all of them up to DUMP_SAMPLE_ROWS, otherwise runs of
    DUMP_RUN_ROWS consecutive rows at seeded starts, so the same output length always gives the same positions."""
    if total <= DUMP_SAMPLE_ROWS:
        return np.arange(total, dtype=np.int64)
    starts = np.random.default_rng(0).integers(0, total - DUMP_RUN_ROWS + 1, size=DUMP_SAMPLE_ROWS // DUMP_RUN_ROWS)
    return np.unique((starts[:, None] + np.arange(DUMP_RUN_ROWS)).ravel())


def copy_positions(positions: np.ndarray, copy, sides: int) -> list[np.ndarray]:
    """RowIDs at `positions`, one device-to-host copy per run of consecutive positions: copy(begin, count, *outputs)."""
    outputs = [np.empty(len(positions), dtype=ROW_ID_DTYPE) for _ in range(sides)]
    starts = np.flatnonzero(np.diff(positions, prepend=-2) != 1)
    for begin, end in zip(starts, np.r_[starts[1:], len(positions)]):
        copy(int(positions[begin]), int(end - begin), *(output[begin:end].ctypes.data for output in outputs))
    return outputs


def row_id_columns(row_ids: np.ndarray) -> np.ndarray:
    return np.stack([row_ids["chunk_id"], row_ids["chunk_offset"]], axis=1).astype(np.float64)


def dump_outputs(directory: str, prefix: str, device, scan, join, aggregate) -> None:
    """What the last timed step returned to its caller, as float64 .npy files: the scan's PosList and the join's RowID
    pairs at the positions of dump_positions (written next to them) with their chunk / radix partition offsets, and the
    whole Q1 result (group RowIDs, one column per aggregate, NULL flags)."""
    os.makedirs(directory, exist_ok=True)
    arrays = {}
    total, _ = scan.info()
    positions = dump_positions(total)
    (rows,) = copy_positions(positions, lambda begin, count, out: capi.check(
        device.lib.hyb_pos_list_copy(device.ptr, scan.handle, begin, count, out)), 1)
    arrays.update(scan_positions=positions, scan_row_ids=row_id_columns(rows), scan_chunk_offsets=scan.chunk_offsets())
    pairs, _, _ = join.info()
    positions = dump_positions(pairs)
    build_rows, probe_rows = copy_positions(positions, lambda begin, count, build, probe: capi.check(
        device.lib.hyb_join_result_copy(device.ptr, join.handle, begin, count, build, probe)), 2)
    arrays.update(join_positions=positions, join_build_row_ids=row_id_columns(build_rows),
                  join_probe_row_ids=row_id_columns(probe_rows), join_partition_offsets=join.partition_offsets())
    arrays.update(aggregate_row_ids=row_id_columns(aggregate.row_ids),
                  aggregate_values=np.stack([values.astype(np.float64) for values in aggregate.values], axis=1),
                  aggregate_nulls=np.stack(aggregate.nulls, axis=1))
    for name, array in arrays.items():
        np.save(os.path.join(directory, f"{prefix}{name}.npy"), np.asarray(array, dtype=np.float64))


def main() -> None:
    parser = argparse.ArgumentParser()
    parser.add_argument("--gpus", type=int, default=1)
    parser.add_argument("--steps", type=int, default=10)
    parser.add_argument("--warmup", type=int, default=3)
    parser.add_argument("--impl", default="ours", choices=["ours", "reference"])
    parser.add_argument("--sf", type=float, default=100.0, help="TPC-H scale factor of the WHOLE job (split over the ranks)")
    parser.add_argument("--cpu-sample-chunks", type=int, default=184,
                        help="lineitem chunks of the CPU arm's bounded sample (92 chunks = SF 1; default SF 2)")
    parser.add_argument("--no-cpu-baseline", action="store_true")
    parser.add_argument("--no-e2e", action="store_true")
    parser.add_argument("--no-verify", action="store_true", help="skip the result self-check (outside the timed region)")
    parser.add_argument("--l2-flush", choices=["auto", "always", "never"], default="auto",
                        help="256 MB memset before every operator: auto = only when an operator input fits the L2")
    parser.add_argument("--dump-outputs", metavar="DIR",
                        help="write the results of the last timed step as DIR/<name>.npy (float64; RowID outputs sampled)")
    args = parser.parse_args()
    if args.steps < 1:
        parser.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 0)
    metric = "TPC-H rows/sec scan+join+agg (TableScan l_shipdate + JoinHash orders x lineitem + Q1 AggregateHash)"
    workload = (f"tpch-sf{args.sf:g} TableScan l_shipdate<'1995-01-01' (config 2 query) + JoinHash orders x lineitem "
                f"(config 3 query) + Q1 AggregateHash (config 4)")
    # identical in both arms (the driver compares them); everything arm-specific lives under "detail" / "cpu_baseline"
    config = {"workload": workload, "scale_factor": args.sf, "chunk_size": capi.DEFAULT_CHUNK_SIZE,
              "tables": "seeded TPC-H-shaped lineitem / orders (dbgen distributions, Hyrise default encodings)"}

    if args.impl == "reference":
        if rank != 0:
            return
        # only the sample is generated: the same generator, seed and encodings, the first chunks of the same tables
        sample_sf = min(args.sf, args.cpu_sample_chunks / 92.0 * 1.15 + 0.1)
        tables = TpchTables(sample_sf, seed=42)
        result = cpu_arm(tables, args.cpu_sample_chunks, max(args.steps, 1), warmup)
        line = {
            "impl": "reference", "metric": metric, "value": result["value"], "unit": "rows/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": warmup, "ms_per_step": result["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int32 keys / u16 value-IDs / f32 arithmetic, f64 sums",
            "data": "synthetic", "config": config,
            "cpu_baseline": {"value": result["value"], "unit": "rows/s", "cores": result["cores"], "kind": "port",
                             "sample": result["sample"]},
            "e2e": {"value": result["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "detail": result["detail"],
        }
        print(json.dumps(line))
        return

    import torch  # device selection / distributed plumbing only

    distributed = world > 1
    if distributed:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if distributed:
            dist.barrier()

    # ---- data: every rank owns the shard [rank * orders, (rank + 1) * orders) of ONE global SF --sf data set (strong
    #      scaling: the job is fixed, the per-GPU share shrinks; key ranges are disjoint, values depend on the global
    #      order index)
    sf_local = args.sf / world
    orders_per_rank = int(round(1_500_000 * sf_local))
    tables = TpchTables(sf_local, seed=42, pinned=not args.no_e2e, first_order=rank * orders_per_rank)
    device = DeviceContext(local_rank)
    lineitem = device.upload(tables.lineitem)
    orders = device.upload(tables.orders)
    device.synchronize()
    rows = tables.lineitem.row_count
    rows_per_step = 3 * rows

    # L2 policy (timing rule: flush L2 between timed iterations OR use inputs larger than L2). --l2-flush auto: when the smallest
    # operator input of this rank — the scanned l_shipdate vector, 2 bytes per row — is larger than the L2, no operator can find
    # any of its input there (and >= 20x the L2 of other traffic passes between two runs of the same operator), so nothing is
    # flushed; otherwise (SF 10 on one GPU: 120 MB < 126 MB) a 256 MB memset precedes every operator inside the timed region.
    l2_bytes = int(torch.cuda.get_device_properties(local_rank).L2_cache_size)
    smallest_input = 2 * rows
    flush_enabled = args.l2_flush == "always" or (args.l2_flush == "auto" and smallest_input <= l2_bytes)
    if distributed:   # one policy for the whole job
        flag = torch.tensor([1 if flush_enabled else 0], device=f"cuda:{local_rank}")
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        flush_enabled = bool(flag.item())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local_rank}")
    stream_ptr = capi.C.c_void_p()
    capi.check(device.lib.hyb_context_stream(device.ptr, capi.C.byref(stream_ptr)))
    hyb_stream = torch.cuda.ExternalStream(stream_ptr.value, device=f"cuda:{local_rank}")

    def flush_l2():
        if flush_enabled:
            with torch.cuda.stream(hyb_stream):
                flush.fill_(1)

    operators = {"scan": [], "join": [], "aggregate": []}
    launches = [0]
    group = None
    phases = {"join": [], "aggregate": []}
    torch_device = torch.device("cuda", local_rank)
    if distributed:
        from hyrise_b200 import distributed as hd
        lineitem_chunk_base = hd.chunk_bases(tables.lineitem.chunk_count, torch_device)[rank]
        orders_chunk_base = hd.chunk_bases(tables.orders.chunk_count, torch_device)[rank]
        rows_per_rank = [None] * world
        dist.all_gather_object(rows_per_rank, rows)
        position_base = sum(rows_per_rank[:rank])
        radix_bits = 8 if args.sf >= 4 else 4
        # every rank receives about 1 / world of all tuples, i.e. about its own share; 25 % head room for skew
        group = hd.connect_peer_group(device, int(1.25 * max(rows_per_rank)) + 65_536)

    def phase_record(stats):
        return {"split_count_ms": stats.split_count_ms, "count_wait_ms": stats.count_wait_ms, "push_ms": stats.push_ms,
                "done_wait_ms": stats.done_wait_ms, "local_ms": stats.local_ms, "finish_ms": stats.finish_ms,
                "tuples_sent": int(stats.tuples_sent), "tuples_received": int(stats.tuples_received),
                "nvlink_bytes": int(stats.nvlink_bytes), "colocated": int(stats.colocated)}

    def distributed_join(table_o=None, table_l=None, record=True):
        """hyb_join_hash_distributed, one C-ABI call per rank: the ranks exchange the key bounds of their shards; co-located
        shards (this data set: a rank's lineitem rows belong to its own orders) are joined locally with global RowIDs, otherwise
        counts are published by kernel, both sides are split and pushed over NVLink, and every rank joins what it received.
        The forced-exchange time of the same call is reported next to the step in phases_rank0."""
        result = group.join_hash(table_o or orders, O_ORDERKEY, table_l or lineitem, L_ORDERKEY, orders_chunk_base,
                                 lineitem_chunk_base, radix_bits)
        return result, (device.last_stats() if record else None)

    def distributed_q1(table_l=None):
        """hyb_aggregate_hash_distributed: local pre-aggregation, partial groups stored into every peer's arena, merged by all"""
        return group.aggregate_hash(table_l or lineitem, Q1_GROUPBY, Q1_AGGREGATES, Q1_PREDICATES, lineitem_chunk_base, position_base)

    kept = []

    def run_step(record: bool, keep: bool = False):
        """One step. record=False (warm-up and the TIMED loop): nothing but the operator calls and the reads of their result
        sizes; record=True (a second, untimed loop of the same steps): per-operator CUDA-event statistics are fetched after
        every call, which synchronises the host with the device and therefore stays out of the timed region. keep=True
        leaves the step's results alive in `kept` for --dump-outputs instead of freeing them."""
        flush_l2()
        scan = device.table_scan(lineitem, SCAN_PREDICATE)
        scan_stats = device.last_stats() if record else None
        flush_l2()
        if distributed:
            join, join_stats = distributed_join(record=record)
            if record:
                phases["join"].append(phase_record(group.stats()))
        else:
            join = device.join_hash(orders, O_ORDERKEY, lineitem, L_ORDERKEY, capi.JOIN_INNER, -1)
            join_stats = device.last_stats() if record else None
        flush_l2()
        if distributed:
            aggregate = distributed_q1()
            if record:
                aggregate_stats = device.last_stats()
                phases["aggregate"].append(phase_record(group.stats()))
        else:
            aggregate = device.aggregate_hash(lineitem, Q1_GROUPBY, Q1_AGGREGATES, predicates=Q1_PREDICATES)
            aggregate_stats = device.last_stats() if record else None
        if record:
            for name, stats in (("scan", scan_stats), ("join", join_stats), ("aggregate", aggregate_stats)):
                operators[name].append((stats.dominant_kernel_ms, stats.device_ms, stats.algorithmic_bytes, stats.output_rows))
                launches[0] += stats.kernel_launches
        result = (scan.info()[0], join.info()[0], aggregate.group_count)
        if keep:
            kept[:] = [scan, join, aggregate]
        else:
            scan.free()
            join.free()
        return result

    for _ in range(warmup):
        run_step(False)
    device.synchronize()
    torch.cuda.synchronize()
    barrier()
    with ClockSampler(local_rank) as clocks:
        begin = time.perf_counter()
        for step in range(args.steps):
            outputs = run_step(False, keep=args.dump_outputs is not None and step == args.steps - 1)
        device.synchronize()
        torch.cuda.synchronize()
        elapsed = time.perf_counter() - begin
    if kept:
        dump_outputs(args.dump_outputs, "" if world == 1 else f"rank{rank}_", device, *kept)
        kept[0].free()
        kept[1].free()
    barrier()
    for _ in range(args.steps):  # the same steps again, instrumented (untimed): per-operator kernel / device times, phases
        run_step(True)
    device.synchronize()
    barrier()
    if distributed:
        tensor = torch.tensor([elapsed], device=f"cuda:{local_rank}", dtype=torch.float64)
        dist.all_reduce(tensor, op=dist.ReduceOp.MAX)
        elapsed = float(tensor.item())
    ms_per_step = elapsed / args.steps * 1e3
    value = rows_per_step * world / (elapsed / args.steps)

    # ---- end to end: host buffers in, host buffers out, every step ---------------------------------------------------
    e2e = None
    if not args.no_e2e:
        join_capacity = rows if not distributed else int(1.25 * max(rows_per_rank)) + 65_536
        scan_out = device.pinned_empty(rows, ROW_ID_DTYPE)
        join_build_out = device.pinned_empty(join_capacity, ROW_ID_DTYPE)
        join_probe_out = device.pinned_empty(join_capacity, ROW_ID_DTYPE)
        host_blocks = tables.host_blocks()
        h2d = sum(block.bytes for block in host_blocks)
        d2h = 0

        trace = os.environ.get("HYB_BENCH_E2E_TRACE") == "1"

        def e2e_step():
            nonlocal d2h
            marks = [("start", time.perf_counter())]

            def mark(name):
                if trace:
                    device.synchronize()
                    marks.append((name, time.perf_counter()))

            # the generator's segment buffers live in a few pinned 256 MB blocks: one DMA per block, tables point into them
            block_set = device.upload_blocks(host_blocks)
            mark("upload_blocks")
            table_l = device.upload_from_blocks(tables.lineitem, block_set)
            table_o = device.upload_from_blocks(tables.orders, block_set)
            mark("tables")
            scan = device.table_scan(table_l, SCAN_PREDICATE)
            mark("scan")
            matched = scan.to_host(scan_out)
            mark("scan d2h")
            if distributed:   # the partitioned path: exchange over NVLink, then this rank's partitions of the result
                join, _ = distributed_join(table_o, table_l)
            else:
                join = device.join_hash(table_o, O_ORDERKEY, table_l, L_ORDERKEY, capi.JOIN_INNER, -1)
            mark("join")
            pairs = join.to_host(join_build_out, join_probe_out)
            mark("join d2h")
            if distributed:
                aggregate = distributed_q1(table_l)
            else:
                aggregate = device.aggregate_hash(table_l, Q1_GROUPBY, Q1_AGGREGATES, predicates=Q1_PREDICATES)
            mark("aggregate")
            d2h = len(matched) * 8 + len(pairs[1]) * 16 + aggregate.group_count * (8 + 8 * len(Q1_AGGREGATES))
            scan.free()
            join.free()
            table_l.drop()
            table_o.drop()
            device.free_blocks(block_set)
            mark("free")
            if trace:
                print("[e2e] " + " ".join(f"{name} {1e3 * (t - marks[i][1]):.1f}" for i, (name, t) in enumerate(marks[1:])),
                      file=sys.stderr, flush=True)

        e2e_steps = max(2, min(args.steps, 5))
        for _ in range(max(3, warmup)):  # the first steps size the library's block cache (cudaMalloc on every miss)
            e2e_step()
        device.synchronize()
        barrier()
        begin = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        device.synchronize()
        e2e_elapsed = time.perf_counter() - begin
        barrier()
        if distributed:
            tensor = torch.tensor([e2e_elapsed], device=f"cuda:{local_rank}", dtype=torch.float64)
            dist.all_reduce(tensor, op=dist.ReduceOp.MAX)
            e2e_elapsed = float(tensor.item())
        e2e = {"value": rows_per_step * world / (e2e_elapsed / e2e_steps), "unit": "rows/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_elapsed / e2e_steps * 1e3, "steps": e2e_steps, "warmup": max(3, warmup)}

    # ---- roofline of the dominant kernel + per-operator breakdown ---------------------------------------------------
    peak, peak_source = measured_peak_gbs()
    breakdown = {}
    for name, samples in operators.items():
        kernel_ms = float(np.mean([s[0] for s in samples]))
        op_ms = float(np.mean([s[1] for s in samples]))
        algorithmic = float(samples[-1][2])
        breakdown[name] = {"kernel_ms": kernel_ms, "operator_ms": op_ms, "algorithmic_bytes": algorithmic,
                           "achieved_gbs": algorithmic / kernel_ms / 1e6, "frac": algorithmic / kernel_ms / 1e6 / peak,
                           "output_rows": int(samples[-1][3])}
    dominant = max(breakdown, key=lambda name: breakdown[name]["kernel_ms"])
    kernels_of = {"scan": ["scan_mask_kernel", "scan_bases_kernel", "scan_expand_kernel"],
                  "join": ["join_build_rank_kernel", "join_span_count_kernel", "exclusive_scan_kernel", "join_span_write_kernel"],
                  "aggregate": ["aggregate_stream_static_kernel"]}
    roofline = {"bound": "hbm", "kernel": " + ".join(kernels_of[dominant]), "achieved": breakdown[dominant]["achieved_gbs"],
                "peak": peak, "peak_source": peak_source, "unit": "GB/s", "frac": breakdown[dominant]["frac"],
                "traffic": ncu_traffic(kernels_of[dominant], args.sf, world),
                "algorithmic_bytes_per_launch": breakdown[dominant]["algorithmic_bytes"],
                "kernel_ms": breakdown[dominant]["kernel_ms"]}

    # ---- self-check, outside the timed region: the numbers above are only worth something if the results are right ------
    verification = None
    if not args.no_verify:
        verification = verify_results(device, tables, lineitem, orders, outputs, distributed, rank, world)
        if distributed:
            # the partitioned operators against the oracle over the union of all shards, at a size the oracle handles
            # (bit-exact RowIDs in reference order, Q1 within 1e-6) — the same checks tests/gpu_distributed_worker.py makes
            sys.path.insert(0, os.path.join(REPO, "tests"))
            from gpu_distributed_worker import run_distributed_checks
            try:
                summary = run_distributed_checks(device, rank, world, torch_device, sf=0.1, legacy_paths=False)
                verification["checks"].append({"name": "distributed scan/join/Q1 vs oracle (SF 0.1 per rank)", "ok": True,
                                               "detail": summary or ""})
            except AssertionError as error:
                verification["checks"].append({"name": "distributed scan/join/Q1 vs oracle (SF 0.1 per rank)", "ok": False,
                                               "detail": str(error)[:400]})
                verification["ok"] = False
            # the timed run itself: every lineitem row joins exactly once, across all ranks
            totals = [None] * world
            dist.all_gather_object(totals, (int(outputs[1]), rows))
            pairs_ok = sum(t[0] for t in totals) == sum(t[1] for t in totals)
            verification["checks"].append({"name": "timed distributed join: pairs over all ranks == lineitem rows", "ok": pairs_ok,
                                           "detail": str(totals)})
            verification["ok"] = verification["ok"] and pairs_ok
            flags = [None] * world
            dist.all_gather_object(flags, verification["ok"])
            verification["all_ranks_ok"] = all(flags)

    phase_summary = None
    if distributed:
        phase_summary = {}
        for name, samples in phases.items():
            if samples:
                phase_summary[name] = {key: float(np.mean([sample[key] for sample in samples])) for key in samples[0]}
        # the same join with the co-location shortcut switched off (outside the timed region): what the radix exchange costs
        device.set_option("join_colocated", "0")
        forced = []
        for _ in range(3):
            flush_l2()
            barrier()
            result, stats = distributed_join()
            forced.append(dict(phase_record(group.stats()), operator_ms=float(stats.device_ms)))
            result.free()
        device.set_option("join_colocated", "1")
        phase_summary["join_exchange_forced"] = {key: float(np.mean([sample[key] for sample in forced[1:]])) for key in forced[0]}
        accounted = sum(breakdown[name]["operator_ms"] for name in breakdown) + (3 * 0.07 if flush_enabled else 0.0)
        phase_summary["host_gap_ms"] = max(0.0, ms_per_step - accounted)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        result = cpu_arm(tables, args.cpu_sample_chunks, 1, 0)
        cpu_baseline = {"value": result["value"], "unit": "rows/s", "cores": result["cores"], "kind": "port",
                        "sample": result["sample"], "detail": result["detail"]}

    if rank == 0:
        line = {
            "metric": metric, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int32 keys / u16 value-IDs / f32 arithmetic, f64 sums", "data": "synthetic",
            "config": config,
            "detail": {"lineitem_rows_per_gpu": rows, "orders_rows_per_gpu": tables.orders.row_count,
                       "l2": ("256 MB memset before every operator, inside the timed region" if flush_enabled else
                              f"inputs larger than L2: the smallest operator input per rank is {smallest_input / 1e6:.0f} MB (scanned "
                              f"column) against {l2_bytes / 1e6:.0f} MB of L2, no flush kernel (--l2-flush auto)"),
                       "parallelism": (f"{world} ranks, each owning 1/{world} of the SF {args.sf:g} tables (orders [r n, (r + 1) n) and their "
                                       f"lineitem rows): chunk-partitioned scan (no collective); join (hyb_join_hash_distributed) = the "
                                       f"ranks exchange the key bounds of their shards through the peer control blocks; these shards "
                                       f"are co-located (no rank's lineitem keys reach another rank's orders keys), so every rank "
                                       f"joins its own shards and emits global RowIDs — the radix exchange the call falls back to "
                                       f"otherwise (counts published by kernel, fused split + NVLink P2P stores, flags polled on the "
                                       f"device, local join of the received tuples) is timed next to the step in "
                                       f"phases_rank0.join_exchange_forced; aggregate (hyb_aggregate_hash_distributed) = local "
                                       f"pre-aggregation, partial groups stored into every peer's arena and merged by all ranks; "
                                       f"no NCCL collective inside the step")
                       if world > 1 else "1 GPU",
                       "outputs_per_step": {"scan_matches": int(outputs[0]), "join_pairs": int(outputs[1]), "groups": int(outputs[2])}},
            "roofline": roofline, "operators": breakdown, "phases_rank0": phase_summary, "cpu_baseline": cpu_baseline, "e2e": e2e,
            "gpu_launches": launches[0], "clocks": clocks.summary(), "verify": verification,
        }
        print(json.dumps(line))
    ok = verification is None or (verification["ok"] and verification.get("all_ranks_ok", True))
    if group is not None:
        barrier()
        group.destroy()
    device.close()
    if distributed:
        dist.destroy_process_group()
    if not ok:
        print(f"[bench] rank {rank}: result verification FAILED: {verification}", file=sys.stderr)
        sys.exit(3)


if __name__ == "__main__":
    main()
