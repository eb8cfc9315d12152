#!/usr/bin/env python
"""bench.py — hash-join probe rows/s on the BASELINE.json workload (lineitem JOIN orders, synthetic SF100,
BIGINT key), plus the Q1 GROUP-BY input rows/s, through the C ABI of libtrino_gpu.so.

  python bench.py --gpus 1 --steps K --warmup W            # this repo's sm_100a operators
  python bench.py --impl reference --gpus N ...            # the reference's CPU algorithm (C++ restatement, all host threads)
  torchrun ... bench.py --gpus N ...                       # partitioned join: hash exchange over NCCL + local probe
  python bench.py --gpus 1 ... --dump-outputs DIR          # also write the joined page of the last timed step to DIR/*.npy

A "step" is one pass of the LookupJoinOperator over the whole probe side (N>1: PagePartitioner + all-to-all + probe).
`value` is timed with inputs resident in HBM; `e2e` feeds HOST pages through the same operator calls and copies the
result back to host memory inside the timed region.  Prints ONE JSON line on rank 0.

The inputs are generated from fixed seeds, so two builds run with the same arguments join the same rows, and their
--dump-outputs directories can be compared file by file.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True      # the benchmark leaves the tree it runs from as it found it (it may be read-only)

import numpy as np  # noqa: E402

SEED_LINEITEM, SEED_ORDERS = 0x7C01, 0x7C02
# --dump-outputs: a joined page of more rows than this is written as DUMP_RUNS runs of DUMP_RUN_ROWS consecutive rows at
# places drawn with SEED_DUMP (4 files x 8 MB of float64 at most)
DUMP_RUNS, DUMP_RUN_ROWS, SEED_DUMP = 512, 2048, 0x7C0D
ALG_BYTES_PROBE_INDEX = 24          # SURVEY.md §8d: 8 key + 12 table entry + 4 position
ALG_BYTES_PROBE_FUSED = 40          # fused probe + gather, this workload: 24 + 8 build payload read + 8 written (probe columns pass through by reference)
ALG_BYTES_Q1_CODES = 38             # shipdate 4 + 4 x FLOAT64 32 + 2 INT8 key codes
ALG_BYTES_Q1_UTF8 = 46              # the reference's key types: 2 x VARCHAR(1) = 2 x (4 offset + 1 byte) instead of the 2 code bytes (SURVEY.md §8d)
ALG_BYTES_GROUPBY_BIGINT = 36       # SURVEY.md §8d: 8 key + 8 value + 20 table entry touched
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures (profiles/r02_kernels.md),
# quoted only for the configuration they were captured on
NCU_TRAFFIC_PROBE_FUSED_SF100 = 8.429180e9 + 7.174483e9      # 600 000 003 rows: 26.0 B/row (join_probe_lean_kernel<2,1,8>, dense order-preserving table)
NCU_TRAFFIC_Q1_SF300 = 68.400325e9 + 4.218368e6               # 1.8 G rows: 38.0 B/row (tg_agg_small_jit, profiles/r02_kernels.md, capture r3k)


def bind_to_gpu_numa_node(local):
    """N > 1: run this rank's host threads (and so first-touch its pinned staging) on the NUMA node its GPU hangs off, so that the
    end-to-end path of 8 ranks does not funnel through one socket's memory controller.  Best effort: silently a no-op when the
    topology files are not there."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(local), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local), "pci_device_id", 0)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        if cpus:
            os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def cpu_probe_measure(args, n_orders, probe_rows, passes, warm):
    """The CPU probe arm, shared by --impl reference and the cpu_baseline block: PartitionedLookupSource of P partitions built in
    parallel (one builder per partition), persistent pool of T probe drivers on 8192-row pages, every buffer of the timed region
    allocated and first-touched by the drivers beforehand (oracle.h: orc_pjoin_*).  Returns the median pass and the spread."""
    import oracle_lib as o
    threads = o.hardware_threads()
    partitions = 2
    while partitions < min(threads, 256):
        partitions <<= 1
    sample = min(probe_rows, args.cpu_sample_rows)
    okeys = o.synth_orders_keys(n_orders, 0, n_orders, SEED_ORDERS, True)
    payload = (okeys % 2557).astype(np.int32)
    pj = o.PartitionedJoin(okeys, payload, partitions, threads)
    lkeys = pj.alloc(sample, np.int64)
    lkeys[:] = o.synth_lineitem_keys(n_orders, 0, sample, SEED_LINEITEM, int(args.shuffle_probe))
    pos = pj.alloc(sample, np.int64)
    pay = pj.alloc(sample, np.int32)
    for _ in range(max(1, warm)):
        pj.probe(lkeys, pos, pay)
    times = sorted(pj.probe(lkeys, pos, pay) for _ in range(passes))
    assert (pos >= 0).all()
    assert (pay[:4096] == (lkeys[:4096] % 2557)).all()
    med = float(np.median(times))
    out = {"value": sample / med, "unit": "rows/s", "cores": threads, "kind": "port", "seconds_median": med, "passes": len(times),
           "spread": {"min_s": times[0], "max_s": times[-1], "rel_iqr": float((np.percentile(times, 75) - np.percentile(times, 25)) / med)},
           "sample": f"{sample} of {probe_rows} probe rows against the full {n_orders}-row build side; PartitionedLookupSource of {pj.partitions} partitions "
                     f"(parallel build {pj.build_seconds:.1f} s, untimed), {threads} persistent probe drivers on 8192-row pages, batched 3-phase "
                     f"getAddressIndex + build payload copy; outputs pre-allocated and first-touched by the drivers; median of {len(times)} passes; "
                     f"{os.cpu_count()} logical CPUs"}
    pj.close()
    return out


def reference_arm(args):
    """The reference's CPU algorithm (oracle port, see cpu_probe_measure) on a bounded sample of the same workload.
    Test infrastructure timed as the baseline; never on the product path."""
    import oracle_lib as o
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    sf = args.sf
    n_orders = int(1_500_000 * sf)
    rows = o.synth_lineitem_rows(n_orders)
    cpu = cpu_probe_measure(args, n_orders, rows, args.steps, args.warmup)
    value = cpu["value"]
    line = {"impl": "reference", "metric": "hash_join_probe_rows_per_sec", "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": cpu["seconds_median"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
            "data": "synthetic", "config": workload_config(args, n_orders, rows, 1), "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def workload_config(args, n_orders, probe_rows, world):
    return {"workload": f"lineitem JOIN orders hash join, synthetic SF{args.sf:g}, BIGINT join key, INNER, build payload o_orderdate (days, BIGINT), "
                        f"probe payload l_extendedprice FLOAT64 (BASELINE.json configs[1])",
            "build_rows_per_gpu": n_orders, "probe_rows_per_gpu": probe_rows, "probe_order": "orderkey-clustered" if not args.shuffle_probe else "shuffled",
            "parallelism": (f"hash-partitioned x{world}, probe side exchanged every step " +
                            ("over NCCL send/recv" if os.environ.get("TGPU_EXCHANGE_NCCL") else
                             "by SM stores into peer HBM (NVLink)" if os.environ.get("TGPU_BENCH_SERIAL") else
                             "into peer HBM over NVLink by the copy engines, two half-pages per step, split-phase: SMs partition page k+1 and probe page k "
                             "while page k+1 is in flight")) if world > 1 else "single GPU",
            "l2": "inputs (9.6 GB probe side, 4.3 GB table at SF100) are far larger than the 126 MB L2; no flush needed"}


def device_col(ctx, nbytes):
    return ctx.malloc(nbytes)


def dump_page(ctx, out, names, path):
    """Write the columns of a device output page as path/<name>.npy in float64 (the BIGINT values here stay below 2^53), with
    path/row.npy = the positions in the page of the rows written: every row of a small page, else the seeded sample of
    DUMP_RUNS runs of DUMP_RUN_ROWS rows, which is the same for every page of the same row count."""
    from trino_b200 import abi
    n = out.rows
    if n <= DUMP_RUNS * DUMP_RUN_ROWS:
        runs = [(0, n)]
    else:
        starts = np.sort(np.random.default_rng(SEED_DUMP).choice(n // DUMP_RUN_ROWS, DUMP_RUNS, replace=False)) * DUMP_RUN_ROWS
        runs = [(int(s), DUMP_RUN_ROWS) for s in starts]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "row.npy"), np.concatenate([np.arange(s, s + m, dtype=np.float64) for s, m in runs]))
    dtypes = {abi.INT64: np.dtype(np.int64), abi.FLOAT64: np.dtype(np.float64)}
    for c, name in enumerate(names):
        col = out.column(c)
        assert not col.validity, f"{name}: NULLs are not written"
        dt = dtypes[col.type]
        vals = np.concatenate([ctx.to_host(col.ptr + s * dt.itemsize, dt, m) for s, m in runs])
        np.save(os.path.join(path, name + ".npy"), vals.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="join", choices=["join", "q3way", "star", "q1"],
                    help="join (default, BASELINE.json configs[1]; the line the driver reads) | q3way (configs[3]) | star (configs[4]) | q1 (configs[2] across GPUs): bench_workloads.py")
    ap.add_argument("--sf", type=float, default=None, help="TPC-H scale factor per GPU (default 100 for the join workload, 37.5 = SF300 / 8 for q3way)")
    ap.add_argument("--ds-sf", type=float, default=125.0, help="TPC-DS scale factor per GPU of the star workload (125 = SF1000 / 8)")
    ap.add_argument("--star-chunks", type=int, default=4, help="pages the fact shard is fed in per step (bounds the intermediate pages)")
    ap.add_argument("--q1-sf", type=float, default=300.0, help="scale factor of the Q1 GROUP-BY side measurement (0 = skip)")
    ap.add_argument("--shuffle-probe", action="store_true", help="variant B: uniformly shuffled probe keys")
    ap.add_argument("--cpu-sample-rows", type=int, default=200_000_000)
    ap.add_argument("--e2e-rows", type=int, default=0, help="probe rows fed from host per e2e step (0 = all)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-shuffled", action="store_true", help="skip the shuffled-probe variant (roofline_shuffled)")
    ap.add_argument("--no-groupby-bigint", action="store_true", help="skip the high-cardinality BIGINT GROUP BY block")
    ap.add_argument("--no-secondary", action="store_true", help="skip the FilterAndProject / PartitionedOutput blocks (secondary_operators)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end (host pages) measurement: kernel experiments only")
    ap.add_argument("--l2-fetch", type=int, default=0, help="cudaLimitMaxL2FetchGranularity to set (32/64/128; 0 = leave the default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the joined page of the last one as DIR/<column>.npy (float64; a fixed seeded sample of "
                         f"{DUMP_RUNS} x {DUMP_RUN_ROWS} rows of a larger page, DIR/row.npy = their positions in the page)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "b200" or args.workload != "join" or dist_env()[1] > 1):
        ap.error("--dump-outputs is implemented for the join workload of --impl b200 on one GPU")
    if args.sf is None:
        args.sf = 37.5 if args.workload == "q3way" else 100.0
    if args.impl == "reference":
        return reference_arm(args)
    if args.workload != "join":
        import bench_workloads
        return bench_workloads.main(args, ClockSampler, dist_env)

    rank, world, local = dist_env()
    from trino_b200 import abi
    from trino_b200 import operators as ops

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        bind_to_gpu_numa_node(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = ops.Context(local)
    lib = ctx.lib
    if args.l2_fetch:
        ctx.check(lib.tgpu_ctx_set_l2_fetch_granularity(ctx.h, args.l2_fetch))
    l2g = C.c_int()
    ctx.check(lib.tgpu_ctx_get_l2_fetch_granularity(ctx.h, C.byref(l2g)))

    def barrier():
        if dist is not None:
            dist.barrier()

    # ---------------- setup (untimed): synthetic columns in HBM, hash build
    sf = args.sf
    n_orders = int(1_500_000 * sf)                   # per GPU
    probe_rows = lib.tgpu_synth_lineitem_rows(n_orders)
    total_orders = n_orders * world
    total_rows = lib.tgpu_synth_lineitem_rows(total_orders)
    # every rank owns a contiguous range shard of the global tables
    from trino_b200.sharding import shard_range
    o_first, _ = shard_range(total_orders, world, rank)
    l_first, l_count = shard_range(total_rows, world, rank)
    d_okeys = ctx.malloc(n_orders * 8)
    ctx.check(lib.tgpu_synth_orders_keys(ctx.h, total_orders, o_first, n_orders, SEED_ORDERS, 1, C.c_void_p(d_okeys)))
    d_lkeys = ctx.malloc(l_count * 8)
    d_lprice = ctx.malloc(l_count * 8)
    ctx.check(lib.tgpu_synth_lineitem_keys(ctx.h, total_orders, l_first, l_count, SEED_LINEITEM, int(args.shuffle_probe), C.c_void_p(d_lkeys)))
    # payload columns: o_orderdate = key % 2557 (INT32), l_extendedprice = key * 0.5 (FLOAT64); produced by the filter/project operator
    def project(ptr, n, dtype_expr, out_type):
        page = ops.DevicePage([ops.DeviceColumn(abi.INT64, ptr, n)], n)
        prog = ops.PageProcessorProgram(None, [dtype_expr])
        op = ops.FilterAndProjectOperatorFactory(ctx, prog).create_operator()
        op.add_input(page)
        out = op.get_output_device()
        op.close()
        return out
    price_page = project(d_lkeys, l_count, ops.Call(abi.EX_MUL, ops.Call(abi.EX_CAST_BIGINT_TO_DOUBLE, ops.Col(0, abi.V_BIGINT)), ops.Const(0.5, abi.V_DOUBLE)), abi.FLOAT64)
    d_lprice_col = price_page.column(0)
    date_page = project(d_okeys, n_orders, ops.Call(abi.EX_MOD, ops.Col(0, abi.V_BIGINT), ops.Const(2557, abi.V_BIGINT)), abi.INT64)
    d_odate_col = date_page.column(0)      # INT64 payload (8 B) — keeps the build payload a plain BIGINT column

    build_page = ops.DevicePage([ops.DeviceColumn(abi.INT64, d_okeys, n_orders), d_odate_col], n_orders)
    probe_page = ops.DevicePage([ops.DeviceColumn(abi.INT64, d_lkeys, l_count), d_lprice_col], l_count)

    partitioner = None
    if world > 1:
        # co-locate build and probe by key: HashBucketFunction over orderkey, bucket == rank (SURVEY.md §8e)
        idb = (C.c_uint8 * abi.COMM_ID_BYTES)()
        if rank == 0:
            ctx.check(lib.tgpu_comm_get_unique_id(C.cast(idb, C.c_void_p)))
        import torch
        t = torch.tensor(list(idb), dtype=torch.uint8, device=f"cuda:{local}")
        dist.broadcast(t, 0)
        idb = (C.c_uint8 * abi.COMM_ID_BYTES)(*t.cpu().tolist())
        ctx.check(lib.tgpu_comm_init(ctx.h, C.cast(idb, C.c_void_p), rank, world))
        partitioner = ops.PartitionedOutputOperatorFactory(ctx, [0], world).create_operator()
        pp = abi.PP()
        ctx.check(lib.tgpu_exchange_partitioned(ctx.h, partitioner.h, build_page.ref(), C.byref(pp)))
        build_in = ops.DeviceOutputPage(ctx, pp)
        build_page_local = build_in.as_device_page()
    else:
        build_page_local = build_page

    # N > 1, pipelined form (default): split-phase exchange - the SMs partition page k+1 and probe page k while the copy
    # engines move page k+1 over NVLink.  TGPU_BENCH_SERIAL=1: exchange then probe, one page per step, no overlap.
    overlap = world > 1 and not os.environ.get("TGPU_BENCH_SERIAL") and not os.environ.get("TGPU_EXCHANGE_NCCL")
    pctx = ctx
    bridge = ops.JoinBridge()
    builder = ops.HashBuilderOperatorFactory(pctx, bridge, [0], [1], n_orders).create_operator()
    t_build0 = time.time()
    builder.add_input(build_page_local)
    builder.finish()
    pctx.synchronize()
    build_s = time.time() - t_build0
    lookup = bridge.lookup_source
    probe_op = ops.LookupJoinOperatorFactory(pctx, bridge, abi.JOIN_INNER, False, [0], [0, 1]).create_operator()
    if world > 1 and not os.environ.get("TGPU_EXCHANGE_NCCL"):
        # peer-memory exchange for the probe side: two receive arenas per rank, IPC handles all-gathered once.
        # (created only now: the build-side page above went through NCCL send/recv and is owned by the lookup source)
        import torch
        arena_bytes = int(l_count * 1.3) * 16 + (4 << 20)
        hb = (C.c_uint8 * (abi.NUM_ARENAS * abi.IPC_HANDLE_BYTES))()
        ctx.check(lib.tgpu_comm_arena_create(ctx.h, arena_bytes, C.cast(hb, C.c_void_p)))
        mine = torch.tensor(list(hb), dtype=torch.uint8, device=f"cuda:{local}")
        gathered = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(gathered, mine)
        allh = (C.c_uint8 * (world * abi.NUM_ARENAS * abi.IPC_HANDLE_BYTES))(*torch.cat(gathered).cpu().tolist())
        ctx.check(lib.tgpu_comm_arena_open(ctx.h, C.cast(allh, C.c_void_p)))

    out_rows_seen = [0]
    kernel_ms = []
    # pipelined form: the step's page is exchanged in two halves through tgpu_exchange_begin/_end; probe(half k) is only
    # enqueued, its output is taken when the next page is handed to the probe
    halves = []
    if overlap:
        h0 = (l_count // 2) // 1024 * 1024
        for first, cnt in ((0, h0), (h0, l_count - h0)):
            halves.append(ops.DevicePage([ops.DeviceColumn(abi.INT64, d_lkeys + first * 8, cnt), ops.DeviceColumn(abi.FLOAT64, d_lprice_col.ptr + first * 8, cnt)], cnt))
    inflight = []
    step_rows = [0]

    check = {"on": False, "rows": 0, "key": 0, "payload": 0, "key_mod": 0, "spot": 0}
    M64 = (1 << 64) - 1

    def column_sum(col, mod=0):
        c = abi.Column()
        c.type, c.flags, c.length, c.data, c.offsets, c.validity = col.type, 0, col.length, col.ptr, col.offsets, col.validity
        v = C.c_int64()
        ctx.check(lib.tgpu_column_sum(ctx.h, C.byref(c), mod, C.byref(v)))
        return v.value & M64

    def check_output(out):
        """closed-form checks of one joined page (untimed verification pass): see `verify` in the JSON line"""
        check["rows"] += out.rows
        check["key"] = (check["key"] + column_sum(out.column(0))) & M64
        check["payload"] = (check["payload"] + column_sum(out.column(2))) & M64
        check["key_mod"] = (check["key_mod"] + column_sum(out.column(0), 2557)) & M64
        if check["spot"] == 0 and out.rows > 0:
            import oracle_lib as o
            from trino_b200.page import Block, Page
            m = min(out.rows, 1 << 20)
            hk, hp, hb = np.empty(m, np.int64), np.empty(m, np.float64), np.empty(m, np.int64)
            for arr, c in ((hk, 0), (hp, 1), (hb, 2)):
                ctx.check(lib.tgpu_memcpy_d2h(ctx.h, C.c_void_p(arr.ctypes.data), C.c_void_p(out.column(c).ptr), m * 8))
            assert (hb == hk % 2557).all() and (hp == hk * 0.5).all(), "joined row carries the wrong payload"
            assert (o.partition_ids(Page(Block.bigint(hk)), [0], world) == rank).all(), "row received by the wrong rank (HashGenerator.java:41-46)"
            check["spot"] = m

    def drain():
        if not inflight:
            return
        out = probe_op.get_output_device()
        step_rows[0] += out.rows if out else 0
        if out:
            if check["on"]:
                check_output(out)
            out.release()
        inflight.pop().release()

    handles = []

    def step_overlapped():
        # per half page k: begin(k) [partition on the SMs, transfer on the copy engines], then end(k-1) + probe(k-1)
        for half in halves:
            h = C.c_void_p()
            ctx.check(lib.tgpu_exchange_begin(ctx.h, partitioner.h, half.ref(), C.byref(h)))
            handles.append(h)
            if len(handles) > 1:
                finish_one()

    def finish_one():
        drain()                      # output of the probe before (needsInput protocol)
        pp = abi.PP()
        ctx.check(lib.tgpu_exchange_end(ctx.h, handles.pop(0), C.byref(pp)))
        inp = ops.DeviceOutputPage(ctx, pp)
        probe_op.add_input(inp.as_device_page())
        inflight.append(inp)

    last_out = [None]

    def step(keep_output=False):
        if overlap:
            step_overlapped()
        elif partitioner is not None:
            pp = abi.PP()
            ctx.check(lib.tgpu_exchange_partitioned(ctx.h, partitioner.h, probe_page.ref(), C.byref(pp)))
            inp = ops.DeviceOutputPage(ctx, pp)
            probe_op.add_input(inp.as_device_page())
            out = probe_op.get_output_device()
            out_rows_seen[0] = out.rows if out else 0
            if out:
                if check["on"]:
                    check_output(out)
                out.release()
            inp.release()
        else:
            probe_op.add_input(probe_page)
            kernel_ms.append(ctx.last_kernel_ms())
            out = probe_op.get_output_device()
            out_rows_seen[0] = out.rows if out else 0
            if out:
                if keep_output:
                    last_out[0] = out          # --dump-outputs: written and released after the timed region
                else:
                    out.release()

    for _ in range(args.warmup):
        step()
    while handles:
        finish_one()
    drain()
    ctx.synchronize()
    pctx.synchronize()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    del kernel_ms[:]
    step_rows[0] = 0
    launches0 = ctx.kernel_launches + 0
    ctx.timer_start()
    for i in range(args.steps):
        step(keep_output=args.dump_outputs is not None and i == args.steps - 1)
    if overlap:
        # pipeline drain: the last exchange is ended and probed, its output taken (host-synchronised) before the stop event
        while handles:
            finish_one()
        drain()
        out_rows_seen[0] = step_rows[0] // args.steps     # every half of every timed step was drained inside the timed region
    ms = ctx.timer_stop_ms()
    launches = ctx.kernel_launches + 0 - launches0
    clocks = sampler.stop()
    if args.dump_outputs is not None:
        assert last_out[0] is not None, "the last timed step produced no page"
        dump_page(ctx, last_out[0], ["l_orderkey", "l_extendedprice", "o_orderdate"], args.dump_outputs)
        last_out[0].release()
    barrier()
    if dist is not None:
        import torch
        tt = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
        rr = torch.tensor([float(out_rows_seen[0])], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(rr)
        total_out = int(rr.item())
    else:
        total_out = out_rows_seen[0]
    assert total_out == total_rows, f"join produced {total_out} rows, expected {total_rows} (100 % match rate)"
    verify = None
    if world > 1:
        # untimed verification pass of the partitioned path: row count and key sum conserved across exchange + join, every joined row
        # carries the build payload of ITS key (sum(payload) == sum(key % 2557), the generator's closed form), and an oracle spot
        # check that received rows belong to this rank under the reference's partition function
        import torch
        check["on"] = True
        step()
        if overlap:
            while handles:
                finish_one()
            drain()
        check["on"] = False
        in_key = column_sum(ops.DeviceColumn(abi.INT64, d_lkeys, l_count))
        mine = torch.tensor([check["rows"], l_count] + [x >> 32 for x in (check["key"], check["payload"], check["key_mod"], in_key)] +
                            [x & 0xFFFFFFFF for x in (check["key"], check["payload"], check["key_mod"], in_key)], dtype=torch.int64, device=f"cuda:{local}")
        dist.all_reduce(mine)
        t = [int(x) for x in mine.tolist()]
        tot = lambda i: ((t[2 + i] << 32) + t[6 + i]) & M64
        verify = {"rows_out": t[0], "rows_in": t[1], "key_sum_conserved": tot(0) == tot(3), "payload_sum_matches_keys": tot(1) == tot(2),
                  "oracle_spot_check_rows_per_rank": check["spot"],
                  "how": "one untimed pass after the timed region: tgpu_column_sum over every joined page, all-reduced; spot check against oracle partition ids"}
        assert verify["rows_out"] == verify["rows_in"] == total_rows, verify
        assert verify["key_sum_conserved"] and verify["payload_sum_matches_keys"], verify
    ms_per_step = ms / args.steps
    value = total_rows / (ms_per_step * 1e-3)

    # ---------------- roofline of the dominant kernel of the step: the fused probe + build-payload gather.
    # Its device time is measured live inside the timed region with CUDA events recorded around the launch on the ctx stream
    # (tgpu_ctx_last_kernel_ms); the index-only probe kernel is timed alone as a second data point.
    roofline = None
    index_probe = None
    if world == 1:
        peak, peak_src = measured_peak()
        kms = float(np.mean(kernel_ms))
        achieved = ALG_BYTES_PROBE_FUSED * l_count / (kms * 1e-3) / 1e9
        traffic = NCU_TRAFFIC_PROBE_FUSED_SF100 if (args.sf == 100.0 and not args.shuffle_probe and not os.environ.get("TGPU_JOIN_HASH")) else None
        roofline = {"kernel": "join_probe_lean_kernel<2,true> (fused probe + payload gather, order-preserving table lines)", "bound": "hbm", "achieved": achieved, "peak": peak,
                    "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                    "traffic_source": "ncu --set full capture of this kernel on this configuration, profiles/r02_kernels.md (bytes per launch)",
                    "frac_of_traffic": (traffic / (kms * 1e-3) / 1e9 / peak) if traffic else None,
                    "note": "algorithmic_bytes_per_row 40 = 8 key + 12 table entry + 4 position + 8 build payload read + 8 written: SURVEY §8(d)'s 52 minus the probe columns, "
                            "which pass through as views (LookupJoinPageBuilder.java:144-150), with an 8-byte BIGINT build payload instead of the survey's INT32.  "
                            "frac can exceed 1: the model charges one table entry per probe ROW, but the ~4 rows of an order share one entry and the "
                            "order-preserving layout reads every table line once; frac_of_traffic = measured DRAM bytes (ncu) / kernel time / peak is the physical utilisation",
                    "peak_source": peak_src, "algorithmic_bytes_per_row": ALG_BYTES_PROBE_FUSED, "rows_per_launch": l_count,
                    "kernel_ms": kms, "kernel_share_of_step": kms / ms_per_step, "launches_timed": len(kernel_ms)}
        d_pos = ctx.malloc(l_count * 4)
        keys_page = ops.DevicePage([ops.DeviceColumn(abi.INT64, d_lkeys, l_count)], l_count)
        for _ in range(3):
            lookup.get_join_positions_device(keys_page, d_pos)
        reps, acc = 10, 0.0
        for _ in range(reps):
            lookup.get_join_positions_device(keys_page, d_pos)
            acc += ctx.last_kernel_ms()
        ims = acc / reps
        ia = ALG_BYTES_PROBE_INDEX * l_count / (ims * 1e-3) / 1e9
        index_probe = {"kernel": "join_probe_lean_kernel<2,false> (index-only probe)", "bound": "hbm", "achieved": ia, "peak": peak, "unit": "GB/s", "frac": ia / peak,
                       "algorithmic_bytes_per_row": ALG_BYTES_PROBE_INDEX, "kernel_ms": ims, "kernel_rows_per_sec": l_count / (ims * 1e-3)}
        ctx.free(d_pos)

    # ---------------- variant B (SURVEY.md §8d): the same join with uniformly shuffled probe keys - no key locality at all
    shuffled = None
    if world == 1 and not args.shuffle_probe and not args.no_shuffled:
        d_skeys = ctx.malloc(l_count * 8)
        ctx.check(lib.tgpu_synth_lineitem_keys(ctx.h, total_orders, l_first, l_count, SEED_LINEITEM, 1, C.c_void_p(d_skeys)))
        spage = ops.DevicePage([ops.DeviceColumn(abi.INT64, d_skeys, l_count), d_lprice_col], l_count)
        sms = []
        for i in range(2 + 3):
            ctx.timer_start()
            probe_op.add_input(spage)
            out = probe_op.get_output_device()
            t = ctx.timer_stop_ms()
            assert out.rows == l_count
            if i == 4:
                ck = column_sum(out.column(0), 2557), column_sum(out.column(2))
                assert ck[0] == ck[1], "shuffled probe: payload sum does not match the keys"
            out.release()
            if i >= 2:
                sms.append(t)
        sm = float(np.mean(sms))
        sa = ALG_BYTES_PROBE_FUSED * l_count / (sm * 1e-3) / 1e9
        shuffled = {"kernel": "LookupJoinOperator step over shuffled probe keys: join_probe_locality_kernel picks join_probe_wide_kernel (32-byte wide slots)",
                    "bound": "hbm", "achieved": sa, "peak": peak, "unit": "GB/s", "frac": sa / peak,
                    "algorithmic_bytes_per_row": ALG_BYTES_PROBE_FUSED, "ms_per_step": sm, "rows_per_sec": l_count / (sm * 1e-3),
                    "sector_floor_rows_per_sec": peak * 1e9 / (8 + 32 + 4 + 8),
                    "line_floor_rows_per_sec": peak * 1e9 / (8 + 128 + 4 + 8),
                    "frac_of_line_floor": (l_count / (sm * 1e-3)) / (peak * 1e9 / (8 + 128 + 4 + 8)),
                    "note": "every probe row reads its own random 32-byte wide slot (key, head and the payload cell in one sector; the 16-byte slots + "
                            "slot-ordered payload array of the key-ordered case cost two random accesses per row: 33 ms).  ncu (profiles/r02_kernels.md): the "
                            "L2 fills a whole 128-byte line from HBM for every random sector (134 DRAM bytes per row, whatever cudaLimitMaxL2FetchGranularity "
                            "or the load's L2 fetch-size qualifier say), so the floor of this access pattern is line_floor = copy peak / (8 key + 128 line + "
                            "4 position + 8 payload written), not sector_floor"}
        ctx.free(d_skeys)

    # ---------------- Q1 GROUP-BY side measurement (BASELINE.json configs[2]) on rank 0 at N=1
    q1 = None
    if world == 1 and args.q1_sf > 0:
        q1 = bench_q1(ctx, args)
    gb = None
    secondary = None
    if world == 1 and args.q1_sf > 0 and not args.no_secondary:
        secondary = bench_secondary(ctx)
    if world == 1 and args.q1_sf > 0 and not args.no_groupby_bigint:
        gb = bench_groupby_bigint(ctx, args)

    # ---------------- end to end: host pages in, host result out, through the same operator calls
    e2e = None
    if args.no_e2e:
        pass
    elif world == 1:
        e2e = bench_e2e(ctx, args, bridge, d_lkeys, d_lprice_col.ptr, l_count)
    elif overlap:
        e2e = bench_e2e_dist(ctx, args, dist, local, world, partitioner, probe_op, d_lkeys, d_lprice_col.ptr, l_count)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args, n_orders, probe_rows)

    if rank == 0:
        line = {"metric": "hash_join_probe_rows_per_sec", "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
                "config": workload_config(args, n_orders, probe_rows, world), "gpu_launches": int(launches), "clocks": clocks,
                "build_seconds": build_s, "output_rows_per_step": total_out, "l2_fetch_granularity": l2g.value}
        if verify:
            line["verify"] = verify
        if roofline:
            line["roofline"] = roofline
            line["roofline_index_probe"] = index_probe
        if cpu:
            line["cpu_baseline"] = cpu
        if e2e:
            line["e2e"] = e2e
        if shuffled:
            line["roofline_shuffled"] = shuffled
        if q1:
            line["groupby_q1"] = q1
        if gb:
            line["groupby_bigint"] = gb
        if secondary is not None:
            line["secondary_operators"] = secondary
        print(json.dumps(line))
    probe_op.close()
    builder.close()
    lookup.close()
    if dist is not None:
        dist.barrier()
        ctx.check(lib.tgpu_comm_destroy(ctx.h))
        dist.destroy_process_group()
    ctx.close()
    return 0


def bench_e2e(ctx, args, bridge, d_keys, d_price, n, drivers=int(os.environ.get("TGPU_E2E_DRIVERS", "4"))):
    """host -> device -> host through add_input / get_output / page_copy_to_host with pinned host memory.
    `drivers` probe operators run concurrently, each on its own context/stream, sharing the lookup source — the shape of a
    Trino task (task.concurrency drivers over one PartitionedLookupSourceFactory).  Probe blocks that the operator passes
    through unchanged (tgpu_page_passthrough_channel) are not copied back: the host already holds them, exactly like the
    probe-side views of LookupJoinPageBuilder.build."""
    from trino_b200 import abi
    from trino_b200 import operators as ops
    from trino_b200.page import Block, Page
    lib = ctx.lib
    total = n if args.e2e_rows <= 0 else min(n, args.e2e_rows)
    try:
        avail = int([l for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0].split()[1]) * 1024
    except Exception:
        avail = 32 << 30
    chunk = 32 << 20    # rows per host page
    need = total * 16 + drivers * chunk * 24
    if need > avail * 0.6:
        total = int((avail * 0.6 - drivers * chunk * 24) // 16)
    h_keys = ctx.pinned_empty(total, np.int64)
    h_price = ctx.pinned_empty(total, np.float64)
    ctx.check(lib.tgpu_memcpy_d2h(ctx.h, C.c_void_p(h_keys.ctypes.data), C.c_void_p(d_keys), total * 8))
    ctx.check(lib.tgpu_memcpy_d2h(ctx.h, C.c_void_p(h_price.ctypes.data), C.c_void_p(d_price), total * 8))
    chunks = [(lo, min(total, lo + chunk)) for lo in range(0, total, chunk)]
    # probe blocks the join passes through (here: both probe channels; the join is 1:1) are views of the caller's blocks, as in
    # LookupJoinPageBuilder.build: only the join key crosses PCIe on the way in, only the build payload on the way out
    by_reference = not os.environ.get("TGPU_E2E_MATERIALIZE")
    d2h_bytes = [0]
    rows_out = [0]
    lock = threading.Lock()

    class Driver:
        def __init__(self, index):
            self.ctx = ops.Context(ctx.device)
            self.op = ops.LookupJoinOperatorFactory(self.ctx, bridge, abi.JOIN_INNER, False, [0], [0, 1]).create_operator()
            if by_reference:
                self.op.set_passthrough_by_reference(True)
            # result landing zone (pinned): probe key, probe price, build payload
            self.bufs = [self.ctx.pinned_empty(chunk, np.int64), self.ctx.pinned_empty(chunk, np.float64), self.ctx.pinned_empty(chunk, np.int64)]
            self.valid = [np.empty(chunk // 8 + 8, np.uint8) for _ in range(3)]
            self.host_cols = (abi.Column * 3)()
            self.mine = chunks[index::drivers]

        def run(self):
            c, l = self.ctx, self.ctx.lib
            rows = copied = 0
            for lo, hi in self.mine:
                page = Page(Block(abi.INT64, h_keys[lo:hi]), Block(abi.FLOAT64, h_price[lo:hi]))
                self.op.add_input(page)
                pp = abi.PP()
                c.check(l.tgpu_op_get_output(self.op.h, C.byref(pp)))
                if not pp:
                    continue
                m = pp.contents.num_rows
                for col, (arr, t) in enumerate(zip(self.bufs, (abi.INT64, abi.FLOAT64, abi.INT64))):
                    src = C.c_int32(-1)
                    c.check(l.tgpu_page_passthrough_channel(pp, col, C.byref(src)))
                    self.host_cols[col].type = t
                    self.host_cols[col].validity = self.valid[col].ctypes.data
                    if src.value >= 0:
                        self.host_cols[col].data = None          # an unchanged view of input block src.value: nothing to copy
                    else:
                        self.host_cols[col].data = arr.ctypes.data
                        copied += m * 8
                hp = abi.Page(3, 0, m, C.cast(self.host_cols, C.POINTER(abi.Column)))
                c.check(l.tgpu_page_copy_to_host(c.h, pp, C.byref(hp)))
                l.tgpu_page_release(c.h, pp)
                rows += m
            with lock:
                rows_out[0] += rows
                d2h_bytes[0] += copied

    ds = [Driver(i) for i in range(drivers)]

    def one_pass():
        rows_out[0] = 0
        d2h_bytes[0] = 0
        ts = [threading.Thread(target=d.run) for d in ds]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        return rows_out[0]

    one_pass()
    reps = 2
    t0 = time.time()
    for _ in range(reps):
        rows = one_pass()
    dt = (time.time() - t0) / reps
    assert rows == total, (rows, total)
    d0 = ds[0]
    lo, hi = d0.mine[-1]
    assert (d0.bufs[2][:8] == (h_keys[lo:lo + 8] % 2557)).all()
    out = {"value": total / dt, "unit": "rows/s", "h2d_bytes_per_step": int(total * (8 if by_reference else 16)), "d2h_bytes_per_step": int(d2h_bytes[0]),
           "rows_per_step": int(total), "host_page_rows": chunk, "drivers": drivers,
           "timing": "wall clock around add_input(host page) + get_output + page_copy_to_host on every driver thread, pinned memory; "
                     "pass-through probe blocks are not copied back" + (" and, being views of the caller's blocks, not uploaded either "
                     "(tgpu_join_probe_set_passthrough_by_reference): H2D = join key, D2H = build payload" if by_reference else "")}
    for d in ds:
        d.op.close()
        d.ctx.close()
    return out


def bench_e2e_dist(ctx, args, dist, local, world, partitioner, probe_op, d_keys, d_price, n):
    """N > 1 end to end: every rank feeds its probe rows from pinned host pages through the split-phase exchange and the probe and
    reads the joined rows back (probe key, probe payload, build payload: received rows are not the host's own blocks, so all three
    columns come back).  Three threads per rank keep the three engines busy at once, the way a Trino task runs several drivers:
    an UPLOADER (own context/stream: H2D of page k+2 on the copy engine), the EXCHANGE + PROBE driver (the rank's communicator; same
    call sequence on every rank) and a DOWNLOADER (own context: D2H of joined page k-1).  Time = wall clock, max over ranks."""
    import queue
    import torch
    from trino_b200 import abi
    from trino_b200 import operators as ops
    lib = ctx.lib
    chunk = 32 << 20
    want = n if args.e2e_rows <= 0 else min(n, args.e2e_rows)
    try:
        avail = int([l for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0].split()[1]) * 1024
    except Exception:
        avail = 32 << 30
    budget = int(avail * 0.5 / world)                       # pinned host memory this rank may take
    if want * 16 + 4 * chunk * 24 > budget:
        want = min(want, max(chunk, (budget - 4 * chunk * 24) // 16))
    cap = torch.tensor([want], dtype=torch.int64, device=f"cuda:{local}")
    dist.all_reduce(cap, op=dist.ReduceOp.MIN)            # identical chunk count on every rank
    total = int(cap.item())
    h_keys = ctx.pinned_empty(total, np.int64)
    h_price = ctx.pinned_empty(total, np.float64)
    ctx.check(lib.tgpu_memcpy_d2h(ctx.h, C.c_void_p(h_keys.ctypes.data), C.c_void_p(d_keys), total * 8))
    ctx.check(lib.tgpu_memcpy_d2h(ctx.h, C.c_void_p(h_price.ctypes.data), C.c_void_p(d_price), total * 8))
    land = int(chunk * 1.5) + 1024                          # a rank may receive more rows than it sent
    chunks = [(lo, min(total, lo + chunk)) for lo in range(0, total, chunk)]
    up_ctx, down_ctx = ops.Context(ctx.device), ops.Context(ctx.device)
    NBUF = 4                                                # rotating device input pages (uploader ahead of the exchange driver)
    dev_in = [(up_ctx.malloc(chunk * 8), up_ctx.malloc(chunk * 8)) for _ in range(NBUF)]
    free_in = queue.Queue()
    bufs = [down_ctx.pinned_empty(land, np.int64), down_ctx.pinned_empty(land, np.float64), down_ctx.pinned_empty(land, np.int64)]
    valid = [np.empty(land // 8 + 8, np.uint8) for _ in range(3)]
    host_cols = (abi.Column * 3)()
    state = {"rows": 0, "d2h": 0, "err": None}

    def uploader(q_up):
        try:
            for k, (lo, hi) in enumerate(chunks):
                b = free_in.get()
                dk, dp = dev_in[b]
                m = hi - lo
                up_ctx.check(lib.tgpu_memcpy_h2d(up_ctx.h, C.c_void_p(dk), C.c_void_p(h_keys[lo:hi].ctypes.data), m * 8))
                up_ctx.check(lib.tgpu_memcpy_h2d(up_ctx.h, C.c_void_p(dp), C.c_void_p(h_price[lo:hi].ctypes.data), m * 8))
                q_up.put((b, ops.DevicePage([ops.DeviceColumn(abi.INT64, dk, m), ops.DeviceColumn(abi.FLOAT64, dp, m)], m)))
        except Exception as e:      # noqa: BLE001 - reported by the driver thread
            state["err"] = e
        q_up.put(None)

    q_done = queue.Queue()

    def release_done():
        while not q_done.empty():
            lib.tgpu_page_release(ctx.h, q_done.get())

    def downloader(q_down):
        try:
            while True:
                pp = q_down.get()
                if pp is None:
                    return
                m = pp.contents.num_rows
                for col, (arr, t) in enumerate(zip(bufs, (abi.INT64, abi.FLOAT64, abi.INT64))):
                    host_cols[col].type = t
                    host_cols[col].validity = valid[col].ctypes.data
                    host_cols[col].data = arr.ctypes.data
                hp = abi.Page(3, 0, m, C.cast(host_cols, C.POINTER(abi.Column)))
                down_ctx.check(lib.tgpu_page_copy_to_host(down_ctx.h, pp, C.byref(hp)))
                q_done.put(pp)           # released by the driver thread: a context (its allocator) is used by one thread at a time
                state["rows"] += m
                state["d2h"] += m * 24
        except Exception as e:      # noqa: BLE001
            state["err"] = e

    def one_pass():
        state["rows"] = state["d2h"] = 0
        while not free_in.empty():
            free_in.get()
        for b in range(NBUF):
            free_in.put(b)
        q_up, q_down = queue.Queue(maxsize=NBUF), queue.Queue(maxsize=2)
        tu = threading.Thread(target=uploader, args=(q_up,))
        td = threading.Thread(target=downloader, args=(q_down,))
        tu.start(); td.start()
        handles, inflight = [], []      # handles: (exchange handle, input buffer index); inflight: (received page, its input buffer)

        def take_output():
            pp = abi.PP()
            ctx.check(lib.tgpu_op_get_output(probe_op.h, C.byref(pp)))   # host-synchronises on the probe of the page before
            page_in, b = inflight.pop()
            lib.tgpu_page_release(ctx.h, page_in)
            if pp:
                q_down.put(pp)

        def finish_one():
            if inflight:
                take_output()
            pp = abi.PP()
            h, b = handles.pop(0)
            ctx.check(lib.tgpu_exchange_end(ctx.h, h, C.byref(pp)))
            free_in.put(b)               # _begin consumed the input page before it returned control of the SMs to later work:
            ctx.check(lib.tgpu_op_add_input(probe_op.h, pp))   # its scatter is ordered before this probe on the context's stream
            inflight.append((pp, b))

        while True:
            item = q_up.get()
            if item is None:
                break
            b, page = item
            release_done()
            h = C.c_void_p()
            # (_begin waits on the host for its count matrix, which is ordered behind the scatter of the exchange before: by the time
            #  finish_one() hands an input buffer back to the uploader, the kernels that read it have completed)
            ctx.check(lib.tgpu_exchange_begin(ctx.h, partitioner.h, page.ref(), C.byref(h)))
            handles.append((h, b))
            if len(handles) > 1:
                finish_one()
        while handles:
            finish_one()
        if inflight:
            take_output()
        q_down.put(None)
        tu.join(); td.join()
        release_done()
        if state["err"] is not None:
            raise state["err"]

    one_pass()
    dist.barrier()
    t0 = time.time()
    one_pass()
    dt = torch.tensor([time.time() - t0], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    rows = torch.tensor([float(state["rows"]), float(state["d2h"])], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(rows)
    assert int(rows[0].item()) == total * world, (int(rows[0].item()), total * world)
    assert (bufs[2][:4096] == bufs[0][:4096] % 2557).all()
    out = {"value": float(rows[0].item()) / float(dt.item()), "unit": "rows/s", "h2d_bytes_per_step": int(total * 16) * world, "d2h_bytes_per_step": int(rows[1].item()),
           "rows_per_step": int(rows[0].item()), "host_page_rows": chunk, "threads_per_rank": 3,
           "timing": "wall clock (max over ranks) around one pass of every rank's probe rows: pinned host pages -> H2D (uploader thread, own stream) -> "
                     "tgpu_exchange_begin/_end -> LookupJoinOperator -> page_copy_to_host of all three output columns (downloader thread, own stream)"}
    for dk, dp in dev_in:
        up_ctx.free(dk); up_ctx.free(dp)
    up_ctx.close(); down_ctx.close()
    return out


def bench_q1(ctx, args):
    """TPC-H Q1 fused scan+filter+project+GROUP BY over device-resident synthetic lineitem columns: with INT8 key codes (A = 38) and
    with the reference's own key types, VARCHAR(1) l_returnflag / l_linestatus (A = 46: the keys go through the device string dictionary)"""
    from q1 import q1_factory
    from trino_b200 import abi
    from trino_b200 import operators as ops
    lib = ctx.lib
    n = int(6_000_000 * args.q1_sf)
    spec = [(abi.INT32, 4), (abi.INT8, 1), (abi.INT8, 1), (abi.FLOAT64, 8), (abi.FLOAT64, 8), (abi.FLOAT64, 8), (abi.FLOAT64, 8)]
    ptrs = [ctx.malloc(n * sz) for _, sz in spec]
    ctx.check(lib.tgpu_synth_lineitem_q1(ctx.h, n, 0, SEED_LINEITEM, *[C.c_void_p(p) for p in ptrs]))
    page = ops.DevicePage([ops.DeviceColumn(t, p, n) for (t, _), p in zip(spec, ptrs)], n)
    d_off = ctx.malloc((n + 1) * 4)                      # VARCHAR(1): offsets 0..n, the bytes are the code columns themselves
    ctx.check(lib.tgpu_synth_sequence32(ctx.h, 0, n + 1, C.c_void_p(d_off)))
    cols_utf8 = [ops.DeviceColumn(t, p, n) for (t, _), p in zip(spec, ptrs)]
    cols_utf8[1] = ops.DeviceColumn(abi.UTF8, ptrs[1], n, offsets=d_off)
    cols_utf8[2] = ops.DeviceColumn(abi.UTF8, ptrs[2], n, offsets=d_off)
    page_utf8 = ops.DevicePage(cols_utf8, n)
    factory = q1_factory(ctx, fused=True)
    peak, peak_src = measured_peak()

    def measure(pg, alg, label, traffic):
        def run():
            op = factory.create_operator()
            op.add_input(pg)
            op.finish()
            out = op.get_output()
            op.close()
            return out

        for _ in range(2):
            out = run()
        reps = 5
        kms = 0.0
        ctx.timer_start()
        for _ in range(reps):
            out = run()
            kms += ctx.last_kernel_ms()
        ms = ctx.timer_stop_ms() / reps
        kms /= reps
        rows = out.rows()
        achieved = alg * n / (kms * 1e-3) / 1e9
        step_achieved = alg * n / (ms * 1e-3) / 1e9
        return {"metric": "groupby_input_rows_per_sec", "value": n / (ms * 1e-3), "unit": "rows/s", "ms_per_step": ms, "rows": n, "groups": len(rows),
                "config": f"TPC-H Q1 GROUP-BY, synthetic SF{args.q1_sf:g} lineitem, {label}, fused filter+project+aggregate (BASELINE.json configs[2])",
                "roofline": {"kernel": "tg_agg_small_jit", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "peak_source": peak_src, "algorithmic_bytes_per_row": alg, "traffic": traffic, "kernel_ms": kms, "kernel_share_of_step": kms / ms,
                             "step_frac": step_achieved / peak},
                "result_count_order": [int(r[-1]) for r in rows]}

    q1 = measure(page, ALG_BYTES_Q1_CODES, "INT8 key codes", NCU_TRAFFIC_Q1_SF300 if args.q1_sf == 300.0 else None)
    q1["utf8_keys"] = measure(page_utf8, ALG_BYTES_Q1_UTF8, "VARCHAR(1) keys (the reference's types: offsets + bytes, device string dictionary)", None)
    assert q1["utf8_keys"]["result_count_order"] == q1["result_count_order"]
    ctx.free(d_off)
    for p in ptrs:
        ctx.free(p)
    return q1


def bench_groupby_bigint(ctx, args):
    """BIGINT-key GROUP BY with many groups (SURVEY.md §8 a3: BigintGroupByHash territory, e.g. GROUP BY orderkey): 150 M rows, 10 M groups,
    sum(bigint) + count(*), one operator per timed run (all groups are new every time)"""
    from trino_b200 import abi
    from trino_b200 import operators as ops
    lib = ctx.lib
    m, groups = 150_000_000, 10_000_000
    d_keys, d_val = ctx.malloc(m * 8), ctx.malloc(m * 8)
    for lo in range(0, m, groups):
        cnt = min(groups, m - lo)
        ctx.check(lib.tgpu_synth_orders_keys(ctx.h, groups, 0, cnt, 0x55 + lo, 1, C.c_void_p(d_keys + lo * 8)))   # every pass a fresh permutation of the keys
    ctx.check(lib.tgpu_synth_lineitem_keys(ctx.h, m, 0, m, 1, 0, C.c_void_p(d_val)))
    page = ops.DevicePage([ops.DeviceColumn(abi.INT64, d_keys, m), ops.DeviceColumn(abi.INT64, d_val, m)], m)
    f = ops.HashAggregationOperatorFactory(ctx, [0], abi.STEP_SINGLE, [ops.Aggregator(abi.AGG_SUM, 1), ops.Aggregator(abi.AGG_COUNT_STAR)], expected_groups=groups)
    got = [0]

    def run():
        op = f.create_operator()
        op.add_input(page)
        got[0] = op.group_count()
        op.close()

    run()
    reps = 3
    ctx.timer_start()
    for _ in range(reps):
        run()
    ms = ctx.timer_stop_ms() / reps
    assert got[0] == groups, got
    peak, peak_src = measured_peak()
    achieved = ALG_BYTES_GROUPBY_BIGINT * m / (ms * 1e-3) / 1e9
    ctx.free(d_keys); ctx.free(d_val)
    return {"metric": "groupby_input_rows_per_sec", "value": m / (ms * 1e-3), "unit": "rows/s", "ms_per_step": ms, "rows": m, "groups": groups,
            "config": "GROUP BY a BIGINT key, 10 M groups, sum(bigint) + count(*), 150 M synthetic rows (SURVEY.md §8 a3), whole addInput incl. table set-up",
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                         "algorithmic_bytes_per_row": ALG_BYTES_GROUPBY_BIGINT, "note": "step-level (operator call), not a single kernel"}}


def bench_secondary(ctx):
    """The other two operators of the path on device-resident synthetic pages (SURVEY.md §8 a8, a13), timed like the headline step:
    FilterAndProject over the Q1 program (300 M lineitem rows) and PartitionedOutput into 8 partitions (150 M rows of BIGINT key + BIGINT payload)"""
    from q1 import q1_program
    from trino_b200 import abi
    from trino_b200 import operators as ops
    lib = ctx.lib
    peak, peak_src = measured_peak()
    out = {}

    def timed(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        ctx.timer_start()
        for _ in range(reps):
            fn()
        return ctx.timer_stop_ms() / reps

    n = 300_000_000
    spec = [(abi.INT32, 4), (abi.INT8, 1), (abi.INT8, 1), (abi.FLOAT64, 8), (abi.FLOAT64, 8), (abi.FLOAT64, 8), (abi.FLOAT64, 8)]
    ptrs = [ctx.malloc(n * sz) for _, sz in spec]
    ctx.check(lib.tgpu_synth_lineitem_q1(ctx.h, n, 0, 0x7C01, *[C.c_void_p(p) for p in ptrs]))
    page = ops.DevicePage([ops.DeviceColumn(t, p, n) for (t, _), p in zip(spec, ptrs)], n)
    fp = ops.FilterAndProjectOperatorFactory(ctx, q1_program()).create_operator()
    rows_out = [0]

    def run_fp():
        fp.add_input(page)
        o = fp.get_output_device()
        rows_out[0] = o.rows
        o.release()
    ms = timed(run_fp)
    sel = rows_out[0] / n
    alg = 38 + sel * (2 + 5 * 8)          # every input column read once, 2 key bytes + 5 doubles written per selected row
    out["filter_project"] = {"config": "FilterAndProject, TPC-H Q1 filter + 7 projections, 300 M synthetic lineitem rows", "rows": n, "ms_per_step": ms,
                             "rows_per_sec": n / (ms * 1e-3), "selectivity": sel,
                             "roofline": {"bound": "hbm", "achieved": alg * n / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                          "frac": alg * n / (ms * 1e-3) / 1e9 / peak, "peak_source": peak_src, "algorithmic_bytes_per_row": alg,
                                          "note": "step-level: tg_fp_filter_chunks_jit + fp_chunk_scan_kernel + tg_fp_project_chunks_jit"}}
    fp.close()
    for p in ptrs:
        ctx.free(p)
    m = 150_000_000
    d_keys, d_val = ctx.malloc(m * 8), ctx.malloc(m * 8)
    ctx.check(lib.tgpu_synth_lineitem_keys(ctx.h, m, 0, m, 0x7C01, 0, C.c_void_p(d_keys)))
    ctx.check(lib.tgpu_synth_lineitem_keys(ctx.h, m, 0, m, 1, 0, C.c_void_p(d_val)))
    gpage = ops.DevicePage([ops.DeviceColumn(abi.INT64, d_keys, m), ops.DeviceColumn(abi.INT64, d_val, m)], m)
    part = ops.PartitionedOutputOperatorFactory(ctx, [0], 8).create_operator()

    def run_part():
        part.add_input(gpage)
        while True:
            o = part.get_output_device()
            if o is None:
                break
            o.release()
    ms = timed(run_part, reps=3, warm=1)
    out["partitioned_output"] = {"config": "PartitionedOutput (PagePartitioner), 8 partitions, BIGINT key + BIGINT payload, 150 M synthetic rows", "rows": m,
                                 "ms_per_step": ms, "rows_per_sec": m / (ms * 1e-3),
                                 "roofline": {"bound": "hbm", "achieved": 36 * m / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                              "frac": 36 * m / (ms * 1e-3) / 1e9 / peak, "peak_source": peak_src, "algorithmic_bytes_per_row": 36,
                                              "note": "step-level: xchg_hist_warp_kernel + xchg_offsets_kernel + xchg_scatter_warp_kernel (SURVEY.md §8d: 8 key + 1 + 1 id + 16 in + 16 out, rounded)"}}
    part.close()
    ctx.free(d_keys); ctx.free(d_val)
    return out


def cpu_baseline(args, n_orders, probe_rows):
    import oracle_lib as o
    out = cpu_probe_measure(args, n_orders, probe_rows, 10, 2)
    threads = out["cores"]
    if args.q1_sf > 0:
        n = 60_000_000
        cols = o.synth_lineitem_q1(n, 0, SEED_LINEITEM)
        o.q1_run(cols, 10471, threads)
        runs = sorted(o.q1_run(cols, 10471, threads)[0] for _ in range(5))
        secs = runs[len(runs) // 2]
        out["groupby_q1"] = {"value": n / secs, "unit": "rows/s", "cores": threads, "kind": "port", "spread": {"min_s": runs[0], "max_s": runs[-1]},
                             "sample": f"{n} synthetic lineitem rows, filter -> 7 projection loops -> FlatHash group ids -> 8 accumulator passes, {threads} partial drivers + final merge; median of 5 passes"}
    return out


if __name__ == "__main__":
    sys.exit(main())
