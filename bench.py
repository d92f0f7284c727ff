#!/usr/bin/env python
"""bench.py — coprocessor rows/sec on B200 (BASELINE.json metric), one JSON line on rank 0.

Headline workload ("C3", BASELINE.json configs[2] with the metric's own filter): a region-sharded synthetic table of
1e9 rows per GPU (HBM-resident, row format v2, one version per key, columns {id PK, key i32 in [0, 1024), val i64 in
[-2^40, 2^40)}), DAG = BatchTableScan -> BatchSelection(val < 0) -> BatchFastHashAggregation GROUP BY key: SUM(val).
A "step" is one pass of the hot path over the whole table followed by the final merge of the per-GPU partial
aggregates (all_gather over NCCL + exact re-aggregation; TiDB's final HashAgg in the reference):
  value : inputs already resident in HBM, result left in HBM (device time, CUDA events on the launch stream)
  e2e   : the same request through the C ABI with HOST buffers (pinned): H2D of every block + D2H of the result inside
          the timed region (cold); e2e_warm: the same with the region blocks pinned in the HBM block cache
  sub   : C2 (scan + selection, 1e8 rows x 8 i64), C4 (TopN + all_gather merge), C5 (checksum + XOR merge), each with
          its own roofline fraction and CPU-arm rate
  --impl reference : the CPU oracle (C++ restatement of the reference algorithm; the Rust reference cannot be
          built in this image) on all host cores, one region task per thread, regions generated on the host by
          oracle/orc_gen.h (no product code on that arm), each step a bounded sample of the workload.
"""
import argparse
import ctypes as C
import json
import os
import struct
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

TABLE_ID = 1000
SEED = 0x525C682A2F7CE3DB  # tests/benches/coprocessor_executors/util/fixture.rs:26
READ_TS = 1000
COMMIT_TS, NEWER_TS = 20, 5000
METRIC = "coprocessor rows/sec (scan+filter+hash-agg) at 1/2/4/8 B200 vs host-CPU ref"
GROUPS = 1024

# ---- workloads (SURVEY.md 8(d)) ------------------------------------------------------------------------------------
TABLES = {
    # name: (n_cols, col_lo, col_range (0 = full-range i64), null_per_million)
    "c3": (2, [0, -(1 << 40)], [GROUPS, 1 << 41], None),
    "c2": (8, [0] * 8, [0] * 8, None),
    "c4": (2, [0, 0], [0, 0], [0, 10000]),
}
TITLES = {
    "c3": f"C3: BatchTableScan + BatchSelection(val < 0) + BatchFastHashAggregation GROUP BY i32 key (G={GROUPS}) SUM(i64), row format v2, 1 version/key (BASELINE.json configs[2] + the metric's filter)",
    "c2": "C2: BatchTableScan + BatchSelection(col0 < 0) on 8 i64 cols, row format v2 (BASELINE.json configs[1])",
    "c4": "C4: BatchTopN ORDER BY c0 DESC, c1 ASC LIMIT 1000 (c1 1 % NULL) + all_gather merge (BASELINE.json configs[3])",
    "c5": "C5: Checksum CRC-64/XZ over the C2 table's KVs + XOR merge (BASELINE.json configs[4])",
}


def build_plan(name="c3"):
    from tikv_b200 import ffi
    from tikv_b200.plan import ColumnDef, Plan, col, const_int, lt
    if name == "c3":
        cols = [ColumnDef(100, pk_handle=True), ColumnDef(1, tp=ffi.TP_LONG), ColumnDef(2)]
        return Plan().table_scan(TABLE_ID, cols).selection(lt(col(2), const_int(0))).aggregation([("sum", col(2))], group_by=[col(1, tp=ffi.TP_LONG)]).build()
    if name == "c2":
        cols = [ColumnDef(100, pk_handle=True)] + [ColumnDef(i + 1) for i in range(8)]
        return Plan().table_scan(TABLE_ID, cols).selection(lt(col(1), const_int(0))).build(output_offsets=list(range(1, 9)))
    if name == "c4":
        cols = [ColumnDef(100, pk_handle=True), ColumnDef(1), ColumnDef(2)]
        return Plan().table_scan(TABLE_ID, cols).topn([(col(1), True), (col(2), False)], 1000).build()
    raise ValueError(name)


def row_key(handle):
    return b"t" + struct.pack(">Q", TABLE_ID ^ (1 << 63)) + b"_r" + struct.pack(">Q", handle ^ (1 << 63))


def table_range(first=None, n=None):
    pre = b"t" + struct.pack(">Q", TABLE_ID ^ (1 << 63))
    if first is None:
        return [(pre + b"_r", pre + b"_s")]
    return [(row_key(first), row_key(first + n))]


def gen_spec(ffi, table, first_handle, n_rows, row_format=2):
    n_cols, lo, rng, nulls = TABLES[table]
    spec = ffi.GenSpec()
    spec.table_id, spec.first_handle, spec.n_rows, spec.n_cols, spec.row_format, spec.seed = TABLE_ID, first_handle, n_rows, n_cols, row_format, SEED
    keep = [(C.c_int64 * n_cols)(*lo), (C.c_uint64 * n_cols)(*rng)]
    spec.col_lo, spec.col_range = keep
    if nulls:
        keep.append((C.c_uint32 * n_cols)(*nulls))
        spec.null_per_million = keep[-1]
    spec.commit_ts, spec.newer_ts = COMMIT_TS, NEWER_TS
    return spec, keep


def gen_blocks(ffi, device, table, n_rows, n_blocks, first_handle=0, row_format=2):
    """Generate the table on the device as `n_blocks` CF_WRITE blocks (one per region).  Returns (gens, GenBlock list)."""
    L = ffi.lib()
    gens, blks = [], []
    per = (n_rows + n_blocks - 1) // n_blocks
    h, left = first_handle, n_rows
    while left > 0:
        n = min(per, left)
        spec, keep = gen_spec(ffi, table, h, n, row_format)
        g, blk = C.c_void_p(), ffi.GenBlock()
        rc = L.b2_gen_create(device, C.byref(spec), C.byref(g), C.byref(blk))
        if rc != 0:
            raise RuntimeError("b2_gen_create: " + L.b2_last_error_message().decode())
        gens.append(g)
        blks.append(blk)
        h += n
        left -= n
    return gens, blks


class Source:
    def __init__(self, ffi, blocks, location, device):
        self.arr = (ffi.CfBlock * len(blocks))(*blocks)
        s = ffi.RegionSource()
        s.location, s.device, s.write, s.n_write = location, device, self.arr, len(blocks)
        s.read_ts, s.isolation_level, s.check_has_newer_ts_data = READ_TS, ffi.ISO_SI, 1
        self.c = s


def blocks_to_pinned_host(ffi, device, blks):
    """D2H copy of generated blocks into pinned host buffers near the GPU (setup, outside every timed region)."""
    L = ffi.lib()
    out, keep = [], []
    for b in blks:
        n = b.block.n
        sizes = [((b.key_bytes + 31) // 16) * 16, 4 * (n + 1), ((b.val_bytes + 31) // 16) * 16, 4 * (n + 1)]
        srcs = [b.block.keys, b.block.key_offs, b.block.vals, b.block.val_offs]
        copy = [b.key_bytes, 4 * (n + 1), b.val_bytes, 4 * (n + 1)]
        ptrs = []
        for sz, src, cb in zip(sizes, srcs, copy):
            p = L.b2_host_alloc_pinned_near(device, sz)
            if not p:
                raise RuntimeError("pinned host allocation failed")
            keep.append(p)
            if L.b2_copy_to_host(device, p, src, cb) != 0:
                raise RuntimeError("D2H copy failed")
            ptrs.append(p)
        hb = ffi.CfBlock()
        hb.keys, hb.key_offs, hb.vals, hb.val_offs, hb.n = ptrs[0], ptrs[1], ptrs[2], ptrs[3], n
        out.append(hb)
    return out, keep


def run_dag(ffi, plan, ranges, src, out_loc, chunk, stream=0, after=None):
    """One request: open the executor, pull batches until drained; `after(ex, batch)` sees every batch while the executor
    is alive (the final merges read its device-resident results).  Returns (rows_out, stats)."""
    from tikv_b200.executor import BatchExecutor
    rows = 0
    with BatchExecutor(plan, ranges, src, output=out_loc, stream=stream) as ex:
        while True:
            rc, b = ex.next_batch_raw(chunk)
            if rc != 0:
                raise RuntimeError("next_batch failed: " + ex.last_error().message.decode())
            rows += b.n_rows
            if after is not None:
                after(ex, b)
            if b.is_drained != ffi.DRAIN_REMAIN:
                break
        st = ex.collect_exec_stats()
    return rows, st


def sst_e2e(ffi, device, blks, plan, after, args, stream, barrier, max_over_ranks, e2e_rows, world):
    """End to end from RocksDB data blocks in pinned host memory.  Setup (untimed): the generated regions are encoded on the
    device (b2_sst_encode, ~32 KiB blocks, restart interval 16, 'z' + internal-key footer + trailer: the stored form of a
    TiKV write-CF block, src/config/mod.rs:966) and copied to the host.  Timed, per step: b2_sst_decode of every region
    (H2D of the compressed bytes + expansion on the device) and the request over the decoded blocks, result to the host."""
    import numpy as np
    import torch
    from tikv_b200.executor import SstDecoder
    L = ffi.lib()
    enc_host, keep, flat_bytes, enc_bytes = [], [], 0, 0
    for b in blks:
        per = max(16, 32768 // max(8, int((b.key_bytes + b.val_bytes) / max(1, b.block.n)) - 9))
        h, enc = C.c_void_p(), ffi.SstEncoded()
        if L.b2_sst_encode(device, C.byref(b.block), per, 16, 1, ord("z"), 8, 5, C.byref(h), C.byref(enc)) != 0:
            raise RuntimeError("b2_sst_encode: " + L.b2_last_error_message().decode())
        p = L.b2_host_alloc_pinned_near(device, enc.data_len + 64)
        if not p:
            raise RuntimeError("pinned host allocation failed")
        keep.append(p)
        offs = np.zeros(enc.n_blocks + 1, dtype=np.uint64)
        if L.b2_copy_to_host(device, p, enc.data, enc.data_len) != 0 or L.b2_copy_to_host(device, offs.ctypes.data, enc.block_offs, 8 * len(offs)) != 0:
            raise RuntimeError("D2H copy failed")
        L.b2_sst_free(h)
        enc_host.append((p, offs))
        flat_bytes += b.key_bytes + b.val_bytes + 8 * b.block.n
        enc_bytes += enc.data_len
    decs = [SstDecoder(device) for _ in blks]
    pool = None
    try:
        from concurrent.futures import ThreadPoolExecutor
        pool = ThreadPoolExecutor(max_workers=2)  # two regions in flight: one expands while the other's bytes cross PCIe

        def step():
            res = list(pool.map(lambda a: a[0].decode(a[1][0], a[1][1]), zip(decs, enc_host)))
            arr = [blk for blk, _ in res]
            h2d = sum(st.h2d_bytes for _, st in res)
            dms = sum(st.decode_ms for _, st in res)
            src = Source(ffi, arr, ffi.LOC_DEVICE, device)
            rows, st = run_dag(ffi, plan, table_range(), src, ffi.LOC_HOST, args.chunk, stream.cuda_stream, after)
            return rows, st, h2d, dms
        for _ in range(2):
            step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        k = args.steps
        dms_acc = 0.0
        for _ in range(k):
            rows, st, h2d, dms = step()
            dms_acc += dms
        e1.record(stream)
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1)) / k
    finally:
        if pool:
            pool.shutdown()
        for d in decs:
            d.close()
        for p in keep:
            L.b2_host_free_pinned(p)
    return {"value": e2e_rows * world / (ms / 1e3), "unit": "rows/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(st.d2h_bytes), "ms_per_step": ms,
            "rows_per_gpu": int(e2e_rows), "rows_out": int(rows), "decode_ms_per_step": dms_acc / k,
            "source": "RocksDB data blocks (uncompressed, prefix-compressed keys, 'z' prefix + internal-key footer + trailer) in pinned host memory, "
                      "expanded on the device by b2_sst_decode",
            "compressed_to_flat_bytes": enc_bytes / max(1, flat_bytes),
            "note": "cold: every data block crosses PCIe inside the timed region"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
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
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def usable_cores():
    """Host threads this process may actually run at once: the affinity mask, capped by the cgroup CPU quota (a
    container can see 128 CPUs and be allowed 32 of them; oversubscribing would understate the CPU arm)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:  # cgroup v2: "<quota|max> <period>"
            q, per = f.read().split()[:2]
            if q != "max":
                quota = int(q) / int(per)
    except (OSError, ValueError):
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:  # cgroup v1
                q, per = int(f.read()), int(g.read())
                if q > 0 and per > 0:
                    quota = q / per
        except (OSError, ValueError):
            pass
    if quota is not None:
        n = min(n, max(1, int(quota + 0.999)))
    return max(1, n)


def host_mem_available():
    """Bytes of host memory this process may still take: MemAvailable, capped by the cgroup limit."""
    avail = None
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    except OSError:
        pass
    for lim, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                     ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            l = open(lim).read().strip()
            if l != "max" and int(l) < (1 << 60):
                room = int(l) - int(open(cur).read().strip())
                avail = room if avail is None else min(avail, room)
        except (OSError, ValueError):
            pass
    return avail if avail is not None else 8 << 30


# ---- CPU arm: the oracle on host-generated regions (nothing of the product library is used here) -----------------------
class _Src:
    def __init__(self, c):
        self.c = c


class CpuArm:
    def __init__(self, table, rows_per_task, tasks, threads, first_handle=0):
        import orc
        from tikv_b200 import ffi
        self.L = orc.lib()
        L = self.L
        L.orc_bench_create.argtypes = [C.POINTER(ffi.GenSpec), C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint32]
        L.orc_bench_create.restype = C.c_void_p
        L.orc_bench_step.argtypes = [C.c_void_p, C.POINTER(ffi.DagPlan), C.POINTER(ffi.KeyRange), C.c_uint32, C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_int)]
        L.orc_bench_step.restype = C.c_uint64
        L.orc_bench_checksum_step.argtypes = [C.c_void_p, C.POINTER(ffi.KeyRange), C.c_uint32, C.c_uint32, C.POINTER(ffi.ChecksumResponse)]
        L.orc_bench_source.argtypes = [C.c_void_p, C.c_uint32]
        L.orc_bench_source.restype = C.POINTER(ffi.RegionSource)
        L.orc_bench_bytes.argtypes = [C.c_void_p]
        L.orc_bench_bytes.restype = C.c_uint64
        L.orc_bench_free.argtypes = [C.c_void_p]
        spec, keep = gen_spec(ffi, table, first_handle, rows_per_task)
        self.ffi, self.rows_per_task, self.tasks, self.threads = ffi, rows_per_task, tasks, threads
        self.h = L.orc_bench_create(C.byref(spec), tasks, rows_per_task, READ_TS, threads)

    def source(self, task=0):
        return self.L.orc_bench_source(self.h, task).contents

    def step(self, plan):
        from tikv_b200.plan import key_ranges
        kr, keep = key_ranges(table_range())
        scanned, status = C.c_uint64(), C.c_int()
        t0 = time.perf_counter()
        rows_out = self.L.orc_bench_step(self.h, C.byref(plan.c), kr, 1, self.threads, C.byref(scanned), C.byref(status))
        dt = time.perf_counter() - t0
        if status.value != 0:
            raise RuntimeError(f"oracle failed with status {status.value}")
        return dt, int(rows_out)

    def checksum_step(self):
        from tikv_b200.plan import key_ranges
        kr, keep = key_ranges(table_range())
        out = self.ffi.ChecksumResponse()
        t0 = time.perf_counter()
        st = self.L.orc_bench_checksum_step(self.h, kr, 1, self.threads, C.byref(out))
        dt = time.perf_counter() - t0
        if st != 0:
            raise RuntimeError(f"oracle checksum failed with status {st}")
        return dt, out

    def rate(self, plan, steps=1, warmup=1):
        times = []
        for it in range(warmup + steps):
            dt, _ = self.step(plan) if plan is not None else self.checksum_step()
            if it >= warmup:
                times.append(dt)
        sec = sum(times) / len(times)
        return self.rows_per_task * self.tasks / sec, sec

    def close(self):
        if self.h:
            self.L.orc_bench_free(self.h)
            self.h = None


def oracle_result(plan, ranges, src):
    """One oracle request -> (status, numpy-friendly columns)."""
    import orc
    from tikv_b200.plan import key_ranges
    import numpy as np
    L = orc.lib()
    kr, keep = key_ranges(ranges)
    h = C.c_void_p()
    L.orc_dag_handle(C.byref(plan.c), kr, len(ranges), C.byref(src), C.byref(h))
    n = L.orc_result_rows(h)
    status = L.orc_result_status(h)
    cols = []
    from tikv_b200 import ffi
    for c in range(L.orc_result_cols(h)):
        kind = L.orc_result_col_kind(h, c)
        nn = np.ctypeslib.as_array(L.orc_result_col_nonnull(h, c), shape=(n,)).astype(bool) if n else np.zeros(0, bool)
        if kind == ffi.COL_DECIMAL:
            vals = [int(L.orc_result_decimal_str(h, c, i).decode()) if nn[i] else None for i in range(n)]
        else:
            a = np.ctypeslib.as_array(L.orc_result_col_i64(h, c), shape=(n,)).copy() if n else np.zeros(0, np.int64)
            vals = (a, nn.copy())
        cols.append(vals)
    L.orc_result_free(h)
    return status, n, cols


def gpu_columns(ffi, b, device):
    """b2_batch with device-resident Int columns -> [(int64 tensor, nonnull bool tensor)] (no copy of the data)."""
    import torch
    from tikv_b200.dist import _CudaArray
    n = int(b.n_rows)
    dev = torch.device("cuda", device)
    out = []
    for i in range(b.n_columns):
        c = b.columns[i]
        if n == 0:
            out.append((torch.zeros(0, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.bool, device=dev)))
            continue
        data = torch.as_tensor(_CudaArray(c.data, (n,), "<i8"), device=dev)
        bm = torch.as_tensor(_CudaArray(c.null_bitmap, ((n + 63) // 64,), "<i8"), device=dev)
        idx = torch.arange(n, device=dev)
        nn = ((bm[idx >> 6] >> (idx & 63)) & 1).bool()
        out.append((data, nn))
    return out


def parity_check(ffi, device, name, plan, dev_src, first_handle, sample_rows, stream):
    """Bench-scale parity: the oracle on host-generated rows [first_handle, +sample_rows) vs the CUDA path on the same
    handles of the resident table (a key-range request).  Raises on any difference."""
    import numpy as np
    import torch
    from tikv_b200.executor import BatchExecutor, _decimal_to_int
    table = "c2" if name == "c5" else name
    arm = CpuArm(table, sample_rows, 1, 1, first_handle=first_handle)
    rng = table_range(first_handle, sample_rows)
    t0 = time.perf_counter()
    info = {"rows": sample_rows, "first_handle": first_handle}
    if name == "c5":
        import orc
        from tikv_b200.executor import checksum
        st, exp, msg = orc.checksum(rng, _Src(arm.source()))
        rc, got, msg2 = checksum(rng, dev_src)
        assert st == 0 and rc == 0, (st, rc, msg, msg2)
        assert tuple(exp) == tuple(got), f"checksum parity: oracle {exp} vs CUDA {got}"
        info["checked"] = "checksum, total_kvs, total_bytes"
    else:
        status, n, cols = oracle_result(plan, rng, arm.source())
        assert status == 0
        with BatchExecutor(plan, rng, dev_src, output=ffi.LOC_HOST, stream=stream) as ex:
            got_cols, got_n = None, 0
            while True:
                r = ex.next_batch(1 << 24)
                assert r.error is None, r.error
                if got_cols is None:
                    got_cols = [list(c) for c in r.columns]
                else:
                    for a, c in zip(got_cols, r.columns):
                        a.extend(c)
                if r.is_drained:
                    break
        got_n = len(got_cols[0]) if got_cols else 0
        assert got_n == n, f"{name} parity: oracle {n} rows vs CUDA {got_n}"
        if name == "c3":  # [SUM(val) decimal, key]: group order is unspecified
            exp = {int(k) if nn else None: s for s, k, nn in zip(cols[0], cols[1][0], cols[1][1])}
            got = {k: s for s, k in zip(got_cols[0], got_cols[1])}
            assert exp == got, f"c3 parity: {sum(1 for k in exp if exp[k] != got.get(k))} of {len(exp)} groups differ"
            info["checked"] = f"{n} groups: key set and exact SUM per group"
        else:  # ordered rows: every cell (NULLs as None)
            for ci, (oc, gc) in enumerate(zip(cols, got_cols)):
                a, nn = oc
                g = np.array([0 if v is None else v for v in gc], dtype=np.int64)
                gn = np.array([v is not None for v in gc], dtype=bool)
                assert np.array_equal(nn, gn) and np.array_equal(np.where(nn, a, 0), g), f"{name} parity: column {ci} differs"
            info["checked"] = f"{n} rows x {len(cols)} columns, every cell in order"
    info["seconds"] = round(time.perf_counter() - t0, 2)
    arm.close()
    return info


def dump_outputs(out_dir, outputs):
    """--dump-outputs: the merged results of the last timed step of each workload, as a caller receives them, one float64
    .npy per array.  An int64 array becomes <name>_hi (its signed upper 32 bits) and <name>_lo (its lower 32 bits), both
    exact in float64.  Files: c3_keys, c3_key_null, c3_acc (one row per group, sorted by key; the accumulator words of
    b2_agg_partials), c4_col<i>, c4_col<i>_null (the top rows in order), c5_checksum ([crc64, total_kvs, total_bytes])."""
    import numpy as np
    import torch
    arrays = {}

    def ints(name, t):
        t = torch.as_tensor(t).to("cpu", torch.int64)
        arrays[name + "_hi"], arrays[name + "_lo"] = (t >> 32).double(), (t & 0xFFFFFFFF).double()

    for name, res in outputs.items():
        if name == "c3":
            keys, nul, acc = res
            ints("c3_keys", keys)
            arrays["c3_key_null"] = nul.double().cpu()
            ints("c3_acc", acc)
        elif name == "c4":
            for i, (c, n) in enumerate(zip(*res)):
                ints(f"c4_col{i}", c)
                arrays[f"c4_col{i}_null"] = n.double().cpu()
        elif name == "c5":
            ints("c5_checksum", [v - (1 << 64) if v >= 1 << 63 else v for v in res])
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_per_entry(kernel):
    p = os.path.join(ROOT, "profiles", f"{kernel}_r2_traffic.json")
    if os.path.exists(p):
        return json.load(open(p)).get("dram_bytes_per_entry")
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of every timed loop")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the results of the last timed step of each workload to DIR/<name>.npy (see dump_outputs)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=1_000_000_000, help="rows per GPU of the headline table")
    ap.add_argument("--blocks", type=int, default=16, help="CF_WRITE blocks (regions) per GPU of the headline table")
    ap.add_argument("--sub-rows", type=int, default=100_000_000, help="rows per GPU of the sub-record tables (C2/C5, C4)")
    ap.add_argument("--chunk", type=int, default=1 << 24, help="CF_WRITE entries per next_batch (scan pipelines)")
    ap.add_argument("--cpu-sample-rows", type=int, default=2_000_000, help="rows per region task of the CPU arm")
    ap.add_argument("--e2e-rows", type=int, default=0, help="rows of the end-to-end (host buffer) request; 0 = as many of --rows as host memory allows")
    ap.add_argument("--parity-rows", type=int, default=1_000_000)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sst", action="store_true", help="end to end from flat CF blocks only (skip the RocksDB data-block source)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the C2 / C4 / C5 sub-records")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-jit", action="store_true", help="generic kernels only")
    ap.add_argument("--only", default="", help="debug: run one workload (c2|c4|c5) as the headline shape")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.only == "c2"):
        ap.error("--dump-outputs: only the CUDA path's aggregation, TopN and checksum results are dumped (C2 leaves its rows on the device)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = usable_cores()

    import __graft_entry__ as ge
    if args.impl == "reference":
        # the reference arm never touches the product library: oracle + host generator only
        if rank != 0:
            return
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
        plan = build_plan("c3")
        arm = CpuArm("c3", args.cpu_sample_rows, cores, cores)
        rate, sec = arm.rate(plan, steps=max(1, args.steps), warmup=args.warmup)
        arm.close()
        sample = f"each step = {cores} region tasks x {args.cpu_sample_rows} rows of that table, one task per thread, each task its own host-generated region (a bounded sample of the workload)"
        line = {
            "impl": "reference", "metric": METRIC, "value": rate, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64", "data": "synthetic",
            "config": {"workload": TITLES["c3"], "rows_per_step": args.cpu_sample_rows * cores, "sample": sample},
            "cpu_baseline": {"value": rate, "unit": "rows/s", "cores": cores, "kind": "port",
                             "sample": sample + " (restated C++ CPU baseline, not the TiKV Rust binary)"},
            "e2e": {"value": rate, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
        return

    if rank == 0:
        ge.build()
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    from tikv_b200 import dist as b2dist
    from tikv_b200 import ffi
    from tikv_b200.executor import checksum as b2_checksum
    L = ffi.lib()
    device = local_rank if world > 1 else 0
    torch.cuda.set_device(device)
    dev = torch.device("cuda", device)
    t_setup = time.time()
    if args.no_jit:
        os.environ["B2_JIT"] = "off"
    plans = {n: build_plan(n) for n in ("c3", "c2", "c4")}
    # prepared plans: the kernels specialised for these DAG shapes are compiled once (NVRTC, disk-cached), like prepared
    # statements; compiled concurrently
    prep = {}
    if not args.no_jit:
        def _prep(n):
            prep[n] = L.b2_plan_prepare(C.byref(plans[n].c), device)
        ths = [threading.Thread(target=_prep, args=(n,)) for n in plans]
        [t.start() for t in ths]
        [t.join() for t in ths]
    kernel_kind = "generic (interpreted plan)" if args.no_jit or any(prep.values()) else "plan-specialised (compiled at run time, cached per plan shape)"
    stream = torch.cuda.Stream(device=device)
    peak, peak_src = peak_hbm()

    def barrier():
        torch.cuda.synchronize(device)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    merge_ms_acc = [0.0]

    def timed_merge(fn):
        """Run a final merge on `stream`, bracketed by its own events (reported as merge_ms)."""
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            a.record(stream)
            out = fn()
            b.record(stream)
        b.synchronize()
        merge_ms_acc[0] += a.elapsed_time(b)
        return out

    merged = {}

    def after_agg(ex, b):
        def fn():
            keys, nul, acc = b2dist.agg_partials_as_tensors(ex, device)
            return b2dist.merge_agg_partials(keys, nul, acc)
        merged["c3"] = timed_merge(fn)

    def after_topn(ex, b):
        def fn():
            cols = gpu_columns(ffi, b, device)
            return b2dist.merge_topn([c for c, _ in cols], [~nn for _, nn in cols], [(1, True, "i64"), (2, False, "i64")], 1000)
        merged["c4"] = timed_merge(fn)

    def run_workload(name, src, steps, warmup, chunk):
        """warm-up + K timed steps of one workload over a resident table; device time, max over ranks."""
        plan = plans.get(name)
        after = {"c3": after_agg, "c4": after_topn}.get(name)

        def one():
            if name == "c5":
                rc, res, msg = b2_checksum(table_range(), src, stream=stream.cuda_stream, want_stats=True)
                if rc != 0:
                    raise RuntimeError("checksum failed: " + msg)
                st = res[3]
                merged["c5"] = timed_merge(lambda: b2dist.merge_checksum(res[0], res[1], res[2], device=dev))
                return res[1], st
            return run_dag(ffi, plan, table_range(), src, ffi.LOC_DEVICE, chunk, stream.cuda_stream, after)
        rows_out, st = 0, None
        for _ in range(warmup):
            rows_out, st = one()
        barrier()
        merge_ms_acc[0] = 0.0
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        kernel_ns = launches = jit_launches = 0
        for _ in range(steps):
            rows_out, st = one()
            kernel_ns += st.kernel_time_ns
            launches += st.kernel_launches
            jit_launches += st.jit_launches
        ev1.record(stream)
        barrier()
        ms_step = max_over_ranks(ev0.elapsed_time(ev1)) / steps
        return {"rows_out": int(rows_out), "ms_per_step": ms_step, "kernel_s": kernel_ns / 1e9 / steps, "launches": int(launches), "jit_launches": int(jit_launches),
                "merge_ms": max_over_ranks(merge_ms_acc[0]) / steps}

    def roofline(kernel, in_bytes, out_bytes, r, n_entries):
        achieved = (in_bytes + out_bytes) / r["kernel_s"] / 1e9 if r["kernel_s"] > 0 else 0.0
        tpe = traffic_per_entry(kernel)
        scan_launches = max(1, r["launches"])
        return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": tpe * n_entries / (scan_launches / max(1, r.get("steps", 1))) if tpe else None,
                "kernel": kernel, "kernel_build": kernel_kind, "algorithmic_bytes_per_step": in_bytes + out_bytes,
                "kernel_ms_per_step": r["kernel_s"] * 1e3, "peak_source": peak_src}

    # ================= headline: C3 =================
    head = args.only or "c3"
    table = "c2" if head == "c5" else head
    gens, blks = gen_blocks(ffi, device, table, args.rows, args.blocks, first_handle=rank * args.rows)
    dev_src = Source(ffi, [b.block for b in blks], ffi.LOC_DEVICE, device)
    n_entries = sum(b.block.n for b in blks)
    in_bytes = sum(b.key_bytes + b.val_bytes + 8 * b.block.n for b in blks)
    parity = {}
    if not args.no_parity:
        parity[head] = parity_check(ffi, device, head, plans.get(head), dev_src, rank * args.rows + (args.rows // 3), min(args.parity_rows, args.rows // 2), stream.cuda_stream)
    sampler = ClockSampler(device)
    sampler.start()
    r = run_workload(head, dev_src, args.steps, args.warmup, args.chunk)
    r["steps"] = args.steps
    outputs = {head: merged[head]} if head in merged else {}  # (the end-to-end requests below overwrite merged["c3"])
    value = args.rows * world / (r["ms_per_step"] / 1e3)
    out_bytes = r["rows_out"] * (8 * 8) + 8 * ((r["rows_out"] + 63) // 64) * 8 if head == "c2" else 0
    kname = {"c3": "scan_kernel<PM_AGG>", "c2": "scan_kernel<PM_SCAN>", "c4": "scan_kernel<PM_TOPN>", "c5": "scan_kernel<PM_CHECKSUM>"}[head]
    kfile = {"c3": "agg_kernel", "c2": "scan_kernel", "c4": "topn_kernel", "c5": "checksum_kernel"}[head]
    roof = roofline(kfile, in_bytes, out_bytes, r, n_entries)
    roof["kernel"] = kname
    if head == "c3" and "c3" in merged:
        n_groups = int(merged["c3"][0].shape[0])
    else:
        n_groups = None

    # ---- end to end with host buffers (cold), then with the blocks pinned in the HBM block cache (warm) ----
    e2e = None
    if not args.no_e2e and head != "c5":
        bytes_per_row = in_bytes / max(1, args.rows)
        budget = host_mem_available() * 0.45 / max(1, min(world, 8))
        want = args.e2e_rows or args.rows
        e2e_blocks = max(1, min(len(blks), int(budget // (bytes_per_row * (args.rows / len(blks))))))
        e2e_blocks = min(e2e_blocks, max(1, -(-want * len(blks) // args.rows)))
        sub_blks = blks[:e2e_blocks]
        e2e_rows = sum(b.n_user_keys for b in sub_blks)
        plan = plans[head]
        after = after_agg if head == "c3" else None  # (the TopN merge reads device-resident columns: HBM-resident steps only)
        # (a) the regions as TiKV's block cache holds them: RocksDB data blocks (uncompressed, prefix-compressed keys, 'z' data
        # prefix, internal-key footer, block trailer) in pinned host memory; every step expands them on the device
        # (b2_sst_decode) and runs the request over the decoded blocks.  Fewer bytes cross PCIe than with flat blocks.
        e2e_sst = None
        if not args.no_sst:
            try:
                e2e_sst = sst_e2e(ffi, device, sub_blks, plan, after, args, stream, barrier, max_over_ranks, e2e_rows, world)
            except Exception as ex:  # the flat-block request below still measures the end-to-end path
                e2e_sst = {"error": str(ex)[:300]}
        host_blocks, pinned = blocks_to_pinned_host(ffi, device, sub_blks)
        host_src = Source(ffi, host_blocks, ffi.LOC_HOST, device)
        for _ in range(2):
            r_e2e, st_e = run_dag(ffi, plan, table_range(), host_src, ffi.LOC_HOST, args.chunk, stream.cuda_stream, after)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        k = args.steps
        for _ in range(k):
            r_e2e, st_e = run_dag(ffi, plan, table_range(), host_src, ffi.LOC_HOST, args.chunk, stream.cuda_stream, after)
        e1.record(stream)
        barrier()
        ms_e = max_over_ranks(e0.elapsed_time(e1)) / k
        part = "" if e2e_rows == args.rows else f"; {e2e_blocks} of {len(blks)} regions of the table (pinned host memory budget), same plan"
        e2e = {"value": e2e_rows * world / (ms_e / 1e3), "unit": "rows/s", "h2d_bytes_per_step": int(st_e.h2d_bytes), "d2h_bytes_per_step": int(st_e.d2h_bytes),
               "ms_per_step": ms_e, "rows_per_gpu": int(e2e_rows), "source": "flat CF blocks (b2_cf_block) in pinned host memory",
               "note": "cold: every block crosses PCIe inside the timed region" + part}
        if e2e_sst and "value" in e2e_sst:
            assert e2e_sst.pop("rows_out") == r_e2e
            flat = e2e
            e2e = e2e_sst
            e2e["note"] += part
            e2e["flat"] = flat
        elif e2e_sst:
            e2e["sst_error"] = e2e_sst["error"]
        # warm: the same host-resident regions pinned in the HBM block cache (b2_region_pin, keyed by region id + data version):
        # a repeated request reads HBM, only the result crosses PCIe
        for g in gens:
            L.b2_gen_destroy(g)
        gens = []
        pinned_src = ffi.RegionSource()
        if L.b2_region_pin(device, 1000 + rank, 1, C.byref(host_src.c), C.byref(pinned_src)) == 0:
            class _P:
                c = pinned_src
            for _ in range(2):
                run_dag(ffi, plan, table_range(), _P, ffi.LOC_HOST, args.chunk, stream.cuda_stream, after)
            barrier()
            w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            w0.record(stream)
            kw = args.steps
            for _ in range(kw):
                r_w, st_w = run_dag(ffi, plan, table_range(), _P, ffi.LOC_HOST, args.chunk, stream.cuda_stream, after)
            w1.record(stream)
            barrier()
            ms_w = max_over_ranks(w0.elapsed_time(w1)) / kw
            assert r_w == r_e2e
            e2e["warm"] = {"value": e2e_rows * world / (ms_w / 1e3), "unit": "rows/s", "ms_per_step": ms_w, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": int(st_w.d2h_bytes),
                           "note": "the regions' blocks pinned in the HBM block cache (b2_region_pin): only the result crosses PCIe"}
            L.b2_region_unpin(device, 1000 + rank, 1)
        for p in pinned:
            L.b2_host_free_pinned(p)
    clocks = sampler.stop()
    for g in gens:
        L.b2_gen_destroy(g)
    gens = []

    # ================= sub-records: C2, C5 (same table), C4 =================
    sub = []
    cpu_sub = {}
    if not args.no_sub and not args.only:
        for tname, names in (("c2", ["c2", "c5"]), ("c4", ["c4"])):
            gens, blks2 = gen_blocks(ffi, device, tname, args.sub_rows, 8, first_handle=rank * args.sub_rows)
            src2 = Source(ffi, [b.block for b in blks2], ffi.LOC_DEVICE, device)
            ne2 = sum(b.block.n for b in blks2)
            ib2 = sum(b.key_bytes + b.val_bytes + 8 * b.block.n for b in blks2)
            for nm in names:
                if not args.no_parity:
                    parity[nm] = parity_check(ffi, device, nm, plans.get(nm), src2, rank * args.sub_rows + args.sub_rows // 3,
                                              min(args.parity_rows // 4 if nm == "c2" else args.parity_rows, args.sub_rows // 2), stream.cuda_stream)
                rr = run_workload(nm, src2, args.steps, 3, args.chunk)
                rr["steps"] = args.steps
                if nm in merged:
                    outputs[nm] = merged[nm]
                ob = rr["rows_out"] * 64 + 8 * ((rr["rows_out"] + 63) // 64) * 8 if nm == "c2" else 0
                kb = ib2 if nm != "c5" else sum(b.key_bytes + b.val_bytes + 8 * b.block.n for b in blks2)
                rf = roofline({"c2": "scan_kernel", "c4": "topn_kernel", "c5": "checksum_kernel"}[nm], kb, ob, rr, ne2)
                rf["kernel"] = {"c2": "scan_kernel<PM_SCAN>", "c4": "scan_kernel<PM_TOPN>", "c5": "scan_kernel<PM_CHECKSUM>"}[nm]
                rec = {"workload": TITLES[nm], "rows_per_gpu": args.sub_rows, "value": args.sub_rows * world / (rr["ms_per_step"] / 1e3), "unit": "rows/s" if nm != "c5" else "KVs/s",
                       "ms_per_step": rr["ms_per_step"], "merge_ms": rr["merge_ms"], "rows_out": rr["rows_out"], "gpu_launches": rr["launches"], "roofline": rf}
                if nm == "c5":
                    rec["GBps"] = kb * world / (rr["ms_per_step"] / 1e3) / 1e9
                sub.append((nm, rec))
            for g in gens:
                L.b2_gen_destroy(g)
            gens = []

    # ================= CPU arm (rank 0): oracle on host-generated regions =================
    cpu = None
    if rank == 0 and not args.no_cpu:
        arm = CpuArm(table, args.cpu_sample_rows, cores, cores)
        rate, sec = (arm.rate(plans[head]) if head != "c5" else arm.rate(None))
        arm.close()
        cpu = {"value": rate, "unit": "rows/s", "cores": cores, "kind": "port",
               "sample": f"{cores} region tasks x {args.cpu_sample_rows} rows of the same workload, one task per thread, host-generated regions (restated C++ CPU baseline, not the TiKV Rust binary)"}
        if sub:
            small = max(200_000, args.cpu_sample_rows // 4)
            for tname, names in (("c2", ["c2", "c5"]), ("c4", ["c4"])):
                arm = CpuArm(tname, small, cores, cores)
                for nm in names:
                    cpu_sub[nm], _ = arm.rate(plans.get(nm))
                arm.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    sub_out = []
    for nm, rec in sub:
        if nm in cpu_sub:
            rec["cpu_rows_per_s"] = cpu_sub[nm]
        if nm in parity:
            rec["parity"] = parity[nm]
        sub_out.append(rec)
    merge_desc = {"c3": "all_gather of the per-GPU partial tables (key, count, SUM limbs) over NCCL + exact re-aggregation, inside the timed step",
                  "c4": "all_gather of per-GPU top-N rows + final selection", "c5": "all_gather of partial CRCs + XOR, all_reduce of counters", "c2": None}[head]
    line = {
        "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": TITLES[head], "table": f"{args.rows:.0e} rows per GPU, HBM-resident ({in_bytes / 1e9:.1f} GB of CF_WRITE blocks per GPU)",
                   "rows_per_gpu": args.rows, "cf_write_entries_per_gpu": n_entries, "blocks_per_gpu": len(blks), "groups": n_groups,
                   "selectivity": 0.5, "parallelism": f"region-sharded x{world}; final merge: {merge_desc}",
                   "l2": f"inputs {in_bytes / 1e9:.1f} GB per pass >> 126 MB L2 (no flush needed)", "setup_s": round(time.time() - t_setup, 1)},
        "merge_ms": r["merge_ms"],
        "roofline": roof, "e2e": e2e, "cpu_baseline": cpu, "gpu_launches": r["launches"], "jit_launches": r["jit_launches"], "clocks": clocks,
        "parity": parity.get(head), "sub": sub_out,
    }
    print(json.dumps(line))


if __name__ == "__main__":
    main()
