#!/usr/bin/env python
"""bench.py — Mrows/s of the arrow::compute hot path (filter + take + add) on B200.

One "step" = one pass of the hot path over one synthetic 1e9-row table per GPU
(BASELINE.json configs[1] + configs[2] shapes):
    filter(Int64 col, predicate 10 % set, 5 % nulls)          arrow-select/src/filter.rs:201
      -> take(Int64 col, UInt32 indices = the selected rows)   arrow-select/src/take.rs:89
      -> add(Float64 a, Float64 b), 5 % nulls each side        arrow-arith/src/numeric.rs:36
      -> sum(taken Int64) [+ NCCL all-reduce when --gpus > 1]  arrow-arith/src/aggregate.rs:943
`value` = rows of the table all ranks processed per second of the step (inputs resident in
HBM); `e2e` = the same step through the C ABI starting from pinned HOST buffers with the
H2D / D2H copies inside the timed region. `roofline` is for the dominant kernel (the Float64
add, 24.375 B/row algorithmic) from its own CUDA-event time inside the timed region.

`--impl reference` times the CPU restatement of the reference (oracle/, arrow-rs cannot be
built here: no Rust toolchain) on the host cores, row-partitioned over all of them.

`--dump-outputs DIR` writes what the last timed step returned (filter, take and add outputs with
their validity, the sum) as .npy files of finite float64 / float32 values, so that two builds can
be compared output for output on the same seeded inputs.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True  # the benchmark may run from a read-only tree: no __pycache__ next to the sources

# The contract is ONE JSON line on stdout. Libraries loaded later (NCCL prints "NCCL version ..." when NCCL_DEBUG is set)
# write to file descriptor 1 directly, so the real stdout is set aside and fd 1 is pointed at stderr for everything else.
_REAL_STDOUT = None


def isolate_stdout():
    """Called by main() only (importing this module must not touch the importer's stdout)."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_line(text):
    if _REAL_STDOUT is None:
        print(text, flush=True)
    else:
        os.write(_REAL_STDOUT, (text + "\n").encode())

import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(REPO, "arrow-rs_b200"))
sys.path.insert(0, os.path.join(REPO, "tests"))

import numpy as np  # noqa: E402

SEED_VALUES, SEED_B, SEED_VALID_A, SEED_VALID_B, SEED_PRED = 42, 43, 44, 45, 46  # SURVEY.md §8(d)
SELECTIVITY, NULL_DENSITY = 0.10, 0.05


def so_sha16():
    """Identity of the kernel build: sha256 over the kernel SOURCES (csrc/*.cu, *.cuh, Makefile, the C header), in name order.
    (nvcc's output is not bit-reproducible from one build to the next, so the binary's own hash would call a clean rebuild of
    the same sources a different build.) tools/gpu_profiles.sh records the same value beside every ncu capture."""
    import glob
    import hashlib
    h = hashlib.sha256()
    src = os.path.join(REPO, "arrow-rs_b200", "csrc")
    files = sorted(glob.glob(os.path.join(src, "*.cu")) + glob.glob(os.path.join(src, "*.cuh")) + [os.path.join(src, "Makefile"),
                   os.path.join(REPO, "include", "arrow_cuda.h")])
    try:
        for f in files:
            h.update(os.path.basename(f).encode() + b"\0")
            h.update(open(f, "rb").read())
        return h.hexdigest()[:16]
    except Exception:
        return None


def profiled_traffic(rows):
    """Per-launch dram__bytes_read.sum + dram__bytes_write.sum of the step's kernels from the newest committed
    ncu --set full capture (profiles/rNN_traffic.json: {"so_sha16", "rows", "kernels": {name: bytes}}; the r01 file is a flat
    {name: bytes}). Returns (dict kernel-prefix -> bytes, source file, sha of the .so the capture was taken on) or ({}, None, None)
    for other row counts."""
    pdir = os.path.join(REPO, "profiles")
    best, src, sha = {}, None, None
    for name in sorted(os.listdir(pdir)) if os.path.isdir(pdir) else []:
        if name.endswith("_traffic.json"):
            try:
                d = json.load(open(os.path.join(pdir, name)))
                if "kernels" in d:
                    if int(d.get("rows", 0)) != rows:
                        continue
                    best, src, sha = {k: float(v) for k, v in d["kernels"].items()}, name, d.get("so_sha16")
                elif rows == 1_000_000_000:
                    best, src, sha = {k: float(v) for k, v in d.items() if isinstance(v, (int, float))}, name, None
            except Exception:
                pass
    return best, src, sha


def traffic_of(traffic, prefix):
    for k, v in traffic.items():
        if k.startswith(prefix):
            return v
    return None


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML, 5 ms period)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index):
        self.gpu, self.samples, self.stop_flag, self.thread, self.max_mhz = gpu_index, [], False, None, None
        self.t_mark = 0.0  # only samples taken after mark() are reported (the timed region)

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical GPUs; honour CUDA_VISIBLE_DEVICES if it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu])
                except Exception:
                    idx = self.gpu
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            return

        def loop():
            while not self.stop_flag:
                try:
                    mhz = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                    try:
                        rs = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:
                        rs = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    self.samples.append((float(mhz), int(rs), time.perf_counter()))
                except Exception:
                    pass
                time.sleep(0.005)

        self.thread = threading.Thread(target=loop, daemon=True)
        self.thread.start()

    def mark(self):
        self.t_mark = time.perf_counter()

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=1.0)
        self.samples = [(m, r) for m, r, t in self.samples if t >= self.t_mark]
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        reasons = set()
        for _, rs in self.samples:
            for bit, name in self.REASONS.items():
                if rs & bit:
                    reasons.add(name)
        return {"sm_mhz": float(np.median([m for m, _ in self.samples])), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
class Workload:
    """Device-resident synthetic table for one rank (deterministic, SURVEY.md §8(d))."""

    def __init__(self, ctx, rows, first_row, share=None):
        """share: another Workload of the same first_row with >= rows rows — view its first `rows` rows (same device
        buffers, own counts / indices) instead of generating a table (used to check a prefix against the oracle)."""
        import acu
        from acu import _abi as abi
        self.ctx, self.abi, self.acu, self.n = ctx, abi, acu, rows
        lib, h = ctx.lib, ctx.h
        bb = abi.bitmap_bytes(rows)
        self.bb = bb
        if share is not None:
            for k in ("d_i64", "d_i64_valid", "d_pred", "d_a", "d_b", "d_a_valid", "d_b_valid"):
                setattr(self, k, getattr(share, k))
        else:
            self.d_i64 = ctx.malloc(rows * 8)
            self.d_i64_valid = ctx.malloc(bb)
            self.d_pred = ctx.malloc(bb)
            self.d_a = ctx.malloc(rows * 8)
            self.d_b = ctx.malloc(rows * 8)
            self.d_a_valid = ctx.malloc(bb)
            self.d_b_valid = ctx.malloc(bb)
            ctx.check(lib.acu_generate_values(h, 0, SEED_VALUES, first_row, 0, self.d_i64, rows))
            ctx.check(lib.acu_generate_values(h, 2, SEED_VALUES, first_row, 0, self.d_a, rows))
            ctx.check(lib.acu_generate_values(h, 2, SEED_B, first_row, 0, self.d_b, rows))
            ctx.check(lib.acu_generate_bits(h, SEED_VALID_A, first_row, 1.0 - NULL_DENSITY, self.d_i64_valid, rows))
            ctx.check(lib.acu_generate_bits(h, SEED_VALID_A + 100, first_row, 1.0 - NULL_DENSITY, self.d_a_valid, rows))
            ctx.check(lib.acu_generate_bits(h, SEED_VALID_B, first_row, 1.0 - NULL_DENSITY, self.d_b_valid, rows))
            ctx.check(lib.acu_generate_bits(h, SEED_PRED, first_row, SELECTIVITY, self.d_pred, rows))
        ctx.sync()
        # exact null counts (cached like NullBuffer does) and the output capacity
        self.nc_i64 = rows - self._count(self.d_i64_valid)
        self.nc_a = rows - self._count(self.d_a_valid)
        self.nc_b = rows - self._count(self.d_b_valid)
        self.m = self._count(self.d_pred)
        # outputs (caller-owned, reused every step)
        mb = abi.bitmap_bytes(self.m)
        if share is not None:
            self.out_filter, self.out_take, self.out_add = share.out_filter, share.out_take, share.out_add
        else:
            self.out_filter = self._out(self.m * 8, mb)
            self.out_take = self._out(self.m * 8, mb)
            self.out_add = self._out(rows * 8, bb)
        # take's indices are an INPUT (as for the CPU arm): the selected rows of the predicate, ascending
        # (index distribution A of SURVEY.md §8(d): what a filter -> take pipeline produces)
        self.d_idx = ctx.malloc(self.m * 4)
        self.rebuild_indices()

    def rebuild_indices(self):
        ctx, lib, h = self.ctx, self.ctx.lib, self.ctx.h
        pred = self.arr(self.d_pred, None, self.n, 0)
        plan = C.c_void_p()
        ctx.check(lib.acu_filter_plan_create(h, C.byref(pred), C.byref(plan)))
        ctx.check(lib.acu_filter_plan_indices(h, plan, self.abi.U32, self.d_idx))
        lib.acu_filter_plan_destroy(h, plan)

    def _count(self, d_bits):
        c = C.c_int64(0)
        self.ctx.check(self.ctx.lib.acu_bitmap_count(self.ctx.h, d_bits, 0, None, 0, self.n, C.byref(c)))
        return c.value

    def _out(self, vbytes, bbytes):
        o = self.abi.ArrayOut()
        o.values = self.ctx.malloc(vbytes)
        o.validity = self.ctx.malloc(bbytes)
        return o

    def arr(self, values, validity, n, null_count, voff=0):
        a = self.abi.Array()
        a.values, a.values_offset = values, voff
        a.validity, a.validity_offset = validity, 0
        a.len, a.null_count, a.is_scalar = n, null_count, 0
        return a

    def step(self, timer=None):
        """filter -> take -> add -> sum. Returns (sum_bits, valid_count)."""
        pred = self.arr(self.d_pred, None, self.n, 0)
        col = self.arr(self.d_i64, self.d_i64_valid, self.n, self.nc_i64)
        idx = self.arr(self.d_idx, None, self.m, 0)
        a = self.arr(self.d_a, self.d_a_valid, self.n, self.nc_a)
        b = self.arr(self.d_b, self.d_b_valid, self.n, self.nc_b)
        return hot_path_step(self.ctx, self.abi, pred, col, idx, a, b, self.out_filter, self.out_take, self.out_add, allreduce=True)


def make_arr(abi, values, validity, n, null_count):
    a = abi.Array()
    a.values, a.values_offset = values, 0
    a.validity, a.validity_offset = validity, 0
    a.len, a.null_count, a.is_scalar = n, null_count, 0
    return a


def gpu_checksums(ctx, abi, wl):
    """Run one rank-local step (no all-reduce) and fold its outputs into the same checksums oracle/refbench.cpp computes
    on the CPU (RefBench.CHECK_KEYS): row / null counts and wrapping Int64 sums of every output buffer's bit patterns
    (all slots, validity ignored) — computed on the device with acu_aggregate."""
    lib, h = ctx.lib, ctx.h
    wl.rebuild_indices()  # the e2e arm used d_idx as scratch for its batch-local indices
    pred = wl.arr(wl.d_pred, None, wl.n, 0)
    col = wl.arr(wl.d_i64, wl.d_i64_valid, wl.n, wl.nc_i64)
    idx = wl.arr(wl.d_idx, None, wl.m, 0)
    a = wl.arr(wl.d_a, wl.d_a_valid, wl.n, wl.nc_a)
    b = wl.arr(wl.d_b, wl.d_b_valid, wl.n, wl.nc_b)
    bits, cnt = hot_path_step(ctx, abi, pred, col, idx, a, b, wl.out_filter, wl.out_take, wl.out_add, allreduce=False)

    def wsum(out):
        arr = make_arr(abi, out.values, None, out.len, 0)
        sb, sc = C.c_uint64(0), C.c_int64(0)
        ctx.check(lib.acu_aggregate(h, abi.I64, abi.SUM, C.byref(arr), C.byref(sb), C.byref(sc)))
        return int(sb.value) if sc.value else 0

    nulls = lambda o: int(o.null_count) if o.has_validity else 0  # noqa: E731
    return {"filter_rows": int(wl.out_filter.len), "filter_nulls": nulls(wl.out_filter), "filter_values_wsum": wsum(wl.out_filter),
            "take_nulls": nulls(wl.out_take), "take_values_wsum": wsum(wl.out_take), "add_nulls": nulls(wl.out_add),
            "add_bits_wsum": wsum(wl.out_add), "sum_valid_rows": int(cnt), "sum_bits": int(bits), "valid_rows": int(cnt)}


# --dump-outputs: an output longer than DUMP_ROWS is sampled as DUMP_ROWS // DUMP_BLOCK blocks of DUMP_BLOCK rows, so the
# three step outputs take 3 x 2^20 rows x (8 B values + 4 B validity) = 36 MiB at any table size (a dump stays under 64 MiB).
DUMP_ROWS, DUMP_BLOCK, DUMP_SEED = 1 << 20, 1 << 12, 47


def dump_rows(length):
    """Rows of a `length`-row output that --dump-outputs writes: all of them up to DUMP_ROWS, else whole DUMP_BLOCK-row
    blocks at seeded random offsets (the same rows on every run; block starts are multiples of 8, so every block's
    validity is whole bitmap bytes)."""
    if length <= DUMP_ROWS:
        return np.arange(length)
    blocks = np.random.default_rng(DUMP_SEED).choice(length // DUMP_BLOCK, DUMP_ROWS // DUMP_BLOCK, replace=False)
    return (np.sort(blocks)[:, None] * DUMP_BLOCK + np.arange(DUMP_BLOCK)).ravel()


def dump_output(ctx, out, dtype, out_dir, name):
    """One step output (8-byte values, validity at bit offset 0), rows dump_rows(out.len): <name>.npy = the values as
    float64, 0 in null slots (their contents are unspecified, so builds may differ there); <name>_valid.npy = the
    validity as float32 1 / 0."""
    n = int(out.len)
    rows = dump_rows(n)
    runs = [(0, n)] if len(rows) == n else [(int(s), DUMP_BLOCK) for s in rows[::DUMP_BLOCK]]
    vals, valid = [], []
    for start, count in runs:
        vals.append(ctx.d2h(out.values + start * 8, count * 8, dtype))
        if out.has_validity:
            bits = ctx.d2h(out.validity + start // 8, (count + 7) // 8)
            valid.append(np.unpackbits(bits, bitorder="little")[:count].astype(bool))
    x = np.concatenate(vals).astype(np.float64)
    v = np.concatenate(valid) if out.has_validity else np.ones(len(x), dtype=bool)
    x[~v] = 0.0
    np.save(os.path.join(out_dir, name + ".npy"), x)
    np.save(os.path.join(out_dir, name + "_valid.npy"), v.astype(np.float32))


def dump_outputs(ctx, wl, sum_bits, sum_valid, out_dir):
    """--dump-outputs: what the last timed step returned to its caller (rank 0's shard when --gpus > 1), as .npy files:
    filter / take (Int64 values) and add (Float64) by dump_output; sum = the all-reduced Int64 sum as float64 (0 when no
    taken row is valid: arrow's None, told apart by the last count); counts = [filter rows, filter nulls, take rows,
    take nulls, add rows, add nulls, valid rows of the sum], whole-output figures. Every value written is finite."""
    os.makedirs(out_dir, exist_ok=True)
    outs = (("filter", wl.out_filter, np.int64), ("take", wl.out_take, np.int64), ("add", wl.out_add, np.float64))
    for name, out, dtype in outs:
        dump_output(ctx, out, dtype, out_dir, name)
    total = float(np.array([sum_bits], dtype=np.uint64).view(np.int64)[0]) if sum_valid else 0.0
    np.save(os.path.join(out_dir, "sum.npy"), np.array([total]))
    counts = [x for _, o, _ in outs for x in (o.len, o.null_count if o.has_validity else 0)] + [sum_valid]
    np.save(os.path.join(out_dir, "counts.npy"), np.array(counts, dtype=np.float64))
    print(f"bench.py: last step's outputs written to {out_dir}", file=sys.stderr)


ALLREDUCE_WALL = [0.0, 0]  # host seconds spent inside the final-reduce call (includes waiting for the slowest rank), calls


STREAM_ORDERED = os.environ.get("ACU_BENCH_SYNC", "0") != "1"


def hot_path_step(ctx, abi, pred, col, idx, a, b, out_filter, out_take, out_add, allreduce):
    """One pass of the hot path through the C ABI (device pointers):
    filter(col, pred) -> take(col, idx) -> add(a, b) -> sum(taken) [-> NCCL all-reduce].
    By default the five calls are queued in ONE stream-ordered section (acu_async_begin ... acu_results_fetch: one D2H and
    one synchronisation per step); ACU_BENCH_SYNC=1 uses the synchronous form of the same entry points (one sync each)."""
    lib, h = ctx.lib, ctx.h
    plan = C.c_void_p()
    bits, cnt = C.c_uint64(0), C.c_int64(0)
    if STREAM_ORDERED:
        ctx.check(lib.acu_async_begin(h))
    try:
        ctx.check(lib.acu_filter_plan_create(h, C.byref(pred), C.byref(plan)))
        ctx.check(lib.acu_filter_primitive(h, plan, 8, C.byref(col), C.byref(out_filter)))
        ctx.check(lib.acu_take_primitive(h, 8, C.byref(col), C.byref(idx), abi.U32, 0, C.byref(out_take)))
        ctx.check(lib.acu_arith(h, abi.F64, abi.ADD, C.byref(a), C.byref(b), C.byref(out_add)))
        if STREAM_ORDERED:
            # the taken column's null count is still on the device: -1 makes the reduction count its valid rows itself
            has_v = bool(col.validity) and col.null_count != 0 or bool(idx.validity)
            taken = make_arr(abi, out_take.values, out_take.validity if has_v else None, idx.len, -1 if has_v else 0)
        else:
            taken = make_arr(abi, out_take.values, out_take.validity if out_take.has_validity else None, out_take.len,
                             out_take.null_count if out_take.has_validity else 0)
        # multi-GPU: sum of the shard + NCCL all-reduce of {sum, valid_count} in place on the call's result block — the
        # partial never bounces through the host between the reduction kernel and the collective (world 1: acu_aggregate)
        t0 = time.perf_counter()
        agg = lib.acu_aggregate_allreduce if allreduce else lib.acu_aggregate
        ctx.check(agg(h, abi.I64, abi.SUM, C.byref(taken), C.byref(bits), C.byref(cnt)))
        if STREAM_ORDERED:
            ctx.check(lib.acu_results_fetch(h))
        if allreduce:
            ALLREDUCE_WALL[0] += time.perf_counter() - t0
            ALLREDUCE_WALL[1] += 1
    except BaseException:
        if STREAM_ORDERED and lib.acu_async_active(h):
            lib.acu_results_fetch(h)  # close the section before the plan goes away
        raise
    finally:
        lib.acu_filter_plan_destroy(h, plan)
    return bits.value, cnt.value


class HostStaged:
    """e2e arm: the same step, inputs start in pinned HOST memory, results end there."""

    def __init__(self, wl):
        self.wl = wl
        ctx, n, bb = wl.ctx, wl.n, wl.bb
        self.bufs = {}
        for name, dptr, nbytes in [("i64", wl.d_i64, n * 8), ("i64_valid", wl.d_i64_valid, bb), ("pred", wl.d_pred, bb),
                                   ("a", wl.d_a, n * 8), ("b", wl.d_b, n * 8), ("a_valid", wl.d_a_valid, bb), ("b_valid", wl.d_b_valid, bb)]:
            p = C.c_void_p()
            ctx.check(ctx.lib.acu_host_alloc(ctx.h, nbytes, C.byref(p)))
            ctx.check(ctx.lib.acu_memcpy_d2h(ctx.h, p, dptr, nbytes))  # host copy of the synthetic table
            self.bufs[name] = (p, dptr, nbytes)
        mb = wl.abi.bitmap_bytes(wl.m)
        self.outs = {}
        for name, out, vbytes, bbytes in [("filter", wl.out_filter, wl.m * 8, mb), ("take", wl.out_take, wl.m * 8, mb),
                                          ("add", wl.out_add, n * 8, bb)]:
            pv, pb = C.c_void_p(), C.c_void_p()
            ctx.check(ctx.lib.acu_host_alloc(ctx.h, vbytes, C.byref(pv)))
            ctx.check(ctx.lib.acu_host_alloc(ctx.h, bbytes, C.byref(pb)))
            self.outs[name] = (out, pv, vbytes, pb, bbytes)
        self.h2d_bytes = sum(b[2] for b in self.bufs.values())
        self.d2h_bytes = sum(o[2] + o[4] for o in self.outs.values()) + 16

    def step(self):
        ctx = self.wl.ctx
        lib, h = ctx.lib, ctx.h
        for p, dptr, nbytes in self.bufs.values():
            ctx.check(lib.acu_memcpy_h2d_async(h, dptr, p, nbytes))
        res = self.wl.step()
        for out, pv, vbytes, pb, bbytes in self.outs.values():
            ctx.check(lib.acu_memcpy_d2h_async(h, pv, out.values, vbytes))
            ctx.check(lib.acu_memcpy_d2h_async(h, pb, out.validity, bbytes))
        ctx.sync()
        return res

    def free(self):
        ctx = self.wl.ctx
        for p, _, _ in self.bufs.values():
            ctx.lib.acu_host_free(ctx.h, p)
        for _, pv, _, pb, _ in self.outs.values():
            ctx.lib.acu_host_free(ctx.h, pv)
            ctx.lib.acu_host_free(ctx.h, pb)


class HostPipelined:
    """e2e arm (default): the table starts in pinned HOST memory and is streamed through the C ABI as
    RecordBatches of `batch_rows` rows (BASELINE.json configs[4] streams 2^26-row batches) by `n_workers`
    contexts = streams = host threads on the same GPU, so one batch's H2D, another's kernels and a third's
    D2H overlap (PCIe is full duplex). Every batch does: H2D of its 8 input buffers -> the hot-path step ->
    D2H of filter / take / add outputs."""

    def __init__(self, wl, device, batch_rows=1 << 26, n_workers=3):
        import acu
        self.wl, self.acu, self.abi, self.device = wl, acu, wl.abi, device
        ctx, abi, n = wl.ctx, wl.abi, wl.n
        lib, h = ctx.lib, ctx.h
        self.n_workers = n_workers
        bb = wl.bb
        self.host = {}
        for name, dptr, nbytes in [("i64", wl.d_i64, n * 8), ("i64_valid", wl.d_i64_valid, bb), ("pred", wl.d_pred, bb),
                                   ("a", wl.d_a, n * 8), ("b", wl.d_b, n * 8), ("a_valid", wl.d_a_valid, bb), ("b_valid", wl.d_b_valid, bb)]:
            p = C.c_void_p()
            ctx.check(lib.acu_host_alloc(h, nbytes, C.byref(p)))
            ctx.check(lib.acu_memcpy_d2h(h, p, dptr, nbytes))
            self.host[name] = p.value
        # batches: 64-row aligned ranges; per-batch counts (selected rows, null counts) are metadata
        # a RecordBatch carries (NullBuffer caches null_count)
        self.batches = []
        m_off = 0

        def count(dptr, lo, rows):
            c = C.c_int64(0)
            ctx.check(lib.acu_bitmap_count(h, dptr + lo // 8, 0, None, 0, rows, C.byref(c)))
            return c.value

        p_idx = C.c_void_p()
        ctx.check(lib.acu_host_alloc(h, max(wl.m, 1) * 4, C.byref(p_idx)))
        self.host["idx"] = p_idx.value
        for lo in range(0, n, batch_rows):
            rows = min(batch_rows, n - lo)
            m_b = count(wl.d_pred, lo, rows)
            ncs = tuple(rows - count(d, lo, rows) for d in (wl.d_i64_valid, wl.d_a_valid, wl.d_b_valid))
            # batch-local take indices (an input of the step, like on the CPU arm)
            pred = make_arr(abi, wl.d_pred + lo // 8, None, rows, 0)
            plan = C.c_void_p()
            ctx.check(lib.acu_filter_plan_create(h, C.byref(pred), C.byref(plan)))
            ctx.check(lib.acu_filter_plan_indices(h, plan, abi.U32, wl.d_idx))
            lib.acu_filter_plan_destroy(h, plan)
            ctx.check(lib.acu_memcpy_d2h(h, p_idx.value + m_off * 4, wl.d_idx, m_b * 4))
            self.batches.append({"lo": lo, "rows": rows, "m": m_b, "m_off": m_off, "ncs": ncs})
            m_off += m_b
        self.m_max = max(b["m"] for b in self.batches)
        self.rows_max = max(b["rows"] for b in self.batches)
        # pinned outputs: add at row offsets; filter/take values at selected-row offsets; per-batch validity bitmaps
        self.out = {}
        mb_max = abi.bitmap_bytes(self.m_max)
        for name, nbytes in [("add", n * 8), ("add_valid", bb + 8 * len(self.batches)), ("filter", m_off * 8), ("take", m_off * 8),
                             ("filter_valid", mb_max * len(self.batches)), ("take_valid", mb_max * len(self.batches))]:
            p = C.c_void_p()
            ctx.check(lib.acu_host_alloc(h, max(nbytes, 8), C.byref(p)))
            self.out[name] = p.value
        self.mb_max = mb_max
        self.h2d_bytes = n * 24 + 4 * bb + m_off * 4
        self.d2h_bytes = n * 8 + bb + 2 * (m_off * 8 + abi.bitmap_bytes(m_off))
        self.workers = [self._make_worker() for _ in range(n_workers)]

    def _make_worker(self):
        acu, abi = self.acu, self.abi
        ctx = acu.Context(self.device)
        rb, mb = abi.bitmap_bytes(self.rows_max), abi.bitmap_bytes(self.m_max)
        w = {"ctx": ctx}
        for name, nbytes in [("i64", self.rows_max * 8), ("i64_valid", rb), ("pred", rb), ("a", self.rows_max * 8), ("b", self.rows_max * 8),
                             ("a_valid", rb), ("b_valid", rb), ("idx", self.m_max * 4)]:
            w[name] = ctx.malloc(nbytes)
        for name, vb, bbytes in [("out_filter", self.m_max * 8, mb), ("out_take", self.m_max * 8, mb), ("out_add", self.rows_max * 8, rb)]:
            o = abi.ArrayOut()
            o.values, o.validity = ctx.malloc(vb), ctx.malloc(bbytes)
            w[name] = o
        return w

    def _run_worker(self, k, result):
        abi, w = self.abi, self.workers[k]
        ctx = w["ctx"]
        lib, h = ctx.lib, ctx.h
        total, valid = 0, 0
        try:
            for bi in range(k, len(self.batches), self.n_workers):
                bt = self.batches[bi]
                lo, rows, m, m_off = bt["lo"], bt["rows"], bt["m"], bt["m_off"]
                rb = abi.bitmap_bytes(rows)
                for name, off, nbytes in [("i64", lo * 8, rows * 8), ("i64_valid", lo // 8, rb), ("pred", lo // 8, rb), ("a", lo * 8, rows * 8),
                                          ("b", lo * 8, rows * 8), ("a_valid", lo // 8, rb), ("b_valid", lo // 8, rb), ("idx", m_off * 4, m * 4)]:
                    ctx.check(lib.acu_memcpy_h2d_async(h, w[name], self.host[name] + off, min(nbytes, self._host_left(name, off))))
                pred = make_arr(abi, w["pred"], None, rows, 0)
                col = make_arr(abi, w["i64"], w["i64_valid"], rows, bt["ncs"][0])
                idx = make_arr(abi, w["idx"], None, m, 0)
                a = make_arr(abi, w["a"], w["a_valid"], rows, bt["ncs"][1])
                b = make_arr(abi, w["b"], w["b_valid"], rows, bt["ncs"][2])
                bits, cnt = hot_path_step(ctx, abi, pred, col, idx, a, b, w["out_filter"], w["out_take"], w["out_add"], allreduce=False)
                total = (total + bits) & 0xFFFFFFFFFFFFFFFF  # wrapping i64 sum of the per-batch sums
                valid += cnt
                mb = abi.bitmap_bytes(m)
                for src, dst, nbytes in [(w["out_add"].values, self.out["add"] + lo * 8, rows * 8),
                                         (w["out_add"].validity, self.out["add_valid"] + lo // 8, rb),
                                         (w["out_filter"].values, self.out["filter"] + m_off * 8, m * 8),
                                         (w["out_filter"].validity, self.out["filter_valid"] + bi * self.mb_max, mb),
                                         (w["out_take"].values, self.out["take"] + m_off * 8, m * 8),
                                         (w["out_take"].validity, self.out["take_valid"] + bi * self.mb_max, mb)]:
                    ctx.check(lib.acu_memcpy_d2h_async(h, dst, src, nbytes))
            ctx.sync()
            result[k] = (total, valid)
        except Exception as e:  # surface worker failures in the main thread
            result[k] = e

    def _host_left(self, name, off):
        n, bb = self.wl.n, self.wl.bb
        size = {"i64": n * 8, "a": n * 8, "b": n * 8, "i64_valid": bb, "pred": bb, "a_valid": bb, "b_valid": bb, "idx": max(self.wl.m, 1) * 4}[name]
        return size - off

    def step(self):
        result = [None] * self.n_workers
        ts = [threading.Thread(target=self._run_worker, args=(k, result)) for k in range(self.n_workers)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        for r in result:
            if isinstance(r, Exception):
                raise r
        total = sum(r[0] for r in result) & 0xFFFFFFFFFFFFFFFF
        return total, sum(r[1] for r in result)

    def free(self):
        ctx = self.wl.ctx
        for w in self.workers:
            w["ctx"].close()
        for p in list(self.host.values()) + list(self.out.values()):
            ctx.lib.acu_host_free(ctx.h, p)


def numa_bind(gpu_index):
    """Default for the e2e arm (ACU_BENCH_NUMA=0 disables): run this rank's host threads, and therefore allocate / first-touch
    its pinned buffers, on the CPUs NVML reports as local to the GPU (round 1: 8 unbound ranks reached 0.41 of 8 x the
    one-GPU e2e rate — half the GPUs streamed from the remote socket's memory). Returns the previous affinity (to restore) or
    None when nothing was changed."""
    try:
        before = os.sched_getaffinity(0)
        cpus = set()
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[gpu_index]) if vis else gpu_index
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        except Exception as e:  # fall back to sysfs: the NUMA node of the GPU's PCI device
            NUMA_NOTE[0] = f"nvml affinity unavailable ({type(e).__name__})"
        if not cpus:
            try:
                import pynvml
                bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(gpu_index)).busId
                bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
                bus = bus[4:] if len(bus) > 12 else bus  # 00000000:17:00.0 -> 0000:17:00.0
                node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
                if node >= 0:
                    spec = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
                    for part in spec.split(","):
                        lo, _, hi = part.partition("-")
                        cpus |= set(range(int(lo), int(hi or lo) + 1))
            except Exception as e:
                NUMA_NOTE[0] = (NUMA_NOTE[0] or "") + f"; sysfs numa_node unavailable ({type(e).__name__})"
        cpus &= before
        if not cpus or cpus == before:
            NUMA_NOTE[0] = (NUMA_NOTE[0] or "") + f" no narrower GPU-local CPU set ({len(cpus)} of {len(before)})"
            return None
        os.sched_setaffinity(0, cpus)
        NUMA_NOTE[0] = f"bound to {len(cpus)} GPU-local CPUs"
        return before
    except Exception as e:
        NUMA_NOTE[0] = f"failed ({type(e).__name__}: {e})"
        return None


NUMA_NOTE = [None]


def algorithmic_bytes(n, m):
    """SURVEY.md §8(d): each input read once, each output written once, bitmaps ceil(rows/8)."""
    return {
        "filter": 8 * n + n / 8 + n / 8 + 8 * m + m / 8,
        "take": 4 * m + 8 * m + m / 8 + 8 * m + m / 8,
        "add": 16 * n + 2 * n / 8 + 8 * n + n / 8,
        "sum": 8 * m + m / 8,
        "filter_plan": n / 8,
    }


def run_gpu(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    import acu
    from acu import _abi as abi
    from acu.rendezvous import Group
    ctx = acu.Context(local_rank)
    lib, h = ctx.lib, ctx.h
    group = Group(ctx, rank, local_rank, world)  # NCCL unique-id exchange + acu_comm_init when world > 1
    barrier = group.barrier

    n = args.rows
    wl = Workload(ctx, n, first_row=rank * n)  # weak scaling: every rank owns its own row range
    for _ in range(args.warmup):
        wl.step()
    # the clock sampler (NVML init, a thread) starts BEFORE the barrier: anything rank 0 alone does between the
    # barrier and its timed region would make the other ranks wait for it inside their first all-reduce
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ctx.check(lib.acu_kernel_stats_reset(h))
    ALLREDUCE_WALL[0], ALLREDUCE_WALL[1] = 0.0, 0
    launches0 = ctx.launch_count()
    barrier()
    sampler.mark()
    ms = C.c_float(0)
    ctx.check(lib.acu_timer_start_slot(h, 1))
    for _ in range(args.steps):
        total_bits, total_cnt = wl.step()
    ctx.check(lib.acu_timer_stop_slot(h, 1, C.byref(ms)))
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.launch_count() - launches0
    step_ms = ms.value / args.steps
    step_ms = group.max_over_ranks(step_ms)  # device time, max over ranks
    # per-kernel-class device time inside the timed region
    kstats = {}
    for cls, name in enumerate(abi.KERNEL_CLASS_NAMES):
        tot, cnt = C.c_double(0), C.c_int64(0)
        ctx.check(lib.acu_kernel_stats(h, cls, C.byref(tot), C.byref(cnt)))
        if cnt.value:
            kstats[name] = {"ms_per_step": tot.value / args.steps, "launches_per_step": cnt.value / args.steps,
                            "share_of_step": tot.value / ms.value}
    if args.dump_outputs and rank == 0:  # here: the e2e arm and the oracle check below run the step again
        dump_outputs(ctx, wl, total_bits, total_cnt, args.dump_outputs)

    # ---- e2e: host buffers, copies inside the timed region --------------------------------
    e2e = None
    if not args.no_e2e:
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = 64 << 30
        need = n * 34 + (64 << 20)
        if need * world < avail * 0.6:
            all_cpus = numa_bind(local_rank) if os.environ.get("ACU_BENCH_NUMA", "1") != "0" else None
            hs = HostStaged(wl) if args.e2e_mode == "serial" else HostPipelined(wl, local_rank, args.e2e_batch_rows, args.e2e_workers)
            e2e_check = hs.step()
            barrier()
            # the pipelined arm spans several streams: time it on the host clock around a full device sync
            # (every worker synchronises its stream before step() returns)
            t_begin = time.perf_counter()
            for _ in range(args.e2e_steps):
                e2e_check = hs.step()
            ctx.sync()
            e2e_ms = (time.perf_counter() - t_begin) * 1e3 / args.e2e_steps
            e2e_ms = group.max_over_ranks(e2e_ms)
            e2e = {"value": n * world / (e2e_ms * 1e-3) / 1e6, "unit": "Mrows/s", "h2d_bytes_per_step": hs.h2d_bytes,
                   "d2h_bytes_per_step": hs.d2h_bytes, "ms_per_step": e2e_ms, "steps": args.e2e_steps, "rows_per_gpu": n,
                   "mode": args.e2e_mode, "batch_rows": args.e2e_batch_rows, "streams": args.e2e_workers,
                   "timer": "host perf_counter around steps that end with a stream sync (spans several streams)",
                   "numa_bound_cpus": len(os.sched_getaffinity(0)) if all_cpus else None, "numa_note": NUMA_NOTE[0],
                   "check": {"sum_bits": int(e2e_check[0]), "valid_rows": int(e2e_check[1])}}
            hs.free()
            if all_cpus:
                os.sched_setaffinity(0, all_cpus)  # the CPU baseline below uses every host core again
        else:
            e2e = {"value": None, "unit": "Mrows/s", "skipped": f"host RAM: need {need * world >> 30} GiB pinned, {avail >> 30} GiB available"}

    if rank != 0:
        group.close()
        ctx.close()
        return
    peak, peak_src = peaks()
    ab = algorithmic_bytes(n, wl.m)
    traffic, traffic_src, traffic_sha = profiled_traffic(n)
    sha = so_sha16()
    roof_ops = {}
    # (op, kernel class, ncu kernel-name prefixes whose per-launch DRAM traffic adds up to the op's real traffic)
    for op, cls, kprefix in [("add", "arith", ["k_arith<double"]), ("filter", "filter", ["k_filter_fused<8", "k_filter_values_async<8", "k_compress_bits"]),
                             ("take", "take", ["k_take<8"]), ("sum", "reduce", ["k_reduce<long"]), ("filter_plan", "filter_plan", ["k_plan_mask"])]:
        if cls in kstats:
            t_ms = kstats[cls]["ms_per_step"]  # all kernels of the class
            gbs = ab[op] / (t_ms * 1e-3) / 1e9
            tr = [traffic_of(traffic, p) for p in kprefix]
            tr = sum(x for x in tr if x is not None) if any(x is not None for x in tr) else None
            roof_ops[op] = {"bound": "hbm", "ms": t_ms, "algorithmic_bytes": ab[op], "achieved": gbs, "achieved_gbs": gbs, "peak": peak, "unit": "GB/s",
                            "frac": gbs / peak, "traffic": tr, "frac_real_traffic": (tr / (t_ms * 1e-3) / 1e9 / peak) if tr else None,
                            "mrows_s": (n if op in ("add", "filter", "filter_plan") else wl.m) / (t_ms * 1e-3) / 1e6}
    dom = roof_ops.get("add", {})
    # rank-local outputs of one more step, folded into checksums the CPU arm reproduces (oracle/refbench.cpp)
    gpu_chk = gpu_checksums(ctx, abi, wl)
    line = {
        "metric": "Mrows/sec filter+take+add on 1e9-row Int64/Float64; % HBM roofline",
        "value": n * world / (step_ms * 1e-3) / 1e6,
        "unit": "Mrows/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "i64 (filter/take/sum) + f64 (add)", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rows_per_gpu": n, "parallelism": f"row-range shards x{world}, NCCL all-reduce of the sum only",
                   "l2": "inputs >> L2 (126 MB): no flush needed", "input_residency": "HBM"},
        "selected_rows": wl.m,
        "roofline": {"bound": "hbm", "kernel": "k_arith<double> (Float64 add, fused validity AND + popcount)",
                     "achieved": dom.get("achieved_gbs"), "peak": peak, "unit": "GB/s", "frac": dom.get("frac"),
                     "traffic": dom.get("traffic"), "traffic_source": f"profiles/{traffic_src} (ncu --set full, per launch)" if traffic_src else None,
                     "traffic_so_sha16": traffic_sha, "so_sha16": sha, "sha_of": "kernel sources (csrc/*.cu, *.cuh, Makefile, include/arrow_cuda.h)",
                     "traffic_same_build": (traffic_sha == sha) if traffic_sha else None,
                     "algorithmic_bytes": ab["add"], "peak_source": peak_src, "per_op": roof_ops},
        "roofline_filter": roof_ops.get("filter"), "roofline_take": roof_ops.get("take"),
        "kernels": kstats,
        "gpu_launches": launches,
        "ms_per_step_rank0": ms.value / args.steps,
        "stream_ordered": STREAM_ORDERED,
        "sync_gap_ms_per_step": step_ms - sum(v.get("ms_per_step", 0.0) for v in kstats.values()),
        "sync_gap_note": "step time minus the CUDA-event time of the step's kernel classes = launch gaps + the ONE result fetch"
                         + (" + NCCL all-reduce of {sum, count} in place on the result block + the wait for the slowest rank" if world > 1 else ""),
        "final_reduce_ms_per_step": ((step_ms - sum(v.get("ms_per_step", 0.0) for v in kstats.values())) if STREAM_ORDERED else
                                     (1e3 * ALLREDUCE_WALL[0] / max(ALLREDUCE_WALL[1], 1) - kstats.get("reduce", {}).get("ms_per_step", 0.0))) if world > 1 else 0.0,
        "final_reduce_note": "stream-ordered step: everything of the step that is not kernel time (upper bound of the all-reduce cost); ACU_BENCH_SYNC=1: host wall time of acu_aggregate_allreduce minus the reduction kernel's device time",
        "clocks": clocks,
        "e2e": e2e,
        "check": {"sum_bits": int(total_bits), "valid_rows": int(total_cnt), "rank0_local": gpu_chk},
    }
    if not args.no_cpu:
        base, _, cpu_chk = cpu_reference(args, args.cpu_steps, 2)
        line["cpu_baseline"] = base
        ok, keys, bad = compare_checks(gpu_chk, cpu_chk) if base["same_config"] else (None, [], {})
        if not base["same_config"]:  # the CPU arm ran a prefix of the table: run the GPU on the same prefix and compare that
            sub = Workload(ctx, base["rows"], first_row=0, share=wl)
            ok, keys, bad = compare_checks(gpu_checksums(ctx, abi, sub), cpu_chk)
        line["check_vs_oracle"] = bool(ok)
        line["check"]["vs_oracle"] = {"equal": bool(ok), "rows": base["rows"], "compared": keys, "mismatch": {k: [str(a), str(b)] for k, (a, b) in bad.items()}}
        if not ok:
            emit_line(json.dumps(line))
            raise SystemExit("bench.py: GPU outputs differ from the oracle's: " + json.dumps(line["check"]["vs_oracle"]))
    if not args.no_configs and world == 1:
        line["configs"] = config_subresults(ctx, abi, wl, args, peak, traffic)
    emit_line(json.dumps(line))
    group.close()
    ctx.close()


def config_subresults(ctx, abi, wl, args, peak, traffic):
    """Driver-visible sub-results for BASELINE.json configs #2-#5 (kernel-only CUDA-event time vs algorithmic bytes,
    SURVEY.md §8(d)); the headline step above is configs #2 + #3 combined. Untimed with respect to `value`."""
    sys.path.insert(0, os.path.join(REPO, "tools"))
    import opbench
    lib, h, n = ctx.lib, ctx.h, wl.n
    b = opbench.Bench(ctx, 3)
    b.quiet = True
    A = wl.arr(wl.d_a, wl.d_a_valid, n, wl.nc_a)
    Bv = wl.arr(wl.d_b, wl.d_b_valid, n, wl.nc_b)
    o = wl.out_add
    out = {}
    try:
        # config #3: mul, lt, eq Float64 (add is the headline roofline)
        b.timed("cfg3 mul f64", [abi.K_ARITH], 24.375 * n, n, lambda: ctx.check(lib.acu_arith(h, abi.F64, abi.MUL, C.byref(A), C.byref(Bv), C.byref(o))))
        for name, op in [("cfg3 lt f64", abi.LT), ("cfg3 eq f64", abi.EQ)]:
            b.timed(name, [abi.K_CMP], 16.5 * n, n, lambda op=op: ctx.check(lib.acu_cmp(h, abi.F64, op, C.byref(A), C.byref(Bv), C.byref(o))))
        # config #2, index distribution B: uniform random UInt32 indices, M = 1e8 (or n/10)
        m = min(100_000_000, max(n // 10, 1))
        col = wl.arr(wl.d_i64, wl.d_i64_valid, n, wl.nc_i64)
        drand = b.gen(3, 47, m, 4, param=n)
        ix = b.arr(drand, None, m, 0)
        ot = b.out(m * 8, m)
        b.timed("cfg2 take i64 uniform random", [abi.K_TAKE], 20.25 * m, m,
                lambda: ctx.check(lib.acu_take_primitive(h, 8, C.byref(col), C.byref(ix), abi.U32, 0, C.byref(ot))), note="index distribution B")
        ctx.free(drand)
        # config #4: cast Int64 -> Float64 and Dictionary<Int32,Utf8> -> Utf8, 1e8 rows
        ns = min(100_000_000, n)
        Is = b.arr(wl.d_i64, wl.d_i64_valid, ns, -1)
        b.timed("cfg4 cast i64->f64", [abi.K_CAST], 16.25 * ns, ns, lambda: ctx.check(lib.acu_cast_numeric(h, abi.I64, abi.F64, 1, C.byref(Is), C.byref(ot))))
        ctx._free_out(ot)
        D = 4096
        rng = np.random.default_rng(1)
        lens = rng.integers(4, 13, D)
        offs = np.zeros(D + 1, dtype=np.int32)
        offs[1:] = np.cumsum(lens)
        data = rng.integers(97, 123, int(offs[-1]) + 16).astype(np.uint8)
        d_off, d_data = ctx.malloc(offs.nbytes + 64), ctx.malloc(data.nbytes + 64)
        ctx.h2d(d_off, offs)
        ctx.h2d(d_data, data)
        dkeys = b.gen(4, 48, ns, 4, param=D)
        kv, nkv = b.bits(49, 0.95, ns)
        keys = b.arr(dkeys, kv, ns, ns - nkv)
        dict_nulls = b.arr(None, None, D, 0)
        d_out_off, d_out_data = ctx.malloc((ns + 1) * 4 + 64), ctx.malloc(ns * 13 + 64)
        on = abi.ArrayOut()
        on.validity = ctx.malloc(abi.bitmap_bytes(ns) + 64)
        total = C.c_int64(0)
        b.timed("cfg4 cast dict<i32,utf8>->utf8", [abi.K_TAKE, abi.K_BYTES], 4 * ns + ns / 8 + 4 * (D + 1) + float(offs[-1]) + 4 * (ns + 1) + 0.95 * ns * 8 + ns / 8, ns,
                lambda: ctx.check(lib.acu_take_bytes(h, 4, d_off, d_data, C.byref(dict_nulls), C.byref(keys), abi.I32, 0, d_out_off, d_out_data, ns * 13, C.byref(total), C.byref(on))),
                note="D=4096, lengths 4..12, 5 % null keys")
        for p in (d_off, d_data, dkeys, kv, d_out_off, d_out_data, on.validity):
            ctx.free(p)
        for r in b.rows:
            key = r["op"].split(" ", 1)
            out.setdefault(key[0], {})[key[1]] = {"rows": r["rows"], "kernel_ms": r["kernel_ms"], "call_ms": r["call_ms"], "algorithmic_bytes": r["algorithmic_bytes"],
                                                  "achieved_gbs": r["achieved_gbs"], "frac": r["frac_of_measured_peak"], "mrows_s": r["mrows_s"], "note": r["note"],
                                                  "traffic": None}
    except Exception as e:  # sub-results never take the headline down
        out["error"] = repr(e)[:300]
    # config #5: RecordBatch pipeline (tools/recordbatch_bench.py body), one GPU's share: 15 x 2^26-row 8-column batches
    try:
        if n >= 1_000_000_000:
            import recordbatch_bench as rbb
            tb = rbb.Table(ctx, abi, 0, 15, 1 << 26, SELECTIVITY, NULL_DENSITY)
            import acu
            # extra lanes (ctx + stream + host thread each): the host gaps of one lane overlap the kernels of the others
            extra = [acu.Context(ctx.device) for _ in range(max(int(os.environ.get("ACU_RB_STREAMS", "3")), 1) - 1)]
            for c in extra:
                tb.add_lane(c)
            lanes = [ctx] + extra
            for _ in range(2):
                tb.step()
            for c in lanes:
                c.sync()
                c.check(lib.acu_kernel_stats_reset(c.h))
            reps = 3
            t0 = time.perf_counter()
            for _ in range(reps):
                sums, cnts, alg = tb.step()
            for c in lanes:
                c.sync()
            step_ms = (time.perf_counter() - t0) * 1e3 / reps  # host clock: every stream idle at both ends
            ksum, kcls = 0.0, {}
            for cls in range(len(abi.KERNEL_CLASS_NAMES)):
                ms_c, n_c = 0.0, 0
                for c in lanes:
                    tot, cnt = C.c_double(0), C.c_int64(0)
                    c.check(lib.acu_kernel_stats(c.h, cls, C.byref(tot), C.byref(cnt)))
                    ms_c += tot.value / reps
                    n_c += cnt.value
                ksum += ms_c
                if n_c:
                    kcls[abi.KERNEL_CLASS_NAMES[cls]] = round(ms_c, 3)
            for c in extra:
                c.close()
            rows = 15 * (1 << 26)
            out["cfg5"] = {"filter_record_batch -> take_record_batch -> 6 sums": {
                "rows": rows, "ms_per_step": step_ms, "kernel_ms": ksum, "kernel_ms_by_class": kcls, "algorithmic_bytes": alg, "achieved_gbs": alg / (step_ms * 1e-3) / 1e9,
                "frac": alg / (step_ms * 1e-3) / 1e9 / peak, "mrows_s": rows / (step_ms * 1e-3) / 1e6, "traffic": None,
                "streams": len(lanes), "timer": "host clock around steps bracketed by a synchronisation of every stream",
                "note": "one GPU's share of BASELINE configs[4]: 15 batches of 2^26 rows x {3 Int64, 3 Float64, 2 Utf8}, every batch resident in HBM; "
                        "frac is whole-pipeline algorithmic bytes / step time (host launch gaps included)"}}
    except Exception as e:
        out["cfg5_error"] = repr(e)[:300]
    return out


# ------------------------------------------------------------------------------------------
# CPU reference arm (oracle port of the arrow-rs algorithms; test infrastructure used as the
# timed CPU baseline only). The harness is native (oracle/refbench.cpp): a persistent pool of
# pinned threads, every thread generating / first-touching its own row range, the timer inside C
# around the barriers. No Python, thread creation or allocation in the timed region.
# ------------------------------------------------------------------------------------------
SEEDS7 = (SEED_VALUES, SEED_VALUES, SEED_B, SEED_VALID_A, SEED_VALID_A + 100, SEED_VALID_B, SEED_PRED)
REF_BYTES_PER_ROW = 36.0  # inputs 24 + bitmaps 0.5 + indices 0.4 + outputs 9.6 + slack


def host_available_bytes():
    try:
        import psutil
        return int(psutil.virtual_memory().available)
    except Exception:
        return 64 << 30


def reference_rows(args):
    """Rows the CPU arm runs per step: the full per-GPU table (same config) when the host has the RAM for it
    (36 B/row), else the largest 64-row multiple that fits in 60 % of the available RAM (stated in the line)."""
    if args.cpu_rows:
        return min(args.cpu_rows, args.rows), "--cpu-rows"
    fit = int(host_available_bytes() * 0.6 / REF_BYTES_PER_ROW) // 64 * 64
    if fit >= args.rows:
        return args.rows, None
    return max(fit, 64), f"host RAM: {host_available_bytes() >> 30} GiB available, {int(args.rows * REF_BYTES_PER_ROW) >> 30} GiB needed for the full table"


def pyarrow_secondary(orc, n):
    """Labelled secondary figure: the same step through pyarrow (Arrow C++ — a different implementation of the same
    format, not arrow-rs and not the oracle), one call per op over an n-row sample."""
    try:
        import pyarrow as pa
        import pyarrow.compute as pc
        from acu import unpack_bits
        data = {"i64": orc.generate_values(0, SEED_VALUES, 0, 0, n, np.int64), "i64_valid": orc.generate_bits(SEED_VALID_A, 0, 1 - NULL_DENSITY, n),
                "pred": orc.generate_bits(SEED_PRED, 0, SELECTIVITY, n), "a": orc.generate_values(2, SEED_VALUES, 0, 0, n, np.float64),
                "b": orc.generate_values(2, SEED_B, 0, 0, n, np.float64), "a_valid": orc.generate_bits(SEED_VALID_A + 100, 0, 1 - NULL_DENSITY, n),
                "b_valid": orc.generate_bits(SEED_VALID_B, 0, 1 - NULL_DENSITY, n)}

        def pa_prim(t, values, valid):
            return pa.Array.from_buffers(t, n, [pa.py_buffer(valid), pa.py_buffer(values)], null_count=-1)

        p_col = pa_prim(pa.int64(), data["i64"], data["i64_valid"])
        p_a, p_b = pa_prim(pa.float64(), data["a"], data["a_valid"]), pa_prim(pa.float64(), data["b"], data["b_valid"])
        p_pred = pa.Array.from_buffers(pa.bool_(), n, [None, pa.py_buffer(data["pred"])], null_count=0)
        p_idx = pa.array(np.nonzero(unpack_bits(data["pred"], 0, n))[0].astype(np.uint32), type=pa.uint32())

        def pa_step():
            t0 = time.perf_counter()
            pc.filter(p_col, p_pred, null_selection_behavior="drop")
            tk = pc.take(p_col, p_idx, boundscheck=False)
            pc.add(p_a, p_b)
            pc.sum(tk)
            return time.perf_counter() - t0

        pa_step()
        return {"impl": f"pyarrow {pa.__version__} (Arrow C++; labelled secondary baseline, not arrow-rs)", "value": n / min(pa_step() for _ in range(2)) / 1e6,
                "unit": "Mrows/s", "rows": n, "threads": "one call per op over the whole sample (pyarrow's own kernel threading)"}
    except Exception as e:  # pyarrow is optional
        return {"impl": "pyarrow", "skipped": repr(e)[:120]}


def cpu_pin_order():
    """Allowed CPUs ordered for pinning: one hyperthread of every physical core first, alternating between the NUMA nodes /
    packages, then the sibling hyperthreads in the same order — so that ANY thread count spreads over all memory controllers."""
    allowed = sorted(os.sched_getaffinity(0))
    try:
        info = {}
        for c in allowed:
            base = f"/sys/devices/system/cpu/cpu{c}/topology/"
            pkg = int(open(base + "physical_package_id").read())
            sib = open(base + "thread_siblings_list").read().strip().replace("-", ",").split(",")
            info[c] = (pkg, min(int(x) for x in sib))
        primaries = [c for c in allowed if info[c][1] == c or info[c][1] not in allowed]
        seconds = [c for c in allowed if c not in primaries]

        def interleave(cs):
            by_pkg = {}
            for c in cs:
                by_pkg.setdefault(info[c][0], []).append(c)
            out, lists = [], [by_pkg[k] for k in sorted(by_pkg)]
            for i in range(max((len(x) for x in lists), default=0)):
                out += [x[i] for x in lists if i < len(x)]
            return out
        return interleave(primaries) + interleave(seconds)
    except Exception:
        return allowed


def cpu_reference(args, steps, warmup, secondary=True, one_thread=True):
    """Run the native reference harness: `warmup` untimed + `steps` timed passes of the hot-path step over
    reference_rows(args) rows. Returns (cpu_baseline dict, per-step seconds, checksums of the outputs)."""
    from oracle import Oracle, RefBench
    orc = Oracle()
    n, why = reference_rows(args)
    os.environ.setdefault("ORC_BENCH_CPU_ORDER", ",".join(str(c) for c in cpu_pin_order()))
    calib = None
    threads_req = args.cpu_threads or 0
    if not threads_req and n >= 200_000_000:
        # "all the host threads it can use" is not always the fastest way to run a memory-bound step: on the round-2 GPU box a
        # plain Float64 add reaches 132 GB/s on 16 threads, 118 on 64 and 64 on all 128 hyperthreads (tools/experiments/membw.c).
        # The arm therefore measures a 1e8-row sample at a few thread counts and runs the full table with the best one.
        ncpu = len(os.sched_getaffinity(0))
        calib = {}
        for t in sorted({ncpu, max(ncpu // 2, 1), max(ncpu // 4, 1), max(ncpu // 8, 1)}):
            with RefBench(100_000_000, SEEDS7, SELECTIVITY, NULL_DENSITY, threads=t, oracle=orc) as rbc:
                rbc.step()
                calib[t] = 100_000_000 / min(rbc.step()[0] for _ in range(2)) / 1e6
        threads_req = max(calib, key=calib.get)
    with RefBench(n, SEEDS7, SELECTIVITY, NULL_DENSITY, threads=threads_req, oracle=orc) as rb:
        for _ in range(max(warmup, 1)):
            rb.step()
        runs = [rb.step() for _ in range(max(steps, 1))]
        secs = [r[0] for r in runs]
        chk = rb.check()
        chk["sum_bits"], chk["valid_rows"] = int(runs[-1][1]), int(runs[-1][2])
        threads, gen_s = rb.threads, rb.generate_seconds
    med, best = float(np.median(secs)), float(min(secs))
    base = {"value": n / med / 1e6, "unit": "Mrows/s", "cores": threads, "kind": "port",
            "sample": (f"{n} rows = " + ("the full per-GPU table (same config)" if n == args.rows else f"first {n} rows of the table [{why}]") +
                       f"; same step (filter+take+add+sum) row-partitioned over {threads} pinned native threads (oracle/refbench.cpp: each thread first-touches "
                       "its own range, outputs pre-allocated, timer inside C); oracle/ C++ restatement of arrow-rs (no Rust toolchain here)"),
            "rows": n, "same_config": n == args.rows, "host_cores": os.cpu_count() or 1, "seconds_median": med, "seconds_min": best,
            "value_best": n / best / 1e6, "spread": (max(secs) - best) / med if med else None, "timed_steps": len(secs), "generate_seconds": gen_s,
            "thread_calibration_mrows_s": {str(k): round(v, 1) for k, v in calib.items()} if calib else None,
            "pinning": "physical cores first, alternating NUMA nodes (ORC_BENCH_CPU_ORDER)"}
    if one_thread and threads > 1:  # arrow-rs kernels themselves are single-threaded: ONE call per op over a 1e8-row sample
        n1 = min(n, 100_000_000)
        with RefBench(n1, SEEDS7, SELECTIVITY, NULL_DENSITY, threads=1, oracle=orc) as rb1:
            rb1.step()
            base["value_1_thread"] = n1 / min(rb1.step()[0] for _ in range(2)) / 1e6
            base["rows_1_thread"] = n1
    if secondary:
        base["secondary"] = pyarrow_secondary(orc, min(n, 100_000_000))
    return base, secs, chk


def compare_checks(gpu_chk, cpu_chk):
    """True when every checksum both sides report is identical (bit-exact integer quantities)."""
    keys = [k for k in cpu_chk if k in gpu_chk]
    bad = {k: (gpu_chk[k], cpu_chk[k]) for k in keys if int(gpu_chk[k]) != int(cpu_chk[k])}
    return (len(keys) > 0 and not bad), keys, bad


WORKLOAD = "filter(Int64, 10% selected, 5% nulls) -> take(UInt32 monotone indices, M=count) -> add(Float64, 5% nulls x2) -> sum(Int64)"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # other ranks exit 0 without work
    # the reference arm never touches the GPU
    base, secs, chk = cpu_reference(args, args.steps, args.warmup, secondary=False, one_thread=True)
    n = base["rows"]
    sec = base["seconds_median"]
    value = n / sec / 1e6
    line = {
        "impl": "reference",
        "metric": "Mrows/sec filter+take+add on 1e9-row Int64/Float64; % HBM roofline",
        "value": value, "unit": "Mrows/s", "n_gpus": args.gpus, "steps": len(secs), "warmup": args.warmup,
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "i64 (filter/take/sum) + f64 (add)", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rows_per_gpu": args.rows, "parallelism": f"row-range shards x{args.gpus}, NCCL all-reduce of the sum only",
                   "l2": "inputs >> L2 (126 MB): no flush needed", "input_residency": "HBM"},
        "rows_per_step": n, "same_config": base["same_config"],
        "timing": {"seconds": secs, "median": sec, "min": base["seconds_min"], "spread": base["spread"]},
        "cpu_baseline": base,
        "check": chk,
        "e2e": {"value": value, "unit": "Mrows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit_line(json.dumps(line))


def main():
    isolate_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=1_000_000_000, help="rows per GPU")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-mode", default="pipelined", choices=["pipelined", "serial"])
    ap.add_argument("--e2e-batch-rows", type=int, default=1 << 26)
    ap.add_argument("--e2e-workers", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows of the CPU arm's step (0 = the full table when host RAM allows)")
    ap.add_argument("--cpu-steps", type=int, default=5, help="timed CPU steps of the cpu_baseline leg of the GPU arm")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config sub-results (configs #2-#5)")
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as .npy files to DIR (GPU arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; the reference arm keeps its outputs inside oracle/refbench.cpp")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
