"""Reductions checked exactly: sum / min / max (k_reduce, csrc/reduce.cu) and sum_checked (csrc/sumchecked.cu).

- Float sums on inputs whose sum is exact in every association order (every value k·2^e, Σ|k| <= 2^p) must equal
  Σx bit for bit, at any size and whatever order the kernel adds in: a dropped, duplicated or misplaced row fails.
- Every dtype past one full grid (N_WAVE rows: most warps run two or more super-group iterations, with a ragged
  tail), the batched launch with short columns sharing a long column's grid, the deferred valid count of a
  stream-ordered section, and one 1-byte column past 2^32 rows. Inputs are generated on the device
  (acu_generate_*); the host twin (oracle.generate_*) is built in chunks, so host memory stays bounded.
- sum_checked over more than 1024 chunks of 4096 rows, so that each scan thread walks several chunks and the
  trailing threads are idle, against the oracle's sequential checked fold.
"""
import ctypes as C

import numpy as np
import pytest

import acu
from acu import _abi as abi
from acu import HostArray

from test_gpu_parity import (EXACT_KINDS, FLOAT_DTYPES, INT_DTYPES, SIZES, exact_float_array, expect_same_error,
                             same_float)

pytestmark = pytest.mark.gpu

ALL_DTYPES = INT_DTYPES + FLOAT_DTYPES
UNSIGNED = {1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}
SIGNED = {1: np.int8, 2: np.int16, 4: np.int32, 8: np.int64}
OPS = (abi.SUM, abi.MIN, abi.MAX)
CHUNK = 1 << 24  # rows per host-twin chunk


@pytest.fixture(scope="module")
def sm_count(gpu):
    return gpu.lib.acu_device_sm_count(gpu.h)


@pytest.fixture(scope="module")
def n_wave(sm_count):
    """Past the reduction's grid cap (8 CTAs of 8 warps per SM, 2048 rows per warp iteration) for any occupancy:
    most warps take two or more super-groups, and the last one is ragged."""
    return 2 * sm_count * (1 << 20) + 12345


# ---- A. float sum, bit-exact on order-independent inputs ------------------------------------------------------
@pytest.mark.parametrize("dtype", FLOAT_DTYPES)
@pytest.mark.parametrize("kind", EXACT_KINDS)
def test_float_sum_exact(gpu, dtype, kind):
    rng = np.random.default_rng(11000 + 10 * dtype + EXACT_KINDS.index(kind))
    for n in SIZES:
        for null_p, off in [(None, 0), (0.1, 1), (0.5, 3), (None, 2), (1.0, 0)]:
            a, exp = exact_float_array(rng, dtype, n, kind, null_p, off)
            got = gpu.sum(a)
            assert same_float(got, exp, dtype), f"sum {kind} dtype={dtype} n={n} nulls={null_p} off={off}: {got!r} != {exp!r}"


@pytest.mark.parametrize("dtype", FLOAT_DTYPES)
def test_float_sum_zero_is_positive_zero(gpu, dtype):
    """Σx = 0 gives +0.0 (T::ZERO + ...), including a column of -0.0 only."""
    npdt = acu.NP_DTYPES[dtype]
    rng = np.random.default_rng(12000 + dtype)
    for n in (1, 2, 100, 4097, 70001):
        half = rng.integers(-50, 50, max(n // 2, 1)).astype(npdt)
        for vals in (np.full(n, -0.0, dtype=npdt), rng.permutation(np.concatenate([half, -half]))):
            # and the same valid rows with a null slot holding 1.0 inserted at a random place
            at = int(rng.integers(0, len(vals) + 1))
            mask = np.insert(np.ones(len(vals), dtype=bool), at, False)
            for a in (HostArray.from_numpy(dtype, vals), HostArray.from_numpy(dtype, np.insert(vals, at, 1.0), mask)):
                got = gpu.sum(a)
                assert same_float(got, 0.0, dtype), f"n={n}: {got!r} is not +0.0"


@pytest.mark.parametrize("dtype", FLOAT_DTYPES)
def test_float_sum_special_values(gpu, dtype):
    """IEEE outcomes that do not depend on the association order."""
    npdt = acu.NP_DTYPES[dtype]
    rng = np.random.default_rng(13000 + dtype)
    for n in (1, 65, 4097, 70001):
        base = rng.integers(-100, 100, n).astype(npdt)  # Σ|x| < 2^24: the finite sums below are exact even in f32
        pos = int(rng.integers(0, n))
        with_inf = base.copy()
        with_inf[pos] = np.inf
        assert gpu.sum(HostArray.from_numpy(dtype, with_inf)) == np.inf, f"finite + inf n={n}"
        neg = base.copy()
        neg[pos] = -np.inf
        assert gpu.sum(HostArray.from_numpy(dtype, neg)) == -np.inf, f"finite - inf n={n}"
        if n > 1:
            both = with_inf.copy()
            both[(pos + n // 2 + 1) % n] = -np.inf
            assert np.isnan(gpu.sum(HostArray.from_numpy(dtype, both))), f"+inf + -inf n={n}"
        nan = base.copy()
        nan[pos] = np.nan
        assert np.isnan(gpu.sum(HostArray.from_numpy(dtype, nan))), f"valid NaN n={n}"
        # the same specials under a null: the validity decides, the result is the exact finite sum
        mask = np.ones(n, dtype=bool)
        mask[pos] = False
        exp = float(np.array(int(base.astype(np.int64)[mask].sum()), dtype=npdt)) if n > 1 else None
        for v in (with_inf, neg, nan):
            assert same_float(gpu.sum(HostArray.from_numpy(dtype, v, mask)), exp, dtype), f"special under a null n={n}"
        assert gpu.sum(HostArray.from_numpy(dtype, nan, np.zeros(n, dtype=bool))) is None, f"all null n={n}"


# ---- C. every reduction past one full grid ----------------------------------------------------------------------
def make_arr(values, n, validity=None, voff=0, null_count=0, scalar=False):
    a = abi.Array()
    a.values, a.values_offset, a.validity, a.validity_offset = values, 0, validity, voff
    a.len, a.null_count, a.is_scalar = n, null_count, 1 if scalar else 0
    return a


def dev_raw(gpu, seed, nbytes):
    """kind-0 generator output: little-endian splitmix64 words, so row r of a `size`-byte column is bytes
    [r·size, (r+1)·size) of the word stream."""
    words = -(-nbytes // 8)
    d = gpu.malloc(words * 8 + 64)
    gpu.check(gpu.lib.acu_generate_values(gpu.h, 0, seed, 0, 0, d, words))
    return d


def dev_bits(gpu, seed, p, nbits):
    d = gpu.malloc(abi.bitmap_bytes(nbits) + 64)
    gpu.check(gpu.lib.acu_generate_bits(gpu.h, seed, 0, p, d, nbits))
    return d


def host_mask(oracle, vseed, p, first_bit, m):
    return acu.unpack_bits(oracle.generate_bits(vseed, first_bit, p, m), 0, m)


def order_keys(u, dtype):
    """Native bit patterns (unsigned view) -> keys whose integer order is the reduction's order (totalOrder for floats)."""
    size = abi.DTYPE_SIZE[dtype]
    if dtype in FLOAT_DTYPES:
        k = u.view(SIGNED[size])
        return k ^ ((k >> (8 * size - 1)) & np.iinfo(SIGNED[size]).max)
    return u.view(SIGNED[size]) if dtype in (abi.I8, abi.I16, abi.I32, abi.I64) else u


def key_bits(key, dtype):
    size = abi.DTYPE_SIZE[dtype]
    k = np.array([key], dtype=SIGNED[size] if (dtype in FLOAT_DTYPES or dtype <= abi.I64) else UNSIGNED[size])
    if dtype in FLOAT_DTYPES:
        k = k ^ ((k >> (8 * size - 1)) & np.iinfo(SIGNED[size]).max)
    return int(k.view(UNSIGNED[size])[0])


def twin_stats(oracle, dtype, seed, start, n, vseed=None, p=None, voff=0):
    """Host twin of rows [start, start + n) of a kind-0 column of `dtype` whose validity bit for row r is generated bit
    voff + r (vseed, p) -> {SUM: wrapping-sum bits, MIN / MAX: bits of the extreme, "count": valid rows}."""
    size = abi.DTYPE_SIZE[dtype]
    assert (start * size) % 8 == 0
    total, count, lo, hi = 0, 0, None, None
    for s in range(start, start + n, CHUNK):
        m = min(CHUNK, start + n - s)
        u = oracle.generate_values(0, seed, s * size // 8, 0, -(-m * size // 8), np.uint64).view(UNSIGNED[size])[:m]
        if vseed is not None:
            u = u[host_mask(oracle, vseed, p, voff + s, m)]
        if not u.size:
            continue
        count += u.size
        total += int(u.astype(np.uint64).sum(dtype=np.uint64))  # an 8-byte sum wraps mod 2^64: all that is kept
        keys = order_keys(u, dtype)
        lo = keys.min() if lo is None else min(lo, keys.min())
        hi = keys.max() if hi is None else max(hi, keys.max())
    if count == 0:
        return {"count": 0}
    return {abi.SUM: total % (1 << (8 * size)), abi.MIN: key_bits(lo, dtype), abi.MAX: key_bits(hi, dtype), "count": count}


def aggregate_bits(gpu, dtype, op, arr):
    bits, cnt = C.c_uint64(0), C.c_int64(0)
    gpu.check(gpu.lib.acu_aggregate(gpu.h, dtype, op, C.byref(arr), C.byref(bits), C.byref(cnt)))
    return bits.value & ((1 << (8 * abi.DTYPE_SIZE[dtype])) - 1), cnt.value


def aggregate_in_section(gpu, dtype, arr, ops=OPS):
    """sum / min / max queued in one stream-ordered section on `arr` (null_count = -1: the kernel counts)."""
    outs = [(C.c_uint64(0), C.c_int64(0)) for _ in ops]
    gpu.async_begin()
    try:
        for op, (bits, cnt) in zip(ops, outs):
            gpu.check(gpu.lib.acu_aggregate(gpu.h, dtype, op, C.byref(arr), C.byref(bits), C.byref(cnt)))
    finally:
        gpu.results_fetch()
    mask = (1 << (8 * abi.DTYPE_SIZE[dtype])) - 1
    return [(b.value & mask, c.value) for b, c in outs]


VOFF = 5  # bit offset of every generated validity


@pytest.mark.parametrize("dtype", ALL_DTYPES)
def test_reduce_past_one_grid(gpu, oracle, n_wave, dtype):
    """sum / min / max over N_WAVE rows of raw bit patterns (floats: every pattern, NaNs of both signs included, for
    min / max), without validity and with a validity at a nonzero bit offset, synchronously and in a section with
    the valid count left to the kernel."""
    n, size = n_wave, abi.DTYPE_SIZE[dtype]
    seed, vseed, p = 600 + dtype, 700 + dtype, 0.9
    d_vals, d_valid = dev_raw(gpu, seed, n * size), dev_bits(gpu, vseed, p, n + VOFF)
    try:
        ops = OPS if dtype not in FLOAT_DTYPES else (abi.MIN, abi.MAX)
        exp = twin_stats(oracle, dtype, seed, 0, n)
        for op in ops:
            assert aggregate_bits(gpu, dtype, op, make_arr(d_vals, n)) == (exp[op], n), f"op {op} without validity"
        exp = twin_stats(oracle, dtype, seed, 0, n, vseed, p, VOFF)
        nc = n - exp["count"]
        for op in ops:
            assert aggregate_bits(gpu, dtype, op, make_arr(d_vals, n, d_valid, VOFF, nc)) == (exp[op], exp["count"]), f"op {op}"
        got = aggregate_in_section(gpu, dtype, make_arr(d_vals, n, d_valid, VOFF, -1), ops)
        assert got == [(exp[op], exp["count"]) for op in ops], "deferred valid count"
    finally:
        gpu.free(d_vals)
        gpu.free(d_valid)


def build_exact_float_column(gpu, dtype, n, kseed, param, d_mask, voff, garbage_seed):
    """Device column of n rows: row r = (k_r - param/2) as `dtype` where mask bit voff + r is set, with k_r the kind-4
    integer in [0, param) (acu_arith subtracts the scalar, acu_cast converts: both exact at these magnitudes), and
    otherwise raw kind-0 bit patterns (garbage_seed) or, with garbage_seed None, 0.0. Built in chunks by acu_zip."""
    size, lib, h = abi.DTYPE_SIZE[dtype], gpu.lib, gpu.h
    step = 1 << 26
    d_out = gpu.malloc(n * size + 64)
    d_k, d_half = gpu.malloc(step * 4 + 64), gpu.malloc(64)
    gpu.h2d(d_half, np.array([param // 2], dtype=np.int32))
    d_zero = gpu.malloc(64)
    gpu.h2d(d_zero, np.zeros(1, dtype=acu.NP_DTYPES[dtype]))
    o_sub, o_cast, o_zip = gpu.alloc_out(step * 4, step), gpu.alloc_out(step * size, step), abi.ArrayOut()
    o_zip.validity = gpu.malloc(abi.bitmap_bytes(step) + 8)
    d_junk = gpu.malloc(step * size + 64) if garbage_seed is not None else None
    try:
        for s in range(0, n, step):
            m = min(step, n - s)
            gpu.check(lib.acu_generate_values(h, 4, kseed, s, param, d_k, m))
            k, half = make_arr(d_k, m), make_arr(d_half, 1, scalar=True)
            gpu.check(lib.acu_arith(h, abi.I32, abi.SUB_WRAPPING, C.byref(k), C.byref(half), C.byref(o_sub)))
            ks = make_arr(o_sub.values, m)
            gpu.check(lib.acu_cast_numeric(h, abi.I32, dtype, 1, C.byref(ks), C.byref(o_cast)))
            if d_junk is not None:
                gpu.check(lib.acu_generate_values(h, 0, garbage_seed, s * size // 8, 0, d_junk, -(-m * size // 8)))
                falsy = make_arr(d_junk, m)
            else:
                falsy = make_arr(d_zero, 1, scalar=True)
            mask = make_arr(d_mask, m)
            mask.values_offset = voff + s
            truthy = make_arr(o_cast.values, m)
            o_zip.values = d_out + s * size
            gpu.check(lib.acu_zip(h, size, C.byref(mask), C.byref(truthy), C.byref(falsy), C.byref(o_zip)))
        gpu.sync()
    finally:
        for o in (o_sub, o_cast):
            gpu._free_out(o)
        for ptr in (o_zip.validity, d_k, d_half, d_zero, d_junk):
            gpu.free(ptr)
    return d_out


def exact_masked_sum(oracle, kseed, param, vseed, p, voff, n, precision):
    """Host twin of build_exact_float_column -> (Σ (k - param/2) over the masked rows, number of masked rows)."""
    total, abs_total, count = 0, 0, 0
    for s in range(0, n, CHUNK):
        m = min(CHUNK, n - s)
        k = oracle.generate_values(4, kseed, s, param, m, np.int32).astype(np.int64) - param // 2
        k = k[host_mask(oracle, vseed, p, voff + s, m)]
        total += int(k.sum())
        abs_total += int(np.abs(k).sum())
        count += k.size
    assert abs_total <= 1 << precision, "inputs must keep every partial sum exact"
    return total, count


@pytest.mark.parametrize("dtype", FLOAT_DTYPES)
def test_float_sum_past_one_grid_exact(gpu, oracle, n_wave, dtype):
    """Order-independent float sums over N_WAVE rows: the values k - param/2 are integers with Σ|k| < 2^p, so the
    result must be Σx exactly. With validity: most rows null for f32 (to keep Σ|k| < 2^24), raw bit patterns (NaN,
    inf, anything) under every null slot. Without validity: the same rows valid, 0.0 everywhere else."""
    n, size = n_wave, abi.DTYPE_SIZE[dtype]
    kseed, vseed = 800 + dtype, 810 + dtype
    p, param = (2.0 ** -8, 16) if dtype == abi.F32 else (0.9, 1 << 20)
    d_valid = dev_bits(gpu, vseed, p, n + VOFF)
    try:
        exp_int, count = exact_masked_sum(oracle, kseed, param, vseed, p, VOFF, n, 24 if dtype == abi.F32 else 53)
        exp = float(np.array(exp_int, dtype=acu.NP_DTYPES[dtype]))
        for garbage_seed in (820 + dtype, None):
            d_vals = build_exact_float_column(gpu, dtype, n, kseed, param, d_valid, VOFF, garbage_seed)
            try:
                if garbage_seed is not None:
                    arrs = [make_arr(d_vals, n, d_valid, VOFF, n - count), make_arr(d_vals, n, d_valid, VOFF, -1)]
                else:
                    arrs = [make_arr(d_vals, n)]
                for arr in arrs:
                    bits, cnt = aggregate_bits(gpu, dtype, abi.SUM, arr)
                    got = float(np.array([bits], dtype=np.uint64).view(np.uint8)[:size].view(acu.NP_DTYPES[dtype])[0])
                    assert same_float(got, exp, dtype), f"sum garbage={garbage_seed is not None}: {got!r} != {exp!r}"
                    assert cnt == (count if arr.validity else n)
                if garbage_seed is not None:  # deferred count
                    (bits, cnt), = aggregate_in_section(gpu, dtype, make_arr(d_vals, n, d_valid, VOFF, -1), (abi.SUM,))
                    got = float(np.array([bits], dtype=np.uint64).view(np.uint8)[:size].view(acu.NP_DTYPES[dtype])[0])
                    assert same_float(got, exp, dtype) and cnt == count, f"sum in a section: {got!r} / {cnt}"
            finally:
                gpu.free(d_vals)
    finally:
        gpu.free(d_valid)


@pytest.mark.parametrize("dtype,op", [(abi.I32, abi.SUM), (abi.U16, abi.MAX), (abi.F32, abi.MIN)])
def test_batched_launch_long_and_short_columns(gpu, oracle, n_wave, dtype, op):
    """One acu_aggregate_columns call: 8 columns of one (dtype, op) share one launch whose grid is sized by the N_WAVE
    column, mixed with short columns (1, 64, 2049, 70001 rows ...) read from other places of the same buffers, an
    all-null and an empty column (None) and a second (dtype, op) group."""
    n, size = n_wave, abi.DTYPE_SIZE[dtype]
    seed, vseed, p = 900 + dtype, 910 + dtype, 0.9
    d_vals, d_valid = dev_raw(gpu, seed, n * size), dev_bits(gpu, vseed, p, n + VOFF)
    d_f64 = dev_raw(gpu, 920, 100_000 * 8)
    d_zero_bits = gpu.malloc(64)
    gpu.check(gpu.lib.acu_memset(gpu.h, d_zero_bits, 0, 64))
    try:
        # (first row, rows, with validity): first rows are multiples of 8 so the host twin starts on a word
        spans = [(0, n, True), (8, 1, True), (4096, 64, False), ((n - 2049) // 8 * 8, 2049, True), (123456, 70001, True),
                 ((n - 70001) // 8 * 8, 70001, False), (1 << 20, 33, True), (8 * 1000003, 300000, True)]
        cols, dtypes, ops, exps = [], [], [], []
        for start, m, with_valid in spans:
            ptr = d_vals + start * size
            if with_valid:
                cols.append(make_arr(ptr, m, d_valid, VOFF + start, -1))
                exps.append(twin_stats(oracle, dtype, seed, start, m, vseed, p, VOFF))
            else:
                cols.append(make_arr(ptr, m))
                exps.append(twin_stats(oracle, dtype, seed, start, m))
            dtypes.append(dtype)
            ops.append(op)
        cols.insert(3, make_arr(d_vals, 100, d_zero_bits, 0, -1))  # all null
        cols.insert(6, make_arr(d_vals, 0))                        # empty
        for at in (3, 6):
            dtypes.insert(at, dtype)
            ops.insert(at, op)
            exps.insert(at, {"count": 0})
        for start, m in ((0, 70001), (8, 5000)):  # a second group: Float64 max over raw bit patterns
            cols.append(make_arr(d_f64 + start * 8, m))
            dtypes.append(abi.F64)
            ops.append(abi.MAX)
            exps.append(twin_stats(oracle, abi.F64, 920, start, m))
        k = len(cols)
        arrs = (abi.Array * k)(*cols)
        bits, cnts = (C.c_uint64 * k)(), (C.c_int64 * k)()
        gpu.check(gpu.lib.acu_aggregate_columns(gpu.h, k, (C.c_int32 * k)(*dtypes), (C.c_int32 * k)(*ops), arrs, bits, cnts))
        for c in range(k):
            e, dt = exps[c], dtypes[c]
            assert cnts[c] == e["count"], f"column {c}: valid count {cnts[c]} != {e['count']}"
            if e["count"]:
                got = bits[c] & ((1 << (8 * abi.DTYPE_SIZE[dt])) - 1)
                assert got == e[ops[c]], f"column {c} ({cols[c].len} rows): {got:#x} != {e[ops[c]]:#x}"
    finally:
        for ptr in (d_vals, d_valid, d_f64, d_zero_bits):
            gpu.free(ptr)


def test_int8_reduce_past_2_pow_32_rows_in_section(gpu, oracle):
    """Int8 sum / min / max with validity past 2^32 rows, queued in a section: the valid count (> 2^32) comes from the
    kernel. The host twin (wrapping sum, extremes, popcount) is built chunk by chunk."""
    n = (1 << 32) + (1 << 28) + 12345
    seed, vseed, p, voff = 1000, 1001, 0.99, 3
    d_vals, d_valid = dev_raw(gpu, seed, n), dev_bits(gpu, vseed, p, n + voff)
    try:
        got = aggregate_in_section(gpu, abi.I8, make_arr(d_vals, n, d_valid, voff, -1))
    finally:
        gpu.free(d_vals)
        gpu.free(d_valid)
    exp = twin_stats(oracle, abi.I8, seed, 0, n, vseed, p, voff)
    assert exp["count"] > 1 << 32
    assert got == [(exp[op], exp["count"]) for op in OPS]


# ---- D. sum_checked over more than 1024 chunks ---------------------------------------------------------------------
SC_CHUNK = 4096
SC_N = 3 * (1 << 22) + 12345  # 3076 chunks: 4 per scan thread, threads 769..1023 idle
SC_PER = 4


def walk_values(rng, dtype, valid):
    """Valid rows whose running sum stays inside the type (signed: every prefix in [1, max/4]; unsigned: small
    non-negative steps, first one >= 1); every null slot holds an extreme value that would overflow if it counted."""
    npdt = acu.NP_DTYPES[dtype]
    info = np.iinfo(npdt)
    n, nv = len(valid), int(valid.sum())
    if info.min < 0:
        prefix = rng.integers(1, info.max // 4, nv, endpoint=True, dtype=np.int64)
        steps = np.diff(prefix, prepend=0)
    else:
        steps = rng.integers(0, info.max // (2 * n), nv, dtype=npdt)
        steps[:1] = np.maximum(steps[:1], 1)
    vals = np.empty(n, dtype=npdt)
    vals[valid] = steps.astype(npdt)
    junk = np.array([info.max, info.min if info.min < 0 else info.max, info.max - 1], dtype=npdt)
    vals[~valid] = junk[rng.integers(0, len(junk), n - nv)]
    return vals


def first_valid_at_or_after(valid, r):
    return r + int(np.argmax(valid[r:]))


SC_CASES = {
    "no_overflow": [],
    "first_chunk_of_a_range": [(300 * SC_PER * SC_CHUNK + 17, "max")],
    "last_chunk_of_a_range": [((500 * SC_PER + SC_PER - 1) * SC_CHUNK + 4000, "max")],
    "final_ragged_chunk": [(SC_N - 5, "max")],
    "two_threads": [((500 * SC_PER + 2) * SC_CHUNK + 9, "max"), (300 * SC_PER * SC_CHUNK + 4095, "max")],
    # the prefix leaves the range at the last row of a thread's range and comes back in the next thread's first row:
    # the total fits, only the prefix check sees it
    "prefix_leaves_and_returns": [((600 * SC_PER + SC_PER - 1) * SC_CHUNK + SC_CHUNK - 1, "max"), ("next", "min")],
}


@pytest.mark.parametrize("case,dtype", [(c, dt) for c in SC_CASES for dt in (abi.I8, abi.I32, abi.I64, abi.U64)
                                        if not (c == "prefix_leaves_and_returns" and dt == abi.U64)])  # unsigned: monotone
def test_sum_checked_many_chunks(gpu, oracle, dtype, case):
    info = np.iinfo(acu.NP_DTYPES[dtype])
    rng = np.random.default_rng(14000 + 31 * dtype + list(SC_CASES).index(case))
    for null_p in (None, 0.3):
        valid = np.ones(SC_N, dtype=bool) if null_p is None else rng.random(SC_N) >= null_p
        vals = walk_values(rng, dtype, valid)
        r = 0
        for where, kind in SC_CASES[case]:
            r = first_valid_at_or_after(valid, r + 1 if where == "next" else where)
            vals[r] = info.max if kind == "max" else info.min
        a = HostArray.from_numpy(dtype, vals, None if null_p is None else valid, bit_offset=int(rng.integers(1, 8)))
        got, exp = expect_same_error(gpu, oracle, lambda be: be.sum_checked(a))
        assert got == exp, f"sum_checked {case} dtype={dtype} nulls={null_p}: {got} != {exp}"
        if case == "no_overflow":
            assert exp is not None
        else:
            with pytest.raises(acu.ArrowError):
                oracle.sum_checked(a)
