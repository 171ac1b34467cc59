"""Config-scale parity: BASELINE.json configs #2-#4 at >= 1e8 rows, the CUDA path (through the C ABI) against the
CPU oracle on the host twin of the device-generated table, compared byte for byte — values including the bytes
under null slots, validity bitmaps, null_count, NullBuffer presence, offsets.

The kernel paths that only exist at this scale (multi-wave grids, the u64 tile-offset scan across > 4096 chunks,
the bulk-copy phase flips of k_take over thousands of tiles per warp, bytes offsets near the i32 limit) are exactly
what the <= 70,001-row fuzz tests cannot reach. Inputs follow SURVEY.md §8(d): counter-based splitmix64 streams
generated ON THE DEVICE (acu_generate_*), seeds 42/43 values, 44/45 validity, 46 predicate, 47 indices; the host
twin is the D2H copy, and a spot check pins the device generator against the oracle's.

Pattern: the reference's fuzz_filter (arrow-select/src/filter.rs:1888-1977) at config scale.
ACU_CONFIG_ROWS overrides the row count (default 1e8).
"""
import ctypes as C
import os

import numpy as np
import pytest

import acu
from acu import _abi as abi
from acu import BOOL, HostArray

from test_gpu_parity import assert_float_sum, assert_same

pytestmark = pytest.mark.gpu

N = int(os.environ.get("ACU_CONFIG_ROWS", "100000000"))
NULL_P, SEL = 0.05, 0.10


def dev_values(gpu, kind, seed, n, np_dtype, param=0):
    d = gpu.malloc(n * np.dtype(np_dtype).itemsize + 64)
    gpu.check(gpu.lib.acu_generate_values(gpu.h, kind, seed, 0, param, d, n))
    out = gpu.d2h(d, n * np.dtype(np_dtype).itemsize, np_dtype)
    gpu.free(d)
    return out


def dev_bits(gpu, seed, p, n):
    d = gpu.malloc(abi.bitmap_bytes(n) + 64)
    gpu.check(gpu.lib.acu_generate_bits(gpu.h, seed, 0, p, d, n))
    out = gpu.d2h(d, abi.bitmap_bytes(n))
    gpu.free(d)
    return np.concatenate([out, np.zeros(8, np.uint8)])


def popcount(bits, n):
    full = np.unpackbits(bits[: (n + 7) // 8], bitorder="little")[:n]
    return int(full.sum())


def prim(dtype, values, validity, n):
    nc = n - popcount(validity, n) if validity is not None else 0
    return HostArray(dtype, values, n, validity, 0, 0, nc)


@pytest.fixture(scope="module")
def table(gpu):
    """The config-2/3/4 columns, generated on the device, downloaded once."""
    t = {}
    t["i64"] = prim(abi.I64, dev_values(gpu, 0, 42, N, np.int64), dev_bits(gpu, 44, 1 - NULL_P, N), N)
    t["pred"] = HostArray(BOOL, dev_bits(gpu, 46, SEL, N), N, None, 0, 0, 0)
    fa, fb = dev_values(gpu, 2, 42, N, np.float64), dev_values(gpu, 2, 43, N, np.float64)
    # specials at ~2^-20 density (SURVEY §8(d)): +-0, +-inf, +-NaN, subnormals
    rng = np.random.default_rng(5)
    sp = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan, 5e-324, -5e-324, 2.2250738585072009e-308], dtype=np.float64)
    for v in (fa, fb):
        pos = rng.integers(0, N, max(N >> 20, 8))
        v[pos] = sp[rng.integers(0, len(sp), len(pos))]
    t["fa"] = prim(abi.F64, fa, dev_bits(gpu, 144, 1 - NULL_P, N), N)
    t["fb"] = prim(abi.F64, fb, dev_bits(gpu, 45, 1 - NULL_P, N), N)
    return t


def test_device_generator_matches_host_twin(gpu, oracle):
    n = 1 << 20
    for kind, dt, param in [(0, np.int64, 0), (1, np.int64, 0), (2, np.float64, 0), (3, np.uint32, 12345), (4, np.int32, 4096)]:
        got = dev_values(gpu, kind, 42, n, dt, param)
        exp = oracle.generate_values(kind, 42, 0, param, n, dt)
        assert np.array_equal(got.view(np.uint8), exp.view(np.uint8)), f"generator kind {kind}"
    for p in (0.1, 0.95, 1.0):
        assert np.array_equal(dev_bits(gpu, 46, p, n)[: n // 8], oracle.generate_bits(46, 0, p, n)[: n // 8])


# ---- config #2: filter + take Int64, s = 0.1, 5 % nulls -------------------------------------------
def test_config2_filter_int64(gpu, oracle, table):
    got, exp = gpu.filter(table["i64"], table["pred"]), oracle.filter(table["i64"], table["pred"])
    assert exp.length > 0.09 * N
    assert_same(got, exp, f"config 2 filter Int64 N={N}")
    assert gpu.filter_plan(table["pred"]) == oracle.filter_plan(table["pred"])


@pytest.mark.parametrize("sel,pred_nulls", [(0.5, False), (0.9, False), (0.1, True), (0.001, False)])
def test_config2_filter_other_selectivities(gpu, oracle, table, sel, pred_nulls):
    """config #1's 50 % selectivity, the dense SlicesIterator regime (> 0.8, filter.rs:346-364), a 5 %-null predicate
    (prep_null_mask_filter) and a sparse one, all at config scale."""
    pv = dev_bits(gpu, 460 + int(sel * 1000), sel, N)
    if pred_nulls:
        nv = dev_bits(gpu, 461, 0.95, N)
        pred = HostArray(BOOL, pv, N, nv, 0, 0, N - popcount(nv, N))
    else:
        pred = HostArray(BOOL, pv, N, None, 0, 0, 0)
    assert_same(gpu.filter(table["i64"], pred), oracle.filter(table["i64"], pred), f"filter Int64 N={N} s={sel} pred_nulls={pred_nulls}")


def test_config2_filter_no_null_column_and_int32(gpu, oracle, table):
    col = HostArray(abi.I64, table["i64"].values, N, None, 0, 0, 0)
    assert_same(gpu.filter(col, table["pred"]), oracle.filter(col, table["pred"]), "filter Int64 without NullBuffer")
    c32 = prim(abi.I32, table["i64"].values.view(np.int32)[:N], table["i64"].validity, N)
    assert_same(gpu.filter(c32, table["pred"]), oracle.filter(c32, table["pred"]), "filter Int32")


def test_config2_take_monotone(gpu, oracle, table):
    """index distribution A: the selected rows of the predicate (what filter -> take produces)."""
    sel = np.nonzero(np.unpackbits(table["pred"].values[: (N + 7) // 8], bitorder="little")[:N])[0].astype(np.uint32)
    idx = HostArray.from_numpy(abi.U32, sel)
    assert_same(gpu.take(table["i64"], idx), oracle.take(table["i64"], idx), f"take monotone M={len(sel)}")


def test_config2_take_dense_monotone(gpu, oracle, table):
    """index distribution A': every other row (M = N/2), UInt64 indices."""
    idx = HostArray.from_numpy(abi.U64, np.arange(0, N, 2, dtype=np.uint64))
    assert_same(gpu.take(table["i64"], idx), oracle.take(table["i64"], idx), "take dense monotone u64")


def test_config2_take_uniform_random_with_null_indices(gpu, oracle, table):
    """index distribution B: uniform random UInt32 in [0, N), 5 % null indices."""
    m = max(N // 10, 1)
    ix = dev_values(gpu, 3, 47, m, np.uint32, N)
    iv = dev_bits(gpu, 470, 0.95, m)
    idx = HostArray(abi.U32, ix, m, iv, 0, 0, m - popcount(iv, m))
    assert_same(gpu.take(table["i64"], idx), oracle.take(table["i64"], idx), f"take uniform random M={m}")
    col = HostArray(abi.I64, table["i64"].values, N, None, 0, 0, 0)
    assert_same(gpu.take(col, idx), oracle.take(col, idx), "take uniform random, values without nulls")


# ---- config #3: add / mul / lt / eq Float64, 5 % nulls each side -------------------------------------
@pytest.mark.parametrize("op", ["add", "mul", "sub", "div"])
def test_config3_arith_float64(gpu, oracle, table, op):
    got, exp = getattr(gpu, op)(table["fa"], table["fb"]), getattr(oracle, op)(table["fa"], table["fb"])
    assert_same(got, exp, f"config 3 {op} Float64 N={N}", float_nan_ok=True)


@pytest.mark.parametrize("op", ["lt", "eq", "gt_eq", "distinct"])
def test_config3_cmp_float64(gpu, oracle, table, op):
    got, exp = getattr(gpu, op)(table["fa"], table["fb"]), getattr(oracle, op)(table["fa"], table["fb"])
    assert_same(got, exp, f"config 3 {op} Float64 N={N}")


def test_config3_add_int64_checked_and_wrapping(gpu, oracle, table):
    a = prim(abi.I64, dev_values(gpu, 1, 42, N, np.int64), table["fa"].validity, N)
    b = prim(abi.I64, dev_values(gpu, 1, 43, N, np.int64), table["fb"].validity, N)
    assert_same(gpu.add(a, b), oracle.add(a, b), "add Int64 checked (no overflow, zero under nulls)")
    assert_same(gpu.add_wrapping(table["i64"], a), oracle.add_wrapping(table["i64"], a), "add_wrapping Int64")
    # overflow injection far into the array: both sides must report the same lowest failing row and text
    a.values[N - 12345] = np.iinfo(np.int64).max
    b.values[N - 12345] = 1
    vm = np.unpackbits(a.validity[: (N + 7) // 8] & b.validity[: (N + 7) // 8], bitorder="little")
    if vm[N - 12345]:
        with pytest.raises(acu.ArrowError) as ge:
            gpu.add(a, b)
        with pytest.raises(acu.ArrowError) as oe:
            oracle.add(a, b)
        assert str(ge.value) == str(oe.value) and ge.value.index == oe.value.index == N - 12345


# ---- config #4: cast Int64 -> Float64; Dictionary<Int32,Utf8> -> Utf8 ------------------------------------
def test_config4_cast_int64_to_float64(gpu, oracle, table):
    assert_same(gpu.cast(table["i64"], abi.F64), oracle.cast(table["i64"], abi.F64), f"config 4 cast Int64->Float64 N={N}")


def test_config4_sum_min_max(gpu, oracle, table):
    assert gpu.sum(table["i64"]) == oracle.sum(table["i64"])
    for op in ("min", "max"):
        assert getattr(gpu, op)(table["i64"]) == getattr(oracle, op)(table["i64"])
        g, e = getattr(gpu, op)(table["fa"]), getattr(oracle, op)(table["fa"])
        assert np.float64(g).tobytes() == np.float64(e).tobytes()
    # fa carries ~N/2^20 specials, so its sum is NaN exactly when a valid NaN or both infinities survive the nulls
    fa = table["fa"]
    valid = np.unpackbits(fa.validity[: (N + 7) // 8], bitorder="little")[:N].astype(bool)
    sm = gpu.lib.acu_device_sm_count(gpu.h)
    assert_float_sum(gpu.sum(fa), fa.values, valid, abi.F64, sm, f"config 4 sum Float64 N={N}")
    # the other ~1e8 rows: the same column with the specials replaced by 0 on the host twin, re-uploaded
    clean = np.where(np.isfinite(fa.values), fa.values, 0.0)
    g = gpu.sum(prim(abi.F64, clean, fa.validity, N))
    assert g is not None and np.isfinite(g)
    assert_float_sum(g, clean, valid, abi.F64, sm, f"config 4 sum Float64 without specials N={N}")


def make_dictionary(d=4096, seed=1):
    rng = np.random.default_rng(seed)
    lens = rng.integers(4, 13, d)
    offs = np.zeros(d + 1, dtype=np.int32)
    offs[1:] = np.cumsum(lens)
    data = rng.integers(97, 123, int(offs[-1]) + 16).astype(np.uint8)
    return offs, data


def test_config4_dictionary_to_utf8(gpu, oracle):
    """cast(Dictionary<Int32,Utf8> -> Utf8) = take_bytes(dictionary, keys) (arrow-cast/src/cast/dictionary.rs:310-317):
    D = 4096 strings of 4..12 bytes, keys uniform with 5 % nulls."""
    d = 4096
    offs, data = make_dictionary(d)
    keys_v = dev_values(gpu, 4, 48, N, np.int32, d)
    kv = dev_bits(gpu, 49, 0.95, N)
    keys = HostArray(abi.I32, keys_v, N, kv, 0, 0, N - popcount(kv, N))
    nulls_of = HostArray(acu.U8, np.zeros(0, np.uint8), d, None, 0, 0, 0)
    g_off, g_data, g_n = gpu.take_bytes(offs, data, nulls_of, keys)
    e_off, e_data, e_n = oracle.take_bytes(offs, data, nulls_of, keys)
    assert np.array_equal(g_off, e_off), "offsets differ"
    assert np.array_equal(g_data, e_data), "value bytes differ"
    assert (g_n.validity is None) == (e_n.validity is None) and g_n.null_count == e_n.null_count
    assert np.array_equal(g_n.validity[: N // 8], e_n.validity[: N // 8])
    # dictionary with null entries: output nulls = keys' nulls AND dictionary nulls (take_nulls, take.rs:419-430)
    dv = acu.pack_bits(np.random.default_rng(2).random(d) >= 0.1)
    nulls_of = HostArray(acu.U8, np.zeros(0, np.uint8), d, dv, 0, 0, d - popcount(dv, d))
    m = min(N, 20_000_000)
    keys_s = HostArray(abi.I32, keys_v[:m], m, kv, 0, 0, -1)
    g_off, g_data, g_n = gpu.take_bytes(offs, data, nulls_of, keys_s)
    e_off, e_data, e_n = oracle.take_bytes(offs, data, nulls_of, keys_s)
    assert np.array_equal(g_off, e_off) and np.array_equal(g_data, e_data) and g_n.null_count == e_n.null_count
    assert np.array_equal(g_n.validity[: m // 8], e_n.validity[: m // 8])


def test_config5_utf8_filter_take_at_batch_scale(gpu, oracle):
    """One config-5 Utf8 column at batch scale (2^26 rows, L = 8: 5.4e8 bytes < 2^31): filter_bytes then take_bytes."""
    n = min(N, 1 << 26)
    d = 4096
    offs_d, data_d = make_dictionary(d, seed=7)
    keys = HostArray(abi.I32, dev_values(gpu, 4, 300, n, np.int32, d), n, None, 0, 0, 0)
    nulls_of = HostArray(acu.U8, np.zeros(0, np.uint8), d, None, 0, 0, 0)
    s_off, s_data, _ = oracle.take_bytes(offs_d, data_d, nulls_of, keys)  # the column itself
    sv = dev_bits(gpu, 400, 0.95, n)
    col_nulls = HostArray(acu.U8, np.zeros(0, np.uint8), n, sv, 0, 0, n - popcount(sv, n))
    pred = HostArray(BOOL, dev_bits(gpu, 46, SEL, n), n, None, 0, 0, 0)
    g = gpu.filter_bytes(s_off, s_data, col_nulls, pred)
    e = oracle.filter_bytes(s_off, s_data, col_nulls, pred)
    assert np.array_equal(g[0], e[0]) and np.array_equal(g[1], e[1]) and g[2].null_count == e[2].null_count
    cnt = len(e[0]) - 1
    assert np.array_equal(g[2].validity[: cnt // 8], e[2].validity[: cnt // 8])
    idx = HostArray.from_numpy(abi.U32, np.arange(0, cnt, 2, dtype=np.uint32))
    gt, et = gpu.take_bytes(e[0], e[1], e[2], idx), oracle.take_bytes(e[0], e[1], e[2], idx)
    assert np.array_equal(gt[0], et[0]) and np.array_equal(gt[1], et[1]) and gt[2].null_count == et[2].null_count


# ---- config #1 twin on the GPU: filter Int32 1e6, s = 0.5 (the CPU run is tests/test_config1_cpu.py) ------
def test_config1_gpu_twin(gpu, oracle):
    from test_config1_cpu import config1
    for null_p, pred_null_p in [(None, None), (0.05, None), (0.05, 0.05), (0.0, None)]:
        col, pred = config1(oracle, null_p, pred_null_p)
        assert_same(gpu.filter(col, pred), oracle.filter(col, pred), f"config 1 nulls={null_p}/{pred_null_p}")
