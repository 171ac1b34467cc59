"""RecordBatch-level entry points (acu_filter_record_batch / acu_take_record_batch /
acu_aggregate_columns) vs the oracle applied column by column — which is exactly what the
reference does: filter_record_batch filters every column with one FilterPredicate
(arrow-select/src/filter.rs:225-244, :459-478) and take_record_batch takes every column with
the same indices (arrow-select/src/take.rs:1123-1133). Bit-exact, including NullBuffer
presence and the bytes under nulls; one stream synchronisation per call on the CUDA side."""
import numpy as np
import pytest

import acu
from acu import _abi as abi
from acu import BOOL, HostArray, Utf8Column
from test_gpu_parity import (assert_same, assert_same_bytes, exact_float_array, expect_same_error, rand_array, rand_bool,
                             rand_strings, same_float)

pytestmark = pytest.mark.gpu


def make_batch(rng, n, nulls=0.1):
    """8+ columns of one length: the config-5 schema {3 x Int64, 3 x Float64, 2 x Utf8} plus a boolean, narrow and
    128-bit columns, with and without validity buffers (and one validity buffer without nulls)."""
    cols = [rand_array(rng, abi.I64, n, nulls), rand_array(rng, abi.I64, n, None), rand_array(rng, abi.I64, n, 0.0),
            rand_array(rng, abi.F64, n, nulls), rand_array(rng, abi.F64, n, nulls, offset=3), rand_array(rng, abi.F64, n, None)]
    for null_p in (nulls, None):
        o, d, nl = rand_strings(rng, n, null_p)
        cols.append(Utf8Column(o, d, nl))
    cols.append(rand_bool(rng, n, 0.5, nulls))
    cols.append(rand_array(rng, abi.I8, n, nulls))
    cols.append(rand_array(rng, abi.U16, n, None, offset=5))
    return cols


def oracle_filter(oracle, col, pred):
    if isinstance(col, Utf8Column):
        return oracle.filter_bytes(col.offsets, col.data, col.nulls, pred)
    return oracle.filter(col, pred)


def oracle_take(oracle, col, idx):
    if isinstance(col, Utf8Column):
        return oracle.take_bytes(col.offsets, col.data, col.nulls, idx)
    return oracle.take(col, idx)


def check_columns(got, cols, expect_fn, what):
    assert len(got) == len(cols)
    for c, col in enumerate(cols):
        exp = expect_fn(col)
        if isinstance(col, Utf8Column):
            assert_same_bytes((got[c].offsets, got[c].data, got[c].nulls), exp, f"{what} col {c} (utf8)")
        else:
            assert_same(got[c], exp, f"{what} col {c}")


@pytest.mark.parametrize("n", [0, 1, 64, 1000, 4097, 70001])
def test_filter_record_batch(gpu, oracle, n):
    rng = np.random.default_rng(500 + n)
    cols = make_batch(rng, n)
    for true_p, pnull in [(0.0, None), (0.1, None), (0.5, 0.05), (0.9, None), (1.0, None)]:
        pred = rand_bool(rng, n, true_p, pnull)
        got = gpu.filter_record_batch(cols, pred)
        check_columns(got, cols, lambda col: oracle_filter(oracle, col, pred), f"filter_record_batch n={n} p={true_p}")


def test_filter_record_batch_no_columns_and_errors(gpu, oracle):
    rng = np.random.default_rng(77)
    pred = rand_bool(rng, 100, 0.5, None)
    assert gpu.filter_record_batch([], pred) == []  # filter.rs:1727 test_filter_record_batch_no_columns
    # predicate longer than a column: the reference's error text, whichever column fails first (filter.rs:537-541)
    cols = [rand_array(rng, abi.I64, 100, 0.1), rand_array(rng, abi.I32, 50, None)]
    with pytest.raises(acu.ArrowError) as e:
        gpu.filter_record_batch(cols, pred)
    assert "Filter predicate of length 100 is larger than target array of length 50" in str(e.value)


@pytest.mark.parametrize("n,m", [(1, 10), (50, 0), (1000, 64), (4097, 20000), (70001, 5000)])
def test_take_record_batch(gpu, oracle, n, m):
    rng = np.random.default_rng(900 + n)
    cols = make_batch(rng, n)
    for idt, inull in [(abi.U32, None), (abi.I32, 0.1), (abi.U64, None), (abi.I64, 0.3)]:
        idx = HostArray.from_numpy(idt, rng.integers(0, n, m).astype(acu.NP_DTYPES[idt]), None if inull is None else rng.random(m) >= inull)
        got = gpu.take_record_batch(cols, idx)
        check_columns(got, cols, lambda col: oracle_take(oracle, col, idx), f"take_record_batch n={n} m={m} idx={idt}")
    # monotone indices (what filter -> take produces), all columns
    if m and n > 1:
        idx = HostArray.from_numpy(abi.U32, np.sort(rng.integers(0, n, m)).astype(np.uint32))
        got = gpu.take_record_batch(cols, idx, check_bounds=True)
        check_columns(got, cols, lambda col: oracle_take(oracle, col, idx), f"take_record_batch monotone n={n}")


def test_take_record_batch_out_of_bounds(gpu, oracle):
    rng = np.random.default_rng(5)
    cols = [rand_array(rng, abi.I64, 20, 0.2), rand_array(rng, abi.F64, 20, None)]
    o, d, nl = rand_strings(rng, 20, 0.2)
    idx = HostArray.from_list(abi.U32, [1, 1000, 2])
    for cb in (False, True):
        got, exp = expect_same_error(gpu, oracle, lambda be: (be.take_record_batch(cols, idx, cb) if be is gpu else be.take(cols[0], idx, cb)))
        assert got is None and exp is None
    # a variable-width column alone: the bytes pass reports the panic (take.rs:517)
    for cb in (False, True):
        got, exp = expect_same_error(gpu, oracle, lambda be: (be.take_record_batch([Utf8Column(o, d, nl)], idx, cb) if be is gpu
                                                               else be.take_bytes(o, d, nl, idx, cb)))
        assert got is None and exp is None


def test_aggregate_columns(gpu, oracle):
    rng = np.random.default_rng(31)
    for n in [0, 1, 65, 1000, 70001]:
        cols = [rand_array(rng, abi.I64, n, 0.1), rand_array(rng, abi.I64, n, None), rand_array(rng, abi.I32, n, 1.0), rand_array(rng, abi.U8, n, 0.5),
                rand_array(rng, abi.F64, n, 0.1), rand_array(rng, abi.F32, n, None)]
        for op_name, op in (("sum", abi.SUM), ("min", abi.MIN), ("max", abi.MAX)):
            use = cols if op != abi.SUM else cols[:4]  # float sums are order-dependent: checked in test_gpu_parity
            got = gpu.aggregate_columns([op] * len(use), use)
            for c, col in enumerate(use):
                exp = getattr(oracle, op_name)(col)
                if isinstance(exp, float) and np.isnan(exp):
                    assert np.isnan(got[c]) and np.signbit(got[c]) == np.signbit(exp)
                else:
                    assert got[c] == exp, f"{op_name} n={n} col {c}: {got[c]} != {exp}"
        # float sums on order-independent inputs (exact in any association order), in one call with integer sums
        exact = [exact_float_array(rng, dt, n, kind, null_p, off)
                 for dt, kind, null_p, off in ((abi.F64, "ints", 0.1, 1), (abi.F32, "dyadic", None, 0),
                                               (abi.F32, "garbage_under_nulls", 0.9, 3), (abi.F64, "subnormal", None, 2))]
        use = [h for h, _ in exact] + cols[:2]
        got = gpu.aggregate_columns([abi.SUM] * len(use), use)
        for c, (h, e) in enumerate(exact):
            assert same_float(got[c], e, h.dtype), f"float sum n={n} col {c}: {got[c]!r} != {e!r}"
        assert got[len(exact):] == [oracle.sum(cols[0]), oracle.sum(cols[1])]
        # mixed ops in one call
        got = gpu.aggregate_columns([abi.SUM, abi.MIN, abi.MAX], cols[:3])
        assert got == [oracle.sum(cols[0]), oracle.min(cols[1]), oracle.max(cols[2])]


def test_pipeline_filter_take_sum_matches_oracle(gpu, oracle):
    """Config 5 in miniature: filter_record_batch -> take_record_batch (monotone half-sample) -> sums."""
    rng = np.random.default_rng(2024)
    n = 50_000
    cols = make_batch(rng, n)[:8]
    pred = rand_bool(rng, n, 0.1, None)
    f_gpu = gpu.filter_record_batch(cols, pred)
    count = f_gpu[0].length
    keep = np.flatnonzero(rng.random(count) < 0.5).astype(np.uint32)
    idx = HostArray.from_numpy(abi.U32, keep)
    t_gpu = gpu.take_record_batch(f_gpu, idx)
    f_or = [oracle_filter(oracle, col, pred) for col in cols]
    f_or_cols = [Utf8Column(*x) if isinstance(x, tuple) else x for x in f_or]
    check_columns(t_gpu, f_or_cols, lambda col: oracle_take(oracle, col, idx), "pipeline take")
    sums = gpu.aggregate_columns([abi.SUM] * 3, t_gpu[:3])
    assert sums == [oracle.sum(oracle_take(oracle, c, idx)) for c in f_or_cols[:3]]


def test_many_columns_share_launches(gpu, oracle):
    """More equal-width columns than one batched launch holds (8), mixed with other widths: every column still right;
    more than ACU_MAX_BATCH_COLUMNS in one call is an argument error (the C++ mirror splits such batches)."""
    rng = np.random.default_rng(4242)
    n = 5000
    cols = [rand_array(rng, abi.I32 if c % 3 else abi.I64, n, 0.1 if c % 2 else None) for c in range(21)]
    cols += [rand_bool(rng, n, 0.5, 0.1) for _ in range(10)]
    pred = rand_bool(rng, n, 0.4, None)
    check_columns(gpu.filter_record_batch(cols, pred), cols, lambda col: oracle_filter(oracle, col, pred), "31 columns filter")
    idx = HostArray.from_numpy(abi.U32, rng.integers(0, n, 3000).astype(np.uint32), rng.random(3000) >= 0.05)
    check_columns(gpu.take_record_batch(cols, idx), cols, lambda col: oracle_take(oracle, col, idx), "31 columns take")
    ops = [abi.SUM, abi.MIN, abi.MAX] * 7
    got = gpu.aggregate_columns(ops, cols[:21])
    exp = [getattr(oracle, ("sum", "min", "max")[op])(col) for op, col in zip(ops, cols[:21])]
    assert got == exp
    with pytest.raises(acu.ArrowError) as e:
        gpu.filter_record_batch([cols[0]] * 65, pred)
    assert e.value.status == abi.ERR_INVALID_ARGUMENT
