"""Stream-ordered sections (acu_async_begin ... acu_results_fetch, include/arrow_cuda.h): a chain of calls queued with ONE
synchronisation must give exactly what the synchronous entry points give one by one — values, validity bits, null counts,
NullBuffer presence, aggregate, and the first error in call order with the reference's text. Checked against the oracle
(which restates the synchronous reference functions: filter.rs:201-213, take.rs:89-105, numeric.rs:36-374,
aggregate.rs:317-366, cmp.rs:79-382)."""
import ctypes as C

import numpy as np
import pytest

import acu
from acu import _abi as abi
from acu import BOOL, ArrowError, HostArray

from test_gpu_parity import assert_float_sum, assert_same, rand_array, rand_bool

pytestmark = pytest.mark.gpu


def selected_rows(pred):
    bits = np.unpackbits(np.asarray(pred.values, dtype=np.uint8), bitorder="little")[pred.values_offset:pred.values_offset + pred.length].astype(bool)
    if pred.validity is not None:
        v = np.unpackbits(pred.validity, bitorder="little")[pred.validity_offset:pred.validity_offset + pred.length].astype(bool)
        bits &= v
    return np.flatnonzero(bits)


@pytest.mark.parametrize("dtype", [abi.I64, abi.I32, abi.F64, abi.I8])
def test_chain_matches_synchronous_calls(gpu, oracle, dtype):
    rng = np.random.default_rng(900 + dtype)
    for n in [1, 63, 64, 1000, 4097, 70001, 300000]:
        for col_null, sel, pred_null, idx_null in [(0.05, 0.1, None, None), (None, 0.5, 0.1, None), (0.3, 0.0, None, 0.2),
                                                   (0.0, 1.0, None, None), (0.5, 1.0, None, None), (None, 0.93, None, None)]:
            col = rand_array(rng, dtype, n, col_null, 0)
            pred = rand_bool(rng, n, sel, pred_null, 0)
            rows = selected_rows(pred)
            if len(rows) == 0:
                rows = np.array([0])
            idx_vals = rows.astype(np.uint32)
            if idx_null is not None:
                iv = np.packbits(rng.random(len(idx_vals)) >= idx_null, bitorder="little")
                iv = np.concatenate([iv, np.zeros(8, np.uint8)])
                nulls = len(idx_vals) - int(np.unpackbits(iv, bitorder="little")[:len(idx_vals)].sum())
                idx = HostArray(abi.U32, idx_vals, len(idx_vals), iv, 0, 0, nulls)
            else:
                idx = HostArray(abi.U32, idx_vals, len(idx_vals))
            a, b = rand_array(rng, dtype, n, 0.1, 0), rand_array(rng, dtype, n, None, 0)
            op = acu.ADD_WRAPPING
            got_f, got_t, got_a, got_s = gpu.chain(col, pred, idx, a, b, arith_op=op, agg_op=acu.SUM)
            what = f"n={n} nulls={col_null} sel={sel}"
            assert_same(got_f, oracle.filter(col, pred), "chain filter " + what)
            exp_t = oracle.take(col, idx)
            assert_same(got_t, exp_t, "chain take " + what)
            assert_same(got_a, oracle.arith(op, a, b), "chain arith " + what)
            exp_s = oracle.aggregate(acu.SUM, exp_t)
            if dtype == abi.F64:
                assert (got_s is None) == (exp_s is None)
                # rand_values injects NaN / inf: NaN exactly when a valid NaN or both infinities were taken
                sm = gpu.lib.acu_device_sm_count(gpu.h)
                assert_float_sum(got_s, exp_t.value_array(), exp_t.valid_mask(), dtype, sm, "chain sum " + what)
                # and the finite rows: the same chain over the column with its specials replaced by 0
                cv = col.value_array()
                clean = HostArray(dtype, np.where(np.isfinite(cv), cv, 0.0), n, col.validity, col.validity_offset, 0,
                                  col.null_count)
                clean_t = oracle.take(clean, idx)
                got_c = gpu.chain(clean, pred, idx, a, b, arith_op=op, agg_op=acu.SUM)[3]
                assert got_c is None or np.isfinite(got_c)
                assert_float_sum(got_c, clean_t.value_array(), clean_t.valid_mask(), dtype, sm, "chain sum without specials " + what)
            else:
                assert got_s == exp_s, "chain sum " + what


def test_chain_boolean_column(gpu, oracle):
    rng = np.random.default_rng(77)
    for n in [65, 5000, 70001]:
        col = rand_bool(rng, n, 0.4, 0.2, 0)
        pred = rand_bool(rng, n, 0.3, None, 0)
        idx = HostArray(abi.U32, selected_rows(pred).astype(np.uint32), len(selected_rows(pred)))
        a, b = rand_array(rng, abi.I32, n, None, 0), rand_array(rng, abi.I32, n, 0.2, 0)
        got_f, got_t, got_a, _ = gpu.chain(col, pred, idx, a, b, arith_op=acu.MUL_WRAPPING)
        assert_same(got_f, oracle.filter(col, pred), f"bool chain filter n={n}")
        assert_same(got_t, oracle.take(col, idx), f"bool chain take n={n}")
        assert_same(got_a, oracle.arith(acu.MUL_WRAPPING, a, b), f"bool chain arith n={n}")


def test_chain_with_comparison_predicate(gpu, oracle):
    """cmp -> fused plan -> filter inside one section (the comparison's own output is checked too)."""
    rng = np.random.default_rng(78)
    for n in [100, 4097, 200000]:
        x, y = rand_array(rng, abi.I64, n, 0.1, 0), rand_array(rng, abi.I64, n, 0.05, 0)
        col = rand_array(rng, abi.F64, n, 0.2, 0)
        pred = oracle.cmp(acu.LT, x, y)
        rows = selected_rows(pred)
        idx = HostArray(abi.U32, rows.astype(np.uint32), len(rows)) if len(rows) else HostArray(abi.U32, np.zeros(1, np.uint32), 1)
        a, b = rand_array(rng, abi.F64, n, None, 0), rand_array(rng, abi.F64, n, None, 0)
        got_f, got_t, got_a, _, got_p = gpu.chain(col, None, idx, a, b, cmp_with=(acu.LT, x, y))
        assert_same(got_p, pred, f"chain cmp n={n}")
        assert_same(got_f, oracle.filter(col, pred), f"chain cmp->filter n={n}")
        assert_same(got_t, oracle.take(col, idx), f"chain take n={n}")
        assert_same(got_a, oracle.arith(acu.ADD, a, b), f"chain add n={n}")


def test_first_error_in_call_order(gpu, oracle):
    """A checked overflow queued in a section surfaces at the fetch with the synchronous call's exact text."""
    n = 5000
    rng = np.random.default_rng(5)
    col = rand_array(rng, abi.I64, n, 0.1, 0)
    pred = rand_bool(rng, n, 0.5, None, 0)
    idx = HostArray(abi.U32, selected_rows(pred).astype(np.uint32), len(selected_rows(pred)))
    av = rng.integers(-100, 100, n).astype(np.int64)
    bv = rng.integers(-100, 100, n).astype(np.int64)
    av[1234], bv[1234] = np.iinfo(np.int64).max, 5
    av[4000], bv[4000] = np.iinfo(np.int64).max, 7
    a, b = HostArray(abi.I64, av, n), HostArray(abi.I64, bv, n)
    with pytest.raises(ArrowError) as sync_err:
        gpu.arith(acu.ADD, a, b)
    with pytest.raises(ArrowError) as async_err:
        gpu.chain(col, pred, idx, a, b, arith_op=acu.ADD)
    assert str(async_err.value) == str(sync_err.value)
    assert async_err.value.index == sync_err.value.index == 1234
    with pytest.raises(ArrowError) as ora:
        oracle.arith(acu.ADD, a, b)
    assert str(ora.value) == str(sync_err.value)
    # the ctx is usable again, synchronously
    assert_same(gpu.arith(acu.ADD_WRAPPING, a, b), oracle.arith(acu.ADD_WRAPPING, a, b), "after a failed section")


def test_out_of_bounds_take_in_section(gpu):
    n = 1000
    rng = np.random.default_rng(6)
    col = rand_array(rng, abi.I32, n, None, 0)
    pred = rand_bool(rng, n, 0.5, None, 0)
    iv = np.arange(10, dtype=np.uint32)
    iv[7] = 5000
    idx = HostArray(abi.U32, iv, 10)
    a = rand_array(rng, abi.I32, n, None, 0)
    with pytest.raises(ArrowError) as e:
        gpu.chain(col, pred, idx, a, a, arith_op=acu.ADD_WRAPPING)
    assert e.value.status == abi.ERR_PANIC_OUT_OF_BOUNDS and "5000" in str(e.value)


def test_section_rules(gpu):
    lib, h = gpu.lib, gpu.h
    rng = np.random.default_rng(7)
    x = rand_array(rng, abi.I64, 1000, 0.1, 0)
    # fetch without a section / nested begin
    assert lib.acu_results_fetch(h) == abi.ERR_INVALID_ARGUMENT
    gpu.async_begin()
    assert lib.acu_async_begin(h) == abi.ERR_INVALID_ARGUMENT
    # an entry point that has to synchronise refuses loudly (cast is not split into enqueue + finalise)
    dx = gpu.upload(x)
    out = gpu.alloc_out(1000 * 8, 1000)
    xd = dx.descriptor()
    st = lib.acu_cast_numeric(h, abi.I64, abi.F64, 1, C.byref(xd), C.byref(out))
    assert st == abi.ERR_INVALID_ARGUMENT
    assert b"not available between acu_async_begin" in lib.acu_last_error(h).contents.message
    # unknown null_count would need a device count
    xd2 = dx.descriptor()
    xd2.null_count = -1
    st = lib.acu_arith(h, abi.I64, acu.ADD_WRAPPING, C.byref(xd2), C.byref(xd2), C.byref(out))
    assert st == abi.ERR_INVALID_ARGUMENT
    # more than 64 queued calls
    sts = [lib.acu_arith(h, abi.I64, acu.ADD_WRAPPING, C.byref(xd), C.byref(xd), C.byref(out)) for _ in range(70)]
    assert sts[:64] == [abi.OK] * 64 and sts[64] == abi.ERR_INVALID_ARGUMENT
    gpu.results_fetch()
    assert lib.acu_async_active(h) == 0
    assert out.len == 1000 and out.has_validity == 1 and out.null_count == x.null_count
    gpu._free_out(out)
    dx.free()
    # and the synchronous ABI works as before
    got = gpu.arith(acu.ADD_WRAPPING, x, x)
    assert got.null_count == x.null_count
