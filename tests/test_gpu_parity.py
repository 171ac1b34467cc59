"""Differential parity: the CUDA path (through the C ABI) vs the CPU oracle on seeded random,
sliced, ragged inputs — the reference's own fuzz pattern (fuzz_filter,
arrow-select/src/filter.rs:1888-1977: random lengths, offsets, null densities vs a naive oracle).

Bar: bit-exact for integer / byte / index / bitmap work, including the bytes written under
null slots and whether the result carries a NullBuffer at all; floating-point arithmetic is
compared bit-for-bit except that any NaN matches any NaN (tolerance stated by north_star:
1 ulp; we hold 0 ulp on non-NaN results). Float `sum` is order-dependent in the reference itself
(arrow-arith/src/aggregate.rs:303-313): it is held to the summation-tree error bound of
float_sum_bound, and to bit-exactness on order-independent inputs (test_gpu_reduce.py).
"""
import ctypes as C
import itertools
import math

import numpy as np
import pytest

import acu
from acu import _abi as abi
from acu import BOOL, HostArray

pytestmark = pytest.mark.gpu

INT_DTYPES = [abi.I8, abi.I16, abi.I32, abi.I64, abi.U8, abi.U16, abi.U32, abi.U64]
FLOAT_DTYPES = [abi.F32, abi.F64]
SIZES = [0, 1, 31, 32, 33, 63, 64, 65, 127, 128, 129, 1000, 4095, 4096, 4097, 8191, 12345, 70001]


def rand_values(rng, dtype, n, small=False):
    npdt = acu.NP_DTYPES[dtype]
    if dtype in FLOAT_DTYPES:
        v = (rng.random(n) * 2e6 - 1e6).astype(npdt)
        if n:
            specials = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan, 5e-324, 1.0, -1.0], dtype=npdt)
            k = max(1, n // 16)
            v[rng.integers(0, n, k)] = specials[rng.integers(0, len(specials), k)]
        return v
    info = np.iinfo(npdt)
    if small:
        lo, hi = max(info.min, -50), min(info.max, 50)
        return rng.integers(lo, hi, n, dtype=np.int64).astype(npdt)
    v = rng.integers(info.min, info.max, n, dtype=npdt, endpoint=True)
    if n:
        k = max(1, n // 16)
        edge = np.array([info.min, info.max, 0, 1, info.max - 1], dtype=npdt)
        v[rng.integers(0, n, k)] = edge[rng.integers(0, len(edge), k)]
    return v


def rand_array(rng, dtype, n, null_p, offset=0, small=False):
    """Random primitive array; `offset` > 0 builds a longer buffer and slices it (bit + element offsets)."""
    total = n + offset
    vals = rand_values(rng, dtype, total, small)
    mask = None if null_p is None else rng.random(total) >= null_p
    h = HostArray.from_numpy(dtype, vals, mask, bit_offset=int(rng.integers(0, 9)) if mask is not None else 0)
    return h.slice(offset, n) if offset else h


PRECISION = {abi.F32: 24, abi.F64: 53}
EXACT_KINDS = ("ints", "dyadic", "subnormal", "garbage_under_nulls")


def exact_float_array(rng, dtype, n, kind, null_p, offset=0):
    """A float array whose sum is exact in every association order -> (HostArray, expected sum as a Python float).

    Every value is k·2^e with Σ|k| <= 2^p over the whole buffer (p = 24 for f32, 53 for f64), so every partial sum
    of any subset, in any order, is representable: the only correct result is Σx itself, bit for bit, and +0.0 when
    Σx = 0 (the accumulator starts at T::ZERO). kinds: small integers (e = 0), dyadic fractions (e = -20),
    subnormals (e = the smallest subnormal exponent), and sparse valid integers with NaN / ±inf / huge values in every
    null slot. `offset` > 0 slices a longer buffer, like rand_array."""
    npdt = acu.NP_DTYPES[dtype]
    total = n + offset
    if kind == "garbage_under_nulls":
        null_p = 0.9 if null_p is None else max(null_p, 0.9)
    e = {"ints": 0, "dyadic": -20, "subnormal": -149 if dtype == abi.F32 else -1074, "garbage_under_nulls": 0}[kind]
    cap = 1000 if dtype == abi.F32 else 1 << 40
    kmax = max(1, min(cap, (1 << PRECISION[dtype]) // max(total, 1)))
    k = rng.integers(-kmax, kmax, total, endpoint=True)
    vals = np.ldexp(k.astype(np.float64), e).astype(npdt)
    mask = None if null_p is None else rng.random(total) >= null_p
    if kind == "garbage_under_nulls":
        junk = np.array([np.nan, -np.nan, np.inf, -np.inf, np.finfo(npdt).max, -np.finfo(npdt).max], dtype=npdt)
        vals[~mask] = junk[rng.integers(0, len(junk), int((~mask).sum()))]
    h = HostArray.from_numpy(dtype, vals, mask, bit_offset=int(rng.integers(0, 9)) if mask is not None else 0)
    if offset:
        h = h.slice(offset, n)
    valid = h.valid_mask()
    kk = k[offset:offset + n][valid]
    if kk.size == 0:
        return h, None
    return h, float(np.array(np.ldexp(float(int(kk.sum())), e), dtype=npdt))


def same_float(got, exp, dtype):
    """Bit-exact float comparison of two Python floats as `dtype` (so +0.0 != -0.0), any NaN matching any NaN."""
    if got is None or exp is None:
        return got is None and exp is None
    if np.isnan(exp):
        return bool(np.isnan(got))
    npdt = acu.NP_DTYPES[dtype]
    return np.array(got, dtype=npdt).tobytes() == np.array(exp, dtype=npdt).tobytes()


def rand_bool(rng, n, true_p, null_p, offset=0):
    total = n + offset
    bools = rng.random(total) < true_p
    mask = None if null_p is None else rng.random(total) >= null_p
    h = HostArray.bool_from_numpy(bools, mask, bit_offset=int(rng.integers(0, 9)), mask_offset=int(rng.integers(0, 9)))
    return h.slice(offset, n) if offset else h


def same_bits(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def assert_same(got, exp, what, float_nan_ok=False, exact_bytes=True):
    assert got.length == exp.length, f"{what}: length {got.length} != {exp.length}"
    assert (got.validity is None) == (exp.validity is None), f"{what}: NullBuffer presence differs"
    n = exp.length
    if exp.validity is not None:
        assert got.null_count == exp.null_count, f"{what}: null_count {got.null_count} != {exp.null_count}"
        assert np.array_equal(got.valid_mask(), exp.valid_mask()), f"{what}: validity bits differ"
    gv, ev = got.value_array(), exp.value_array()
    if not exact_bytes:  # logical equality only (arrow-data/src/equal/mod.rs:161-166)
        m = exp.valid_mask()
        gv, ev = gv[m], ev[m]
    if float_nan_ok and exp.dtype in FLOAT_DTYPES:
        gn, en = np.isnan(gv), np.isnan(ev)
        assert np.array_equal(gn, en), f"{what}: NaN positions differ"
        assert same_bits(gv[~gn], ev[~en]), f"{what}: non-NaN float bits differ"
    else:
        if not same_bits(gv[:n], ev[:n]):
            bad = np.nonzero(gv[:n] != ev[:n])[0]
            raise AssertionError(f"{what}: values differ at {bad[:8]}: {gv[bad[:8]]} vs {ev[bad[:8]]}")


UNIT_ROUNDOFF = {abi.F32: 2.0 ** -24, abi.F64: 2.0 ** -53}


def float_sum_bound(n, dtype, sm_count):
    """Relative forward-error bound of k_reduce's float sum over an n-row launch: |sum - Σx| <= bound · Σ|x|.

    Recursive summation whose evaluation tree has depth D errs by at most γ_D·Σ|x|, γ_D = D·u / (1 - D·u)
    (Higham, Accuracy and Stability of Numerical Algorithms, §4.2). D follows the design in reduce.cu's header:
    sgroups = ⌈n/2048⌉ super-groups, W = ⌈sgroups/8⌉ work blocks of one warp-per-super-group CTA of 8 warps, and a
    real grid between G_min = min(W, 8·sm_count) (at least one CTA per SM, one wave) and G_max = min(W, 64·sm_count)
    (at most 8 CTAs per SM, 8 waves). Along any path from a row to the result there are
      64·⌈sgroups / (8·G_min)⌉   adds into one lane's accumulator (2 rows per 64-row strip, 32 strips per super-group)
      + 5                        the warp's shuffle tree
      + 7                        the CTA's fold of its 8 warp partials
      + ⌈G_max / 32⌉             the last CTA's lane-strided fold of the per-CTA partials
      + 5                        the final shuffle tree,
    plus one for the rounding of the reference (math.fsum, correctly rounded in double). Below the grid cap
    G_min = G_max = W and the bound is exact for the launch; at 70001 rows D = 82 + 1."""
    if n == 0:
        return 0.0
    sgroups = -(-n // 2048)
    w = -(-sgroups // 8)
    g_min, g_max = min(w, 8 * sm_count), min(w, 64 * sm_count)
    depth = 64 * -(-sgroups // (8 * g_min)) + 5 + 7 + -(-g_max // 32) + 5 + 1
    u = UNIT_ROUNDOFF[dtype]
    return depth * u / (1 - depth * u)


def exact_fsum(x, chunk=1 << 20):
    """math.fsum over a float array without materialising it as one Python list."""
    return math.fsum(itertools.chain.from_iterable(x[i:i + chunk].tolist() for i in range(0, len(x), chunk)))


def assert_float_sum(got, values, valid, dtype, sm_count, what):
    """got = the device's float sum of an array of len(values) rows, valid rows marked by `valid`.
    IEEE outcomes that do not depend on the order are checked exactly (a valid NaN or both infinities: NaN; one
    infinity: that infinity; no valid row: None); finite sums against math.fsum within float_sum_bound."""
    x = np.asarray(values)[np.asarray(valid, dtype=bool)].astype(np.float64)
    if x.size == 0:
        assert got is None, f"{what}: {got} for a column without valid rows"
        return
    assert got is not None, f"{what}: None for {x.size} valid rows"
    pinf, ninf = bool((x == np.inf).any()), bool((x == -np.inf).any())
    if np.isnan(x).any() or (pinf and ninf):
        assert np.isnan(got), f"{what}: {got}, expected NaN"
    elif pinf or ninf:
        assert got == (np.inf if pinf else -np.inf), f"{what}: {got}, expected {'+' if pinf else '-'}inf"
    else:
        exact = exact_fsum(x)
        tol = float_sum_bound(len(values), dtype, sm_count) * float(np.abs(x).sum())
        assert abs(got - exact) <= tol, f"{what}: {got!r} vs fsum {exact!r}: error {abs(got - exact):.3g} > bound {tol:.3g}"


def expect_same_error(gpu, oracle, fn):
    try:
        exp = fn(oracle)
    except acu.ArrowError as e:
        with pytest.raises(acu.ArrowError) as gi:
            fn(gpu)
        assert gi.value.status == e.status
        assert str(gi.value) == str(e), f"{gi.value} != {e}"
        assert gi.value.index == e.index
        return None, None
    return fn(gpu), exp


# ---- filter ------------------------------------------------------------------------------
@pytest.mark.parametrize("width_dtype", [abi.I8, abi.I16, abi.I32, abi.I64, abi.F64])
@pytest.mark.parametrize("true_p", [0.0, 0.01, 0.1, 0.5, 0.9, 1.0])
def test_filter_primitive_fuzz(gpu, oracle, width_dtype, true_p):
    rng = np.random.default_rng(1000 + width_dtype * 17 + int(true_p * 100))
    for n in SIZES:
        for null_p, pred_null_p, off in [(None, None, 0), (0.05, None, 3), (0.5, 0.1, 1), (0.0, 0.3, 0)]:
            values = rand_array(rng, width_dtype, n + int(rng.integers(0, 3)), null_p, off)
            pred = rand_bool(rng, n, true_p, pred_null_p, off)
            got, exp = gpu.filter(values, pred), oracle.filter(values, pred)
            assert_same(got, exp, f"filter n={n} p={true_p} nulls={null_p}/{pred_null_p} off={off}")
            assert gpu.filter_plan(pred) == oracle.filter_plan(pred)


def test_filter_boolean_fuzz(gpu, oracle):
    rng = np.random.default_rng(7)
    for n in SIZES:
        for true_p in [0.1, 0.5, 0.95]:
            values = rand_bool(rng, n, 0.5, 0.2, 2)
            pred = rand_bool(rng, n, true_p, 0.1, 5)
            assert_same(gpu.filter(values, pred), oracle.filter(values, pred), f"filter_boolean n={n} p={true_p}")


def test_filter_predicate_shorter_and_longer(gpu, oracle):
    rng = np.random.default_rng(8)
    values = rand_array(rng, abi.I64, 5000, 0.1)
    pred = rand_bool(rng, 4000, 0.3, None)
    assert_same(gpu.filter(values, pred), oracle.filter(values, pred), "shorter predicate")
    pred = rand_bool(rng, 5001, 0.3, None)
    got, exp = expect_same_error(gpu, oracle, lambda be: be.filter(values, pred))
    assert got is None


@pytest.mark.parametrize("width", [16, 32])
def test_filter_wide_elements(gpu, oracle, width):
    """Decimal128/256-sized elements: modelled as `width`-byte records over uint64 lanes."""
    rng = np.random.default_rng(9 + width)
    lanes = width // 8
    for n in [0, 1, 100, 4097, 9000]:
        raw = rng.integers(0, 2**63, n * lanes, dtype=np.uint64)
        mask = rng.random(n) >= 0.2
        pred = rand_bool(rng, n, 0.3, None)
        # run through the C ABI directly with elem_bytes = width
        import ctypes as C
        from oracle import Oracle  # noqa: F401
        vals = HostArray(abi.U64, raw, n, acu.pack_bits(mask), 0, 0, int(n - mask.sum()))
        dv, dp = gpu.upload(HostArray(abi.U64, raw, n * lanes)), gpu.upload(pred)
        dn = gpu.malloc(len(vals.validity) + 8)
        gpu.h2d(dn, vals.validity)
        plan = C.c_void_p()
        pd = dp.descriptor()
        gpu.check(gpu.lib.acu_filter_plan_create(gpu.h, C.byref(pd), C.byref(plan)))
        count = gpu.lib.acu_filter_plan_count(plan)
        out = gpu.alloc_out(count * width, count)
        vd = abi.Array()
        vd.values, vd.validity, vd.validity_offset, vd.len, vd.null_count = dv.d_values, dn, 0, n, vals.null_count
        gpu.check(gpu.lib.acu_filter_primitive(gpu.h, plan, width, C.byref(vd), C.byref(out)))
        got_vals = gpu.d2h(out.values, count * width, np.uint64).reshape(count, lanes)
        sel = pred.value_array() & pred.valid_mask()
        assert np.array_equal(got_vals, raw.reshape(n, lanes)[sel])
        exp_valid = mask[sel]
        if out.has_validity:
            got_valid = acu.unpack_bits(gpu.d2h(out.validity, abi.bitmap_bytes(count)), 0, count)
            assert np.array_equal(got_valid, exp_valid) and out.null_count == int((~exp_valid).sum())
        else:
            assert exp_valid.all()
        gpu.lib.acu_filter_plan_destroy(gpu.h, plan)
        gpu._free_out(out)
        gpu.free(dn)
        dv.free()
        dp.free()


# ---- take --------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [abi.I8, abi.I16, abi.I32, abi.I64, abi.F64])
@pytest.mark.parametrize("idx_dtype", [abi.U8, abi.I8, abi.U16, abi.I16, abi.U32, abi.I32, abi.U64, abi.I64])
def test_take_primitive_fuzz(gpu, oracle, dtype, idx_dtype):
    rng = np.random.default_rng(2000 + dtype * 31 + idx_dtype)
    idx_max = min(int(np.iinfo(acu.NP_DTYPES[idx_dtype]).max), 100000)
    for nv in [1, 7, 100, 5000]:
        nv = min(nv, idx_max)
        for m in [0, 1, 33, 2047, 2048, 2049, 10000]:
            for vnull, inull, off in [(None, None, 0), (0.1, None, 0), (None, 0.2, 3), (0.3, 0.3, 2)]:
                values = rand_array(rng, dtype, nv, vnull, off)
                raw = rng.integers(0, nv, m + off).astype(acu.NP_DTYPES[idx_dtype])
                imask = None if inull is None else rng.random(m + off) >= inull
                if imask is not None and m:  # out-of-bounds values hidden under null index slots
                    hidden = np.nonzero(~imask)[0]
                    raw[hidden[: len(hidden) // 2]] = idx_max
                idx = HostArray.from_numpy(idx_dtype, raw, imask, bit_offset=int(rng.integers(0, 9)) if imask is not None else 0)
                if off:
                    idx = idx.slice(off, m)
                if imask is not None and nv > idx_max - 1:
                    continue
                got, exp = expect_same_error(gpu, oracle, lambda be: be.take(values, idx))
                if exp is not None:
                    assert_same(got, exp, f"take nv={nv} m={m} nulls={vnull}/{inull} off={off}")


def test_take_boolean_fuzz(gpu, oracle):
    rng = np.random.default_rng(11)
    for nv, m in [(10, 100), (1000, 5000), (70000, 33)]:
        values = rand_bool(rng, nv, 0.5, 0.2, 3)
        idx = HostArray.from_numpy(abi.U32, rng.integers(0, nv, m).astype(np.uint32), rng.random(m) >= 0.1)
        assert_same(gpu.take(values, idx), oracle.take(values, idx), f"take_boolean nv={nv} m={m}")


def test_take_out_of_bounds_contract(gpu, oracle):
    values = HostArray.from_list(abi.I64, [0, 1, 2, 3])
    for dt, bad in [(abi.U32, 1000), (abi.I32, -1), (abi.I64, -5), (abi.I8, -1), (abi.U64, 2**40)]:
        idx = HostArray.from_list(dt, [1, bad, 2])
        for cb in (False, True):
            got, exp = expect_same_error(gpu, oracle, lambda be: be.take(values, idx, cb))
            assert got is None and exp is None


# ---- variable width ------------------------------------------------------------------------
def rand_strings(rng, n, null_p):
    lens = rng.integers(0, 13, n)
    offsets = np.zeros(n + 1, dtype=np.int32)
    offsets[1:] = np.cumsum(lens)
    data = rng.integers(97, 123, int(offsets[-1]) + 16).astype(np.uint8)
    mask = rng.random(n) >= null_p if null_p is not None else None
    nulls = HostArray(abi.U8, np.zeros(0, np.uint8), n, None if mask is None else acu.pack_bits(mask), 0, 0,
                      0 if mask is None else int(n - mask.sum()))
    return offsets, data, nulls


def assert_same_bytes(got, exp, what):
    go, gd, gn = got
    eo, ed, en = exp
    assert np.array_equal(go, eo), f"{what}: offsets differ"
    assert np.array_equal(gd, ed), f"{what}: bytes differ"
    assert (gn.validity is None) == (en.validity is None), f"{what}: NullBuffer presence"
    if en.validity is not None:
        assert np.array_equal(gn.valid_mask(), en.valid_mask()) and gn.null_count == en.null_count


def test_take_bytes_fuzz(gpu, oracle):
    """Also the Dictionary<Int32,Utf8> -> Utf8 cast (arrow-cast/src/cast/dictionary.rs:310-317)."""
    rng = np.random.default_rng(12)
    for nv, m in [(1, 10), (50, 0), (4096, 20000), (300, 5000)]:
        for vnull, inull in [(None, None), (0.2, None), (None, 0.1), (0.2, 0.1)]:
            o, d, n = rand_strings(rng, nv, vnull)
            idx = HostArray.from_numpy(abi.I32, rng.integers(0, nv, m).astype(np.int32),
                                       None if inull is None else rng.random(m) >= inull)
            assert_same_bytes(gpu.take_bytes(o, d, n, idx), oracle.take_bytes(o, d, n, idx), f"take_bytes nv={nv} m={m}")


def test_filter_bytes_fuzz(gpu, oracle):
    rng = np.random.default_rng(13)
    for n in [0, 1, 100, 4096, 4097, 30000]:
        for true_p in [0.0, 0.1, 0.9, 1.0]:
            o, d, nulls = rand_strings(rng, n, 0.15)
            pred = rand_bool(rng, n, true_p, 0.05)
            assert_same_bytes(gpu.filter_bytes(o, d, nulls, pred), oracle.filter_bytes(o, d, nulls, pred),
                              f"filter_bytes n={n} p={true_p}")


def test_bytes_long_and_mixed_rows(gpu, oracle):
    """Rows longer than the 16-byte fast window, CTAs whose output exceeds the shared-memory staging
    buffer (direct-store path), empty rows, and i64 offsets (LargeUtf8) + every index width."""
    rng = np.random.default_rng(14)
    for n, max_len, odt in [(5000, 200, np.int32), (3000, 40, np.int64), (6000, 17, np.int32), (2500, 1, np.int32), (9000, 30, np.int32), (4100, 48, np.int32)]:
        lens = rng.integers(0, max_len + 1, n)
        lens[rng.random(n) < 0.2] = 0
        offsets = np.zeros(n + 1, dtype=odt)
        offsets[1:] = np.cumsum(lens)
        data = rng.integers(0, 256, int(offsets[-1]) + 16).astype(np.uint8)
        for null_p in (None, 0.1):
            mask = rng.random(n) >= null_p if null_p is not None else None
            nulls = HostArray(abi.U8, np.zeros(0, np.uint8), n, None if mask is None else acu.pack_bits(mask), 0, 0,
                              0 if mask is None else int(n - mask.sum()))
            pred = rand_bool(rng, n, 0.6, None)
            assert_same_bytes(gpu.filter_bytes(offsets, data, nulls, pred), oracle.filter_bytes(offsets, data, nulls, pred),
                              f"filter_bytes long n={n} max_len={max_len}")
            for idt in (abi.U32, abi.I64, abi.U16, abi.I8):
                hi = min(n, int(np.iinfo(acu.NP_DTYPES[idt]).max))
                m = 7000
                idx = HostArray.from_numpy(idt, rng.integers(0, hi, m).astype(acu.NP_DTYPES[idt]), rng.random(m) >= 0.1)
                assert_same_bytes(gpu.take_bytes(offsets, data, nulls, idx), oracle.take_bytes(offsets, data, nulls, idx),
                                  f"take_bytes long n={n} max_len={max_len} idx={idt}")


def test_bytes_many_blocks(gpu, oracle):
    """More 2048-row blocks than resident CTAs: the persistent copy kernel's three-stage load pipeline (indices two rounds
    ahead, offsets one round ahead) runs over several rounds per CTA, with blocks of short rows (shared-memory image path),
    blocks of long rows (direct path) and a ragged last block in the same launch."""
    rng = np.random.default_rng(16)
    n = 300_000
    lens = rng.integers(0, 25, n)
    lens[100_000:120_000] = rng.integers(30, 90, 20_000)  # a region of long rows
    offsets = np.zeros(n + 1, dtype=np.int32)
    offsets[1:] = np.cumsum(lens)
    data = rng.integers(0, 256, int(offsets[-1]) + 16).astype(np.uint8)
    mask = rng.random(n) >= 0.1
    nulls = HostArray(abi.U8, np.zeros(0, np.uint8), n, acu.pack_bits(mask), 0, 0, int(n - mask.sum()))
    m = 1_400_003
    iv = np.sort(rng.integers(0, n, m)).astype(np.uint32)  # monotone (filter-like) first half, random second half
    iv[m // 2:] = rng.integers(0, n, m - m // 2).astype(np.uint32)
    idx = HostArray.from_numpy(abi.U32, iv, rng.random(m) >= 0.05)
    assert_same_bytes(gpu.take_bytes(offsets, data, nulls, idx), oracle.take_bytes(offsets, data, nulls, idx), "take_bytes 1.4M rows")
    pred = rand_bool(rng, n, 0.7, None)
    big_o, big_d, big_n = gpu.take_bytes(offsets, data, nulls, idx)
    pred2 = rand_bool(rng, m, 0.6, 0.02)
    assert_same_bytes(gpu.filter_bytes(big_o, big_d, big_n, pred2), oracle.filter_bytes(big_o, big_d, big_n, pred2), "filter_bytes 1.4M rows")
    assert_same_bytes(gpu.filter_bytes(offsets, data, nulls, pred), oracle.filter_bytes(offsets, data, nulls, pred), "filter_bytes 300k rows")


def test_dictionary_filter_take_on_keys(gpu, oracle):
    """filter_dict (filter.rs:999-1007) and take_dict (take.rs:932-938) touch only the KEYS and share the dictionary
    values, so at the C ABI a dictionary column is its Int32 key array: decode(filter(keys)) == filter(decode(keys)),
    and the same for take (decode = the Dictionary<Int32,Utf8> -> Utf8 cast, dictionary.rs:310-317)."""
    rng = np.random.default_rng(15)
    d_off, d_data, d_nulls = rand_strings(rng, 300, 0.1)  # the dictionary (with null entries)
    for n in [0, 1, 1000, 20000]:
        keys = HostArray.from_numpy(abi.I32, rng.integers(0, 300, n).astype(np.int32), rng.random(n) >= 0.1)
        decoded = gpu.take_bytes(d_off, d_data, d_nulls, keys)
        pred = rand_bool(rng, n, 0.3, 0.05)
        fk = gpu.filter(keys, pred)
        assert_same(fk, oracle.filter(keys, pred), f"filter_dict keys n={n}")
        assert_same_bytes(gpu.take_bytes(d_off, d_data, d_nulls, fk), gpu.filter_bytes(decoded[0], decoded[1], decoded[2], pred), f"filter_dict n={n}")
        if n:
            idx = HostArray.from_numpy(abi.U32, rng.integers(0, n, 777).astype(np.uint32), rng.random(777) >= 0.1)
            tk = gpu.take(keys, idx)
            assert_same(tk, oracle.take(keys, idx), f"take_dict keys n={n}")
            assert_same_bytes(gpu.take_bytes(d_off, d_data, d_nulls, tk), gpu.take_bytes(decoded[0], decoded[1], decoded[2], idx), f"take_dict n={n}")


def test_take_bytes_offset_overflow(gpu, oracle):
    """take.rs:2877-2910 test_take_bytes_offset_overflow(_nullable): one 1 MB value selected i32::MAX / 1e6 + 1 times
    => Err(OffsetOverflowError(capacity)) on the no-null fast path and on the nullable path, with the reference's
    capacity (the running total at the first index that no longer fits i32). Sizing mode: no bytes are copied."""
    value_len = 1_000_000
    n = (2**31 - 1) // value_len + 1
    offsets = np.array([0, value_len], dtype=np.int32)
    data = np.full(value_len + 16, ord("a"), dtype=np.uint8)
    nulls = HostArray(abi.U8, np.zeros(0, np.uint8), 1, None, 0, 0, 0)
    for idx in (HostArray.from_numpy(abi.I32, np.zeros(n, dtype=np.int32)),
                HostArray.from_numpy(abi.I32, np.zeros(n + 1, dtype=np.int32), np.arange(n + 1) != 0)):
        errs = []
        for be in (gpu, oracle):
            with pytest.raises(acu.ArrowError) as e:
                be.take_bytes(offsets, data, nulls, idx)
            errs.append(e.value)
        assert errs[0].status == errs[1].status == abi.ERR_OFFSET_OVERFLOW
        assert str(errs[0]) == str(errs[1]) == f"Offset overflow error: {n * value_len}"


# ---- 16 / 32-byte elements: Decimal128/256, intervals, and Utf8View / BinaryView ----------------
def _wide_column(gpu, raw_u64, n, width, mask):
    """Device descriptor of n `width`-byte records (given as uint64 lanes) with an optional validity mask."""
    import ctypes as C  # noqa: F401
    dv = gpu.malloc(raw_u64.nbytes + 64)
    if raw_u64.nbytes:
        gpu.h2d(dv, raw_u64)
    dn = None
    if mask is not None:
        bits = acu.pack_bits(mask)
        dn = gpu.malloc(len(bits) + 8)
        gpu.h2d(dn, bits)
    a = abi.Array()
    a.values, a.validity, a.len, a.null_count = dv, dn, n, 0 if mask is None else int(n - mask.sum())
    return a, [p for p in (dv, dn) if p]


def _wide_result(gpu, out, width):
    n = out.len
    vals = gpu.d2h(out.values, n * width, np.uint64).reshape(n, width // 8)
    valid = acu.unpack_bits(gpu.d2h(out.validity, abi.bitmap_bytes(n)), 0, n) if out.has_validity else np.ones(n, dtype=bool)
    return vals, valid


@pytest.mark.parametrize("width", [16, 32])
def test_take_wide_elements(gpu, oracle, width):
    import ctypes as C
    rng = np.random.default_rng(90 + width)
    lanes = width // 8
    for n, m in [(1, 5), (100, 0), (4097, 9000), (9000, 4097)]:
        raw = rng.integers(0, 2**63, n * lanes, dtype=np.uint64)
        mask = rng.random(n) >= 0.2
        col, owned = _wide_column(gpu, raw, n, width, mask)
        idx_h = HostArray.from_numpy(abi.U32, rng.integers(0, n, m).astype(np.uint32), rng.random(m) >= 0.1)
        di = gpu.upload(idx_h)
        out = gpu.alloc_out(m * width, m)
        idd = di.descriptor()
        gpu.check(gpu.lib.acu_take_primitive(gpu.h, width, C.byref(col), C.byref(idd), abi.U32, 0, C.byref(out)))
        vals, valid = _wide_result(gpu, out, width)
        ix, iv = idx_h.value_array(), idx_h.valid_mask()
        assert np.array_equal(valid, mask[ix] & iv)
        assert np.array_equal(vals[iv], raw.reshape(n, lanes)[ix[iv]])  # the value is gathered wherever the index is valid
        gpu._free_out(out)
        di.free()
        for p in owned:
            gpu.free(p)


def test_byte_view_filter_take(gpu, oracle):
    """Utf8View / BinaryView: filter_byte_view (filter.rs:931-944) and take_byte_view (take.rs:630-640) run
    filter_native / take_native over the 16-byte views and share the data buffers, i.e. they ARE the 16-byte primitive
    kernels. Views are built here as arrow's u128 layout (len | 12 inline bytes, or len | prefix | buffer | offset)."""
    import ctypes as C
    rng = np.random.default_rng(77)
    n = 6000
    strings = ["".join(chr(c) for c in rng.integers(97, 123, rng.integers(0, 30))) for _ in range(n)]
    buf = bytearray()
    views = np.zeros((n, 4), dtype=np.uint32)
    for i, s in enumerate(strings):
        b = s.encode()
        views[i, 0] = len(b)
        if len(b) <= 12:
            views[i, 1:4] = np.frombuffer(b.ljust(12, b"\0"), dtype=np.uint32)
        else:
            views[i, 1] = np.frombuffer(b[:4], dtype=np.uint32)[0]
            views[i, 2], views[i, 3] = 0, len(buf)
            buf += b

    def decode(v):
        out = []
        for row in v.view(np.uint32).reshape(-1, 4):
            ln = int(row[0])
            out.append(row[1:4].tobytes()[:ln].decode() if ln <= 12 else bytes(buf[int(row[3]): int(row[3]) + ln]).decode())
        return out

    mask = rng.random(n) >= 0.1
    col, owned = _wide_column(gpu, views.view(np.uint64).reshape(-1), n, 16, mask)
    pred = rand_bool(rng, n, 0.3, 0.05)
    dp = gpu.upload(pred)
    plan = C.c_void_p()
    pd = dp.descriptor()
    gpu.check(gpu.lib.acu_filter_plan_create(gpu.h, C.byref(pd), C.byref(plan)))
    count = gpu.lib.acu_filter_plan_count(plan)
    out = gpu.alloc_out(count * 16, count)
    gpu.check(gpu.lib.acu_filter_primitive(gpu.h, plan, 16, C.byref(col), C.byref(out)))
    vals, valid = _wide_result(gpu, out, 16)
    sel = pred.value_array() & pred.valid_mask()
    assert decode(vals) == [s for s, k in zip(strings, sel) if k] and np.array_equal(valid, mask[sel])
    gpu.lib.acu_filter_plan_destroy(gpu.h, plan)
    gpu._free_out(out)
    idx_h = HostArray.from_numpy(abi.I64, rng.integers(0, n, 5000).astype(np.int64))
    di = gpu.upload(idx_h)
    out = gpu.alloc_out(5000 * 16, 5000)
    idd = di.descriptor()
    gpu.check(gpu.lib.acu_take_primitive(gpu.h, 16, C.byref(col), C.byref(idd), abi.I64, 1, C.byref(out)))
    vals, valid = _wide_result(gpu, out, 16)
    assert decode(vals) == [strings[i] for i in idx_h.value_array()] and np.array_equal(valid, mask[idx_h.value_array()])
    gpu._free_out(out)
    di.free()
    dp.free()
    for p in owned:
        gpu.free(p)


def test_arith_in_place(gpu, oracle):
    """binary_mut / unary_mut (arrow-arith/src/arity.rs:137-252,301-363): the output aliases the first operand's buffers."""
    rng = np.random.default_rng(99)
    for dtype in (abi.I64, abi.F64, abi.I32):
        for n in (1, 64, 4097, 70001):
            a, b = rand_array(rng, dtype, n, 0.1, 0), rand_array(rng, dtype, n, 0.05, 0)
            exp = oracle.arith(acu.MUL_WRAPPING, a, b)
            da, db = gpu.upload(a), gpu.upload(b)
            ad, bd = da.descriptor(), db.descriptor()
            out = abi.ArrayOut()
            out.values = ad.values
            aliased_validity = ad.validity_offset == 0
            out.validity = ad.validity if aliased_validity else gpu.malloc(acu.bitmap_bytes(n) + 8)
            gpu.check(gpu.lib.acu_arith(gpu.h, dtype, acu.MUL_WRAPPING, C.byref(ad), C.byref(bd), C.byref(out)))
            vals = gpu.d2h(out.values, n * abi.DTYPE_SIZE[dtype], acu.NP_DTYPES[dtype])
            validity = gpu.d2h(out.validity, acu.bitmap_bytes(n)) if out.has_validity else None
            got = HostArray(dtype, vals, n, validity, 0, 0, out.null_count if out.has_validity else 0)
            assert_same(got, exp, f"in-place mul dtype={dtype} n={n}", float_nan_ok=True)
            if not aliased_validity:
                gpu.free(out.validity)
            da.free()
            db.free()


# ---- numeric -------------------------------------------------------------------------------
ARITH_OPS = ["add", "add_wrapping", "sub", "sub_wrapping", "mul", "mul_wrapping", "div", "rem"]


@pytest.mark.parametrize("dtype", INT_DTYPES + FLOAT_DTYPES)
@pytest.mark.parametrize("op", ARITH_OPS)
def test_arith_fuzz(gpu, oracle, dtype, op):
    rng = np.random.default_rng(3000 + dtype * 13 + ARITH_OPS.index(op))
    for n in [0, 1, 63, 64, 65, 255, 256, 257, 1000, 5000, 33333]:
        for an, bn, off, small in [(None, None, 0, True), (0.1, None, 1, True), (0.1, 0.2, 3, False), (0.0, 0.0, 0, True),
                                   (None, None, 1, False)]:
            a = rand_array(rng, dtype, n, an, off, small)
            b = rand_array(rng, dtype, n, bn, off and 2, small)
            got, exp = expect_same_error(gpu, oracle, lambda be: getattr(be, op)(a, b))
            if exp is not None:
                assert_same(got, exp, f"{op} dtype={dtype} n={n} nulls={an}/{bn} off={off}", float_nan_ok=True)


@pytest.mark.parametrize("dtype", [abi.I32, abi.I64, abi.U64, abi.F32, abi.F64])
@pytest.mark.parametrize("op", ARITH_OPS)
def test_arith_scalar_fuzz(gpu, oracle, dtype, op):
    rng = np.random.default_rng(4000 + dtype * 13 + ARITH_OPS.index(op))
    for n in [0, 1, 100, 4097]:
        for null_p in [None, 0.2]:
            arr = rand_array(rng, dtype, n, null_p, 1, small=True)
            for sv in [rand_array(rng, dtype, 1, None, 0, small=True).scalar(), HostArray.from_list(dtype, [None]).scalar()]:
                for fn in (lambda be: getattr(be, op)(arr, sv), lambda be: getattr(be, op)(sv, arr)):
                    got, exp = expect_same_error(gpu, oracle, fn)
                    if exp is not None:
                        assert_same(got, exp, f"{op} scalar dtype={dtype} n={n}", float_nan_ok=True)


@pytest.mark.parametrize("dtype", [abi.I8, abi.I32, abi.I64, abi.F32, abi.F64])
def test_neg_fuzz(gpu, oracle, dtype):
    rng = np.random.default_rng(5000 + dtype)
    for n in [0, 1, 100, 5000]:
        for null_p in [None, 0.3]:
            a = rand_array(rng, dtype, n, null_p, 2)
            for checked in (True, False):
                got, exp = expect_same_error(gpu, oracle, lambda be: be.neg(a, checked))
                if exp is not None:
                    assert_same(got, exp, f"neg dtype={dtype} n={n} checked={checked}", float_nan_ok=True)


# ---- cmp -----------------------------------------------------------------------------------
CMP_OPS = ["eq", "neq", "lt", "lt_eq", "gt", "gt_eq", "distinct", "not_distinct"]


@pytest.mark.parametrize("dtype", [abi.I8, abi.I32, abi.I64, abi.U32, abi.U64, abi.F32, abi.F64])
@pytest.mark.parametrize("op", CMP_OPS)
def test_cmp_fuzz(gpu, oracle, dtype, op):
    rng = np.random.default_rng(6000 + dtype * 13 + CMP_OPS.index(op))
    for n in [0, 1, 63, 64, 65, 1000, 4097, 20000]:
        for an, bn, off in [(None, None, 0), (0.1, None, 1), (0.1, 0.2, 3), (0.0, 0.0, 0)]:
            a = rand_array(rng, dtype, n, an, off, small=True)
            b = rand_array(rng, dtype, n, bn, off, small=True)
            got, exp = gpu.cmp(abi.EQ + CMP_OPS.index(op), a, b), oracle.cmp(abi.EQ + CMP_OPS.index(op), a, b)
            assert_same(got, exp, f"{op} dtype={dtype} n={n} nulls={an}/{bn}")
        if n:
            arr = rand_array(rng, dtype, n, 0.2, 1, small=True)
            for sv in [rand_array(rng, dtype, 1, None, 0, small=True).scalar(), HostArray.from_list(dtype, [None]).scalar()]:
                for x, y in ((arr, sv), (sv, arr), (sv, sv)):
                    code = abi.EQ + CMP_OPS.index(op)
                    assert_same(gpu.cmp(code, x, y), oracle.cmp(code, x, y), f"{op} scalar dtype={dtype} n={n}", exact_bytes=False)


# ---- cast ----------------------------------------------------------------------------------
@pytest.mark.parametrize("frm", INT_DTYPES + FLOAT_DTYPES)
@pytest.mark.parametrize("to", INT_DTYPES + FLOAT_DTYPES)
def test_cast_fuzz(gpu, oracle, frm, to):
    rng = np.random.default_rng(7000 + frm * 10 + to)
    for n in [0, 1, 65, 1000, 4097]:
        for null_p in [None, 0.1]:
            a = rand_array(rng, frm, n, null_p, 1)
            assert_same(gpu.cast(a, to), oracle.cast(a, to), f"cast {frm}->{to} n={n}", float_nan_ok=True)
            got, exp = expect_same_error(gpu, oracle, lambda be: be.cast(a, to, safe=False))
            if exp is not None:
                assert_same(got, exp, f"cast unsafe {frm}->{to} n={n}", float_nan_ok=True)


# ---- boolean (arrow-arith/src/boolean.rs) ----------------------------------------------------
@pytest.mark.parametrize("op", ["and_", "or_", "and_not", "and_kleene", "or_kleene"])
def test_boolean_binary_fuzz(gpu, oracle, op):
    rng = np.random.default_rng(6000 + len(op))
    for n in SIZES:
        for an, bn in [(None, None), (0.2, None), (None, 0.2), (0.3, 0.3), (0.0, None)]:
            a, b = rand_bool(rng, n, 0.5, an, offset=int(rng.integers(0, 70))), rand_bool(rng, n, 0.4, bn, offset=int(rng.integers(0, 9)))
            assert_same(getattr(gpu, op)(a, b), getattr(oracle, op)(a, b), f"{op} n={n} nulls=({an},{bn})")
    got, exp = expect_same_error(gpu, oracle, lambda be: getattr(be, op)(rand_bool(np.random.default_rng(1), 5, 0.5, None), rand_bool(np.random.default_rng(2), 6, 0.5, None)))
    assert got is None and exp is None


def test_boolean_unary_fuzz(gpu, oracle):
    rng = np.random.default_rng(6100)
    for n in SIZES:
        for null_p in (None, 0.25, 1.0):
            a = rand_bool(rng, n, 0.5, null_p, offset=int(rng.integers(0, 70)))
            assert_same(gpu.not_(a), oracle.not_(a), f"not n={n}")
            for src in (a, rand_array(rng, abi.I64, n, null_p, offset=3), rand_array(rng, abi.I8, n, null_p)):
                assert_same(gpu.is_null(src), oracle.is_null(src), f"is_null n={n}")
                assert_same(gpu.is_not_null(src), oracle.is_not_null(src), f"is_not_null n={n}")


def test_predicate_pipeline_on_device(gpu, oracle):
    """cmp -> and_kleene -> filter: the mask a query engine builds, then applies (SURVEY.md §8(f) rank 2)."""
    rng = np.random.default_rng(6200)
    n = 50_000
    x, y = rand_array(rng, abi.F64, n, 0.1), rand_array(rng, abi.F64, n, 0.1)
    k = rand_array(rng, abi.I64, n, 0.05, small=True)
    zero = HostArray.from_list(abi.I64, [0], scalar=True)
    for be_name in ("gpu",):
        mask_g = gpu.and_kleene(gpu.lt(x, y), gpu.gt_eq(k, zero))
        mask_o = oracle.and_kleene(oracle.lt(x, y), oracle.gt_eq(k, zero))
        assert_same(mask_g, mask_o, "predicate")
        assert_same(gpu.filter(k, mask_g), oracle.filter(k, mask_o), "filter by device-built predicate")


# ---- aggregate -----------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [abi.I8, abi.I32, abi.I64, abi.U64, abi.F32, abi.F64])
def test_aggregate_fuzz(gpu, oracle, dtype):
    rng = np.random.default_rng(8000 + dtype)
    for n in [0, 1, 63, 64, 65, 1000, 70001]:
        for null_p in [None, 0.1, 1.0]:
            a = rand_array(rng, dtype, n, null_p, 1)
            for op in ("min", "max"):
                g, e = getattr(gpu, op)(a), getattr(oracle, op)(a)
                if isinstance(e, float) and np.isnan(e):
                    assert np.isnan(g) and np.signbit(g) == np.signbit(e)
                else:
                    assert g == e, f"{op} dtype={dtype} n={n}: {g} != {e}"
            if dtype in FLOAT_DTYPES:  # order-dependent: finite inputs, the summation-tree error bound
                vals = (rng.random(n) * 2e3 - 1e3).astype(acu.NP_DTYPES[dtype])
                b = HostArray.from_numpy(dtype, vals, None if null_p is None else rng.random(n) >= null_p)
                g = gpu.sum(b)
                assert (g is None) == (oracle.sum(b) is None)
                assert_float_sum(g, vals, b.valid_mask(), dtype, gpu.lib.acu_device_sm_count(gpu.h), f"sum dtype={dtype} n={n}")
            else:
                assert gpu.sum(a) == oracle.sum(a), f"sum dtype={dtype} n={n}"


@pytest.mark.parametrize("dtype", [abi.I8, abi.I16, abi.I32, abi.I64, abi.U8, abi.U32, abi.U64])
def test_sum_checked_fuzz(gpu, oracle, dtype):
    """sum_checked = the in-order checked fold (aggregate.rs:897-937): same value, or the same error text / failing row /
    operands as the oracle's sequential fold — including prefixes that overflow while the total would fit."""
    rng = np.random.default_rng(8100 + dtype)
    npdt = acu.NP_DTYPES[dtype]
    info = np.iinfo(npdt)
    for n in [0, 1, 15, 16, 17, 4095, 4096, 4097, 20000, 70001]:
        for null_p in (None, 0.2, 1.0):
            for regime in ("small", "edge", "full"):
                if regime == "small":      # never overflows
                    span = max(1, int(info.max // max(n, 1) // 2))
                    vals = rng.integers(max(info.min, -span), span, n, dtype=np.int64 if info.min < 0 else np.uint64, endpoint=True).astype(npdt)
                elif regime == "edge":     # mostly zeros with a few extreme values: late, sparse overflows
                    vals = np.zeros(n, dtype=npdt)
                    if n:
                        k = max(1, n // 500)
                        vals[rng.integers(0, n, k)] = rng.choice(np.array([info.max, info.min, info.max - 1, 1], dtype=npdt), k)
                else:
                    vals = rng.integers(info.min, info.max, n, dtype=npdt, endpoint=True)
                a = HostArray.from_numpy(dtype, vals, None if null_p is None else rng.random(n) >= null_p, bit_offset=int(rng.integers(0, 9)))
                if n > 40:
                    a = a.slice(7, n - 20)
                got, exp = expect_same_error(gpu, oracle, lambda be: be.sum_checked(a))
                assert got == exp, f"sum_checked dtype={dtype} n={n} {regime}: {got} != {exp}"


def test_generators_match_host_twin(gpu, oracle):
    import ctypes as C
    n = 100003
    for kind, npdt, param in [(0, np.uint64, 0), (1, np.int64, 0), (2, np.float64, 0), (3, np.uint32, 12345), (4, np.int32, 777)]:
        d = gpu.malloc(n * 8)
        gpu.check(gpu.lib.acu_generate_values(gpu.h, kind, 42, 1000, param, d, n))
        got = gpu.d2h(d, n * np.dtype(npdt).itemsize, npdt)
        gpu.free(d)
        assert same_bits(got, oracle.generate_values(kind, 42, 1000, param, n, npdt))
    d = gpu.malloc(abi.bitmap_bytes(n))
    gpu.check(gpu.lib.acu_generate_bits(gpu.h, 46, 5, 0.1, d, n))
    got = acu.unpack_bits(gpu.d2h(d, abi.bitmap_bytes(n)), 0, n)
    gpu.free(d)
    assert np.array_equal(got, acu.unpack_bits(oracle.generate_bits(46, 5, 0.1, n), 0, n))
    cnt = C.c_int64(0)
