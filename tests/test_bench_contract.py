"""The reference arm of bench.py is runnable without a GPU: its JSON line must carry the contract's keys
(metric / unit / config shared with the GPU arm, cpu_baseline describing the run, a zero-copy e2e object)."""
import json
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_reference(extra_env=None, args=()):
    env = dict(os.environ)
    env.update(extra_env or {})
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-rows", "300000", *args],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout


def test_reference_arm_line():
    lines = [ln for ln in run_reference().splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    base = json.load(open(os.path.join(REPO, "BASELINE.json")))
    assert d["impl"] == "reference" and d["metric"] == base["metric"] and d["unit"] == "Mrows/s"
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb and cb["unit"] == "Mrows/s"
    assert d["e2e"] == {"value": d["value"], "unit": "Mrows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0


def test_reference_arm_other_ranks_exit_quietly():
    """Under torchrun (N > 1) rank 0 alone runs and prints the reference arm."""
    out = run_reference({"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, ("--gpus", "2"))
    assert out.strip() == ""


def test_refbench_checksums_match_single_call_oracle():
    """oracle/refbench.cpp (the native multi-threaded harness behind cpu_baseline / --impl reference) must compute exactly
    what one oracle call per op over the whole table computes: its folded checksums are partition-independent."""
    sys.path.insert(0, os.path.join(REPO, "arrow-rs_b200"))
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import numpy as np
    import acu
    from acu import _abi as abi
    from acu import HostArray, BOOL
    from oracle import Oracle, RefBench
    n, seeds = 200_003, (42, 42, 43, 44, 144, 45, 46)
    orc = Oracle()
    chks = []
    for threads in (1, 3, 8):
        with RefBench(n, seeds, 0.1, 0.05, threads=threads, oracle=orc) as rb:
            _, bits, valid = rb.step()
            c = rb.check()
            c["sum_bits"], c["valid_rows"] = bits, valid
            chks.append(c)
    assert chks[0] == chks[1] == chks[2]
    # the same quantities from single calls through the Python oracle wrapper
    col = HostArray(abi.I64, orc.generate_values(0, 42, 0, 0, n, np.int64), n, orc.generate_bits(44, 0, 0.95, n), 0, 0, -1)
    pred = HostArray(BOOL, orc.generate_bits(46, 0, 0.1, n), n, None, 0, 0, 0)
    a = HostArray(abi.F64, orc.generate_values(2, 42, 0, 0, n, np.float64), n, orc.generate_bits(144, 0, 0.95, n), 0, 0, -1)
    b = HostArray(abi.F64, orc.generate_values(2, 43, 0, 0, n, np.float64), n, orc.generate_bits(45, 0, 0.95, n), 0, 0, -1)
    f = orc.filter(col, pred)
    idx = HostArray.from_numpy(abi.U32, np.nonzero(pred.value_array())[0].astype(np.uint32))
    t = orc.take(col, idx)
    s = orc.add(a, b)
    wsum = lambda x: int(np.asarray(x).view(np.uint64).sum(dtype=np.uint64))  # noqa: E731
    c = chks[0]
    assert c["filter_rows"] == f.length and c["filter_nulls"] == f.null_count and c["filter_values_wsum"] == wsum(f.values[: f.length])
    assert c["take_nulls"] == t.null_count and c["take_values_wsum"] == wsum(t.values[: t.length])
    assert c["add_nulls"] == s.null_count and c["add_bits_wsum"] == wsum(s.values[: s.length])
    total = orc.sum(t)
    assert c["sum_bits"] == (int(total) & 0xFFFFFFFFFFFFFFFF) and c["valid_rows"] == t.length - t.null_count


@pytest.mark.parametrize("args, message", [(("--steps", "0"), "--steps must be at least 1"),
                                           (("--impl", "reference", "--dump-outputs", "out"), "--dump-outputs writes the GPU arm")])
def test_bench_rejects_bad_arguments(args, message):
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *args], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and message in r.stderr and not r.stdout


def test_dump_rows_is_a_fixed_sample():
    sys.path.insert(0, REPO)
    import numpy as np
    import bench
    assert np.array_equal(bench.dump_rows(1000), np.arange(1000))
    rows = bench.dump_rows(10 ** 9)
    assert len(rows) == bench.DUMP_ROWS and np.array_equal(rows, bench.dump_rows(10 ** 9))
    assert np.all(np.diff(rows) > 0) and rows[-1] < 10 ** 9 and np.all(rows[:: bench.DUMP_BLOCK] % 8 == 0)


@pytest.mark.gpu
def test_dump_outputs_are_the_steps_outputs(tmp_path):
    """--dump-outputs writes the last timed step's filter / take / add outputs (values and validity) and sum, all finite and
    equal to the oracle's on the same seeded table: at 3e6 rows the add output (3e6 rows) is a sample, the filter and take
    outputs are whole."""
    sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, "arrow-rs_b200"))
    sys.path.insert(0, os.path.join(REPO, "tests"))
    import numpy as np
    import bench
    from acu import _abi as abi
    from acu import HostArray, BOOL
    from oracle import Oracle
    n, out = 3_000_000, tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--rows", str(n), "--steps", "2", "--warmup", "1", "--no-e2e",
                        "--no-cpu", "--no-configs", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert line["steps"] == 2
    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert sorted(got) == ["add", "add_valid", "counts", "filter", "filter_valid", "sum", "take", "take_valid"]
    assert all(v.dtype == (np.float32 if k.endswith("_valid") else np.float64) for k, v in got.items())
    assert all(np.isfinite(v).all() for v in got.values()) and sum(v.nbytes for v in got.values()) <= 64 << 20
    orc = Oracle()
    col = HostArray(abi.I64, orc.generate_values(0, 42, 0, 0, n, np.int64), n, orc.generate_bits(44, 0, 0.95, n), 0, 0, -1)
    pred = HostArray(BOOL, orc.generate_bits(46, 0, 0.1, n), n, None, 0, 0, 0)
    a = HostArray(abi.F64, orc.generate_values(2, 42, 0, 0, n, np.float64), n, orc.generate_bits(144, 0, 0.95, n), 0, 0, -1)
    b = HostArray(abi.F64, orc.generate_values(2, 43, 0, 0, n, np.float64), n, orc.generate_bits(45, 0, 0.95, n), 0, 0, -1)
    idx = HostArray.from_numpy(abi.U32, np.nonzero(pred.value_array())[0].astype(np.uint32))
    expect = {"filter": orc.filter(col, pred), "take": orc.take(col, idx), "add": orc.add(a, b)}
    counts = []
    for name, e in expect.items():
        x, v = e.value_array()[: e.length].astype(np.float64), e.valid_mask()
        x[~v] = 0.0
        rows = bench.dump_rows(e.length)
        assert np.array_equal(got[name], x[rows]) and np.array_equal(got[name + "_valid"], v[rows].astype(np.float32)), name
        counts += [e.length, e.null_count]
    assert len(got["add"]) == bench.DUMP_ROWS < n and len(got["filter"]) == expect["filter"].length
    total = orc.sum(expect["take"])
    assert got["sum"].tolist() == [float(total)]
    assert got["counts"].tolist() == counts + [expect["take"].length - expect["take"].null_count]
