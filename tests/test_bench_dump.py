"""bench.py --dump-outputs: the rows of the last timed step, for a fixed sample of reads, as float .npy files that two builds can be
compared by.  CPU: the sampling, gathering and size cap of dump_outputs on a synthetic result whose CIGAR words lie out of order in
their pool.  GPU: the option end to end on the timed path, against the step's digest and the oracle's rows for the same reads."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from oracle_lib import ROW_DTYPE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _result(n_reads, seed=5):
    rng = np.random.default_rng(seed)
    counts = rng.integers(0, 4, size=n_reads)
    row_off = np.concatenate(([0], np.cumsum(counts))).astype(np.uint64)
    n_rows = int(row_off[-1])
    rows = np.zeros(n_rows, dtype=ROW_DTYPE)
    for name in rows.dtype.names:
        rows[name] = rng.integers(0, 1 << 20, size=n_rows).astype(rows.dtype[name])
    rows["hash"] = rng.integers(0, np.iinfo(np.uint64).max, size=n_rows, dtype=np.uint64)
    rows["ref_id"] = rng.integers(np.iinfo(np.int64).min, np.iinfo(np.int64).max, size=n_rows, dtype=np.int64)
    rows["n_cigar"] = rng.integers(1, 6, size=n_rows)
    perm = rng.permutation(n_rows)                      # rows' CIGAR words in a shuffled pool order
    sizes = rows["n_cigar"].astype(np.int64)[perm]
    rows["cigar_off"][perm] = np.concatenate(([0], np.cumsum(sizes)[:-1]))
    cigar = rng.integers(0, 1 << 20, size=int(sizes.sum())).astype(np.uint32)
    return row_off, rows, cigar


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def _restore(d):
    """The dump back in the library's types: (row_off, rows, cigar words in row order)."""
    row_off = np.concatenate(([0], np.cumsum(d["rows_per_read"]))).astype(np.uint64)
    rows = np.zeros(len(d["row_score"]), dtype=ROW_DTYPE)
    for name in ROW_DTYPE.names:
        t = ROW_DTYPE[name]
        if name == "cigar_off":
            continue
        if t.kind in "iu" and t.itemsize == 8:
            rows[name] = d["row_%s_hi" % name].astype(np.int64).astype(t) << t.type(32) | d["row_%s_lo" % name].astype(t)
        else:
            rows[name] = d["row_" + name].astype(t)
    return row_off, rows, d["cigar"].astype(np.uint32)


def _digest(row_off, rows, cigar):
    """bench.rows_digest of a result whose CIGAR words are stored in row order."""
    dg = hashlib.sha1()
    dg.update(row_off.tobytes())
    for name in rows.dtype.names:
        if name != "cigar_off":
            dg.update(np.ascontiguousarray(rows[name]).tobytes())
    dg.update(cigar.tobytes())
    return dg.hexdigest()


def test_dump_outputs_sample(tmp_path):
    row_off, rows, cigar = _result(3000)
    pick = bench.dump_sample(3000, 150)
    assert np.array_equal(pick, np.arange(3000))
    nbytes = bench.dump_outputs(str(tmp_path / "a"), pick, row_off, rows, cigar)
    bench.dump_outputs(str(tmp_path / "b"), pick, row_off, rows, cigar)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)
    assert sum(x.nbytes for x in a.values()) == nbytes <= bench.DUMP_BYTES
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert "row_cigar_off" not in a
    r_off, r_rows, r_cig = _restore(a)
    assert np.array_equal(r_off, row_off)
    for name in ROW_DTYPE.names:
        if name != "cigar_off":
            assert np.array_equal(r_rows[name], rows[name]), name
    want = np.concatenate([cigar[int(o):int(o) + int(c)] for o, c in zip(rows["cigar_off"], rows["n_cigar"])])
    assert np.array_equal(r_cig, want)


def test_dump_sample_fixed_by_inputs():
    a = bench.dump_sample(1_000_000, 150)
    assert len(a) == bench.DUMP_READS and np.all(np.diff(a) > 0) and np.array_equal(a, bench.dump_sample(1_000_000, 150))
    assert len(bench.dump_sample(12_500, 10_000)) == bench.DUMP_READS * 150 // 10_000


def test_dump_outputs_size_cap(tmp_path, monkeypatch):
    row_off, rows, cigar = _result(5000)
    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    pick = bench.dump_sample(5000, 150)
    nbytes = bench.dump_outputs(str(tmp_path), pick, row_off, rows, cigar)
    d = _load(tmp_path)
    assert nbytes <= 200_000
    k = len(d["read_index"])
    assert 0 < k < 5000 and np.array_equal(d["read_index"], pick[:k])
    # the longest prefix that fits: one more read would not have
    ro = row_off.astype(np.int64)
    nxt = int(pick[k])
    extra = 16 + (ro[nxt + 1] - ro[nxt]) * (nbytes - 16 * k - 8 * len(d["cigar"])) / max(len(d["row_score"]), 1) \
        + 8 * int(rows["n_cigar"][ro[nxt]:ro[nxt + 1]].sum())
    assert nbytes + extra > 200_000
    sel = np.concatenate([np.arange(ro[i], ro[i + 1]) for i in pick[:k]])
    assert np.array_equal(d["rows_per_read"], ro[pick[:k] + 1] - ro[pick[:k]])
    assert np.array_equal(d["row_score"], rows["score"][sel])


@pytest.mark.gpu
def test_bench_dump_outputs(gpu_lib, tmp_path):
    """c1 (10 k reads): the sample covers every read, so the dump rebuilds the digest of the last timed step; and the reference arm's
    dump of the same reads (the oracle) is the same, array for array."""
    env = {k: v for k, v in os.environ.items() if k not in ("BSQ_SMALL_BATCH_READS", "BSQ_FIN_SHORT_LIST")}
    runs = {}
    for impl in ("ours", "reference"):
        p = subprocess.run([sys.executable, "bench.py", "--impl", impl, "--config", "c1", "--steps", "2", "--warmup", "1", "--cpu-seconds", "1",
                            "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(tmp_path / impl)], cwd=ROOT, env=env, capture_output=True, timeout=600)
        assert p.returncode == 0, (impl, p.stdout.decode()[-1500:], p.stderr.decode()[-1500:])
        runs[impl] = json.loads(p.stdout.decode().strip().split("\n")[-1]), _load(tmp_path / impl)
    line, d = runs["ours"]
    assert line["steps"] == 2
    assert np.array_equal(d["read_index"], np.arange(10_000))
    assert _digest(*_restore(d)) == line["rows_sha1_rank0"]
    ref = runs["reference"][1]
    assert sorted(ref) == sorted(d)
    for k in d:
        assert np.array_equal(ref[k], d[k]), k
