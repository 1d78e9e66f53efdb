"""bsq_multi_result_tuples: the bwa_result tuples of a multi-GPU batch, each device materialising the rows of its own block of reads, must
be byte-identical to the single-device route (bsq_result_tuples on the built handle), whether a device serves its block from HBM or
stages it.  A device may repeat in the device list, so every case runs on a one-GPU box; with two GPUs the blocks go to both."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as O
from bioseqdb_b200 import BsqError, MultiBwaIndex, synth
from bioseqdb_b200._lib import BsqResult, check, ptr
from bioseqdb_b200.loader import nuclseq_image_block
from helpers import build_pair, read_arrays

pytestmark = pytest.mark.gpu
HARNESS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bioseqdb_b200", "host", "harness")


@pytest.fixture
def devs(gpu_lib):
    """devs(k): a device list of k entries, over two GPUs when the box has them, else k handles on GPU 0"""
    two = gpu_lib.bsq_device_count() >= 2
    return lambda k: [d % 2 if two else 0 for d in range(k)]


def _reference(seed, n_reads, rng):
    """reference rows with ambiguity runs (un-rebased holes) and reads over them, plus N / R / Y letters in the reads"""
    rows = []
    for n in (30_001, 20_002, 9_999):
        t = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=n)].copy()
        for _ in range(12):
            a = int(rng.integers(0, n - 40)); l = int(rng.integers(1, 30))
            t[a:a + l] = ord(rng.choice(list("NNRYKM")))
        rows.append(t)
    seqs, offs, _ = synth.simulate_reads(rows, n_reads, 150, seed=seed)
    seqs = seqs.copy()
    seqs[rng.integers(0, len(seqs), size=n_reads // 2)] = np.frombuffer(b"NNNRY", dtype=np.uint8)[rng.integers(0, 5, size=n_reads // 2)]
    return rows, seqs, offs


def _same(a, b):
    assert np.array_equal(a.off, b.off)
    assert np.array_equal(a.ref_match, b.ref_match)
    assert np.array_equal(a.data, b.data)


def _multi_align(multi, seqs, offs, ids):
    """bsq_multi_align_batch, the library's result kept (not collected), so that its tuples can be served from HBM"""
    res = C.POINTER(BsqResult)()
    check(multi.L.bsq_multi_align_batch(multi.m, ptr(seqs), ptr(offs), ptr(ids), len(offs) - 1, C.byref(res)))
    return res


def _multi_align_datums(multi, data, off, ids):
    res = C.POINTER(BsqResult)()
    check(multi.L.bsq_multi_align_batch_datums(multi.m, ptr(data), ptr(off), ptr(ids), len(off) - 1, C.byref(res)))
    return res


@pytest.mark.parametrize("datums", [False, True])
def test_latest_multi_result_from_hbm(devs, datums):
    rng = np.random.default_rng(201)
    rows, seqs, offs = _reference(202, 1500, rng)
    orc, gpu = build_pair(rows, O.sql_default_opts(3))
    n = len(offs) - 1
    ids = synth.lrand48_ids_fast(n)
    multi = MultiBwaIndex(gpu, devs(2))
    data, off, _ = nuclseq_image_block(seqs, offs)
    raw = _multi_align_datums(multi, data, off, ids) if datums else _multi_align(multi, seqs, offs, ids)
    try:
        got = {f: multi._fetch_tuples(raw, None, None, f) for f in (0, 1, 3)}
    finally:
        res = gpu._collect(raw)
    assert int(res.row_off[-1]) >= n
    for f, tup in got.items():
        _same(tup, gpu.tuples(res, seqs, offs, f))                       # the staged single-device route
        one_res, one = gpu.align_tuples_datums(data, off, ids, f)         # the single-device datum call, served from its own HBM
        assert np.array_equal(one_res.row_off, res.row_off)
        _same(tup, one)
    # the datum call of the Python mirror returns the same pair
    res2, tup2 = multi.align_tuples_datums(data, off, ids, 3)
    assert np.array_equal(res2.row_off, res.row_off)
    _same(tup2, got[3])
    multi.close()


def test_three_blocks_with_an_empty_one(devs):
    """three blocks of 1000, 1000 and 1001 reads; the middle one is all reads shorter than min_seed_len, so it has no rows and the third
    block's byte offsets are rebased across an empty piece"""
    rng = np.random.default_rng(211)
    rows, seqs, offs = _reference(212, 3001, rng)
    orc, gpu = build_pair(rows, O.sql_default_opts(3))
    reads = [seqs[int(offs[i]):int(offs[i + 1])].tobytes() for i in range(3001)]
    for i in range(1000, 2000):
        reads[i] = reads[i][:12]
    seqs, offs = read_arrays(reads)
    ids = synth.lrand48_ids_fast(3001)
    multi = MultiBwaIndex(gpu, devs(3))
    raw = _multi_align(multi, seqs, offs, ids)
    try:
        tup = multi._fetch_tuples(raw, None, None, 0)
    finally:
        res = gpu._collect(raw)
    assert res.row_off[1000] == res.row_off[2000] and res.row_off[1000] > 0 and res.row_off[-1] > res.row_off[2000]
    _same(tup, gpu.tuples(res, seqs, offs))
    _same(multi.tuples(res, seqs, offs), tup)                           # the same result staged across the three handles
    multi.close()


def test_edge_sizes(devs):
    rng = np.random.default_rng(221)
    rows, seqs, offs = _reference(222, 8, rng)
    orc, gpu = build_pair(rows, O.sql_default_opts(3))
    multi = MultiBwaIndex(gpu, devs(3))
    for n in (1, 2):                                                     # fewer reads than devices: empty blocks
        s, o = seqs[:int(offs[n])], offs[:n + 1]
        ids = synth.lrand48_ids_fast(n)
        raw = _multi_align(multi, s, o, ids)
        try:
            tup = multi._fetch_tuples(raw, None, None, 0)
        finally:
            res = gpu._collect(raw)
        assert int(res.row_off[-1]) >= n
        _same(tup, gpu.tuples(res, s, o))
    s, o = read_arrays([b"ACGTACGTAC", b"NNNN", b"ACGTTT"])              # no rows at all
    raw = _multi_align(multi, s, o, synth.lrand48_ids_fast(3))
    try:
        tup = multi._fetch_tuples(raw, None, None, 0)
    finally:
        res = gpu._collect(raw)
    assert int(res.row_off[-1]) == 0
    assert tup.off.tolist() == [0] and tup.ref_match.shape == (0, 3) and len(tup.data) == 0
    multi.close()


def test_mixed_resident_and_staged(devs):
    """a single-device align_batch after the multi call overwrites device 0's batch: device 0 stages its block, the others serve theirs"""
    rng = np.random.default_rng(231)
    rows, seqs, offs = _reference(232, 1200, rng)
    orc, gpu = build_pair(rows, O.sql_default_opts(3))
    ids = synth.lrand48_ids_fast(1200)
    multi = MultiBwaIndex(gpu, devs(2))
    raw = _multi_align(multi, seqs, offs, ids)
    try:
        gpu.align_batch(seqs[:int(offs[100])], offs[:101], ids[:100])
        with pytest.raises(BsqError, match="null argument"):
            multi._fetch_tuples(raw, None, None, 0)
        tup = multi._fetch_tuples(raw, ptr(seqs), ptr(offs), 1)
    finally:
        res = gpu._collect(raw)
    _same(tup, gpu.tuples(res, seqs, offs, 1))
    multi.close()


def test_non_resident_results_leave_the_batches(devs):
    """a host-assembled result and an earlier multi result are staged across the devices; the latest multi result is still served from
    HBM afterwards, with the same tuples"""
    rng = np.random.default_rng(241)
    rows, seqs, offs = _reference(242, 2000, rng)
    orc, gpu = build_pair(rows, O.sql_default_opts(3))
    ids = synth.lrand48_ids_fast(2000)
    cut = int(offs[900])
    sa, oa = seqs[:cut], offs[:901]
    sb, ob = seqs[cut:], offs[900:] - offs[900]
    host = gpu.align_batch(sa, oa, ids[:900])                            # a result that lives on the host only
    multi = MultiBwaIndex(gpu, devs(2))
    earlier = _multi_align(multi, sa, oa, ids[:900])
    latest = _multi_align(multi, sb, ob, ids[900:])
    try:
        before = multi._fetch_tuples(latest, None, None, 0)
        with pytest.raises(BsqError, match="null argument"):
            multi._fetch_tuples(earlier, None, None, 0)
        from_earlier = multi._fetch_tuples(earlier, ptr(sa), ptr(oa), 0)
        from_host = multi.tuples(host, sa, oa)
        after = multi._fetch_tuples(latest, None, None, 0)
    finally:
        res_a = gpu._collect(earlier)
        res_b = gpu._collect(latest)
    want = gpu.tuples(host, sa, oa)
    _same(from_host, want)
    assert np.array_equal(res_a.row_off, host.row_off)
    _same(from_earlier, want)
    _same(after, before)
    _same(after, gpu.tuples(res_b, sb, ob))
    multi.close()


def test_harness_on_several_devices(gpu_lib, tmp_path):
    if not os.path.exists(HARNESS):
        pytest.fail("host harness is not built (run __graft_entry__.build())")
    rng = np.random.default_rng(251)
    rows, seqs, offs = _reference(252, 400, rng)
    ref = tmp_path / "ref.tsv"; qry = tmp_path / "q.tsv"
    ref.write_bytes(b"".join(b"%d\t%s\n" % (i + 1, r.tobytes()) for i, r in enumerate(rows)))
    qry.write_bytes(b"".join(b"%d\t%s\n" % (i + 100, seqs[int(offs[i]):int(offs[i + 1])].tobytes()) for i in range(400)))
    one = subprocess.run([HARNESS, str(ref), str(qry)], capture_output=True, timeout=300)
    assert one.returncode == 0, one.stderr.decode()[-2000:]
    assert len(one.stdout.splitlines()) >= 400
    lists = ["0,0"] + (["0,1"] if gpu_lib.bsq_device_count() >= 2 else [])
    for devices in lists:
        p = subprocess.run([HARNESS, str(ref), str(qry), "devices=" + devices, "check_tuples=1"], capture_output=True, timeout=300)
        assert p.returncode == 0, p.stderr.decode()[-2000:]
        assert "rows identical" in p.stderr.decode()
        assert p.stdout == one.stdout, devices
