"""The compact index layout: when the full suffix array (and its inverse) cannot be allocated, the index keeps every 32nd SA entry only and
resolves the positions of its SA lookups by LF walks on the GPU.  Rows must not change.  Compact indexes are reached here through the test
hook BSQ_TEST_COMPACT=1 (the inverse SA's allocation and a load's full-SA allocation "fail") and, for the batch-pool rung, through
BSQ_TEST_POOL_OOM."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

import oracle_lib as O
from bioseqdb_b200 import BwaIndex, BwaIndexCache, BsqError, MultiBwaIndex, _lib, bwa_opts, synth
from bioseqdb_b200.loader import nuclseq_image_block
from helpers import build_pair, compare_results, to_bsq

pytestmark = pytest.mark.gpu

NOTE_SA_COMPACTED = 4
SA_SAMPLES_SECTION = 2            # index of the sa_samples section in the file's section table
HEADER_SECTIONS_AT, HEADER_CHECKSUM_AT = 136, 304
HARNESS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bioseqdb_b200", "host", "harness")


# ---- fixtures: row lengths not multiples of 4, ambiguity codes (holes), a planted repeat
def reference(lens=(3001, 2003, 997), seed=5151):
    rows = synth.reference_rows(list(lens), seed=seed)
    rng = np.random.default_rng(seed + 1)
    for r in rows:
        for _ in range(4):
            a = int(rng.integers(0, len(r) - 30))
            r[a:a + int(rng.integers(1, 12))] = ord(rng.choice(list("NRYW")))
    n = min(len(rows[0]), len(rows[1])) // 3
    rows[1][100:100 + n] = rows[0][200:200 + n]
    return rows


def big_reference():
    """large enough for the seeding prefix table, with repeat families of eight copies (above a small max_occ)"""
    rows = synth.reference_rows([90_001, 60_003, 1_001], seed=6161)
    rows = synth.plant_repeats(rows, n_families=6, copies=8, unit=(200, 900), divergence=0.01, seed=6162)
    for r in rows[:2]:
        r[5000:5007] = ord("N")
    return rows


def compact_pair(rows, opts, monkeypatch, wide=False):
    """(oracle, full index, compact index) over the same rows"""
    if wide:
        monkeypatch.setenv("BSQ_FORCE_WIDE", "1")
    orc, full = build_pair(rows, opts)
    _, comp = build_pair(rows, opts)
    with monkeypatch.context() as m:
        m.setenv("BSQ_TEST_COMPACT", "1")
        comp.L.bsq_index_prepare(comp.h, None)
    assert full.meta().sa_interval == 1 and comp.meta().sa_interval == 32
    assert full.meta().sa_bytes == comp.meta().sa_bytes == (8 if wide else 4)
    return orc, full, comp


def same_rows(a, b):
    return not compare_results(a, {"row_off": b.row_off, "rows": b.rows, "cigar": b.cigar})


def oracle_sa(orc, n):
    return np.array([n] + [orc.bwt_sa(k) for k in range(1, n + 1)], dtype=np.uint64)


# ---- 1. bwt_sa on every row
@pytest.mark.parametrize("wide", [False, True])
def test_sa_lookup_every_row(gpu_lib, monkeypatch, wide):
    orc, full, comp = compact_pair(reference(), O.sql_default_opts(3), monkeypatch, wide)
    n = int(comp.meta().seq_len)
    rows = np.arange(n + 1, dtype=np.uint64)
    want = oracle_sa(orc, n)
    assert np.array_equal(comp.sa_lookup(rows), want)
    assert np.array_equal(full.sa_lookup(rows), want)
    assert np.array_equal(comp.sa_lookup(rows[::-1].copy()), want[::-1])
    assert np.array_equal(comp.sa_sampled(), full.sa_sampled())
    with pytest.raises(BsqError, match="outside"):
        comp.sa_lookup(np.array([n + 1], dtype=np.uint64))


# ---- 2. parity
PARITY_CASES = {
    "sql": (lambda: O.sql_default_opts(3), 150, False),
    "canonical_wide": (lambda: O.canonical_opts(3), 150, True),
    "max_occ_3": (lambda: O.Opts(**{**{f: getattr(O.sql_default_opts(3), f) for f, _ in O.Opts._fields_}, "max_occ": 3}), 150, False),
    "long_reads": (lambda: O.canonical_opts(3), 700, False),
}


@pytest.mark.parametrize("case", list(PARITY_CASES))
def test_rows_equal_oracle_and_full(gpu_lib, monkeypatch, case):
    opts_fn, rlen, wide = PARITY_CASES[case]
    rows = big_reference()
    orc, full, comp = compact_pair(rows, opts_fn(), monkeypatch, wide)
    for ix in (full, comp):
        ix.set_rows_ext(True)
    n = 1500 if rlen < 496 else 300
    seqs, offs, _ = synth.simulate_reads(rows, n, rlen, sub=0.01, seed=6163, n_frac=0.002)
    ids = synth.lrand48_ids_fast(n)
    rc, rf = comp.align_batch(seqs, offs, ids), full.align_batch(seqs, offs, ids)
    bad = compare_results(rc, orc.align_batch(seqs, offs, ids, 4))
    assert not bad, "\n".join(bad)
    assert same_rows(rc, rf)
    assert comp.meta().sa_interval == 32
    data, off, _ = nuclseq_image_block(seqs, offs)
    assert same_rows(comp.align_batch_datums(data, off, ids), rf)


def test_three_chunks(gpu_lib, monkeypatch):
    rows = big_reference()
    orc, full, comp = compact_pair(rows, O.sql_default_opts(3), monkeypatch)
    monkeypatch.setenv("BSQ_CHUNK_READS", "1024")
    n = 3 * 1024 + 517
    seqs, offs, _ = synth.simulate_reads(rows, n, 120, seed=6164)
    ids = synth.lrand48_ids_fast(n)
    rc = comp.align_batch(seqs, offs, ids)
    assert same_rows(rc, full.align_batch(seqs, offs, ids))
    assert not compare_results(rc, orc.align_batch(seqs, offs, ids, 4))


# ---- 3. each rung
def test_prepare_rung(gpu_lib, monkeypatch):
    rows = big_reference()
    _, full = build_pair(rows, O.sql_default_opts(3))
    _lib.check(full.L.bsq_index_prepare(full.h, None))
    _, gpu = build_pair(rows, O.sql_default_opts(3))
    m = gpu.meta()
    monkeypatch.setenv("BSQ_TEST_COMPACT", "1")
    _lib.check(gpu.L.bsq_index_prepare(gpu.h, None))
    assert gpu.timing().notes & NOTE_SA_COMPACTED
    mc = gpu.meta()
    samples = (int(m.seq_len) + 32) // 32 * m.sa_bytes
    assert mc.sa_interval == 32 and mc.arr_bytes[_lib.ARR_SA] == samples and gpu.download(_lib.ARR_SA).size == samples
    # against the full layout after the same call: SA + inverse SA became the samples
    assert full.device_bytes() - gpu.device_bytes() >= 2 * (m.seq_len + 1) * m.sa_bytes - samples


def test_batch_pool_rung(gpu_lib, monkeypatch):
    """a reference too small for the prefix table: no table level to give back, so the pools' shortage compacts the index"""
    rows = reference()
    orc, gpu = build_pair(rows, O.sql_default_opts(3))
    seqs, offs, _ = synth.simulate_reads(rows, 400, 100, seed=5152)
    ids = synth.lrand48_ids_fast(400)
    want = gpu.align_batch(seqs, offs, ids)
    assert gpu.meta().sa_interval == 1 and not gpu.timing().notes & NOTE_SA_COMPACTED
    monkeypatch.setenv("BSQ_TEST_POOL_OOM", "1")
    gpu2 = BwaIndex(0, to_bsq(O.sql_default_opts(3)))
    for i, r in enumerate(rows):
        gpu2.add_ref_sequence(i + 1, r.tobytes())
    gpu2.build()
    got = gpu2.align_batch(seqs, offs, ids)
    assert gpu2.timing().notes & NOTE_SA_COMPACTED and gpu2.meta().sa_interval == 32
    assert gpu2.L.bsq_last_error() == b""
    assert same_rows(got, want)
    assert not compare_results(got, orc.align_batch(seqs, offs, ids, 2))
    got2 = gpu2.align_batch(seqs, offs, ids)
    assert not gpu2.timing().notes & NOTE_SA_COMPACTED and same_rows(got2, want)


def test_load_rung_and_files(gpu_lib, monkeypatch, tmp_path):
    rows = big_reference()
    orc, full = build_pair(rows, O.sql_default_opts(3))
    path = tmp_path / "i.bsqidx"
    full.save(str(path), key=b"k" * 16)
    seqs, offs, _ = synth.simulate_reads(rows, 800, 150, seed=6165)
    ids = synth.lrand48_ids_fast(800)
    want, full_sa = full.align_batch(seqs, offs, ids), full.download(_lib.ARR_SA)
    monkeypatch.setenv("BSQ_TEST_COMPACT", "1")
    ld = BwaIndex(0, to_bsq(O.sql_default_opts(3)))
    ld.load(str(path), key=b"k" * 16)
    m = ld.meta()
    assert m.sa_interval == 32 and m.arr_bytes[_lib.ARR_SA] == (m.seq_len + 32) // 32 * m.sa_bytes
    assert ld.last_load()["lf_steps"] == 0
    assert same_rows(ld.align_batch(seqs, offs, ids), want)
    # compact -> file: byte for byte the file it was loaded from
    again = tmp_path / "again.bsqidx"
    ld.save(str(again), key=b"k" * 16)
    assert again.read_bytes() == path.read_bytes()
    # a compact index saved by itself loads as a full index again
    monkeypatch.delenv("BSQ_TEST_COMPACT")
    back = BwaIndex(0, to_bsq(O.sql_default_opts(3)))
    back.load(str(again), key=b"k" * 16)
    assert back.meta().sa_interval == 1
    assert np.array_equal(back.download(_lib.ARR_SA), full_sa)


def _checksum(b: bytes) -> int:
    w = np.frombuffer(bytes(b) + b"\0" * (-len(b) % 8), dtype="<u8")
    g = np.uint64(0x9E3779B97F4A7C15)
    with np.errstate(over="ignore"):
        z = (w ^ (np.arange(len(w), dtype=np.uint64) * g)) + g
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
        return int(z.sum(dtype=np.uint64))


def _with_sample(data: bytes, k: int, value: int) -> bytes:
    """the file with sample k replaced, its section and header checksums recomputed: damage that passes the checksums"""
    d = bytearray(data)
    off, nbytes = struct.unpack_from("<QQ", d, HEADER_SECTIONS_AT + 24 * SA_SAMPLES_SECTION)
    struct.pack_into("<Q", d, off + 8 * k, value)
    struct.pack_into("<Q", d, HEADER_SECTIONS_AT + 24 * SA_SAMPLES_SECTION + 16, _checksum(bytes(d[off:off + nbytes])))
    struct.pack_into("<Q", d, HEADER_CHECKSUM_AT, _checksum(bytes(d[:HEADER_CHECKSUM_AT])))
    return bytes(d)


def test_compact_load_refuses_bad_samples(gpu_lib, monkeypatch, tmp_path):
    rows = reference()
    _, full = build_pair(rows, O.sql_default_opts(3))
    path = tmp_path / "good.bsqidx"
    full.save(str(path))
    data = path.read_bytes()
    n = int(full.meta().seq_len)
    monkeypatch.setenv("BSQ_TEST_COMPACT", "1")
    bad = tmp_path / "bad.bsqidx"
    for k, v, msg in [(7, n + 1, "SA sample 7 is larger than seq_len"), (0, n - 1, "SA sample 0 is not seq_len")]:
        bad.write_bytes(_with_sample(data, k, v))
        ix = BwaIndex(0)
        with pytest.raises(BsqError, match=msg):
            ix.load(str(bad))
        assert ix.meta().built == 0


def test_without_hook_everything_stays_full(gpu_lib, monkeypatch, tmp_path):
    monkeypatch.delenv("BSQ_TEST_COMPACT", raising=False)
    rows = big_reference()
    _, gpu = build_pair(rows, O.sql_default_opts(3))
    _lib.check(gpu.L.bsq_index_prepare(gpu.h, None))
    seqs, offs, _ = synth.simulate_reads(rows, 300, 150, seed=6166)
    gpu.align_batch(seqs, offs)
    assert gpu.meta().sa_interval == 1 and not gpu.timing().notes & NOTE_SA_COMPACTED
    path = str(tmp_path / "i.bsqidx")
    gpu.save(path)
    ld = BwaIndex(0)
    ld.load(path)
    assert ld.meta().sa_interval == 1


# ---- 4. tuples
@pytest.mark.parametrize("flags", [0, 3])
def test_tuples_equal_full(gpu_lib, monkeypatch, flags):
    rows = big_reference()
    _, full, comp = compact_pair(rows, O.sql_default_opts(3), monkeypatch)
    seqs, offs, _ = synth.simulate_reads(rows, 1200, 150, seed=6167, n_frac=0.002)
    ids = synth.lrand48_ids_fast(1200)
    data, off, _ = nuclseq_image_block(seqs, offs)
    (rf, tf), (rc, tc) = full.align_tuples_datums(data, off, ids, flags), comp.align_tuples_datums(data, off, ids, flags)   # resident
    assert same_rows(rc, rf)
    assert np.array_equal(tf.off, tc.off) and np.array_equal(tf.ref_match, tc.ref_match) and np.array_equal(tf.data, tc.data)
    sf, sc = full.tuples(rf, seqs, offs, flags), comp.tuples(rc, seqs, offs, flags)                                     # staged
    assert np.array_equal(sf.off, sc.off) and np.array_equal(sf.ref_match, sc.ref_match) and np.array_equal(sf.data, sc.data)
    assert np.array_equal(sc.data, tc.data)


# ---- 6. multi
@pytest.mark.parametrize("devices", [[0, 0], [0, 1]])
def test_multi_from_compact(gpu_lib, monkeypatch, devices):
    if max(devices) >= _lib.lib().bsq_device_count():
        pytest.skip("needs %d GPUs" % (max(devices) + 1))
    rows = big_reference()
    _, full, comp = compact_pair(rows, O.sql_default_opts(3), monkeypatch)
    seqs, offs, _ = synth.simulate_reads(rows, 2000, 150, seed=6168)
    ids = synth.lrand48_ids_fast(2000)
    want = comp.align_batch(seqs, offs, ids)
    mi = MultiBwaIndex(comp, devices)
    try:
        assert same_rows(mi.align_batch(seqs, offs, ids), want)
    finally:
        mi.close()
    assert same_rows(want, full.align_batch(seqs, offs, ids))


# ---- 7. verify
def _device_view(gpu, what, dtype):
    import torch
    from bioseqdb_b200.dist import _CudaArray
    p = C.c_void_p()
    _lib.check(gpu.L.bsq_index_device_ptr(gpu.h, what, C.byref(p)))
    n = int(gpu.meta().arr_bytes[what])
    return torch.as_tensor(_CudaArray(p.value, n), device="cuda").view(dtype)


def test_verify_compact(gpu_lib, monkeypatch):
    import torch
    _, _, comp = compact_pair(reference(), O.sql_default_opts(3), monkeypatch)
    ok = comp.verify(n_samples=1 << 40)
    assert ok["sa_permutation_ok"] == 0 and ok["exhaustive"] == 0 and ok["l2_ok"] == 1, ok
    assert all(ok[k] == 0 for k in ok if k.endswith("_bad")) and ok["sa_out_of_range"] == 0 and ok["order_undecided"] == 0, ok
    n_sa = (int(comp.meta().seq_len) + 32) // 32
    assert ok["rows_checked"] == n_sa and ok["order_checked"] == n_sa - 1, ok
    sa = _device_view(comp, _lib.ARR_SA, torch.int32)
    occ = _device_view(comp, _lib.ARR_OCC, torch.int32)
    keep = int(sa[20])
    sa[20] = int(sa[21])
    torch.cuda.synchronize()
    bad = comp.verify(n_samples=1 << 40)
    assert bad["order_bad"] >= 1 or bad["bwt_bad"] >= 1, bad
    sa[20] = keep
    occ[16 * 5] += 1                                  # block 5's count of A
    torch.cuda.synchronize()
    bad = comp.verify(n_samples=1 << 40)
    assert bad["occ_bad"] >= 1, bad
    occ[16 * 5] -= 1
    torch.cuda.synchronize()
    assert all(v == 0 for k, v in comp.verify(n_samples=1 << 40).items() if k.endswith("_bad"))


# ---- 8. cache
def test_cache_budget_counts_compact_size(gpu_lib, monkeypatch):
    texts = reference()
    rows = [(i + 1, t.tobytes()) for i, t in enumerate(texts)]
    full_cache = BwaIndexCache(max_bytes=8 << 30)
    f = full_cache.get(rows, bwa_opts())
    _lib.check(f.index.L.bsq_index_prepare(f.index.h, None))
    monkeypatch.setenv("BSQ_TEST_COMPACT", "1")
    cache = BwaIndexCache(max_bytes=8 << 30)
    lease = cache.get(rows, bwa_opts())
    _lib.check(lease.index.L.bsq_index_prepare(lease.index.h, None))
    m = lease.index.meta()
    assert m.sa_interval == 32 and cache.total_bytes() == lease.index.device_bytes()
    # no batch has run yet: the full twin holds SA + ISA where the compact one holds the samples
    assert full_cache.total_bytes() - cache.total_bytes() >= 2 * (m.seq_len + 1) * m.sa_bytes - m.arr_bytes[_lib.ARR_SA]
    seqs, offs, _ = synth.simulate_reads(texts, 300, 100, seed=5153)
    assert same_rows(lease.align_batch(seqs, offs), f.align_batch(seqs, offs))   # both sessions draw the same first ids
    assert cache.total_bytes() == lease.index.device_bytes()


# ---- the host harness reports the layout on stderr, its rows unchanged
def test_harness_reports_layout(gpu_lib, tmp_path):
    if not os.path.exists(HARNESS):
        pytest.fail("host harness is not built (run __graft_entry__.build())")
    rows = reference()
    seqs, offs, _ = synth.simulate_reads(rows, 200, 100, seed=5154)
    ref = tmp_path / "ref.tsv"; qry = tmp_path / "q.tsv"
    ref.write_bytes(b"".join(b"%d\t%s\n" % (i + 1, r.tobytes()) for i, r in enumerate(rows)))
    qry.write_bytes(b"".join(b"%d\t%s\n" % (i + 100, seqs[int(offs[i]):int(offs[i + 1])].tobytes()) for i in range(200)))
    env = {k: v for k, v in os.environ.items() if k != "BSQ_TEST_COMPACT"}
    full = subprocess.run([HARNESS, str(ref), str(qry)], capture_output=True, timeout=300, env=env)
    assert full.returncode == 0, full.stderr.decode()[-2000:]
    assert "index: layout=full sa_compacted=0" in full.stderr.decode()
    env["BSQ_TEST_COMPACT"] = "1"
    comp = subprocess.run([HARNESS, str(ref), str(qry)], capture_output=True, timeout=300, env=env)
    assert comp.returncode == 0, comp.stderr.decode()[-2000:]
    assert "index: layout=compact sa_compacted=1" in comp.stderr.decode()          # the alignment call compacted the index
    assert comp.stdout == full.stdout
    multi = subprocess.run([HARNESS, str(ref), str(qry), "devices=0,0"], capture_output=True, timeout=300, env=env)
    assert multi.returncode == 0, multi.stderr.decode()[-2000:]
    assert "index: layout=compact" in multi.stderr.decode()                         # compacted while the replicas were prepared
    assert multi.stdout == full.stdout
