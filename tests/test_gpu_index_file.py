"""Index files (bsq_index_save / bsq_index_load): a saved index loads into a fresh handle that holds the same arrays, host state and meta,
aligns exactly like the index it was saved from, and a damaged file is refused with a message that names what is wrong.  The file format
is read here by a small reader of its own (header, section table, checksum), independent of the library's."""
import os
import struct
import subprocess

import numpy as np
import pytest

import oracle_lib as O
from bioseqdb_b200 import BwaIndex, BsqError, _lib, bwa_opts, synth
from bioseqdb_b200.bwa import TUPLES_FIX_HOLE_OFFSETS, TUPLES_FIX_REVERSE
from helpers import build_pair, compare_results, to_bsq

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HARNESS = os.path.join(ROOT, "bioseqdb_b200", "host", "harness")

# ---- the file format, as a reader outside the library sees it
HEADER_FMT = "<8sIIqQQ5QQIIdQQ16s21QQ"
HEADER_FIELDS = ["magic", "version", "byte_order", "l_pac", "seq_len", "primary", "L2", "n_anns", "sa_bytes", "sa_interval", "build_ms",
                 "build_launches", "sort_pass_bytes", "key", "sections", "header_checksum"]
SECTIONS = ["pac", "occ", "sa_samples", "ann_offset", "ann_len", "ann_id", "host_state"]
assert struct.calcsize(HEADER_FMT) == 312


def checksum(b: bytes) -> int:
    """sum of splitmix64(w_i ^ i * 0x9e3779b97f4a7c15) over the u64 words of b (tail zero-padded), mod 2^64"""
    w = np.frombuffer(bytes(b) + b"\0" * (-len(b) % 8), dtype="<u8")
    g = np.uint64(0x9E3779B97F4A7C15)
    with np.errstate(over="ignore"):
        z = (w ^ (np.arange(len(w), dtype=np.uint64) * g)) + g
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
        return int(z.sum(dtype=np.uint64))


def read_header(data: bytes) -> dict:
    v = struct.unpack_from(HEADER_FMT, data)
    h = dict(zip(HEADER_FIELDS[:6], v[:6]))
    h["L2"] = list(v[6:11])
    h.update(zip(HEADER_FIELDS[7:14], v[11:18]))
    sec = v[18:39]
    h["sections"] = {name: {"offset": sec[3 * i], "bytes": sec[3 * i + 1], "checksum": sec[3 * i + 2]} for i, name in enumerate(SECTIONS)}
    h["header_checksum"] = v[39]
    return h


def section(data: bytes, h: dict, name: str) -> bytes:
    s = h["sections"][name]
    return data[s["offset"]:s["offset"] + s["bytes"]]


def reseal(data: bytearray, name: str):
    """Recompute the checksum of section `name` and of the header after an edit: a damaged file that got past its checksums."""
    h = read_header(bytes(data))
    i = SECTIONS.index(name)
    struct.pack_into("<Q", data, 136 + 24 * i + 16, checksum(section(bytes(data), h, name)))
    struct.pack_into("<Q", data, 304, checksum(bytes(data[:304])))


# ---- fixtures: several rows, lengths not multiples of 4 (filler bases), ambiguity codes (holes), a planted repeat
def reference():
    rows = synth.reference_rows([60_001, 40_003, 997, 25_002], seed=4242)
    rng = np.random.default_rng(4243)
    for r in rows[:3]:
        for _ in range(6):
            a = int(rng.integers(0, len(r) - 30))
            r[a:a + int(rng.integers(1, 15))] = ord(rng.choice(list("NRYW")))
    rows[1][5000:7000] = rows[0][1000:3000]
    return rows


def opts():
    return O.sql_default_opts(4)


def fresh(device=0):
    return BwaIndex(device, to_bsq(opts()))


def meta_tuple(m):
    return (m.l_pac, m.seq_len, m.primary, list(m.L2), m.n_anns, m.sa_bytes, m.built, list(m.arr_bytes), m.build_ms, m.build_launches, m.sort_pass_bytes)


def as_expected(res):
    """an AlignResult in the form compare_results takes as its second argument"""
    return {"row_off": res.row_off, "rows": res.rows, "cigar": res.cigar}


def reads(rows, n=600, seed=4244):
    seqs, offs, _ = synth.simulate_reads(rows, n, 150, seed=seed, n_frac=0.01)
    return seqs, offs, synth.lrand48_ids_fast(n)


@pytest.fixture(scope="module")
def built():
    rows = reference()
    orc, gpu = build_pair(rows, opts())
    return rows, orc, gpu


@pytest.mark.parametrize("wide", [False, True])
def test_round_trip(gpu_lib, monkeypatch, tmp_path, wide):
    """Build, save, load into a fresh handle: every array, the host state and the meta come back, and the loaded index passes the
    exhaustive device check.  wide: the 64-bit suffix array (BSQ_FORCE_WIDE is read by every build call)."""
    if wide:
        monkeypatch.setenv("BSQ_FORCE_WIDE", "1")
    _, gpu = build_pair(reference(), opts())
    m = gpu.meta()
    assert m.sa_bytes == (8 if wide else 4)
    path = str(tmp_path / "i.bsqidx")
    gpu.save(path)
    ld = fresh()
    ms = ld.load(path)
    assert ms > 0 and ld.n_rows == 4
    for what in range(_lib.ARR_COUNT):
        assert np.array_equal(ld.download(what), gpu.download(what)), what
    assert ld.host_state() == gpu.host_state()
    assert meta_tuple(ld.meta()) == meta_tuple(m)
    chk = ld.verify(n_samples=1 << 40)
    assert chk["sound"] and chk["exhaustive"] == 1 and chk["rows_checked"] == m.seq_len + 1, chk
    info = ld.last_load()
    assert info["file_bytes"] == os.path.getsize(path)
    assert info["lf_steps"] == m.seq_len + 1 and info["lf_steps"] <= info["lane_slots"]


def test_file_contents_against_oracle(gpu_lib, built, tmp_path):
    rows, orc, gpu = built
    path = tmp_path / "i.bsqidx"
    gpu.save(str(path))
    data = path.read_bytes()
    h = read_header(data)
    oi = orc.info()
    assert h["magic"] == b"BSQIDX\0\0" and h["version"] == 1 and h["byte_order"] == 0x01020304 and h["sa_interval"] == 32
    assert h["header_checksum"] == checksum(data[:304])
    assert (h["l_pac"], h["seq_len"], h["primary"], h["L2"], h["n_anns"]) == (oi["l_pac"], oi["seq_len"], oi["primary"], oi["L2"], 4)
    for name in SECTIONS:
        s = h["sections"][name]
        assert s["offset"] % 64 == 0 and s["checksum"] == checksum(section(data, h, name)), name
    samples = np.frombuffer(section(data, h, "sa_samples"), dtype="<u8")
    want = orc.sa()
    assert len(samples) == len(want) == (oi["seq_len"] + 32) // 32
    assert int(samples[0]) == oi["seq_len"] and np.array_equal(samples[1:], want[1:])
    assert np.array_equal(np.frombuffer(section(data, h, "pac"), dtype=np.uint8), orc.pac())
    occ = np.frombuffer(section(data, h, "occ"), dtype="<u4")
    n_full = oi["seq_len"] // 128
    assert np.array_equal(occ[:n_full * 16], orc.bwt_interleaved()[:n_full * 16])
    assert h["key"] == b"\0" * 16


def test_alignment_through_loaded_index(gpu_lib, built, tmp_path):
    """Rows, CIGARs, the extension fields and the GPU-built tuple columns (with the hole overlay) of the loaded index equal those of the
    index it was saved from and the oracle's.  Options come from the composite after the load, so max_occ's default counts the rows."""
    rows, orc, gpu = built
    path = str(tmp_path / "i.bsqidx")
    gpu.save(path)
    ld = BwaIndex(0)
    ld.load(path)
    ld.set_options_from_composite(bwa_opts())
    assert [getattr(ld.options, f) for f, _ in _lib.BsqOpts._fields_] == [getattr(gpu.options, f) for f, _ in _lib.BsqOpts._fields_]
    seqs, offs, ids = reads(rows)
    rb, rl = gpu.align_batch(seqs, offs, ids), ld.align_batch(seqs, offs, ids)
    assert rl.rows["is_rev"].any() and (seqs == ord("N")).any()
    assert not compare_results(rl, as_expected(rb))
    assert not compare_results(rl, orc.align_batch(seqs, offs, ids, 2))
    flags = TUPLES_FIX_HOLE_OFFSETS | TUPLES_FIX_REVERSE
    tb, tl = gpu.tuples(rb, seqs, offs, flags), ld.tuples(rl, seqs, offs, flags)
    assert np.array_equal(tb.ref_match, tl.ref_match)
    for i in range(len(rb.rows)):
        assert (tb.ref_subseq(i), tb.query_subseq(i), tb.cigar(i)) == (tl.ref_subseq(i), tl.query_subseq(i), tl.cigar(i)), i


def test_save_is_deterministic(gpu_lib, built, tmp_path):
    _, _, gpu = built
    a, b = tmp_path / "a.bsqidx", tmp_path / "b.bsqidx"
    key = bytes(range(16))
    gpu.save(str(a), key=key)
    ld = fresh()
    ld.load(str(a), key=key)
    ld.save(str(b), key=key)
    assert a.read_bytes() == b.read_bytes()


def _load_error(path, key=None) -> str:
    ix = fresh()
    with pytest.raises(BsqError) as e:
        ix.load(str(path), key=key)
    assert ix.meta().built == 0 and ix.n_rows == 0
    return str(e.value)


def test_damaged_files_are_refused(gpu_lib, built, tmp_path):
    _, _, gpu = built
    good = tmp_path / "good.bsqidx"
    gpu.save(str(good), key=b"k" * 16)
    data = good.read_bytes()
    h = read_header(data)
    bad = tmp_path / "bad.bsqidx"
    for name in SECTIONS:                         # one flipped byte inside each section: the checksum names it
        s = h["sections"][name]
        d = bytearray(data)
        d[s["offset"] + s["bytes"] // 2] ^= 0x40
        bad.write_bytes(bytes(d))
        assert "checksum mismatch in section '%s'" % name in _load_error(bad), name
    bad.write_bytes(data[:len(data) // 2])
    assert "shorter than its section table" in _load_error(bad)
    bad.write_bytes(data[:100])
    assert "shorter than the 320-byte header" in _load_error(bad)
    bad.write_bytes(b"NOTANIDX" + data[8:])
    assert "wrong magic" in _load_error(bad)
    d = bytearray(data)
    struct.pack_into("<I", d, 8, 2)
    bad.write_bytes(bytes(d))
    assert "format version 2" in _load_error(bad)
    assert "key mismatch" in _load_error(good, key=b"x" * 16)
    # sizes that disagree with seq_len, and 4-byte SA entries for 2^32 rows: refused on the host before anything is allocated
    d = bytearray(data)
    struct.pack_into("<Q", d, 136 + 24 * 1 + 8, h["sections"]["occ"]["bytes"] + 64)
    struct.pack_into("<Q", d, 304, checksum(bytes(d[:304])))
    bad.write_bytes(bytes(d))
    assert "section 'occ' has" in _load_error(bad)
    d = bytearray(data)
    struct.pack_into("<qQ", d, 16, 1 << 31, 1 << 32)
    struct.pack_into("<Q", d, 304, checksum(bytes(d[:304])))
    bad.write_bytes(bytes(d))
    assert "4-byte SA entries" in _load_error(bad)
    # past the checksums: a sample above seq_len, and an Occ checkpoint that sends LF out of the rows, stop the rebuild
    d = bytearray(data)
    s = h["sections"]["sa_samples"]
    struct.pack_into("<Q", d, s["offset"] + 8 * 7, h["seq_len"] + 5)
    reseal(d, "sa_samples")
    bad.write_bytes(bytes(d))
    assert "SA sample 7 is larger than seq_len" in _load_error(bad)
    d = bytearray(data)
    o = h["sections"]["occ"]
    for blk in range(h["seq_len"] // 128):
        for c in range(4):
            struct.pack_into("<Q", d, o["offset"] + 64 * blk + 8 * c, 1 << 40)
    reseal(d, "occ")
    bad.write_bytes(bytes(d))
    assert "left the rows" in _load_error(bad)
    # a failed load leaves the handle fresh: the good file loads into it afterwards
    ix = fresh()
    with pytest.raises(BsqError):
        ix.load(str(bad))
    ix.load(str(good), key=b"k" * 16)
    assert ix.meta().built == 1


def test_save_and_load_misuse(gpu_lib, built, tmp_path):
    rows, _, gpu = built
    p = tmp_path / "i.bsqidx"
    gpu.save(str(p))
    ix = fresh()
    ix.add_ref_sequence(1, rows[2].tobytes())
    with pytest.raises(BsqError, match="fresh handle"):
        ix.load(str(p))
    with pytest.raises(BsqError, match="not built"):
        ix.save(str(tmp_path / "unbuilt.bsqidx"))
    empty = fresh()
    empty.build()                                  # the empty reference builds nothing
    with pytest.raises(BsqError, match="not built"):
        empty.save(str(tmp_path / "empty.bsqidx"))
    missing = tmp_path / "no" / "such" / "dir"
    with pytest.raises(BsqError, match="No such file or directory"):
        gpu.save(str(missing / "i.bsqidx"))
    with pytest.raises(BsqError, match="cannot open"):
        fresh().load(str(missing / "i.bsqidx"))
    assert sorted(os.listdir(tmp_path)) == ["i.bsqidx"]    # no temporary file left anywhere


def _harness(ref, qry, *extra):
    return subprocess.run([HARNESS, str(ref), str(qry), *extra], capture_output=True, timeout=300)


def test_harness_cross_process(gpu_lib, tmp_path):
    """Two processes with the same index_cache directory: the first builds and writes the file, the second loads it (the file is not
    rewritten) and prints the same rows -- which are also those of a run without the cache."""
    if not os.path.exists(HARNESS):
        pytest.fail("host harness is not built (run __graft_entry__.build())")
    rows = reference()
    seqs, offs, _ = reads(rows, 300, seed=4245)
    ref, qry = tmp_path / "ref.tsv", tmp_path / "q.tsv"
    ref.write_bytes(b"".join(b"%d\t%s\n" % (i + 1, r.tobytes()) for i, r in enumerate(rows)))
    qry.write_bytes(b"".join(b"%d\t%s\n" % (i + 100, seqs[int(offs[i]):int(offs[i + 1])].tobytes()) for i in range(300)))
    cache = tmp_path / "cache"
    cache.mkdir()
    first = _harness(ref, qry, "index_cache=%s" % cache)
    assert first.returncode == 0, first.stderr.decode()[-2000:]
    assert "index_cache: disk_hits=0 disk_saves=1 disk_errors=0" in first.stderr.decode()
    files = os.listdir(cache)
    assert len(files) == 1 and files[0].endswith(".bsqidx")
    mtime = os.stat(cache / files[0]).st_mtime_ns
    second = _harness(ref, qry, "index_cache=%s" % cache)
    assert second.returncode == 0, second.stderr.decode()[-2000:]
    assert "index_cache: disk_hits=1 disk_saves=0 disk_errors=0" in second.stderr.decode()
    assert os.listdir(cache) == files and os.stat(cache / files[0]).st_mtime_ns == mtime
    plain = _harness(ref, qry)
    assert plain.returncode == 0
    assert first.stdout and second.stdout == first.stdout == plain.stdout


def test_python_cache_across_instances(gpu_lib, tmp_path):
    """Two BwaIndexCache objects on one directory, standing in for two backends: the second loads what the first built."""
    from bioseqdb_b200 import BwaIndexCache
    rows = reference()
    trows = [(i + 1, r.tobytes()) for i, r in enumerate(rows)]
    seqs, offs, ids = reads(rows, 400, seed=4246)
    a = BwaIndexCache(directory=str(tmp_path))
    ra = a.get(trows, bwa_opts()).align_batch(seqs, offs, ids)
    assert (a.misses, a.disk_hits, a.disk_saves, a.disk_errors) == (1, 0, 1, 0)
    b = BwaIndexCache(directory=str(tmp_path))
    lease = b.get(trows, bwa_opts())
    assert (b.misses, b.disk_hits, b.disk_saves, b.disk_errors) == (1, 1, 0, 0)
    assert lease.index.last_load()["lf_steps"] == lease.index.meta().seq_len + 1     # this index came from the file
    assert not compare_results(lease.align_batch(seqs, offs, ids), as_expected(ra))
    a.clear(); b.clear()


def test_load_on_other_device(gpu_lib, built, tmp_path):
    if gpu_lib.bsq_device_count() < 2:
        pytest.skip("needs two GPUs")
    rows, _, gpu = built
    path = str(tmp_path / "i.bsqidx")
    gpu.save(path)
    ld = fresh(device=1)
    ld.load(path)
    seqs, offs, ids = reads(rows, 300, seed=4247)
    assert not compare_results(ld.align_batch(seqs, offs, ids), as_expected(gpu.align_batch(seqs, offs, ids)))
