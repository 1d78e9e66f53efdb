"""The slim wire format (VERDICT r1 #9): reads handed over as NUCLSEQ datum images (bsq_align_batch_datums), ids drawn by the library from
the session's lrand48 stream (ids = NULL), 64-byte public rows with the mem_alnreg_t extension optional -- each against the plain ASCII
entry point and, through it, the oracle."""
import numpy as np
import pytest

import oracle_lib as O
from bioseqdb_b200 import synth
from bioseqdb_b200.loader import nuclseq_image_block
from helpers import build_pair, compare_results, read_arrays, PARITY_FIELDS

pytestmark = pytest.mark.gpu


def _same(a, b, fields=PARITY_FIELDS):
    assert np.array_equal(a.row_off, b.row_off)
    for f in fields:
        assert np.array_equal(a.rows[f], b.rows[f]), f
    for i in range(len(a.rows)):
        assert a.cigar_of(a.rows[i]) == b.cigar_of(b.rows[i])


def test_datum_batch_equals_ascii_batch(gpu_lib):
    rows = synth.reference_rows([300_001, 200_003], seed=101)
    orc, gpu = build_pair(rows, O.sql_default_opts(2))
    seqs, offs, _ = synth.simulate_reads(rows, 5000, 150, seed=102, n_frac=0.004)      # some reads carry N
    r0 = rows[0].tobytes()
    extra = [r0[1000:1070] + b"NNNNNRRYK" + r0[1079:1150], b"N" * 40, r0[5:24], b"", r0[2000:2301], b"ACGTN"]    # IUPAC runs, all-N, 19 bases, empty, 301 bases
    es, eo = read_arrays(extra)
    seqs = np.concatenate([seqs, es]); offs = np.concatenate([offs, eo[1:] + offs[-1]])
    n = len(offs) - 1
    ids = synth.lrand48_ids_fast(n)
    a = gpu.align_batch(seqs, offs, ids)
    data, off, _ = nuclseq_image_block(seqs, offs)
    d = gpu.align_batch_datums(data, off, ids)
    _same(a, d)
    o = orc.align_batch(seqs, offs, ids, 4)
    assert not compare_results(d, o)


def test_datum_batch_chunked(gpu_lib, monkeypatch):
    """large batch => the two-lane chunk pipeline; chunks are cut out of the datum block by their offsets"""
    monkeypatch.setenv("BSQ_CHUNK_READS", "65536")
    rows = synth.reference_rows([400_001], seed=111)
    _, gpu = build_pair(rows, O.sql_default_opts(1))
    seqs, offs, _ = synth.simulate_reads(rows, 2 * 65536 + 4321, 100, seed=112)     # 2 x 64 K reads at least: the batch is chunked
    ids = synth.lrand48_ids_fast(len(offs) - 1)
    data, off, _ = nuclseq_image_block(seqs, offs)
    d = gpu.align_batch_datums(data, off, ids)
    chunked_launches = gpu.timing().launches
    gpu.upload(seqs, offs, ids); gpu.align_resident()
    assert chunked_launches >= 3 * gpu.timing().launches     # three chunks ran, each a pipeline pass
    r = gpu.download_result()
    _same(d, r)


def test_session_ids(gpu_lib):
    """ids = NULL: the library draws lrand48() itself, one per read, continuing across calls (mem_align1's id, SURVEY A.10)"""
    rows = synth.reference_rows([200_001], seed=121)
    rows = synth.plant_repeats(rows, n_families=6, copies=6, unit=(150, 400), divergence=0.0, seed=122)   # exact repeats: equal scores, order decided by hash(id)
    _, gpu = build_pair(rows, O.sql_default_opts(1))
    seqs, offs, _ = synth.simulate_reads(rows, 3000, 150, seed=123)
    ids = synth.lrand48_ids_fast(3000)
    want = gpu.align_batch(seqs, offs, ids)
    assert gpu.session_lrand48() == 0
    cut = 1234
    a = gpu.align_batch(seqs[:int(offs[cut])], offs[:cut + 1], None)
    data, off, _ = nuclseq_image_block(seqs[int(offs[cut]):], offs[cut:] - offs[cut])
    b = gpu.align_batch_datums(data, off, None)
    assert np.array_equal(want.rows["hash"], np.concatenate([a.rows["hash"], b.rows["hash"]]))
    assert np.array_equal(want.rows["rb"], np.concatenate([a.rows["rb"], b.rows["rb"]]))
    st = gpu.session_lrand48()
    assert st != 0
    gpu.session_lrand48(0)                               # a fresh backend: the stream starts again
    again = gpu.align_batch(seqs[:int(offs[cut])], offs[:cut + 1], None)
    assert np.array_equal(again.rows["hash"], a.rows["hash"])
    assert gpu.session_lrand48() == synth.lrand48_ids(cut)[1]      # glibc's state after `cut` draws


def test_public_rows_without_extension(gpu_lib):
    """default C-ABI results carry the 64-byte bsq_row only; the extension fields are not transferred (zero in the joined view)"""
    pub = ["rid", "rb", "re", "qb", "qe", "is_rev", "score", "pos", "NM", "mapq", "flag", "n_cigar", "ref_id"]
    rows = synth.reference_rows([150_001, 100_003], seed=131)
    _, gpu = build_pair(rows, O.sql_default_opts(2))
    seqs, offs, _ = synth.simulate_reads(rows, 2000, 150, seed=132)
    ids = synth.lrand48_ids_fast(2000)
    full = gpu.align_batch(seqs, offs, ids)
    gpu.set_rows_ext(False)
    slim = gpu.align_batch(seqs, offs, ids)
    t = gpu.timing()
    gpu.set_rows_ext(True)
    _same(full, slim, pub)
    assert not slim.rows["hash"].any() and full.rows["hash"].any()
    assert int(t.d2h_bytes) < 2000 * 8 + 16 + len(slim.rows) * 64 + len(slim.cigar) * 4 + 64


def test_tuples_from_resident_batch(gpu_lib):
    """bsq_result_tuples on the library's own result of a batch that is still in HBM uploads nothing (VERDICT r1 #6); its datums, CIGAR
    strings and ref_match_* must equal the general path's (rows, CIGARs and reads uploaded again), for one-pass and two-chunk batches,
    holes in the reference and in the reads included."""
    rows = [r.tobytes() for r in synth.reference_rows([250_001, 150_003], seed=141)]
    rows[0] = rows[0][:5000] + b"N" * 30 + rows[0][5030:90_000] + b"RRY" + rows[0][90_003:]
    _, gpu = build_pair(rows, O.sql_default_opts(2))
    clean = [np.frombuffer(r.replace(b"N", b"A").replace(b"R", b"G").replace(b"Y", b"C"), dtype=np.uint8) for r in rows]
    for n in (3000, 2 * 65536 + 777):
        seqs, offs, _ = synth.simulate_reads(clean, n, 100, seed=142 + n, n_frac=0.003)
        extra = [rows[0][4950:5100], rows[0][89_950:90_100]]      # reads over the reference's holes (their own N / R / Y become holes of query_subseq)
        es, eo = read_arrays(extra)
        seqs = np.concatenate([seqs, es]); offs = np.concatenate([offs, eo[1:] + offs[-1]])
        ids = synth.lrand48_ids_fast(len(offs) - 1)
        data, off, _ = nuclseq_image_block(seqs, offs)
        res, tup = gpu.align_tuples_datums(data, off, ids)
        ref = gpu.tuples(res, seqs, offs)                          # general path: host result, everything uploaded
        assert len(res.rows) > n * 0.9
        assert np.array_equal(tup.off, ref.off) and np.array_equal(tup.ref_match, ref.ref_match)
        assert np.array_equal(tup.data, ref.data)
        for flags in (1, 3):
            res2, tup2 = gpu.align_tuples_datums(data, off, ids, flags)
            ref2 = gpu.tuples(res2, seqs, offs, flags)
            assert np.array_equal(tup2.off, ref2.off) and np.array_equal(tup2.data, ref2.data) and np.array_equal(tup2.ref_match, ref2.ref_match)


def test_tuples_of_another_result_leave_the_resident_batch(gpu_lib):
    """bsq_result_tuples on a result that is not resident works in buffers of its own: a tuples call on another, host-assembled result
    between the alignment of a batch and the tuples of that batch's result must leave the batch servable (no reads passed) and its
    tuples unchanged."""
    import ctypes as C
    from bioseqdb_b200._lib import BsqResult, check, ptr
    rows = synth.reference_rows([250_001, 150_003], seed=161)
    _, gpu = build_pair(rows, O.sql_default_opts(2))
    s_other, o_other, _ = synth.simulate_reads(rows, 6000, 150, seed=162)
    other = gpu.align_batch(s_other, o_other, synth.lrand48_ids_fast(6000))     # copied to the host: no longer the library's own result
    seqs, offs, _ = synth.simulate_reads(rows, 4000, 100, seed=163, n_frac=0.003)
    ids = synth.lrand48_ids_fast(4000)
    res = C.POINTER(BsqResult)()
    check(gpu.L.bsq_align_batch(gpu.h, ptr(seqs), ptr(offs), ptr(ids), 4000, C.byref(res)))
    try:
        before = gpu._fetch_tuples(res, None, None, 0)
        staged = gpu.tuples(other, s_other, o_other)
        after = gpu._fetch_tuples(res, None, None, 0)
    finally:
        gpu.L.bsq_result_free(res)
    assert len(other.rows) > 5000 and len(staged.off) == 3 * len(other.rows) + 1
    assert len(before.off) > 3 * 3600
    assert np.array_equal(before.off, after.off) and np.array_equal(before.ref_match, after.ref_match)
    assert np.array_equal(before.data, after.data)


def test_pool_oom_drops_a_table_level(gpu_lib, monkeypatch):
    """Device memory short while sizing the batch pools (simulated: BSQ_TEST_POOL_OOM makes one pool allocation fail): the library gives back
    the deepest level of the seeding prefix table, rebuilds the shallower one and finishes the call; the rows do not change (the table
    only shortcuts bwt_extend), the call says so in bsq_timing.notes, and the next call runs without incident."""
    from helpers import compare_results
    monkeypatch.setenv("BSQ_TEST_POOL_OOM", "1")
    rows = synth.reference_rows([150_001, 100_003], seed=151)
    orc, gpu = build_pair(rows, O.sql_default_opts(2))
    seqs, offs, _ = synth.simulate_reads(rows, 3000, 150, seed=152)
    ids = synth.lrand48_ids_fast(3000)
    g = gpu.align_batch(seqs, offs, ids)
    assert gpu.timing().notes & 2                       # BSQ_NOTE_TABLE_DOWNGRADED
    assert gpu.L.bsq_last_error() == b""
    o = orc.align_batch(seqs, offs, ids, 4)
    bad = compare_results(g, o)
    assert not bad, "\n".join(bad)
    g2 = gpu.align_batch(seqs, offs, ids)
    assert not (gpu.timing().notes & 2)
    assert not compare_results(g2, o)
