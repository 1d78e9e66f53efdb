"""End-to-end parity through the C ABI (bsq_align_batch) vs the oracle: identical ordered rows --
rid, rb, re, qb, qe, strand, score, truesc, secondary, sub, sub_n, CIGAR, NM, MAPQ, hash order."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O
from bioseqdb_b200 import synth
from helpers import build_pair, compare_results, read_arrays

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("opts_fn", [O.sql_default_opts, O.canonical_opts])
def test_align_simulated(gpu_lib, opts_fn):
    rows = synth.reference_rows([400_003, 300_001, 250_002, 49_999], seed=21)
    orc, gpu = build_pair(rows, opts_fn(len(rows)))
    seqs, offs, _ = synth.simulate_reads(rows, 6000, 150, seed=22)
    ids = synth.lrand48_ids_fast(6000)
    g = gpu.align_batch(seqs, offs, ids)
    o = orc.align_batch(seqs, offs, ids, 4)
    bad = compare_results(g, o)
    assert not bad, "\n".join(bad)
    assert int(g.row_off[-1]) >= 6000 * 0.99


def test_align_repeats_and_noise(gpu_lib):
    """repeat families => multiple chains, secondaries, sub/sub_n, dedup; higher error => clipping, band retries"""
    rows = synth.reference_rows([300_000, 200_001], seed=31)
    rows = synth.plant_repeats(rows, n_families=12, copies=10, unit=(150, 1200), divergence=0.03)
    orc, gpu = build_pair(rows, O.sql_default_opts(2))
    seqs, offs, _ = synth.simulate_reads(rows, 4000, 150, sub=0.03, ins=0.006, dele=0.006, seed=32, n_frac=0.002)
    ids = synth.lrand48_ids_fast(4000)
    g = gpu.align_batch(seqs, offs, ids)
    o = orc.align_batch(seqs, offs, ids, 4)
    bad = compare_results(g, o)
    assert not bad, "\n".join(bad)
    assert (g.rows["secondary"] >= 0).sum() > 0


def test_align_edge_cases(gpu_lib):
    rows = synth.reference_rows([60_001, 1_003, 501], seed=41)
    orc, gpu = build_pair(rows, O.canonical_opts(3))
    r0, r1, r2 = [r.tobytes() for r in rows]
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    reads = [
        r0[1000:1150],                       # perfect forward
        r0[2000:2150].translate(comp)[::-1],  # perfect reverse
        r0[0:150], r0[60_001 - 150:],        # flush with the row ends
        r1[1_003 - 150:], r2[:150], r2[501 - 100:],
        r0[5:23], r0[5:24], b"", b"A", b"N" * 150,   # shorter than min_seed_len / exactly 19 / empty / all N
        r0[3000:3070] + b"N" * 10 + r0[3080:3150],
        r0[4000:4075] + r0[4090:4165],       # 15-base deletion
        r0[5000:5075] + b"ACGTACGTACGT" + r0[5075:5138],  # 12-base insertion
        r0[6000:6100] + r1[100:150],         # chimera across rows
        r0[7000:7100] + r0[9000:9050],       # split within a row
        b"ACGT" * 37,
    ]
    seqs, offs = read_arrays(reads)
    ids = synth.lrand48_ids_fast(len(reads))
    g = gpu.align_batch(seqs, offs, ids)
    o = orc.align_batch(seqs, offs, ids, 1)
    bad = compare_results(g, o)
    assert not bad, "\n".join(bad)
    assert g.cigar_of(g.rows_of(0)[0]) == "150M" and g.rows_of(0)[0]["mapq"] == 60
    assert len(g.rows_of(7)) == 0 and len(g.rows_of(9)) == 0 and len(g.rows_of(11)) == 0


def test_align_single_read_entry(gpu_lib):
    """nuclseq_search_bwa shape: one read per call, ids continue across calls (SURVEY.md A.10)."""
    rows = synth.reference_rows([80_000], seed=51)
    orc, gpu = build_pair(rows, O.sql_default_opts(1))
    seqs, offs, _ = synth.simulate_reads(rows, 5, 150, seed=52)
    ids = synth.lrand48_ids(5)[0]
    for i in range(5):
        read = seqs[int(offs[i]):int(offs[i + 1])]
        g = gpu.align_batch(read, np.array([0, 150], dtype=np.uint64))   # the index object draws its own ids
        o = orc.align_batch(read, np.array([0, 150], dtype=np.uint64), ids[i:i + 1], 1)
        bad = compare_results(g, o)
        assert not bad, "\n".join(bad)


def test_align_many_short_contigs(gpu_lib):
    """C5-like: thousands of short rows whose lengths are not multiples of 4 (inter-row filler bases in the
    text), max_occ = max(500, 2 * rows) by the reference's rule; reads flush with contig ends."""
    rng = np.random.default_rng(61)
    lens = rng.integers(500, 1501, size=3000)
    lens = (lens + (lens % 4 == 0)).tolist()
    rows = synth.reference_rows(lens, seed=62)
    orc, gpu = build_pair(rows, O.sql_default_opts(len(rows)))
    assert orc.opts.max_occ == 6000
    seqs, offs, _ = synth.simulate_reads(rows, 3000, 150, seed=63)
    extra = [rows[i].tobytes()[-150:] for i in range(0, 3000, 97)] + [rows[i].tobytes()[:150] for i in range(5, 3000, 101)]
    s2, o2 = read_arrays(extra)
    seqs = np.concatenate([seqs, s2]); offs = np.concatenate([offs, o2[1:] + offs[-1]])
    n = len(offs) - 1
    ids = synth.lrand48_ids_fast(n)
    g = gpu.align_batch(seqs, offs, ids)
    o = orc.align_batch(seqs, offs, ids, 4)
    bad = compare_results(g, o)
    assert not bad, "\n".join(bad)


def test_align_small_max_occ_and_options(gpu_lib):
    """max_occ below the repeat copy number => the k/step sampling rule, frac_rep > 0 and MAPQ scaling;
    non-default match score / penalties / band / zdrop / clip penalties flow through every kernel."""
    rows = synth.reference_rows([200_000], seed=71)
    rows = synth.plant_repeats(rows, n_families=4, copies=40, unit=(300, 500), divergence=0.0, seed=72)
    opts = O.Opts(17, 8, 2, 5, 7, 3, 60, 40, 5, 2, 4, 1)
    orc, gpu = build_pair(rows, opts)
    seqs, offs, _ = synth.simulate_reads(rows, 3000, 150, sub=0.02, ins=0.004, dele=0.004, seed=73)
    ids = synth.lrand48_ids_fast(3000)
    g = gpu.align_batch(seqs, offs, ids)
    o = orc.align_batch(seqs, offs, ids, 4)
    bad = compare_results(g, o)
    assert not bad, "\n".join(bad)
    assert (g.rows["frac_rep"] > 0).sum() > 0


def test_align_read_lengths_ragged(gpu_lib):
    """ragged batch: read lengths 19..700 in one call (the batch's max length sizes every per-warp scratch)"""
    rows = synth.reference_rows([150_000, 90_001], seed=81)
    orc, gpu = build_pair(rows, O.canonical_opts(2))
    rng = np.random.default_rng(82)
    reads = []
    cat = [r.tobytes() for r in rows]
    for i in range(600):
        ln = int(rng.choice([19, 20, 35, 76, 100, 151, 250, 400, 700]))
        r = int(rng.integers(0, 2)); p = int(rng.integers(0, len(cat[r]) - ln))
        t = bytearray(cat[r][p:p + ln])
        for k in range(len(t)):
            if rng.random() < 0.02:
                t[k] = b"ACGT"[int(rng.integers(0, 4))]
        reads.append(bytes(t))
    seqs, offs = read_arrays(reads)
    ids = synth.lrand48_ids_fast(len(reads))
    g = gpu.align_batch(seqs, offs, ids)
    o = orc.align_batch(seqs, offs, ids, 4)
    bad = compare_results(g, o)
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("opts_fn,rlen,err", [(O.canonical_opts, 1000, (0.02, 0.005, 0.005)), (O.sql_default_opts, 2500, (0.04, 0.03, 0.03)),
                                              (O.canonical_opts, 6000, (0.04, 0.03, 0.03))])
def test_align_long_reads(gpu_lib, opts_fn, rlen, err):
    """C4-like: reads long enough (> ~730 bp) for mem_flt_chained_seeds' per-seed local SW, many seeds per
    chain, wide-band ksw_extend2 with band retries, wide ksw_global2 tracebacks."""
    rows = synth.reference_rows([400_000, 250_003], seed=101)
    orc, gpu = build_pair(rows, opts_fn(2))
    n = 120 if rlen <= 2500 else 40
    seqs, offs, _ = synth.simulate_reads(rows, n, rlen, sub=err[0], ins=err[1], dele=err[2], seed=102 + rlen)
    ids = synth.lrand48_ids_fast(n)
    g = gpu.align_batch(seqs, offs, ids)
    o = orc.align_batch(seqs, offs, ids, 4)
    bad = compare_results(g, o)
    assert not bad, "\n".join(bad)
    assert o["counters"]["sw_calls"] > 0
    assert int(g.row_off[-1]) >= n


def _flat_cigars(res):
    """per-row CIGAR words concatenated in row order (independent of where the pool put them)"""
    off, n = res.rows["cigar_off"].astype(np.int64), res.rows["n_cigar"].astype(np.int64)
    if len(n) == 0 or n.sum() == 0:
        return np.zeros(0, dtype=np.uint32)
    idx = np.repeat(off - np.concatenate(([0], np.cumsum(n)[:-1])), n) + np.arange(n.sum())
    return res.cigar[idx]


def _own_result(gpu, call):
    """a result as the library hands it out (`call` fills the bsq_result pointer), so that bsq_result_tuples recognises it as its own"""
    from bioseqdb_b200._lib import BsqResult, check
    res = C.POINTER(BsqResult)()
    check(call(C.byref(res)))
    return res


def test_align_batch_chunked_pipeline(gpu_lib, monkeypatch):
    """bsq_align_batch cuts a large batch into chunks on two lanes (copies overlapped with compute): rows, their order
    and the rebased CIGAR offsets must equal the single-lane resident path's, and the oracle's on a sample.  With three chunks
    the lanes no longer hold the whole result: its tuples take the path that uploads rows and reads, and must equal the tuples
    the resident batch of the same reads serves."""
    from helpers import PARITY_FIELDS
    from bioseqdb_b200._lib import ptr
    monkeypatch.setenv("BSQ_CHUNK_READS", str(1 << 17))
    rows = synth.reference_rows([600_001, 400_003], seed=71)
    rows = synth.plant_repeats(rows, n_families=6, copies=6, unit=(200, 800), divergence=0.02)
    orc, gpu = build_pair(rows, O.sql_default_opts(2))
    n = 2 * (1 << 17) + 12_345                      # two full chunks and a ragged third
    seqs, offs, _ = synth.simulate_reads(rows, n, 100, sub=0.015, ins=0.002, dele=0.002, seed=72, n_frac=0.001)
    ids = synth.lrand48_ids_fast(n)
    g_res = _own_result(gpu, lambda p: gpu.L.bsq_align_batch(gpu.h, ptr(seqs), ptr(offs), ptr(ids), n, p))   # chunked
    chunked_launches = gpu.timing().launches
    g_tup = gpu._fetch_tuples(g_res, ptr(seqs), ptr(offs), 0)
    g = gpu._collect(g_res)
    gpu.upload(seqs, offs, ids); gpu.align_resident()
    # three pipeline passes; two would stay below three resident passes (the chunks add only a few copy kernels each)
    assert chunked_launches >= 3 * gpu.timing().launches
    r_res = _own_result(gpu, lambda p: gpu.L.bsq_result_download(gpu.h, p))
    r_tup = gpu._fetch_tuples(r_res, None, None, 0)      # served from the resident batch: nothing uploaded
    r = gpu._collect(r_res)
    assert np.array_equal(g.row_off, r.row_off)
    for f in PARITY_FIELDS:
        assert np.array_equal(g.rows[f], r.rows[f]), f
    assert np.array_equal(_flat_cigars(g), _flat_cigars(r))
    assert np.array_equal(g_tup.off, r_tup.off) and np.array_equal(g_tup.ref_match, r_tup.ref_match)
    assert np.array_equal(g_tup.data, r_tup.data)
    # the oracle on reads that straddle the chunk boundaries and the tail
    pick = np.concatenate([np.arange((1 << 17) - 600, (1 << 17) + 600), np.arange(2 * (1 << 17) - 600, 2 * (1 << 17) + 600), np.arange(n - 800, n)])
    s_offs = np.zeros(len(pick) + 1, dtype=np.uint64)
    lens = (offs[pick + 1] - offs[pick]).astype(np.int64)
    s_offs[1:] = np.cumsum(lens)
    s_seqs = np.concatenate([seqs[int(offs[i]):int(offs[i + 1])] for i in pick])
    o = orc.align_batch(s_seqs, s_offs, ids[pick], 4)
    cnt_g = np.diff(g.row_off.astype(np.int64))[pick]
    assert np.array_equal(cnt_g, np.diff(o["row_off"].astype(np.int64)))
    sel = np.concatenate([np.arange(int(g.row_off[i]), int(g.row_off[i + 1])) for i in pick]).astype(np.int64)
    for f in PARITY_FIELDS:
        assert np.array_equal(g.rows[f][sel], o["rows"][f]), f
    gc = _flat_cigars(type(g)(g.row_off, g.rows[sel], g.cigar))
    oo, on = o["rows"]["cigar_off"].astype(np.int64), o["rows"]["n_cigar"].astype(np.int64)
    oc = np.concatenate([o["cigar"][int(a):int(a + b)] for a, b in zip(oo, on)]) if on.sum() else np.zeros(0, dtype=np.uint32)
    assert np.array_equal(gc, oc)


def test_align_batch_chunked_fallback(gpu_lib, monkeypatch):
    """When the rows outgrow the result block extrapolated from the first chunk, the call drains both lanes and runs one
    plain pass: same rows as the resident path."""
    from helpers import PARITY_FIELDS
    monkeypatch.setenv("BSQ_TEST_TIGHT_RESULT", "1")
    rows = synth.reference_rows([300_001, 200_003], seed=81)
    _, gpu = build_pair(rows, O.sql_default_opts(2))
    n = 2 * (1 << 16) + 4321
    seqs, offs, _ = synth.simulate_reads(rows, n, 80, seed=82)
    ids = synth.lrand48_ids_fast(n)
    g = gpu.align_batch(seqs, offs, ids)
    assert gpu.timing().notes & 1                              # BSQ_NOTE_CHUNK_FALLBACK: the fallback really ran (the call itself succeeded)
    assert gpu.L.bsq_last_error() == b""                        # ... and a successful call leaves no error text behind
    gpu.upload(seqs, offs, ids); gpu.align_resident(); r = gpu.download_result()
    assert np.array_equal(g.row_off, r.row_off)
    for f in PARITY_FIELDS:
        assert np.array_equal(g.rows[f], r.rows[f]), f
    assert np.array_equal(_flat_cigars(g), _flat_cigars(r))


def test_small_batch_routing(gpu_lib):
    """Default routing of a small batch (warp-cooperative DP kernels instead of the thread-per-extension / thread-per-region ones):
    the smoke check -- 2000 reads against the oracle, bit for bit -- in a fresh process without this suite's BSQ_SMALL_BATCH_READS=0."""
    import os
    import subprocess
    import sys
    env = {k: v for k, v in os.environ.items() if k not in ("BSQ_SMALL_BATCH_READS", "BSQ_FIN_SHORT_LIST")}
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.smoke()"], cwd=root, env=env, capture_output=True, timeout=600)
    assert p.returncode == 0, (p.stdout.decode()[-1500:], p.stderr.decode()[-1500:])
    assert b"smoke ok" in p.stdout
