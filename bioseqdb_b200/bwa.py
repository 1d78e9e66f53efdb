"""Python mirror of the reference's bwa adapter interface (bioseqdb/bwa.h:15-48): ``BwaIndex`` with
``add_ref_sequence`` / ``build`` / ``align_sequence`` and ``BwaMatch`` rows, plus the batched entry point
that replaces the per-read loop of ``nuclseq_multi_search_bwa`` (bioseqdb/extension.cpp:362-370).
Everything below the class runs on the GPU through the C ABI (include/bioseqdb_gpu.h)."""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import BsqMeta, BsqOpts, BsqResult, BsqTiming, EXT_ROW_DTYPE, PUB_ROW_DTYPE, ROW_DTYPE, check, ptr
from .sequence import NucleotideSequence, nuclseq_from_text, nuclseq_to_text

_CIGAR_CHR = "MIDNSHP=XB"  # htslib's table applied to bwa op codes (bwa.cpp:70-77): soft clip prints as 'N'


@dataclass
class BwaMatch:  # bwa.h:15-30
    ref_id: int
    ref_subseq: bytes
    ref_match_begin: int
    ref_match_end: int
    ref_match_len: int
    query_subseq: bytes
    query_match_begin: int
    query_match_end: int
    query_match_len: int
    is_primary: bool
    is_secondary: bool
    is_reverse: bool
    cigar: str
    score: int


def bwa_opts(min_seed_len=19, max_occ=None, match_score=1, mismatch_penalty=4, pen_clip3=5, pen_clip5=5, zdrop=100,
             bandwidth=100, o_del=6, o_ins=6, e_del=1, e_ins=1):
    """The SQL function bwa_opts() (bioseqdb--0.0.0.sql:175-194) INCLUDING its positional mix-up: the ROW is
    built as (..., o_del, o_ins, e_del, e_ins) but the composite's fields are (..., o_del, e_del, o_ins, e_ins),
    so a caller's o_ins lands in e_del and e_del in o_ins (SURVEY.md B#1). Returns the composite as a dict
    keyed by the field names the C side reads (extension.cpp:220-231); None = SQL NULL."""
    row = (min_seed_len, max_occ, match_score, mismatch_penalty, pen_clip3, pen_clip5, zdrop, bandwidth, o_del, o_ins, e_del, e_ins)
    names = ("min_seed_len", "max_occ", "match_score", "mismatch_penalty", "pen_clip3", "pen_clip5", "zdrop", "bandwidth",
             "o_del", "e_del", "o_ins", "e_ins")
    return dict(zip(names, row))


def cigar_to_string(words) -> str:
    return "".join("%d%s" % (int(w) >> 4, _CIGAR_CHR[int(w) & 0xF]) for w in words)


class AlignResult:
    """Rows of one batch: ``row_off`` (n+1), ``rows`` (ROW_DTYPE), ``cigar`` (u32 words)."""

    def __init__(self, row_off, rows, cigar):
        self.row_off, self.rows, self.cigar = row_off, rows, cigar

    def rows_of(self, i):
        return self.rows[int(self.row_off[i]):int(self.row_off[i + 1])]

    def cigar_of(self, row) -> str:
        return cigar_to_string(self.cigar[int(row["cigar_off"]):int(row["cigar_off"]) + int(row["n_cigar"])])


def nuclseq_image(s) -> bytes:
    """The NUCLSEQ datum as PostgreSQL stores it (sequence.h:18-38, alloc_raw_nucls sequence.cpp:59-69): varlena length word of an
    uncompressed 4-byte header, holes_num, len, the hole records, the packed codes."""
    import struct
    body = s.holes.tobytes() + s.pac.tobytes()
    return struct.pack("<III", (12 + len(body)) << 2, len(s.holes), s.len) + body


TUPLES_FIX_HOLE_OFFSETS, TUPLES_FIX_REVERSE = 1, 2   # opt-in fix-ups of bsq_result_tuples (SURVEY.md 8f-3)


class Tuples:
    """Result of BwaIndex.tuples: per row: images at off[3i] and off[3i+1], NUL-terminated CIGAR string at off[3i+2]."""

    def __init__(self, off, ref_match, data, device_ms):
        self.off, self.ref_match, self.data, self.device_ms = off, ref_match, data, device_ms

    def _image(self, at: int) -> bytes:
        size = int(np.frombuffer(self.data[at:at + 4].tobytes(), dtype="<u4")[0]) >> 2
        return self.data[at:at + size].tobytes()

    def ref_subseq(self, i: int) -> bytes:
        return self._image(int(self.off[3 * i]))

    def query_subseq(self, i: int) -> bytes:
        return self._image(int(self.off[3 * i + 1]))

    def cigar(self, i: int) -> str:
        return self.data[int(self.off[3 * i + 2]):int(self.off[3 * i + 3])].tobytes().split(b"\0", 1)[0].decode()


class BwaIndex:
    """BwaIndex of bioseqdb/bwa.h:32-48 over libbioseqdb_gpu.so."""

    def __init__(self, device: int = 0, opts: BsqOpts | None = None):
        self.L = _lib.lib()
        if opts is None:
            opts = BsqOpts()
            self.L.bsq_opts_init(C.byref(opts))
        self.options = opts
        self.h = self.L.bsq_index_new(C.byref(opts), device)
        if not self.h:
            raise _lib.BsqError(self.L.bsq_last_error().decode())
        self.device = device
        self.set_rows_ext(True)      # the Python mirror drives the parity tests: it asks for every field (bench's e2e leg switches it off)
        self.n_rows = 0
        self._refs = []  # ids of the reference rows added through this object (the rows themselves live in the library)

    def close(self):
        if getattr(self, "h", None):
            self.L.bsq_index_free(self.h)
            self.h = None

    def __del__(self):
        self.close()

    # ---- options: bwa_index_from_query's writes (extension.cpp:220-231)
    def set_options_from_composite(self, opts: dict | None):
        o = opts or {}

        def get(name, default):
            v = o.get(name)
            if v is None:
                return default
            if v < 0:
                raise ValueError("bwa_opt %s must be nonnegative" % name)
            return int(v)
        b = BsqOpts(get("min_seed_len", 19), get("max_occ", max(500, self.n_rows * 2)), get("match_score", 1), get("mismatch_penalty", 4),
                    get("pen_clip3", 5), get("pen_clip5", 5), get("zdrop", 100), get("bandwidth", 100),
                    get("o_del", 6), get("e_del", 1), get("o_ins", 6), get("e_ins", 1))
        self.set_options(b)

    def set_options(self, b: BsqOpts):
        check(self.L.bsq_index_set_opts(self.h, C.byref(b)))
        self.options = b

    # ---- reference rows
    def add_ref_sequence(self, ref_id: int, seq):
        if not isinstance(seq, NucleotideSequence):
            seq = nuclseq_from_text(seq)
        holes = np.ascontiguousarray(seq.holes)
        pac = np.ascontiguousarray(seq.pac)
        check(self.L.bsq_index_add_ref(self.h, int(ref_id), ptr(pac), seq.len, ptr(holes) if len(holes) else None, len(holes)))
        self._refs.append(int(ref_id))
        self.n_rows += 1

    def add_ref_sequences(self, ref_ids, texts):
        """Many reference rows in two calls: the texts become NUCLSEQ datums on the GPU (bsq_nuclseq_from_text_batch = nuclseq_in of
        every row) and the datum images go to bsq_index_add_ref_datums -- the batched form of the add_ref_sequence loop of
        bwa_index_from_query (extension.cpp:211-219).  texts: bytes or uint8 arrays of upper-case letters."""
        from ._lib import BsqNuclseqs
        n = len(texts)
        if n == 0:
            return
        arrs = [t if isinstance(t, np.ndarray) else np.frombuffer(bytes(t), dtype=np.uint8) for t in texts]
        offs = np.zeros(n + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(a) for a in arrs])
        ids = np.ascontiguousarray(ref_ids, dtype=np.int64)
        # rows are converted in groups of at most ~1 G bases so that the device staging stays bounded
        lo = 0
        while lo < n:
            hi = lo + 1
            while hi < n and int(offs[hi + 1] - offs[lo]) <= (1 << 30):
                hi += 1
            cat = np.concatenate(arrs[lo:hi]) if hi - lo > 1 else np.ascontiguousarray(arrs[lo])
            if len(cat) == 0:
                cat = np.zeros(1, dtype=np.uint8)
            rel = np.ascontiguousarray(offs[lo:hi + 1] - offs[lo])
            res = C.POINTER(BsqNuclseqs)()
            check(self.L.bsq_nuclseq_from_text_batch(self.device, ptr(cat), ptr(rel), hi - lo, C.byref(res)))
            try:
                r = res.contents
                check(self.L.bsq_index_add_ref_datums(self.h, hi - lo, ptr(ids[lo:hi]), C.cast(r.bytes, C.c_void_p), C.cast(r.off, C.c_void_p)))
            finally:
                self.L.bsq_nuclseqs_free(res)
            lo = hi
        self._refs.extend(int(i) for i in ids)
        self.n_rows += n

    def build(self):
        check(self.L.bsq_index_build(self.h))
        self._view = None

    def meta(self) -> BsqMeta:
        m = BsqMeta()
        check(self.L.bsq_index_get_meta(self.h, C.byref(m)))
        return m

    def save(self, path, key: bytes | None = None):
        """Write the built index to one file (bsq_index_save): pac, Occ, annotations, host state and every 32nd suffix-array entry.
        The file appears under `path` only when complete.  key: 16 opaque bytes kept in the header (BwaIndexCache stores its digest)."""
        check(self.L.bsq_index_save(self.h, os.fsencode(path), _key_arg(key)))

    def load(self, path, key: bytes | None = None) -> float:
        """Fill this fresh index (nothing added, not built) from a file written by save(); the full suffix array is rebuilt on the GPU.
        key: when given, the file's key must equal it.  Returns the wall milliseconds of the load."""
        ms = C.c_float(0)
        check(self.L.bsq_index_load(self.h, os.fsencode(path), _key_arg(key), C.byref(ms)))
        self.n_rows = int(self.meta().n_anns)        # max_occ's default counts the rows, as replica_finish does
        self._view = None
        return float(ms.value)

    def last_load(self) -> dict:
        """Where the last load() spent its time (bsq_index_last_load)."""
        from ._lib import BsqLoadInfo
        i = BsqLoadInfo()
        check(self.L.bsq_index_last_load(self.h, C.byref(i)))
        return {k: getattr(i, k) for k, _ in BsqLoadInfo._fields_}

    def verify(self, n_samples: int = 1 << 22, seed: int = 20261018) -> dict:
        """Device-side check of the index against its text (bsq_index_verify): every `*_bad` must be 0 and every `*_ok` 1."""
        from ._lib import BsqIndexCheck
        c = BsqIndexCheck()
        check(self.L.bsq_index_verify(self.h, int(n_samples), int(seed), C.byref(c)))
        d = {k: (float(getattr(c, k)) if k == "ms" else int(getattr(c, k))) for k, _ in BsqIndexCheck._fields_}
        d["sound"] = bool(d["sa_permutation_ok"] and d["l2_ok"] and not (d["sa_out_of_range"] or d["order_bad"] or d["bwt_bad"] or d["lf_bad"] or d["occ_bad"]))
        return d

    def device_bytes(self) -> int:
        b = C.c_uint64(0)
        check(self.L.bsq_index_device_bytes(self.h, C.byref(b)))
        return int(b.value)

    def download(self, what: int) -> np.ndarray:
        m = self.meta()
        n = int(m.arr_bytes[what])
        out = np.empty(n, dtype=np.uint8)
        check(self.L.bsq_index_download(self.h, what, ptr(out), n))
        return out

    def bwt_plain(self) -> np.ndarray:
        m = self.meta()
        out = np.zeros((int(m.seq_len) + 15) // 16, dtype=np.uint32)
        check(self.L.bsq_index_bwt_plain(self.h, ptr(out)))
        return out

    def sa_lookup(self, rows) -> np.ndarray:
        """bwt_sa of each row in [0, seq_len] (bsq_debug_sa_lookup): SA[row] on a full index, the LF walk of the alignment pipeline's
        position resolve pass on a compact one (meta().sa_interval == 32).  Row 0 gives seq_len."""
        r = np.ascontiguousarray(rows, dtype=np.uint64)
        out = np.empty(len(r), dtype=np.uint64)
        check(self.L.bsq_debug_sa_lookup(self.h, ptr(r), len(r), ptr(out)))
        return out

    def sa_sampled(self) -> np.ndarray:
        m = self.meta()
        n_sa = (int(m.seq_len) + 32) // 32
        out = np.zeros(n_sa, dtype=np.uint64)
        check(self.L.bsq_index_sa_sampled(self.h, ptr(out), n_sa))
        return out

    # ---- lrand48 ids: mem_align1 draws one per read (SURVEY.md A.10).  The library keeps the session's generator state in the handle
    # and draws the ids on the device whenever a call passes none; _lrand_state is a view of that state (the index cache moves it
    # from one cached index to the next, bioseqdb_b200/cache.py).
    @property
    def _lrand_state(self) -> int:
        return self.session_lrand48()

    @_lrand_state.setter
    def _lrand_state(self, v: int):
        self.session_lrand48(int(v))

    # ---- alignment
    def set_rows_ext(self, on: bool):
        """Ask for (or drop) the bsq_row_ext records: the mem_alnreg_t fields only parity checks read (hash, truesc, sub, ...)."""
        self.rows_ext = bool(on)
        self._apply_flags()

    def _apply_flags(self):
        check(self.L.bsq_index_set_flags(self.h, (_lib.FLAG_ROWS_EXT if self.rows_ext else 0) | (_lib.FLAG_TWO_CHUNKS if getattr(self, "two_chunks", False) else 0)))

    def _collect(self, res_p) -> AlignResult:
        r = res_p.contents
        n = int(r.n_reads)
        row_off = np.ctypeslib.as_array(r.row_off, shape=(n + 1,)).copy()
        total = int(row_off[n])
        rows = np.zeros(total, dtype=ROW_DTYPE)
        if total:
            pub = np.frombuffer((C.c_uint8 * (total * PUB_ROW_DTYPE.itemsize)).from_address(r.rows), dtype=PUB_ROW_DTYPE)
            for f in PUB_ROW_DTYPE.names:
                rows[f] = pub[f]
            if r.rows_ext:
                ext = np.frombuffer((C.c_uint8 * (total * EXT_ROW_DTYPE.itemsize)).from_address(r.rows_ext), dtype=EXT_ROW_DTYPE)
                for f in EXT_ROW_DTYPE.names:
                    rows[f] = ext[f]
        ncw = int(r.n_cigar_words)
        cigar = np.ctypeslib.as_array(r.cigar, shape=(max(ncw, 1),))[:ncw].copy()
        self.L.bsq_result_free(res_p)
        return AlignResult(row_off, rows, cigar)

    def align_batch(self, seqs: np.ndarray, offs: np.ndarray, ids: np.ndarray | None = None) -> AlignResult:
        """reads: concatenated ASCII bytes, offs (n+1). One call = the whole per-read loop of extension.cpp:362-370."""
        seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        n = len(offs) - 1
        if ids is not None:
            ids = np.ascontiguousarray(ids, dtype=np.int64)
        res = C.POINTER(BsqResult)()
        check(self.L.bsq_align_batch(self.h, ptr(seqs), ptr(offs), ptr(ids) if ids is not None else None, n, C.byref(res)))
        return self._collect(res)

    def align_batch_datums(self, data: np.ndarray, off: np.ndarray, ids: np.ndarray | None = None) -> AlignResult:
        """The same call with the reads as NUCLSEQ datum images (image i at data[off[i]:], off has n + 1 entries): what the PG glue holds
        for the query rows (extension.cpp:362) before to_text_palloc.  ids=None: the library continues the session's lrand48 stream."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = len(off) - 1
        if ids is not None:
            ids = np.ascontiguousarray(ids, dtype=np.int64)
        res = C.POINTER(BsqResult)()
        check(self.L.bsq_align_batch_datums(self.h, ptr(data), ptr(off), ptr(ids) if ids is not None else None, n, C.byref(res)))
        return self._collect(res)

    def align_tuples_raw(self, data_ptr: int, off_ptr: int, ids_ptr: int | None, n: int, flags: int = 0):
        """bench helper: one bsq_align_batch_datums call on raw (pinned) host pointers followed by bsq_result_tuples on its result, which
        the library serves from the still-resident batch.  Returns (device ms of both calls, bytes that came back)."""
        from ._lib import BsqTuples
        if not getattr(self, "two_chunks", False):
            self.two_chunks = True
            self._apply_flags()
        res = C.POINTER(BsqResult)()
        check(self.L.bsq_align_batch_datums(self.h, C.c_void_p(data_ptr), C.c_void_p(off_ptr), C.c_void_p(ids_ptr) if ids_ptr else None, n, C.byref(res)))
        t = self.timing()
        tp = C.POINTER(BsqTuples)()
        try:
            check(self.L.bsq_result_tuples(self.h, res, None, None, int(flags), C.byref(tp)))
            ms = float(t.total) + float(tp.contents.device_ms)
            nbytes = int(t.d2h_bytes) + int(tp.contents.n_bytes) + int(tp.contents.n_rows) * 36 + 8
            self.L.bsq_tuples_free(tp)
        finally:
            self.L.bsq_result_free(res)
        return ms, nbytes

    def align_tuples_datums(self, data: np.ndarray, off: np.ndarray, ids: np.ndarray | None = None, flags: int = 0):
        """Rows and their materialised columns in one go: bsq_align_batch_datums, then bsq_result_tuples served from the resident batch
        (no re-upload).  Returns (AlignResult, Tuples)."""
        if not getattr(self, "two_chunks", False):
            self.two_chunks = True
            self._apply_flags()
        data = np.ascontiguousarray(data, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = len(off) - 1
        if ids is not None:
            ids = np.ascontiguousarray(ids, dtype=np.int64)
        res = C.POINTER(BsqResult)()
        check(self.L.bsq_align_batch_datums(self.h, ptr(data), ptr(off), ptr(ids) if ids is not None else None, n, C.byref(res)))
        try:
            tup = self._fetch_tuples(res, None, None, flags)
        except Exception:
            self.L.bsq_result_free(res)
            raise
        return self._collect(res), tup

    def session_lrand48(self, state: int | None = None) -> int:
        """Read (state=None) or set the lrand48 state the library draws read ids from when a call passes none."""
        v = C.c_uint64(0 if state is None else state)
        check(self.L.bsq_session_lrand48(self.h, 0 if state is None else 1, C.byref(v)))
        return int(v.value)

    def upload(self, seqs, offs, ids):
        seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        ids = np.ascontiguousarray(ids, dtype=np.int64)
        check(self.L.bsq_reads_upload(self.h, ptr(seqs), ptr(offs), ptr(ids), len(offs) - 1))

    def align_resident(self):
        check(self.L.bsq_align_resident(self.h))

    def download_result(self) -> AlignResult:
        res = C.POINTER(BsqResult)()
        check(self.L.bsq_result_download(self.h, C.byref(res)))
        return self._collect(res)

    def tuples(self, res: AlignResult, seqs: np.ndarray, offs: np.ndarray, flags: int = 0) -> "Tuples":
        """Row materialisation on the GPU (SURVEY.md 8f-2): for every row of `res` the NUCLSEQ datum images of ref_subseq and
        query_subseq, the CIGAR string and ref_match_* -- what build_tuple_bwa (extension.cpp:282-305) assembles from a BwaMatch."""
        r, keep = _host_result(res)
        seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        return self._fetch_tuples(C.byref(r), ptr(seqs), ptr(offs), flags)

    def _fetch_tuples(self, res, seqs, offs, flags: int) -> "Tuples":
        """bsq_result_tuples on `res` (a pointer to a bsq_result; seqs / offs: the reads, or None when the library serves the result
        from its resident batch), copied out"""
        from ._lib import BsqTuples
        tp = C.POINTER(BsqTuples)()
        check(self.L.bsq_result_tuples(self.h, res, seqs, offs, int(flags), C.byref(tp)))
        return _take_tuples(self.L, tp)

    def timing(self) -> BsqTiming:
        t = BsqTiming()
        check(self.L.bsq_last_timing(self.h, C.byref(t)))
        return t

    def set_counters(self, on: bool):
        check(self.L.bsq_set_counters(self.h, int(on)))

    def counters(self) -> dict:
        v = np.zeros(8, dtype=np.uint64)
        check(self.L.bsq_get_counters(self.h, ptr(v)))
        names = ["n_extend", "n_sa", "dup_chain_pos", "ext_cells", "ext_calls", "ext_rows", "glb_cells", "glb_calls"]
        return {k: int(x) for k, x in zip(names, v)}

    def align_sequence(self, seq) -> list[BwaMatch]:
        """BwaIndex::align_sequence (bwa.cpp:141-181) for one read."""
        if not self.n_rows:
            return []
        text = nuclseq_to_text(seq) if isinstance(seq, NucleotideSequence) else bytes(seq)
        q = np.frombuffer(text, dtype=np.uint8)
        res = self.align_batch(q, np.array([0, len(q)], dtype=np.uint64))
        return self.matches(res, 0, text)

    def host_state(self) -> bytes:
        """The index's host-only state (ambiguity holes of the reference rows + their row numbers) as bsq_index_host_state_get writes it."""
        nb = C.c_uint64(0)
        check(self.L.bsq_index_host_state_size(self.h, C.byref(nb)))
        buf = np.zeros(int(nb.value), dtype=np.uint8)
        check(self.L.bsq_index_host_state_get(self.h, ptr(buf), int(nb.value)))
        return buf.tobytes()

    def replica_finish(self, host_state: bytes | None):
        """After the device arrays of a replica were filled (dist.broadcast_index): rebuild the library's host mirrors."""
        if host_state is None:
            check(self.L.bsq_index_replica_finish(self.h, None, 0))
        else:
            buf = np.frombuffer(host_state, dtype=np.uint8)
            check(self.L.bsq_index_replica_finish(self.h, ptr(buf), len(buf)))
        self.n_rows = int(self.meta().n_anns)
        self._view = None

    def _host_view(self):
        """(forward text as ASCII, row offsets, holes) read back from the library -- the same on the index that was built and on
        every replica of it, so ref_subseq does not depend on which rank answers."""
        v = getattr(self, "_view", None)
        if v is None:
            from ._lib import ARR_PAC, ARR_ANN_OFFSET, HOLE_DTYPE
            p = self.download(ARR_PAC)
            codes = np.empty((len(p), 4), dtype=np.uint8)
            codes[:, 0] = p >> 6; codes[:, 1] = (p >> 4) & 3; codes[:, 2] = (p >> 2) & 3; codes[:, 3] = p & 3
            cat = np.frombuffer(b"ACGT", dtype=np.uint8)[codes.reshape(-1)]
            offsets = self.download(ARR_ANN_OFFSET).view(np.int64)
            st = self.host_state()
            nh = int(np.frombuffer(st[:8], dtype="<u8")[0])
            holes = np.frombuffer(st[8:8 + 16 * nh], dtype=HOLE_DTYPE)
            v = self._view = (cat, offsets, holes)
        return v

    def matches(self, res: AlignResult, i: int, text: bytes) -> list[BwaMatch]:
        out = []
        m = self.meta()
        cat, offsets, holes = self._host_view()
        for row in res.rows_of(i):
            rid = int(row["rid"])
            ref_offset = int(offsets[rid])
            rb, re_ = int(row["rb"]), int(row["re"])
            out.append(BwaMatch(
                ref_id=int(row["ref_id"]),
                ref_subseq=self._ref_subseq(rb, re_, int(m.l_pac), cat, holes),
                ref_match_begin=_i32(rb - ref_offset), ref_match_end=_i32(re_ - ref_offset), ref_match_len=_i32(re_ - rb),
                query_subseq=text[int(row["qb"]):int(row["qe"])],
                query_match_begin=int(row["qb"]), query_match_end=int(row["qe"]), query_match_len=int(row["qe"] - row["qb"]),
                is_primary=(int(row["flag"]) & 0x100) == 0, is_secondary=(int(row["flag"]) & 0x100) != 0, is_reverse=bool(row["is_rev"]),
                cigar=res.cigar_of(row), score=int(row["score"])))
        return out

    @staticmethod
    def _ref_subseq(rb, re_, l_pac, cat, holes) -> bytes:
        """extract_reference_subseq (bwa.cpp:55-68). Forward hits: the reference's own arithmetic, holes
        overlaid with their un-rebased offsets (SURVEY.md B#2). Reverse hits index past the reference's
        vector (UB, B#3): defined here as the reverse-strand text."""
        comp = bytes.maketrans(b"ACGT", b"TGCA")
        if rb >= l_pac:
            fwd = cat[2 * l_pac - re_:2 * l_pac - rb].tobytes()
            out = bytearray(fwd.translate(comp)[::-1])
        else:
            out = bytearray(cat[rb:re_].tobytes())
        for h in holes:
            lo, hi = max(int(h["offset"]), rb), min(int(h["offset"]) + int(h["len"]), re_)
            for k in range(lo, hi):
                out[k - rb] = ord(h["amb"])
        return bytes(out)


class MultiBwaIndex:
    """One process, one thread, several GPUs (bsq_multi_*): the built index `ix` replicated to `devices` (devices[0] = ix.device), a
    batch split into contiguous blocks of reads, one result in read order.  Options / flags / the lrand48 session are those of `ix`."""

    def __init__(self, ix: BwaIndex, devices):
        self.ix = ix
        self.L = ix.L
        devs = np.ascontiguousarray(devices, dtype=np.int32)
        self.m = self.L.bsq_multi_new(ix.h, ptr(devs), len(devs))
        if not self.m:
            raise _lib.BsqError(self.L.bsq_last_error().decode())
        self.devices = list(int(d) for d in devs)

    def close(self):
        if getattr(self, "m", None):
            self.L.bsq_multi_free(self.m)
            self.m = None

    def __del__(self):
        self.close()

    def align_batch(self, seqs, offs, ids=None) -> AlignResult:
        seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        if ids is not None:
            ids = np.ascontiguousarray(ids, dtype=np.int64)
        res = C.POINTER(BsqResult)()
        check(self.L.bsq_multi_align_batch(self.m, ptr(seqs), ptr(offs), ptr(ids) if ids is not None else None, len(offs) - 1, C.byref(res)))
        return self.ix._collect(res)

    def align_batch_datums(self, data, off, ids=None) -> AlignResult:
        data = np.ascontiguousarray(data, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        if ids is not None:
            ids = np.ascontiguousarray(ids, dtype=np.int64)
        res = C.POINTER(BsqResult)()
        check(self.L.bsq_multi_align_batch_datums(self.m, ptr(data), ptr(off), ptr(ids) if ids is not None else None, len(off) - 1, C.byref(res)))
        return self.ix._collect(res)

    def timing(self) -> BsqTiming:
        t = BsqTiming()
        check(self.L.bsq_multi_last_timing(self.m, C.byref(t)))
        return t

    def tuples(self, res: AlignResult, seqs: np.ndarray, offs: np.ndarray, flags: int = 0) -> Tuples:
        """BwaIndex.tuples on every device (bsq_multi_result_tuples): each device materialises the rows of its block of reads.  A host
        result is staged: every device uploads its block's rows, CIGAR words and reads."""
        r, keep = _host_result(res)
        seqs = np.ascontiguousarray(seqs, dtype=np.uint8)
        offs = np.ascontiguousarray(offs, dtype=np.uint64)
        return self._fetch_tuples(C.byref(r), ptr(seqs), ptr(offs), flags)

    def _fetch_tuples(self, res, seqs, offs, flags: int) -> Tuples:
        from ._lib import BsqTuples
        tp = C.POINTER(BsqTuples)()
        check(self.L.bsq_multi_result_tuples(self.m, res, seqs, offs, int(flags), C.byref(tp)))
        return _take_tuples(self.L, tp)

    def align_tuples_datums(self, data, off, ids=None, flags: int = 0):
        """bsq_multi_align_batch_datums, then the tuples of its result, which every device serves from its resident block (no
        re-upload, no reads passed).  Returns (AlignResult, Tuples)."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        if ids is not None:
            ids = np.ascontiguousarray(ids, dtype=np.int64)
        res = C.POINTER(BsqResult)()
        check(self.L.bsq_multi_align_batch_datums(self.m, ptr(data), ptr(off), ptr(ids) if ids is not None else None, len(off) - 1, C.byref(res)))
        try:
            tup = self._fetch_tuples(res, None, None, flags)
        except Exception:
            self.L.bsq_result_free(res)
            raise
        return self.ix._collect(res), tup

    def align_tuples_raw(self, data_ptr: int, off_ptr: int, ids_ptr: int | None, n: int, flags: int = 0):
        """bench helper, as BwaIndex.align_tuples_raw: one bsq_multi_align_batch_datums call on raw (pinned) host pointers, then
        bsq_multi_result_tuples on its result.  Returns (device ms of both calls, bytes that came back, tuple bytes)."""
        from ._lib import BsqTuples
        res = C.POINTER(BsqResult)()
        check(self.L.bsq_multi_align_batch_datums(self.m, C.c_void_p(data_ptr), C.c_void_p(off_ptr), C.c_void_p(ids_ptr) if ids_ptr else None, n, C.byref(res)))
        t = self.timing()
        tp = C.POINTER(BsqTuples)()
        try:
            check(self.L.bsq_multi_result_tuples(self.m, res, None, None, int(flags), C.byref(tp)))
            ms = float(t.total) + float(tp.contents.device_ms)
            tb = int(tp.contents.n_bytes)
            nbytes = int(t.d2h_bytes) + tb + int(tp.contents.n_rows) * 36 + 8
            self.L.bsq_tuples_free(tp)
        finally:
            self.L.bsq_result_free(res)
        return ms, nbytes, tb


def _host_result(res: AlignResult):
    """A bsq_result over the arrays of a host AlignResult; the second value keeps those arrays alive."""
    row_off = np.ascontiguousarray(res.row_off, dtype=np.uint64)
    rows = np.zeros(len(res.rows), dtype=PUB_ROW_DTYPE)
    for f in PUB_ROW_DTYPE.names:
        rows[f] = res.rows[f]
    cigar = np.ascontiguousarray(res.cigar, dtype=np.uint32)
    r = BsqResult()
    r.n_reads = len(row_off) - 1
    r.row_off = row_off.ctypes.data_as(C.POINTER(C.c_uint64))
    r.rows = rows.ctypes.data
    r.cigar = cigar.ctypes.data_as(C.POINTER(C.c_uint32))
    r.n_cigar_words = len(cigar)
    return r, (row_off, rows, cigar)


def _take_tuples(L, tp) -> Tuples:
    """Copies a bsq_tuples out of the library's pinned block and frees it."""
    t = tp.contents
    n = int(t.n_rows)
    off = np.ctypeslib.as_array(t.off, shape=(3 * n + 1,)).copy()
    ref_match = np.ctypeslib.as_array(t.ref_match, shape=(max(3 * n, 1),))[:3 * n].copy().reshape(n, 3)
    nb = int(t.n_bytes)
    data = np.ctypeslib.as_array(t.bytes, shape=(max(nb, 1),))[:nb].copy()
    ms = float(t.device_ms)
    L.bsq_tuples_free(tp)
    return Tuples(off, ref_match, data, ms)


def _key_arg(key):
    if key is None:
        return None
    key = bytes(key)
    if len(key) != 16:
        raise ValueError("an index file key is 16 bytes")
    return key


def _i32(v: int) -> int:
    v &= 0xFFFFFFFF
    return v - (1 << 32) if v & 0x80000000 else v
