"""Index cache keyed by the CONTENT of the reference rows (SURVEY.md 8f-1).

The reference builds a fresh BwaIndex inside every SQL call (`bwa_index_from_query`, extension.cpp:211-236, called from
:326 and :359) and throws it away afterwards, so `nuclseq_search_bwa` is build-bound.  Here a built index stays resident
in HBM and is found again by a digest of what went into it: (id, length, packed payload, holes) of every row, in order.
Alignment options are not part of the key -- they do not influence the index (extension.cpp:220-231 writes them into
mem_opt_t, which only the aligner reads) -- and are applied to the cached handle on every lookup.

The reference's per-read id comes from glibc's process-wide lrand48 state, which survives across SQL calls of one
session; the cache therefore owns that state and lends it to whichever index serves a call.

With a `directory` the cache also has a disk tier, for what one process cannot keep: in PostgreSQL every backend is its own
process, and a new one would build the same index again.  A built index is written to `<directory>/<digest hex>.bsqidx`
(BwaIndex.save: atomic replace, the digest kept in the file's header) and a memory miss loads it from there when it exists.
A file that does not load (damaged, or written for other content) is rebuilt and replaced; a file that cannot be written
(disk full, read-only directory) costs the next process a build, never this call.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
from collections import OrderedDict

import numpy as np

from .sequence import NucleotideSequence, nuclseq_from_text


def rows_digest(rows) -> bytes:
    """rows: iterable of (id, NucleotideSequence).  Order matters (row order fixes the text, bwa.cpp:82-105)."""
    h = hashlib.blake2b(digest_size=16)
    for rid, seq in rows:
        h.update(np.array([int(rid), int(seq.len), len(seq.holes)], dtype=np.int64).tobytes())
        h.update(np.ascontiguousarray(seq.pac).tobytes())
        if len(seq.holes):
            h.update(np.ascontiguousarray(seq.holes).tobytes())
    return h.digest()


class BwaIndexCache:
    def __init__(self, device: int = 0, max_bytes: int = 96 << 30, factory=None, directory=None):
        """max_bytes: HBM budget for resident indexes (index arrays + derived arrays + batch pools, as reported by
        bsq_index_device_bytes).  factory(device) -> a BwaIndex-like object; defaults to the CUDA-backed BwaIndex.
        directory: where the disk tier keeps its index files (None: no disk tier)."""
        self.device, self.max_bytes = device, max_bytes
        self._factory = factory
        self.directory = directory
        self._lru: OrderedDict[bytes, object] = OrderedDict()
        self.hits = self.misses = self.evictions = 0
        self.disk_hits = self.disk_saves = self.disk_errors = 0
        self.lrand_state = 0

    def _new_index(self):
        if self._factory is not None:
            return self._factory(self.device)
        from .bwa import BwaIndex
        return BwaIndex(self.device)

    @staticmethod
    def _bytes_of(ix) -> int:
        if hasattr(ix, "device_bytes"):
            return int(ix.device_bytes())
        return 0

    def total_bytes(self) -> int:
        return sum(self._bytes_of(ix) for ix in self._lru.values())

    def get(self, rows, opts: dict | None = None):
        """bwa_index_from_query with a memory: rows = iterable of (id, text | NucleotideSequence); opts = the bwa_options
        composite as a dict (None fields take the reference's defaults).  Returns a built index."""
        rows = [(int(r), s if isinstance(s, NucleotideSequence) else nuclseq_from_text(s)) for r, s in rows]
        key = rows_digest(rows)
        ix = self._lru.get(key)
        if ix is not None:
            self._lru.move_to_end(key)
            self.hits += 1
        else:
            self.misses += 1
            # an empty reference builds nothing (bwa.cpp:108-109): there is no index to keep on disk
            path = self.file_path(key) if self.directory is not None and any(seq.len for _, seq in rows) else None
            ix = self._load(path, key) if path is not None and os.path.exists(path) else None
            if ix is None:
                ix = self._new_index()
                for rid, seq in rows:
                    ix.add_ref_sequence(rid, seq)
                ix.set_options_from_composite(opts)     # max_occ's default depends on the row count: set before build as the reference does
                ix.build()
                if path is not None:
                    self._save(ix, path, key)
            self._lru[key] = ix
            self._evict(keep=key)
        ix.set_options_from_composite(opts)
        return _Lease(self, ix)

    def file_path(self, key: bytes) -> str:
        return os.path.join(self.directory, key.hex() + ".bsqidx")

    def _load(self, path, key):
        """The index saved under `path` for `key`, or None when the file does not load (the caller rebuilds and replaces it)."""
        ix = self._new_index()
        try:
            ix.load(path, key=key)
        except (RuntimeError, OSError, ValueError):
            self.disk_errors += 1
            if hasattr(ix, "close"):
                ix.close()
            return None
        self.disk_hits += 1
        return ix

    def _save(self, ix, path, key):
        try:
            ix.save(path, key=key)
        except (RuntimeError, OSError, ValueError):
            self.disk_errors += 1            # the index is built and serves this call; only the next process pays
            return
        self.disk_saves += 1

    def _evict(self, keep):
        while len(self._lru) > 1 and self.total_bytes() > self.max_bytes:
            k = next(iter(self._lru))
            if k == keep:
                break
            old = self._lru.pop(k)
            if hasattr(old, "close"):
                old.close()
            self.evictions += 1

    def clear(self):
        for ix in self._lru.values():
            if hasattr(ix, "close"):
                ix.close()
        self._lru.clear()


class _Lease:
    """A cached index for the duration of one call: forwards to the index with the session's lrand48 state."""

    def __init__(self, cache: BwaIndexCache, ix):
        self._cache, self.index = cache, ix

    def _with_state(self, fn, *a):
        self.index._lrand_state = self._cache.lrand_state
        try:
            return fn(*a)
        finally:
            self._cache.lrand_state = self.index._lrand_state

    def align_sequence(self, seq):
        return self._with_state(self.index.align_sequence, seq)

    def align_batch(self, seqs, offs, ids=None):
        return self._with_state(self.index.align_batch, seqs, offs, ids)

    def __getattr__(self, name):
        return getattr(self.index, name)
