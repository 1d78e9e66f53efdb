"""The disk tier of BwaIndexCache (index files shared by processes): hit, miss and write-through, recovery from a file that does not load,
a write that fails, empty references, and no disk tier without a directory -- host logic only, with a stand-in index that records its
save / load calls."""
import ast
import os

import pytest

from bioseqdb_b200 import synth
from bioseqdb_b200.cache import BwaIndexCache, rows_digest
from bioseqdb_b200.sequence import nuclseq_from_text


class DiskIndex:
    """Stand-in for BwaIndex: save writes the key and the rows, load reads them back and fails like the library on a wrong key or a
    damaged file."""
    log = []
    fail_save = False

    def __init__(self, device):
        self.rows, self.opts, self.is_built, self.loaded, self.closed, self._lrand_state = [], None, False, False, False, 0

    def add_ref_sequence(self, rid, seq):
        self.rows.append((rid, seq.len))

    def set_options_from_composite(self, o):
        self.opts = o

    def build(self):
        self.is_built = True
        DiskIndex.log.append(("build",))

    def save(self, path, key=None):
        DiskIndex.log.append(("save", path, key))
        if DiskIndex.fail_save:
            raise OSError(28, "No space left on device")
        with open(path, "wb") as f:
            f.write(b"IDX" + key + repr(self.rows).encode())

    def load(self, path, key=None):
        DiskIndex.log.append(("load", path, key))
        with open(path, "rb") as f:
            data = f.read()
        if not data.startswith(b"IDX"):
            raise RuntimeError("bsq_index_load: %s is not an index file (wrong magic)" % path)
        if data[3:19] != key:
            raise RuntimeError("bsq_index_load: %s: key mismatch" % path)
        self.rows, self.loaded = ast.literal_eval(data[19:].decode()), True

    def device_bytes(self):
        return 100

    def close(self):
        self.closed = True


@pytest.fixture(autouse=True)
def _reset():
    DiskIndex.log, DiskIndex.fail_save = [], False


def _rows(seed, n=3):
    return [(i + 1, r.tobytes()) for i, r in enumerate(synth.reference_rows([50 + 7 * i for i in range(n)], seed=seed))]


def _key(rows):
    return rows_digest([(rid, nuclseq_from_text(t)) for rid, t in rows])


def _ops():
    return [e[0] for e in DiskIndex.log]


def test_miss_writes_through_and_other_process_loads(tmp_path):
    rows = _rows(1)
    a = BwaIndexCache(factory=DiskIndex, directory=str(tmp_path))
    la = a.get(rows, {"min_seed_len": 21})
    path = str(tmp_path / (_key(rows).hex() + ".bsqidx"))
    assert a.file_path(_key(rows)) == path and os.path.exists(path)
    assert _ops() == ["build", "save"] and DiskIndex.log[1][1:] == (path, _key(rows))
    assert (a.misses, a.disk_hits, a.disk_saves, a.disk_errors) == (1, 0, 1, 0) and la.index.is_built
    assert a.get(rows).index is la.index and _ops() == ["build", "save"]          # a memory hit touches no file
    b = BwaIndexCache(factory=DiskIndex, directory=str(tmp_path))                 # another process: loads, builds nothing
    lb = b.get(rows, {"min_seed_len": 23})
    assert _ops() == ["build", "save", "load"] and DiskIndex.log[2][1:] == (path, _key(rows))
    assert lb.index.loaded and not lb.index.is_built and lb.index.rows == la.index.rows
    assert lb.index.opts == {"min_seed_len": 23}                                   # options are applied after the load
    assert (b.misses, b.disk_hits, b.disk_saves, b.disk_errors) == (1, 1, 0, 0)
    other = _rows(2)
    b.get(other)
    assert _ops()[-2:] == ["build", "save"] and len(os.listdir(tmp_path)) == 2    # one file per reference


@pytest.mark.parametrize("damage", ["garbage", "other key"])
def test_failed_load_rebuilds_and_replaces(tmp_path, damage):
    rows = _rows(3)
    path = tmp_path / (_key(rows).hex() + ".bsqidx")
    path.write_bytes(b"garbage" if damage == "garbage" else b"IDX" + b"\0" * 16 + b"[]")
    c = BwaIndexCache(factory=DiskIndex, directory=str(tmp_path))
    lease = c.get(rows)
    assert _ops() == ["load", "build", "save"] and lease.index.is_built
    assert (c.disk_hits, c.disk_saves, c.disk_errors) == (0, 1, 1)
    assert path.read_bytes().startswith(b"IDX" + _key(rows))                       # replaced by a good file
    d = BwaIndexCache(factory=DiskIndex, directory=str(tmp_path))
    assert d.get(rows).index.loaded and d.disk_hits == 1


def test_failed_save_does_not_fail_the_call(tmp_path):
    DiskIndex.fail_save = True
    c = BwaIndexCache(factory=DiskIndex, directory=str(tmp_path))
    lease = c.get(_rows(4))
    assert lease.index.is_built
    assert (c.disk_saves, c.disk_errors) == (0, 1) and os.listdir(tmp_path) == []


def test_empty_reference_is_not_written(tmp_path):
    c = BwaIndexCache(factory=DiskIndex, directory=str(tmp_path))
    c.get([])
    c.get([(1, b"")])
    assert _ops() == ["build", "build"] and os.listdir(tmp_path) == []
    assert (c.disk_hits, c.disk_saves, c.disk_errors) == (0, 0, 0)


def test_no_directory_no_disk_tier(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    c = BwaIndexCache(factory=DiskIndex)
    a = c.get(_rows(5))
    assert c.get(_rows(5)).index is a.index
    assert _ops() == ["build"] and os.listdir(tmp_path) == []
    assert (c.hits, c.misses, c.disk_hits, c.disk_saves, c.disk_errors) == (1, 1, 0, 0, 0)
