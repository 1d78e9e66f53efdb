"""Index files at the bench configurations: what a process pays to build an index, to save it, and to load it instead.

For each configuration (c2, c5, c3: synth.config_row_lengths with bench.py's seeds) one JSON line with
  build wall / device time, save wall time and file bytes,
  load wall time split into read + upload, device checksums, k_sa_from_samples (CUDA events) and host mirrors, plus the lane
  efficiency of the suffix-array rebuild,
  bsq_index_prepare of the loaded index, bsq_index_verify of the loaded index over every row,
  whether a sample of the bench's reads gives the same rows (row offsets, fields, CIGARs) through the built and the loaded index,
  the GPU's name and power limit.
The index files go to a temporary directory (the c3 file is 5.4 GB), which is deleted before exit.  Nothing here can drop the page
cache, so every load reads a file that was just written: the load figures are "file in page cache".

  python scripts/index_file.py [--configs c2,c5,c3] [--reads 20000] [--out DIR]
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bioseqdb_b200 import BwaIndex, BsqOpts, synth  # noqa: E402

LAYOUT = {"c2": "C2", "c5": "C5", "c3": "C3"}


def gpu_card():
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=60).stdout.strip()
    return out or None


def rows_digest(res) -> str:
    """SHA-1 of row offsets, every row field but cigar_off (a pool position) and the CIGAR words of every row."""
    dg = hashlib.sha1()
    dg.update(np.ascontiguousarray(res.row_off).tobytes())
    for name in res.rows.dtype.names:
        if name != "cigar_off":
            dg.update(np.ascontiguousarray(res.rows[name]).tobytes())
    for r in res.rows:
        dg.update(np.ascontiguousarray(res.cigar[int(r["cigar_off"]):int(r["cigar_off"]) + int(r["n_cigar"])]).tobytes())
    return dg.hexdigest()


def new_index(n_rows):
    ix = BwaIndex(0, BsqOpts(19, max(500, 2 * n_rows), 1, 4, 5, 5, 100, 100, 6, 6, 1, 1))   # bench.py's SQL options
    ix.set_rows_ext(False)
    return ix


def run(cfg, n_reads, tmpdir):
    lens = synth.config_row_lengths(LAYOUT[cfg])
    rows = synth.reference_rows(lens)
    seqs, offs, _ = synth.simulate_reads(rows, n_reads, 150, seed=synth.SEED_READS)
    ids = synth.lrand48_ids_fast(n_reads)
    path = os.path.join(tmpdir, "%s.bsqidx" % cfg)

    built = new_index(len(rows))
    built.add_ref_sequences(list(range(1, len(rows) + 1)), rows)
    t = time.perf_counter()
    built.build()
    build_wall = time.perf_counter() - t
    m = built.meta()
    t = time.perf_counter()
    built.save(path)
    save_wall = time.perf_counter() - t
    digest_built = rows_digest(built.align_batch(seqs, offs, ids))
    built.close()                      # at c3 two resident indexes with their inverse SAs would not fit beside each other

    ld = new_index(len(rows))
    load_ms = ld.load(path)
    info = ld.last_load()
    prep = C.c_float(0)
    ld.L.bsq_index_prepare(ld.h, C.byref(prep))
    chk = ld.verify(n_samples=1 << 40)
    digest_loaded = rows_digest(ld.align_batch(seqs, offs, ids))
    ld.close()
    os.unlink(path)
    return {
        "config": cfg, "ref_bases": int(sum(lens)), "ref_rows": len(lens), "seq_len": int(m.seq_len), "sa_bytes": int(m.sa_bytes),
        "build_wall_s": build_wall, "build_device_ms": float(m.build_ms),
        "save_wall_s": save_wall, "file_bytes": int(info["file_bytes"]),
        "load_wall_s": load_ms / 1e3, "load_note": "file in page cache (written just before; the page cache cannot be dropped here)",
        "load_read_upload_ms": info["read_ms"], "load_checksum_ms": info["checksum_ms"], "load_sa_from_samples_ms": info["sa_ms"],
        "load_host_mirrors_ms": info["host_ms"],
        "sa_lf_steps": int(info["lf_steps"]), "sa_lane_efficiency": info["lf_steps"] / max(1, info["lane_slots"]),
        "prepare_ms": float(prep.value),
        "verify": {"sound": chk["sound"], "exhaustive": chk["exhaustive"], "rows_checked": chk["rows_checked"], "ms": chk["ms"]},
        "sample_reads": n_reads, "rows_equal_built_vs_loaded": digest_built == digest_loaded, "rows_sha1": digest_loaded,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c2,c5,c3")
    ap.add_argument("--reads", type=int, default=20_000)
    ap.add_argument("--out", default=None, help="also write DIR/r03_index_file_<config>.json")
    args = ap.parse_args()
    card = gpu_card()
    for cfg in args.configs.split(","):
        tmpdir = tempfile.mkdtemp(prefix="bsqidx-")
        try:
            line = run(cfg, args.reads, tmpdir)
        finally:
            shutil.rmtree(tmpdir, ignore_errors=True)
        line["gpu"] = card
        s = json.dumps(line)
        print(s, flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, "r03_index_file_%s.json" % cfg), "w") as f:
                f.write(s + "\n")


if __name__ == "__main__":
    main()
