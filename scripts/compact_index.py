"""The compact index layout (1/32 of the suffix array in HBM, positions resolved by LF walks) against the full layout, on the bench
configurations.  The index is built once and saved; every run loads it into a fresh handle, alternating full and compact (the compact
runs set BSQ_TEST_COMPACT=1, so the load and bsq_index_prepare take the library's real selection code).  One JSON line per run with
  device bytes after bsq_index_prepare, load wall time and its device SA step (k_sa_from_samples, or the check of the samples),
  resident reads/s (bsq_align_resident, one batch of --reads, best of --steps after one warm-up) and e2e reads/s (bsq_align_batch),
  the resident call's stage times (seed, chain including the resolve pass, extend, finalize),
  SA lookups per read, and on the compact layout LF steps per lookup and the resolve pass's lane efficiency,
  whether the rows (every field and CIGAR) equal those of the first full run on the whole sample,
  the GPU's name and power limit.

  python scripts/compact_index.py [--configs c2] [--reads 1000000] [--runs 4] [--out DIR]
"""
from __future__ import annotations

import argparse
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
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from bioseqdb_b200 import synth  # noqa: E402
from index_file import LAYOUT, gpu_card, new_index, rows_digest  # noqa: E402


def one_run(path, n_rows, compact, seqs, offs, ids, steps):
    if compact:
        os.environ["BSQ_TEST_COMPACT"] = "1"
    else:
        os.environ.pop("BSQ_TEST_COMPACT", None)
    ix = new_index(n_rows)
    try:
        load_ms = ix.load(path)
        info = ix.last_load()
        ix.L.bsq_index_prepare(ix.h, None)
        dev_bytes = ix.device_bytes()
        m = ix.meta()
        n = len(offs) - 1
        ix.upload(seqs, offs, ids)
        ix.align_resident()                                # warm-up
        best = None
        for _ in range(steps):
            t = time.perf_counter()
            ix.align_resident()
            wall = time.perf_counter() - t
            T = ix.timing()
            if best is None or wall < best[0]:
                best = (wall, {k: float(getattr(T, k)) for k in ("seed", "chain", "extend", "finalize", "total")})
        res = ix.download_result()
        ix.set_counters(True)
        ix.align_resident()
        ctr = ix.counters()
        ctl = np.zeros(64, dtype=np.uint32)
        ix.L.bsq_debug_ctl(ix.h, ctl.ctypes.data)
        ix.set_counters(False)
        lf_steps = int(ctl[28]) | int(ctl[29]) << 32
        warp_iters = int(ctl[54]) | int(ctl[55]) << 32
        t = time.perf_counter()
        ix.align_batch(seqs, offs, ids)
        e2e = time.perf_counter() - t
        return {
            "layout": "compact" if m.sa_interval == 32 else "full", "sa_interval": int(m.sa_interval), "sa_bytes": int(m.sa_bytes),
            "device_bytes_after_prepare": int(dev_bytes), "load_wall_ms": load_ms, "load_sa_step_ms": info["sa_ms"],
            "resident_reads_per_s": n / best[0], "e2e_reads_per_s": n / e2e, "stage_ms": best[1],
            "sa_lookups_per_read": ctr["n_sa"] / n,
            "lf_steps_per_lookup": (lf_steps / ctr["n_sa"]) if m.sa_interval == 32 and ctr["n_sa"] else None,
            "resolve_lane_efficiency": (lf_steps / (32 * warp_iters)) if m.sa_interval == 32 and warp_iters else None,
        }, rows_digest(res)
    finally:
        ix.close()
        os.environ.pop("BSQ_TEST_COMPACT", None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c2")
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--runs", type=int, default=4, help="alternating full, compact, full, compact, ...")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write DIR/r03_compact_<config>.json (all runs, one line each)")
    args = ap.parse_args()
    card = gpu_card()
    for cfg in args.configs.split(","):
        lens = synth.config_row_lengths(LAYOUT[cfg])
        rows = synth.reference_rows(lens)
        seqs, offs, _ = synth.simulate_reads(rows, args.reads, 150, seed=synth.SEED_READS)
        ids = synth.lrand48_ids_fast(args.reads)
        tmpdir = tempfile.mkdtemp(prefix="bsqcompact-")
        lines = []
        try:
            path = os.path.join(tmpdir, "%s.bsqidx" % cfg)
            built = new_index(len(rows))
            built.add_ref_sequences(list(range(1, len(rows) + 1)), rows)
            built.build()
            built.save(path)
            built.close()
            ref_digest = None
            for i in range(args.runs):
                line, digest = one_run(path, len(rows), i % 2 == 1, seqs, offs, ids, args.steps)
                if ref_digest is None:
                    ref_digest = digest
                line.update({"config": cfg, "run": i, "reads": args.reads, "ref_bases": int(sum(lens)),
                             "rows_equal_first_full_run": digest == ref_digest, "rows_sha1": digest, "gpu": card})
                s = json.dumps(line)
                print(s, flush=True)
                lines.append(s)
                if args.out:                       # rewritten after every run: a long configuration keeps what it measured
                    os.makedirs(args.out, exist_ok=True)
                    with open(os.path.join(args.out, "r03_compact_%s.json" % cfg), "w") as f:
                        f.write("\n".join(lines) + "\n")
        finally:
            shutil.rmtree(tmpdir, ignore_errors=True)


if __name__ == "__main__":
    main()
