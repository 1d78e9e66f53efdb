#!/usr/bin/env python
"""One process, one host thread, N GPUs: bsq_multi_align_batch_datums on one batch of (reads_per_gpu x N) reads from pinned host memory,
rows of every device back in one pinned result (the shape of a PostgreSQL backend, reference extension.cpp:346-377).
  python scripts/bench_multi.py --gpus N [--config c2|c3] [--steps K] [--tuples]      (prints one JSON line; e2e only: host buffers in, host rows out)
With --tuples every timed step also materialises the bwa_result tuples of its result on every device (bsq_multi_result_tuples, served
from HBM), and the same run times the single-device route on the same result (bsq_result_tuples on the built handle, which stages the
rows and the ASCII reads on device 0) outside the timed steps."""
import argparse, ctypes as C, json, os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import bench  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=2); ap.add_argument("--config", default="c2"); ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--tuples", action="store_true")
    a = ap.parse_args()
    import torch
    from bioseqdb_b200 import BwaIndex, BsqOpts, MultiBwaIndex, _lib, synth
    from bioseqdb_b200.loader import nuclseq_image_block
    sys.argv = ["bench.py", "--config", a.config, "--gpus", str(a.gpus)]
    args = bench.parse()
    per = args.reads
    args.reads = per * a.gpus
    rows, seqs, offs, ids, _ = bench.workload(args, 0)
    ot = bench.opts_tuple(args, len(rows))
    ix = BwaIndex(0, BsqOpts(*ot))
    ix.add_ref_sequences(list(range(1, len(rows) + 1)), rows)
    t0 = time.time(); ix.build(); build_s = time.time() - t0
    t0 = time.time(); m = MultiBwaIndex(ix, list(range(a.gpus))); repl_s = time.time() - t0
    img, off, _ = nuclseq_image_block(seqs, offs, 0)
    img_pin = torch.from_numpy(img).pin_memory(); off_pin = torch.from_numpy(off.view(np.int64)).pin_memory()
    ix.set_rows_ext(False)
    n = args.reads
    res = C.POINTER(_lib.BsqResult)()
    tp = C.POINTER(_lib.BsqTuples)()
    tup = {"ms": 0.0, "bytes": 0, "single_ms": [], "single_wall_ms": []}
    if a.tuples:
        seqs_pin = torch.from_numpy(seqs).pin_memory(); offs_pin = torch.from_numpy(offs.view(np.int64)).pin_memory()

    def one():
        ix.session_lrand48(0)
        _lib.check(ix.L.bsq_multi_align_batch_datums(m.m, C.c_void_p(img_pin.data_ptr()), C.c_void_p(off_pin.data_ptr()), None, n, C.byref(res)))
        rows_n = int(res.contents.row_off[n])
        if a.tuples:
            _lib.check(ix.L.bsq_multi_result_tuples(m.m, res, None, None, 0, C.byref(tp)))
            tup["ms"] += float(tp.contents.device_ms); tup["bytes"] = int(tp.contents.n_bytes)
            ix.L.bsq_tuples_free(tp)
        ix.L.bsq_result_free(res)
        return rows_n

    def single_route():
        """the route without this call: bsq_result_tuples on the built handle stages the whole multi result on device 0"""
        ix.session_lrand48(0)
        _lib.check(ix.L.bsq_multi_align_batch_datums(m.m, C.c_void_p(img_pin.data_ptr()), C.c_void_p(off_pin.data_ptr()), None, n, C.byref(res)))
        w = time.time()
        _lib.check(ix.L.bsq_result_tuples(ix.h, res, C.c_void_p(seqs_pin.data_ptr()), C.c_void_p(offs_pin.data_ptr()), 0, C.byref(tp)))
        tup["single_wall_ms"].append(1e3 * (time.time() - w)); tup["single_ms"].append(float(tp.contents.device_ms))
        assert int(tp.contents.n_bytes) == tup["bytes"]
        ix.L.bsq_tuples_free(tp)
        ix.L.bsq_result_free(res)
    for _ in range(a.warmup):
        one()
    tup["ms"] = 0.0
    ms = 0.0; w0 = time.time()
    for _ in range(a.steps):
        rows_n = one(); ms += m.timing().total
    wall = time.time() - w0
    t = m.timing()
    extra = {}
    if a.tuples:
        single_route()                      # warm-up of the single-device route
        tup["single_ms"].clear(); tup["single_wall_ms"].clear()
        for _ in range(a.steps):
            single_route()
        import subprocess
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
        extra = {"e2e_rows_reads_per_s_device_time": n * a.steps / ((ms + tup["ms"]) * 1e-3), "e2e_rows_reads_per_s_wall": n * a.steps / wall,
                 "tuples_bytes_per_call": tup["bytes"], "tuples_ms_per_call_device_multi": tup["ms"] / a.steps,
                 "tuples_ms_per_call_device_single": sorted(tup["single_ms"]), "tuples_ms_per_call_wall_single": sorted(tup["single_wall_ms"]),
                 "gpus": [line.strip() for line in q.splitlines() if line.strip()][:a.gpus]}
    print(json.dumps({"what": "one process, one thread, %d GPUs: bsq_multi_align_batch_datums (host datum images in, one pinned result out)" % a.gpus,
                      "config": a.config, "n_gpus": a.gpus, "reads_per_call": n, "rows_per_call": rows_n,
                      "e2e_reads_per_s_device_time": n * a.steps / (ms * 1e-3), "e2e_reads_per_s_wall": n * a.steps / wall,
                      "ms_per_call_device": ms / a.steps, "ms_per_call_wall": 1e3 * wall / a.steps,
                      "h2d_bytes": int(t.h2d_bytes), "d2h_bytes": int(t.d2h_bytes), "launches": int(t.launches),
                      "index_build_s": build_s, "replicate_and_derive_s": repl_s, **extra}))


if __name__ == "__main__":
    main()
