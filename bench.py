#!/usr/bin/env python
"""bench.py -- 150 bp reads aligned per second through the bwa hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c1|c2|c3|c4|c5] [--dump-outputs DIR]

A step = one pass of the hot path (seed -> chain -> extend -> finalize -> rows in read order with MAPQ) over one batch of
simulated reads against the resident FM-index.  --config picks a BASELINE.json configuration with BASELINE.md's exact row layout
(default c2 = configs[1]: 1 M simulated 150 bp reads, 1 % error, vs 10 rows x 10 Mbp on one B200; "SQL default" options, i.e. what
bwa_opts() really delivers, SURVEY.md B#1):

  c1  configs[0]  10 k x 150 bp reads vs 5 x 1 Mbp
  c2  configs[1]  1 M x 150 bp reads vs 10 x 10 Mbp                                   <- the line the driver records
  c3  configs[2]  10 M x 150 bp reads vs 24 human-chromosome-proportional rows, 3.1 Gbp: 1.25 M reads per GPU (10 M at N = 8)
  c4  configs[3]  100 k x 10 kbp reads (10 % error) vs the c2 reference: 12.5 k reads per GPU (100 k at N = 8)
  c5  configs[4]  1 M x 150 bp reads vs 500 k contigs of 500-1500 bp (index build reported in `index`)

  value     whole-job reads/s with the reads already resident in HBM (device time, CUDA events on the library's launching stream,
            max over ranks)
  e2e       the same metric through the C-ABI call bsq_align_batch with HOST buffers: pinned host reads in, host rows out, H2D and
            D2H inside the timed region
  roofline  for the dominant kernel; cpu_baseline = the CPU oracle on this box's host cores (bounded sample), with `parity`: the
            oracle's rows compared with the GPU's for every read of that sample (all 24 parity fields + CIGAR words)

--impl reference times the CPU path only (the reference cannot be compiled here -- no PostgreSQL / libbwa sources -- so this is the
oracle port, all host threads, bounded sample per step).  N > 1 (torchrun): the index is built on rank 0 and broadcast over NCCL,
reads are sharded per rank (weak scaling: every rank aligns its own batch), no collective in the per-read path.

PARITY UNPINNED: the oracle restates lh3/bwa from its published algorithm; no libbwa binary or reference-held vector exists to pin
it (DESIGN.md section 5).  Every ratio this file prints is against that oracle.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from bioseqdb_b200 import synth  # noqa: E402

METRIC = "150bp_reads_aligned_per_sec"
UNIT = "reads/s"

# BASELINE.md section 3: (rows layout, reads per GPU, read length, error rates sub/ins/del, BASELINE.json configs index)
CONFIGS = {
    "c1": ("C1", 10_000, 150, "0.008,0.001,0.001", 0),
    "c2": ("C2", 1_000_000, 150, "0.008,0.001,0.001", 1),
    "c3": ("C3", 1_250_000, 150, "0.008,0.001,0.001", 2),
    "c4": ("C2", 12_500, 10_000, "0.04,0.03,0.03", 3),
    "c5": ("C5", 1_000_000, 150, "0.008,0.001,0.001", 4),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--reads", type=int, default=None, help="reads per GPU (default: the configuration's)")
    ap.add_argument("--ref-mbp", type=int, default=None, help="ad hoc reference of 10 equal rows instead of the configuration's layout")
    ap.add_argument("--repeats", action="store_true", help="plant repeat families in the reference (SURVEY.md 8d realism knob: 4 families x 8 copies per Mbp, 300-6000 bp, 2 %% divergence)")
    ap.add_argument("--opts", default="sql", choices=["sql", "canonical"])
    ap.add_argument("--read-len", type=int, default=None)
    ap.add_argument("--err", default=None, help="substitution,insertion,deletion rates per base")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU seconds of the cpu_baseline sample")
    ap.add_argument("--no-extras", action="store_true", help="skip the tuple / loader / microbenchmark probes after the timed legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the rows of the last timed step (rank 0) to DIR/*.npy for a fixed, seeded sample of reads (dump_sample, "
                         "dump_outputs); --impl reference writes the oracle's rows for the same reads")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    layout, reads, rlen, err, idx = CONFIGS[args.config]
    args.layout = layout
    args.baseline_index = idx
    if args.reads is None:
        args.reads = reads
    if args.read_len is None:
        args.read_len = rlen
    if args.err is None:
        args.err = err
    return args


def reference_rows(args):
    if args.ref_mbp is not None:
        lens = [args.ref_mbp * 1_000_000 // 10] * 10
    else:
        lens = synth.config_row_lengths(args.layout)
    rows = synth.reference_rows(lens)
    if args.repeats:
        mbp = max(1, int(sum(lens) // 1_000_000))
        rows = synth.plant_repeats(rows, n_families=max(20, 4 * mbp), copies=8)
    args.ref_bases = int(sum(lens))
    args.ref_rows = len(lens)
    return rows


def workload(args, rank):
    rows = reference_rows(args)
    sub, ins, dele = [float(x) for x in args.err.split(",")]
    seqs, offs, truth = synth.simulate_reads(rows, args.reads, args.read_len, sub=sub, ins=ins, dele=dele, seed=synth.SEED_READS + rank,
                                             chunk=max(1, min(200_000, 40_000_000 // max(args.read_len, 1))))
    ids = synth.lrand48_ids_fast(args.reads)
    return rows, seqs, offs, ids, truth


def opts_tuple(args, n_rows):
    # (min_seed_len, max_occ, a, b, clip3, clip5, zdrop, w, o_del, e_del, o_ins, e_ins)
    if args.opts == "sql":
        return (19, max(500, 2 * n_rows), 1, 4, 5, 5, 100, 100, 6, 6, 1, 1)
    return (19, max(500, 2 * n_rows), 1, 4, 5, 5, 100, 100, 6, 1, 6, 1)


def config_dict(args):
    """The same dict in both arms (the driver compares them)."""
    if args.ref_mbp is not None:
        ref = "%d Mbp synthetic reference (10 equal rows, ad hoc)" % args.ref_mbp
    else:
        ref = {"C1": "5 rows x 1 Mbp", "C2": "10 rows x 10 Mbp", "C3": "24 human-chromosome-proportional rows, 3.1 Gbp",
               "C5": "500 k contigs of 500-1500 bp (lengths not multiples of 4)"}[args.layout]
    standard = args.ref_mbp is None and (args.reads, args.read_len, args.err) == CONFIGS[args.config][1:4] and not args.repeats
    return {"workload": ("BASELINE configs[%d]: " % args.baseline_index if standard else "ad hoc: ") +
                        "%d simulated %d bp reads (error sub/ins/del %s) per GPU vs %s%s, index resident" % (
                            args.reads, args.read_len, args.err, ref, ", repeat families planted" if args.repeats else ""),
            "config": args.config,
            "options": "SQL default (o_del 6, e_del 6, o_ins 1, e_ins 1)" if args.opts == "sql" else "canonical bwa (6/1/6/1)",
            "reads_per_gpu": args.reads, "read_len": args.read_len, "ref_layout": args.layout if args.ref_mbp is None else "10 equal rows",
            "l2_policy": "per-step working set (FM-index + full SA + batch pools, > 1 GB) exceeds the 126 MB L2; no explicit flush",
            "parallelism": "reads sharded over %d GPU(s), index replicated" % args.gpus}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index):
        self.rows = []
        self.stop = threading.Event()
        self.idx = gpu_index
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = max(int(r[1]) for r in self.rows if r[1].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(self.rows)}


def seed_traffic(args):
    """dram__bytes_read + dram__bytes_write of one launch of the dominant seeding kernel from the committed ncu --set full capture of
    THIS workload (profiles/seed_traffic.json: one record per profiled workload and kernel version); None for any other workload."""
    path = os.path.join(ROOT, "profiles", "seed_traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)
    except (OSError, ValueError):
        return None
    for rec in (t if isinstance(t, list) else [t]):
        w = rec.get("workload", {})
        if w.get("config") == args.config and w.get("reads") == args.reads and w.get("read_len") == args.read_len and w.get("opts") == args.opts \
                and args.ref_mbp is None and not args.repeats:
            return rec
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def sized_sample(orc, args, seqs, offs, ids, cores):
    """Reads of the workload that cost about --cpu-seconds of all-core CPU work (probed), capped at the batch."""
    probe = max(16, min(20_000, args.reads, 3_000_000 // max(args.read_len, 1)))
    r = orc.align_batch(seqs[:int(offs[probe])], offs[:probe + 1], ids[:probe], cores)
    rate = probe / max(r["seconds"], 1e-9)
    return int(min(args.reads, max(probe, rate * args.cpu_seconds))), probe, rate


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args, rank, world):
    if rank != 0:
        return
    import oracle_lib as O
    rows, seqs, offs, ids, _truth = workload(args, 0)
    cores = os.cpu_count() or 1
    ot = opts_tuple(args, len(rows))
    orc = O.OracleIndex(O.Opts(*ot))
    for i, r in enumerate(rows):
        orc.add_ref_text(i + 1, r.tobytes())
    if args.ref_bases * 2 >= (1 << 31):
        # the reference itself cannot index this text (is_bwt takes an int length, bwa.cpp:10,26,47) and the oracle's SA-IS would run for
        # the better part of an hour: the FM-index arrays (mathematically unique) are taken from the GPU build; the timed path is alignment only
        from bioseqdb_b200 import BwaIndex, BsqOpts
        ix = BwaIndex(0, BsqOpts(*ot))
        ix.add_ref_sequences(list(range(1, len(rows) + 1)), rows)
        ix.build()
        orc.adopt(ix.bwt_plain(), int(ix.meta().primary), ix.sa_sampled())
        ix.close()
        how = "FM-index arrays adopted from the GPU build (the reference's is_bwt(int n) cannot index this text; not in the step)"
    else:
        build_s = orc.build()
        how = "index built once by the oracle's SA-IS in %.1f s (not in the step)" % build_s
    sample, _probe, _rate = sized_sample(orc, args, seqs, offs, ids, cores)
    times = []
    for s in range(args.warmup + args.steps):
        r = orc.align_batch(seqs[:int(offs[sample])], offs[:sample + 1], ids[:sample], cores)
        if s >= args.warmup:
            times.append(r["seconds"])
    if args.dump_outputs:
        # the timed batch size comes from a timing probe; the dump covers dump_sample's reads, as the GPU arm's does, aligned once more
        pick = dump_sample(args.reads, args.read_len)
        lens = (offs[pick + 1] - offs[pick]).astype(np.int64)
        d = orc.align_batch(seqs[ranges(offs[pick], lens)], np.concatenate(([0], np.cumsum(lens))), ids[pick], cores)
        dump_outputs(args.dump_outputs, pick, d["row_off"], d["rows"], d["cigar"], at=np.arange(len(pick)))
    total = sum(times)
    value = sample * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
        "data": "synthetic", "config": config_dict(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d of %d reads per step, all %d host threads; %s" % (sample, args.reads, cores, how)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "parity_pinning": "unpinned (oracle restates lh3/bwa; no libbwa binary or reference vector to pin it)",
        "note": "the reference cannot be compiled in this image (no PostgreSQL, libbwa, htslib sources): this arm is the CPU oracle port of the same path",
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ outputs
def ranges(starts, counts):
    """Indices of the concatenated ranges [starts[i], starts[i] + counts[i])."""
    counts = np.asarray(counts, dtype=np.int64)
    return np.repeat(np.asarray(starts, dtype=np.int64) - (np.cumsum(counts) - counts), counts) + np.arange(int(counts.sum()), dtype=np.int64)


def rows_digest(res):
    """SHA-1 over everything the step produced (row offsets, row fields, CIGAR words): two builds / code paths compare run to run."""
    import hashlib
    total_rows = int(res.row_off[-1])
    dg = hashlib.sha1()
    dg.update(np.ascontiguousarray(res.row_off).tobytes())
    rr = res.rows[:total_rows]
    for name in rr.dtype.names:
        if name != "cigar_off":            # pool positions depend on the order warps allocate in; the words they point at do not
            dg.update(np.ascontiguousarray(rr[name]).tobytes())
    if total_rows:
        dg.update(np.ascontiguousarray(res.cigar[ranges(rr["cigar_off"], rr["n_cigar"])]).tobytes())
    return dg.hexdigest()


DUMP_BYTES = 64 << 20
DUMP_READS = 1 << 16          # sampled 150 bp reads; longer reads are sampled fewer in proportion
DUMP_SEED = 20261021


def dump_sample(n, read_len):
    """The reads a dump covers, in read order: a seeded choice fixed by the batch size and the read length alone."""
    k = min(n, max(1, DUMP_READS * 150 // max(read_len, 150)))
    return np.sort(np.random.Generator(np.random.PCG64(DUMP_SEED)).permutation(n)[:k])


def _dump_arrays(read_index, row_off, rows, cigar, at):
    row_off = np.asarray(row_off, dtype=np.int64)
    counts = row_off[at + 1] - row_off[at]
    rr = rows[ranges(row_off[at], counts)]
    out = {"read_index": read_index.astype(np.float64), "rows_per_read": counts.astype(np.float64)}
    for name in rr.dtype.names:
        v = rr[name]
        if name == "cigar_off":
            continue
        if v.dtype.kind in "iu" and v.dtype.itemsize == 8:
            out["row_%s_hi" % name] = (v >> v.dtype.type(32)).astype(np.float64)
            out["row_%s_lo" % name] = (v & v.dtype.type(0xFFFFFFFF)).astype(np.float64)
        else:
            out["row_" + name] = v.astype(np.float32 if v.dtype.kind == "f" else np.float64)
    out["cigar"] = np.asarray(cigar)[ranges(rr["cigar_off"], rr["n_cigar"])].astype(np.float64)
    return out


def dump_outputs(out_dir, read_index, row_off, rows, cigar, at=None):
    """Writes the rows of the reads read_index (from dump_sample) as .npy files in out_dir: read_index, rows_per_read, row_<field> for
    every row field in read order, and cigar (the CIGAR words of those rows in the same order).  row_off / rows / cigar are a result
    whose read at[i] (default: read_index[i]) is read read_index[i].  cigar_off is left out for the reason rows_digest gives.  Every
    array is float64 (frac_rep float32) and exact: each 64-bit integer field goes in two 32-bit halves, row_<field>_hi (signed for a
    signed field) and row_<field>_lo.  When the arrays would exceed DUMP_BYTES, the longest prefix of the reads that fits is written.
    Returns the number of bytes written."""
    at = read_index if at is None else at
    out = _dump_arrays(read_index, row_off, rows, cigar, at)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_BYTES:
        counts = out["rows_per_read"].astype(np.int64)
        words = np.bincount(np.repeat(np.arange(len(counts)), counts), weights=out["row_n_cigar"], minlength=len(counts))
        row_bytes = sum(a.itemsize for k, a in out.items() if k.startswith("row_"))
        per_read = 16 + counts * row_bytes + words * 8
        keep = max(1, int(np.searchsorted(np.cumsum(per_read), DUMP_BYTES, side="right")))
        out = _dump_arrays(read_index[:keep], row_off, rows, cigar, at[:keep])
        total = sum(a.nbytes for a in out.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return total


# ------------------------------------------------------------------------------------------ our arm
def run_ours(args, rank, world, local_rank):
    import ctypes as C
    import torch
    from bioseqdb_b200 import BwaIndex, BsqOpts, _lib
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
    dev = local_rank if world > 1 else 0
    rows, seqs, offs, ids, truth = workload(args, rank)
    ot = opts_tuple(args, len(rows))
    ix = BwaIndex(dev, BsqOpts(*ot))
    bcast_bytes = 0
    bcast_s = 0.0
    t0 = time.time()
    t_add = 0.0
    if world == 1 or rank == 0:
        ix.add_ref_sequences(list(range(1, len(rows) + 1)), rows)
        t_add = time.time() - t0
        ix.build()
    build_wall = time.time() - t0
    if world > 1:
        from bioseqdb_b200.dist import broadcast_index
        dist.barrier()
        tb = time.time()
        bcast_bytes = broadcast_index(ix, rank, dist)
        dist.barrier()
        bcast_s = time.time() - tb
    meta = ix.meta()
    prep_ms = C.c_float(0)
    _lib.check(ix.L.bsq_index_prepare(ix.h, C.byref(prep_ms)))     # per-device derived arrays (inverse SA, prefix table)
    n = args.reads

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # pinned host staging for the e2e leg
    seqs_pin = torch.from_numpy(seqs).pin_memory()
    offs_pin = torch.from_numpy(offs.view(np.int64)).pin_memory()
    ids_pin = torch.from_numpy(ids).pin_memory()

    # ---------------- value: inputs resident in HBM
    ix.upload(seqs, offs, ids)
    ix.set_counters(True)
    ix.align_resident()          # also sizes the pools (first run may re-run on overflow)
    ctr = ix.counters()
    ix.set_counters(False)
    for _ in range(max(args.warmup, 3)):
        ix.align_resident()
    stage = {"seed": 0.0, "chain": 0.0, "extend": 0.0, "finalize": 0.0}
    dev_ms = 0.0
    launches = 0
    barrier()
    with ClockSampler(dev) as clk:
        w0 = time.time()
        for _ in range(args.steps):
            ix.align_resident()
            t = ix.timing()
            dev_ms += t.total
            launches += t.launches
            for k in stage:
                stage[k] += getattr(t, k)
        barrier()
        wall = time.time() - w0
    clocks = clk.summary()
    res = ix.download_result()
    total_rows = int(res.row_off[-1])
    # sanity against the simulator's truth (parity is GPU vs oracle below and in tests/; this is a scale check): the first row of a
    # read is its best hit -- same reference row, same strand, position within the indel slack
    first = res.row_off[:-1].astype(np.int64)
    has = np.diff(res.row_off.astype(np.int64)) > 0
    pr = res.rows[np.minimum(first, max(total_rows - 1, 0))]
    okk = has & (pr["rid"] == truth[0]) & (pr["is_rev"] == truth[2].astype(np.int32)) & (np.abs(pr["pos"] - truth[1]) <= 16 + args.read_len // 8)
    truth_frac = float(okk.mean())
    digest = rows_digest(res)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dump_sample(n, args.read_len), res.row_off, res.rows, res.cigar)

    # ---------------- e2e: host buffers through the C ABI.  The reference-facing form of the call takes the reads as the PG glue holds them
    # (NUCLSEQ datum images, extension.cpp:362) and returns the 64-byte public rows; the ASCII form (bsq_align_batch) is timed beside it.
    from bioseqdb_b200.loader import nuclseq_image_block
    img, img_off, _ = nuclseq_image_block(seqs, offs, dev)
    img_pin = torch.from_numpy(img).pin_memory()
    img_off_pin = torch.from_numpy(img_off.view(np.int64)).pin_memory()
    ix.set_rows_ext(False)
    resp = C.POINTER(_lib.BsqResult)()

    def one_e2e():
        ix.session_lrand48(0)      # ids = NULL: drawn on the device from the session's lrand48 stream, the same stream every step
        _lib.check(ix.L.bsq_align_batch_datums(ix.h, C.c_void_p(img_pin.data_ptr()), C.c_void_p(img_off_pin.data_ptr()), None, n, C.byref(resp)))
        ix.L.bsq_result_free(resp)

    def one_e2e_ascii():
        _lib.check(ix.L.bsq_align_batch(ix.h, C.c_void_p(seqs_pin.data_ptr()), C.c_void_p(offs_pin.data_ptr()), C.c_void_p(ids_pin.data_ptr()), n, C.byref(resp)))
        ix.L.bsq_result_free(resp)

    def timed(fn):
        for _ in range(2):
            fn()
        barrier()
        t0_ = time.time()
        dev_ms_ = h2d_ms_ = d2h_ms_ = 0.0
        hb = db = 0
        for _ in range(args.steps):
            fn()
            t_ = ix.timing()
            dev_ms_ += t_.total; h2d_ms_ += t_.h2d; d2h_ms_ += t_.d2h
            hb, db = int(t_.h2d_bytes), int(t_.d2h_bytes)
        barrier()
        return dev_ms_, time.time() - t0_, h2d_ms_, d2h_ms_, hb, db
    e2e_dev_ms, e2e_wall, e2e_h2d_ms, e2e_d2h_ms, h2d, d2h = timed(one_e2e)
    asc_dev_ms, asc_wall, asc_h2d_ms, asc_d2h_ms, asc_h2d, asc_d2h = timed(one_e2e_ascii)
    ix.set_rows_ext(True)

    # ---------------- e2e_rows: the reference's unit of output (the 15-column tuple, extension.cpp:282-305) through bsq_align_tuples
    e2e_rows = None
    if hasattr(ix, "align_tuples_raw"):
        def one_rows():
            ix.session_lrand48(0)
            return ix.align_tuples_raw(img_pin.data_ptr(), img_off_pin.data_ptr(), None, n)
        ix.set_rows_ext(False)
        for _ in range(2):
            one_rows()
        barrier()
        r0 = time.time()
        tup_ms = 0.0
        tb = 0
        for _ in range(args.steps):
            tup_ms_i, tb = one_rows()
            tup_ms += tup_ms_i
        barrier()
        e2e_rows = {"ms": tup_ms, "wall": time.time() - r0, "d2h_bytes": tb}
        ix.set_rows_ext(True)
        ix.two_chunks = False
        ix._apply_flags()

    # ---------------- max over ranks
    def allmax(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    # every rank checks ITS copy of the index (built or received by broadcast) against the text: bsq_index_verify over EVERY row and
    # block (30 ms at c2, about a second for the 6.2 G rows of c3)
    verify = ix.verify(1 << 40)
    verify["unsound_ranks"] = int(allmax(0.0 if verify["sound"] else 1.0) > 0) if dist is not None else int(not verify["sound"])
    dev_ms_max = allmax(dev_ms)
    e2e_ms_max = allmax(e2e_dev_ms)
    asc_ms_max = allmax(asc_dev_ms)
    wall_max = allmax(wall)
    e2e_wall_max = allmax(e2e_wall)
    prep_ms_max = allmax(float(prep_ms.value))
    e2e_rows_ms_max = allmax(e2e_rows["ms"]) if e2e_rows else None
    if dist is not None:
        tot = torch.tensor([float(launches)], dtype=torch.float64, device="cuda")
        dist.all_reduce(tot)
        launches_all = int(tot.item())
    else:
        launches_all = launches

    # ---------------- results gathered on the host (SURVEY.md 8e): every rank's rows to rank 0 over a gloo side group, timed
    gather = None
    if dist is not None:
        from bioseqdb_b200.dist import gather_rows_host
        gg = dist.new_group(backend="gloo")
        dist.barrier()
        g0 = time.time()
        out = gather_rows_host(res.row_off, res.rows, res.cigar, dist, gg, rank, world)
        dist.barrier()
        gather = {"seconds": time.time() - g0, "rows_on_rank0": int(out[0][-1]) if out is not None else None,
                  "how": "gloo gather of row offsets, rows and CIGAR words to rank 0 (host memory to host memory, one process per GPU)"}

    if rank == 0:
        peaks, peak_src = measured_peaks()
        value = n * world * args.steps / (dev_ms_max * 1e-3)
        e2e_value = n * world * args.steps / max(e2e_ms_max * 1e-3, 1e-9)
        # roofline of the dominant kernel (by device time share)
        dom = max(stage, key=stage.get)
        seed_bytes = 64.0 * 2.0 * ctr["n_extend"]                 # per launch: two 64-byte Occ blocks per bwt_extend
        seed_s = stage["seed"] / args.steps * 1e-3
        roof = {"kernel": "seed_calls", "bound": "hbm", "achieved": seed_bytes / seed_s / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": seed_bytes / seed_s / 1e9 / peaks["hbm_gbs"], "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": seed_bytes, "dominant_kernel_by_time": dom,
                "stage": "seed (seed_pack + seed_calls + seed_last + seed_smem for declined reads; seed_calls is ~85 % of it)",
                "note": "algorithmic bytes = 2 Occ blocks x the reference's bwt_extend count (SURVEY 8d); the kernels resolve most of "
                        "those extends from the prefix table / by text comparison, so measured DRAM traffic is below the algorithmic figure"}
        tr = seed_traffic(args)
        if tr is not None:
            roof["traffic"] = tr["dram_bytes_per_launch"]
            roof["traffic_source"] = tr["source"]
            roof["traffic_gbs"] = tr["dram_bytes_per_launch"] / seed_s / 1e9
            roof["traffic_frac_of_hbm_peak"] = roof["traffic_gbs"] / peaks["hbm_gbs"]
        ext_s = stage["extend"] / args.steps * 1e-3
        fin_s = stage["finalize"] / args.steps * 1e-3
        sw = {"ksw_extend2_gcups": ctr["ext_cells"] / max(ext_s, 1e-12) / 1e9, "ksw_global2_gcups_incl_finalize": ctr["glb_cells"] / max(fin_s, 1e-12) / 1e9,
              "ext_cells_per_launch": ctr["ext_cells"], "glb_cells_per_launch": ctr["glb_cells"]}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
            "data": "synthetic", "config": config_dict(args),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms_max / args.steps, "wall_ms_per_step": 1e3 * e2e_wall_max / args.steps,
                    "h2d_ms_per_step": e2e_h2d_ms / args.steps, "d2h_ms_per_step": e2e_d2h_ms / args.steps,
                    "call": "bsq_align_batch_datums: reads as NUCLSEQ datum images in pinned host memory, ids drawn by the library (session lrand48 stream), 64-byte rows + CIGAR words back in pinned host memory"},
            "e2e_ascii": {"value": n * world * args.steps / max(asc_ms_max * 1e-3, 1e-9), "unit": UNIT, "h2d_bytes_per_step": asc_h2d, "d2h_bytes_per_step": asc_d2h,
                          "ms_per_step": asc_ms_max / args.steps, "call": "bsq_align_batch: ASCII reads + u64 offsets + ids"},
            "gpu_launches": launches_all,
            "clocks": clocks,
            "roofline": roof, "sw": sw,
            "stage_ms_per_step": {k: v / args.steps for k, v in stage.items()},
            "wall_ms_per_step": 1e3 * wall_max / args.steps,
            "rows_per_step_rank0": total_rows, "truth_match_frac_rank0": truth_frac, "rows_sha1_rank0": digest,
            "index": {"build_ms_device": meta.build_ms, "build_wall_s": build_wall, "add_ref_wall_s": t_add, "build_launches": int(meta.build_launches),
                      "sort_pass_gbs": (meta.sort_pass_bytes / (meta.build_ms * 1e-3) / 1e9) if meta.build_ms else None,
                      "seq_len": int(meta.seq_len), "broadcast_bytes": bcast_bytes, "broadcast_s": bcast_s,
                      "derived_arrays_ms_max_over_ranks": prep_ms_max, "device_bytes": ix.device_bytes(),
                      "verify": verify},
            "counters_per_launch": ctr,
            "parity_pinning": "unpinned (oracle restates lh3/bwa; no libbwa binary or reference vector to pin it)",
        }
        if e2e_rows:
            line["e2e_rows"] = {"value": n * world * args.steps / max(e2e_rows_ms_max * 1e-3, 1e-9), "unit": UNIT, "ms_per_step": e2e_rows_ms_max / args.steps,
                                "d2h_bytes_per_step": e2e_rows["d2h_bytes"], "frac_of_e2e": (e2e_ms_max / max(e2e_rows_ms_max, 1e-9)),
                                "wall_ms_per_step": 1e3 * e2e_rows["wall"] / args.steps,
                                "what": "bsq_align_batch_datums + bsq_result_tuples (served from the resident batch) with host buffers: rows + NUCLSEQ datum images of ref_subseq / query_subseq + CIGAR strings (the bwa_result tuple of extension.cpp:282-305) on the host"}
        if gather:
            line["gather"] = gather
        if not args.no_extras:
            gather_gbs = C.c_double(0)
            _lib.check(ix.L.bsq_bench_gather(ix.h, 1 << 28, 3, C.byref(gather_gbs)))
            dpx = C.c_double(0)
            _lib.check(ix.L.bsq_bench_dpx(dev, 3, C.byref(dpx)))
            roof["random_gather_peak_gbs"] = gather_gbs.value
            roof["frac_of_random_gather"] = seed_bytes / seed_s / 1e9 / max(gather_gbs.value, 1e-9)
            if roof.get("traffic_gbs"):
                roof["traffic_frac_of_random_gather"] = roof["traffic_gbs"] / max(gather_gbs.value, 1e-9)
            sw["dpx_peak_ginstr_s"] = dpx.value
            # SURVEY 8d: DPX fraction = DPX instructions per cell of the shipped kernel x cells/s over the whole extension stage, against
            # the measured DPX issue peak
            sw["ksw_extend2_dpx_per_cell"] = 3
            sw["ksw_extend2_dpx_frac_of_peak"] = 3 * ctr["ext_cells"] / max(ext_s, 1e-12) / 1e9 / dpx.value
            # row materialisation from a host result (SURVEY 8f-2, the re-upload path) and the bulk loader (8f-4)
            t0 = time.time()
            tup = ix.tuples(res, seqs, offs)
            tup_wall = time.time() - t0
            from bioseqdb_b200.loader import nuclseq_images
            ld_texts, ld_bases = [], 0
            for r_ in rows:
                if ld_bases + len(r_) > 400_000_000:
                    break
                ld_texts.append(r_.tobytes()); ld_bases += len(r_)
            _, ld_ms = nuclseq_images(ld_texts, local_rank) if ld_texts else ([], 0.0)
            line["loader"] = {"sequences": len(ld_texts), "bases": ld_bases, "device_ms_incl_copies": ld_ms,
                              "gbases_per_s_device": ld_bases / max(ld_ms * 1e-3, 1e-9) / 1e9}
            line["tuples"] = {"rows": total_rows, "bytes": int(len(tup.data)), "device_ms_incl_copies": tup.device_ms, "wall_ms_python": 1e3 * tup_wall,
                              "rows_per_s_device": total_rows / max(tup.device_ms * 1e-3, 1e-9)}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"], line["parity"] = cpu_baseline(args, rows, seqs, offs, ids, ix, ot, res)
            if line["parity"]["mismatching_reads"]:
                line["PARITY_FAILED"] = "%d of %d reads differ from the oracle" % (line["parity"]["mismatching_reads"], line["parity"]["reads_checked"])
                print("PARITY FAILED: %s" % line["PARITY_FAILED"], file=sys.stderr, flush=True)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def cpu_baseline(args, rows, seqs, offs, ids, ix, ot, gres):
    """The oracle port on this box's host cores, bounded sample; the index arrays are adopted from the GPU build (they are
    mathematically unique) so that the sample budget goes to alignment.  The oracle's rows for the sample are then compared with
    the GPU's rows for the same reads: all PARITY_FIELDS and every CIGAR word (tests/helpers.py parity_report)."""
    import oracle_lib as O
    from helpers import parity_report
    cores = os.cpu_count() or 1
    orc = O.OracleIndex(O.Opts(*ot))
    for i, r in enumerate(rows):
        orc.add_ref_text(i + 1, r.tobytes())
    orc.adopt(ix.bwt_plain(), int(ix.meta().primary), ix.sa_sampled())
    sample, probe, rate = sized_sample(orc, args, seqs, offs, ids, cores)
    r = orc.align_batch(seqs[:int(offs[sample])], offs[:sample + 1], ids[:sample], cores)
    parity = parity_report(gres, r, sample)
    parity["against"] = "CPU oracle port (parity unpinned: no libbwa binary or reference vector exists to pin the oracle)"
    probe1 = max(8, min(probe, int(rate / cores * 3.0)))   # ~3 s of single-core work
    r1 = orc.align_batch(seqs[:int(offs[probe1])], offs[:probe1 + 1], ids[:probe1], 1)
    # index build on a bounded 8 Mbp sample, 1 core
    small = O.OracleIndex(O.Opts(*ot))
    head = rows[0][:8_000_000] if len(rows[0]) >= 8_000_000 else np.concatenate(rows[:16000])[:8_000_000]
    small.add_ref_text(1, head.tobytes())
    bs = small.build()
    base = {"value": sample / r["seconds"], "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d of %d reads, %d threads, FM-index arrays adopted from the GPU build" % (sample, args.reads, cores),
            "one_core_reads_per_s": probe1 / r1["seconds"], "index_build_s_8Mbp_1core": bs,
            "oracle_counters_per_read": {k: v / sample for k, v in r["counters"].items()}}
    return base, parity


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
