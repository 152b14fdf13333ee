"""FASTA vs FASTQ input, end to end: utb_search_mem from a page-locked buffer on the L2S workload (bench.py's tree and
reads; the FASTQ is the same reads with seeded qualities of an Illumina-like profile, '+' separators).  Formats alternate, three timed runs each
after a warm-up; then one profiled run per format gives the time of the framing and mask kernels.  One JSON line per
format on stdout.

    python scripts/bench_fastq.py [--reads N] [--runs 3] [--min-qual 20] [--trace-dir DIR]
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (ensure_ctr, make_reads, CONFIGS)

FRAME_KERNELS = ("nl_count_kernel", "frame_setup_kernel", "nl_index_kernel", "frame_parse_kernel", "frame_parse_fastq_kernel")
MASK_KERNELS = ("qual_mask_kernel",)


def to_fastq(fa, n, read_len, seed):
    """Fixed-length bench.py records (header line, sequence line) -> pinned FASTQ with seeded qualities: Phred 38 at
    the start of a read, falling by 1 every 20 bases, +-3 of noise, and 1 % of the bases at Phred 2 (short-read
    instruments give mostly high qualities that fall along the read, with scattered low-quality calls)."""
    import torch
    rec = fa.size // n
    rows = fa.reshape(n, rec)
    fq = torch.empty(n * (rec + 2 + read_len + 1), dtype=torch.uint8, pin_memory=True).numpy().reshape(n, -1)
    fq[:, :rec] = rows
    fq[:, 0] = ord("@")
    fq[:, rec] = ord("+")
    fq[:, rec + 1] = ord("\n")
    rng = np.random.default_rng(seed)
    step = 1 << 20
    trend = (38 - np.arange(read_len) // 20).astype(np.int16)
    for a in range(0, n, step):
        k = min(step, n - a)
        q = trend + rng.integers(-3, 4, (k, read_len), dtype=np.int16)
        q[rng.integers(0, 100, (k, read_len), dtype=np.uint8) == 0] = 2
        fq[a:a + k, rec + 2:rec + 2 + read_len] = (np.clip(q, 0, 41) + 33).astype(np.uint8)
    fq[:, -1] = ord("\n")
    return fq.reshape(-1)


def kernel_ms(searcher, buf, trace_dir, tag):
    """Device time per kernel name over one search, from torch.profiler (CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rc, ex, n, st = searcher.search_mem(None, do_rc=True, ptr=buf.ctypes.data, n=buf.size, copy=False)
        torch.cuda.synchronize()
    assert rc == 0, rc
    if trace_dir:
        prof.export_chrome_trace(os.path.join(trace_dir, f"fastq_{tag}.pt.trace.json"))
    out = {}
    for e in prof.key_averages():
        name = e.key.split("(")[0].split("<")[0].replace("void ", "").strip()
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        out[name] = out.get(name, 0.0) + t / 1e3
    return out, st["batches"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=0, help="reads (default: the L2S config's 10 M)")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--min-qual", type=int, default=20, help="masking threshold of the fastq_mask leg")
    ap.add_argument("--trace-dir", default="")
    args = ap.parse_args()
    import torch
    from utree_b200 import build, capi
    build.build()
    cfg = bench.CONFIGS["l2s"]
    n = args.reads or cfg["reads"]
    ctr_path, meta = bench.ensure_ctr("l2s", cfg, 0)
    fa, off = bench.make_reads(cfg, 0, n, 0, pin=True)
    t = time.time()
    fq = to_fastq(fa, n, cfg["read_len"], bench.SEED + 7)
    bench.log(f"{n} reads: FASTA {fa.size / 1e9:.2f} GB, FASTQ {fq.size / 1e9:.2f} GB (built in {time.time() - t:.1f} s)")
    ctr = capi.Ctr(ctr_path)
    s = capi.Searcher(ctr, devices=(0,), host_threads=max(2, len(bench.ALL_CPUS)))
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    legs = [("fasta", fa, False, 0), ("fastq", fq, True, 0), ("fastq_mask", fq, True, args.min_qual)]
    qual = fq.reshape(n, -1)[:, -1 - cfg["read_len"]:-1]
    masked = float(np.count_nonzero(qual < 33 + args.min_qual)) / qual.size

    def run(leg, copy=False):
        name, buf, fastq, q = leg
        s.set_input(fastq, q)
        t0 = time.perf_counter()
        rc, ex, text, st = s.search_mem(None, do_rc=True, ptr=buf.ctypes.data, n=buf.size, copy=copy)
        dt = time.perf_counter() - t0                              # utb_search_mem returns after its last device copy
        assert (rc, ex) == (0, 0), (name, rc, capi.lib().utb_last_error())
        return dt, text, st

    digest = {}
    for leg in legs:                                               # warm-up (page-locks the output arena), and the outputs
        dt, text, st = run(leg, copy=True)
        digest[leg[0]] = hashlib.sha256(text).hexdigest()
        del text
    assert digest["fasta"] == digest["fastq"], "FASTQ output differs from the FASTA output"
    times = {leg[0]: [] for leg in legs}
    stats = {}
    for _ in range(args.runs):
        for leg in legs:
            dt, _, st = run(leg)
            times[leg[0]].append(dt)
            stats[leg[0]] = st
    kern = {}
    for leg in legs:
        s.set_input(leg[2], leg[3])
        kern[leg[0]] = kernel_ms(s, leg[1], args.trace_dir, leg[0])
    for name, buf, fastq, q in legs:
        ts = times[name]
        mean = sum(ts) / len(ts)
        k, batches = kern[name]
        frame = sum(v for kname, v in k.items() if kname in FRAME_KERNELS)
        mask = sum(v for kname, v in k.items() if kname in MASK_KERNELS)
        line = {
            "metric": "utb_search_mem from a page-locked buffer, L2S (10 M x 150 bp), RC", "format": name,
            "min_qual": q, "reads": n, "input_bytes": int(buf.size),
            "reads_per_s": round(n / mean, 1), "input_gb_per_s": round(buf.size / mean / 1e9, 2),
            "ms_per_search": [round(1e3 * x, 2) for x in ts],
            "batches": batches,
            "frame_kernels_ms": round(frame, 3), "frame_kernels_ms_per_batch": round(frame / max(1, batches), 3),
            "mask_kernel_ms": round(mask, 3), "mask_kernel_ms_per_batch": round(mask / max(1, batches), 3),
            "kernels_ms": {kname: round(v, 3) for kname, v in sorted(k.items())
                           if kname in FRAME_KERNELS + MASK_KERNELS + ("pack_kernel",)},
            "masked_base_fraction": round(masked, 4) if q else 0.0,
            "output_sha256": digest[name], "out_bytes": stats[name]["out_bytes"],
            "gpu": gpu,
        }
        print(json.dumps(line), flush=True)
    s.destroy(); ctr.close()


if __name__ == "__main__":
    main()
