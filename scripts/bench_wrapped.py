"""Linear vs wrapped FASTA input, end to end: utb_search_mem from a page-locked buffer.  Two workloads from bench.py:
L2S (10 M x 150 bp, RC), linear against wrapped at 60 columns; LONG (10 kb - 16 Mb queries, RC), linear against
wrapped at 80 (and, with --crlf, at 60 with CRLF line ends).  Legs alternate, three timed runs each after a warm-up;
then one profiled run per leg gives the time of the framing and join kernels.  Wrapped and linear outputs must have
equal sha256.  One JSON line per leg on stdout.

    python scripts/bench_wrapped.py [--workloads l2s,long] [--runs 3] [--crlf] [--trace-dir DIR]
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

HDR = 12                                                           # bench.py records: 12-byte header line, sequence, '\n'
FRAME_KERNELS = ("nl_count_kernel", "frame_setup_kernel", "nl_index_kernel", "frame_parse_kernel")
WRAP_KERNELS = ("wrap_tile_kernel", "wrap_keep_kernel", "wrap_join_kernel", "wrap_record_kernel", "frame_setup_kernel",
                "scan_sums_kernel", "scan_top_kernel", "scan_apply_kernel")


def rewrap(fa, off, width, crlf):
    """bench.py's linear records (fa, record offsets) -> a page-locked wrapped FASTA: the sequence cut into lines of
    `width` bases, each ended by '\\n' (or '\\r\\n')."""
    import torch
    eol = np.frombuffer(b"\r\n" if crlf else b"\n", dtype=np.uint8)
    lens = np.diff(off).astype(np.int64) - HDR - 1
    lines = (lens + width - 1) // width
    out_off = np.zeros(lens.size + 1, dtype=np.int64)
    out_off[1:] = np.cumsum(HDR + lens + lines * eol.size)
    out = torch.empty(int(out_off[-1]), dtype=torch.uint8, pin_memory=True).numpy()
    if np.all(lens == lens[0]):                                    # fixed length: all records at once
        n, L, k = lens.size, int(lens[0]), int(lines[0])
        rows, dst = fa.reshape(n, -1), out.reshape(n, -1)
        dst[:, :HDR] = rows[:, :HDR]
        for j in range(k):
            a, b = j * width, min(L, (j + 1) * width)
            o = HDR + a + j * eol.size
            dst[:, o:o + b - a] = rows[:, HDR + a:HDR + b]
            dst[:, o + b - a:o + b - a + eol.size] = eol
        return out
    for i in range(lens.size):                                     # one record at a time (long queries)
        s, d, L, k = int(off[i]), int(out_off[i]), int(lens[i]), int(lines[i])
        out[d:d + HDR] = fa[s:s + HDR]
        seq = fa[s + HDR:s + HDR + L]
        full = L // width
        body = out[d + HDR:int(out_off[i + 1])]
        if full:
            blk = body[:full * (width + eol.size)].reshape(full, width + eol.size)
            blk[:, :width] = seq[:full * width].reshape(full, width)
            blk[:, width:] = eol
        if L > full * width:
            rest = L - full * width
            body[full * (width + eol.size):full * (width + eol.size) + rest] = seq[full * width:]
            body[-eol.size:] = eol
    return out


def kernel_ms(searcher, buf, trace_dir, tag):
    """Device time per kernel name over one search, from torch.profiler (CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rc, ex, n, st = searcher.search_mem(None, do_rc=True, ptr=buf.ctypes.data, n=buf.size, copy=False)
        torch.cuda.synchronize()
    assert rc == 0, rc
    if trace_dir:
        prof.export_chrome_trace(os.path.join(trace_dir, f"wrapped_{tag}.pt.trace.json"))
    out = {}
    for e in prof.key_averages():
        name = e.key.split("(")[0].split("<")[0].replace("void ", "").strip()
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        out[name] = out.get(name, 0.0) + t / 1e3
    return out, st["batches"]


def run_workload(wl, args, gpu):
    from utree_b200 import capi
    cfg = bench.CONFIGS[wl]
    n = cfg["reads"]
    ctr_path, meta = bench.ensure_ctr(wl, cfg, 0)
    fa, off = bench.make_reads(cfg, 0, n, 0, pin=True)
    bases = int(off[-1]) - n * (HDR + 1)
    widths = [(60, False)] if wl == "l2s" else [(80, False)] + ([(60, True)] if args.crlf else [])
    legs = [("linear", fa, False)]
    for w, crlf in widths:
        t = time.time()
        legs.append((f"wrapped{w}{'_crlf' if crlf else ''}", rewrap(fa, off, w, crlf), True))
        bench.log(f"{wl}: {legs[-1][0]} {legs[-1][1].size / 1e9:.2f} GB from {fa.size / 1e9:.2f} GB (built in {time.time() - t:.1f} s)")
    ctr = capi.Ctr(ctr_path)
    s = capi.Searcher(ctr, devices=(0,), host_threads=max(2, len(bench.ALL_CPUS)))

    def run(leg, copy=False):
        name, buf, wrapped = leg
        s.set_input(False, 0, wrapped=wrapped)
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
    for leg in legs[1:]:
        assert digest[leg[0]] == digest["linear"], f"{wl}: {leg[0]} output differs from the linear output"
    times = {leg[0]: [] for leg in legs}
    stats = {}
    for _ in range(args.runs):
        for leg in legs:
            dt, _, st = run(leg)
            times[leg[0]].append(dt)
            stats[leg[0]] = st
    for name, buf, wrapped in legs:
        s.set_input(False, 0, wrapped=wrapped)
        k, batches = kernel_ms(s, buf, args.trace_dir, f"{wl}_{name}")
        ts = times[name]
        mean = sum(ts) / len(ts)
        names = WRAP_KERNELS if wrapped else FRAME_KERNELS
        # the wrapped path's scans are the framing's; the grp_off scan that both paths run is counted in neither
        frame = sum(v for kname, v in k.items() if kname in names and not kname.startswith("scan_"))
        scans = sum(v for kname, v in k.items() if kname.startswith("scan_"))
        line = {
            "metric": f"utb_search_mem from a page-locked buffer, {wl.upper()} ({cfg['desc']}), RC", "workload": wl, "format": name,
            "reads": n, "bases": bases, "input_bytes": int(buf.size),
            "reads_per_s": round(n / mean, 1), "g_bases_per_s": round(bases / mean / 1e9, 2),
            "input_gb_per_s": round(buf.size / mean / 1e9, 2),
            "ms_per_search": [round(1e3 * x, 2) for x in ts],
            "batches": batches,
            "frame_kernels_ms": round(frame, 3), "frame_kernels_ms_per_batch": round(frame / max(1, batches), 3),
            "scan_kernels_ms_per_batch": round(scans / max(1, batches), 3),
            "kernels_ms": {kname: round(v, 3) for kname, v in sorted(k.items())
                           if kname in FRAME_KERNELS + WRAP_KERNELS + ("pack_kernel",)},
            "output_sha256": digest[name], "out_bytes": stats[name]["out_bytes"],
            "gpu": gpu,
        }
        print(json.dumps(line), flush=True)
    s.destroy(); ctr.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="l2s,long")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--crlf", action="store_true", help="LONG also wrapped at 60 with CRLF line ends")
    ap.add_argument("--trace-dir", default="")
    args = ap.parse_args()
    from utree_b200 import build
    build.build()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    for wl in args.workloads.split(","):
        run_workload(wl, args, gpu)


if __name__ == "__main__":
    main()
