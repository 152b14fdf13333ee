#!/usr/bin/env python
"""bench.py -- reads/s and k-mer lookups/s of the SEARCH_GG hot path on B200.

Default workload (BASELINE.json configs[1], "l2s"): a synthetic L2-scale CTR (5,000
prokaryote-sized genomes, complevel 2, ~1.1 G records, ~8 GB) against 10 M synthetic
150 bp reads per GPU with reverse complement.  A "step" is one pass of the hot path over
the whole read set.  `--config toy | l4 | long | u32` runs the other BASELINE configs the same
way (their lines are committed under profiles/).

  value     reads/s with the FASTA bytes already resident in HBM: device time of
            pack -> sieve -> table lookup -> vote from CUDA events on the launching
            stream (utb_batch_rerun_device), summed over the chunks of the read set
  e2e       reads/s through the C ABI with HOST buffers (utb_search_mem: H2D of the
            raw FASTA from a page-locked buffer, framing + search + output formatting
            on the device, D2H of the text straight into the searcher's page-locked
            output arena), wall clock; the arena is allocated by the warm-up steps
  e2e_file  utb_search_file (FASTA file -> output file, both on /dev/shm) on the
            resident searcher, wall clock of the call
  e2e_cli   the drop-in CLI (bin/utree-search_gg, files on /dev/shm), wall minus a
            1-read run of the same command -- the recipe the reference arm uses
  e2e_pageable  utb_search_mem from an ordinary (pageable) buffer
  roofline  the LONGEST kernel of the resident step (every stage kernel is listed in
            roofline.kernels): algorithmic bytes per launch / its CUDA-event time,
            against MEASURED_PEAKS.json hbm_gbs (streaming kernels) or the live random
            32-byte-sector gather rate (utb_measure_rand32, gather kernels); traffic =
            ncu dram bytes of that kernel at this shape (profiles/traffic.json)
  cpu_baseline / --impl reference: the UNMODIFIED reference binary
            (oracle/_ref/utree-search_gg) on the host cores, same CTR + reads
  parity    asserted inside this run: e2e text == host-formatted records of the
            resident pass == CLI output file, and its head == the CPU checker's output

`--dump-outputs DIR` writes, after the timed steps, the output text of the last timed e2e
step (rank 0's reads) for a fixed, seeded sample of reads, so that two builds can be compared
output for output on identical inputs (see dump_outputs).

Multi-GPU (torchrun, one rank per GPU): reads sharded, CTR replicated, no collective on the
data path; weak scaling.  `single_process` additionally times ONE utb_searcher over all
N devices on one FASTA of N x the reads (one upload + NVLink fan-out of the tables, one
dispatcher thread, ordered merge of the per-GPU output).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import re
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from oracle import oracle_api  # noqa: E402  (CPU checker: used only by the cpu_baseline / reference / parity legs)

CONFIGS = {
    # universe = (phyla, genera, species, strains, genome_len); one strain per species, like a RefSeq-representative
    # set: little k-mer sharing, so 20 Gb of genome sampled 1/16 (complevel 2) keeps ~1.1 G records (~8 GB), README.md:2
    "l2s": dict(universe=(50, 20, 5, 1, 4_000_000), complevel=2, ix_bytes=2, reads=10_000_000, read_len=150,
                desc="L2-scale synthetic CTR (5000 genomes x 4 Mb, complevel 2) vs 10M x 150bp reads, RC"),
    "l4": dict(universe=(50, 20, 5, 1, 4_000_000), complevel=4, ix_bytes=2, reads=50_000_000, read_len=150,
               desc="L4 synthetic CTR (5000 genomes x 4 Mb, complevel 4, ~0.5 GB) vs 50M x 150bp reads, RC"),
    # 10 kb - 1 Mb log-uniform reads + whole-genome queries of 5 - 16 Mb against the L2-scale CTR.  Default: a 1/12.5
    # sample of the named 200k-read set (3.6 GB of FASTA per step, one resident batch); --reads 200000 is the full set
    "long": dict(universe=(50, 20, 5, 1, 4_000_000), complevel=2, ix_bytes=2, reads=16_000, read_len=None, genomes_per_1k=1,
                 desc="long-read workload: 16k synthetic 10 kb-1 Mb reads (log-uniform) + 16 whole-genome 5-16 Mb queries "
                      "vs the L2-scale CTR, RC (a 1/12.5 sample of the named 200k reads per step)"),
    # IXTYPE=uint32_t (SZ=9), > 65,536 labels, complevel 0 (dense sampling), 250 bp reads (BASELINE.json configs[4])
    "u32": dict(universe=(60, 11, 10, 10, 6000), complevel=0, ix_bytes=4, reads=10_000_000, read_len=250,
                desc="uint32-label synthetic CTR (66000 genomes x 6 kb, 73500 labels, complevel 0) vs 10M x 250bp reads, RC"),
    # BASELINE.json configs[0]: the reference's own CPU-runnable case
    "toy": dict(universe=(2, 2, 5, 1, 1_000_000), complevel=2, ix_bytes=2, reads=100_000, read_len=150,
                desc="toy CTR (20 synthetic genomes x 1 Mb, complevel 2) vs 100k x 150bp reads, RC"),
    "small": dict(universe=(4, 3, 3, 3, 400_000), complevel=2, ix_bytes=2, reads=400_000, read_len=150,
                  desc="small synthetic CTR (108 genomes x 0.4 Mb, complevel 2) vs 400k x 150bp reads, RC"),
}
SEED = 20260101
ALL_CPUS = os.sched_getaffinity(0)
CHUNK_BYTES = 1_900_000_000          # raw bytes of one resident batch (positions x 2 strands must fit 32 bits)
DUMP_READS = 1 << 15                 # reads whose output lines --dump-outputs writes (< 64 MB at any label length in CONFIGS)


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def work_dir():
    d = os.environ.get("UTB_BENCH_DIR")
    if not d:
        d = "/dev/shm/utb_bench" if os.path.isdir("/dev/shm") else "/tmp/utb_bench"
    os.makedirs(d, exist_ok=True)
    return d


def cfg_key(name, cfg):
    return hashlib.sha1(json.dumps([cfg["universe"], cfg["complevel"], cfg["ix_bytes"], SEED]).encode()).hexdigest()[:10]


def ensure_ctr(name, cfg, device):
    """Synthesises the CTR once per box (cached so both arms, and the configs that share a tree, see the same file)."""
    from utree_b200 import build
    from tools import synthgpu
    build.build_synth()
    path = os.path.join(work_dir(), f"ctr_{cfg_key(name, cfg)}.ctr")
    meta = path + ".json"
    if os.path.exists(path) and os.path.exists(meta):
        return path, json.load(open(meta))
    uni = synthgpu.Universe(SEED, *cfg["universe"])
    t = time.time()
    tmp = path + f".tmp{os.getpid()}"
    n, nl = uni.build_ctr(tmp, complevel=cfg["complevel"], ix_bytes=cfg["ix_bytes"], device=device)
    os.replace(tmp, path)
    m = {"records": n, "labels": nl, "bytes": os.path.getsize(path), "synth_s": round(time.time() - t, 1)}
    json.dump(m, open(meta, "w"))
    log(f"synthesised {path}: {n} records, {nl} labels, {m['bytes'] / 1e9:.2f} GB in {m['synth_s']} s")
    return path, m


def read_lengths(cfg, first, n_reads):
    """Lengths of reads [first, first + n_reads) of a variable-length config (seeded per read index)."""
    idx = np.arange(first, first + n_reads, dtype=np.uint64)
    h = (idx * np.uint64(0x9E3779B97F4A7C15) + np.uint64(SEED)) & np.uint64(0xFFFFFFFFFFFFFFFF)
    h ^= h >> np.uint64(29); h *= np.uint64(0xBF58476D1CE4E5B9); h ^= h >> np.uint64(32)
    u = (h >> np.uint64(11)).astype(np.float64) / float(1 << 53)
    lens = np.floor(10.0 ** (4.0 + 2.0 * u)).astype(np.uint32)                       # log-uniform 10 kb .. 1 Mb
    every = 1000 // max(1, cfg.get("genomes_per_1k", 1))
    whole = (idx % np.uint64(every)) == np.uint64(every - 1)                          # whole-genome queries, 5 .. 16 Mb
    lens[whole] = np.minimum(16_777_214, np.floor(5e6 + 11e6 * u[whole])).astype(np.uint32)
    return lens


def make_reads(cfg, first, n_reads, device, pin=False):
    """(uint8 FASTA array, record byte offsets [n + 1]) of reads [first, first + n_reads)."""
    import torch
    from tools import synthgpu
    uni = synthgpu.Universe(SEED, *cfg["universe"])
    if cfg["read_len"]:
        rec = 12 + cfg["read_len"] + 1
        off = np.arange(n_reads + 1, dtype=np.uint64) * np.uint64(rec)
        lens = None
    else:
        lens = read_lengths(cfg, first, n_reads)
        off = np.zeros(n_reads + 1, dtype=np.uint64)
        off[1:] = np.cumsum(lens.astype(np.uint64) + 13)
    nb = int(off[-1])
    buf = torch.empty(nb, dtype=torch.uint8, pin_memory=pin).numpy()
    if lens is None:
        uni.make_reads(n_reads, read_len=cfg["read_len"], read_seed=SEED + 1, first=first, device=device, out=buf)
    else:
        uni.make_long_reads(lens, read_seed=SEED + 1, first=first, device=device, out=buf)
    return buf, off


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu_index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        self.stop_flag = True
        sm = sorted(int(r[1]) for r in self.rows if r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if r[2].isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ---------------------------------------------------------------------------
# reference arm helpers (CPU): the unmodified reference binary
# ---------------------------------------------------------------------------
def ref_binary(cfg):
    exe = os.path.join(ROOT, "oracle", "_ref", "utree-search_gg" + ("_u32" if cfg["ix_bytes"] == 4 else ""))
    return exe if os.path.exists(exe) else None


def run_reference(exe, ctr, fasta, threads):
    out = os.path.join(work_dir(), f"ref_{os.getpid()}.out")
    t = time.time()
    p = subprocess.run([exe, ctr, fasta, out, str(threads), "RC"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    dt = time.time() - t
    if p.returncode:
        raise RuntimeError(f"reference exited {p.returncode}: {p.stderr[-300:]}")
    return dt, out


def cpu_reference_rate(cfg, ctr_path, reads, off, budget_s, threads, state=None):
    """reads/s of the reference binary = sample / (wall - wall of a 1-read run) (BASELINE.md 3).  The sample is a
    prefix of the same reads sized for ~budget_s of search time."""
    exe = ref_binary(cfg)
    wd = work_dir()
    n_avail = off.size - 1
    if state is None:
        state = {}
    if "t_load" not in state:
        one = os.path.join(wd, f"one_{os.getpid()}.fa")
        reads[:int(off[1])].tofile(one)
        state["t_load"] = min(run_reference(exe, ctr_path, one, threads)[0] for _ in range(2))
        # calibrate on a prefix of ~3 Mb of sequence
        n_cal = max(1, min(n_avail, int(np.searchsorted(off, 3_300_000))))
        cal = os.path.join(wd, f"cal_{os.getpid()}.fa")
        reads[:int(off[n_cal])].tofile(cal)
        dt, _ = run_reference(exe, ctr_path, cal, threads)
        rate_bytes = float(off[n_cal]) / max(dt - state["t_load"], 1e-3)
        state["sample"] = max(n_cal, min(n_avail, int(np.searchsorted(off, rate_bytes * budget_s))))
        os.remove(cal)
    n = state["sample"]
    fa = os.path.join(wd, f"sample_{os.getpid()}.fa")
    if state.get("fa_n") != n:
        reads[:int(off[n])].tofile(fa)
        state["fa_n"] = n
    dt, out = run_reference(exe, ctr_path, fa, threads)
    search = max(dt - state["t_load"], 1e-6)
    state["last_out"] = out
    return n / search, n, search, state


def oracle_sample(ctr_path, reads, off, n_sample, threads):
    """The CPU checker on a prefix of the reads: its output text (parity of this very run) and SURVEY 8d's
    algorithmic bytes per lookup (sectors the reference's own probe sequence touches)."""
    fa = os.path.join(work_dir(), f"sect_{os.getpid()}.fa")
    reads[:int(off[n_sample])].tofile(fa)
    orc = oracle_api.OracleDb(ctr_path)
    t = time.time()
    rc, st, err = orc.search_file(fa, fa + ".out", do_rc=True, threads=threads)
    dt = time.time() - t
    orc.free()
    assert rc == 0, err
    text = open(fa + ".out", "rb").read()
    os.remove(fa); os.remove(fa + ".out")
    bpl = 32.0 * (st["sect_idx"] + st["sect_bkt"]) / max(st["lookups"], 1)
    return {"bytes_per_lookup": bpl, "lookups_per_read": st["lookups"] / n_sample, "sample_reads": n_sample,
            "port_reads_per_s": n_sample / dt, "text": text}


_REAL_STDOUT = None


def emit_json(line):
    """The ONE JSON line goes to the process's original stdout; everything else (NCCL banners, library
    chatter) was redirected to stderr at start-up."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def chunks_of(off, limit=CHUNK_BYTES, max_reads=10_000_000):
    """Consecutive record ranges [a, b) of at most `limit` raw bytes / max_reads records (one resident batch each)."""
    out, a, n = [], 0, off.size - 1
    while a < n:
        b = int(np.searchsorted(off, off[a] + np.uint64(limit), side="right")) - 1
        b = max(a + 1, min(b, a + max_reads, n))
        out.append((a, b))
        a = b
    return out


def bind_near_gpu(index):
    """N > 1: run this rank (and so page-lock its host buffers) on the cores of the NUMA node its GPU hangs off, the way
    one would start it under numactl.  Returns what it did, for the JSON line; any failure leaves the affinity alone."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(index)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        base = f"/sys/bus/pci/devices/{bdf}/"
        node = int(open(base + "numa_node").read())
        cpus = set()
        for part in open(base + "local_cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if node < 0 or not cpus:
            return {"numa_node": node, "bound": False}
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "bound": True, "cpus": len(cpus)}
    except Exception as e:                                           # noqa: BLE001
        return {"bound": False, "why": str(e)[:80]}


def mem_interleave(on):
    """Page placement of what this process allocates next: spread over all NUMA nodes (a buffer every GPU reads) or the
    default again.  Best effort."""
    try:
        import ctypes, platform
        nr = {"x86_64": 238, "aarch64": 237}.get(platform.machine())
        if nr is None:
            return False
        mask = 0
        if on:
            for part in open("/sys/devices/system/node/online").read().strip().split(","):
                a, _, b = part.partition("-")
                for n in range(int(a), int(b or a) + 1):
                    mask |= 1 << n
            if mask & (mask - 1) == 0:
                return False
        m = ctypes.c_ulong(mask)
        return ctypes.CDLL(None, use_errno=True).syscall(nr, 3 if on else 0, ctypes.byref(m) if on else None, 65 if on else 0) == 0
    except Exception:                                                # noqa: BLE001
        return False


def cli_run(exe, ctr_path, fasta, out, threads):
    t = time.time()
    p = subprocess.run([exe, ctr_path, fasta, out, str(threads), "RC"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                       env=dict(os.environ, UTB_STATS="1"))
    dt = time.time() - t
    if p.returncode:
        raise RuntimeError(f"{exe} exited {p.returncode}: {p.stderr[-300:]}")
    log(f"cli {os.path.basename(fasta)}: wall {dt:.2f} s | " + " | ".join(p.stderr.strip().splitlines()[-2:]))
    m = re.search(r"([0-9.]+) s total", p.stderr)                   # UTB_STATS: the search itself (utb_search_file), without tree load / table build
    return dt, (float(m.group(1)) if m else None)


def search_mem_unread(capi, searcher, ptr, n):
    """Searcher.search_mem(copy=False) that also returns where the text is: it stays in the searcher's arena until the
    next search, so it can be copied once the clock has stopped.  -> (rc, text address, text length, stats)."""
    import ctypes as C
    st, ex = capi.Stats(), C.c_int()
    out, out_len = C.c_void_p(), C.c_size_t()
    rc = capi.lib().utb_search_mem(searcher.h, ptr, n, 1, C.byref(out), C.byref(out_len), C.byref(st), C.byref(ex))
    return rc, out.value, out_len.value, st.as_dict()


def dump_outputs(d, text, first_read, n_reads):
    """The output lines of DUMP_READS reads drawn with a fixed seed from reads [first_read, first_read + n_reads) (all
    of them when there are fewer), as d/read_index.npy (float64, the sampled read numbers, ascending),
    d/line_offsets.npy (float64, n + 1: read i's line is line_bytes[off[i]:off[i + 1]] without its newline, empty when
    the read has no line) and d/line_bytes.npy (float32, the bytes of those lines).  Reads are named r%09u after their
    number and their lines come in input order."""
    t = np.frombuffer(text, dtype=np.uint8)
    ends = np.flatnonzero(t == 10)
    starts = np.concatenate([[0], ends + 1])[:ends.size].astype(np.int64)
    num = np.zeros(starts.size, dtype=np.int64)
    for k in range(1, 10):
        num = num * 10 + t[starts + k].astype(np.int64) - 48
    rng = np.random.default_rng(SEED)
    reads = first_read + np.sort(rng.choice(n_reads, min(n_reads, DUMP_READS), replace=False)).astype(np.int64)
    pos = np.minimum(np.searchsorted(num, reads), max(num.size - 1, 0))
    has = num[pos] == reads if num.size else np.zeros(reads.size, dtype=bool)
    lens = np.zeros(reads.size, dtype=np.int64)
    lens[has] = ends[pos[has]] - starts[pos[has]]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    line_bytes = t[np.repeat(starts[pos[has]] - off[:-1][has], lens[has]) + np.arange(off[-1])].astype(np.float32)
    assert line_bytes.nbytes + 16 * (reads.size + 1) <= 64 << 20, "dump over 64 MB"
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "read_index.npy"), reads.astype(np.float64))
    np.save(os.path.join(d, "line_offsets.npy"), off.astype(np.float64))
    np.save(os.path.join(d, "line_bytes.npy"), line_bytes)
    log(f"dumped the lines of {int(has.sum())} of {reads.size} sampled reads ({line_bytes.size} bytes) to {d}")


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=os.environ.get("UTB_BENCH_CONFIG", "l2s"), choices=sorted(CONFIGS))
    ap.add_argument("--reads", type=int, default=0, help="reads per GPU (default: the config's)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the e2e_file / e2e_cli / e2e_pageable / single_process legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the output of the last timed e2e step there (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = dict(CONFIGS[args.config])
    if args.reads:
        cfg["reads"] = args.reads
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    ncpu = os.cpu_count() or 1
    workload = {"workload": cfg["desc"], "config": args.config, "reads_per_gpu": cfg["reads"], "read_len": cfg["read_len"] or "10kb-16Mb",
                "rc": True, "sharding": f"reads x{world}, CTR replicated", "l2_policy": "inputs larger than L2 (no flush needed)"}

    import torch
    if args.impl == "reference":
        return reference_arm(args, cfg, rank, world, local, ncpu, workload)

    import torch.distributed as dist
    from utree_b200 import build, capi
    build.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback")
    torch.cuda.set_device(local)
    cpu_group = None
    numa = bind_near_gpu(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        cpu_group = dist.new_group(backend="gloo")          # host-side waits that must not park a kernel on the GPUs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- inputs ------------------------------------------------------------
    if rank == 0:
        ctr_path, ctr_meta = ensure_ctr(args.config, cfg, local)
    barrier()
    if rank != 0:
        ctr_path, ctr_meta = ensure_ctr(args.config, cfg, local)
    n_reads = cfg["reads"]
    t = time.time()
    from utree_b200.shard import shard_range
    lo_read, hi_read = shard_range(world * n_reads, rank, world)    # this rank's contiguous range of the job's reads
    reads_np, off = make_reads(cfg, lo_read, hi_read - lo_read, local, pin=True)
    n_bases = int(off[-1]) - 13 * n_reads
    log(f"rank {rank}: {n_reads} reads ({reads_np.size / 1e9:.2f} GB FASTA, {n_bases / 1e9:.2f} G bases) in {time.time() - t:.1f} s")

    # ---- database resident in HBM ---------------------------------------------
    t = time.time()
    ctr = capi.Ctr(ctr_path)
    db = capi.Db(ctr, local)
    db_load_s = time.time() - t
    log(f"rank {rank}: CTR resident in HBM in {db_load_s:.1f} s ({ctr.num_nodes} records, {ctr.max_ix} labels)")

    # ---- value: device-resident pass over the chunks of the read set ---------------------
    chunks = chunks_of(off)
    cap_bytes = max(int(off[b] - off[a]) for a, b in chunks)
    cap_reads = max(b - a for a, b in chunks)
    batch = capi.Batch(db, cap_bytes, cap_reads)

    def load_chunk(a, b):
        """Stages chunk [a, b) in the batch and runs it once (H2D + kernels + D2H of the result records)."""
        base, nb = int(off[a]), int(off[b] - off[a])
        batch.bytes[:nb] = reads_np[base:base + nb]
        batch.seq_off[:b - a] = off[a:b] - np.uint64(base) + np.uint64(12)
        batch.seq_len[:b - a] = (off[a + 1:b + 1] - off[a:b] - np.uint64(13)).astype(np.uint32)
        batch.submit(nb, b - a, True)
        return batch.wait()

    sampler = ClockSampler(local)
    sampler.start()
    lookups = hits = 0
    resident_records = []                                   # result records of the resident pass (parity leg, rank 0)
    ms_sum = np.zeros(4)
    det_ms, det_sect = np.zeros(2), np.zeros(2)
    launches = 0
    single = len(chunks) == 1
    for step in range(-args.warmup, args.steps):
        if step == 0:
            barrier()
        for ci, (a, b) in enumerate(chunks):
            if not single or step == -args.warmup:
                res = load_chunk(a, b)                      # untimed: puts the chunk's bytes in HBM
                if step == -args.warmup:
                    lk, ht = batch.counts()
                    lookups += lk; hits += ht
                    if rank == 0:
                        resident_records.append(res)
            ms, l = batch.rerun_device(1)                   # timed on the device: CUDA events on the launching stream
            if step >= 0:
                ms_sum += np.array(ms)
                launches += l
                dm, ds = batch.lookup_detail()
                det_ms += np.array(dm)
                if step == 0:
                    det_sect += np.array(ds, dtype=np.float64)
    barrier()
    dev_s = ms_sum[3] / 1e3
    lookup_mode, hbm_bytes = db.lookup_mode(), int(db.hbm_bytes())
    batch.destroy(); db.free()          # the e2e searcher below uploads its own copy: never both resident at once
    host_threads = max(2, ncpu // max(world, 1))
    searcher = capi.Searcher(ctr, devices=(local,), host_threads=host_threads)

    # ---- e2e: host buffers through the C ABI --------------------------------------
    ptr = reads_np.ctypes.data
    out_text = None
    for _ in range(max(1, args.warmup)):
        rc_, ex, out_text, st = searcher.search_mem(None, do_rc=True, ptr=ptr, n=reads_np.size, copy=(rank == 0))
        assert rc_ == 0, capi.lib().utb_last_error()
    out_len = len(out_text) if rank == 0 else out_text
    barrier()
    t0 = time.time()
    e2e_stats, last_text = [], None
    for i in range(args.steps):
        if args.dump_outputs and rank == 0 and i == args.steps - 1:
            rc_, last_text, nbytes, st = search_mem_unread(capi, searcher, ptr, reads_np.size)
        else:
            rc_, ex, nbytes, st = searcher.search_mem(None, do_rc=True, ptr=ptr, n=reads_np.size, copy=False)
        assert rc_ == 0 and nbytes == out_len
        e2e_stats.append(st)
    own_e2e_s = time.time() - t0                                   # this rank alone; the figure uses the time up to the barrier, i.e. the slowest rank
    barrier()
    e2e_s = time.time() - t0
    if last_text is not None:
        import ctypes
        dump_outputs(args.dump_outputs, ctypes.string_at(last_text, nbytes) if nbytes else b"", lo_read, n_reads)
    clocks = sampler.summary()
    log(f"rank {rank}: e2e {own_e2e_s * 1e3 / args.steps:.1f} ms per step on its own ({ncpu} cores visible, {host_threads} host threads)")

    # ---- reduce over ranks: max time, sum of units -----------------------------------
    tt = torch.tensor([dev_s, e2e_s], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([float(lookups), float(hits), float(launches), float(n_bases)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    dev_s_max, e2e_s_max = tt.tolist()
    per_rank_ms = [round(own_e2e_s * 1e3 / args.steps, 1)]
    if world > 1:
        gathered = [torch.zeros(1, dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(gathered, torch.tensor([own_e2e_s * 1e3 / args.steps], dtype=torch.float64, device="cuda"))
        per_rank_ms = [round(float(g.item()), 1) for g in gathered]
    lookups_all, hits_all, launches_all, bases_all = cnt.tolist()

    # ---- extra legs (rank 0; the other ranks wait on the host) ----------------------------
    extra = {}
    if rank == 0 and not args.no_extra:
        extra = extra_legs(args, cfg, capi, searcher, ctr, ctr_path, reads_np, off, out_text, host_threads, world, local)
    if world > 1:
        dist.barrier(group=cpu_group)

    line = None
    if rank == 0:
        total_reads = n_reads * world * args.steps
        value = total_reads / dev_s_max
        lookups_per_s = lookups_all * args.steps / dev_s_max
        e2e_value = total_reads / e2e_s_max
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        stream_peak = peaks.get("hbm_gbs", 6650.0)
        rand32 = capi.measure_rand32(local, ws_bytes=8 << 30, loads=1 << 28, iters=3)
        # ---- parity of this very run -------------------------------------------------------
        n_chk = min(n_reads, 100_000 if cfg["read_len"] else 40)
        sect = oracle_sample(ctr_path, reads_np, off, n_chk, ncpu)
        assert out_text.startswith(sect["text"]), "bench output differs from the oracle"
        pos = 0
        for (a, b), res in zip(chunks, resident_records):   # the resident pass's records, formatted on the host, slice by slice
            for c0 in range(a, b, 2_000_000):
                c1 = min(b, c0 + 2_000_000)
                base = int(off[c0])
                txt = capi.format_results(ctr, reads_np[base:int(off[c1])], (off[c0:c1] - np.uint64(base) + np.uint64(1)).astype(np.uint32),
                                          np.full(c1 - c0, 10, dtype=np.uint32), res[c0 - a:c1 - a])
                assert out_text[pos:pos + len(txt)] == txt, f"resident records of reads [{c0}, {c1}) differ from the e2e text"
                pos += len(txt)
        assert pos == len(out_text), "e2e text longer than the resident pass's"
        parity = {"oracle_sample_reads": n_chk, "resident_vs_e2e_bytes": pos, "ok": True}
        if "e2e_cli" in extra:
            parity["cli_output_identical"] = extra["e2e_cli"].pop("identical")
            assert parity["cli_output_identical"], "CLI output file differs from the e2e text"
        if "e2e_file" in extra:
            parity["file_output_identical"] = extra["e2e_file"].pop("identical")
            assert parity["file_output_identical"], "utb_search_file output differs from the e2e text"
        # ---- roofline ----------------------------------------------------------------------
        steps = args.steps
        lookup_ms = ms_sum[1] / steps
        two_phase = det_ms[0] > 0
        ref_bytes = sect["bytes_per_lookup"] * lookups        # SURVEY 8d: what the reference's probe sequence would touch
        ref_equiv = ref_bytes / (lookup_ms * 1e-3) / 1e9
        n_pos = float(np.sum(((off[1:] - off[:-1] - np.uint64(13) + np.uint64(1) + np.uint64(31)) // np.uint64(32)) * np.uint64(32)))
        probes = det_sect[0] / 2.0                                  # ONE sieve fetch per position serves both strands
        surv_ms, sieve_ms = det_ms[1] / steps, det_ms[0] / steps
        vote_ms, pack_ms = ms_sum[2] / steps, ms_sum[0] / steps
        # candidates: (kernel, ms per step, algorithmic bytes per step, peak it is held against, what the bytes are)
        cand = []
        if two_phase:
            sieve_bytes = 8.0 * probes + (8 + 8 + 4) / 32.0 * n_pos + 12.0 * det_sect[1]
            cand.append(("sieve_kernel<2> (minimizer-keyed blocked Bloom: one 8 B block per position serves both strands, "
                         "one DRAM line per minimizer run)", sieve_ms, sieve_bytes, "stream",
                         "8 B sieve block per valid position + the packed streams in (pk, pkr, bad: 20 B per 32 positions) + one "
                         "12 B queue entry per survivor"))
            cand.append(("queue_lookup_kernel (exact sector-hash-table lookup of the sieve survivors)", surv_ms, 32.0 * det_sect[1],
                         "rand32", "32 B x the table sectors touched (counted on the device): the random accesses, which is what the peak it is "
                                   "held against measures; the 12 B queue entry read and the 4 B per hit appended to its read's list are sequential"))
            stage_bytes = sieve_bytes + 44.0 * det_sect[1]
        elif lookup_mode:
            cand.append(("lookup_kernel<2,true> (sector hash table, sieve off: dense tree)", lookup_ms, 32.0 * det_sect[1] + 20 / 32.0 * n_pos, "rand32",
                         "32 B x the table sectors touched, counted on the device"))
            stage_bytes = 32.0 * det_sect[1]
        else:
            cand.append(("lookup_kernel<2,false> (reference probe sequence)", lookup_ms, ref_bytes, "rand32", "SURVEY 8d reference-layout bytes"))
            stage_bytes = ref_bytes
        cand.append(("vote kernels (vote_thread / vote_warp / vote_block / vote_big_*: label multiset and aufbau walk)", vote_ms,
                     (4.0 * n_reads if two_phase else 8.0 * lookups) + 4.0 * hits + 32.0 * n_reads, "stream",
                     "per read: its hit count (4 B), its hit list (4 B per hit; sieve off: the dense hit slots), one 32 B result"))
        cand.append(("pack_kernel", pack_ms, float(n_bases) + 20 / 32.0 * n_pos, "stream", "1 B per base in, pk + pkr + bad out"))
        k_name, k_ms, k_bytes, k_peak, k_alg = max(cand, key=lambda c: c[1])
        achieved = k_bytes / (k_ms * 1e-3) / 1e9
        peak = stream_peak if k_peak == "stream" else rand32
        traffic = None
        try:        # ncu dram__bytes_read + dram__bytes_write of the kernel at exactly this shape (one --set full capture per round)
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(args.config, {})
            if tr.get("reads") == n_reads:
                traffic = tr.get(k_name.split("<")[0].split(" ")[0])
        except Exception:
            pass
        roofline = {"bound": "hbm", "kernel": k_name, "achieved": round(achieved, 1), "peak": round(peak, 1),
                    "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic,
                    "algorithmic_bytes": k_alg,
                    "peak_kind": ("MEASURED_PEAKS.json hbm_gbs (streaming copy)" if k_peak == "stream" else
                                  "measured random 32B-sector gather, 8 GiB working set (utb_measure_rand32)"),
                    "rand32_peak": round(rand32, 1), "stream_peak": stream_peak,
                    "stream_peak_kind": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback",
                    "kernels": [{"kernel": c[0].split(" ")[0], "ms": round(float(c[1]), 3),
                                 "alg_gbs": round(c[2] / (c[1] * 1e-3) / 1e9, 1) if c[1] > 0 else None,
                                 "frac": round(c[2] / (c[1] * 1e-3) / 1e9 / (stream_peak if c[3] == "stream" else rand32), 4) if c[1] > 0 else None,
                                 "peak": c[3]} for c in cand],
                    "sieve_probes_per_s": round(probes / (sieve_ms * 1e-3), 1) if two_phase else None,
                    "phase_a_ms": {"sieve_kernel": round(float(sieve_ms), 3)} if two_phase else None,
                    "kernel_ms": round(float(k_ms), 3), "kernel_share_of_step": round(float(k_ms * steps / ms_sum[3]), 4),
                    "lookups_per_step": lookups,
                    "lookup_stage": {"ms": round(float(lookup_ms), 3), "bytes": stage_bytes,
                                     "gbs": round(stage_bytes / (lookup_ms * 1e-3) / 1e9, 1),
                                     "survivor_kernel_ms": round(float(surv_ms), 3),
                                     "survivors_per_lookup": round(det_sect[1] / max(lookups, 1), 4) if two_phase else None},
                    "reference_layout_equiv": {"bytes_per_lookup": round(sect["bytes_per_lookup"], 2), "gbs": round(ref_equiv, 1),
                                               "ratio_to_rand32_peak": round(ref_equiv / rand32, 3),
                                               "note": "SURVEY 8d figure: what the reference's bisection would touch per lookup; "
                                                       "above 1 because the path no longer performs those probes"},
                    "stage_ms": {"pack": round(float(pack_ms), 3), "lookup": round(float(lookup_ms), 3), "vote": round(float(vote_ms), 3)}}
        cpu = None
        if world == 1 and not args.no_cpu:
            exe = ref_binary(cfg)
            if exe:
                rate, n_s, secs, _ = cpu_reference_rate(cfg, ctr_path, reads_np, off, 12.0, ncpu)
                bps = float(off[n_s] - 13 * n_s) / secs
                cpu = {"value": round(rate, 1), "unit": "reads/s", "cores": ncpu, "kind": "reference",
                       "sample": f"first {n_s} of the same reads, reference binary threads={ncpu}, wall minus 1-read run, {secs:.1f} s",
                       "bases_per_s": round(bps, 1), "lookups_per_s": round(rate * sect["lookups_per_read"], 1)}
                try:                                                  # and single-threaded (the parity configuration)
                    r1, n1, s1, _ = cpu_reference_rate(cfg, ctr_path, reads_np, off, 4.0, 1)
                    cpu["value_1thread"] = round(r1, 1)
                    cpu["sample_1thread"] = f"first {n1} reads, threads=1, {s1:.1f} s"
                except Exception as e:                                # never fail the bench line over the extra figure
                    cpu["value_1thread"] = None
                    log(f"1-thread reference run failed: {e}")
            else:
                cpu = {"value": round(sect["port_reads_per_s"], 1), "unit": "reads/s", "cores": ncpu, "kind": "port",
                       "sample": f"first {n_chk} of the same reads, oracle port with {ncpu} OpenMP threads (with sector accounting)",
                       "lookups_per_s": round(sect["port_reads_per_s"] * sect["lookups_per_read"], 1)}
        st = e2e_stats[-1]
        line = {
            "metric": "reads/sec (150bp, L2-scale CTR, RC); k-mer lookups/sec in lookups_per_s",
            "value": round(value, 1), "unit": "reads/s", "lookups_per_s": round(lookups_per_s, 1),
            "bases_per_s": round(bases_all * args.steps / dev_s_max, 1),
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(dev_s_max * 1e3 / args.steps, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": workload,
            "e2e": {"value": round(e2e_value, 1), "unit": "reads/s", "h2d_bytes_per_step": int(st["h2d_bytes"]),
                    "d2h_bytes_per_step": int(st["d2h_bytes"]), "ms_per_step": round(e2e_s_max * 1e3 / args.steps, 1), "per_rank_ms": per_rank_ms,
                    "bases_per_s": round(bases_all * args.steps / e2e_s_max, 1),
                    "api": "utb_search_mem (page-locked host FASTA buffer -> text in the searcher's page-locked arena, "
                           "allocated once by the warm-up steps)", "out_bytes_per_step": int(st["out_bytes"]),
                    "host_phase_s": {k: round(st[k], 3) for k in ("rd_wait_slot", "rd_fill", "rd_frame", "rd_submit",
                                                                 "fm_wait_gpu", "fm_format", "fm_emit", "seconds_device")}},
            "gpu_launches": int(launches_all), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "parity": parity,
            "db": {"records": int(ctr.num_nodes), "labels": int(ctr.max_ix), "file_bytes": ctr_meta["bytes"],
                   "hbm_bytes": hbm_bytes, "load_s": round(db_load_s, 1)},
            "hit_rate": round(hits / max(lookups, 1), 4), "lookups_per_read": round(lookups / n_reads, 2),
        }
        if numa is not None:
            line["host_affinity"] = dict(numa, note="each rank runs on the cores local to its GPU (rank 0 shown)")
        line.update(extra)
    searcher.destroy(); ctr.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line:
        emit_json(line)


def extra_legs(args, cfg, capi, searcher, ctr, ctr_path, reads_np, off, out_text, host_threads, world, local):
    """Rank 0, after the main figures: the drop-in CLI file -> file, a pageable caller buffer, and (N > 1) ONE
    searcher over all N devices.  Each is bounded to a few steps."""
    import torch
    n_reads = off.size - 1
    ex = {}
    wd = work_dir()
    try:    # ---- the CLI, file -> file on /dev/shm (reference arm's recipe: wall minus a 1-read run)
        exe = os.path.join(ROOT, "bin", "utree-search_gg")
        fa, one, out = (os.path.join(wd, f"cli_{os.getpid()}.{x}") for x in ("fa", "one.fa", "out"))
        reads_np.tofile(fa)
        reads_np[:int(off[1])].tofile(one)
        t_one = min(cli_run(exe, ctr_path, one, out, host_threads)[0] for _ in range(2))
        runs = [cli_run(exe, ctr_path, fa, out, host_threads) for _ in range(2)]
        t_full = min(r[0] for r in runs)
        t_search = min((r[1] for r in runs if r[1]), default=None)
        same = os.path.getsize(out) == len(out_text) and open(out, "rb").read() == out_text
        ex["e2e_cli"] = {"value": round(n_reads / t_search, 1) if t_search else None, "unit": "reads/s", "search_s": t_search,
                         "wall_s": round(t_full, 2), "wall_1read_s": round(t_one, 2),
                         "how": "bin/utree-search_gg ctr fasta out <threads> RC, files on " + wd + ", best of 2; value = reads / the search "
                                "time the process reports (UTB_STATS), wall_s = the whole process incl. tree load + table build, "
                                "wall_1read_s = the same command on a 1-read FASTA", "identical": same}
        # the same file -> file search through the C ABI of the searcher that is already up (what a long-lived
        # caller pays per FASTA): utb_search_file, input and output on tmpfs
        best, st_best = None, None
        for _ in range(3):
            t = time.time()
            rc_, _, st_ = searcher.search_file(fa, out, do_rc=True)
            dt = time.time() - t
            assert rc_ == 0
            if best is None or dt < best:
                best, st_best = dt, st_
        same2 = os.path.getsize(out) == len(out_text) and open(out, "rb").read() == out_text
        ex["e2e_file"] = {"value": round(n_reads / best, 1), "unit": "reads/s", "ms": round(best * 1e3, 1), "identical": same2,
                          "in_bytes": int(reads_np.size), "out_bytes": len(out_text),
                          "host_phase_s": {k: round(st_best[k], 3) for k in ("rd_wait_slot", "rd_fill", "rd_frame", "rd_submit", "fm_wait_gpu", "fm_emit", "seconds_device")},
                          "how": "utb_search_file(fasta, out) on the resident searcher, files on " + wd + ", best of 3 (host-side "
                                 "pread into page-locked slots and pwrite of the text bound it, not the GPU)"}
        for f in (fa, one, out):
            os.remove(f)
    except Exception as e:
        log(f"e2e_file leg failed: {e}")
        ex["e2e_file_error"] = str(e)[:200]
    try:    # ---- pageable caller buffer (staged through the batch's page-locked buffers by the reader threads)
        pageable = np.array(reads_np, copy=True)
        searcher.search_mem(None, do_rc=True, ptr=pageable.ctypes.data, n=pageable.size, copy=False)
        t = time.time()
        rc_, _, nb, _ = searcher.search_mem(None, do_rc=True, ptr=pageable.ctypes.data, n=pageable.size, copy=False)
        dt = time.time() - t
        assert rc_ == 0 and nb == len(out_text)
        ex["e2e_pageable"] = {"value": round(n_reads / dt, 1), "unit": "reads/s", "ms": round(dt * 1e3, 1),
                              "how": f"utb_search_mem from an ordinary numpy buffer, {host_threads} host threads"}
        del pageable
    except Exception as e:
        log(f"e2e_pageable leg failed: {e}")
    if world > 1:
        try:    # ---- ONE searcher over all devices: strong scaling of one FASTA of world x the reads
            os.sched_setaffinity(0, ALL_CPUS)                       # this leg drives every GPU from one process: all cores, input spread over the nodes
            spread = mem_interleave(True)
            big, boff = make_reads(cfg, 0, n_reads * world, local, pin=True)
            mem_interleave(False)
            s2 = capi.Searcher(ctr, devices=tuple(range(world)), host_threads=max(2, (os.cpu_count() or 2) // 2))
            n_out = None
            for _ in range(2):
                rc_, _, n_out, _ = s2.search_mem(None, do_rc=True, ptr=big.ctypes.data, n=big.size, copy=False)
                assert rc_ == 0
            t = time.time()
            k = max(1, min(args.steps, 3))
            for _ in range(k):
                rc_, _, nb, st = s2.search_mem(None, do_rc=True, ptr=big.ctypes.data, n=big.size, copy=False)
                assert rc_ == 0 and nb == n_out
            dt = (time.time() - t) / k
            ex["single_process"] = {"value": round(n_reads * world / dt, 1), "unit": "reads/s", "ms_per_step": round(dt * 1e3, 1),
                                    "n_devices": world, "reads": n_reads * world, "out_bytes": int(n_out), "input_interleaved_over_numa_nodes": bool(spread),
                                    "how": "ONE utb_searcher over all devices (tables uploaded once, cloned over NVLink), one FASTA, "
                                           "ordered merge; the other ranks idle on the host"}
            s2.destroy()
            del big
        except Exception as e:
            log(f"single_process leg failed: {e}")
            ex["single_process_error"] = str(e)[:200]
    return ex


def reference_arm(args, cfg, rank, world, local, ncpu, workload):
    """`--impl reference`: the reference's own CPU implementation of the path, all host threads,
    bounded sample per step.  Rank 0 alone works."""
    if rank != 0:
        return
    import torch
    have_gpu = torch.cuda.is_available()
    ctr_path = os.path.join(work_dir(), f"ctr_{cfg_key(args.config, cfg)}.ctr")
    if not os.path.exists(ctr_path):
        if not have_gpu:
            emit_json({"impl": "reference", "unavailable": "synthetic CTR needs the GPU synthesiser and no GPU is visible"})
            return
        ctr_path, _ = ensure_ctr(args.config, cfg, local)
    n_avail = min(cfg["reads"], 2_000_000 if cfg["read_len"] else 400)
    reads_np, off = make_reads(cfg, 0, n_avail, local)
    exe = ref_binary(cfg)
    steps_total = args.steps + args.warmup
    budget = max(2.0, min(12.0, 150.0 / steps_total))
    times, state = [], None
    kind = "reference" if exe else "port"
    if exe:
        for i in range(steps_total):
            rate, n_s, secs, state = cpu_reference_rate(cfg, ctr_path, reads_np, off, budget, ncpu, state)
            if i >= args.warmup:
                times.append((n_s, secs))
    else:
        orc = oracle_api.OracleDb(ctr_path)
        fa = os.path.join(work_dir(), f"refport_{os.getpid()}.fa")
        n_s = min(n_avail, 200_000 if cfg["read_len"] else 20)
        reads_np[:int(off[n_s])].tofile(fa)
        for i in range(steps_total):
            t = time.time()
            orc.search_file(fa, fa + ".out", do_rc=True, threads=ncpu)
            if i >= args.warmup:
                times.append((n_s, time.time() - t))
        orc.free()
    tot_reads = sum(n for n, _ in times)
    tot_s = sum(s for _, s in times)
    value = tot_reads / tot_s
    line = {"impl": "reference", "metric": "reads/sec (150bp, L2-scale CTR, RC); k-mer lookups/sec in lookups_per_s",
            "value": round(value, 1), "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(tot_s * 1e3 / args.steps, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": workload,
            "cpu_baseline": {"value": round(value, 1), "unit": "reads/s", "cores": ncpu, "kind": kind,
                             "sample": f"{times[0][0]} reads per step of the same synthetic reads; search time = wall minus a 1-read run"},
            "e2e": {"value": round(value, 1), "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit_json(line)


if __name__ == "__main__":
    main()
