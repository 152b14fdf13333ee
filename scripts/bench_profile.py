"""Sample profile cost on the L2S workload (10 M x 150 bp reads, RC) on one GPU: reads/s and bytes over PCIe for the
text alone, the text plus the profile, and the profile alone, through utb_search_mem from a page-locked buffer and
utb_search_file file to file on /dev/shm; then profile_kernel + profile_compact_kernel time per batch from a
torch.profiler run of its own.  The profile is checked against Counter(column 2 of the text) inside the run.

    python scripts/bench_profile.py [--reads N] [--repeats R] [--out DIR]

Prints one JSON line per mode and one for the kernels; with --out also writes them there."""
import argparse
import collections
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = q.stdout.splitlines()[0].split(", ")
    return {"gpu": name, "power_limit": power}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import bench
    from utree_b200 import build, capi
    build.build()
    info = gpu_info()
    cfg = dict(bench.CONFIGS["l2s"])
    ctr_path, _ = bench.ensure_ctr("l2s", cfg, 0)
    reads, off = bench.make_reads(cfg, 0, args.reads, 0, pin=True)
    n = off.size - 1
    ctr = capi.Ctr(ctr_path)
    threads = min(os.cpu_count() or 1, 64)
    s = capi.Searcher(ctr, devices=(0,), host_threads=threads)
    wd = bench.work_dir()
    fa, out = os.path.join(wd, f"prof_{os.getpid()}.fa"), os.path.join(wd, f"prof_{os.getpid()}.out")
    reads.tofile(fa)
    lines = []

    def emit(d):
        d.update(info, workload=cfg["desc"], reads=n)
        lines.append(json.dumps(d))
        print(lines[-1], flush=True)

    def timed(fn):
        fn()                                                       # warm-up
        best, st = None, None
        for _ in range(args.repeats):
            t = time.time()
            st_ = fn()
            dt = time.time() - t
            if best is None or dt < best:
                best, st = dt, st_
        return best, st

    ptr = reads.ctypes.data
    legs = {
        "mem_text": (False, lambda: s.search_mem(None, do_rc=True, ptr=ptr, n=reads.size, copy=False)[3]),
        "mem_text_profile": (True, lambda: s.search_mem(None, do_rc=True, ptr=ptr, n=reads.size, copy=False)[3]),
        "mem_profile": (True, lambda: s.search_mem(None, do_rc=True, ptr=ptr, n=reads.size, text=False)[3]),
        "file_text": (False, lambda: s.search_file(fa, out, do_rc=True)[2]),
        "file_text_profile": (True, lambda: s.search_file(fa, out, do_rc=True)[2]),
        "file_profile": (True, lambda: s.search_file(fa, None, do_rc=True)[2]),
    }
    profiles = {}
    for name, (on, fn) in legs.items():
        s.set_profile(on)
        dt, st = timed(fn)
        if on:
            profiles[name] = s.profile()
        emit({"leg": name, "reads_per_s": round(n / dt, 1), "ms": round(dt * 1e3, 1), "h2d_bytes": st["h2d_bytes"],
              "d2h_bytes": st["d2h_bytes"], "out_bytes": st["out_bytes"], "batches": st["batches"],
              "kernel_launches": st["kernel_launches"], "good_finds": st["good_finds"], "best_of": args.repeats})
    # the oracle: column 2 of the text of the same search
    s.set_profile(True)
    rc, _, text, st = s.search_mem(None, do_rc=True, ptr=ptr, n=reads.size)
    assert rc == 0
    want = sorted(collections.Counter(line.split(b"\t")[-4] for line in text.split(b"\n")[:-1]).items())
    del text
    got = [(t, c) for t, c, _ in s.profile()[0]]
    assert got == want, "profile differs from the text"
    assert all(p == profiles["mem_text_profile"] for p in profiles.values()), "profiles differ between modes"
    # kernel time: a profiled run of its own (profile only)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rc, _, _, st = s.search_mem(None, do_rc=True, ptr=ptr, n=reads.size, text=False)
        torch.cuda.synchronize()
    ks = collections.defaultdict(lambda: [0, 0.0])
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and ("profile_kernel" in e.name or "profile_compact_kernel" in e.name):
            k = "profile_compact_kernel" if "compact" in e.name else "profile_kernel"
            ks[k][0] += 1
            ks[k][1] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
    emit({"leg": "kernels", "batches": st["batches"], "rows": len(got),
          **{k: {"launches": c, "us_total": round(t, 1), "us_per_batch": round(t / max(c, 1), 1)} for k, (c, t) in ks.items()},
          "us_per_10M_reads": round(sum(t for _, t in ks.values()) * 1e7 / n, 1), "how": "torch.profiler, CUDA activities"})
    for f in (fa, out):
        if os.path.exists(f):
            os.remove(f)
    s.destroy(); ctr.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_profile.jsonl"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
