import hashlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")
REFDIR = os.path.join(ROOT, "oracle", "_ref")
REFERENCE_RUNS = os.path.join(GOLD, "reference_runs.json")


def _digest(data, text):
    e = {"bytes": len(data), "sha256": hashlib.sha256(data).hexdigest()}
    if text:
        lines = data.split(b"\n")
        idx = np.random.default_rng(len(lines)).choice(len(lines), min(40, len(lines)), replace=False)
        e["lines"] = len(lines)
        e["sample"] = {str(i): lines[i].decode("latin-1") for i in sorted(idx.tolist())}
    return e


def check_reference_run(name, got, text=True):
    """`got` == the bytes the reference wrote for case `name`.  tests/golden/reference_runs.json keeps their size and
    sha256 and, for text, the line count and a seeded sample of lines, compared first so that a mismatch names a line.
    UTB_RECORD_REFERENCE_RUNS=1 writes the entry instead of comparing (see "_about" in that file)."""
    runs = json.load(open(REFERENCE_RUNS)) if os.path.exists(REFERENCE_RUNS) else {}
    if os.environ.get("UTB_RECORD_REFERENCE_RUNS") == "1":
        runs[name] = _digest(got, text)
        with open(REFERENCE_RUNS, "w") as f:
            json.dump(runs, f, indent=1, sort_keys=True)
        return
    assert name in runs, f"no recorded reference output for {name}"
    want = runs[name]
    if text:
        lines = got.split(b"\n")
        assert len(lines) == want["lines"], name
        for i, line in want["sample"].items():
            assert lines[int(i)].decode("latin-1") == line, (name, int(i))
    assert (len(got), hashlib.sha256(got).hexdigest()) == (want["bytes"], want["sha256"]), name


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def built():
    """Product library + oracle built in-tree (no-op when up to date)."""
    from utree_b200 import build
    build.build()
    if not os.path.exists(os.path.join(ROOT, "oracle", "liboracle.so")):
        import subprocess
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "liboracle.so", "oracle_search"], check=True)
    return True


@pytest.fixture(scope="session")
def meta():
    return json.load(open(os.path.join(GOLD, "meta.json")))


@pytest.fixture(scope="session")
def ctrs(tmp_path_factory, built):
    """The golden .ubt fixtures compressed to .ctr the way utree-compress
    does (synth.compress is checked against the reference's sha256)."""
    from tools import synth
    d = tmp_path_factory.mktemp("ctr")
    out = {}
    for name in ("toyA", "toyB_u32", "quirk", "dense"):
        p = str(d / (name + ".ctr"))
        synth.compress(os.path.join(GOLD, name + ".ubt"), p)
        out[name] = p
    return out


# (db, reads, golden output, RC)
CASES = [
    ("toyA", "toyA_reads.fa", "toyA_rc.out", 1),
    ("toyA", "toyA_reads.fa", "toyA_norc.out", 0),
    ("toyB_u32", "toyB_reads.fa", "toyB_u32_rc.out", 1),
    ("quirk", "quirk_reads.fa", "quirk_rc.out", 1),
    ("quirk", "quirk_reads.fa", "quirk_norc.out", 0),
    ("dense", "dense_reads.fa", "dense_rc.out", 1),
    ("dense", "dense_reads.fa", "dense_norc.out", 0),
    ("toyA", "long_reads.fa", "long_rc.out", 1),
    ("toyA", "edge_reads.fa", "edge_rc.out", 1),
]
BAD_CASES = ["bad_noheader.fa", "bad_seq_is_header.fa", "bad_truncated.fa"]


def gold(name):
    return os.path.join(GOLD, name)


def read_fasta(path):
    """[(name, seq)] using the reference reader's trimming rules."""
    recs = []
    with open(path, "rb") as f:
        while True:
            h = f.readline()
            if not h:
                break
            s = f.readline()
            name = h[1:].split(b" ")[0].split(b"\n")[0]
            if s.endswith(b"\n"):
                s = s[:-1]
            if s.endswith(b"\r"):
                s = s[:-1]
            recs.append((name, s))
    return recs
