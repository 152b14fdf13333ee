"""ctypes mirror of include/utree_b200.h (the product's C ABI).  No compute
happens in Python: every call below lands in libutree_b200.so, and a missing
library or a missing GPU is a hard error -- there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LIB_PATH = os.path.join(HERE, "csrc", "libutree_b200.so")

UTB_NONE, UTB_STAR, UTB_WALK = 0, 1, 2
CUT_EMPTY, CUT_FULL = 0xFFFFFFFF, 0xFFFFFFFE
BAD32 = 0xFFFFFFFF
INPUT_FASTA, INPUT_FASTQ, INPUT_FASTA_WRAPPED = 0, 1, 2
FQ_NOHEADER, FQ_NOSEPARATOR, FQ_QUALLEN, FQ_TOOLONG, FQ_TRUNCATED = 1, 2, 3, 4, 5
FW_NOHEADER, FW_TOOLONG = 1, 4


class UtbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"utb error {code}: {msg}")
        self.code = code


class Result(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("kind", "label", "cut", "found", "uix", "sl", "ol", "_pad")]


RESULT_DTYPE = np.dtype([(n, "<u4") for n in ("kind", "label", "cut", "found", "uix", "sl", "ol", "_pad")])


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("reads", "good_finds", "lookups", "hits", "batches",
                                          "kernel_launches", "h2d_bytes", "d2h_bytes", "out_bytes")] + \
               [(n, C.c_double) for n in ("seconds_total", "seconds_device", "rd_wait_slot", "rd_fill", "rd_frame",
                                          "rd_submit", "fm_wait_gpu", "fm_format", "fm_emit")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


# every symbol include/utree_b200.h declares (tests check the .so exports all)
EXPORTS = [
    "utb_last_error", "utb_ctr_open", "utb_ctr_close", "utb_ctr_num_nodes", "utb_ctr_ix_bytes",
    "utb_ctr_binix_bytes", "utb_ctr_max_ix", "utb_ctr_last_bin", "utb_ctr_label", "utb_ctr_label_rank",
    "utb_device_count", "utb_db_upload", "utb_db_free", "utb_db_hbm_bytes", "utb_db_lookup_mode",
    "utb_batch_create", "utb_batch_destroy", "utb_batch_bytes", "utb_batch_seq_off", "utb_batch_seq_len",
    "utb_batch_max_bytes", "utb_batch_max_reads", "utb_read_slots", "utb_batch_max_slots",
    "utb_batch_submit", "utb_batch_wait", "utb_batch_name_off", "utb_batch_name_len", "utb_batch_rerun_device", "utb_batch_counts", "utb_batch_lookup_detail", "utb_db_clone", "utb_db_device",
    "utb_lookup_words", "utb_pack_sequence", "utb_vote_hits", "utb_vote_hits_sparse", "utb_frame_records", "utb_frame_fastq_records", "utb_frame_wrapped_records", "utb_format_results",
    "utb_searcher_create", "utb_searcher_destroy", "utb_search_file", "utb_search_mem", "utb_free",
    "utb_main", "utb_main_shallow", "utb_build_ubt", "utb_build_main", "utb_searcher_set_shallow", "utb_searcher_set_input",
    "utb_searcher_set_profile", "utb_searcher_profile", "utb_profile_main", "utb_measure_rand32", "utb_compress_ubt", "utb_compress_main",
]

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise UtbError(-1, f"{LIB_PATH} is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                               "there is no fallback implementation")
        L = C.CDLL(LIB_PATH)
        L.utb_last_error.restype = C.c_char_p
        L.utb_ctr_num_nodes.restype = C.c_uint64
        L.utb_ctr_last_bin.restype = C.c_uint64
        L.utb_ctr_label.restype = C.c_char_p
        L.utb_ctr_label.argtypes = [C.c_void_p, C.c_uint32]
        L.utb_ctr_label_rank.argtypes = [C.c_void_p, C.c_uint32]
        L.utb_ctr_label_rank.restype = C.c_uint32
        for f in ("utb_ctr_num_nodes", "utb_ctr_ix_bytes", "utb_ctr_binix_bytes", "utb_ctr_max_ix", "utb_ctr_last_bin",
                  "utb_ctr_close", "utb_db_free", "utb_db_hbm_bytes", "utb_batch_destroy", "utb_searcher_destroy",
                  "utb_batch_bytes", "utb_batch_seq_off", "utb_batch_seq_len", "utb_batch_max_bytes",
                  "utb_batch_max_reads", "utb_batch_max_slots", "utb_free"):
            getattr(L, f).argtypes = [C.c_void_p]
        for f in ("utb_ctr_close", "utb_db_free", "utb_batch_destroy", "utb_searcher_destroy", "utb_free"):
            getattr(L, f).restype = None
        for f in ("utb_batch_bytes", "utb_batch_seq_off", "utb_batch_seq_len"):
            getattr(L, f).restype = C.c_void_p
        for f in ("utb_db_hbm_bytes", "utb_batch_max_slots", "utb_read_slots"):
            getattr(L, f).restype = C.c_uint64
        for f in ("utb_batch_max_bytes", "utb_batch_max_reads"):
            getattr(L, f).restype = C.c_size_t
        L.utb_read_slots.argtypes = [C.c_uint32]
        L.utb_ctr_open.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
        L.utb_device_count.argtypes = [C.POINTER(C.c_int)]
        L.utb_db_upload.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        L.utb_batch_create.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.POINTER(C.c_void_p)]
        L.utb_batch_submit.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int]
        L.utb_batch_wait.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.utb_batch_rerun_device.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_uint64)]
        L.utb_batch_counts.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.utb_lookup_words.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.utb_pack_sequence.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.utb_vote_hits.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.utb_frame_records.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.c_int, C.c_size_t] + [C.c_void_p] * 4 + \
            [C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_int)]
        L.utb_searcher_create.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.utb_search_file.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p, C.c_int, C.POINTER(Stats), C.POINTER(C.c_int)]
        L.utb_search_mem.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p),
                                     C.POINTER(C.c_size_t), C.POINTER(Stats), C.POINTER(C.c_int)]
        L.utb_main.argtypes = [C.c_int, C.POINTER(C.c_char_p)]
        L.utb_measure_rand32.argtypes = [C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.POINTER(C.c_double)]
        _lib = L
    return _lib


def _ck(rc):
    if rc:
        raise UtbError(rc, lib().utb_last_error().decode(errors="replace"))


class Ctr:
    """Host view of a CTR file (utb_ctr_open)."""

    def __init__(self, path):
        self.h = C.c_void_p()
        _ck(lib().utb_ctr_open(os.fsencode(path), C.byref(self.h)))
        L = lib()
        self.num_nodes = L.utb_ctr_num_nodes(self.h)
        self.ix_bytes = L.utb_ctr_ix_bytes(self.h)
        self.binix_bytes = L.utb_ctr_binix_bytes(self.h)
        self.max_ix = L.utb_ctr_max_ix(self.h)
        self.last_bin = L.utb_ctr_last_bin(self.h)

    def label(self, ix):
        return lib().utb_ctr_label(self.h, ix)

    def rank(self, ix):
        return lib().utb_ctr_label_rank(self.h, ix)

    def close(self):
        if self.h:
            lib().utb_ctr_close(self.h)
            self.h = C.c_void_p()


def frame_records(buf: bytes, eof=True, threads=1, max_reads=None):
    """Host framer (utb_frame_records).  Returns (rc, ref_exit, used, [(name, seq)])."""
    cap = max_reads if max_reads is not None else len(buf) // 2 + 2
    seq_off = np.zeros(cap, dtype=np.uint64)
    seq_len = np.zeros(cap, dtype=np.uint32)
    name_off = np.zeros(cap, dtype=np.uint32)
    name_len = np.zeros(cap, dtype=np.uint32)
    n, used, ex = C.c_size_t(), C.c_size_t(), C.c_int()
    rc = lib().utb_frame_records(buf, len(buf), int(eof), threads, cap, seq_off.ctypes.data, seq_len.ctypes.data,
                                 name_off.ctypes.data, name_len.ctypes.data, C.byref(n), C.byref(used), C.byref(ex))
    recs = [(buf[name_off[i]:name_off[i] + name_len[i]], buf[seq_off[i]:seq_off[i] + seq_len[i]]) for i in range(n.value)]
    return rc, ex.value, used.value, recs, (name_off[:n.value].copy(), name_len[:n.value].copy())


def frame_fastq_records(buf: bytes, eof=True, threads=1, max_reads=None):
    """Host FASTQ framer (utb_frame_fastq_records).  Returns (rc, used, [(name, seq, qual)], (err_record, err_code));
    err_record is 1-based, (0, 0) when every record is well formed."""
    cap = max_reads if max_reads is not None else len(buf) // 4 + 2
    seq_off = np.zeros(cap, dtype=np.uint64)
    qual_off = np.zeros(cap, dtype=np.uint64)
    seq_len = np.zeros(cap, dtype=np.uint32)
    name_off = np.zeros(cap, dtype=np.uint32)
    name_len = np.zeros(cap, dtype=np.uint32)
    n, used, er, ec = C.c_size_t(), C.c_size_t(), C.c_size_t(), C.c_int()
    L = lib()
    L.utb_frame_fastq_records.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.c_int, C.c_size_t] + [C.c_void_p] * 5 + \
        [C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_int)]
    rc = L.utb_frame_fastq_records(buf, len(buf), int(eof), threads, cap, seq_off.ctypes.data, seq_len.ctypes.data,
                                   qual_off.ctypes.data, name_off.ctypes.data, name_len.ctypes.data,
                                   C.byref(n), C.byref(used), C.byref(er), C.byref(ec))
    recs = [(buf[name_off[i]:name_off[i] + name_len[i]], buf[seq_off[i]:seq_off[i] + seq_len[i]],
             buf[qual_off[i]:qual_off[i] + seq_len[i]]) for i in range(n.value)]
    return rc, used.value, recs, (er.value, ec.value)


def frame_wrapped_records(buf: bytes, eof=True, threads=1, max_reads=None):
    """Host wrapped-FASTA framer (utb_frame_wrapped_records).  Returns (rc, used, [(name, joined sequence)],
    (err_record, err_code)); err_record is 1-based, (0, 0) when every record is well formed."""
    cap = max_reads if max_reads is not None else len(buf) // 2 + 2
    seq_out = np.zeros(len(buf) + 1, dtype=np.uint8)
    seq_off = np.zeros(cap, dtype=np.uint64)
    seq_len = np.zeros(cap, dtype=np.uint32)
    name_off = np.zeros(cap, dtype=np.uint32)
    name_len = np.zeros(cap, dtype=np.uint32)
    n, used, er, ec = C.c_size_t(), C.c_size_t(), C.c_size_t(), C.c_int()
    L = lib()
    L.utb_frame_wrapped_records.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_size_t] + \
        [C.c_void_p] * 4 + [C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_int)]
    rc = L.utb_frame_wrapped_records(buf, len(buf), int(eof), threads, cap, seq_out.ctypes.data, len(buf), seq_off.ctypes.data,
                                     seq_len.ctypes.data, name_off.ctypes.data, name_len.ctypes.data,
                                     C.byref(n), C.byref(used), C.byref(er), C.byref(ec))
    joined = seq_out.tobytes()
    recs = [(buf[name_off[i]:name_off[i] + name_len[i]], joined[seq_off[i]:seq_off[i] + seq_len[i]]) for i in range(n.value)]
    return rc, used.value, recs, (er.value, ec.value)


def format_results(ctr, buf, name_off, name_len, results):
    """Host formatter (utb_format_results) -> bytes.  buf: bytes or a uint8 numpy array holding the names."""
    results = np.ascontiguousarray(results, dtype=RESULT_DTYPE)
    name_off = np.ascontiguousarray(name_off, dtype=np.uint32)
    name_len = np.ascontiguousarray(name_len, dtype=np.uint32)
    src = np.frombuffer(buf, dtype=np.uint8) if isinstance(buf, (bytes, bytearray)) else np.ascontiguousarray(buf, dtype=np.uint8)
    if not hasattr(ctr, "_max_label"):
        ctr._max_label = max((len(ctr.label(i)) for i in range(ctr.max_ix)), default=0)
    cap = int(name_len.sum()) + results.size * (ctr._max_label + 64) + 64
    out = np.empty(cap, dtype=np.uint8)
    n = C.c_size_t()
    L = lib()
    L.utb_format_results.argtypes = [C.c_void_p, C.c_void_p] + [C.c_void_p] * 3 + [C.c_size_t, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
    _ck(L.utb_format_results(ctr.h, src.ctypes.data, name_off.ctypes.data, name_len.ctypes.data, results.ctypes.data,
                             results.size, out.ctypes.data, cap, C.byref(n)))
    return out[:n.value].tobytes()


def compress_ubt(ubt_path, ctr_path):
    """utree-compress equivalent (utb_compress_ubt).  Returns (n_records, n_labels)."""
    n, nl = C.c_uint64(), C.c_uint32()
    lib().utb_compress_ubt.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]
    _ck(lib().utb_compress_ubt(os.fsencode(ubt_path), os.fsencode(ctr_path), C.byref(n), C.byref(nl)))
    return n.value, nl.value


class BuildStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("map_bytes", "map_lines", "sequences", "kmers_seen", "kmers_made", "records")] + [("labels", C.c_uint32)]


def build_ubt(fasta, map_path, out, complevel=1, gg=True, ix_bytes=2, device=0):
    """utree-build_gg on the GPU (utb_build_ubt).  Returns (rc, ref_exit, stats dict)."""
    st, ex = BuildStats(), C.c_int()
    L = lib()
    L.utb_build_ubt.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint32, C.c_int, C.c_int, C.c_int, C.POINTER(BuildStats), C.POINTER(C.c_int)]
    rc = L.utb_build_ubt(os.fsencode(fasta), os.fsencode(map_path), os.fsencode(out), complevel, int(gg), ix_bytes, device, C.byref(st), C.byref(ex))
    return rc, ex.value, {n: getattr(st, n) for n, _ in st._fields_}


def device_count():
    n = C.c_int()
    _ck(lib().utb_device_count(C.byref(n)))
    return n.value


class Db:
    """CTR resident in one GPU's HBM (utb_db_upload) + stage-level calls."""

    def __init__(self, ctr: Ctr, device=0):
        self.ctr = ctr
        self.h = C.c_void_p()
        _ck(lib().utb_db_upload(ctr.h, device, C.byref(self.h)))

    def lookup_words(self, words):
        words = np.ascontiguousarray(words, dtype=np.uint64)
        out = np.empty(words.size, dtype=np.uint32)
        _ck(lib().utb_lookup_words(self.h, words.ctypes.data, words.size, out.ctypes.data))
        return out

    def pack_sequence(self, seq: bytes):
        n = len(seq)
        fwd = np.zeros(n, dtype=np.uint64)
        rc = np.zeros(n, dtype=np.uint64)
        valid = np.zeros(n, dtype=np.uint8)
        _ck(lib().utb_pack_sequence(self.h, seq, n, fwd.ctypes.data, rc.ctypes.data, valid.ctypes.data))
        return fwd, rc, valid

    def vote_hits(self, hits, off, sparse=False):
        """sparse=True: through the pipeline's per-read hit lists (thread -> warp -> block kernels)."""
        hits = np.ascontiguousarray(hits, dtype=np.uint32)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        n = off.size - 1
        res = np.zeros(n, dtype=RESULT_DTYPE)
        fn = lib().utb_vote_hits_sparse if sparse else lib().utb_vote_hits
        fn.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        _ck(fn(self.h, hits.ctypes.data, off.ctypes.data, n, res.ctypes.data))
        return res

    def hbm_bytes(self):
        return lib().utb_db_hbm_bytes(self.h)

    def lookup_mode(self):
        """1: sector hash table (+ sieve) on a regular CTR; 0: reference probe sequence."""
        lib().utb_db_lookup_mode.argtypes = [C.c_void_p]
        return lib().utb_db_lookup_mode(self.h)

    def clone(self, device):
        """The finished tables copied to another GPU (peer copy; utb_db_clone)."""
        other = Db.__new__(Db)
        other.ctr, other.h = self.ctr, C.c_void_p()
        lib().utb_db_clone.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        _ck(lib().utb_db_clone(self.h, device, C.byref(other.h)))
        return other

    def free(self):
        if self.h:
            lib().utb_db_free(self.h)
            self.h = C.c_void_p()


class Batch:
    """One stream slot (utb_batch_*): pinned staging + device buffers."""

    def __init__(self, db: Db, max_bytes, max_reads):
        self.db = db
        self.h = C.c_void_p()
        _ck(lib().utb_batch_create(db.h, max_bytes, max_reads, C.byref(self.h)))
        L = lib()
        self.max_bytes, self.max_reads = max_bytes, max_reads
        self.bytes = np.ctypeslib.as_array(C.cast(L.utb_batch_bytes(self.h), C.POINTER(C.c_uint8)), (max_bytes,))
        self.seq_off = np.ctypeslib.as_array(C.cast(L.utb_batch_seq_off(self.h), C.POINTER(C.c_uint64)), (max_reads,))
        self.seq_len = np.ctypeslib.as_array(C.cast(L.utb_batch_seq_len(self.h), C.POINTER(C.c_uint32)), (max_reads,))
        self.n_reads = 0

    def submit(self, n_bytes, n_reads, do_rc):
        self.n_reads = n_reads
        _ck(lib().utb_batch_submit(self.h, n_bytes, n_reads, int(do_rc)))

    def wait(self):
        p = C.c_void_p()
        _ck(lib().utb_batch_wait(self.h, C.byref(p)))
        if not self.n_reads:
            return np.zeros(0, dtype=RESULT_DTYPE)
        buf = (C.c_uint8 * (self.n_reads * RESULT_DTYPE.itemsize)).from_address(p.value)
        return np.frombuffer(buf, dtype=RESULT_DTYPE).copy()

    def rerun_device(self, iters=1):
        ms = (C.c_float * 4)()
        launches = C.c_uint64()
        _ck(lib().utb_batch_rerun_device(self.h, iters, ms, C.byref(launches)))
        return [ms[i] for i in range(4)], launches.value

    def counts(self):
        a, b = C.c_uint64(), C.c_uint64()
        _ck(lib().utb_batch_counts(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def lookup_detail(self):
        ms, sec = (C.c_float * 2)(), (C.c_uint64 * 2)()
        lib().utb_batch_lookup_detail.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_uint64)]
        _ck(lib().utb_batch_lookup_detail(self.h, ms, sec))
        return [ms[0], ms[1]], [sec[0], sec[1]]

    def destroy(self):
        if self.h:
            lib().utb_batch_destroy(self.h)
            self.h = C.c_void_p()


class ProfileRow(C.Structure):
    _fields_ = [("label", C.c_uint32), ("len", C.c_uint32), ("reads", C.c_uint64)]


class Searcher:
    """Whole search over one or more GPUs (utb_searcher_* / utb_search_*)."""

    def __init__(self, ctr: Ctr, devices=(0,), host_threads=1):
        self.ctr = ctr
        self.h = C.c_void_p()
        arr = (C.c_int * len(devices))(*devices)
        _ck(lib().utb_searcher_create(ctr.h, arr, len(devices), host_threads, C.byref(self.h)))

    def set_shallow(self, on=True):
        """The non-GG binary's search (utb_searcher_set_shallow)."""
        lib().utb_searcher_set_shallow.argtypes = [C.c_void_p, C.c_int]
        _ck(lib().utb_searcher_set_shallow(self.h, int(on)))

    def set_input(self, fastq=True, min_qual=0, wrapped=False):
        """Input format of the following searches (utb_searcher_set_input): 4-line FASTQ, bases whose quality byte is
        below 33 + min_qual counted as N (0: no masking); fastq=False: FASTA, linearised, or with wrapped=True
        wrapped (multi-line) FASTA."""
        if fastq and wrapped:
            raise ValueError("set_input: wrapped input is FASTA only (fastq=False, wrapped=True)")
        lib().utb_searcher_set_input.argtypes = [C.c_void_p, C.c_int, C.c_uint32]
        fmt = INPUT_FASTQ if fastq else INPUT_FASTA_WRAPPED if wrapped else INPUT_FASTA
        _ck(lib().utb_searcher_set_input(self.h, fmt, min_qual))

    def set_profile(self, on=True):
        """Count reads per taxonomy string in the following searches (utb_searcher_set_profile)."""
        lib().utb_searcher_set_profile.argtypes = [C.c_void_p, C.c_int]
        _ck(lib().utb_searcher_set_profile(self.h, int(on)))

    def profile(self):
        """The last search's profile (utb_searcher_profile): ([(taxonomy bytes, reads, label)] in row order,
        unclassified reads)."""
        L = lib()
        L.utb_searcher_profile.argtypes = [C.c_void_p, C.POINTER(C.POINTER(ProfileRow)), C.POINTER(C.c_size_t), C.POINTER(C.c_uint64)]
        rows, n, uncl = C.POINTER(ProfileRow)(), C.c_size_t(), C.c_uint64()
        _ck(L.utb_searcher_profile(self.h, C.byref(rows), C.byref(n), C.byref(uncl)))
        return [(self.ctr.label(rows[i].label)[:rows[i].len], rows[i].reads, rows[i].label) for i in range(n.value)], uncl.value

    def search_file(self, fasta, out, do_rc=True):
        """out=None: no output file (with the profile on: the profile alone)."""
        st, ex = Stats(), C.c_int()
        rc = lib().utb_search_file(self.h, os.fsencode(fasta), None if out is None else os.fsencode(out), int(do_rc),
                                   C.byref(st), C.byref(ex))
        return rc, ex.value, st.as_dict()

    def search_mem(self, fasta: bytes, do_rc=True, ptr=None, n=None, copy=True, text=True):
        """copy=False: the output text is not copied into Python (returns its length instead).  text=False: no output
        is asked for (NULL out and out_len; with the profile on: the profile alone); returns None for the text."""
        st, ex = Stats(), C.c_int()
        out, out_len = C.c_void_p(), C.c_size_t()
        if ptr is None:
            keep = C.create_string_buffer(fasta, len(fasta))
            ptr, n = C.addressof(keep), len(fasta)
        if not text:
            rc = lib().utb_search_mem(self.h, ptr, n, int(do_rc), None, None, C.byref(st), C.byref(ex))
            return rc, ex.value, None, st.as_dict()
        rc = lib().utb_search_mem(self.h, ptr, n, int(do_rc), C.byref(out), C.byref(out_len), C.byref(st), C.byref(ex))
        data = out_len.value
        if copy:
            data = C.string_at(out.value, out_len.value) if out.value else b""
        if out.value:
            lib().utb_free(out)
        return rc, ex.value, data, st.as_dict()

    def destroy(self):
        if self.h:
            lib().utb_searcher_destroy(self.h)
            self.h = C.c_void_p()


def measure_rand32(device=0, ws_bytes=8 << 30, loads=1 << 28, iters=3):
    g = C.c_double()
    _ck(lib().utb_measure_rand32(device, ws_bytes, loads, iters, C.byref(g)))
    return g.value
