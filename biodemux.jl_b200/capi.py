"""ctypes binding of libbdx (include/bdx.h) and the ``Engine`` convenience wrapper.

This is the Python twin of the ``ccall`` shim in ``julia/BioDemuXB200.jl``: it fills
``bdx_params`` from a ``DemuxConfig`` and drives submit / fetch.  It never classifies
on the CPU -- if the shared library or a CUDA device is missing it raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional, Sequence

import numpy as np

from .config import DemuxConfig
from .demux import DETAIL_DTYPE, RESULT_DTYPE, pack_reads

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BDX_LIB") or os.path.join(_HERE, "csrc", "libbdx.so")
ABI_VERSION = 1

BDX_OK, BDX_ERR_INVALID, BDX_ERR_CUDA, BDX_ERR_NOMEM, BDX_ERR_STATE, BDX_ERR_TOO_LARGE = 0, -1, -2, -3, -4, -5

# every symbol include/bdx.h declares (tests check that the library exports all of them)
DEBUG_NO_FILTER, DEBUG_NO_PREFILTER, DEBUG_NO_SEEDS, DEBUG_NO_SEED_DEEP = 1, 2, 4, 8
DEBUG_ONE_SEED_LEVEL, DEBUG_NO_GRAPHS, DEBUG_NO_HAMMING_PACKED, DEBUG_PREFER_SEED_VAR = 16, 32, 64, 128
DEBUG_NO_QGRAM_FILTER = 256

EXPORTS = [
    "bdx_last_error", "bdx_abi_version", "bdx_device_count", "bdx_config_create", "bdx_config_create_debug", "bdx_config_destroy",
    "bdx_stream_work_counters", "bdx_config_code_table", "bdx_config_describe", "bdx_pack_reads4", "bdx_submit_packed4", "bdx_submit_packed4_pinned",
    "bdx_window_spans", "bdx_window_reads", "bdx_submit_windows", "bdx_submit_windows_pinned",
    "bdx_stream_create", "bdx_stream_destroy", "bdx_submit", "bdx_acquire", "bdx_commit",
    "bdx_submit_pinned", "bdx_host_alloc", "bdx_host_free", "bdx_stream_enable_details",
    "bdx_fetch", "bdx_fetch_view", "bdx_classify", "bdx_classify_device", "bdx_stream_sync",
    "bdx_stream_cuda_stream", "bdx_stream_launch_count", "bdx_stream_profile", "bdx_stream_profile_read", "bdx_stream_profile_read_stages", "bdx_stream_path_counters", "bdx_stats_layout_get", "bdx_stats_fetch",
    "bdx_stats_device_ptr", "bdx_stats_reset", "bdx_synth_reads_device", "bdx_int_alu_peak",
    "bdx_fastq_scan", "bdx_fastq_pack", "bdx_demux_block", "bdx_demux_stage_ms",
    "bdx_barcode_table_load", "bdx_barcode_table_destroy", "bdx_barcode_table_count", "bdx_barcode_table_id_count",
    "bdx_barcode_table_bytes", "bdx_barcode_table_offsets", "bdx_barcode_table_lengths_no_n", "bdx_barcode_table_id",
    "bdx_barcode_table_error", "bdx_stats_entries",
    "bdx_pool_create", "bdx_pool_destroy", "bdx_pool_submit", "bdx_pool_submit_pinned", "bdx_pool_fetch",
    "bdx_pool_fetch_view", "bdx_pool_in_flight", "bdx_pool_stats_fetch", "bdx_stats_overflow_fetch",
]


class BdxError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libbdx error {code}: {msg}")
        self.code = code


class Range(C.Structure):
    _fields_ = [("start_offset", C.c_int64), ("start_from_end", C.c_int32), ("end_from_end", C.c_int32),
                ("end_offset", C.c_int64)]


class BarcodeSet(C.Structure):
    _fields_ = [("n_barcodes", C.c_int32), ("trim_side", C.c_int32), ("bytes", C.c_void_p),
                ("offsets", C.c_void_p), ("lengths_no_n", C.c_void_p), ("ref_search_range", Range),
                ("barcode_start_range", Range), ("barcode_end_range", Range)]


class Params(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("abi_version", C.c_uint32), ("max_error_rate", C.c_double),
                ("min_delta", C.c_double), ("match", C.c_int64), ("mismatch", C.c_int64),
                ("indel", C.c_int64), ("nindel", C.c_int64), ("has_nindel", C.c_int32),
                ("algorithm", C.c_int32), ("is_dual", C.c_int32), ("want_stats", C.c_int32),
                ("set1", BarcodeSet), ("set2", BarcodeSet)]


class StatsLayout(C.Structure):
    _fields_ = [("total_len", C.c_int64), ("sample_off", C.c_int64), ("b1", C.c_int32), ("b2", C.c_int32),
                ("pos_bins", C.c_int32), ("len_bins", C.c_int32), ("dist_bins", C.c_int32),
                ("pos_bias", C.c_int32), ("dist_bias", C.c_int32), ("reserved", C.c_int32),
                ("pos_off", C.c_int64 * 2), ("len_off", C.c_int64 * 2),
                ("dist_off", C.c_int64 * 2)]


class SynthSpec(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("first_read", C.c_int64), ("read_len", C.c_int32),
                ("plant_permille", C.c_int32), ("start_lo", C.c_int32), ("start_hi", C.c_int32),
                ("n_permille_x10", C.c_int32), ("set2_mode", C.c_int32), ("end_lo", C.c_int32),
                ("end_hi", C.c_int32)]


class DemuxOut(C.Structure):
    _fields_ = [("n_records", C.c_int32), ("n_buckets", C.c_int32), ("consumed1", C.c_int64),
                ("consumed2", C.c_int64), ("out1", C.c_void_p), ("out1_len", C.c_int64), ("out2", C.c_void_p),
                ("out2_len", C.c_int64), ("buckets", C.c_void_p), ("results", C.c_void_p)]


# bdx_demux_bucket (include/bdx.h)
BUCKET_DTYPE = np.dtype([("status", "<i4"), ("bc1", "<i4"), ("bc2", "<i4"), ("n_records", "<i4"),
                         ("offset1", "<i8"), ("length1", "<i8"), ("offset2", "<i8"), ("length2", "<i8")])
DEMUX_SINGLE, DEMUX_MATES, DEMUX_BOTH, DEMUX_DEVICE_IO = 0, 1, 2, 16

FASTQ_REC_DTYPE = np.dtype([("header_off", "<i8"), ("seq_off", "<i8"), ("plus_off", "<i8"), ("qual_off", "<i8"),
                            ("header_len", "<i4"), ("seq_len", "<i4"), ("plus_len", "<i4"), ("qual_len", "<i4")])

_LIB = None


def build_library(force: bool = False) -> str:
    """Compile csrc/ with nvcc for sm_100a (works without a GPU)."""
    if force or not os.path.exists(LIB_PATH):
        subprocess.run(["make", "-s", "-C", os.path.join(_HERE, "csrc")], check=True,
                       stdout=subprocess.DEVNULL)
    return LIB_PATH


def load_library():
    """Loads libbdx.so; raises if it is missing (no fallback)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise BdxError(BDX_ERR_CUDA, f"{LIB_PATH} not built: run `make -C biodemux.jl_b200/csrc` "
                                     "(or __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    L.bdx_last_error.restype = C.c_char_p
    L.bdx_abi_version.restype = C.c_int
    L.bdx_device_count.restype = C.c_int
    L.bdx_config_create.argtypes = [C.POINTER(Params), C.POINTER(vp)]
    L.bdx_config_create_debug.argtypes = [C.POINTER(Params), C.c_uint32, C.POINTER(vp)]
    L.bdx_config_code_table.argtypes = [vp, vp]
    L.bdx_config_describe.argtypes = [vp, C.c_int, C.c_char_p, C.c_int]
    L.bdx_pack_reads4.argtypes = [vp, vp, i64, vp]
    L.bdx_submit_packed4.argtypes = [vp, vp, vp, C.c_int32, C.c_uint64]
    L.bdx_submit_packed4_pinned.argtypes = [vp, vp, vp, C.c_int32, C.c_uint64]
    L.bdx_window_spans.argtypes = [vp, i32, vp]
    L.bdx_window_reads.argtypes = [vp, vp, vp, i32, vp, vp]
    L.bdx_submit_windows.argtypes = [vp, vp, vp, vp, i32, C.c_int, u64]
    L.bdx_submit_windows_pinned.argtypes = [vp, vp, vp, vp, i32, C.c_int, u64]
    L.bdx_config_destroy.argtypes = [vp]
    L.bdx_config_destroy.restype = None
    L.bdx_stream_create.argtypes = [vp, C.c_int, i32, i64, C.POINTER(vp)]
    L.bdx_stream_destroy.argtypes = [vp]
    L.bdx_stream_destroy.restype = None
    L.bdx_submit.argtypes = [vp, vp, vp, i32, u64]
    L.bdx_submit_pinned.argtypes = [vp, vp, vp, i32, u64]
    L.bdx_acquire.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    L.bdx_commit.argtypes = [vp, i32, u64]
    L.bdx_host_alloc.argtypes = [C.c_size_t]
    L.bdx_host_alloc.restype = vp
    L.bdx_host_free.argtypes = [vp]
    L.bdx_host_free.restype = None
    L.bdx_stream_enable_details.argtypes = [vp, C.c_int]
    L.bdx_fetch.argtypes = [vp, C.POINTER(u64), C.POINTER(i32), vp, vp]
    L.bdx_fetch_view.argtypes = [vp, C.POINTER(u64), C.POINTER(i32), C.POINTER(vp), C.POINTER(vp)]
    L.bdx_classify.argtypes = [vp, vp, vp, i32, vp, vp]
    L.bdx_classify_device.argtypes = [vp, vp, vp, i32, vp, vp]
    L.bdx_stream_sync.argtypes = [vp]
    L.bdx_stream_cuda_stream.argtypes = [vp]
    L.bdx_stream_cuda_stream.restype = vp
    L.bdx_stream_launch_count.argtypes = [vp]
    L.bdx_stream_launch_count.restype = i64
    L.bdx_stream_profile.argtypes = [vp, C.c_int]
    L.bdx_stream_profile_read.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(i32)]
    L.bdx_stream_profile_read_stages.argtypes = [vp, C.POINTER(C.c_double * 8), C.POINTER(i32 * 8)]
    L.bdx_stream_path_counters.argtypes = [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.c_int]
    L.bdx_stats_layout_get.argtypes = [vp, C.POINTER(StatsLayout)]
    L.bdx_stats_fetch.argtypes = [vp, vp, i64]
    L.bdx_stats_overflow_fetch.argtypes = [vp, vp, i64, C.POINTER(i64), C.POINTER(i64)]
    L.bdx_stats_entries.argtypes = [vp, vp, vp, i64]
    L.bdx_stats_entries.restype = i64
    L.bdx_stats_device_ptr.argtypes = [vp]
    L.bdx_stats_device_ptr.restype = vp
    L.bdx_stats_reset.argtypes = [vp]
    L.bdx_synth_reads_device.argtypes = [vp, C.POINTER(SynthSpec), i32, vp, vp]
    L.bdx_int_alu_peak.argtypes = [C.c_int, C.POINTER(C.c_double)]
    L.bdx_fastq_scan.argtypes = [vp, i64, C.c_int, i32, vp, C.POINTER(i32), C.POINTER(i64)]
    L.bdx_fastq_pack.argtypes = [vp, vp, i32, vp, i64, vp]
    L.bdx_pool_create.argtypes = [vp, C.POINTER(C.c_int), C.c_int, C.c_int, i32, i64, C.POINTER(vp)]
    L.bdx_pool_destroy.argtypes = [vp]
    L.bdx_pool_destroy.restype = None
    L.bdx_pool_submit.argtypes = [vp, vp, vp, i32, u64]
    L.bdx_pool_submit_pinned.argtypes = [vp, vp, vp, i32, u64]
    L.bdx_pool_fetch.argtypes = [vp, C.POINTER(u64), C.POINTER(i32), vp, vp]
    L.bdx_pool_fetch_view.argtypes = [vp, C.POINTER(u64), C.POINTER(i32), C.POINTER(vp), C.POINTER(vp)]
    L.bdx_pool_in_flight.argtypes = [vp]
    L.bdx_pool_stats_fetch.argtypes = [vp, vp, i64]
    L.bdx_barcode_table_load.argtypes = [C.c_char_p, C.c_int, C.c_int, C.POINTER(vp)]
    L.bdx_barcode_table_destroy.argtypes = [vp]
    L.bdx_barcode_table_destroy.restype = None
    for name in ("count", "id_count"):
        getattr(L, "bdx_barcode_table_" + name).argtypes = [vp]
        getattr(L, "bdx_barcode_table_" + name).restype = i32
    for name in ("bytes", "offsets", "lengths_no_n"):
        getattr(L, "bdx_barcode_table_" + name).argtypes = [vp]
        getattr(L, "bdx_barcode_table_" + name).restype = vp
    L.bdx_barcode_table_id.argtypes = [vp, i32]
    L.bdx_barcode_table_id.restype = C.c_char_p
    L.bdx_barcode_table_error.restype = C.c_char_p
    L.bdx_demux_block.argtypes = [vp, vp, i64, vp, i64, C.c_int, C.c_int, C.POINTER(DemuxOut)]
    L.bdx_demux_stage_ms.argtypes = [vp, C.POINTER(C.c_float * 8)]
    _LIB = L
    return L


def _check(rc: int):
    if rc != BDX_OK:
        raise BdxError(rc, load_library().bdx_last_error().decode("utf-8", "replace"))


def _range(dr) -> Range:
    return Range(dr.start_offset, int(dr.start_from_end), int(dr.end_from_end), dr.end_offset)


def fastq_scan(buf: np.ndarray, final_block: bool, max_records: int):
    """bdx_fastq_scan over a uint8 array -> (records structured array, bytes consumed)."""
    recs = np.zeros(max_records, dtype=FASTQ_REC_DTYPE)
    n, consumed = C.c_int32(), C.c_int64()
    _check(load_library().bdx_fastq_scan(buf.ctypes.data if buf.size else None, buf.size, int(final_block),
                                         max_records, recs.ctypes.data, C.byref(n), C.byref(consumed)))
    return recs[:n.value], consumed.value


def fastq_pack(buf: np.ndarray, recs: np.ndarray, seq_out: Optional[np.ndarray] = None):
    """bdx_fastq_pack -> (packed sequence bytes, int32 offsets)."""
    recs = np.ascontiguousarray(recs)
    total = int(recs["seq_len"].sum())
    if seq_out is None:
        seq_out = np.zeros(max(total, 1), dtype=np.uint8)
    off = np.zeros(len(recs) + 1, dtype=np.int32)
    _check(load_library().bdx_fastq_pack(buf.ctypes.data if buf.size else None, recs.ctypes.data, len(recs),
                                         seq_out.ctypes.data, seq_out.size, off.ctypes.data))
    return seq_out[:total], off


STATS_OVERFLOW_DTYPE = np.dtype([("pass", "<i4"), ("bc", "<i4"), ("start", "<i4"), ("length", "<i4")])
STATS_ENTRY_DTYPE = np.dtype([("pass", "<i4"), ("kind", "<i4"), ("bc", "<i4"), ("reserved", "<i4"),
                              ("key", "<i8"), ("score", "<f8"), ("count", "<i8")])


def stats_entries(config: "Config", counters: np.ndarray) -> np.ndarray:
    """bdx_stats_entries: the DemuxStats Dict entries of a (summed) counter buffer."""
    L = load_library()
    counters = np.ascontiguousarray(counters, dtype=np.int64)
    n = L.bdx_stats_entries(config.handle, counters.ctypes.data, None, 0)
    if n < 0:
        _check(int(n))
    out = np.zeros(int(n), dtype=STATS_ENTRY_DTYPE)
    L.bdx_stats_entries(config.handle, counters.ctypes.data, out.ctypes.data, int(n))
    return out


def load_barcode_table(path: str, complement: bool = False, rev: bool = False):
    """bdx_barcode_table_load -> ``(sequences, lengths_no_N, ids)`` like preprocess_bc_file (fileio.jl:7-72)."""
    L = load_library()
    h = C.c_void_p()
    rc = L.bdx_barcode_table_load(os.fsencode(path), int(complement), int(rev), C.byref(h))
    if rc != BDX_OK:
        raise BdxError(rc, L.bdx_barcode_table_error().decode("utf-8", "replace"))
    try:
        n, n_ids = L.bdx_barcode_table_count(h), L.bdx_barcode_table_id_count(h)
        off = np.ctypeslib.as_array(C.cast(L.bdx_barcode_table_offsets(h), C.POINTER(C.c_int32)), (n + 1,)).copy()
        blob = C.string_at(L.bdx_barcode_table_bytes(h), int(off[-1]))
        lens = (np.ctypeslib.as_array(C.cast(L.bdx_barcode_table_lengths_no_n(h), C.POINTER(C.c_int32)), (n,)).tolist()
                if n else [])
        seqs = [blob[off[i]:off[i + 1]].decode("utf-8", "replace") for i in range(n)]
        ids = [L.bdx_barcode_table_id(h, i).decode("utf-8", "replace") for i in range(n_ids)]
    finally:
        L.bdx_barcode_table_destroy(h)
    return seqs, lens, ids


class Config:
    """Owns a ``bdx_config`` (immutable; shareable across streams)."""

    def __init__(self, cfg: DemuxConfig, want_stats: Optional[bool] = None, debug: int = 0):
        """debug: BDX_DEBUG_* flags (tests only: single pipeline stages switched off)."""
        self.lib = load_library()
        self.cfg = cfg
        self._keep = []
        p = Params()
        p.struct_size = C.sizeof(Params)
        p.abi_version = ABI_VERSION
        p.max_error_rate = float(cfg.max_error_rate)
        p.min_delta = float(cfg.min_delta)
        p.match, p.mismatch, p.indel = int(cfg.match), int(cfg.mismatch), int(cfg.indel)
        p.has_nindel = 0 if cfg.nindel is None else 1
        p.nindel = 0 if cfg.nindel is None else int(cfg.nindel)
        p.algorithm = cfg.algorithm_code
        p.is_dual = int(bool(cfg.is_dual))
        p.want_stats = int(bool(cfg.summary if want_stats is None else want_stats))
        p.set1 = self._set(cfg.bc_seqs, cfg.bc_lengths_no_N, cfg.ref_search_range, cfg.barcode_start_range,
                           cfg.barcode_end_range, cfg.trim_side)
        if cfg.is_dual:
            p.set2 = self._set(cfg.bc_seqs2, cfg.bc_lengths_no_N2, cfg.ref_search_range2,
                               cfg.barcode_start_range2, cfg.barcode_end_range2, cfg.trim_side2)
        self.params = p
        self.handle = C.c_void_p()
        if debug:
            _check(self.lib.bdx_config_create_debug(C.byref(p), int(debug), C.byref(self.handle)))
        else:
            _check(self.lib.bdx_config_create(C.byref(p), C.byref(self.handle)))
        self.layout = StatsLayout()
        _check(self.lib.bdx_stats_layout_get(self.handle, C.byref(self.layout)))

    def describe(self, pass_: int = 0) -> str:
        """bdx_config_describe: one line per table built for barcode set ``pass_`` (0 / 1) -- diagnostics and tests."""
        n = self.lib.bdx_config_describe(self.handle, pass_, None, 0)
        if n < 0:
            _check(n)
        buf = C.create_string_buffer(n + 1)
        self.lib.bdx_config_describe(self.handle, pass_, buf, n + 1)
        return buf.value.decode()

    def code_table(self) -> np.ndarray:
        """byte -> 4-bit code of the packed input (raises when the config has > 15 distinct barcode bytes)."""
        t = np.zeros(256, np.uint8)
        rc = self.lib.bdx_config_code_table(self.handle, t.ctypes.data)
        if rc < 0:
            _check(rc)
        return t

    def pack4(self, seq: np.ndarray, out: Optional[np.ndarray] = None) -> np.ndarray:
        """bdx_pack_reads4: the concatenated read bytes as 4-bit codes, two per byte."""
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        if out is None:
            out = np.zeros((seq.size + 1) // 2, np.uint8)
        _check(self.lib.bdx_pack_reads4(self.handle, seq.ctypes.data, seq.size, out.ctypes.data))
        return out

    def window_spans(self, read_len: int):
        """bdx_window_spans: ((lo1, hi1, lo2, hi2), window length) of a read of ``read_len`` bases."""
        sp = np.zeros(4, np.int32)
        n = self.lib.bdx_window_spans(self.handle, int(read_len), sp.ctypes.data)
        if n < 0:
            _check(n)
        return tuple(int(x) for x in sp), int(n)

    def window_reads(self, seq: np.ndarray, off: np.ndarray):
        """bdx_window_reads: (window bytes, int32 window offsets) of the concatenated reads ``seq`` / ``off``."""
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.int32)
        n = len(off) - 1
        win_off = np.zeros(n + 1, np.int32)
        _check(self.lib.bdx_window_reads(self.handle, None, off.ctypes.data, n, None, win_off.ctypes.data))
        win = np.zeros(max(int(win_off[-1]), 1), np.uint8)
        _check(self.lib.bdx_window_reads(self.handle, seq.ctypes.data if seq.size else None, off.ctypes.data, n,
                                         win.ctypes.data, win_off.ctypes.data))
        return win[:int(win_off[-1])], win_off

    def _set(self, seqs: Sequence[str], lens: Sequence[int], rs, bs, be, trim) -> BarcodeSet:
        raw = [s.encode("latin-1") if isinstance(s, str) else bytes(s) for s in seqs]
        blob = np.frombuffer(b"".join(raw) + b"\0", dtype=np.uint8).copy()
        off = np.zeros(len(raw) + 1, dtype=np.int32)
        off[1:] = np.cumsum([len(x) for x in raw])
        ln = np.asarray(list(lens), dtype=np.int32) if len(lens) else np.zeros(1, np.int32)
        self._keep += [blob, off, ln]
        s = BarcodeSet()
        s.n_barcodes = len(raw)
        s.trim_side = 0 if trim is None else int(trim)
        s.bytes = blob.ctypes.data
        s.offsets = off.ctypes.data
        s.lengths_no_n = ln.ctypes.data
        s.ref_search_range = _range(rs)
        s.barcode_start_range = _range(bs)
        s.barcode_end_range = _range(be)
        return s

    def close(self):
        if self.handle:
            self.lib.bdx_config_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Stream:
    """Owns a ``bdx_stream`` (one per host worker)."""

    def __init__(self, config: Config, device: int = 0, max_reads: int = 4000, max_bytes: Optional[int] = None):
        self.lib = config.lib
        self.config = config
        self.max_reads = int(max_reads)
        self.max_bytes = int(max_bytes if max_bytes is not None else max(self.max_reads, 1) * 1024)
        self.handle = C.c_void_p()
        _check(self.lib.bdx_stream_create(config.handle, device, self.max_reads, self.max_bytes,
                                          C.byref(self.handle)))
        self.details = bool(config.params.want_stats)

    def enable_details(self, on: bool = True):
        _check(self.lib.bdx_stream_enable_details(self.handle, int(on)))
        self.details = bool(on)

    def submit(self, seq: np.ndarray, off: np.ndarray, tag: int = 0, pinned: bool = False):
        n = len(off) - 1
        fn = self.lib.bdx_submit_pinned if pinned else self.lib.bdx_submit
        _check(fn(self.handle, seq.ctypes.data, off.ctypes.data, n, tag))

    def submit_packed4(self, packed: np.ndarray, off: np.ndarray, tag: int = 0, pinned: bool = False):
        """4-bit packed reads (Config.pack4) + the offsets of the unpacked reads."""
        fn = self.lib.bdx_submit_packed4_pinned if pinned else self.lib.bdx_submit_packed4
        _check(fn(self.handle, packed.ctypes.data, off.ctypes.data, len(off) - 1, tag))

    def submit_windows(self, win: np.ndarray, win_off: np.ndarray, off: np.ndarray, packed4: bool = False,
                       pinned: bool = False, tag: int = 0):
        """The reads' window bytes (Config.window_reads; packed4: those packed by Config.pack4) + the window offsets
        + the offsets of the full reads."""
        fn = self.lib.bdx_submit_windows_pinned if pinned else self.lib.bdx_submit_windows
        _check(fn(self.handle, win.ctypes.data if win.size else None, win_off.ctypes.data, off.ctypes.data,
                  len(off) - 1, int(packed4), tag))

    def fetch(self, want_details: bool = False, copy: bool = True):
        """Oldest in-flight batch.  copy=False returns views into the stream's pinned result
        staging (valid until BDX_MAX_IN_FLIGHT - 1 further submits)."""
        tag, n = C.c_uint64(), C.c_int32()
        res_p, det_p = C.c_void_p(), C.c_void_p()
        _check(self.lib.bdx_fetch_view(self.handle, C.byref(tag), C.byref(n), C.byref(res_p), C.byref(det_p)))
        nn = n.value
        if nn == 0:
            res = np.zeros(0, RESULT_DTYPE)
            det = np.zeros((2, 0), DETAIL_DTYPE)
        else:
            buf = (C.c_char * (nn * RESULT_DTYPE.itemsize)).from_address(res_p.value)
            res = np.frombuffer(buf, dtype=RESULT_DTYPE, count=nn)
            if copy:
                res = res.copy()
            det = None
            if want_details:
                if not det_p.value:
                    raise BdxError(BDX_ERR_STATE, "details not enabled on this stream")
                dbuf = (C.c_char * (2 * nn * DETAIL_DTYPE.itemsize)).from_address(det_p.value)
                det = np.frombuffer(dbuf, dtype=DETAIL_DTYPE, count=2 * nn).reshape(2, nn)
                if copy:
                    det = det.copy()
        return (tag.value, res, det) if want_details else (tag.value, res)

    def classify(self, seq: np.ndarray, off: np.ndarray, want_details: bool = False):
        """One batch through bdx_classify (host buffers in, host results out)."""
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.int32)
        n = len(off) - 1
        res = np.zeros(n, RESULT_DTYPE)
        det = np.zeros((2, n), DETAIL_DTYPE) if want_details else None
        if seq.size == 0:
            seq = np.zeros(1, np.uint8)
        _check(self.lib.bdx_classify(self.handle, seq.ctypes.data, off.ctypes.data, n, res.ctypes.data,
                                     det.ctypes.data if det is not None else None))
        return (res, det) if want_details else res

    def classify_device(self, d_seq: int, d_off: int, n: int, d_res: int, d_det: int = 0):
        _check(self.lib.bdx_classify_device(self.handle, d_seq, d_off, n, d_res, d_det or None))

    def synth_device(self, spec: SynthSpec, n: int, d_seq: int, d_off: int):
        _check(self.lib.bdx_synth_reads_device(self.handle, C.byref(spec), n, d_seq, d_off))

    def sync(self):
        _check(self.lib.bdx_stream_sync(self.handle))

    @property
    def cuda_stream(self) -> int:
        return int(self.lib.bdx_stream_cuda_stream(self.handle) or 0)

    @property
    def launch_count(self) -> int:
        return int(self.lib.bdx_stream_launch_count(self.handle))

    def profile(self, on: bool):
        _check(self.lib.bdx_stream_profile(self.handle, int(on)))

    def profile_read(self):
        ms, n = C.c_double(), C.c_int32()
        _check(self.lib.bdx_stream_profile_read(self.handle, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    # "k_seed": k_seed levels / k_seed_var level 1; "k_seed_deep": k_seed_deep / k_seed_var's complete level
    STAGES = ("k_prefilter", "k_seed", "k_seed_deep", "k_filter", "k_literal", "k_hamming_scan", "k_finalize", "other")

    def profile_read_stages(self):
        """{stage: (summed ms, launches)} of the launches profiled since the last read."""
        ms, n = (C.c_double * 8)(), (C.c_int32 * 8)()
        _check(self.lib.bdx_stream_profile_read_stages(self.handle, C.byref(ms), C.byref(n)))
        return {name: (ms[k], n[k]) for k, name in enumerate(self.STAGES)}

    def path_counters(self, reset: bool = False):
        """(reads resolved by the perfect-occurrence prefilter, by the seed-and-verify kernel,
        reads that ran the full-range automaton)."""
        a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
        _check(self.lib.bdx_stream_path_counters(self.handle, C.byref(a), C.byref(b), C.byref(c), int(reset)))
        return a.value, b.value, c.value

    def work_counters(self, reset: bool = False):
        """(prefilter reads, seed reads, automaton reads, verified hit-columns of k_seed_var, its input reads,
        q-mers probed by k_seed, hit-columns verified by k_seed, positions scanned by k_seed_var, diagonals its
        3-gram filter tested) -- include/bdx.h."""
        out = (C.c_int64 * 12)()
        _check(self.lib.bdx_stream_work_counters(self.handle, out, int(reset)))
        return tuple(int(x) for x in out)[:9]

    def demux_block(self, fastq1, fastq2=None, final_block: int = 1, mode: int = DEMUX_SINGLE):
        """bdx_demux_block over host uint8 arrays (or ``(device_ptr, length)`` pairs with
        DEMUX_DEVICE_IO).  Returns the raw ``DemuxOut``; host-mode helpers: ``demux_views``."""
        def ptr_len(x):
            if x is None:
                return None, 0
            if isinstance(x, tuple):
                return x[0], int(x[1])
            return (x.ctypes.data if x.size else None), int(x.size)
        p1, l1 = ptr_len(fastq1)
        p2, l2 = ptr_len(fastq2)
        out = DemuxOut()
        _check(self.lib.bdx_demux_block(self.handle, p1, l1, p2, l2, int(final_block), int(mode), C.byref(out)))
        return out

    @staticmethod
    def demux_views(out: "DemuxOut"):
        """numpy views (no copy; valid until the next demux_block) of a host-mode DemuxOut:
        (buckets, out1 bytes, out2 bytes, per-record results)."""
        def view(ptr, nbytes, dtype=np.uint8):
            if not ptr or nbytes == 0:
                return np.zeros(0, dtype)
            buf = (C.c_char * nbytes).from_address(ptr)
            return np.frombuffer(buf, dtype=dtype)
        buckets = view(out.buckets, out.n_buckets * BUCKET_DTYPE.itemsize, BUCKET_DTYPE)
        res = view(out.results, out.n_records * RESULT_DTYPE.itemsize, RESULT_DTYPE)
        return buckets, view(out.out1, out.out1_len), view(out.out2, out.out2_len), res

    def demux_stage_ms(self):
        ms = (C.c_float * 8)()
        _check(self.lib.bdx_demux_stage_ms(self.handle, C.byref(ms)))
        return list(ms)

    def stats(self) -> np.ndarray:
        out = np.zeros(self.config.layout.total_len, dtype=np.int64)
        _check(self.lib.bdx_stats_fetch(self.handle, out.ctypes.data, out.size))
        return out

    def stats_overflow(self) -> np.ndarray:
        """Exact records of the matched passes that did not fit the pos / len histograms."""
        n, lost = C.c_int64(), C.c_int64()
        _check(self.lib.bdx_stats_overflow_fetch(self.handle, None, 0, C.byref(n), C.byref(lost)))
        if lost.value:
            raise BdxError(BDX_ERR_TOO_LARGE, f"{lost.value} stats overflow records were lost")
        out = np.zeros(n.value, dtype=STATS_OVERFLOW_DTYPE)
        if n.value:
            _check(self.lib.bdx_stats_overflow_fetch(self.handle, out.ctypes.data, n.value, C.byref(n), C.byref(lost)))
        return out

    @property
    def stats_device_ptr(self) -> int:
        return int(self.lib.bdx_stats_device_ptr(self.handle) or 0)

    def stats_reset(self):
        _check(self.lib.bdx_stats_reset(self.handle))

    def close(self):
        if self.handle:
            self.lib.bdx_stream_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Pool:
    """``bdx_pool``: batches dealt round-robin to streams on several GPUs, results in submission order."""

    def __init__(self, config: Config, devices: Sequence[int], streams_per_device: int = 2, max_reads: int = 4000,
                 max_bytes: Optional[int] = None):
        self.lib, self.config = config.lib, config
        devs = (C.c_int * len(devices))(*devices)
        mb = int(max_bytes if max_bytes is not None else max(max_reads, 1) * 1024)
        self.handle = C.c_void_p()
        _check(self.lib.bdx_pool_create(config.handle, devs, len(devices), streams_per_device, max_reads, mb,
                                        C.byref(self.handle)))

    def submit(self, seq: np.ndarray, off: np.ndarray, tag: int = 0, pinned: bool = False):
        fn = self.lib.bdx_pool_submit_pinned if pinned else self.lib.bdx_pool_submit
        _check(fn(self.handle, seq.ctypes.data, off.ctypes.data, len(off) - 1, tag))

    def try_submit(self, seq, off, tag=0, pinned=False) -> bool:
        """False when the stream whose turn it is is full (fetch first)."""
        try:
            self.submit(seq, off, tag, pinned)
            return True
        except BdxError as e:
            if e.code == BDX_ERR_STATE:
                return False
            raise

    def fetch(self, copy: bool = True):
        """Oldest batch of the pool.  copy=False: a view into the owning stream's pinned result staging (valid
        until that stream has taken BDX_MAX_IN_FLIGHT - 1 further batches)."""
        tag, n = C.c_uint64(), C.c_int32()
        res_p, det_p = C.c_void_p(), C.c_void_p()
        _check(self.lib.bdx_pool_fetch_view(self.handle, C.byref(tag), C.byref(n), C.byref(res_p), C.byref(det_p)))
        if n.value == 0:
            return tag.value, np.zeros(0, RESULT_DTYPE)
        buf = (C.c_char * (n.value * RESULT_DTYPE.itemsize)).from_address(res_p.value)
        res = np.frombuffer(buf, dtype=RESULT_DTYPE, count=n.value)
        return tag.value, (res.copy() if copy else res)

    @property
    def in_flight(self) -> int:
        return int(self.lib.bdx_pool_in_flight(self.handle))

    def stats(self) -> np.ndarray:
        out = np.zeros(self.config.layout.total_len, dtype=np.int64)
        _check(self.lib.bdx_pool_stats_fetch(self.handle, out.ctypes.data, out.size))
        return out

    def close(self):
        if self.handle:
            self.lib.bdx_pool_destroy(self.handle)
            self.handle = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False


class Engine:
    """Config + one stream: what a single reference worker thread would own."""

    def __init__(self, cfg: DemuxConfig, device: int = 0, max_reads: int = 4000,
                 max_bytes: Optional[int] = None, want_stats: Optional[bool] = None, debug: int = 0,
                 windows: bool = False):
        """windows: classify_packed sends only the reads' search-window bytes (bdx_submit_windows)."""
        self.cfg = cfg
        self.windows = windows
        self.config = Config(cfg, want_stats=want_stats, debug=debug)
        self._device = device
        self.stream = Stream(self.config, device=device, max_reads=max_reads, max_bytes=max_bytes)

    def classify_reads(self, seqs: Sequence[bytes]) -> np.ndarray:
        blob, off = pack_reads(seqs)
        return self.classify_packed(blob, off)

    def classify_packed(self, blob: np.ndarray, off: np.ndarray, want_details: bool = False):
        """Any number of reads of any length (the reference has no limits either): the batch is split into
        sub-batches that fit the stream's staging buffers, and a single read longer than max_bytes makes the
        engine re-create its stream with larger buffers."""
        off = np.ascontiguousarray(off, dtype=np.int64)
        n = len(off) - 1
        st = self.stream
        lens = np.diff(off)
        if n and int(lens.max()) > st.max_bytes:
            new_bytes = max(2 * st.max_bytes, int(lens.max()))
            details, dev = st.details, self._device
            st.close()
            self.stream = st = Stream(self.config, device=dev, max_reads=st.max_reads, max_bytes=new_bytes)
            if details != st.details:
                st.enable_details(details)
        if n <= st.max_reads and (n == 0 or int(off[-1]) <= st.max_bytes):
            return self._classify(blob, off.astype(np.int32), want_details)
        res = np.zeros(n, RESULT_DTYPE)
        det = np.zeros((2, n), DETAIL_DTYPE) if want_details else None
        a = 0
        while a < n:
            # the longest run of reads from a that fits both limits
            b = min(n, a + st.max_reads)
            b = min(b, int(np.searchsorted(off, off[a] + st.max_bytes, side="right")) - 1)
            b = max(b, a + 1)
            out = self._classify(blob[off[a]:off[b]], (off[a:b + 1] - off[a]).astype(np.int32), want_details)
            if want_details:
                res[a:b], det[:, a:b] = out
            else:
                res[a:b] = out
            a = b
        return (res, det) if want_details else res

    def _classify(self, blob: np.ndarray, off: np.ndarray, want_details: bool):
        """One batch that fits the stream: the whole reads (bdx_classify), or their window bytes."""
        if not self.windows:
            return self.stream.classify(blob, off, want_details=want_details)
        win, win_off = self.config.window_reads(blob, off)
        self.stream.submit_windows(win, win_off, off)
        out = self.stream.fetch(want_details=want_details)
        return out[1:] if want_details else out[1]

    def demux_stats(self):
        from .stats import stats_from_counters
        return stats_from_counters(self.stream.stats(), self.config.layout, self.cfg, self.stream.stats_overflow())

    def close(self):
        self.stream.close()
        self.config.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False
