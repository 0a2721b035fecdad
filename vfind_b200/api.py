"""ctypes binding of include/vfind_b200.h and the Python mirror of `vfind.find_variants`.

The reference's boundary is the PyO3 function `find_variants`
(/root/reference/src/lib.rs:168-232): same names, positional order, defaults, coercions and
exception types here.  All compute happens in libvfind_b200.so (hand-written sm_100a CUDA);
there is no CPU path — importing works anywhere, calling needs a CUDA device and the
built library, and fails loudly otherwise.
"""
from __future__ import annotations

import ctypes as C
import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvfind_b200.so")

VFB_OK, VFB_ERR_VALUE, VFB_ERR_IO, VFB_ERR_FORMAT, VFB_ERR_CUDA, VFB_ERR_ARG, VFB_ERR_NOMEM = range(7)
NONE = 0xFFFFFFFF
INT32_MIN = -(2 ** 31)

SPAN_DTYPE = np.dtype([("off", "<u4"), ("len", "<u4")])
DIAG_DTYPE = np.dtype([("exact_prefix", "<i4"), ("exact_suffix", "<i4"),
                       ("score_prefix", "<i4"), ("len_prefix", "<i4"),
                       ("score_suffix", "<i4"), ("len_suffix", "<i4"),
                       ("start", "<i4"), ("end", "<i4")])


class Params(C.Structure):
    _fields_ = [("struct_size", C.c_uint32),
                ("prefix", C.c_char_p), ("prefix_len", C.c_uint64),
                ("suffix", C.c_char_p), ("suffix_len", C.c_uint64),
                ("match_score", C.c_int32), ("mismatch_score", C.c_int32),
                ("gap_open_penalty", C.c_int32), ("gap_extend_penalty", C.c_int32),
                ("accept_prefix_alignment", C.c_double), ("accept_suffix_alignment", C.c_double),
                ("n_threads", C.c_uint32), ("queue_len", C.c_uint64),
                ("skip_translation", C.c_int32), ("show_progress", C.c_int32),
                ("device", C.c_int32), ("diagnostics", C.c_int32),
                ("batch_reads", C.c_uint64), ("batch_bytes", C.c_uint64),
                ("table_capacity_hint", C.c_uint64),
                ("debug_hash_bits", C.c_int32), ("force_generic_dp", C.c_int32),
                ("dp_compute_all", C.c_int32), ("force_general_scan", C.c_int32),
                ("dp_mode", C.c_int32), ("debug_win_cap", C.c_int32), ("both_strands", C.c_int32),
                ("collapse_ratio", C.c_double)]


class Table(C.Structure):
    _fields_ = [("rows", C.c_uint64), ("key_bytes", C.c_uint64),
                ("offsets", C.POINTER(C.c_uint64)), ("data", C.POINTER(C.c_uint8)),
                ("counts", C.POINTER(C.c_uint64)), ("owner", C.c_void_p)]


class ArrowSchema(C.Structure):
    """struct ArrowSchema of the Arrow C Data Interface (72 bytes)."""
    _fields_ = [("format", C.c_char_p), ("name", C.c_char_p), ("metadata", C.c_char_p), ("flags", C.c_int64),
                ("n_children", C.c_int64), ("children", C.c_void_p), ("dictionary", C.c_void_p),
                ("release", C.c_void_p), ("private_data", C.c_void_p)]


class ArrowArray(C.Structure):
    """struct ArrowArray of the Arrow C Data Interface (80 bytes)."""
    _fields_ = [("length", C.c_int64), ("null_count", C.c_int64), ("offset", C.c_int64), ("n_buffers", C.c_int64),
                ("n_children", C.c_int64), ("buffers", C.c_void_p), ("children", C.c_void_p),
                ("dictionary", C.c_void_p), ("release", C.c_void_p), ("private_data", C.c_void_p)]


PROGRESS_FN = C.CFUNCTYPE(None, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p)


class Stats(C.Structure):
    _fields_ = [("reads", C.c_uint64), ("dp_prefix", C.c_uint64), ("dp_suffix", C.c_uint64),
                ("dp_cells", C.c_uint64), ("counted", C.c_uint64), ("unique", C.c_uint64),
                ("text_bytes", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("ms_scan", C.c_double), ("ms_worklist", C.c_double), ("ms_dp", C.c_double),
                ("ms_translate", C.c_double), ("ms_count", C.c_double), ("ms_total", C.c_double),
                ("dp_kernel_launches", C.c_uint64), ("dp_kernel_kind", C.c_int32),
                ("reserved", C.c_int32), ("dp_cells_computed", C.c_uint64), ("dp_windows", C.c_uint64),
                ("ms_dp_filter", C.c_double), ("ms_dp_window", C.c_double),
                ("fused_batches", C.c_uint64), ("fused_hits", C.c_uint64),
                ("reverse_reads", C.c_uint64), ("reverse_counted", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class CollapseInfo(C.Structure):
    _fields_ = [("rows_in", C.c_uint64), ("rows_out", C.c_uint64), ("ms", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class UmiInfo(C.Structure):
    _fields_ = [("pairs", C.c_uint64), ("rows_out", C.c_uint64), ("reads_short", C.c_uint64), ("ms", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class SynthCfg(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("read_len", C.c_uint32), ("adapter_len", C.c_uint32),
                ("region_len", C.c_uint32), ("n_variants", C.c_uint32), ("zipf", C.c_uint32),
                ("p_err_ppm", C.c_uint32), ("indel_ppm", C.c_uint32), ("force_indel", C.c_uint32),
                ("frameshift_ppm", C.c_uint32), ("noise_ppm", C.c_uint32), ("n_ppm", C.c_uint32),
                ("reserved", C.c_uint32)]


_lib = None


def load_library():
    """Load the CUDA library.  Raises (never falls back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "vfind_b200: %s is missing — build it with `python -m vfind_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    L.vfb_last_error.restype = C.c_char_p
    L.vfb_abi_version.restype = i32
    L.vfb_default_params.argtypes = [C.POINTER(Params)]
    L.vfb_default_params.restype = None
    L.vfb_create.argtypes = [C.POINTER(Params), C.POINTER(vp)]
    L.vfb_destroy.argtypes = [vp]
    L.vfb_reset.argtypes = [vp]
    L.vfb_set_profiling.argtypes = [vp, i32]
    L.vfb_submit_host.argtypes = [vp, vp, u64, vp, u64]
    L.vfb_submit_device.argtypes = [vp, vp, u64, vp, u64]
    L.vfb_run_file.argtypes = [vp, C.c_char_p, C.POINTER(u64)]
    L.vfb_sync.argtypes = [vp]
    L.vfb_set_compute_stream.argtypes = [vp, vp]
    L.vfb_fence.argtypes = [vp]
    L.vfb_set_lanes.argtypes = [vp, i32]
    L.vfb_finish.argtypes = [vp, C.POINTER(Table)]
    L.vfb_table_free.argtypes = [C.POINTER(Table)]
    L.vfb_table_free.restype = None
    L.vfb_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.vfb_get_diag.argtypes = [vp, vp, u64]
    L.vfb_get_diag_reverse.argtypes = [vp, vp, u64]
    L.vfb_debug_revcomp.argtypes = [C.c_char_p, u64, vp]
    L.vfb_table_partition_sizes.argtypes = [vp, u32, C.POINTER(u64)]
    L.vfb_table_partition_fill.argtypes = [vp, u32, vp, C.POINTER(u64)]
    L.vfb_table_clear.argtypes = [vp]
    L.vfb_table_absorb.argtypes = [vp, vp, u64]
    L.vfb_chunk_rows.argtypes = [vp, u64, C.POINTER(u64)]
    L.vfb_hash_key.argtypes = [C.c_char_p, u32]
    L.vfb_hash_key.restype = u64
    L.vfb_key_owner.argtypes = [u64, u32]
    L.vfb_key_owner.restype = u32
    L.vfb_synth_adapters.argtypes = [C.POINTER(SynthCfg), vp, vp]
    L.vfb_synth_host.argtypes = [C.POINTER(SynthCfg), u64, u64, vp, vp]
    L.vfb_synth_device.argtypes = [C.POINTER(SynthCfg), u64, u64, vp, vp, i32]
    L.vfb_measure_int_peak.argtypes = [i32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.vfb_host_alloc.argtypes = [C.POINTER(vp), u64]
    L.vfb_host_free.argtypes = [vp]
    L.vfb_finish_arrow.argtypes = [vp, vp, vp]
    L.vfb_run_file_ex.argtypes = [vp, C.c_char_p, u32, C.POINTER(u64)]
    L.vfb_set_progress.argtypes = [vp, vp, vp]
    L.vfb_pinned_pool_trim.argtypes = []
    L.vfb_device_pool_trim.argtypes = []
    L.vfb_multi_create.argtypes = [C.POINTER(Params), C.POINTER(C.c_int32), u32, C.POINTER(vp)]
    L.vfb_multi_destroy.argtypes = [vp]
    L.vfb_multi_devices.argtypes = [vp]
    L.vfb_multi_devices.restype = u32
    L.vfb_multi_ctx.argtypes = [vp, u32]
    L.vfb_multi_ctx.restype = vp
    L.vfb_multi_run_file.argtypes = [vp, C.c_char_p, u32, C.POINTER(u64)]
    L.vfb_multi_set_progress.argtypes = [vp, vp, vp]
    L.vfb_multi_sync.argtypes = [vp]
    L.vfb_multi_reset.argtypes = [vp]
    L.vfb_multi_merge.argtypes = [vp]
    L.vfb_multi_finish.argtypes = [vp, C.POINTER(Table)]
    L.vfb_multi_finish_arrow.argtypes = [vp, vp, vp]
    L.vfb_multi_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.vfb_get_collapse_info.argtypes = [vp, C.POINTER(CollapseInfo)]
    L.vfb_multi_get_collapse_info.argtypes = [vp, C.POINTER(CollapseInfo)]
    L.vfb_collapse.argtypes = [C.POINTER(Table), C.c_double, i32, i32, C.POINTER(Table), C.POINTER(CollapseInfo)]
    L.vfb_set_umi.argtypes = [vp, u32, u32]
    L.vfb_multi_set_umi.argtypes = [vp, u32, u32]
    L.vfb_get_umi_info.argtypes = [vp, C.POINTER(UmiInfo)]
    L.vfb_multi_get_umi_info.argtypes = [vp, C.POINTER(UmiInfo)]
    L.vfb_get_molecules.argtypes = [vp, C.POINTER(C.POINTER(C.c_uint64))]
    L.vfb_multi_get_molecules.argtypes = [vp, C.POINTER(C.POINTER(C.c_uint64))]
    L.vfb_nccl_available.restype = i32
    L.vfb_nccl_unique_id.argtypes = [vp]
    L.vfb_nccl_comm_init.argtypes = [vp, u32, u32, i32, C.POINTER(vp)]
    L.vfb_nccl_comm_destroy.argtypes = [vp]
    L.vfb_merge_nccl.argtypes = [vp, vp, u32, u32]
    _lib = L
    return L


class PanicException(RuntimeError):
    """Where the reference panics (malformed gzip/FASTQ, src/lib.rs:308) this build raises
    a RuntimeError subclass named after pyo3_runtime.PanicException."""


def _check(rc: int):
    if rc == VFB_OK:
        return
    msg = load_library().vfb_last_error().decode("utf-8", "replace")
    if rc == VFB_ERR_VALUE:
        raise ValueError(msg)
    if rc == VFB_ERR_IO:
        if "No such file" in msg:
            raise FileNotFoundError(msg)
        raise OSError(msg)
    if rc == VFB_ERR_FORMAT:
        raise PanicException(msg)
    if rc == VFB_ERR_NOMEM:
        raise MemoryError(msg)
    raise RuntimeError(msg)


def _as_bytes(s, what):
    if isinstance(s, str):
        return s.encode("utf-8")
    if isinstance(s, (bytes, bytearray)):
        return bytes(s)
    raise TypeError("%s must be str" % what)


def _make_params(L, adapters, match_score, mismatch_score, gap_open_penalty, gap_extend_penalty,
                 accept_prefix_alignment, accept_suffix_alignment, n_threads, queue_len, skip_translation,
                 show_progress, device, diagnostics, batch_reads, batch_bytes, table_capacity_hint,
                 debug_hash_bits, force_generic_dp, dp_compute_all, force_general_scan, dp_mode, debug_win_cap,
                 both_strands=False, collapse_ratio=None):
    p = Params()
    L.vfb_default_params(C.byref(p))
    pre = _as_bytes(adapters[0], "adapters[0]")
    suf = _as_bytes(adapters[1], "adapters[1]")
    p.prefix, p.prefix_len = pre, len(pre)
    p.suffix, p.suffix_len = suf, len(suf)
    p.match_score, p.mismatch_score = match_score, mismatch_score
    p.gap_open_penalty, p.gap_extend_penalty = gap_open_penalty, gap_extend_penalty
    p.accept_prefix_alignment = accept_prefix_alignment
    p.accept_suffix_alignment = accept_suffix_alignment
    p.n_threads, p.queue_len = n_threads, queue_len
    p.skip_translation = 1 if skip_translation else 0
    p.show_progress = 1 if show_progress else 0
    p.device = -1 if device is None else int(device)
    p.diagnostics = 1 if diagnostics else 0
    p.batch_reads, p.batch_bytes = int(batch_reads), int(batch_bytes)
    p.table_capacity_hint = int(table_capacity_hint)
    p.debug_hash_bits = int(debug_hash_bits)
    p.force_generic_dp = 1 if force_generic_dp else 0
    p.dp_compute_all = 1 if dp_compute_all else 0
    p.force_general_scan = 1 if force_general_scan else 0
    p.dp_mode = int(dp_mode)
    p.debug_win_cap = int(debug_win_cap)
    p.both_strands = 1 if both_strands else 0
    p.collapse_ratio = collapse_ratio or 0.0          # validated by the callers
    return p, pre, suf          # the byte strings must outlive the call that reads p


class Context:
    """One configured variant-recovery pipeline on one GPU (vfb_ctx)."""

    def __init__(self, adapters, match_score=3, mismatch_score=-2, gap_open_penalty=5,
                 gap_extend_penalty=2, accept_prefix_alignment=0.75, accept_suffix_alignment=0.75,
                 n_threads=3, queue_len=2, skip_translation=False, show_progress=True, *,
                 device=None, diagnostics=False, batch_reads=0, batch_bytes=0,
                 table_capacity_hint=0, debug_hash_bits=0, force_generic_dp=False,
                 dp_compute_all=False, force_general_scan=False, dp_mode=0, debug_win_cap=0, both_strands=False,
                 collapse_ratio=None, umi_length=None, umi_offset=0):
        """both_strands: a read without a region is searched once more as its reverse complement, on the device, and
        a region found there is counted in the same table (a read counts on at most one strand).
        collapse_ratio: every finish folds sequencing-error keys into their more abundant neighbours first (see
        collapse_variants); the count table keeps every key, so further reads and another finish collapse them all.
        umi_length / umi_offset: count distinct UMIs per variant (see find_variants); molecules() gives the column of
        the last finish, finish_arrow() returns it as a third column."""
        collapse_ratio = _ratio_arg(collapse_ratio, "collapse_ratio", True) or None
        umi = _umi_args(umi_length, umi_offset, collapse_ratio)
        L = load_library()
        self._lib = L
        self._h = C.c_void_p()
        self._owned = True
        p, self._pre, self._suf = _make_params(L, adapters, match_score, mismatch_score, gap_open_penalty,
                                               gap_extend_penalty, accept_prefix_alignment, accept_suffix_alignment,
                                               n_threads, queue_len, skip_translation, show_progress, device,
                                               diagnostics, batch_reads, batch_bytes, table_capacity_hint,
                                               debug_hash_bits, force_generic_dp, dp_compute_all, force_general_scan,
                                               dp_mode, debug_win_cap, both_strands, collapse_ratio)
        _check(L.vfb_create(C.byref(p), C.byref(self._h)))
        if umi[1]:
            _check(L.vfb_set_umi(self._h, umi[0], umi[1]))

    @classmethod
    def _borrowed(cls, lib, handle):
        """A view of a context owned by a MultiContext (not destroyed on close)."""
        self = cls.__new__(cls)
        self._lib, self._h, self._owned = lib, C.c_void_p(handle), False
        return self

    # -- lifetime
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            if self._owned:
                self._lib.vfb_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- the hot loop
    def submit_host(self, text, spans):
        """text: uint8 array / bytes; spans: SPAN_DTYPE array or (n,2) uint32."""
        text = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray)) else text
        assert text.dtype == np.uint8 and text.flags.c_contiguous
        spans = np.ascontiguousarray(spans)
        n = spans.shape[0]
        assert spans.nbytes == n * 8
        _check(self._lib.vfb_submit_host(self._h, text.ctypes.data if text.size else None, text.size,
                                         spans.ctypes.data if n else None, n))

    def submit_host_ptr(self, text_ptr, text_bytes, spans_ptr, n):
        _check(self._lib.vfb_submit_host(self._h, text_ptr, text_bytes, spans_ptr, n))

    def submit_device(self, text_ptr, text_bytes, spans_ptr, n):
        _check(self._lib.vfb_submit_device(self._h, text_ptr, text_bytes, spans_ptr, n))

    def run_file(self, path, allow_text=False) -> int:
        """Ingest one FASTQ file; the table accumulates over calls.  allow_text: a file without the gzip
        magic is read as uncompressed text instead of failing like the reference."""
        n = C.c_uint64(0)
        _check(self._lib.vfb_run_file_ex(self._h, os.fsencode(path), 1 if allow_text else 0, C.byref(n)))
        return int(n.value)

    def sync(self):
        _check(self._lib.vfb_sync(self._h))

    def reset(self):
        _check(self._lib.vfb_reset(self._h))

    def set_compute_stream(self, stream_ptr: int):
        _check(self._lib.vfb_set_compute_stream(self._h, stream_ptr))

    def fence(self):
        """The compute stream waits (on the device) for everything submitted so far: call before recording your own
        events or queueing your own consumers on it."""
        _check(self._lib.vfb_fence(self._h))

    def set_lanes(self, n: int):
        """1 = every batch on the compute stream itself (per-stage profiling), 2 = two overlapping lanes (default)."""
        _check(self._lib.vfb_set_lanes(self._h, n))

    def set_progress(self, fn):
        """fn(records, bytes_done, bytes_total) is called from run_file about ten times per second and once at
        the end (None removes it)."""
        if fn is None:
            self._progress_cb = None
            _check(self._lib.vfb_set_progress(self._h, None, None))
            return
        self._progress_cb = PROGRESS_FN(lambda r, d, t, _u: fn(int(r), int(d), int(t)))
        _check(self._lib.vfb_set_progress(self._h, C.cast(self._progress_cb, C.c_void_p), None))

    def set_profiling(self, on: bool):
        _check(self._lib.vfb_set_profiling(self._h, 1 if on else 0))

    def stats(self) -> dict:
        s = Stats()
        _check(self._lib.vfb_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    def collapse_info(self) -> dict:
        """What the last collapsing finish did: rows_in (keys with a count), rows_out (roots), ms (elapsed time of
        the collapse on the device stream)."""
        s = CollapseInfo()
        _check(self._lib.vfb_get_collapse_info(self._h, C.byref(s)))
        return s.as_dict()

    def umi_info(self) -> dict:
        """umi_length: pairs ((variant, UMI) rows grouped by the last finish), rows_out (variant rows it returned),
        reads_short (reads not counted because they are shorter than umi_offset + umi_length, since creation or reset)
        and ms (device time of the group-by)."""
        s = UmiInfo()
        _check(self._lib.vfb_get_umi_info(self._h, C.byref(s)))
        return s.as_dict()

    def molecules(self):
        """umi_length: the molecules column (uint64) of the last finish_arrays / finish_dict, aligned with its rows."""
        return _molecules(self._lib.vfb_get_molecules, self._h, getattr(self, "_rows", 0))

    def diag(self, n):
        out = np.zeros(n, dtype=DIAG_DTYPE)
        _check(self._lib.vfb_get_diag(self._h, out.ctypes.data, n))
        return out

    def diag_reverse(self, n):
        """both_strands: diagnostics of the reverse-complement pass over the last batch, in read order; rows of reads
        that were not retried hold the absent markers (-1, INT32_MIN for scores)."""
        out = np.zeros(n, dtype=DIAG_DTYPE)
        _check(self._lib.vfb_get_diag_reverse(self._h, out.ctypes.data, n))
        return out

    # -- results
    def finish_arrays(self, copy=True):
        """(offsets uint64[rows+1], data uint8[key_bytes], counts uint64[rows]) on the host.

        copy=False returns views of the context's pinned buffers: valid only until the next
        finish on this context or its close()."""
        t = Table()
        _check(self._lib.vfb_finish(self._h, C.byref(t)))
        self._rows = int(t.rows)
        return _table_views(self._lib, t, copy)

    def finish_arrow(self):
        """The table as a pyarrow.RecordBatch {sequence: large_string, count: uint64} imported through the
        Arrow C Data Interface: its buffers are the pinned host columns the device wrote, nothing is copied.
        The batch owns them (they return to the pinned pool when it is garbage-collected) and outlives
        this context."""
        import pyarrow as pa
        arr, sch = ArrowArray(), ArrowSchema()
        _check(self._lib.vfb_finish_arrow(self._h, C.byref(arr), C.byref(sch)))
        return pa.RecordBatch._import_from_c(C.addressof(arr), C.addressof(sch))

    def finish_dict(self) -> dict:
        offsets, data, counts = self.finish_arrays()
        raw = data.tobytes()
        return {raw[int(offsets[i]):int(offsets[i + 1])]: int(counts[i]) for i in range(len(counts))}

    # -- multi-GPU merge plumbing (see vfind_b200/distributed.py)
    def partition_sizes(self, n_parts: int):
        out = (C.c_uint64 * n_parts)()
        _check(self._lib.vfb_table_partition_sizes(self._h, n_parts, out))
        return [int(x) for x in out]

    def partition_fill(self, n_parts: int, buf_ptr: int, offsets):
        arr = (C.c_uint64 * n_parts)(*[int(o) for o in offsets])
        _check(self._lib.vfb_table_partition_fill(self._h, n_parts, buf_ptr, arr))

    def table_clear(self):
        _check(self._lib.vfb_table_clear(self._h))

    def absorb(self, chunk_ptr: int, chunk_bytes: int):
        _check(self._lib.vfb_table_absorb(self._h, chunk_ptr, chunk_bytes))

    def merge_nccl(self, comm, rank: int, n_ranks: int):
        """Keep-own-keys merge over NCCL send/recv inside the library (one process per GPU); `comm` from
        nccl_comm_init.  Afterwards this context holds exactly the keys it owns, with global counts."""
        _check(self._lib.vfb_merge_nccl(self._h, comm, rank, n_ranks))


def _molecules(getter, h, rows):
    col = C.POINTER(C.c_uint64)()
    _check(getter(h, C.byref(col)))
    return np.ctypeslib.as_array(col, shape=(rows,)).copy() if rows else np.zeros(0, np.uint64)


def _table_views(lib, t, copy):
    try:
        rows, kb = int(t.rows), int(t.key_bytes)
        offsets = np.ctypeslib.as_array(t.offsets, shape=(rows + 1,))
        data = np.ctypeslib.as_array(t.data, shape=(kb,)) if kb else np.zeros(0, np.uint8)
        counts = np.ctypeslib.as_array(t.counts, shape=(rows,)) if rows else np.zeros(0, np.uint64)
        if copy:
            offsets, data, counts = offsets.copy(), data.copy(), counts.copy()
    finally:
        lib.vfb_table_free(C.byref(t))
    return offsets, data, counts


class MultiContext:
    """One pipeline per GPU behind one handle (vfb_multi): one process drives `devices` (None = all visible).
    run_file deals the file's segments round robin; finish_* merge the per-device tables over peer copies
    (NVLink) and return ONE table.  `contexts` are the per-device Context views (submit_host / submit_device)."""

    def __init__(self, adapters, match_score=3, mismatch_score=-2, gap_open_penalty=5,
                 gap_extend_penalty=2, accept_prefix_alignment=0.75, accept_suffix_alignment=0.75,
                 n_threads=3, queue_len=2, skip_translation=False, show_progress=True, *,
                 devices=None, batch_reads=0, batch_bytes=0, table_capacity_hint=0, debug_hash_bits=0, dp_mode=0,
                 both_strands=False, collapse_ratio=None, umi_length=None, umi_offset=0):
        collapse_ratio = _ratio_arg(collapse_ratio, "collapse_ratio", True) or None
        umi = _umi_args(umi_length, umi_offset, collapse_ratio)
        L = load_library()
        self._lib = L
        self._h = C.c_void_p()
        p, self._pre, self._suf = _make_params(L, adapters, match_score, mismatch_score, gap_open_penalty,
                                               gap_extend_penalty, accept_prefix_alignment, accept_suffix_alignment,
                                               n_threads, queue_len, skip_translation, show_progress, None, False,
                                               batch_reads, batch_bytes, table_capacity_hint, debug_hash_bits,
                                               False, False, False, dp_mode, 0, both_strands, collapse_ratio)
        if devices is None:
            _check(L.vfb_multi_create(C.byref(p), None, 0, C.byref(self._h)))
        else:
            devs = [int(d) for d in devices]
            arr = (C.c_int32 * len(devs))(*devs)
            if not devs:
                raise ValueError("devices must not be empty")
            _check(L.vfb_multi_create(C.byref(p), arr, len(devs), C.byref(self._h)))
        if umi[1]:
            _check(L.vfb_multi_set_umi(self._h, umi[0], umi[1]))
        self.n_devices = int(L.vfb_multi_devices(self._h))
        self.contexts = [Context._borrowed(L, L.vfb_multi_ctx(self._h, i)) for i in range(self.n_devices)]

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            for c in self.contexts:
                c.close()
            self._lib.vfb_multi_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run_file(self, path, allow_text=False) -> int:
        n = C.c_uint64(0)
        _check(self._lib.vfb_multi_run_file(self._h, os.fsencode(path), 1 if allow_text else 0, C.byref(n)))
        return int(n.value)

    def set_progress(self, fn):
        if fn is None:
            self._progress_cb = None
            _check(self._lib.vfb_multi_set_progress(self._h, None, None))
            return
        self._progress_cb = PROGRESS_FN(lambda r, d, t, _u: fn(int(r), int(d), int(t)))
        _check(self._lib.vfb_multi_set_progress(self._h, C.cast(self._progress_cb, C.c_void_p), None))

    def sync(self):
        _check(self._lib.vfb_multi_sync(self._h))

    def reset(self):
        _check(self._lib.vfb_multi_reset(self._h))

    def merge(self):
        _check(self._lib.vfb_multi_merge(self._h))

    def stats(self) -> dict:
        s = Stats()
        _check(self._lib.vfb_multi_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    def collapse_info(self) -> dict:
        """The collapse of the merged table by the last finish (collapse_ratio)."""
        s = CollapseInfo()
        _check(self._lib.vfb_multi_get_collapse_info(self._h, C.byref(s)))
        return s.as_dict()

    def umi_info(self) -> dict:
        """Context.umi_info summed over the devices (ms: the slowest device's group-by)."""
        s = UmiInfo()
        _check(self._lib.vfb_multi_get_umi_info(self._h, C.byref(s)))
        return s.as_dict()

    def molecules(self):
        return _molecules(self._lib.vfb_multi_get_molecules, self._h, getattr(self, "_rows", 0))

    def finish_arrays(self, copy=True):
        t = Table()
        _check(self._lib.vfb_multi_finish(self._h, C.byref(t)))
        self._rows = int(t.rows)
        return _table_views(self._lib, t, copy)

    def finish_dict(self) -> dict:
        offsets, data, counts = self.finish_arrays()
        raw = data.tobytes()
        return {raw[int(offsets[i]):int(offsets[i + 1])]: int(counts[i]) for i in range(len(counts))}

    def finish_arrow(self):
        import pyarrow as pa
        arr, sch = ArrowArray(), ArrowSchema()
        _check(self._lib.vfb_multi_finish_arrow(self._h, C.byref(arr), C.byref(sch)))
        return pa.RecordBatch._import_from_c(C.addressof(arr), C.addressof(sch))


def nccl_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    _check(load_library().vfb_nccl_unique_id(buf))
    return buf.raw


def nccl_comm_init(unique_id: bytes, n_ranks: int, rank: int, device: int = -1):
    comm = C.c_void_p()
    _check(load_library().vfb_nccl_comm_init(unique_id, n_ranks, rank, device, C.byref(comm)))
    return comm


def nccl_comm_destroy(comm):
    _check(load_library().vfb_nccl_comm_destroy(comm))


def batch_to_frame(batch):
    """pyarrow.RecordBatch -> polars.DataFrame when polars is importable (zero-copy: polars' String is
    large_utf8), else a pyarrow.Table with columns `sequence` and `count` (src/lib.rs:312-317)."""
    import pyarrow as pa
    tbl = pa.Table.from_batches([batch])
    try:
        import polars as pl
    except ImportError:
        return tbl
    return pl.from_arrow(tbl)


def table_to_frame(offsets, data, counts):
    """Columns `sequence` (String) and `count` (UInt64) (src/lib.rs:312-317) as a
    polars.DataFrame when polars is importable, else a pyarrow.Table with the same schema."""
    import pyarrow as pa
    rows = len(counts)
    if rows and int(offsets[-1]) >= 2 ** 31:
        seq = pa.Array.from_buffers(pa.large_string(), rows,
                                    [None, pa.py_buffer(offsets.astype(np.int64)), pa.py_buffer(data)])
    else:
        seq = pa.Array.from_buffers(pa.string(), rows,
                                    [None, pa.py_buffer(offsets.astype(np.int32)), pa.py_buffer(data)])
    cnt = pa.array(counts, type=pa.uint64())
    tbl = pa.table({"sequence": seq, "count": cnt})
    try:
        import polars as pl
    except ImportError:
        return tbl
    return pl.from_arrow(tbl)


def _int_arg(v, name, lo, hi):
    if isinstance(v, bool) or not hasattr(v, "__index__"):
        if isinstance(v, bool):
            v = int(v)
        else:
            raise TypeError("argument '%s': '%s' object cannot be interpreted as an integer"
                            % (name, type(v).__name__))
    v = v.__index__()
    if v < lo or v > hi:
        raise OverflowError("argument '%s': out of range integral type conversion attempted" % name)
    return v


def _float_arg(v, name):
    if isinstance(v, (int, float, np.floating, np.integer)) and not isinstance(v, bool):
        return float(v)
    if isinstance(v, bool):
        return float(v)
    raise TypeError("argument '%s': must be real number, not %s" % (name, type(v).__name__))


def _ratio_arg(v, name, optional):
    """collapse_ratio: None (off, where optional) -> 0.0; else a finite real >= 1."""
    if v is None and optional:
        return 0.0
    if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, float, np.floating, np.integer)):
        raise TypeError("argument '%s': must be real number, not %s" % (name, type(v).__name__))
    r = float(v)
    if not (r >= 1.0 and r != float("inf")):
        raise ValueError("argument '%s': must be a finite number >= 1, got %r" % (name, v))
    return r


def _umi_args(umi_length, umi_offset, collapse_ratio):
    """(offset, length) for vfb_set_umi; (0, 0) = off.  Checked before any file is opened or device is used."""
    if umi_length is None:
        if umi_offset is not None and _int_arg(umi_offset, "umi_offset", 0, 2 ** 32 - 1):
            raise ValueError("argument 'umi_offset': needs umi_length")
        return 0, 0
    k = _int_arg(umi_length, "umi_length", -(2 ** 63), 2 ** 63 - 1)
    o = _int_arg(umi_offset, "umi_offset", -(2 ** 63), 2 ** 63 - 1)
    if not 1 <= k <= 64:
        raise ValueError("argument 'umi_length': must be between 1 and 64, got %d" % k)
    if o < 0 or o + k > 65536:
        raise ValueError("argument 'umi_offset': must be >= 0 with umi_offset + umi_length <= 65536, got %d" % o)
    if collapse_ratio:
        raise ValueError("umi_length cannot be combined with collapse_ratio")
    return o, k


def _bool_arg(v, name):
    if isinstance(v, (bool, np.bool_)):
        return bool(v)
    raise TypeError("argument '%s': '%s' object cannot be converted to 'PyBool'" % (name, type(v).__name__))


def find_variants(fq_path, adapters, match_score=3, mismatch_score=-2, gap_open_penalty=5,
                  gap_extend_penalty=2, accept_prefix_alignment=0.75, accept_suffix_alignment=0.75,
                  n_threads=3, queue_len=2, skip_translation=False, show_progress=True, *,
                  device=None, devices=None, batch_reads=0, table_capacity_hint=0, progress=None, allow_text=False,
                  both_strands=False, collapse_ratio=None, umi_length=None, umi_offset=0):
    """Find variable regions flanked by adapters in a gzipped FASTQ dataset.

    Drop-in for `vfind.find_variants` (/root/reference/src/lib.rs:168-232): same positional
    order, defaults and error behaviour; the work runs on a B200.

    Returns a table with columns `sequence` (string) and `count` (uint64): a
    polars.DataFrame when polars is installed, else a pyarrow.Table.  Row order is
    unspecified (as in the reference, src/lib.rs:312).

    Extra keyword-only arguments: device (one CUDA ordinal) or devices (a list of ordinals, or "all": one
    process drives them all, the file's segments are dealt round robin and the per-GPU tables are merged over
    NVLink inside the library; default: every visible GPU that gets at least 64 MB of the compressed input —
    VFB_DEVICES=n caps it), batch_reads, table_capacity_hint,
    progress (callable(records, bytes_done, bytes_total), called about ten times per second),
    allow_text (read a file without the gzip magic as uncompressed FASTQ; the reference panics on it),
    both_strands (a read in which no region is found is searched once more as its reverse complement, on the GPU, and
    counted in the same table: for libraries sequenced from both ends; a read counts on at most one strand),
    collapse_ratio (a real >= 1: fold sequencing-error variants into a more abundant variant of the same length one
    substitution away, on the GPU before the table leaves it; see collapse_variants — not for libraries whose members
    are themselves one substitution apart),
    umi_length / umi_offset (an integer 1..64 and an offset >= 0: bytes [umi_offset, umi_offset + umi_length) of each
    counted read, in the orientation its region was found in, are its UMI; the result gains a column `molecules` = the
    number of distinct UMIs among the variant's reads.  UMIs are compared as raw bytes with no error correction, so a
    UMI with a sequencing error counts as one more molecule.  A read shorter than umi_offset + umi_length is not
    counted.  Cannot be combined with collapse_ratio).
    With show_progress (the default) and a terminal on stderr a one-line progress display is shown
    and cleared at the end, like the reference's spinner (src/lib.rs:265-269, :310).
    """
    if isinstance(fq_path, os.PathLike):
        fq_path = os.fspath(fq_path)
    if not isinstance(fq_path, str):
        raise TypeError("argument 'fq_path': '%s' object cannot be converted to 'PyString'"
                        % type(fq_path).__name__)
    return _find_variants([fq_path], adapters, match_score, mismatch_score, gap_open_penalty, gap_extend_penalty,
                          accept_prefix_alignment, accept_suffix_alignment, n_threads, queue_len, skip_translation,
                          show_progress, device, devices, batch_reads, table_capacity_hint, progress, allow_text,
                          both_strands, collapse_ratio, umi_length, umi_offset)


def find_variants_multi(fq_paths, adapters, match_score=3, mismatch_score=-2, gap_open_penalty=5,
                        gap_extend_penalty=2, accept_prefix_alignment=0.75, accept_suffix_alignment=0.75,
                        n_threads=3, queue_len=2, skip_translation=False, show_progress=True, *,
                        device=None, devices=None, batch_reads=0, table_capacity_hint=0, progress=None, allow_text=False,
                        both_strands=False, collapse_ratio=None, umi_length=None, umi_offset=0):
    """find_variants over several FASTQ files (lanes, split runs) counted into ONE table, on one context
    (SURVEY §8(f) next-4).  Same arguments as find_variants; fq_paths is a non-empty sequence of paths."""
    if isinstance(fq_paths, (str, bytes, os.PathLike)) or not hasattr(fq_paths, "__iter__"):
        raise TypeError("argument 'fq_paths': expected a sequence of paths")
    paths = [os.fspath(p) if isinstance(p, os.PathLike) else p for p in fq_paths]
    if not paths or not all(isinstance(p, str) for p in paths):
        raise TypeError("argument 'fq_paths': expected a non-empty sequence of str / os.PathLike")
    return _find_variants(paths, adapters, match_score, mismatch_score, gap_open_penalty, gap_extend_penalty,
                          accept_prefix_alignment, accept_suffix_alignment, n_threads, queue_len, skip_translation,
                          show_progress, device, devices, batch_reads, table_capacity_hint, progress, allow_text,
                          both_strands, collapse_ratio, umi_length, umi_offset)


def _find_variants(paths, adapters, match_score, mismatch_score, gap_open_penalty, gap_extend_penalty,
                   accept_prefix_alignment, accept_suffix_alignment, n_threads, queue_len, skip_translation,
                   show_progress, device, devices, batch_reads, table_capacity_hint, progress, allow_text, both_strands,
                   collapse_ratio, umi_length=None, umi_offset=0):
    if not isinstance(adapters, (tuple, list)):
        raise TypeError("argument 'adapters': '%s' object cannot be converted to 'PyTuple'"
                        % type(adapters).__name__)
    if len(adapters) != 2:
        raise ValueError("argument 'adapters': expected tuple of length 2, but got tuple of length %d"
                         % len(adapters))
    for a in adapters:
        if not isinstance(a, str):
            raise TypeError("argument 'adapters': '%s' object cannot be converted to 'PyString'"
                            % type(a).__name__)
    i32 = (-(2 ** 31), 2 ** 31 - 1)
    match_score = _int_arg(match_score, "match_score", *i32)
    mismatch_score = _int_arg(mismatch_score, "mismatch_score", *i32)
    gap_open_penalty = _int_arg(gap_open_penalty, "gap_open_penalty", *i32)
    gap_extend_penalty = _int_arg(gap_extend_penalty, "gap_extend_penalty", *i32)
    accept_prefix_alignment = _float_arg(accept_prefix_alignment, "accept_prefix_alignment")
    accept_suffix_alignment = _float_arg(accept_suffix_alignment, "accept_suffix_alignment")
    n_threads = _int_arg(n_threads, "n_threads", 0, 2 ** 32 - 1)
    queue_len = _int_arg(queue_len, "queue_len", 0, 2 ** 64 - 1)
    skip_translation = _bool_arg(skip_translation, "skip_translation")
    show_progress = _bool_arg(show_progress, "show_progress")
    both_strands = _bool_arg(both_strands, "both_strands")
    collapse_ratio = _ratio_arg(collapse_ratio, "collapse_ratio", True) or None
    umi_offset, umi_length = _umi_args(umi_length, umi_offset, collapse_ratio)
    umi_length = umi_length or None

    # The reference opens the file before validating thresholds (src/lib.rs:233 vs :239).
    for p in paths:
        with open(p, "rb"):
            pass
    devs = _pick_devices(device, devices, paths)
    if not table_capacity_hint:
        # a count table that starts near its final size never has to grow in the middle of the run (a rehash stalls the
        # pipeline): about one distinct variant per 512 compressed bytes per device covers the BASELINE shapes; the table
        # still grows by itself when that is not enough.  Small inputs keep the library's default (2 M rows).
        total = sum(os.path.getsize(p) for p in paths)
        guess = total // (512 * len(devs))
        if guess > (2 << 20):
            table_capacity_hint = int(min(guess, 48 << 20))
    if len(devs) == 1:
        ctx = Context(adapters, match_score, mismatch_score, gap_open_penalty, gap_extend_penalty,
                      accept_prefix_alignment, accept_suffix_alignment, n_threads, queue_len,
                      skip_translation, show_progress, device=devs[0], batch_reads=batch_reads,
                      table_capacity_hint=table_capacity_hint, both_strands=both_strands,
                      collapse_ratio=collapse_ratio, umi_length=umi_length, umi_offset=umi_offset)
    else:
        ctx = MultiContext(adapters, match_score, mismatch_score, gap_open_penalty, gap_extend_penalty,
                           accept_prefix_alignment, accept_suffix_alignment, n_threads, queue_len,
                           skip_translation, show_progress, devices=devs, batch_reads=batch_reads,
                           table_capacity_hint=table_capacity_hint, both_strands=both_strands,
                           collapse_ratio=collapse_ratio, umi_length=umi_length, umi_offset=umi_offset)
    with ctx:
        shown = show_progress and progress is None and sys.stderr.isatty()
        if progress is not None:
            ctx.set_progress(progress)
        elif shown:
            def spin(records, done, total, _f="|/-\\", _i=[0]):
                _i[0] += 1
                pct = " %3d%%" % (100 * done // total) if total else ""
                sys.stderr.write("\r%s Finding variants... %d reads%s" % (_f[_i[0] % 4], records, pct))
                sys.stderr.flush()
            ctx.set_progress(spin)
        try:
            for p in paths:
                ctx.run_file(p, allow_text=allow_text)
        finally:
            if shown:
                sys.stderr.write("\r" + " " * 60 + "\r")       # finish_and_clear
                sys.stderr.flush()
        return batch_to_frame(ctx.finish_arrow())


def collapse_variants(table, ratio, *, device=None, debug_hash_bits=0):
    """Fold sequencing-error variants into their parents, on the GPU (directional clustering, as UMI-tools does).

    `table` has columns `sequence` (string or binary) and `count` (unsigned): a pyarrow Table / RecordBatch or a
    polars DataFrame, such as find_variants returns.  Rows are ordered by count descending, then sequence bytes
    ascending.  Sequence a may be the parent of b when both have the same length and differ in exactly one byte
    (Hamming distance 1: no indels), a comes first in the order and count(a) >= ratio * count(b) in float64.  parent(b)
    is the first such a; each row's count goes to the end of its parent chain, so a sequence two substitutions from its
    root can be folded in through an intermediate one.  One row per root comes back (rows with count 0 are dropped), in
    the frame type find_variants returns, the sequence column as a string column if it was one, else binary.

    ratio: a finite real >= 1 (ValueError otherwise; TypeError for a non-number).  A sequence that appears twice is a
    ValueError.  Not for libraries whose true members are one substitution apart (single-mutant deep mutational
    scanning): the wild type would absorb the mutants.  debug_hash_bits: tests only."""
    import pyarrow as pa
    ratio = _ratio_arg(ratio, "ratio", False)
    if not isinstance(table, (pa.Table, pa.RecordBatch)) and hasattr(table, "to_arrow"):
        table = table.to_arrow()                                       # polars.DataFrame
    if isinstance(table, pa.RecordBatch):
        table = pa.Table.from_batches([table])
    if not isinstance(table, pa.Table):
        raise TypeError("collapse_variants: expected a pyarrow Table / RecordBatch or a polars DataFrame, not %s"
                        % type(table).__name__)
    seq, cnt = table.column("sequence").combine_chunks(), table.column("count").combine_chunks()
    # (polars exports its strings as string_view on recent versions)
    is_type = lambda name: getattr(pa.types, "is_" + name, lambda t: False)(seq.type)
    text = is_type("string") or is_type("large_string") or is_type("string_view")
    if not (text or is_type("binary") or is_type("large_binary") or is_type("binary_view")):
        raise TypeError("collapse_variants: column 'sequence' must be string or binary, not %s" % seq.type)
    if seq.null_count or cnt.null_count:
        raise ValueError("collapse_variants: null sequence or count")
    try:
        cnt = cnt.cast(pa.uint64())
    except (pa.ArrowInvalid, pa.ArrowNotImplementedError) as e:
        raise ValueError("collapse_variants: column 'count' must hold non-negative integers (%s)" % e) from None
    seq = seq.cast(pa.large_binary())
    n = len(seq)
    offsets = np.zeros(n + 1, dtype=np.uint64)
    data = np.zeros(0, dtype=np.uint8)
    if n:
        offsets = np.frombuffer(seq.buffers()[1], dtype=np.int64)[seq.offset:seq.offset + n + 1].astype(np.uint64)
        if seq.buffers()[2] is not None:
            data = np.frombuffer(seq.buffers()[2], dtype=np.uint8)
    counts = np.ascontiguousarray(cnt.to_numpy(zero_copy_only=False), dtype=np.uint64)
    L = load_library()
    t_in = Table(n, data.size, offsets.ctypes.data_as(C.POINTER(C.c_uint64)), data.ctypes.data_as(C.POINTER(C.c_uint8)),
                 counts.ctypes.data_as(C.POINTER(C.c_uint64)), None)
    t_out = Table()
    _check(L.vfb_collapse(C.byref(t_in), ratio, -1 if device is None else int(device), int(debug_hash_bits),
                          C.byref(t_out), None))
    o, d, c = _table_views(L, t_out, True)
    typ = pa.large_string() if text else pa.large_binary()
    tbl = pa.table({"sequence": pa.Array.from_buffers(typ, len(c), [None, pa.py_buffer(o.astype(np.int64)), pa.py_buffer(d)]),
                    "count": pa.array(c, type=pa.uint64())})
    try:
        import polars as pl
    except ImportError:
        return tbl
    return pl.from_arrow(tbl)


def _visible_devices() -> int:
    L = load_library()
    L.vfb_device_count.restype = C.c_int
    return int(L.vfb_device_count())


def _pick_devices(device, devices, paths):
    """[ordinal or None] for one context, or the list a MultiContext gets."""
    if device is not None and devices is not None:
        raise ValueError("give either device or devices, not both")
    if device is not None:
        return [int(device)]
    if devices is not None and not (isinstance(devices, str) and devices == "all"):
        devs = [int(d) for d in devices]
        if not devs:
            raise ValueError("devices must not be empty")
        return devs
    n = _visible_devices()
    if devices is None:
        # a GPU is worth starting for about 64 MB of compressed input (context creation costs more than that)
        size = sum(os.path.getsize(p) for p in paths)
        n = min(n, max(1, size >> 26))
        cap = os.environ.get("VFB_DEVICES")
        if cap:
            n = max(1, min(n, int(cap)))
    if n <= 1:
        return [None]
    return list(range(n))


def read_diagnostics(reads, adapters, match_score=3, mismatch_score=-2, gap_open_penalty=5, gap_extend_penalty=2,
                     accept_prefix_alignment=0.75, accept_suffix_alignment=0.75, skip_translation=False, *,
                     device=None, both_strands=False, umi_length=None, umi_offset=0):
    """What find_variants decides for each read, as a pyarrow.Table with one row per read (SURVEY §8(f) next-3):

    exact_prefix / exact_suffix  leftmost exact adapter position, null when absent      (src/lib.rs:148)
    score_* / len_*              semi-global alignment score and length statistic of the
                                 alignments the reference computes, null where none ran  (src/lib.rs:155-160)
    accept_prefix / accept_suffix  the adapter was located (exactly or by an accepted alignment)
    start / end                  region boundaries, null when not located               (src/lib.rs:278-286)
    region                       the variable region (null unless both located and start < end, src/lib.rs:288)

    With both_strands the columns above describe the forward pass, and these follow:

    strand                       +1: the read has a region as given, -1: its reverse complement has one (the read was
                                 retried), null: neither
    rev_exact_prefix ... rev_end the columns above for the reverse complement of the read; null where no reverse pass
                                 ran (the read has a forward region, or is empty)
    region                       the bases that were counted: reverse-complemented for strand -1

    With umi_length:

    umi                          bytes [umi_offset, umi_offset + umi_length) of the read in the orientation its region
                                 was found in (the reverse complement for strand -1); null where there is no region or
                                 the read is too short

    `reads` is a sequence of str / bytes.  Runs the full DP (exact scores also for rejected alignments)."""
    import pyarrow as pa
    umi_offset, umi_length = _umi_args(umi_length, umi_offset, None)

    def with_umi(cols, oriented):
        """oriented[i]: read i in its counted orientation, or None without a region"""
        if umi_length:
            cols["umi"] = pa.array([r[umi_offset:umi_offset + umi_length] if r is not None and len(r) >= umi_offset + umi_length
                                    else None for r in oriented], type=pa.binary())
        return pa.table(cols)

    seqs = [r if isinstance(r, bytes) else r.encode() for r in reads]
    n = len(seqs)
    length = np.array([len(s) for s in seqs], dtype=np.uint64)
    if int(length.sum()) >= 2 ** 32:
        raise ValueError("read_diagnostics takes at most 4 GiB of reads per call")
    spans = np.zeros(n, dtype=SPAN_DTYPE)
    spans["len"] = length
    if n:
        spans["off"][1:] = np.cumsum(length[:-1])
    text = np.frombuffer(b"".join(seqs), dtype=np.uint8)
    d = rd = np.zeros(0, dtype=DIAG_DTYPE)
    if n:
        ad = tuple(a if isinstance(a, bytes) else a.encode() for a in adapters)
        with Context(ad, match_score, mismatch_score, gap_open_penalty, gap_extend_penalty, accept_prefix_alignment,
                     accept_suffix_alignment, skip_translation=skip_translation, device=device, diagnostics=True,
                     batch_reads=max(n, 1), both_strands=both_strands) as ctx:
            ctx.submit_host(text, spans)
            d = ctx.diag(n)
            if both_strands:
                rd = ctx.diag_reverse(n)

    def columns(d, prefix="", ran_pass=None):
        cols = {}
        absent = np.zeros(len(d), dtype=bool) if ran_pass is None else ~ran_pass
        for f in ("exact_prefix", "exact_suffix"):
            cols[prefix + f] = pa.array(d[f], mask=(d[f] < 0) | absent, type=pa.int32())
        for side in ("prefix", "suffix"):
            ran = d["len_" + side] >= 0
            cols[prefix + "score_" + side] = pa.array(d["score_" + side], mask=~ran | absent, type=pa.int32())
            cols[prefix + "len_" + side] = pa.array(d["len_" + side], mask=~ran | absent, type=pa.int32())
        cols[prefix + "accept_prefix"] = pa.array(d["start"] >= 0, mask=absent)
        cols[prefix + "accept_suffix"] = pa.array(d["end"] >= 0, mask=absent)
        cols[prefix + "start"] = pa.array(d["start"], mask=(d["start"] < 0) | absent, type=pa.int32())
        cols[prefix + "end"] = pa.array(d["end"], mask=(d["end"] < 0) | absent, type=pa.int32())
        return cols

    cols = columns(d)
    if not both_strands:
        ok = (d["start"] >= 0) & (d["end"] >= 0) & (d["start"] < d["end"])
        cols["region"] = pa.array([seqs[i][d["start"][i]:d["end"][i]] if ok[i] else None for i in range(n)], type=pa.binary())
        return with_umi(cols, [seqs[i] if ok[i] else None for i in range(n)])
    # the predicate that decides the retry (and that the key kernels use): both located, start < end <= len
    fwd = (d["start"] >= 0) & (d["end"] >= 0) & (d["start"] < d["end"]) & (d["end"].astype(np.int64) <= length.astype(np.int64))
    retried = ~fwd & (length > 0)
    rev = retried & (rd["start"] >= 0) & (rd["end"] >= 0) & (rd["start"] < rd["end"]) & \
        (rd["end"].astype(np.int64) <= length.astype(np.int64))
    cols["strand"] = pa.array(np.where(fwd, 1, -1).astype(np.int8), mask=~(fwd | rev), type=pa.int8())
    cols.update(columns(rd, "rev_", retried))
    cols["region"] = pa.array([seqs[i][d["start"][i]:d["end"][i]] if fwd[i] else
                               reverse_complement(seqs[i])[rd["start"][i]:rd["end"][i]] if rev[i] else None
                               for i in range(n)], type=pa.binary())
    return with_umi(cols, [seqs[i] if fwd[i] else reverse_complement(seqs[i]) if rev[i] else None for i in range(n)])


_RC = bytes.maketrans(b"ACGTUacgtu", b"TGCAAtgcaa")


def reverse_complement(seq: bytes) -> bytes:
    """The reverse complement both_strands searches: A<->T, C<->G (either case), U->A, u->a, other bytes unchanged."""
    return bytes(seq)[::-1].translate(_RC)


# ---- synthetic reads (bench + tests) ----------------------------------------------------
def synth_cfg(seed=1003, read_len=250, adapter_len=20, region_len=198, n_variants=1000000, zipf=1,
              p_err=0.30, indel=0.5, force_indel=1, frameshift=0.05, noise=0.001, n_rate=1e-4) -> SynthCfg:
    ppm = lambda x: int(round(x * 1e6))
    return SynthCfg(seed, read_len, adapter_len, region_len, n_variants, zipf, ppm(p_err), ppm(indel),
                    force_indel, ppm(frameshift), ppm(noise), ppm(n_rate), 0)


def synth_adapters(cfg: SynthCfg):
    L = load_library()
    a = C.create_string_buffer(64)
    b = C.create_string_buffer(64)
    _check(L.vfb_synth_adapters(C.byref(cfg), a, b))
    return a.raw[:cfg.adapter_len], b.raw[:cfg.adapter_len]


def synth_host(cfg: SynthCfg, first: int, n: int):
    L = load_library()
    text = np.zeros(n * cfg.read_len, dtype=np.uint8)
    spans = np.zeros(n, dtype=SPAN_DTYPE)
    _check(L.vfb_synth_host(C.byref(cfg), first, n, text.ctypes.data, spans.ctypes.data))
    return text, spans


def synth_device(cfg: SynthCfg, first: int, n: int, text_ptr: int, spans_ptr: int, device: int = -1):
    _check(load_library().vfb_synth_device(C.byref(cfg), first, n, text_ptr, spans_ptr, device))


def hash_key(key: bytes) -> int:
    return int(load_library().vfb_hash_key(key, len(key)))


def key_owner(h: int, n_parts: int) -> int:
    return int(load_library().vfb_key_owner(h, n_parts))


def pinned_pool_trim():
    """Free the process-wide cache of pinned staging buffers."""
    _check(load_library().vfb_pinned_pool_trim())


def measure_int_peak(device: int = -1):
    a, d = C.c_double(0), C.c_double(0)
    _check(load_library().vfb_measure_int_peak(device, C.byref(a), C.byref(d)))
    return a.value, d.value
