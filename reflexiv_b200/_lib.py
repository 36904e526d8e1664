"""ctypes binding of include/reflexiv_cuda.h (the same symbols a JNI / Panama driver would bind)."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class RfxError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libreflexiv_cuda error {code}: {msg}")
        self.code = code


# rfx_status
RFX_OK, RFX_E_INVALID, RFX_E_CUDA, RFX_E_NOMEM, RFX_E_STATE, RFX_E_CAPACITY, RFX_E_GRAPH, RFX_E_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6, -7
FASTQ_RUN, FASTQ_COUNTER, FASTQ_LINE = 0, 1, 2


class RfxParams(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "struct_size", "kmer_size", "min_kmer_coverage", "max_kmer_coverage", "min_error_coverage", "min_contig",
        "front_clip", "end_clip", "bubble", "min_iter", "max_iter", "partitions", "shuffle_partitions", "counter_mode",
        "fastq_mode", "device", "minimizer_len", "reserved0")] + [("table_capacity", C.c_int64), ("bin_target_kmers", C.c_int64)]


class RfxStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "n_reads", "n_bases", "n_instances", "n_distinct", "n_rows", "n_records", "n_bins", "n_bin_splits", "n_oriented",
        "n_budget_junctions", "n_budget_admissible", "n_cycles", "n_contigs", "n_contig_bases", "kernel_launches")] + [
        (n, C.c_float) for n in ("ms_parse", "ms_partition", "ms_count", "ms_graph", "ms_extend", "ms_contigs",
                                 "ms_kernel_bin_histogram", "ms_kernel_bin_scatter", "ms_kernel_count", "reserved1")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


RFX_SHARD_HANDLE_BYTES = 128


class RfxShardStats(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32)] + [(n, C.c_uint64) for n in (
        "arena_bytes", "arena_used", "n_instances_global", "n_shard_instances", "n_rows_global", "n_oriented_global", "n_contigs_global",
        "n_contig_bases_global", "n_remote_probes", "n_l1_splitters", "n_l2_splitters")] + [("ms_comm", C.c_float), ("fell_back", C.c_int32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class RfxStitchStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("n_probes", "n_reads", "n_fragments", "n_after_pass1", "n_joined", "n_stitched", "n_rings")] + [
        ("ms_stitch", C.c_float), ("reserved", C.c_float)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "reserved"}


# every symbol include/reflexiv_cuda.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "rfx_version": (C.c_char_p, []),
    "rfx_params_default": (C.c_int, [C.POINTER(RfxParams)]),
    "rfx_create": (C.c_int, [C.POINTER(_P), C.POINTER(RfxParams)]),
    "rfx_destroy": (None, [_P]),
    "rfx_last_error": (C.c_char_p, [_P]),
    "rfx_reset": (C.c_int, [_P]),
    "rfx_push_fastq": (C.c_int, [_P, _P, C.c_size_t]),
    "rfx_push_fastq_device": (C.c_int, [_P, _P, C.c_size_t]),
    "rfx_push_reads": (C.c_int, [_P, _P, _P, C.c_uint64]),
    "rfx_count": (C.c_int, [_P]),
    "rfx_counts_size": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_int32)]),
    "rfx_counts_copy": (C.c_int, [_P, _P, _P]),
    "rfx_counts_csv": (C.c_int, [_P, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
    "rfx_load_counts": (C.c_int, [_P, _P, _P, C.c_uint64]),
    "rfx_load_counts_csv": (C.c_int, [_P, _P, C.c_size_t, C.c_int64, C.c_int64, C.c_int32]),
    "rfx_assemble": (C.c_int, [_P]),
    "rfx_contigs_size": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "rfx_contigs_copy": (C.c_int, [_P, _P, _P, _P, _P]),
    "rfx_oriented_size": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "rfx_oriented_copy": (C.c_int, [_P, _P, _P, _P, _P]),
    "rfx_sort_kmers": (C.c_int, [_P, C.c_int32, C.c_double, C.c_int32]),
    "rfx_sorted_size": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "rfx_sorted_copy": (C.c_int, [_P, _P, _P, _P, _P]),
    "rfx_sorted_csv": (C.c_int, [_P, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
    "rfx_stitch_begin": (C.c_int, [_P]),
    "rfx_stitch_finish": (C.c_int, [_P]),
    "rfx_stitch_stats": (C.c_int, [_P, C.POINTER(RfxStitchStats)]),
    "rfx_stats": (C.c_int, [_P, C.POINTER(RfxStats)]),
    "rfx_partition": (C.c_int, [_P, C.c_int32, C.c_uint32]),
    "rfx_choose_bins": (C.c_uint32, [_P, C.c_uint64, C.c_int32]),
    "rfx_rx_buffer": (C.c_int, [_P, C.c_uint64, C.POINTER(C.c_void_p)]),
    "rfx_shard_records": (C.c_int, [_P, C.c_int32, C.POINTER(_P), C.POINTER(C.c_uint64)]),
    "rfx_begin_shard": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_uint32]),
    "rfx_load_records_device": (C.c_int, [_P, _P, C.c_uint64]),
    "rfx_record_bytes": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "rfx_shard_bin_offsets": (C.c_int, [_P, C.c_int32, C.POINTER(_P), C.POINTER(C.c_uint32)]),
    "rfx_load_segment_device": (C.c_int, [_P, _P, C.c_uint64, _P]),
    "rfx_counts_device": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_P), C.POINTER(C.c_uint64), C.POINTER(C.c_int32)]),
    "rfx_load_counts_device": (C.c_int, [_P, _P, _P, C.c_uint64, C.c_int32]),
    "rfx_shard_init": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_uint64]),
    "rfx_shard_export": (C.c_int, [_P, _P]),
    "rfx_shard_connect": (C.c_int, [_P, _P, C.c_int32]),
    "rfx_shard_set_bins": (C.c_int, [_P, C.c_uint32]),
    "rfx_count_sharded": (C.c_int, [_P]),
    "rfx_shard_table": (C.c_int, [_P]),
    "rfx_assemble_sharded": (C.c_int, [_P]),
    "rfx_sort_kmers_sharded": (C.c_int, [_P, C.c_int32, C.c_double, C.c_int32]),
    "rfx_stitch_begin_sharded": (C.c_int, [_P]),
    "rfx_stitch_finish_sharded": (C.c_int, [_P]),
    "rfx_shard_stats": (C.c_int, [_P, C.POINTER(RfxShardStats)]),
    "rfx_device_count": (C.c_int, [C.POINTER(C.c_int32)]),
}


def lib_path() -> str:
    return os.path.join(_HERE, "libreflexiv_cuda.so")


def load_library():
    """Loads the in-tree libreflexiv_cuda.so.  No fallback: a missing library is an error."""
    global _LIB
    if _LIB is None:
        path = lib_path()
        if not os.path.exists(path):
            raise RfxError(RFX_E_STATE, f"{path} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                        f"or `make -C reflexiv_b200/csrc`")
        L = C.CDLL(path)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the header and the library disagree
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB
