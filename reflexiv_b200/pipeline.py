"""Host-side mirror of the reference's pipeline entry points on top of libreflexiv_cuda.

* ``ReflexivContext``                    one rfx_ctx (one GPU): push reads, count, assemble, fetch results
* ``Pipelines.reflexivDSCounterPipe``    <- pipeline/Pipelines.java:148-152 -> ReflexivDataFrameCounter.assembly() (:139-236)
* ``Pipelines.reflexivDSMainPipe``       <- pipeline/Pipelines.java:90-98   -> ReflexivDSMain.assembly() (:123-357)
                                            and assemblyFromKmer() (:362-713) when -kmerc is given
* ``Pipelines.reflexivLeftAndRightSortingPipe`` <- pipeline/Pipelines.java:1309-1313 -> ReflexivDSKmerLeftAndRightSorting
                                            .assemblyFromKmer() (:105-243): Count_<k> CSV -> ``<out>/Count_<k>_sorted``

Same output trees as the reference: ``<out>/Count_<k>/part-*.csv[.gz]`` + ``_SUCCESS`` (rows ``KMER,count``) and
``<out>/part-NNNNN`` contig files (``>Contig-<len>-(<left>,<right>)-<idx>`` + sequence wrapped at 100).
"""
from __future__ import annotations

import ctypes as C
import glob
import gzip
import os
import uuid
from typing import Iterable, List, Optional, Tuple

import numpy as np

from . import _lib
from ._lib import RfxError, RfxParams, RfxStats, load_library
from .params import DefaultParam


def _as_u8(buf) -> np.ndarray:
    if isinstance(buf, np.ndarray):
        return np.ascontiguousarray(buf, dtype=np.uint8)
    return np.frombuffer(bytes(buf), dtype=np.uint8)


class ReflexivContext:
    """One libreflexiv_cuda context.  All heavy lifting happens in the library; this class only moves
    numpy buffers across the C ABI."""

    def __init__(self, param: Optional[DefaultParam] = None, *, counter_mode: bool = False, fastq_mode: Optional[int] = None,
                 device: int = 0, minimizer_len: int = 0, table_capacity: int = 0, bin_target_kmers: int = 0):
        self.L = load_library()
        param = param or DefaultParam()
        p = RfxParams()
        self._check(self.L.rfx_params_default(C.byref(p)), None)
        p.kmer_size = param.kmerSize
        p.min_kmer_coverage = param.minKmerCoverage
        p.max_kmer_coverage = param.maxKmerCoverage
        p.min_error_coverage = param.minErrorCoverage
        p.min_contig = param.minContig
        p.front_clip = param.frontClip
        p.end_clip = param.endClip
        p.bubble = 1 if param.bubble else 0
        p.min_iter = param.minimumIteration
        p.max_iter = param.maximumIteration
        p.partitions = param.partitions
        p.shuffle_partitions = param.shufflePartition
        p.counter_mode = 1 if counter_mode else 0
        if fastq_mode is None:
            # `run` uses the 4-line state machine; `counter` the heuristic, or every line with -infmt line
            fastq_mode = _lib.FASTQ_RUN if not counter_mode else (_lib.FASTQ_LINE if param.inputFormat == "line" else _lib.FASTQ_COUNTER)
        p.fastq_mode = fastq_mode
        p.device = device
        p.minimizer_len = minimizer_len
        p.table_capacity = table_capacity
        p.bin_target_kmers = bin_target_kmers
        self.params = p
        self.k = param.kmerSize
        self._ctx = C.c_void_p()
        rc = self.L.rfx_create(C.byref(self._ctx), C.byref(p))
        if rc != 0:
            raise RfxError(rc, (self.L.rfx_last_error(None) or b"").decode())

    # ---- plumbing ----
    def _check(self, rc: int, ctx):
        if rc != 0:
            raise RfxError(rc, (self.L.rfx_last_error(ctx) or b"").decode())

    def close(self):
        if self._ctx:
            self.L.rfx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        self._check(self.L.rfx_reset(self._ctx), self._ctx)

    # ---- input ----
    def push_fastq(self, text):
        a = _as_u8(text)
        self._check(self.L.rfx_push_fastq(self._ctx, a.ctypes.data, a.size), self._ctx)

    def push_fastq_device(self, dev_ptr: int, n_bytes: int):
        self._check(self.L.rfx_push_fastq_device(self._ctx, dev_ptr, n_bytes), self._ctx)

    def push_reads(self, bases, offsets):
        b = _as_u8(bases)
        o = np.ascontiguousarray(offsets, dtype=np.uint64)
        self._check(self.L.rfx_push_reads(self._ctx, b.ctypes.data, o.ctypes.data, len(o) - 1), self._ctx)

    # ---- counting ----
    def count(self):
        self._check(self.L.rfx_count(self._ctx), self._ctx)
        return self.stats()

    def counts(self) -> Tuple[np.ndarray, np.ndarray]:
        """(keys uint64[n_rows, words_per_key] in the reference's key layout, counts uint32[n_rows]); row order unspecified."""
        n, w = C.c_uint64(), C.c_int32()
        self._check(self.L.rfx_counts_size(self._ctx, C.byref(n), C.byref(w)), self._ctx)
        keys = np.empty((n.value, w.value), dtype=np.uint64)
        cnt = np.empty(n.value, dtype=np.uint32)
        self._check(self.L.rfx_counts_copy(self._ctx, keys.ctypes.data, cnt.ctypes.data), self._ctx)
        return keys, cnt

    def counts_csv(self) -> bytes:
        n = C.c_uint64()
        self._check(self.L.rfx_counts_csv(self._ctx, None, 0, C.byref(n)), self._ctx)
        buf = np.empty(n.value, dtype=np.uint8)
        self._check(self.L.rfx_counts_csv(self._ctx, buf.ctypes.data, buf.size, C.byref(n)), self._ctx)
        return buf.tobytes()

    def load_counts(self, keys: np.ndarray, counts: np.ndarray):
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        counts = np.ascontiguousarray(counts, dtype=np.uint32)
        self._check(self.L.rfx_load_counts(self._ctx, keys.ctypes.data, counts.ctypes.data, len(counts)), self._ctx)

    def load_counts_csv(self, text, min_count: int, max_count: int, append: bool = False):
        """Count_<k> text (`KMER,count` / `(KMER,count)` rows) parsed on the device into the table: rows with
        min_count <= count <= max_count, in text order, behind the current table if append.  The row rule is the `reflexiv`
        binary's (include/reflexiv_cuda.h); a malformed row raises RfxError (RFX_E_INVALID) naming its line."""
        a = _as_u8(text)
        self._check(self.L.rfx_load_counts_csv(self._ctx, a.ctypes.data, a.size, min_count, max_count, 1 if append else 0), self._ctx)

    # ---- assembly ----
    def assemble(self):
        self._check(self.L.rfx_assemble(self._ctx), self._ctx)
        return self.stats()

    # ---- -stitch (ReflexivDSMain.java:585-672) ----
    def stitch_begin(self):
        """Assembles (every record kept) and builds the probe table of the low-coverage contig ends; until stitch_finish()
        the push_* calls scan reads for fragments instead of storing them."""
        self._check(self.L.rfx_stitch_begin(self._ctx), self._ctx)
        return self.stitch_stats()

    def stitch_finish(self):
        """Joins contig + fragment + contig chains; contigs() then returns the stitched set."""
        self._check(self.L.rfx_stitch_finish(self._ctx), self._ctx)
        return self.stitch_stats()

    def stitch_stats(self) -> dict:
        st = _lib.RfxStitchStats()
        self._check(self.L.rfx_stitch_stats(self._ctx, C.byref(st)), self._ctx)
        return st.as_dict()

    def contigs(self):
        """[(sequence, left_flag, right_flag)], both strands of every contig, order unspecified."""
        n, tot = C.c_uint64(), C.c_uint64()
        self._check(self.L.rfx_contigs_size(self._ctx, C.byref(n), C.byref(tot)), self._ctx)
        bases = np.empty(tot.value, dtype=np.uint8)
        offs = np.empty(n.value + 1, dtype=np.uint64)
        left = np.empty(n.value, dtype=np.int32)
        right = np.empty(n.value, dtype=np.int32)
        self._check(self.L.rfx_contigs_copy(self._ctx, bases.ctypes.data, offs.ctypes.data, left.ctypes.data, right.ctypes.data), self._ctx)
        blob = bases.tobytes()
        return [(blob[int(offs[i]):int(offs[i + 1])].decode(), int(left[i]), int(right[i])) for i in range(n.value)]

    def contigs_raw(self, out=None):
        """Contigs as flat arrays (bases uint8[total], offsets uint64[n+1], left int32[n], right int32[n]): the D2H read
        without building Python strings.  `out` may carry preallocated (e.g. pinned) arrays of sufficient size."""
        n, tot = C.c_uint64(), C.c_uint64()
        self._check(self.L.rfx_contigs_size(self._ctx, C.byref(n), C.byref(tot)), self._ctx)
        if out is not None and out[0].size >= tot.value and out[1].size >= n.value + 1 and out[2].size >= n.value:
            bases, offs, left, right = out
        else:
            bases = np.empty(tot.value, dtype=np.uint8)
            offs = np.empty(n.value + 1, dtype=np.uint64)
            left = np.empty(n.value, dtype=np.int32)
            right = np.empty(n.value, dtype=np.int32)
        self._check(self.L.rfx_contigs_copy(self._ctx, bases.ctypes.data, offs.ctypes.data, left.ctypes.data, right.ctypes.data), self._ctx)
        return bases[:tot.value], offs[:n.value + 1], left[:n.value], right[:n.value]

    def oriented(self):
        """Oriented k-mers that survive both fork filters: (keys_hi, keys_lo, left, right)."""
        n = C.c_uint64()
        self._check(self.L.rfx_oriented_size(self._ctx, C.byref(n)), self._ctx)
        hi = np.empty(n.value, dtype=np.uint64)
        lo = np.empty(n.value, dtype=np.uint64)
        le = np.empty(n.value, dtype=np.int32)
        ri = np.empty(n.value, dtype=np.int32)
        if n.value:
            self._check(self.L.rfx_oriented_copy(self._ctx, hi.ctypes.data, lo.ctypes.data, le.ctypes.data, ri.ctypes.data), self._ctx)
        return hi, lo, le, ri

    # ---- Count_<k>_sorted (ReflexivDSKmerLeftAndRightSorting.java:105-243) ----
    def sort_kmers(self, min_error_coverage: int = 8, min_repeat_fold: float = 1.5, max_kmer_size: int = 95) -> int:
        """Runs that stage's two fork filters over both orientations of the count table; returns the number of rows."""
        self._check(self.L.rfx_sort_kmers(self._ctx, min_error_coverage, min_repeat_fold, max_kmer_size), self._ctx)
        n = C.c_uint64()
        self._check(self.L.rfx_sorted_size(self._ctx, C.byref(n)), self._ctx)
        return n.value

    def sorted_rows(self):
        """(keys_hi, keys_lo, left, right) of the rows of Count_<k>_sorted, order unspecified."""
        n = C.c_uint64()
        self._check(self.L.rfx_sorted_size(self._ctx, C.byref(n)), self._ctx)
        hi = np.empty(n.value, dtype=np.uint64)
        lo = np.empty(n.value, dtype=np.uint64)
        le = np.empty(n.value, dtype=np.int32)
        ri = np.empty(n.value, dtype=np.int32)
        if n.value:
            self._check(self.L.rfx_sorted_copy(self._ctx, hi.ctypes.data, lo.ctypes.data, le.ctypes.data, ri.ctypes.data), self._ctx)
        return hi, lo, le, ri

    def sorted_csv(self) -> bytes:
        n = C.c_uint64()
        self._check(self.L.rfx_sorted_csv(self._ctx, None, 0, C.byref(n)), self._ctx)
        buf = np.empty(n.value, dtype=np.uint8)
        if n.value:
            self._check(self.L.rfx_sorted_csv(self._ctx, buf.ctypes.data, buf.size, C.byref(n)), self._ctx)
        return buf.tobytes()

    def stats(self) -> dict:
        s = RfxStats()
        self._check(self.L.rfx_stats(self._ctx, C.byref(s)), self._ctx)
        return s.as_dict()

    # ---- sharded counting ----
    def record_bytes(self) -> int:
        n = C.c_int32()
        self._check(self.L.rfx_record_bytes(self._ctx, C.byref(n)), self._ctx)
        return n.value

    def choose_bins(self, global_instances: int, n_shards: int = 1) -> int:
        """The library's bin count for `global_instances` k-mer instances over `n_shards` shards."""
        return int(self.L.rfx_choose_bins(self._ctx, global_instances, n_shards))

    def partition(self, n_shards: int, n_bins_total: int = 0):
        self._check(self.L.rfx_partition(self._ctx, n_shards, n_bins_total), self._ctx)

    def shard_records(self, shard: int) -> Tuple[int, int]:
        p, n = C.c_void_p(), C.c_uint64()
        self._check(self.L.rfx_shard_records(self._ctx, shard, C.byref(p), C.byref(n)), self._ctx)
        return (p.value or 0), n.value

    def begin_shard(self, shard_id: int, n_shards: int, n_bins_total: int):
        self._check(self.L.rfx_begin_shard(self._ctx, shard_id, n_shards, n_bins_total), self._ctx)

    def load_records_device(self, dev_ptr: int, n_bytes: int):
        self._check(self.L.rfx_load_records_device(self._ctx, dev_ptr, n_bytes), self._ctx)

    def shard_bin_offsets(self, shard: int) -> Tuple[int, int]:
        p, n = C.c_void_p(), C.c_uint32()
        self._check(self.L.rfx_shard_bin_offsets(self._ctx, shard, C.byref(p), C.byref(n)), self._ctx)
        return (p.value or 0), n.value

    def load_segment_device(self, rec_ptr: int, n_bytes: int, offsets_ptr: int):
        self._check(self.L.rfx_load_segment_device(self._ctx, rec_ptr, n_bytes, offsets_ptr), self._ctx)

    def rx_buffer(self, n_bytes: int) -> int:
        p = C.c_void_p()
        self._check(self.L.rfx_rx_buffer(self._ctx, n_bytes, C.byref(p)), self._ctx)
        return p.value or 0

    def counts_device(self):
        """(keys device pointer, counts device pointer, n_rows, key_bytes) of the filtered table in HBM."""
        pk, pc, n, kb = C.c_void_p(), C.c_void_p(), C.c_uint64(), C.c_int32()
        self._check(self.L.rfx_counts_device(self._ctx, C.byref(pk), C.byref(pc), C.byref(n), C.byref(kb)), self._ctx)
        return (pk.value or 0), (pc.value or 0), n.value, kb.value

    def load_counts_device(self, keys_ptr: int, counts_ptr: int, n_rows: int, append: bool = False):
        self._check(self.L.rfx_load_counts_device(self._ctx, keys_ptr, counts_ptr, n_rows, 1 if append else 0), self._ctx)

    # ---- multi-GPU over peer memory (include/reflexiv_cuda.h: rfx_shard_*) ----
    def shard_init(self, rank: int, world: int, arena_bytes: int = 0):
        self._check(self.L.rfx_shard_init(self._ctx, rank, world, arena_bytes), self._ctx)

    def shard_export(self) -> bytes:
        buf = C.create_string_buffer(_lib.RFX_SHARD_HANDLE_BYTES)
        self._check(self.L.rfx_shard_export(self._ctx, buf), self._ctx)
        return buf.raw

    def shard_connect(self, handles: bytes, world: int):
        assert len(handles) == world * _lib.RFX_SHARD_HANDLE_BYTES
        self._check(self.L.rfx_shard_connect(self._ctx, handles, world), self._ctx)

    def shard_set_bins(self, n_bins_total: int):
        self._check(self.L.rfx_shard_set_bins(self._ctx, n_bins_total), self._ctx)

    def count_sharded(self):
        """Collective: every rank calls it.  On return this context holds the rows whose minimiser bin it owns."""
        self._check(self.L.rfx_count_sharded(self._ctx), self._ctx)
        return self.stats()

    def shard_table(self):
        """Collective: every rank calls it after loading any slice of a count table (load_counts*, may be empty).  On return
        this context holds the rows whose minimiser bin it owns, as after count_sharded()."""
        self._check(self.L.rfx_shard_table(self._ctx), self._ctx)
        return self.stats()

    def assemble_sharded(self):
        """Collective.  On return this context holds the contigs whose first k-mer it owns."""
        self._check(self.L.rfx_assemble_sharded(self._ctx), self._ctx)
        return self.stats()

    def sort_kmers_sharded(self, min_error_coverage: int = 8, min_repeat_fold: float = 1.5, max_kmer_size: int = 95) -> int:
        """Collective sort_kmers() on a table sharded by minimiser bin (after count_sharded() or shard_table()).  On return this
        context holds the Count_<k>_sorted rows of its shard (sorted_rows(), sorted_csv()); returns their number."""
        self._check(self.L.rfx_sort_kmers_sharded(self._ctx, min_error_coverage, min_repeat_fold, max_kmer_size), self._ctx)
        n = C.c_uint64()
        self._check(self.L.rfx_sorted_size(self._ctx, C.byref(n)), self._ctx)
        return n.value

    def stitch_begin_sharded(self):
        """Collective stitch_begin() on a table sharded by minimiser bin (after count_sharded() or shard_table()).  Until
        stitch_finish_sharded() the push_* calls of this rank scan its own reads for fragments (not collective: any split of
        the reads, a rank may push none)."""
        self._check(self.L.rfx_stitch_begin_sharded(self._ctx), self._ctx)
        return self.stitch_stats()

    def stitch_finish_sharded(self):
        """Collective stitch_finish(): contigs() then returns the stitched records whose head contig this rank owns; their
        union over the ranks is the one-context result."""
        self._check(self.L.rfx_stitch_finish_sharded(self._ctx), self._ctx)
        return self.stitch_stats()

    def shard_stats(self) -> dict:
        s = _lib.RfxShardStats()
        self._check(self.L.rfx_shard_stats(self._ctx, C.byref(s)), self._ctx)
        return s.as_dict()


# ------------------------------------------------------------------------------------------------------
# helpers shared by the pipelines
# ------------------------------------------------------------------------------------------------------

def decode_keys(keys: np.ndarray, k: int) -> List[str]:
    """DSBinaryKmerToString (Counter.java:405-428, Counter64.java:340-369) for a key matrix in the reference layout."""
    out = []
    if k <= 31:
        for v in keys[:, 0].tolist():
            out.append("".join("ACGT"[(v >> (2 * (k - 1 - i))) & 3] for i in range(k)))
    else:
        res = k % 32
        for row in keys.tolist():
            s = []
            for i in range(k // 32 * 32):
                s.append("ACGT"[(row[i // 32] >> (2 * (31 - i % 32))) & 3])
            for i in range(k // 32 * 32, k):
                s.append("ACGT"[(row[i // 32] >> (2 * (res - 1 - i % 32))) & 3])
            out.append("".join(s))
    return out


def keys_to_int(keys: np.ndarray, k: int) -> List[int]:
    """Reference key layout -> one Python int per k-mer (right-aligned 2k bits)."""
    if k <= 31:
        return [int(v) for v in keys[:, 0]]
    res = k % 32
    return [(int(r[0]) << (2 * res)) | int(r[1]) for r in keys]


def encode_kmer_rows(kmers: Iterable[str], k: int) -> np.ndarray:
    """KmerBinarizer (DSMain.java:3872-3948): ACGT strings -> key matrix in the reference layout."""
    code = {"A": 0, "C": 1, "G": 2}
    w = 1 if k <= 31 else k // 32 + 1
    rows = []
    for s in kmers:
        v = 0
        for ch in s:
            v = (v << 2) | code.get(ch, 3)
        if k <= 31:
            rows.append([v])
        else:
            res = k % 32
            rows.append([(v >> (2 * res)) & 0xFFFFFFFFFFFFFFFF, v & ((1 << (2 * res)) - 1)])
    return np.array(rows, dtype=np.uint64).reshape(-1, w)


def format_contig(seq: str, left: int, right: int, idx: int) -> str:
    """DSKmerToContig + changeLine + TagRowContigID (DSMain.java:743-794, 717-725)."""
    body = "\n".join(seq[i:i + 100] for i in range(0, len(seq), 100))
    return f">Contig-{len(seq)}-({left},{right})-{idx}\n{body}"


def _input_paths(pattern: str) -> List[str]:
    paths = sorted(glob.glob(pattern)) or ([pattern] if os.path.exists(pattern) else [])
    if not paths:
        raise FileNotFoundError(f"Input path does not exist: {pattern}")
    out = []
    for p in paths:
        if os.path.isdir(p):
            out += [os.path.join(p, q) for q in sorted(os.listdir(p)) if not q.startswith(("_", "."))]
        else:
            out.append(p)
    return out


def iter_input_files(pattern: str, readers: Optional[int] = None):
    """spark.read().text(glob): the text of every matching file in path order, .gz inflated on a few host threads ahead of
    the consumer (zlib releases the GIL), every chunk ending on a newline.  Same scheme as the `reflexiv` binary
    (csrc/reflexiv_main.cpp: stream_inputs): the host holds a look-ahead window, not the whole input."""
    from concurrent.futures import ThreadPoolExecutor
    paths = _input_paths(pattern)
    readers = max(1, min(readers or (os.cpu_count() or 4), 16, len(paths)))
    with ThreadPoolExecutor(max_workers=readers) as pool:
        pending = [pool.submit(_read_one, p) for p in paths[:readers]]
        nxt = len(pending)
        while pending:
            c = pending.pop(0).result()
            if nxt < len(paths):
                pending.append(pool.submit(_read_one, paths[nxt]))
                nxt += 1
            if c:
                yield c if c.endswith(b"\n") else c + b"\n"


def read_input_text(pattern: str) -> bytes:
    """All matching files concatenated (small inputs: count tables, tests)."""
    return b"".join(iter_input_files(pattern))


def _read_one(path: str) -> bytes:
    if path.endswith(".4mc"):
        raise RfxError(_lib.RFX_E_UNSUPPORTED, f"{path}: 4mc input needs hadoop-4mc; decompress first or use gzip/plain text")
    if path.endswith(".gz"):
        with gzip.open(path, "rb") as f:
            data = f.read()
    else:
        with open(path, "rb") as f:
            data = f.read()
    # Hadoop's LineRecordReader also ends a line at a lone "\r"; the library takes "\n" and "\r\n" only (csrc/reflexiv_main.cpp)
    head = data[:65536]
    if any(head[i:i + 1] == b"\r" and head[i + 1:i + 2] != b"\n" for i in range(len(head) - 1) if head[i] == 13):
        raise RfxError(_lib.RFX_E_UNSUPPORTED, f"{path}: lone '\\r' line ends (classic Mac text) are not supported; convert with tr '\\r' '\\n'")
    return data


def parse_count_csv(text: bytes, k: int) -> Tuple[np.ndarray, np.ndarray]:
    """KmerBinarizer input forms: `KMER,count` and the legacy `(KMER,count)`; counts of >= 10 digits clamp to 10^9
    (DSMain.java:3895-3910).  Vectorised over the rows (numpy): a table of millions of rows parses in seconds.
    Returns (keys uint64[n, words] in the reference layout, counts uint32[n])."""
    a = np.frombuffer(bytes(text), dtype=np.uint8)
    w = 1 if k <= 31 else k // 32 + 1
    if a.size == 0:
        return np.empty((0, w), np.uint64), np.empty(0, np.uint32)
    nl = np.flatnonzero(a == 10)
    starts = np.concatenate(([0], nl + 1)).astype(np.int64)
    ends = np.concatenate((nl, [a.size])).astype(np.int64)
    pad = np.concatenate((a, np.zeros(16, np.uint8)))          # so that fixed-width gathers may look past the end
    ends = ends - ((ends > starts) & (pad[np.maximum(ends - 1, 0)] == 13))                  # "\r\n"
    keep = ends > starts
    starts, ends = starts[keep], ends[keep]
    starts = starts + (pad[starts] == ord("("))
    ends = ends - (pad[np.maximum(ends - 1, 0)] == ord(")"))
    if np.any(ends - starts < k + 2) or np.any(pad[starts + k] != ord(",")):
        raise ValueError("malformed k-mer count row")
    # k-mer: A=0 C=1 G=2, anything else 3 (nucleotideValue, DSMain.java:3935-3947)
    chars = pad[starts[:, None] + np.arange(k)[None, :]]
    codes = np.full(chars.shape, 3, np.uint64)
    codes[chars == ord("A")] = 0
    codes[chars == ord("C")] = 1
    codes[chars == ord("G")] = 2
    keys = np.zeros((len(starts), w), np.uint64)
    if k <= 31:
        for i in range(k):
            keys[:, 0] = (keys[:, 0] << np.uint64(2)) | codes[:, i]
    else:                                                        # 32 bases per word, the last word holds k % 32 right aligned
        for i in range(k):
            j = i // 32
            keys[:, j] = (keys[:, j] << np.uint64(2)) | codes[:, i]
    nd = ends - (starts + k + 1)
    counts = np.zeros(len(starts), np.int64)
    for d in range(int(min(nd.max(), 9)) if len(nd) else 0):
        ch = pad[starts + k + 1 + d].astype(np.int64)
        use = (d < nd) & (nd < 10)
        if np.any(use & ((ch < 48) | (ch > 57))):
            raise ValueError("malformed k-mer count row")
        counts = np.where(use, counts * 10 + (ch - 48), counts)
    counts[nd >= 10] = 1_000_000_000
    return keys, counts.astype(np.uint32)


class Pipelines:
    """pipeline/Pipelines.java: one method per workflow."""

    def __init__(self, param: DefaultParam, device: int = 0):
        self.param = param
        self.device = device

    def reflexivDSCounterPipe(self) -> dict:
        p = self.param
        with ReflexivContext(p, counter_mode=True, device=self.device) as ctx:
            n_files = 0
            for chunk in iter_input_files(p.inputFqPath):  # one push per file, the next files inflate meanwhile
                ctx.push_fastq(chunk)
                n_files += 1
            if not n_files:
                ctx.push_fastq(b"")
            st = ctx.count()
            csv = ctx.counts_csv()
        out_dir = os.path.join(p.outputPath, f"Count_{p.kmerSize}")
        os.makedirs(out_dir, exist_ok=True)  # SaveMode.Overwrite, Counter.java:224-231
        for f in os.listdir(out_dir):
            os.remove(os.path.join(out_dir, f))
        name = f"part-00000-{uuid.uuid4()}-c000.csv"
        if p.gzip:
            with gzip.open(os.path.join(out_dir, name + ".gz"), "wb") as f:
                f.write(csv)
        else:
            with open(os.path.join(out_dir, name), "wb") as f:
                f.write(csv)
        open(os.path.join(out_dir, "_SUCCESS"), "w").close()
        return st

    def reflexivDSMainPipe(self) -> dict:
        p = self.param
        from_kmer = p.inputKmerPath is not None
        out_dir = os.path.join(p.outputPath, f"Assemble_{p.kmerSize}") if from_kmer else p.outputPath  # DSMain.java:706-710 / 354
        if os.path.exists(out_dir):
            raise FileExistsError(f"Output directory {out_dir} already exists")  # Hadoop FileAlreadyExistsException
        with ReflexivContext(p, counter_mode=False, device=self.device) as ctx:
            if from_kmer:
                keys, counts = parse_count_csv(read_input_text(p.inputKmerPath), p.kmerSize)
                keep = (counts >= p.minKmerCoverage) & (counts <= p.maxKmerCoverage)  # DSMain.java:405-412
                ctx.load_counts(keys[keep], counts[keep])
            else:
                n_files = 0
                for chunk in iter_input_files(p.inputFqPath):
                    ctx.push_fastq(chunk)
                    n_files += 1
                if not n_files:
                    ctx.push_fastq(b"")
                ctx.count()
            if from_kmer and p.stitch:
                # ReflexivDSMain.java:585-672: the FASTQ is read a second time, by the stitch branch only (Parameter.java:571-575)
                if p.inputFqPath is None:
                    raise ValueError("-stitch reads the FASTQ (ReflexivDSMain.java:599): give -fastq next to -kmerc")
                ctx.stitch_begin()
                for chunk in iter_input_files(p.inputFqPath):
                    ctx.push_fastq(chunk)
                stitch = ctx.stitch_finish()
                st = ctx.stats()
                st["stitch"] = stitch
            else:
                st = ctx.assemble()
            contigs = ctx.contigs()
        os.makedirs(out_dir)
        data = "".join(format_contig(s, l, r, i) + "\n" for i, (s, l, r) in enumerate(contigs)).encode()
        if p.gzip and from_kmer:
            with gzip.open(os.path.join(out_dir, "part-00000.gz"), "wb") as f:
                f.write(data)
        else:
            with open(os.path.join(out_dir, "part-00000"), "wb") as f:
                f.write(data)
        open(os.path.join(out_dir, "_SUCCESS"), "w").close()
        return st

    def reflexivLeftAndRightSortingPipe(self) -> dict:
        """Count_<k> CSV (param.inputKmerPath) -> <out>/Count_<k>_sorted/part-*.csv[.gz] + _SUCCESS, rows `KMER,1|left|right`
        (ReflexivDSKmerLeftAndRightSorting.java:168-240).  K-mers whose length is not in the k-mer list are dropped by the
        reference's binarizer (:1695), so a k outside the list writes an empty table."""
        p = self.param
        keys, counts = parse_count_csv(read_input_text(p.inputKmerPath), p.kmerSize)
        keep = counts <= p.maxKmerCoverage  # :186-193, the lower bound is commented out in the reference
        if p.kmerSize not in p.kmerListInt:
            keep &= False
        with ReflexivContext(p, counter_mode=False, device=self.device) as ctx:
            ctx.load_counts(keys[keep], counts[keep])
            n = ctx.sort_kmers(p.minErrorCoverage, p.minRepeatFold, p.kmerListInt[-1])
            csv = ctx.sorted_csv()
            st = ctx.stats()
        out_dir = os.path.join(p.outputPath, f"Count_{p.kmerSize}_sorted")
        os.makedirs(out_dir, exist_ok=True)  # SaveMode.Overwrite, :226-238
        for f in os.listdir(out_dir):
            os.remove(os.path.join(out_dir, f))
        name = f"part-00000-{uuid.uuid4()}-c000.csv"
        if p.gzip:
            with gzip.open(os.path.join(out_dir, name + ".gz"), "wb") as f:
                f.write(csv)
        else:
            with open(os.path.join(out_dir, name), "wb") as f:
                f.write(csv)
        open(os.path.join(out_dir, "_SUCCESS"), "w").close()
        st["n_sorted_rows"] = n
        return st
