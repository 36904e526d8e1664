#!/usr/bin/env python
"""bench.py -- headline benchmark of the Reflexiv hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...            (one rank per GPU)

Workloads (BASELINE.json `configs`, selected by --config; the default and the driver's run is 2):
  2  configs[1]  synthetic E. coli-size genome (4.6 Mbp), 150 bp paired reads at 100x, k = 31, full `reflexiv run` path:
                 FASTQ text -> 2-bit reads -> canonical k-mer count table -> coverage filter -> fork filters -> contig
                 extension -> contig bases.  WEAK scaling: every GPU holds 3.07 M reads, the genome grows with N.
  3  configs[2]  `reflexiv counter` only, 10^8 x 150 bp reads (150 Mbp genome at 100x), k = 31; STRONG scaling: the reads
                 are split over the ranks.
  4  configs[3]  k = 61 (two-word keys), 100 Mbp genome, 1 % substitution errors, cover 2, 30x, full run path; strong.
  5  configs[4]  250 Mbp genome, 60x, k = 31, full run path; strong (the 8-GPU configuration).
  --scale f shrinks genome and read set of configs 3-5 (the line then says so).

A step is one pass of the path over the whole read set.  At N > 1 every rank is one process with one context; the
contexts map each other's device arenas (CUDA IPC) and the library's sharded calls do the rest inside CUDA kernels over
NVLink: the owner of a minimiser bin counts it straight out of every rank's super-k-mer slabs (that read IS the
exchange), the graph stages run on the rows a rank owns with neighbour probes, chain links and contig bases crossing
GPUs through peer pointers (include/reflexiv_cuda.h: rfx_shard_*).  torch.distributed (NCCL) is used for the set-up
(handle exchange), the barriers around the timed region and the max-over-ranks of the time.

`value`    k-mer instances per second over the whole step, inputs (FASTQ text) resident in HBM.
`e2e`      same metric through the public API with host buffers: H2D of the FASTQ text from pinned memory and D2H of
           the result (contigs; the count table for config 3) inside the timed region.
`roofline` the counting stage against the measured HBM copy bandwidth, algorithmic bytes per SURVEY 8(d); three
           denominators are reported: kernel events only, the library's stage timers, and from device-resident FASTQ.
`parity`   N > 1 only, outside the timed region: rank 0 runs the single-GPU library path over the union of all ranks'
           reads and the run fails unless row count, sum of counts, an order-independent digest of the table and the
           canonical contig set equal what the sharded run produced.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

READ_LEN = 150
UNIT = "k-mers/s"
CONFIGS = {
    2: dict(name="configs[1]", genome=4_600_000, coverage=100.0, k=31, error=0.0, cover=2, mode="run", scaling="weak"),
    3: dict(name="configs[2]", genome=150_000_000, coverage=100.0, k=31, error=0.0, cover=2, mode="counter", scaling="strong"),
    4: dict(name="configs[3]", genome=100_000_000, coverage=30.0, k=61, error=0.01, cover=2, mode="run", scaling="strong"),
    5: dict(name="configs[4]", genome=250_000_000, coverage=60.0, k=31, error=0.0, cover=2, mode="run", scaling="strong"),
}
METRIC = {"run": "canonical k-mers counted/sec (full reflexiv run path: count + contig extension)",
          "counter": "canonical k-mers counted/sec (reflexiv counter path: FASTQ text -> filtered count table)"}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


class Workload:
    """Which reads a rank holds.  Weak scaling: genome = N x the per-GPU genome, every rank the same number of pairs.
    Strong scaling: one genome, the pairs split evenly over the ranks."""

    def __init__(self, cfg_id: int, world: int, scale: float = 1.0, read_len_min: int = 0):
        from workload import synth
        c = dict(CONFIGS[cfg_id])
        self.cfg_id, self.cfg, self.world, self.scale = cfg_id, c, world, scale
        g = int(c["genome"] * (scale if cfg_id != 2 else 1.0))
        self.genome_len = g * world if c["scaling"] == "weak" else g
        total_pairs = synth.n_pairs_for(g, c["coverage"], READ_LEN) * (world if c["scaling"] == "weak" else 1)
        self.pairs = [total_pairs * (r + 1) // world - total_pairs * r // world for r in range(world)]
        self.first = [total_pairs * r // world for r in range(world)]
        self.total_reads = 2 * total_pairs
        self.k = c["k"]
        self.read_len_min = read_len_min
        self._genome = None

    def text(self, rank: int):
        from workload import synth
        if self._genome is None:
            self._genome = synth.genome(self.genome_len)
        txt = synth.fastq(self._genome, self.pairs[rank], read_len=READ_LEN, frag_len=400, first_pair=self.first[rank], error_rate=self.cfg["error"])
        if self.read_len_min:
            txt = trim_reads(txt, self.read_len_min, seed=rank)
        return txt

    def instances(self, rank=None):
        if self.read_len_min:
            return None  # known after the run (ragged reads)
        per_read = READ_LEN - self.k + 1
        return (2 * self.pairs[rank] if rank is not None else self.total_reads) * per_read

    def describe(self):
        c = self.cfg
        s = (f"{c['name']}: synthetic {self.genome_len} bp genome, {self.total_reads} x {READ_LEN} bp paired reads at {c['coverage']:.0f}x, k={c['k']}, "
             f"cover {c['cover']}, " + ("full run path (FASTQ text -> counts -> fork filters -> contigs)" if c["mode"] == "run" else "counter path (FASTQ text -> filtered count table)"))
        if c["error"]:
            s += f", {c['error'] * 100:g} % substitution errors"
        if c.get("variant_error"):
            s += " [variant: error rate overridden]"
        if self.scale != 1.0 and self.cfg_id != 2:
            s += f" [SCALED to {self.scale:g} of the configuration's size]"
        if self.read_len_min:
            s += f" [variant: reads quality-trimmed to {self.read_len_min}..{READ_LEN} bp]"
        return s


def trim_reads(txt, lo: int, seed: int = 0):
    """Quality-trimmed variant of a synthetic FASTQ: every read keeps a random prefix of lo..READ_LEN bases."""
    import numpy as np
    a = np.asarray(txt)
    nl = np.flatnonzero(a == 10)
    starts = np.concatenate(([0], nl[:-1] + 1))
    lens = nl - starts
    n_rec = len(nl) // 4
    rng = np.random.default_rng(1234 + seed)
    keep = rng.integers(lo, READ_LEN + 1, n_rec)
    new_len = lens.copy()
    new_len[1::4] = np.minimum(lens[1::4], keep)
    new_len[3::4] = new_len[1::4]
    out_start = np.concatenate(([0], np.cumsum(new_len + 1)[:-1]))
    out = np.empty(int((new_len + 1).sum()), dtype=np.uint8)
    step = 1 << 20  # lines per block: one fancy-index gather each, bounded scratch
    for b in range(0, len(nl), step):
        e = min(len(nl), b + step)
        o0, o1 = int(out_start[b]), int(out_start[e - 1] + new_len[e - 1] + 1)
        idx = np.repeat(starts[b:e] - out_start[b:e], new_len[b:e] + 1) + np.arange(o0, o1)
        out[o0:o1] = a[np.minimum(idx, a.size - 1)]
    out[out_start + new_len] = 10
    return out


def cpu_reference_run(wl: Workload, rank: int = 0, threads: int = 0):
    """The reference's algorithm on the host cores (oracle: extract -> hash-partition -> per-partition aggregate ->
    filter -> fork filters -> sort + merge passes) on one rank's share of the workload."""
    from oracle import orc
    threads = threads or os.cpu_count() or 1
    txt = wl.text(rank)
    k, cover = wl.k, wl.cfg["cover"]
    orc.set_threads(threads)  # sorts on all threads, one scan task per range partition (Spark local[threads])
    t0 = time.perf_counter()
    starts, lens = orc.fastq_reads(txt, orc.FASTQ_RUN if wl.cfg["mode"] == "run" else orc.FASTQ_COUNTER)
    cnt = orc.count_kmers(txt, starts, lens, k, 0, 0, cover, 10_000_000, threads)
    t1 = time.perf_counter()
    n_passes = 0
    if wl.cfg["mode"] == "run":
        ff = orc.fork_filter(cnt["keys_hi"], cnt["keys_lo"], cnt["counts"], k, 8)
        asm = orc.assemble(ff["keys_hi"], ff["keys_lo"], ff["left"], ff["right"], k, 500, orc.ASM_REFSIM)
        n_passes = asm["n_passes"]
    t2 = time.perf_counter()
    orc.set_threads(1)
    n_inst = cnt["n_instances"]
    share = "the whole workload" if wl.world == 1 else f"rank 0's share (1/{wl.world}) of the workload"
    return {"value": n_inst / (t2 - t0), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{share}: {len(starts)} reads x {READ_LEN} bp ({n_inst} k-mers), k={k}; count {t1 - t0:.2f}s"
                      + (f" + fork filters and {n_passes} sort+merge passes {t2 - t1:.2f}s" if wl.cfg["mode"] == "run" else "")
                      + f", all on {threads} threads (parallel sorts, one scan task per range partition); "
                      "CPU restatement of the reference algorithm, the JVM/Spark reference cannot run in this image",
            "count_stage_kmers_per_s": n_inst / (t1 - t0), "reads_per_s": len(starts) / (t2 - t0), "seconds": t2 - t0}


def run_reference(args, emit):
    """--impl reference: the CPU restatement of the reference algorithm on the SAME input as the GPU arm (one rank's share
    of it at N > 1), every step one full pass; passes beyond a ~150 s budget are not run (the line says how many were)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = Workload(args.config, world, args.scale)
    vals, t_start = [], time.perf_counter()
    want = max(1, args.warmup) - 1 + max(1, args.steps)
    for _ in range(want):
        vals.append(cpu_reference_run(wl))
        if time.perf_counter() - t_start > 150 and len(vals) >= 2:
            break
    timed = vals[-max(1, min(args.steps, len(vals) - (1 if len(vals) > 1 else 0))):]
    best = sorted(timed, key=lambda r: r["value"])[len(timed) // 2]
    mode = wl.cfg["mode"]
    line = {"impl": "reference", "metric": METRIC[mode], "value": best["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": best["seconds"] * 1e3, "higher_is_better": True, "scaling": wl.cfg["scaling"], "vs_baseline": None,
            "dtype": "u64" if wl.k <= 31 else "u128", "data": "synthetic",
            "config": {"workload": wl.describe(), "note": best["sample"], "passes_run": len(vals), "passes_timed": len(timed)},
            "cpu_baseline": {k: best[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": best["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def files_end_to_end(wl, text, total_inst):
    """SURVEY 8d's outermost timed region: the `reflexiv` command itself -- process start, CUDA context, file read (mapped /
    inflated on host threads), upload, the whole path, contig (or count-table) files written -- wall clock of the command."""
    import gzip
    import shutil
    import tempfile
    exe = os.path.join(ROOT, "reflexiv_b200", "reflexiv")
    tmp = tempfile.mkdtemp(prefix="rfx_bench_")
    out = {}
    try:
        plain = os.path.join(tmp, "reads.fq")
        with open(plain, "wb") as f:
            f.write(memoryview(text))
        gz = os.path.join(tmp, "reads_gz.fq.gz")
        with open(plain, "rb") as f, gzip.open(gz, "wb", compresslevel=1) as g:
            shutil.copyfileobj(f, g, 1 << 24)
        cmd = "counter" if wl.cfg["mode"] == "counter" else "run"
        for label, path in (("plain", plain), ("gzip", gz)):
            best = None
            for rep in range(2):  # the second run finds the file in the page cache
                target = os.path.join(tmp, f"out_{label}_{rep}")
                t0 = time.perf_counter()
                r = subprocess.run([exe, cmd, "-fastq", path, "-outfile", target, "-kmer", str(wl.k), "-cover", str(wl.cfg["cover"])], capture_output=True, text=True)
                dt = time.perf_counter() - t0
                if r.returncode != 0:
                    out[label] = {"error": (r.stderr or r.stdout)[-300:]}
                    break
                best = dt if best is None else min(best, dt)
            if best is not None:
                out[label] = {"seconds": best, "value": total_inst / best, "unit": UNIT, "input_bytes": os.path.getsize(path)}
        out["note"] = ("wall clock of `reflexiv %s -fastq <file> -outfile <dir>`: process start and CUDA context creation, file mapped (plain) or inflated with zlib on "
                       "host threads (gzip, one member: one thread), chunked upload overlapped with parsing, the whole path, output tree written; best of two runs" % cmd)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return out


def table_digest(keys, counts):
    """Order-independent digest of a (k-mer, count) table: (rows, sum of counts, sum of mixed rows mod 2^64)."""
    import numpy as np
    if len(counts) == 0:
        return 0, 0, 0
    k64 = keys.reshape(len(counts), -1).astype(np.uint64)
    with np.errstate(over="ignore"):
        h = np.zeros(len(counts), dtype=np.uint64)
        for j in range(k64.shape[1]):
            h = (h ^ k64[:, j]) * np.uint64(0x9E3779B97F4A7C15)
            h ^= h >> np.uint64(29)
        h = (h + counts.astype(np.uint64)) * np.uint64(0xD6E8FEB86659FD93)
        h ^= h >> np.uint64(32)
        return len(counts), int(counts.astype(np.uint64).sum()), int(h.sum(dtype=np.uint64))


def contig_digests(bases, offs):
    """sha256 of every contig in canonical orientation (the smaller of the contig and its reverse complement)."""
    import numpy as np
    comp = np.zeros(256, dtype=np.uint8)
    for a, b in zip(b"ACGT", b"TGCA"):
        comp[a] = b
    out = []
    for i in range(len(offs) - 1):
        s = np.asarray(bases[int(offs[i]):int(offs[i + 1])])
        rc = comp[s[::-1]]
        neq = np.flatnonzero(s != rc)
        canon = s if (len(neq) == 0 or s[neq[0]] < rc[neq[0]]) else rc
        out.append(hashlib.sha256(canon.tobytes()).hexdigest())
    return sorted(out)


DUMP_BYTES = 64 << 20


def result_arrays(ctx, mode: str) -> dict:
    """What a caller of the timed path receives from `ctx`, as float arrays that hold every value exactly.  The library
    leaves the order of table rows and of contigs unspecified, so rows are sorted by key and contigs by sequence: two
    runs or two builds that compute the same result give the same arrays."""
    import numpy as np
    if mode == "counter":
        keys, cnts = ctx.counts()
        order = np.lexsort(keys.T)
        # a 64-bit key word does not fit a float64 mantissa, its two 32-bit halves do
        return {"count_keys": keys[order].view(np.uint32).astype(np.float64), "count_values": cnts[order].astype(np.float64)}
    bases, offs, left, right = ctx.contigs_raw()
    seqs = [bases[int(offs[i]):int(offs[i + 1])].tobytes() for i in range(len(left))]
    order = sorted(range(len(seqs)), key=lambda i: (seqs[i], left[i], right[i]))
    return {"contig_bases": np.frombuffer(b"".join(seqs[i] for i in order), dtype=np.uint8).astype(np.float32),
            "contig_lengths": np.array([len(seqs[i]) for i in order], dtype=np.float64),
            "contig_left": left[order].astype(np.float64), "contig_right": right[order].astype(np.float64)}


def dump_outputs(arrays: dict, out_dir: str, limit: int = DUMP_BYTES, suffix: str = "") -> None:
    """Writes every array as out_dir/<name><suffix>.npy, at most `limit` bytes in all.  Small arrays are kept whole; one
    that does not fit its share of what is left is cut to a seeded sample of its rows, the same rows for the same shape."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    room = limit - 4096 * len(arrays)  # what the .npy headers leave
    names = sorted(arrays, key=lambda n: arrays[n].nbytes)
    for i, name in enumerate(names):
        a = arrays[name]
        share = room // (len(names) - i)
        if a.nbytes > share:
            rows = share // (a.nbytes // len(a))
            a = a[np.unique(np.random.default_rng(0).integers(0, len(a), rows))]
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)
        room -= a.nbytes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--scale", type=float, default=1.0, help="configs 3-5 only: fraction of the configuration's genome / read set")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer pass (large configurations on small hosts)")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the single-GPU cross-check after the timed region")
    ap.add_argument("--files", action="store_true", help="N = 1: also time the `reflexiv` command line end to end through files (plain and gzip input, output tree written)")
    ap.add_argument("--trim-to", type=int, default=0, help="variant: reads quality-trimmed to a random length in [trim-to, 150]")
    ap.add_argument("--error-rate", type=float, default=None, help="variant: override the configuration's per-base substitution rate")
    ap.add_argument("--minimizer", type=int, default=0)
    ap.add_argument("--bin-target", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (contigs, or the count table for config 3) as DIR/<name>.npy, "
                         "float32 / float64, at most 64 MB in all (a seeded sample of rows beyond that); N > 1: one file set per rank")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm returns no arrays")
    # stdout carries exactly one JSON line: everything else any library prints goes to stderr, and the line itself is
    # written to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    if args.impl == "reference":
        run_reference(args, emit)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import reflexiv_b200 as R
    from reflexiv_b200 import sharded

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libreflexiv_cuda has no CPU path")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    args.warmup = max(args.warmup, 3)

    wl = Workload(args.config, world, args.scale, args.trim_to)
    if args.error_rate is not None:
        wl.cfg["variant_error"] = wl.cfg["error"] != args.error_rate
        wl.cfg["error"] = args.error_rate
    cfg, kk, mode = wl.cfg, wl.k, wl.cfg["mode"]
    txt = wl.text(rank)
    n_reads = 2 * wl.pairs[rank]
    n_bytes = len(txt)
    e2e_on = not args.no_e2e
    pinned = torch.empty(n_bytes + 64, dtype=torch.uint8, pin_memory=e2e_on)
    pinned[:n_bytes] = torch.from_numpy(np.asarray(txt))
    pinned[n_bytes:] = 0
    host_view = pinned.numpy()[:n_bytes]
    del txt

    param = R.DefaultParam(kmerSize=kk, minKmerCoverage=cfg["cover"])
    ctx = R.ReflexivContext(param, device=local, counter_mode=(mode == "counter"), minimizer_len=args.minimizer, bin_target_kmers=args.bin_target)
    if world > 1:
        free_b, _ = torch.cuda.mem_get_info(device)
        sharded.connect(ctx, dist, arena_bytes=int(free_b * 0.62) - n_bytes)  # the rest: the device copy of the text + the cross-check on rank 0
        inst_guess = wl.instances() or wl.total_reads * (READ_LEN - kk + 1)
        ctx.shard_set_bins(ctx.choose_bins(inst_guess, world))  # known up front: rfx_push_fastq scans every chunk straight into the slabs
    d_text = torch.zeros(n_bytes + 64, dtype=torch.uint8, device=device)
    d_text[:n_bytes].copy_(pinned[:n_bytes])
    torch.cuda.synchronize()

    # pinned landing buffers for the end-to-end result read
    if mode == "run":
        n_ctg_max = 1 << 20
        out_bases = torch.empty(2 * wl.genome_len + (1 << 22), dtype=torch.uint8, pin_memory=e2e_on).numpy()
        out_offs = torch.empty(n_ctg_max, dtype=torch.int64, pin_memory=e2e_on).numpy().view(np.uint64)
        out_left = torch.empty(n_ctg_max, dtype=torch.int32, pin_memory=e2e_on).numpy()
        out_right = torch.empty(n_ctg_max, dtype=torch.int32, pin_memory=e2e_on).numpy()
    e2e_parts = {"push_fastq": 0.0, "count": 0.0, "assemble": 0.0, "fetch_result": 0.0}

    def step(from_host: bool):
        ctx.reset()
        t0 = time.perf_counter()
        if from_host:
            ctx.push_fastq(host_view)
        else:
            ctx.push_fastq_device(d_text.data_ptr(), n_bytes)
        t1 = time.perf_counter()
        st = ctx.count() if world == 1 else ctx.count_sharded()
        t2 = time.perf_counter()
        if mode == "run":
            st = ctx.assemble() if world == 1 else ctx.assemble_sharded()
        t3 = time.perf_counter()
        d2h = 0
        if from_host:
            if mode == "run":
                bases, offs, left, right = ctx.contigs_raw((out_bases, out_offs, out_left, out_right))
                d2h = bases.nbytes + offs.nbytes + left.nbytes + right.nbytes
            else:
                keys, cnts = ctx.counts()
                d2h = keys.nbytes + cnts.nbytes
            t4 = time.perf_counter()
            for key, dt in zip(e2e_parts, (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
                e2e_parts[key] += dt
        return st, d2h

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(n_steps: int, from_host: bool):
        barrier()
        launches0 = ctx.stats()["kernel_launches"]
        t0 = time.perf_counter()
        stats, d2h = [], 0
        for _ in range(n_steps):
            st, d2h = step(from_host)
            stats.append(st)
        barrier()
        wall = time.perf_counter() - t0
        t = torch.tensor([wall], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), stats, ctx.stats()["kernel_launches"] - launches0, d2h

    # raw pinned-host -> device copy rate of this box (what bounds the end-to-end path)
    h2d_gbs = None
    if e2e_on:
        h2d_ev0, h2d_ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        scratch = torch.empty(n_bytes, dtype=torch.uint8, device=device)
        scratch.copy_(pinned[:n_bytes], non_blocking=True)
        torch.cuda.synchronize()
        h2d_ev0.record()
        scratch.copy_(pinned[:n_bytes], non_blocking=True)
        h2d_ev1.record()
        torch.cuda.synchronize()
        h2d_gbs = n_bytes / (h2d_ev0.elapsed_time(h2d_ev1) * 1e-3) / 1e9
        del scratch
        torch.cuda.empty_cache()

    for _ in range(args.warmup):
        step(False)
    sampler = ClockSampler(local)
    sampler.start()
    t_dev, stats, launches, _ = timed(args.steps, False)
    clocks = sampler.stop()
    shard_st = ctx.shard_stats() if world > 1 else None
    if args.dump_outputs:
        dump_outputs(result_arrays(ctx, mode), args.dump_outputs, DUMP_BYTES // world, f"_rank{rank}" if world > 1 else "")
    d_text = None  # the end-to-end steps upload from the pinned host copy: give the device copy back first
    torch.cuda.empty_cache()
    t_e2e, d2h_bytes = None, 0
    if e2e_on:
        step(True)
        for key in e2e_parts:
            e2e_parts[key] = 0.0
        t_e2e, _, _, d2h_bytes = timed(args.steps, True)

    def med(key, ss=stats):
        v = sorted(s[key] for s in ss)
        return v[len(v) // 2]

    st = stats[-1]
    # k-mer instances of the whole job: known in closed form for fixed-length reads, summed over the ranks otherwise
    total_inst = wl.instances()
    inst_local = st["n_instances"]
    if total_inst is None:
        t = torch.tensor([inst_local], dtype=torch.int64, device=device)
        if world > 1:
            dist.all_reduce(t)
        total_inst = int(t.item())
    ms_step = t_dev / args.steps * 1e3
    value = total_inst / (t_dev / args.steps)
    stage_ms = {k: med(k) for k in ("ms_parse", "ms_partition", "ms_count", "ms_graph", "ms_extend", "ms_contigs")}
    kern_ms = {"ms_kernel_scan": med("ms_kernel_bin_histogram") + med("ms_kernel_bin_scatter"), "ms_kernel_count": med("ms_kernel_count")}

    # Roofline of the counting stage.  Algorithmic bytes (SURVEY 8d, stated in DESIGN.md):
    #   B_count = sum(read_len) + 16 * N * W + (8 * W + 4) * D'     (W = 1 word per key for k <= 31; 17.25 B per k-mer at L = 150)
    # for what THIS rank processes: its reads through the minimiser scan, its bins through the counting kernel.
    peak, peak_src = hbm_peak()
    wkey = 1 if kk <= 31 else 2
    rows_local = st["n_rows"]
    b_count = st["n_bases"] + 16 * wkey * inst_local + (8 * wkey + 4) * rows_local
    count_kernels_ms = sum(kern_ms.values())
    stage_timer_ms = stage_ms["ms_partition"] + stage_ms["ms_count"]
    from_fastq_ms = stage_timer_ms + stage_ms["ms_parse"]

    def gbs(ms):
        return b_count / (ms * 1e-3) / 1e9 if ms else None

    ach = gbs(count_kernels_ms)
    roofline = {"bound": "hbm",
                "kernel": "counting stage = bin_scan_fast_kernel / bin_scan_kernel (minimiser scan + super-k-mer record store) + count_bins_kernel (per-bin count + coverage filter)",
                "dominant_kernel": max(kern_ms, key=kern_ms.get),
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak if ach else None, "traffic": None, "peak_source": peak_src,
                "denominators": {
                    "kernel_events_ms": count_kernels_ms, "frac_kernel_events": ach / peak if ach else None,
                    "stage_timers_ms": stage_timer_ms, "frac_stage_timers": (gbs(stage_timer_ms) or 0) / peak if stage_timer_ms else None,
                    "from_device_fastq_ms": from_fastq_ms, "frac_from_device_fastq": (gbs(from_fastq_ms) or 0) / peak if from_fastq_ms else None,
                    "note": "`achieved` / `frac` divide by the CUDA-event durations of the two counting kernels; stage_timers adds what the library's stage "
                            "timers see around them (extent tables, overflow handling, host readbacks); from_device_fastq also adds K1 (line scan, FASTQ "
                            "state machine, 2-bit encoding), which is what actually reads the ASCII bases the numerator charges"},
                "algorithmic_bytes_per_launch": b_count, "algorithmic_bytes_per_kmer": b_count / inst_local if inst_local else None,
                "kernel_ms": kern_ms, "stage_kmers_per_s": inst_local / (count_kernels_ms * 1e-3) if count_kernels_ms else None,
                "bound_observed": "instruction issue / shared-memory latency, not DRAM (ncu summaries in profiles/)"}
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if world == 1 and args.config == 2 and not args.trim_to and os.path.exists(prof):
        try:
            tj = json.load(open(prof))
            roofline["traffic"] = tj.get("counting_stage_dram_bytes")
            roofline["traffic_source"] = "constant from profiles/traffic.json (ncu --set full capture of this workload: dram__bytes_read.sum + dram__bytes_write.sum of the two kernels), not measured in this run"
        except Exception:
            pass

    line = {"metric": METRIC[mode], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "u64" if kk <= 31 else "u128", "data": "synthetic",
            "config": {"workload": wl.describe(),
                       "l2_policy": f"inputs larger than L2: {n_bytes / 1e6:.0f} MB of FASTQ text per GPU per step, nothing reused across steps",
                       "parallelism": "1 GPU" if world == 1 else f"{world} GPUs, one process each: minimiser-bin shards; the counting kernel of a bin's owner pulls the bin's super-k-mer "
                                      "records out of every rank's slab over NVLink (cp.async.bulk from peer memory), graph stages on the own rows with peer-memory probes / links / "
                                      "contig writes; flag barriers in peer memory; no collective library on the data path (NCCL: set-up and timing only)",
                       "timing": "host clock around blocking C-ABI calls bracketed by barrier + cuda synchronize, max over ranks; per-stage and per-kernel times from CUDA events on the library's stream"},
            "reads_per_s": wl.total_reads / (t_dev / args.steps),
            "stage_ms": stage_ms, "result": {k: st[k] for k in ("n_reads", "n_instances", "n_distinct", "n_rows", "n_records", "n_bins", "n_bin_splits",
                                                              "n_oriented", "n_contigs", "n_contig_bases", "n_budget_junctions", "n_budget_admissible", "n_cycles")},
            "roofline": roofline, "gpu_launches": launches, "clocks": clocks}
    if world > 1:
        line["result_scope"] = "rank 0's shard (rows / contigs it owns); global figures under `shard`"
        line["shard"] = {k: shard_st[k] for k in ("n_instances_global", "n_rows_global", "n_oriented_global", "n_contigs_global", "n_contig_bases_global",
                                                   "n_remote_probes", "n_l1_splitters", "n_l2_splitters", "ms_comm", "fell_back", "arena_used")}
    if e2e_on:
        line["e2e"] = {"value": total_inst / (t_e2e / args.steps), "unit": UNIT, "h2d_bytes_per_step": n_bytes, "d2h_bytes_per_step": d2h_bytes,
                       "ms_per_step": t_e2e / args.steps * 1e3, "h2d_gbs_raw_copy": h2d_gbs, "h2d_ms_raw_copy": n_bytes / h2d_gbs / 1e6,
                       "host_ms_per_call": {k2: v / args.steps * 1e3 for k2, v in e2e_parts.items()},
                       "note": "per rank: FASTQ text uploaded in 96 MB chunks on a copy stream while the previous chunk is parsed and scanned; result read back into host arrays"}

    # ---- N > 1: the sharded result against the single-GPU library path on the same reads (outside the timed region) ----
    if world > 1 and not args.no_parity:
        keys, cnts = ctx.counts()
        mine = {"table": table_digest(keys, cnts)}
        if mode == "run":
            bases, offs, _, _ = ctx.contigs_raw()
            mine["contigs"] = contig_digests(bases, offs)
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        if rank == 0:
            got_rows = sum(g["table"][0] for g in gathered)
            got_sum = sum(g["table"][1] for g in gathered)
            got_dig = sum(g["table"][2] for g in gathered) & ((1 << 64) - 1)
            got_ctg = sorted(x for g in gathered for x in g.get("contigs", []))
            with R.ReflexivContext(param, device=local, counter_mode=(mode == "counter")) as one:
                for r in range(world):
                    one.push_fastq(wl.text(r))
                one.count()
                k1, c1 = one.counts()
                exp_rows, exp_sum, exp_dig = table_digest(k1, c1)
                exp_ctg = []
                if mode == "run":
                    one.assemble()
                    b1, o1, _, _ = one.contigs_raw()
                    exp_ctg = contig_digests(b1, o1)
            parity = {"checked": True, "against": "single-GPU library path (rfx_count + rfx_assemble) on the union of all ranks' reads, run on rank 0 after the timed region",
                      "n_rows": [got_rows, exp_rows], "sum_counts": [got_sum, exp_sum], "table_digest_equal": got_dig == exp_dig,
                      "n_contigs": [len(got_ctg), len(exp_ctg)], "contig_set_equal": got_ctg == exp_ctg}
            line["parity"] = parity
            ok = got_rows == exp_rows and got_sum == exp_sum and got_dig == exp_dig and got_ctg == exp_ctg
            if not ok:
                print("PARITY FAILURE:", json.dumps(parity), file=sys.stderr)
                raise SystemExit(3)
    if rank == 0 and world == 1 and args.files:
        line["e2e_files"] = files_end_to_end(wl, host_view, total_inst)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = {k: v for k, v in cpu_reference_run(wl).items() if k in ("value", "unit", "cores", "kind", "sample", "count_stage_kmers_per_s", "reads_per_s")}
    if rank == 0:
        emit(line)
    if world > 1:
        dist.barrier()
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
