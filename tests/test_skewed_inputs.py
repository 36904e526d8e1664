"""Low-complexity and skewed reads against the oracle.

Reads made of one short motif -- poly-G reads and tails of two-colour runs, poly-A of RNA-seq, telomeric (TTAGGG)n,
microsatellites -- have the same minimiser in every window: all their super-k-mer records go to one or two bins and one
k-mer can reach a count in the millions.  That is what reaches the code paths that random-genome reads never do: the
slab overflow list, the fallback of rfx_count to the two-pass partition, the spill pass of that partition, a streamed
partition sized from an unrepresentative first chunk, counts beyond 2^16 / 2^20, the sort kernel meeting a class that one
k-mer fills, and a rank of a sharded run that holds most of the records.  Every result is compared with the oracle.

tests/hooks/librfx_testhooks.so: rfx_debug_partition tells which partition a count ran on, so that every regime the
tests claim to reach is asserted, not hoped for."""
import os
import sys
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

INFO = ("slab_cap", "n_ovf", "ovf_cap", "n_bins", "n_records", "spill", "arena_used", "ovf_at", "ovf_bytes")


@pytest.fixture(scope="module")
def R():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import reflexiv_b200 as R
    R.load_library()
    return R


def _partition_info(hooks, ctx) -> dict:
    """rfx_debug_partition: the partition the context's records are in (read after the call that made them returned)."""
    C = hooks.C
    out = (C.c_uint64 * len(INFO))()
    hooks.L.rfx_debug_partition.argtypes = [C.c_void_p, C.c_void_p]
    assert hooks.L.rfx_debug_partition(ctx._ctx, out) == 0
    return dict(zip(INFO, [int(x) for x in out]))


def _regime(info) -> str:
    if info["slab_cap"] == 0:
        return "twopass"
    return "overflow" if info["n_ovf"] else "slab"


# ---- inputs --------------------------------------------------------------------------------------------------------------
def _fq(seqs, tag) -> bytes:
    return "".join(f"@{tag}{i}\n{s}\n+\n{'I' * len(s)}\n" for i, s in enumerate(seqs)).encode()


def _records(txt: bytes):
    """FASTQ text (4-line records) -> list of records (bytes, newline-terminated)."""
    lines = txt.split(b"\n")
    return [b"\n".join(lines[i:i + 4]) + b"\n" for i in range(0, len(lines) - 3, 4)]


def _shuffle(recs, seed) -> bytes:
    rng = np.random.default_rng(seed)
    return b"".join(recs[i] for i in rng.permutation(len(recs)))


def _genome_reads(n_reads, seed, glen=200_000, err=0.0, g=None) -> bytes:
    from workload import synth
    if g is None:
        g = synth.genome(glen, 500 + seed)
    return bytes(synth.fastq(g, n_reads // 2, read_len=150, frag_len=400, error_rate=err, seed_reads=7 + seed, seed_errors=8 + seed))


def _homopolymer_reads(n, tag="h", length=150) -> bytes:
    """all-A and all-G reads, alternating"""
    return _fq(["AG"[i & 1] * length for i in range(n)], tag)


def _motif_reads(n, motif, tag, length=150) -> bytes:
    rep = motif * (length // len(motif) + 2)
    return _fq([rep[i % len(motif):i % len(motif) + length] for i in range(n)], tag)


def _poly_g_tails(txt: bytes, seed) -> bytes:
    """genome reads whose last 20-80 bases are G"""
    rng = np.random.default_rng(seed)
    out = []
    for rec in _records(txt):
        h, s, p, q = rec.split(b"\n")[:4]
        t = int(rng.integers(20, 81))
        out.append(b"\n".join([h, s[:-t] + b"G" * t, p, q]) + b"\n")
    return b"".join(out)


def _microsatellite_genome(glen, seed):
    """random genome with a few hundred (CA)n, (AGC)n and (TTAGGG)n loci of 30-300 bp"""
    from workload import synth
    g = synth.genome(glen, 600 + seed)
    rng = np.random.default_rng(seed)
    for j, at in enumerate(range(1000, glen - 1000, 600)):
        motif = (b"CA", b"AGC", b"TTAGGG")[j % 3]
        n = int(rng.integers(30, 301))
        g[at:at + n] = np.frombuffer((motif * (n // len(motif) + 1))[:n], np.uint8)
    return g


def _zoo(k) -> bytes:
    """microsatellite genome reads + one adapter dimer read 10^4 times + reads shorter than k"""
    rng = np.random.default_rng(77)
    adapter = "".join("ACGT"[i] for i in rng.integers(0, 4, 96))
    g = _microsatellite_genome(120_000, 3)
    short = ["".join("ACGT"[i] for i in rng.integers(0, 4, int(n))) for n in rng.integers(1, k, 3000)]
    recs = _records(_genome_reads(16_000, 3, g=g)) + _records(_fq([adapter] * 10_000, "d")) + _records(_fq(short, "s"))
    return _shuffle(recs, 5)


def _mixture(frac, n_total=20_000, seed=1) -> bytes:
    """n_total reads, `frac` of them homopolymers, the rest reads of a random genome"""
    n_h = int(round(n_total * frac))
    recs = _records(_genome_reads(n_total - n_h, seed)) + _records(_homopolymer_reads(n_h))
    return _shuffle(recs, seed)


# ---- checks --------------------------------------------------------------------------------------------------------------
def _table(R, ctx, k):
    keys, cnt = ctx.counts()
    ints = np.array(R.pipeline.keys_to_int(keys, k), dtype=object)
    order = np.argsort(ints) if len(ints) else np.array([], dtype=np.int64)
    return [int(x) for x in ints[order]], cnt[order]


def _oracle_table(orc, txt, k, mode, minc=1, maxc=2**62):
    s, l = orc.fastq_reads(txt, mode)
    c = orc.count_kmers(txt, s, l, k, 0, 0, minc, maxc)
    return [(int(h) << 64) | int(lo) for h, lo in zip(c["keys_hi"], c["keys_lo"])], c["counts"], c


def _check_run(R, orc, hooks, txt, k, cover=2, E=8, min_contig=100):
    """Count (and assemble) on one context; table, fork survivors and contigs against the oracle (the checks of
    test_gpu_parity._check_assembly).  Returns the partition the count ran on."""
    ref = orc.run_pipeline(txt, k=k, cover=cover, min_error_cov=E, min_contig=min_contig)
    rc = ref["counts"]
    ints = [(int(h) << 64) | int(lo) for h, lo in zip(rc["keys_hi"], rc["keys_lo"])]
    with R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=cover, minErrorCoverage=E, minContig=min_contig)) as ctx:
        ctx.push_fastq(txt)
        ctx.count()
        info = _partition_info(hooks, ctx)
        g_ints, g_counts = _table(R, ctx, k)
        assert g_ints == ints and np.array_equal(g_counts, rc["counts"])
        st = ctx.assemble()
        hi, lo, le, ri = ctx.oriented()
        contigs = ctx.contigs()
    order = np.lexsort((lo, hi))
    f = ref["forks"]
    assert np.array_equal(hi[order], f["keys_hi"]) and np.array_equal(lo[order], f["keys_lo"])
    assert np.array_equal(le[order], f["left"]) and np.array_equal(ri[order], f["right"])
    a = ref["asm"]
    assert st["n_oriented"] == len(f["left"])
    assert (st["n_budget_junctions"], st["n_budget_admissible"], st["n_cycles"]) == (a["n_budget_junctions"], a["n_budget_admissible"], a["n_cycles"])
    assert sorted(contigs) == sorted(zip(a["contigs"], a["left"].tolist(), a["right"].tolist()))
    print(f"k={k} regime={_regime(info)} {info}")
    return info


# ---- A.1 mixture sweep: the three regimes of the single-pass partition -------------------------------------------------
@pytest.mark.parametrize("k", [31, 61])
@pytest.mark.parametrize("frac,regimes", [(0.0, ("slab", "slab")), (0.05, ("overflow", "overflow")), (0.35, ("overflow", "overflow")),
                                          (0.40, ("twopass", "overflow")), (0.90, ("twopass", "twopass"))])
def test_homopolymer_mixture(R, orc, hooks, k, frac, regimes):
    """20 000 reads, a growing share of them poly-A / poly-G: slab only, slab + overflow segment, fallback to two passes.
    (k = 31, 35 %: 33 341 records overflow a list of 33 868; 40 %: the list does not suffice.)"""
    info = _check_run(R, orc, hooks, _mixture(frac), k)
    assert _regime(info) == regimes[k == 61]
    if _regime(info) == "twopass":
        assert info["n_ovf"] > info["ovf_cap"]  # the fallback was taken because the list was too small


@pytest.mark.parametrize("k", [21, 31, 33, 61])
def test_poly_g_tails(R, orc, hooks, k):
    _check_run(R, orc, hooks, _poly_g_tails(_genome_reads(20_000, 2), 4), k)


@pytest.mark.parametrize("k", [21, 31, 33, 61])
def test_microsatellites_adapter_dimers_and_short_reads(R, orc, hooks, k):
    _check_run(R, orc, hooks, _zoo(k), k)


# ---- A.2 forced two passes -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,cover,E,err", [(21, 1, 8, 0.02), (31, 2, 8, 0.01), (33, 2, 8, 0.0), (61, 2, 8, 0.005)])
def test_two_pass_partition_assembles_like_the_oracle(R, orc, hooks, monkeypatch, k, cover, E, err):
    """RFX_PARTITION=twopass: rfx_count on the compact layout (the noisy reads of test_gpu_parity.test_assembly_matches_oracle)."""
    from workload import synth
    monkeypatch.setenv("RFX_PARTITION", "twopass")
    g = synth.genome(30_000, 100 + k)
    g[12000:12800] = g[3000:3800]
    g[20000:20040] = np.frombuffer(b"AT" * 20, np.uint8)
    txt = bytes(synth.fastq(g, 6000, read_len=150, frag_len=400, error_rate=err, seed_reads=5, seed_errors=6))
    info = _check_run(R, orc, hooks, txt, k, cover, E)
    assert _regime(info) == "twopass"


@pytest.mark.parametrize("k", [31, 61])
def test_spill_pass_of_the_two_pass_partition(R, orc, hooks, k):
    """Reads far longer than the descriptor slots of the two-pass scan: emit_spill_kernel places the runs pass 1 could not
    store (the reads of test_gpu_parity.test_long_and_ragged_reads)."""
    rng = np.random.default_rng(9)
    g = "".join("ACGT"[i] for i in rng.integers(0, 4, 20_000))
    seqs = [g[a:a + n] for a, n in ((0, 5000), (3000, 4000), (100, k), (200, k + 1), (300, k + 2), (400, 150), (9000, 11000), (0, 0), (5, 3))]
    seqs += [orc.revcomp_str(g[a:a + 700]) for a in range(0, 19000, 450)]
    txt = ("\n".join(seqs) + "\n").encode()
    ints, counts, c = _oracle_table(orc, txt, k, orc.FASTQ_LINE)
    with R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=1), fastq_mode=2) as ctx:
        ctx.push_fastq(txt)
        ctx.partition(1)
        info = _partition_info(hooks, ctx)
        st = ctx.count()
        g_ints, g_counts = _table(R, ctx, k)
    print(f"k={k} regime={_regime(info)} {info}")
    assert info["slab_cap"] == 0 and info["spill"] > 0
    assert st["n_instances"] == c["n_instances"]
    assert g_ints == ints and np.array_equal(g_counts, counts)


# ---- A.3 streamed partition sized from the first chunk ---------------------------------------------------------------------
def _streamed_input(which, k):
    genome = _records(_genome_reads(4_000, 11))
    heavy = _records(_genome_reads(2_000, 12)) + _records(_homopolymer_reads(18_000))
    if which == "short_first":  # the first chunk holds only reads shorter than k: no k-mer to size anything from
        rng = np.random.default_rng(13)
        short = _fq(["".join("ACGT"[i] for i in rng.integers(0, 4, int(n))) for n in rng.integers(1, k, 25_000)], "s")
        return short + _mixture(0.05)
    if which == "clean_first":
        return b"".join(genome) + _shuffle(heavy, 14)
    return _shuffle(heavy, 14) + b"".join(genome)  # heavy_first


@pytest.mark.parametrize("k", [31, 61])
@pytest.mark.parametrize("which", ["short_first", "clean_first", "heavy_first"])
def test_streamed_partition_from_an_unrepresentative_first_chunk(R, orc, hooks, monkeypatch, k, which):
    txt = _streamed_input(which, k)
    monkeypatch.setenv("RFX_FASTQ_CHUNK_BYTES", str(1 << 20))
    assert len(txt) >= 3 << 20
    ints, counts, c = _oracle_table(orc, txt, k, orc.FASTQ_RUN, minc=2, maxc=10_000_000)
    tables = []
    for stream in ("1", "0"):
        monkeypatch.setenv("RFX_STREAM_PARTITION", stream)
        with R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=2)) as ctx:
            ctx.push_fastq(txt)
            st = ctx.count()
            info = _partition_info(hooks, ctx)
            tables.append(_table(R, ctx, k))
        print(f"k={k} {which} stream={stream} regime={_regime(info)} {info}")
        assert st["n_instances"] == c["n_instances"]
    for g_ints, g_counts in tables:
        assert g_ints == ints and np.array_equal(g_counts, counts)


# ---- A.4 / A.5 heavy k-mers, coverage bounds, the sort kernel ------------------------------------------------------------
def _heavy_kmer_input(n_poly_a):
    return _shuffle(_records(_genome_reads(4_000, 21)) + _records(_fq(["A" * 150] * n_poly_a, "a")), 22)


def _check_heavy(R, orc, txt, k, heavy, counter_mode=False, cover=1, maxcov=10_000_000):
    if counter_mode:
        lo, hi = (cover if cover > 1 else 1), (maxcov if maxcov < 10_000_000 else 2**62)
    else:
        lo, hi = cover, maxcov
    mode = orc.FASTQ_COUNTER if counter_mode else orc.FASTQ_RUN
    ints, counts, c = _oracle_table(orc, txt, k, mode, minc=max(lo, 1), maxc=hi)
    with R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=cover, maxKmerCoverage=maxcov), counter_mode=counter_mode) as ctx:
        ctx.push_fastq(txt)
        ctx.count()
        g_ints, g_counts = _table(R, ctx, k)
    assert g_ints == ints and np.array_equal(g_counts, counts)
    return dict(zip(g_ints, g_counts.tolist())).get(heavy)


@pytest.mark.parametrize("k,n_poly_a", [(31, 600), (31, 9000), (61, 9000)])
@pytest.mark.parametrize("variant", ["", "sort"])
def test_heavy_kmer_counts_and_the_maxcov_boundary(R, orc, monkeypatch, k, n_poly_a, variant):
    """One k-mer (A^k) with n_poly_a * (151 - k) instances: 72 000 > 2^16, 1.08 M > 2^20 at k = 31; its poly-A reads are
    9000 x 4 identical records in one bin (far beyond one 768-record chunk of the hash kernel).  The exact count, and -maxcov
    at exactly that count (kept) and one below (dropped), in `run` and `counter` filter modes.  variant: RFX_COUNT_VARIANT."""
    if variant:
        monkeypatch.setenv("RFX_COUNT_VARIANT", variant)
    txt = _heavy_kmer_input(n_poly_a)
    n = n_poly_a * (151 - k)
    assert n > 1 << 16 and (n > 1 << 20 or n_poly_a < 9000 or k != 31)
    heavy = 0  # A^k: all bits zero
    assert _check_heavy(R, orc, txt, k, heavy) == n
    for counter_mode in (False, True):
        assert _check_heavy(R, orc, txt, k, heavy, counter_mode, cover=2, maxcov=n) == n
        assert _check_heavy(R, orc, txt, k, heavy, counter_mode, cover=2, maxcov=n - 1) is None


@pytest.mark.parametrize("k", [31, 61])
def test_sort_kernel_on_the_homopolymer_mixture(R, orc, hooks, monkeypatch, k):
    """RFX_COUNT_VARIANT=sort on 90 % poly-A / poly-G reads: one k-mer fills a hash class of its bin on its own."""
    monkeypatch.setenv("RFX_COUNT_VARIANT", "sort")
    _check_run(R, orc, hooks, _mixture(0.90), k)


# ---- A.6 / A.7 a heavy rank of a sharded run ------------------------------------------------------------------------------
def _heavy_rank_parts(world, k, motif):
    """rank 0: 30 000 reads of one motif; the other ranks: reads of a random genome"""
    from test_multi_gpu import _split
    rank0 = _homopolymer_reads(30_000) if motif == "AG" else _motif_reads(30_000, motif, "m")
    return [rank0] + _split(_genome_reads(12_000, 31 + k, glen=60_000), world - 1)


def _sharded_body(parts, bins, stream, results, hooks=None, infos=None):
    def body(rank, ctx):
        ctx.reset()
        if stream:
            ctx.shard_set_bins(bins)  # before the push: the streamed scan follows the upload with the run's bins
        if parts[rank]:
            ctx.push_fastq(parts[rank])
        if bins and not stream:
            ctx.shard_set_bins(bins)
        st = ctx.count_sharded()
        if infos is not None:
            infos[rank] = _partition_info(hooks, ctx)
        keys, cnt = ctx.counts()
        st2 = ctx.assemble_sharded()
        sh = ctx.shard_stats()
        ori = ctx.oriented() if not sh["fell_back"] else None
        results[rank] = dict(keys=keys, cnt=cnt, st=st, st2=st2, sh=sh, ori=ori, contigs=ctx.contigs())
    return body


@pytest.mark.parametrize("world,k", [(2, 31), (2, 61), (3, 31), (3, 61)])
@pytest.mark.parametrize("how", ["agreed", "set_bins", "set_bins_streamed"])
def test_heavy_rank_sharing_one_device(R, orc, hooks, monkeypatch, world, k, how):
    """Rank 0 holds only poly-A / poly-G (world 2) or (CA)n (world 3) reads: its slab overflow list cannot hold what its one
    or two bins overflow by, so it re-scans with a list of the counted size.  Union of the shard tables, fork survivors and
    contigs against the oracle; then the same run again on the same contexts."""
    from reflexiv_b200 import sharded
    from test_multi_gpu import _check_against_oracle
    parts = _heavy_rank_parts(world, k, "AG" if world == 2 else "CA")
    bins = 0 if how == "agreed" else 96 * world
    if how == "set_bins_streamed":
        monkeypatch.setenv("RFX_FASTQ_CHUNK_BYTES", str(1 << 20))
    ctxs = [R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=2, minContig=100), device=0) for _ in range(world)]
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=1 << 30)
        for _ in range(2):  # arenas, barrier epochs and published blocks are reused
            results, infos = [None] * world, [None] * world
            grp.run(_sharded_body(parts, bins, how == "set_bins_streamed", results, hooks, infos))
            print(f"world={world} k={k} {how} rank0 {infos[0]}")
            assert infos[0]["slab_cap"] > 0 and infos[0]["n_ovf"] == infos[0]["ovf_cap"] > 0  # the list of the re-scan: exactly the counted size
            _check_against_oracle(orc, b"".join(parts), k, 2, 8, 100, results)
    finally:
        for c in ctxs:
            c.close()


def test_heavy_rank_with_an_arena_too_small_fails_on_every_rank_at_once(R, orc, hooks):
    """The arena holds everything of the normal rank and the heavy rank's first scan, not the overflow list of its re-scan:
    every rank returns RFX_E_CAPACITY within seconds (no peer waits out a barrier), and the contexts stay usable."""
    from reflexiv_b200 import _lib, sharded
    from test_multi_gpu import _check_against_oracle, _split
    k, world = 31, 2
    parts = [_homopolymer_reads(30_000), _genome_reads(2_000, 41, glen=20_000)]

    def make(arena):
        ctxs = [R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=2, minContig=100), device=0) for _ in range(world)]
        return ctxs, sharded.LocalRanks(ctxs, arena_bytes=arena)

    # where the re-scan puts its overflow list, from a run in a large arena (the layout of a bump allocator is deterministic)
    infos = [None] * world
    ctxs, grp = make(1 << 30)
    try:
        def count_only(rank, ctx):
            ctx.reset()
            ctx.push_fastq(parts[rank])
            ctx.count_sharded()
            infos[rank] = _partition_info(hooks, ctx)
        grp.run(count_only)
    finally:
        for c in ctxs:
            c.close()
    heavy = infos[0]
    assert heavy["n_ovf"] == heavy["ovf_cap"] > 0 and heavy["ovf_at"] > 0
    arena = heavy["ovf_at"] + heavy["ovf_bytes"] // 4  # the re-scan's list does not fit
    assert infos[1]["arena_used"] < arena  # ... everything the normal rank needed does
    print(f"heavy {heavy} normal {infos[1]} arena {arena}")

    ctxs, grp = make(arena)
    try:
        errs = [None] * world

        def count_fails(rank, ctx):
            ctx.reset()
            ctx.push_fastq(parts[rank])
            try:
                ctx.count_sharded()
            except R.RfxError as e:
                errs[rank] = e
        t0 = time.perf_counter()
        grp.run(count_fails)
        took = time.perf_counter() - t0
        print(f"errors after {took:.2f} s: {errs}")
        assert all(e is not None and e.code == _lib.RFX_E_CAPACITY for e in errs), errs
        assert took < 10
        # a normal run on the same contexts
        txt = _genome_reads(4_000, 42, glen=20_000)
        results = [None] * world
        grp.run(_sharded_body(_split(txt, world), 0, False, results))
        _check_against_oracle(orc, txt, k, 2, 8, 100, results)
    finally:
        for c in ctxs:
            c.close()


# ---- one process per GPU ------------------------------------------------------------------------------------------------
def _ipc_worker(rank, world, port, k, out_dir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import pickle
    import torch
    import torch.distributed as dist
    import reflexiv_b200 as R
    from reflexiv_b200 import sharded
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    ctx = R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=2, minContig=100), device=rank)
    sharded.connect(ctx, dist, arena_bytes=1 << 30)
    results = [None] * world
    _sharded_body(_heavy_rank_parts(world, k, "AG"), 0, False, results)(rank, ctx)
    with open(os.path.join(out_dir, f"res_{rank}.pkl"), "wb") as f:
        pickle.dump(results[rank], f)
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("k", [31, 61])
def test_heavy_rank_one_process_per_gpu_over_ipc(tmp_path, orc, k):
    import pickle
    import torch
    import torch.multiprocessing as mp
    from test_multi_gpu import _check_against_oracle
    world = torch.cuda.device_count()
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    world = min(world, 4)
    port = 29300 + os.getpid() % 1000 + k
    mp.spawn(_ipc_worker, args=(world, port, k, str(tmp_path)), nprocs=world, join=True)
    results = [pickle.load(open(tmp_path / f"res_{r}.pkl", "rb")) for r in range(world)]
    _check_against_oracle(orc, b"".join(_heavy_rank_parts(world, k, "AG")), k, 2, 8, 100, results)
