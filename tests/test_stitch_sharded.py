"""-stitch across ranks (include/reflexiv_cuda.h: rfx_stitch_begin_sharded / rfx_stitch_finish_sharded): every rank holds a shard
of the table and any part of the reads; the union of the ranks' stitched records must equal, as a multiset of (sequence, left,
right), the oracle and rfx_stitch_begin / rfx_stitch_finish on one context, for every split of rows and reads.

Ranks are host threads of one process sharing device 0 (runs on a one-GPU box); the last test maps the arenas of one process
per GPU through CUDA IPC (needs >= 2 GPUs)."""
import functools
import os
import sys
import time

import numpy as np
import pytest

from test_stitch import _gpu_stitch, assembled, gap_scenario, natural_scenario, random_scenarios, triples

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
ARENA = 1 << 30


@pytest.fixture(scope="module")
def R():
    import reflexiv_b200 as R
    return R


def records(txt):
    """FASTQ text -> its 4-line records (bytes each)."""
    lines = txt.split(b"\n")
    if lines and lines[-1] == b"":
        lines = lines[:-1]
    return [b"\n".join(lines[i:i + 4]) + b"\n" for i in range(0, len(lines), 4)]


def split_reads(txt, world, seed, empty_rank=None):
    """Uneven split on record boundaries; `empty_rank` gets nothing."""
    recs = records(txt)
    rng = np.random.default_rng(seed)
    takers = [r for r in range(world) if r != empty_rank] or [0]
    owner = np.asarray(takers)[rng.choice(len(takers), len(recs), p=np.arange(1, len(takers) + 1) / sum(range(1, len(takers) + 1)))]
    return [b"".join(recs[i] for i in np.flatnonzero(owner == r)) for r in range(world)]


@functools.lru_cache(maxsize=None)
def _table(txt, k, cover):
    """The filtered count table of one context, in the reference key layout rfx_load_counts takes."""
    import reflexiv_b200 as R
    with R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=cover), device=0) as ctx:
        ctx.push_fastq(txt)
        ctx.count()
        return ctx.counts()


def _ctxs(R, world, k, cover=3, min_contig=0):
    return [R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=cover, minContig=min_contig), device=0) for _ in range(world)]


def _push(ctx, part, device):
    if not part:
        return
    if device:
        import torch
        n = len(part)
        d = torch.zeros((n + 127) // 64 * 64, dtype=torch.uint8, device="cuda:0")
        d[:n] = torch.frombuffer(bytearray(part), dtype=torch.uint8).cuda()
        torch.cuda.synchronize()
        ctx.push_fastq_device(d.data_ptr(), n)
    else:
        ctx.push_fastq(part)


def stitch_body(txt, k, cover, read_parts, table="load", device_reads=False, seed=0, cuts=None):
    """One sharded run: the table (slices of the one-context table cut at `cuts`, or at random, re-sharded; or counted across
    the ranks from `read_parts`), begin, each rank's reads, finish."""
    world = len(read_parts)
    if table == "load":
        keys, cnt = _table(txt, k, cover)
        if cuts is None:
            rng = np.random.default_rng(seed)
            cuts = [0] + sorted(rng.integers(0, len(cnt) + 1, world - 1).tolist()) + [len(cnt)]

    def body(rank, ctx):
        ctx.reset()
        if table == "load":
            ctx.load_counts(keys[cuts[rank]:cuts[rank + 1]], cnt[cuts[rank]:cuts[rank + 1]])
            ctx.shard_table()
        else:
            if read_parts[rank]:
                ctx.push_fastq(read_parts[rank])
            ctx.count_sharded()
        st0 = ctx.stitch_begin_sharded()
        _push(ctx, read_parts[rank], device_reads)
        st = ctx.stitch_finish_sharded()
        return dict(st0=st0, st=st, contigs=ctx.contigs(), sh=ctx.shard_stats())
    return body


def run_sharded(R, body, world, k, min_contig=0, cover=3, arena=ARENA):
    from reflexiv_b200 import sharded
    ctxs = _ctxs(R, world, k, cover, min_contig)
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=arena)
        return grp.run(body)
    finally:
        for c in ctxs:
            c.close()


def union(res):
    return sorted(x for r in res for x in r["contigs"])


STATS = ["n_probes", "n_fragments", "n_after_pass1", "n_joined", "n_stitched", "n_rings"]


def check_stats(res, want_stats, n_reads=None):
    """n_fragments, n_stitched, n_rings (and n_reads) add up over the ranks; n_probes, n_after_pass1, n_joined are global."""
    want = dict(zip(STATS, want_stats))
    for r in res:
        for s in ("n_probes", "n_after_pass1", "n_joined"):
            assert r["st"][s] == want[s], (s, r["st"], want)
        assert r["st0"]["n_probes"] == want["n_probes"]
    for s in ("n_fragments", "n_stitched", "n_rings"):
        assert sum(r["st"][s] for r in res) == want[s], (s, [r["st"] for r in res], want)
    if n_reads is not None:
        assert sum(r["st"]["n_reads"] for r in res) == n_reads
    n_global = res[0]["sh"]["n_contigs_global"]
    assert all(r["sh"]["n_contigs_global"] == n_global for r in res) and n_global == sum(len(r["contigs"]) for r in res)
    assert all(r["sh"]["n_contig_bases_global"] == sum(len(s) for x in res for s, _, _ in x["contigs"]) for r in res)


def _scenarios():
    return [(31, gap_scenario(5, 6000, 100, [(2000, 2060), (4000, 4070)])[1]), (31, gap_scenario(6, 6000, 100, [(2000, 2060), (4000, 4070)], err=0.02)[1]),
            (21, gap_scenario(7, 3000, 80, [(1000, 1050), (2000, 2040)], circular=True)[1])] + list(random_scenarios(6))


def test_sharded_stitch_matches_oracle_and_one_context(R, orc, monkeypatch):
    stitched = rings = 0
    for i, (k, txt) in enumerate(_scenarios()):
        contigs, left, right = assembled(txt, k)
        for min_contig in (0, 300):
            want = orc.stitch(contigs, left, right, txt, k, min_contig=min_contig)
            one, one_st = _gpu_stitch(txt, k, min_contig=min_contig)
            assert one == triples(want)
            for world in (1, 2, 3, 4):
                table = "count" if (i == 1 and world == 3) else "load"
                empty = i % world if world > 1 and table == "load" else None
                parts = split_reads(txt, world, seed=10 * i + world, empty_rank=empty)
                if (i + world) % 3 == 0:
                    monkeypatch.setenv("RFX_FASTQ_CHUNK_BYTES", "4096")  # many chunks: fragments accumulate across them
                res = run_sharded(R, stitch_body(txt, k, 3, parts, table=table, seed=i + world), world, k, min_contig)
                monkeypatch.delenv("RFX_FASTQ_CHUNK_BYTES", raising=False)
                assert union(res) == one, (i, k, min_contig, world, table)
                check_stats(res, list(want["stats"].values()), one_st["n_reads"])
                if empty is not None:
                    assert res[empty]["st"]["n_reads"] == 0 and res[empty]["st"]["n_fragments"] == 0
        stitched += want["stats"]["stitched_records"]
        rings += want["stats"]["rings"]
    assert stitched > 10 and rings > 0


def test_chains_cross_ranks(R, orc):
    """At least one stitched record is made of plain contigs that two different ranks hold (found from a plain
    assemble_sharded(min_contig=0) on the same split, by substring test)."""
    k = 31
    txt = natural_scenario(300_000, 8)
    world = 3
    keys, cnt = _table(txt, k, 3)
    cuts = [0, len(cnt) // 3, 2 * len(cnt) // 3, len(cnt)]

    def plain(rank, ctx):
        ctx.reset()
        ctx.load_counts(keys[cuts[rank]:cuts[rank + 1]], cnt[cuts[rank]:cuts[rank + 1]])
        ctx.shard_table()
        ctx.assemble_sharded()
        return [s for s, _, _ in ctx.contigs()]
    held = run_sharded(R, plain, world, k)
    res = run_sharded(R, stitch_body(txt, k, 3, split_reads(txt, world, seed=3), cuts=cuts), world, k)
    contigs, left, right = assembled(txt, k)
    want = orc.stitch(contigs, left, right, txt, k, min_contig=0)
    assert union(res) == triples(want)
    owner = {s: r for r, ss in enumerate(held) for s in ss}
    rc = orc.revcomp_str
    cross = 0
    for r in res:
        for s, _, _ in r["contigs"]:
            holders = {o for c, o in owner.items() if c != s and (c in s or rc(c) in s)}
            cross += len(holders) > 1
    assert cross > 0


def test_thinly_covered_reads(R, orc, monkeypatch):
    for glen, cov, err in ((1_000_000, 8, 0.0), (400_000, 10, 0.005)):
        txt = natural_scenario(glen, cov, err=err)
        contigs, left, right = assembled(txt, 31)
        want = orc.stitch(contigs, left, right, txt, 31, min_contig=200)
        one, _ = _gpu_stitch(txt, 31, min_contig=200)
        assert one == triples(want)
        for world in (2, 4):
            parts = split_reads(txt, world, seed=world, empty_rank=world - 1 if world == 4 else None)
            monkeypatch.setenv("RFX_FASTQ_CHUNK_BYTES", str(8 << 20))
            res = run_sharded(R, stitch_body(txt, 31, 3, parts, seed=world), world, 31, min_contig=200)
            monkeypatch.delenv("RFX_FASTQ_CHUNK_BYTES", raising=False)
            assert union(res) == one
            check_stats(res, list(want["stats"].values()))
            assert sum(r["st"]["n_stitched"] for r in res) > 100


def test_rings_and_the_closed_path_fallback(R, orc):
    """A circular genome with a bridged gap: rings; and a table whose sharded assembly falls back to rank 0 (a closed path:
    a circular genome without a gap), so that rank 0 holds every contig and the other ranks none."""
    k = 21
    txt = gap_scenario(7, 3000, 80, [(1000, 1050), (2000, 2040)], circular=True)[1]
    contigs, left, right = assembled(txt, k)
    want = orc.stitch(contigs, left, right, txt, k, min_contig=0)
    assert want["stats"]["rings"] > 0
    for world in (2, 3):
        res = run_sharded(R, stitch_body(txt, k, 3, split_reads(txt, world, seed=world), seed=world), world, k)
        assert union(res) == triples(want)
        check_stats(res, list(want["stats"].values()))
    # closed path somewhere (a whole circular genome at full coverage) next to a bridged gap on a linear one
    from workload import synth
    g = bytes(synth.genome(2000, 9)).decode()
    circ = g + g[:200]
    extra = [circ[i:i + 120] for i in range(0, 2000, 7)] * 2
    txt2 = gap_scenario(5, 6000, 100, [(2000, 2060), (4000, 4070)], extra=extra)[1]
    contigs, left, right = assembled(txt2, 31)
    want = orc.stitch(contigs, left, right, txt2, 31, min_contig=0)
    assert want["stats"]["stitched_records"] > 0
    one, _ = _gpu_stitch(txt2, 31)
    res = run_sharded(R, stitch_body(txt2, 31, 3, split_reads(txt2, 2, seed=5), seed=5), 2, 31)
    assert any(r["sh"]["fell_back"] for r in res)
    assert union(res) == one
    assert one == triples(want)
    check_stats(res, list(want["stats"].values()))


def test_k_above_31_is_the_sharded_plain_assembly(R):
    k = 41
    txt = gap_scenario(5, 3000, 100, [(1500, 1560)])[1]
    keys, cnt = _table(txt, k, 3)
    world = 2
    cuts = [0, len(cnt) // 2, len(cnt)]

    def plain(rank, ctx):
        ctx.reset()
        ctx.load_counts(keys[cuts[rank]:cuts[rank + 1]], cnt[cuts[rank]:cuts[rank + 1]])
        ctx.shard_table()
        ctx.assemble_sharded()
        return dict(contigs=ctx.contigs())

    def stitched(rank, ctx):
        ctx.reset()
        ctx.load_counts(keys[cuts[rank]:cuts[rank + 1]], cnt[cuts[rank]:cuts[rank + 1]])
        ctx.shard_table()
        st0 = ctx.stitch_begin_sharded()
        ctx.push_fastq(txt)
        st = ctx.stitch_finish_sharded()
        return dict(st0=st0, st=st, contigs=ctx.contigs())
    want = union(run_sharded(R, plain, world, k, min_contig=100))
    res = run_sharded(R, stitched, world, k, min_contig=100)
    assert all(r["st0"]["n_probes"] == 0 and r["st"]["n_probes"] == 0 and r["st"]["n_fragments"] == 0 and r["st"]["n_reads"] > 0 for r in res)
    assert union(res) == want and len(want) > 0


def test_reads_pushed_from_device_memory(R, orc):
    k, txt = 31, gap_scenario(6, 6000, 100, [(2000, 2060), (4000, 4070)], err=0.02)[1]
    contigs, left, right = assembled(txt, k)
    want = orc.stitch(contigs, left, right, txt, k, min_contig=500)
    for world in (2, 3):
        res = run_sharded(R, stitch_body(txt, k, 3, split_reads(txt, world, seed=world + 7, empty_rank=1), device_reads=True, seed=1), world, k, min_contig=500)
        assert union(res) == triples(want)
        check_stats(res, list(want["stats"].values()))


def test_errors_come_back_from_every_rank_at_once(R, orc):
    from reflexiv_b200 import _lib, sharded
    k = 31
    txt = gap_scenario(5, 6000, 100, [(2000, 2060), (4000, 4070)])[1]
    contigs, left, right = assembled(txt, k)
    want = triples(orc.stitch(contigs, left, right, txt, k, min_contig=0))
    keys, cnt = _table(txt, k, 3)
    # contexts without an arena
    with R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=3), device=0) as ctx:
        ctx.load_counts(keys, cnt)
        for call in (ctx.stitch_begin_sharded, ctx.stitch_finish_sharded):
            with pytest.raises(_lib.RfxError) as e:
                call()
            assert e.value.code == _lib.RFX_E_STATE
    world = 3
    parts = split_reads(txt, world, seed=1)
    cuts = [0, len(cnt) // 3, 2 * len(cnt) // 3, len(cnt)]
    ctxs = _ctxs(R, world, k)
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=ARENA)

        def load(rank, ctx):
            ctx.reset()
            ctx.load_counts(keys[cuts[rank]:cuts[rank + 1]], cnt[cuts[rank]:cuts[rank + 1]])
            ctx.shard_table()

        def good(rank, ctx):
            load(rank, ctx)
            ctx.stitch_begin_sharded()
            _push(ctx, parts[rank], False)
            ctx.stitch_finish_sharded()
            return ctx.contigs()

        def codes(fn):
            def body(rank, ctx):
                try:
                    fn(rank, ctx)
                except _lib.RfxError as err:
                    return err.code
                return 0
            t0 = time.perf_counter()
            out = grp.run(body)
            assert time.perf_counter() - t0 < 10.0  # caught by an exchange: nobody waits for a barrier to time out
            return out

        def case_no_table(rank, ctx):
            load(rank, ctx)
            if rank == 1:
                ctx.reset()
            ctx.stitch_begin_sharded()

        def case_finish_without_begin(rank, ctx):
            load(rank, ctx)
            ctx.stitch_finish_sharded()

        def case_abandoned(rank, ctx):
            load(rank, ctx)
            ctx.stitch_begin_sharded()
            ctx.shard_table()  # abandons the open stage
            ctx.stitch_finish_sharded()

        def case_one_rank_not_open(rank, ctx):
            load(rank, ctx)
            ctx.stitch_begin_sharded()
            if rank == 0:
                ctx.reset()
            ctx.stitch_finish_sharded()

        # after every error the next collective call on the same contexts succeeds
        for case in (case_no_table, case_finish_without_begin, case_abandoned, case_one_rank_not_open):
            assert codes(case) == [_lib.RFX_E_STATE] * world, case.__name__
            assert union([dict(contigs=c) for c in grp.run(good)]) == want, case.__name__

        # the single-context calls on a sharded stage: refused, the stage stays open and the sharded finish completes it
        def single_calls(rank, ctx):
            ctx.reset()
            ctx.load_counts(keys[cuts[rank]:cuts[rank + 1]], cnt[cuts[rank]:cuts[rank + 1]])
            ctx.shard_table()
            ctx.stitch_begin_sharded()
            with pytest.raises(_lib.RfxError) as e:
                ctx.stitch_finish()
            assert e.value.code == _lib.RFX_E_STATE
            with pytest.raises(_lib.RfxError) as e:
                ctx.stitch_begin()  # the one-context begin on a sharded context
            assert e.value.code == _lib.RFX_E_UNSUPPORTED
            _push(ctx, parts[rank], False)
            ctx.stitch_finish_sharded()
            return ctx.contigs()
        assert union([dict(contigs=c) for c in grp.run(single_calls)]) == want
    finally:
        for c in ctxs:
            c.close()
    # one rank with another min_contig: caught in the first exchange, before the assembly; the same contexts then assemble
    ctxs = [R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=3, minContig=300 if r == 2 else 0), device=0) for r in range(world)]
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=ARENA)

        def begin(rank, ctx):
            ctx.reset()
            ctx.load_counts(keys[cuts[rank]:cuts[rank + 1]], cnt[cuts[rank]:cuts[rank + 1]])
            ctx.shard_table()
            try:
                ctx.stitch_begin_sharded()
            except _lib.RfxError as err:
                return err.code
            return 0
        assert grp.run(begin) == [_lib.RFX_E_INVALID] * world

        def plain(rank, ctx):
            ctx.shard_table()
            ctx.assemble_sharded()
            return len(ctx.contigs())
        assert sum(grp.run(plain)) > 0
    finally:
        for c in ctxs:
            c.close()


def test_same_contexts_twice(R, orc):
    """Stitch across ranks, then reset -> count_sharded -> assemble_sharded on the same contexts: the plain result equals a
    fresh run (arena reuse, barrier epochs)."""
    from reflexiv_b200 import sharded
    k, world = 31, 3
    txt = gap_scenario(5, 6000, 100, [(2000, 2060), (4000, 4070)])[1]
    contigs, left, right = assembled(txt, k)
    want = triples(orc.stitch(contigs, left, right, txt, k, min_contig=0))
    parts = split_reads(txt, world, seed=2)

    def plain(rank, ctx):
        ctx.reset()
        ctx.push_fastq(parts[rank])
        ctx.count_sharded()
        ctx.assemble_sharded()
        return dict(contigs=ctx.contigs())
    fresh = union(run_sharded(R, plain, world, k))
    ctxs = _ctxs(R, world, k)
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=ARENA)
        for _ in range(2):
            assert union(grp.run(stitch_body(txt, k, 3, parts, seed=4))) == want
            assert union(grp.run(plain)) == fresh
    finally:
        for c in ctxs:
            c.close()


# ---- one process per GPU, arenas mapped through CUDA IPC ------------------------------------------------------------------
def _worker(rank, world, port, out_dir):
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
    z = np.load(os.path.join(out_dir, "input.npz"))
    txt = z["txt"].tobytes()
    keys, cnt = z["keys"], z["cnt"]
    n = len(cnt)
    ctx = R.ReflexivContext(R.DefaultParam(kmerSize=31, minKmerCoverage=3, minContig=200), device=rank)
    sharded.connect(ctx, dist, arena_bytes=2 << 30)
    ctx.reset()
    ctx.load_counts(keys[n * rank // world:n * (rank + 1) // world], cnt[n * rank // world:n * (rank + 1) // world])
    ctx.shard_table()
    ctx.stitch_begin_sharded()
    ctx.push_fastq(split_reads(txt, world, seed=9)[rank])
    st = ctx.stitch_finish_sharded()
    with open(os.path.join(out_dir, f"res_{rank}.pkl"), "wb") as f:
        pickle.dump(dict(st=st, contigs=ctx.contigs()), f)
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


def test_one_process_per_gpu_over_ipc(tmp_path, orc):
    import pickle
    import torch
    import torch.multiprocessing as mp
    world = torch.cuda.device_count()
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    world = min(world, 4)
    txt = natural_scenario(400_000, 8)
    keys, cnt = _table(txt, 31, 3)
    np.savez(tmp_path / "input.npz", txt=np.frombuffer(txt, np.uint8), keys=keys, cnt=cnt)
    port = 29900 + os.getpid() % 1000
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    res = [pickle.load(open(tmp_path / f"res_{r}.pkl", "rb")) for r in range(world)]
    contigs, left, right = assembled(txt, 31)
    want = orc.stitch(contigs, left, right, txt, 31, min_contig=200)
    assert union(res) == triples(want)
    assert sum(r["st"]["n_stitched"] for r in res) == want["stats"]["stitched_records"]
