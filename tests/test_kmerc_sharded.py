"""A loaded Count_<k> table assembled across ranks (include/reflexiv_cuda.h: rfx_shard_table): every rank loads any slice of
the table, rfx_shard_table sends every row to the rank that owns its minimiser bin, rfx_assemble_sharded assembles the
shards.  The union of the shard tables must be the loaded multiset, the shards disjoint, and fork-filter survivors,
contigs and budget / cycle statistics equal to the oracle and to rfx_load_counts + rfx_assemble on one context.

Ranks are host threads of one process sharing device 0 (runs on a one-GPU box); the last test maps the arenas of one
process per GPU through CUDA IPC (needs >= 2 GPUs)."""
import functools
import os
import sys
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def R():
    import reflexiv_b200 as R
    return R


def _genome_reads(k, err, seed=0, glen=30_000, pairs=6000, at=False):
    from workload import synth
    g = synth.genome(glen, 400 + k + seed)
    if glen >= 13000:
        g[12000:12800] = g[3000:3800]    # repeat: real forks, budget junctions
    if at:
        g[20000:20040] = np.frombuffer(b"AT" * 20, np.uint8)  # palindromic low-complexity stretch: closed paths
    return bytes(synth.fastq(g, pairs, read_len=150, frag_len=400, error_rate=err, seed_reads=5 + seed, seed_errors=6 + seed))


def _oracle_table(orc, txt, k, cover):
    starts, lens = orc.fastq_reads(txt, orc.FASTQ_RUN)
    return orc.count_kmers(txt, starts, lens, k, 0, 0, cover, 10_000_000, 1)


def _ref_layout(t, k):
    """Oracle rows (128-bit split keys) -> the reference key layout rfx_load_counts takes."""
    hi, lo = t["keys_hi"].astype(np.uint64), t["keys_lo"].astype(np.uint64)
    if k <= 31:
        return lo.reshape(-1, 1).copy()
    res = k % 32
    w0 = (hi << np.uint64(64 - 2 * res)) | (lo >> np.uint64(2 * res))
    w1 = lo & np.uint64((1 << (2 * res)) - 1)
    return np.stack([w0, w1], axis=1)


@functools.lru_cache(maxsize=None)
def _table(k, at=False):
    from oracle import orc
    orc.lib()
    txt = _genome_reads(k, 0.01, at=at)
    t = _oracle_table(orc, txt, k, 2)
    return txt, t, _ref_layout(t, k), t["counts"].astype(np.uint32)


def _contiguous(keys, cnt, world):
    n = len(cnt)
    return [(keys[n * r // world:n * (r + 1) // world], cnt[n * r // world:n * (r + 1) // world]) for r in range(world)]


def _load_body(slices, results, bins=0):
    def body(rank, ctx):
        ctx.reset()
        ctx.load_counts(*slices[rank])
        if bins:
            ctx.shard_set_bins(bins)
        st = ctx.shard_table()
        keys, cnt = ctx.counts()
        st2 = ctx.assemble_sharded()
        sh = ctx.shard_stats()
        ori = ctx.oriented() if not sh["fell_back"] else None
        results[rank] = dict(keys=keys, cnt=cnt, st=st, st2=st2, sh=sh, ori=ori, contigs=ctx.contigs())
    return body


def _check_against_oracle(orc, t, k, E, min_contig, results):
    from reflexiv_b200.pipeline import keys_to_int
    f = orc.fork_filter(t["keys_hi"], t["keys_lo"], t["counts"], k, E)
    a = orc.assemble(f["keys_hi"], f["keys_lo"], f["left"], f["right"], k, min_contig, orc.ASM_CANONICAL)
    ref_ints = [(int(h) << 64) | int(l) for h, l in zip(t["keys_hi"], t["keys_lo"])]
    got = {}
    for res in results:
        for key, n in zip(keys_to_int(res["keys"], k), res["cnt"].tolist()):
            assert key not in got  # shard tables are disjoint
            got[key] = n
    assert sorted(got) == ref_ints
    assert [got[x] for x in ref_ints] == t["counts"].tolist()
    assert sum(r["st"]["n_rows"] for r in results) == len(ref_ints)
    fell_back = any(r["sh"]["fell_back"] for r in results)
    if not fell_back:
        hi = np.concatenate([r["ori"][0] for r in results]); lo = np.concatenate([r["ori"][1] for r in results])
        le = np.concatenate([r["ori"][2] for r in results]); ri = np.concatenate([r["ori"][3] for r in results])
        order = np.lexsort((lo, hi))
        assert np.array_equal(hi[order], f["keys_hi"]) and np.array_equal(lo[order], f["keys_lo"])
        assert np.array_equal(le[order], f["left"]) and np.array_equal(ri[order], f["right"])
    got_c = sorted((s, l, r) for res in results for s, l, r in res["contigs"])
    exp_c = sorted(zip(a["contigs"], a["left"].tolist(), a["right"].tolist()))
    assert got_c == exp_c
    tot = lambda name: sum(r["st2"][name] for r in results)  # noqa: E731
    assert tot("n_oriented") == len(f["left"])
    assert (tot("n_budget_junctions"), tot("n_budget_admissible"), tot("n_cycles")) == (a["n_budget_junctions"], a["n_budget_admissible"], a["n_cycles"])
    assert results[0]["sh"]["n_contigs_global"] == len(a["contigs"])
    return a, fell_back


def _ctxs(R, world, k, cover=2, E=8, min_contig=100):
    return [R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=cover, minErrorCoverage=E, minContig=min_contig), device=0) for _ in range(world)]


def _run_loaded(R, slices, k, bins=0, arena=1 << 30, min_contig=100):
    from reflexiv_b200 import sharded
    ctxs = _ctxs(R, len(slices), k, min_contig=min_contig)
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=arena)
        results = [None] * len(slices)
        grp.run(_load_body(slices, results, bins))
    finally:
        for c in ctxs:
            c.close()
    return results


def _single(R, keys, cnt, k, min_contig=100):
    with R.ReflexivContext(R.DefaultParam(kmerSize=k, minContig=min_contig), device=0) as ctx:
        ctx.load_counts(keys, cnt)
        ctx.assemble()
        return sorted(ctx.contigs())


@pytest.mark.parametrize("k", [21, 24, 31, 61])
@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_loaded_table_matches_oracle_and_one_gpu(R, orc, world, k):
    txt, t, keys, cnt = _table(k, at=(k == 24))
    results = _run_loaded(R, _contiguous(keys, cnt, world), k)
    a, fell_back = _check_against_oracle(orc, t, k, 8, 100, results)
    assert len(a["contigs"]) >= 2
    assert sorted(x for r in results for x in r["contigs"]) == _single(R, keys, cnt, k)
    assert all(r["sh"]["n_rows_global"] == len(cnt) for r in results)
    if world > 1:
        assert all(r["st"]["n_rows"] > 0 for r in results)  # every rank owns bins with rows


def test_uneven_slices(R, orc):
    txt, t, keys, cnt = _table(31)
    n, world = len(cnt), 3
    empty = (keys[:0], cnt[:0])
    rng = np.random.default_rng(7)
    perm = rng.permutation(n)
    cuts = sorted(rng.choice(np.arange(1, n), world - 1, replace=False).tolist())
    bounds = [0] + cuts + [n]
    cases = [
        [(keys, cnt), empty, empty],                                                                       # all on rank 0
        [(keys[perm[bounds[r]:bounds[r + 1]]], cnt[perm[bounds[r]:bounds[r + 1]]]) for r in range(world)],  # random order, random cuts
        [(keys[:1], cnt[:1]), (keys[1:n // 2], cnt[1:n // 2]), (keys[n // 2:], cnt[n // 2:])],             # one rank with one row
    ]
    for slices in cases:
        _check_against_oracle(orc, t, 31, 8, 100, _run_loaded(R, slices, 31))


def test_explicit_bins_same_contigs(R, orc):
    txt, t, keys, cnt = _table(31)
    auto = _run_loaded(R, _contiguous(keys, cnt, 2), 31)
    fixed = _run_loaded(R, _contiguous(keys, cnt, 2), 31, bins=2 * 300)
    assert all(r["st"]["n_bins"] == 600 for r in fixed)
    assert len({r["st"]["n_bins"] for r in auto}) == 1 and auto[0]["st"]["n_bins"] % 2 == 0
    _check_against_oracle(orc, t, 31, 8, 100, fixed)
    assert sorted(x for r in auto for x in r["contigs"]) == sorted(x for r in fixed for x in r["contigs"])


def test_reads_then_table_then_reads_on_the_same_contexts(R, orc):
    """Arena reuse and barrier epochs: count_sharded + assemble_sharded, load_counts + shard_table + assemble_sharded, the first again."""
    from reflexiv_b200 import sharded
    txt, t, keys, cnt = _table(31)
    world = 3
    cuts = [0] + [txt.find(b"\n@r", len(txt) * r // world) + 1 for r in range(1, world)] + [len(txt)]
    parts = [txt[cuts[r]:cuts[r + 1]] for r in range(world)]

    def from_reads(results):
        def body(rank, ctx):
            ctx.reset()
            ctx.push_fastq(parts[rank])
            st = ctx.count_sharded()
            k2, c2 = ctx.counts()
            st2 = ctx.assemble_sharded()
            sh = ctx.shard_stats()
            results[rank] = dict(keys=k2, cnt=c2, st=st, st2=st2, sh=sh, ori=ctx.oriented() if not sh["fell_back"] else None, contigs=ctx.contigs())
        return body

    ctxs = _ctxs(R, world, 31)
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=1 << 30)
        for step in ("reads", "table", "reads"):
            results = [None] * world
            grp.run(from_reads(results) if step == "reads" else _load_body(_contiguous(keys, cnt, world), results))
            _check_against_oracle(orc, t, 31, 8, 100, results)
    finally:
        for c in ctxs:
            c.close()


def _tiled_table(orc, glen, seed, circular):
    """Error-free reads tiling a genome of glen bases every 7 bases, twice: oracle table and its rfx_load_counts layout."""
    from workload import synth
    g = bytes(synth.genome(glen, seed))
    src = g + g[:200] if circular else g
    reads = [src[i:i + 120] for i in range(0, glen if circular else glen - 119, 7)] * 2
    txt = "".join(f"@r{i}\n{r.decode()}\n+\n{'I' * len(r)}\n" for i, r in enumerate(reads)).encode()
    t = _oracle_table(orc, txt, 31, 2)
    return t, _ref_layout(t, 31), t["counts"].astype(np.uint32)


def test_closed_paths(R, orc):
    """A circular genome has no head: the sharded assembly falls back to rank 0 assembling the whole table."""
    t, keys, cnt = _tiled_table(orc, 2000, 9, circular=True)
    results = _run_loaded(R, _contiguous(keys, cnt, 2), 31, min_contig=50)
    a, fell_back = _check_against_oracle(orc, t, 31, 8, 50, results)
    assert fell_back and a["n_cycles"] >= 1


def test_closed_paths_fallback_failing_on_rank_0_fails_on_every_rank_at_once(R, orc):
    """The arena holds everything both ranks need up to the whole-table fallback, not rank 0's copy of the whole table and
    the single-GPU stages on it: every rank returns rank 0's RFX_E_NOMEM within seconds, and the contexts stay usable."""
    from reflexiv_b200 import _lib, sharded
    t, keys, cnt = _tiled_table(orc, 2000, 9, circular=True)
    slices = _contiguous(keys, cnt, 2)
    # how much of the arena every rank uses, from a run in a large arena (the layout of a bump allocator is deterministic);
    # only rank 0 reserves anything in the fallback
    used = [r["sh"]["arena_used"] for r in _run_loaded(R, slices, 31, min_contig=50)]
    arena = (used[0] - 1) & ~4095  # rfx_shard_init rounds up to 4 KiB: below what rank 0 needs at the end of its fallback
    assert max(used[1:]) <= arena, (used, arena)  # ... and above what rank 1 needs, and rank 0 before the fallback

    ctxs = _ctxs(R, 2, 31, min_contig=50)
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=arena)

        def body(rank, ctx):
            ctx.reset()
            ctx.load_counts(*slices[rank])
            ctx.shard_table()
            try:
                ctx.assemble_sharded()
            except _lib.RfxError as err:
                return err
            return None
        t0 = time.perf_counter()
        errs = grp.run(body)
        took = time.perf_counter() - t0
        assert all(e is not None and e.code == _lib.RFX_E_NOMEM for e in errs), errs
        assert "arena exhausted" in str(errs[0]) and "rank 0" in str(errs[1])
        assert took < 5.0  # the fallback's exchange carries rank 0's status: rank 1 does not wait for a barrier to time out
        assert ctxs[0].shard_stats()["fell_back"] and ctxs[1].shard_stats()["fell_back"]
        # the ranks stay in step: the same contexts then assemble a linear genome correctly
        t2, keys2, cnt2 = _tiled_table(orc, 1000, 10, circular=False)
        results = [None] * 2
        grp.run(_load_body(_contiguous(keys2, cnt2, 2), results))
        _check_against_oracle(orc, t2, 31, 8, 50, results)
    finally:
        for c in ctxs:
            c.close()


def test_errors_come_back_from_every_rank_at_once(R, orc):
    from reflexiv_b200 import _lib, sharded
    with R.ReflexivContext(R.DefaultParam(kmerSize=31), device=0) as ctx:
        ctx.load_counts(np.zeros((1, 1), np.uint64), np.ones(1, np.uint32))
        with pytest.raises(_lib.RfxError) as e:
            ctx.shard_table()
        assert e.value.code == _lib.RFX_E_STATE
    txt, t, keys, cnt = _table(31)
    world = 3
    slices = _contiguous(keys, cnt, world)
    ctxs = _ctxs(R, world, 31)
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=1 << 30)
        # rank 1 holds no table: it never loads one (shard_table), or it drops its shard before the assembly
        for case in ("shard_table", "assemble_sharded"):
            def body(rank, ctx):
                ctx.reset()
                if rank != 1 or case == "assemble_sharded":
                    ctx.load_counts(*slices[rank])
                try:
                    ctx.shard_table()
                    if case == "assemble_sharded":
                        if rank == 1:
                            ctx.reset()
                        ctx.assemble_sharded()
                except _lib.RfxError as err:
                    return err.code
                return 0
            t0 = time.perf_counter()
            codes = grp.run(body)
            assert codes == [_lib.RFX_E_STATE] * world, case
            assert time.perf_counter() - t0 < 5.0  # the first exchange catches it: nobody waits for a barrier to time out
            # the ranks stay in step: the same contexts then re-shard and assemble correctly
            results = [None] * world
            grp.run(_load_body(slices, results))
            _check_against_oracle(orc, t, 31, 8, 100, results)
    finally:
        for c in ctxs:
            c.close()


def _parts(d):
    return sorted(f for f in os.listdir(d) if f.startswith("part-"))


def _records(d):
    import gzip
    text = "".join((gzip.open(d / f).read().decode() if f.endswith(".gz") else (d / f).read_text()) for f in _parts(d))
    recs = text.strip().split(">")[1:]
    return [x.split("\n")[0] for x in recs], ["".join(x.strip().split("\n")[1:]) for x in recs]


@pytest.mark.parametrize("gz", [False, True])
def test_reflexiv_binary_kmerc_with_gpus_option(tmp_path, orc, golden, gz):
    """`reflexiv run -kmerc <Count_31> --gpus 3` (csrc/reflexiv_main.cpp: run_kmerc_sharded): one part file per rank, the
    same contig set as the one-GPU -kmerc run."""
    import subprocess
    from conftest import GOLDEN
    exe = os.path.join(ROOT, "reflexiv_b200", "reflexiv")
    env = dict(os.environ, REFLEXIV_ARENA_MB="768", CUDA_MODULE_LOADING="EAGER", CUDA_DEVICE_MAX_CONNECTIONS="32")
    cout = tmp_path / "c"
    r = subprocess.run([exe, "counter", "-fastq", os.path.join(GOLDEN, "paired_dat*.fq.gz"), "-outfile", str(cout), "-kmer", "31"], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr + r.stdout
    table = str(cout / "Count_31" / "part*")
    extra = ["-gzip"] if gz else []
    outs = {}
    for gpus in (3, 1):
        out = tmp_path / f"r{gpus}"
        r = subprocess.run([exe, "run", "--gpus", str(gpus), "-kmerc", table, "-outfile", str(out), "-kmer", "31", "-cover", "3"] + extra,
                           capture_output=True, text=True, env=env)
        assert r.returncode == 0, r.stderr + r.stdout
        assert "--gpus" not in r.stderr, r.stderr
        d = out / "Assemble_31"
        assert (d / "_SUCCESS").exists()
        assert len(_parts(d)) == gpus and all(f.endswith(".gz") == gz for f in _parts(d))
        outs[gpus] = _records(d)
    heads, seqs = outs[3]
    assert sorted(heads) == ["Contig-4558-(-4,-4)-0", "Contig-4558-(-4,-4)-1"]
    assert sum(s.startswith(golden["documented"]["prefix_1200"]) for s in seqs) == 1
    assert orc.canonical_contig_set(seqs) == orc.canonical_contig_set(outs[1][1])


# ---- one process per GPU, arenas mapped through CUDA IPC ------------------------------------------------------------------
def _worker(rank, world, port, k, out_dir):
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
    z = np.load(os.path.join(out_dir, "table.npz"))
    ctx = R.ReflexivContext(R.DefaultParam(kmerSize=k, minContig=200), device=rank)
    sharded.connect(ctx, dist, arena_bytes=2 << 30)
    results = [None] * world
    _load_body(_contiguous(z["keys"], z["cnt"], world), results)(rank, ctx)
    with open(os.path.join(out_dir, f"res_{rank}.pkl"), "wb") as f:
        pickle.dump(results[rank], f)
    dist.barrier()
    ctx.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("k", [31, 61])
def test_one_process_per_gpu_over_ipc(tmp_path, orc, k):
    import pickle
    import torch
    import torch.multiprocessing as mp
    world = torch.cuda.device_count()
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    world = min(world, 4)
    txt = _genome_reads(k, 0.005, glen=60_000, pairs=12_000)
    t = _oracle_table(orc, txt, k, 2)
    np.savez(tmp_path / "table.npz", keys=_ref_layout(t, k), cnt=t["counts"].astype(np.uint32))
    port = 29800 + os.getpid() % 1000 + k
    mp.spawn(_worker, args=(world, port, k, str(tmp_path)), nprocs=world, join=True)
    results = [pickle.load(open(tmp_path / f"res_{r}.pkl", "rb")) for r in range(world)]
    _check_against_oracle(orc, t, k, 8, 200, results)
