"""Count_<k>_sorted across ranks (include/reflexiv_cuda.h: rfx_sort_kmers_sharded): every rank holds its shard of a table
sharded by minimiser bin (rfx_shard_table or rfx_count_sharded), the two fork filters of the sorting stage run across the
ranks, every rank keeps the sorted rows of its own shard.  The union must equal the oracle's restatement of
ReflexivDSKmerLeftAndRightSorting and rfx_sort_kmers on one context holding the whole table, bit for bit.

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

# the cases of test_gpu_parity.py::test_sorted_stage_matches_oracle: (k, E, fold, kmax, cover, err)
CASES = [(31, 8, 1.5, 95, 1, 0.01), (31, 6, 2.0, 31, 2, 0.01), (23, 8, 1.5, 95, 1, 0.02),
         (41, 8, 1.5, 95, 1, 0.01), (53, 24, 2.0, 95, 1, 0.005), (12, 3, 1.5, 53, 1, 0.02)]


@pytest.fixture(scope="module")
def R():
    import reflexiv_b200 as R
    return R


def _reads(k, err):
    from workload import synth
    g = synth.genome(30_000, 300 + k)
    g[12000:12800] = g[3000:3800]
    g[20000:20040] = np.frombuffer(b"AT" * 20, np.uint8)
    return bytes(synth.fastq(g, 6000, read_len=150, frag_len=400, error_rate=err, seed_reads=9, seed_errors=10))


@functools.lru_cache(maxsize=None)
def _table(k, cover, err):
    """The oracle's count table with some counts past the 30000 saturation, in the layout rfx_load_counts takes."""
    from oracle import orc
    import reflexiv_b200 as R
    orc.lib()
    txt = _reads(k, err)
    s, l = orc.fastq_reads(txt, orc.FASTQ_RUN)
    c = orc.count_kmers(txt, s, l, k, min_count=cover)
    c["counts"][::131] = 40000 + np.arange(len(c["counts"][::131]), dtype=np.uint32)
    keys = R.pipeline.encode_kmer_rows([orc.decode_kmer(h, lo, k) for h, lo in zip(c["keys_hi"], c["keys_lo"])], k)
    return c, keys, c["counts"].astype(np.uint32)


def _contiguous(keys, cnt, world):
    n = len(cnt)
    return [(keys[n * r // world:n * (r + 1) // world], cnt[n * r // world:n * (r + 1) // world]) for r in range(world)]


def _ctxs(R, world, k, cover=1, E=8):
    return [R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=cover, minErrorCoverage=E, minContig=100), device=0) for _ in range(world)]


def _sort_body(R, slices, results, E, fold, kmax):
    def body(rank, ctx):
        ctx.reset()
        ctx.load_counts(*slices[rank])
        ctx.shard_table()
        n = ctx.sort_kmers_sharded(E, fold, kmax)
        with pytest.raises(R.RfxError) as e:
            ctx.contigs()
        assert e.value.code == R._lib.RFX_E_STATE
        keys, cnt = ctx.counts()
        results[rank] = dict(n=n, rows=ctx.sorted_rows(), csv=ctx.sorted_csv(), keys=keys, sh=ctx.shard_stats(), st=ctx.stats())
    return body


def _run(R, slices, k, E, fold, kmax):
    from reflexiv_b200 import sharded
    ctxs = _ctxs(R, len(slices), k)
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=1 << 30)
        results = [None] * len(slices)
        grp.run(_sort_body(R, slices, results, E, fold, kmax))
    finally:
        for c in ctxs:
            c.close()
    return results


def _rc(x, k):
    y = 0
    for _ in range(k):
        y = (y << 2) | (3 - (x & 3))
        x >>= 2
    return y


def _union(results):
    hi = np.concatenate([r["rows"][0] for r in results]); lo = np.concatenate([r["rows"][1] for r in results])
    le = np.concatenate([r["rows"][2] for r in results]); ri = np.concatenate([r["rows"][3] for r in results])
    order = np.lexsort((lo, hi))
    return hi[order], lo[order], le[order], ri[order]


def _check(orc, R, results, ref, k):
    """Union = oracle (arrays and CSV), ranks disjoint, every rank's rows keys of its own shard.  Returns key -> owner."""
    from reflexiv_b200.pipeline import keys_to_int
    hi, lo, le, ri = _union(results)
    assert np.array_equal(hi, ref["keys_hi"]) and np.array_equal(lo, ref["keys_lo"])
    assert np.array_equal(le, ref["left"]) and np.array_equal(ri, ref["right"])
    assert sorted(b"".join(r["csv"] for r in results).decode().splitlines()) == sorted(orc.sorted_rows_text(ref, k).splitlines())
    assert sum(r["n"] for r in results) == len(ref["left"])
    owner = {}
    for rank, res in enumerate(results):
        for key in keys_to_int(res["keys"], k):
            assert key not in owner  # shard tables are disjoint
            owner[key] = rank
    for rank, res in enumerate(results):
        assert res["n"] == len(res["rows"][0])
        for h, l in zip(res["rows"][0].tolist(), res["rows"][1].tolist()):
            x = (h << 64) | l
            assert owner[min(x, _rc(x, k))] == rank  # a sorted row lives with its canonical k-mer
    return owner


def _remote_left_candidates(results, owner, k):
    """Sorted rows (right-filter survivors) with a left candidate in the table that another rank owns: the left filter of
    their rank asked that owner for the candidate's coverage and right flag."""
    mask = (1 << (2 * (k - 1))) - 1
    n = 0
    for rank, res in enumerate(results):
        for h, l in zip(res["rows"][0].tolist(), res["rows"][1].tolist()):
            x = (h << 64) | l
            for a in range(4):
                y = (a << (2 * (k - 1))) | (x & mask)
                if y == x:
                    continue
                o = owner.get(min(y, _rc(y, k)))
                n += o is not None and o != rank
    return n


def _single(R, keys, cnt, k, E, fold, kmax):
    with R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=1), device=0) as ctx:
        ctx.load_counts(keys, cnt)
        ctx.sort_kmers(E, fold, kmax)
        hi, lo, le, ri = ctx.sorted_rows()
    order = np.lexsort((lo, hi))
    return hi[order], lo[order], le[order], ri[order]


@pytest.mark.parametrize("k,E,fold,kmax,cover,err,world", [c + (2,) for c in CASES] + [CASES[0] + (w,) for w in (1, 3, 4)])
def test_sorted_sharded_matches_oracle_and_one_gpu(R, orc, k, E, fold, kmax, cover, err, world):
    c, keys, cnt = _table(k, cover, err)
    ref = orc.sorted_rows(c["keys_hi"], c["keys_lo"], c["counts"], k, E, fold, kmax)
    results = _run(R, _contiguous(keys, cnt, world), k, E, fold, kmax)
    owner = _check(orc, R, results, ref, k)
    assert len(ref["left"]) > 0
    single = _single(R, keys, cnt, k, E, fold, kmax)
    assert all(np.array_equal(a, b) for a, b in zip(_union(results), single))
    if k == 31 and kmax == 95:
        _, _, le, ri = _union(results)
        assert (le == kmax + 3).any() and (ri == kmax + 3).any()  # fork winners on both sides
    if world >= 2:
        assert sum(r["sh"]["n_remote_probes"] for r in results) > 0
        assert all(r["sh"]["n_oriented_global"] == len(ref["left"]) for r in results)
        if k == 12:
            assert _remote_left_candidates(results, owner, k) > 0


def test_uneven_and_empty_slices(R, orc):
    k, E, fold, kmax = 31, 8, 1.5, 95
    c, keys, cnt = _table(k, 1, 0.01)
    ref = orc.sorted_rows(c["keys_hi"], c["keys_lo"], c["counts"], k, E, fold, kmax)
    n = len(cnt)
    empty = (keys[:0], cnt[:0])
    for slices in ([(keys, cnt), empty, empty],                          # all rows on one rank
                   [(keys[:n // 2], cnt[:n // 2]), empty, (keys[n // 2:], cnt[n // 2:])]):  # a rank with no rows
        _check(orc, R, _run(R, slices, k, E, fold, kmax), ref, k)
    results = _run(R, [empty] * 3, k, E, fold, kmax)                   # an all-empty table
    assert [r["n"] for r in results] == [0, 0, 0] and all(r["csv"] == b"" for r in results)


def test_from_reads(R, orc):
    """Slices of the FASTQ -> count_sharded -> sort_kmers_sharded, against the oracle's count table fed to its sorted stage."""
    from reflexiv_b200 import sharded
    k, E, fold, kmax, world = 31, 8, 1.5, 95, 3
    txt = _reads(k, 0.01)
    s, l = orc.fastq_reads(txt, orc.FASTQ_RUN)
    t = orc.count_kmers(txt, s, l, k, 0, 0, 2, 10_000_000, 1)
    ref = orc.sorted_rows(t["keys_hi"], t["keys_lo"], t["counts"], k, E, fold, kmax)
    cuts = [0] + [txt.find(b"\n@r", len(txt) * r // world) + 1 for r in range(1, world)] + [len(txt)]
    results = [None] * world

    def body(rank, ctx):
        ctx.reset()
        ctx.push_fastq(txt[cuts[rank]:cuts[rank + 1]])
        ctx.count_sharded()
        keys, _ = ctx.counts()
        n = ctx.sort_kmers_sharded(E, fold, kmax)
        results[rank] = dict(n=n, rows=ctx.sorted_rows(), csv=ctx.sorted_csv(), keys=keys, sh=ctx.shard_stats())
    ctxs = _ctxs(R, world, k, cover=2)
    try:
        sharded.LocalRanks(ctxs, arena_bytes=1 << 30).run(body)
    finally:
        for c in ctxs:
            c.close()
    _check(orc, R, results, ref, k)


def test_sort_assemble_sort_on_the_same_contexts(R, orc):
    from reflexiv_b200 import sharded
    k, world = 31, 3
    c, keys, cnt = _table(k, 1, 0.01)
    slices = _contiguous(keys, cnt, world)
    f = orc.fork_filter(c["keys_hi"], c["keys_lo"], c["counts"], k, 8)
    a = orc.assemble(f["keys_hi"], f["keys_lo"], f["left"], f["right"], k, 100, orc.ASM_CANONICAL)
    ctxs = _ctxs(R, world, k)
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=1 << 30)
        for E, fold in ((8, 1.5), (6, 2.0)):
            results = [None] * world
            grp.run(_sort_body(R, slices, results, E, fold, 95))
            _check(orc, R, results, orc.sorted_rows(c["keys_hi"], c["keys_lo"], c["counts"], k, E, fold, 95), k)
            contigs = grp.run(lambda rank, ctx: (ctx.assemble_sharded(), ctx.contigs())[1])
            assert sorted((s, l, r) for cs in contigs for s, l, r in cs) == sorted(zip(a["contigs"], a["left"].tolist(), a["right"].tolist()))
    finally:
        for x in ctxs:
            x.close()


def _expect_all(grp, body, code, world):
    t0 = time.perf_counter()
    codes = grp.run(body)
    assert codes == [code] * world
    assert time.perf_counter() - t0 < 5.0  # the agreement exchange catches it: nobody waits for a barrier to time out


def test_errors_come_back_from_every_rank_at_once(R, orc):
    from reflexiv_b200 import _lib, sharded
    world = 3
    for k, case in ((31, "E0"), (31, "fold"), (31, "unsharded"), (32, "k32")):
        c, keys, cnt = _table(k, 1, 0.01)
        slices = _contiguous(keys, cnt, world)
        ctxs = _ctxs(R, world, k)
        try:
            grp = sharded.LocalRanks(ctxs, arena_bytes=1 << 30)

            def bad(rank, ctx):
                ctx.reset()
                ctx.load_counts(*slices[rank])
                if case != "unsharded":
                    ctx.shard_table()
                E = 0 if case == "E0" else 8
                fold = 2.0 if case == "fold" and rank == 1 else 1.5
                try:
                    ctx.sort_kmers_sharded(E, fold, 95)
                except _lib.RfxError as err:
                    return err.code
                return 0
            want = {"E0": _lib.RFX_E_UNSUPPORTED, "k32": _lib.RFX_E_UNSUPPORTED, "fold": _lib.RFX_E_INVALID, "unsharded": _lib.RFX_E_STATE}[case]
            _expect_all(grp, bad, want, world)
            if k == 31:  # the ranks stay in step: the same contexts then sort correctly
                results = [None] * world
                grp.run(_sort_body(R, slices, results, 8, 1.5, 95))
                _check(orc, R, results, orc.sorted_rows(c["keys_hi"], c["keys_lo"], c["counts"], k, 8, 1.5, 95), k)
        finally:
            for x in ctxs:
                x.close()


def _sorted_lines(d):
    import gzip
    parts = sorted(f for f in os.listdir(d) if f.startswith("part-"))
    text = "".join((gzip.open(d / f).read().decode() if f.endswith(".gz") else (d / f).read_text()) for f in parts)
    return parts, sorted(text.splitlines())


def test_reflexiv_binary_sort_with_gpus_option(tmp_path):
    """`reflexiv sort -kmerc <Count_31> --gpus 3` (csrc/reflexiv_main.cpp: run_kmerc_sharded with a sort stage): one part file
    per rank whose lines together are those of the one-GPU `reflexiv sort`."""
    import subprocess
    from conftest import GOLDEN
    exe = os.path.join(ROOT, "reflexiv_b200", "reflexiv")
    env = dict(os.environ, REFLEXIV_ARENA_MB="768", CUDA_MODULE_LOADING="EAGER", CUDA_DEVICE_MAX_CONNECTIONS="32")
    fastq = os.path.join(GOLDEN, "paired_dat*.fq.gz")
    cout = tmp_path / "c"
    r = subprocess.run([exe, "counter", "-fastq", fastq, "-outfile", str(cout), "-kmer", "31"], capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr + r.stdout
    table = str(cout / "Count_31" / "part*")
    for extra in ([], ["-gzip"], ["-accurate", "-error", "6"], ["-klist", "23,41"]):
        outs = {}
        for gpus in (3, 1):
            out = tmp_path / f"s{gpus}_{len(extra)}_{'gz' if '-gzip' in extra else ''}"
            r = subprocess.run([exe, "sort", "--gpus", str(gpus), "-kmerc", table, "-outfile", str(out), "-kmer", "31"] + extra, capture_output=True, text=True, env=env)
            assert r.returncode == 0, r.stderr + r.stdout
            assert "--gpus" not in r.stderr, r.stderr
            d = out / "Count_31_sorted"
            assert (d / "_SUCCESS").exists()
            parts, lines = _sorted_lines(d)
            assert len(parts) == gpus and all(f.endswith(".gz") == ("-gzip" in extra) for f in parts)
            outs[gpus] = lines
        assert outs[3] == outs[1]
        assert (len(outs[3]) == 0) == ("-klist" in extra)
    r = subprocess.run([exe, "run", "--gpus", "2", "-kmerc", table, "-fastq", fastq, "-stitch", "-outfile", str(tmp_path / "st"), "-kmer", "31", "-cover", "3"],
                       capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stderr + r.stdout
    assert "--gpus applies to" in r.stderr  # -kmerc -stitch stays on one GPU


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
    z = np.load(os.path.join(out_dir, "table.npz"))
    ctx = R.ReflexivContext(R.DefaultParam(kmerSize=31, minKmerCoverage=1), device=rank)
    sharded.connect(ctx, dist, arena_bytes=2 << 30)
    results = [None] * world
    _sort_body(R, _contiguous(z["keys"], z["cnt"], world), results, 8, 1.5, 95)(rank, ctx)
    with open(os.path.join(out_dir, f"res_{rank}.pkl"), "wb") as f:
        pickle.dump(results[rank], f)
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
    c, keys, cnt = _table(31, 1, 0.01)
    np.savez(tmp_path / "table.npz", keys=keys, cnt=cnt)
    port = 29900 + os.getpid() % 1000
    mp.spawn(_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    results = [pickle.load(open(tmp_path / f"res_{r}.pkl", "rb")) for r in range(world)]
    import reflexiv_b200 as R
    _check(orc, R, results, orc.sorted_rows(c["keys_hi"], c["keys_lo"], c["counts"], 31, 8, 1.5, 95), 31)
