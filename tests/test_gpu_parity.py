"""GPU parity tests: every stage of libreflexiv_cuda, through the C ABI, against the CPU oracle on identical inputs.
Bit-exact everywhere (integer / byte work).  Run with `pytest -m gpu` on a B200."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from conftest import make_reads

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def R():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import reflexiv_b200 as R
    R.load_library()
    return R


def _sorted_table(R, ctx, k):
    keys, cnt = ctx.counts()
    ints = np.array(R.pipeline.keys_to_int(keys, k), dtype=object)
    order = np.argsort(ints) if len(ints) else np.array([], dtype=np.int64)
    return [int(x) for x in ints[order]], cnt[order]


def _oracle_table(orc, txt, k, mode, fc=0, ec=0, minc=1, maxc=2**62):
    s, l = orc.fastq_reads(txt, mode)
    c = orc.count_kmers(txt, s, l, k, fc, ec, minc, maxc)
    ints = [(int(h) << 64) | int(lo) for h, lo in zip(c["keys_hi"], c["keys_lo"])]
    return ints, c["counts"], c, (s, l)


def _param(R, **kw):
    return R.DefaultParam(**kw)


# ---------------------------------------------------------------------------------------------------------
# K1: FASTQ filters + 2-bit encoder
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("k,fc,ec", [(31, 0, 0), (21, 3, 5), (61, 0, 0)])
def test_k1_reads_and_packing(R, orc, hostemu, hooks, example_text, mode, k, fc, ec):
    txt = example_text[:300_000]
    txt = txt[:txt.rfind(b"\n@NODE")] + b"\n"
    if mode == 2:
        txt = b"\n".join(txt.split(b"\n")[1::4]) + b"\nACGTNNNNNACGT\n\nAC"  # sequence lines only, ragged tail
    s, l = orc.fastq_reads(txt, mode)
    a = np.frombuffer(txt, dtype=np.uint8)
    elen = np.zeros(len(s), np.uint32); woff = np.zeros(len(s), np.uint64)
    nw = hostemu.emu_pack_reads(a.ctypes.data, s.ctypes.data, l.ctypes.data, len(s), k, fc, ec, elen.ctypes.data, woff.ctypes.data, None)
    words = np.zeros(nw + 1, np.uint64)
    hostemu.emu_pack_reads(a.ctypes.data, s.ctypes.data, l.ctypes.data, len(s), k, fc, ec, elen.ctypes.data, woff.ctypes.data, words.ctypes.data)
    with R.ReflexivContext(_param(R, kmerSize=k, frontClip=fc, endClip=ec), fastq_mode=mode) as ctx:
        ctx.push_fastq(txt)
        g_len, g_woff, g_words = hooks.reads(ctx)
        st = ctx.stats()
    assert st["n_reads"] == len(s)
    assert np.array_equal(g_len, elen)
    assert np.array_equal(g_woff, woff)
    assert np.array_equal(g_words, words[:nw])
    assert st["n_bases"] == int(elen.sum())


def test_k1_state_machine_edge_cases(R, orc, hooks):
    txt = (b"garbage before the first record\n"
           b"@r1\nACGTACGTACGTACGTACGTACGTACGTACGTACGT\n+\n@IIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIII\n"
           b"@r2\nTTTTACGTACGTACGTACGTACGAACGTACGTACGT\n+r2\n+IIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIII\n"
           b"@r3\n@r3b\nACGTNNNNACGTACGTACGTACGTACGTACGTACGT\r\n+\r\nIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIIII\r\n"
           b"\n@r4\nGGGGGGGGGGGGGGGGGGGGGGGGGGGGGGGGGGGG\n+\n")  # last unit lacks its quality line
    for tail in (b"", b"IIII", b"IIII\n", b"IIII\n@r5\nACGT"):
        t = txt + tail
        s, l = orc.fastq_reads(t, orc.FASTQ_RUN)
        with R.ReflexivContext(_param(R, kmerSize=15)) as ctx:
            ctx.push_fastq(t)
            g_len, _, _ = hooks.reads(ctx)
        assert g_len.tolist() == l.tolist()
    with R.ReflexivContext(_param(R, kmerSize=15)) as ctx:
        ctx.push_fastq(b"")
        ctx.push_fastq(b"\n\n\n")
        assert ctx.stats()["n_reads"] == 0
        st = ctx.count()
        assert st["n_rows"] == 0 and st["n_instances"] == 0
        assert ctx.assemble()["n_contigs"] == 0 and ctx.contigs() == []


def test_chunked_upload_carries_the_fastq_state(R, orc, hooks, example_text, monkeypatch):
    """rfx_push_fastq uploads big inputs in chunks cut at arbitrary newlines (here: every ~3 KB, so chunks start in
    the middle of records, on '+' lines and on quality lines that begin with '@'); the carried lineMark must make
    that invisible."""
    monkeypatch.setenv("RFX_FASTQ_CHUNK_BYTES", "3000")
    for txt in (example_text, example_text[:100_003], example_text + b"@tail\nACGTACGTACGTACGTACGTACGTACGTACGTACGT\n+\n"):
        s, l = orc.fastq_reads(txt, orc.FASTQ_RUN)
        with R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=1)) as ctx:
            ctx.push_fastq(txt)
            g_len, _, _ = hooks.reads(ctx)
            assert ctx.stats()["n_reads"] == len(s)
            assert np.array_equal(g_len, np.where(l.astype(np.int64) - 31 > 1, l, 0).astype(np.uint32))
    ints, counts, c, _ = _oracle_table(orc, example_text, 31, orc.FASTQ_RUN)
    with R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=1)) as ctx:
        ctx.push_fastq(example_text)
        ctx.count()
        g_ints, g_counts = _sorted_table(R, ctx, 31)
    assert g_ints == ints and np.array_equal(g_counts, counts)


def test_dos_line_ends(R, example_text, golden):
    """"\\r\\n" line ends give the table of the Unix file (K1 strips the "\\r" like Hadoop's LineRecordReader), in both FASTQ modes."""
    dos = example_text.replace(b"\n", b"\r\n")
    for counter_mode in (False, True):
        rows = []
        for txt in (example_text, dos):
            with R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=2), counter_mode=counter_mode) as ctx:
                ctx.push_fastq(txt)
                ctx.count()
                rows.append(sorted(ctx.counts_csv().decode().splitlines()))
        assert rows[0] == rows[1]
        if not counter_mode:
            assert hashlib.sha256(("\n".join(rows[1]) + "\n").encode()).hexdigest() == golden["oracle"]["count_ge2"]["sha256_sorted_csv"]


def test_regular_layout_shortcut_and_general_state_machine_agree(R, orc, hooks, example_text, monkeypatch):
    """K1 takes a shortcut when a chunk is made of whole 4-line records (reads = every fourth line, at the phase the carried
    lineMark gives) and runs the scan of transition functions otherwise.  Same read table either way, with chunk cuts at
    every phase; a single stray line flips the chunk to the general path without changing the answer."""
    stray = example_text[:50_000] + b"stray line\n" + example_text[50_000:]
    for txt in (example_text, stray):
        s, l = orc.fastq_reads(txt, orc.FASTQ_RUN)
        want = np.where(l.astype(np.int64) - 31 > 1, l, 0).astype(np.uint32)
        for chunk in ("", "2777", "50021"):
            for general in ("", "1"):
                monkeypatch.setenv("RFX_FASTQ_CHUNK_BYTES", chunk) if chunk else monkeypatch.delenv("RFX_FASTQ_CHUNK_BYTES", raising=False)
                monkeypatch.setenv("RFX_FASTQ_GENERAL", general) if general else monkeypatch.delenv("RFX_FASTQ_GENERAL", raising=False)
                with R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=1)) as ctx:
                    ctx.push_fastq(txt)
                    g_len, _, _ = hooks.reads(ctx)
                assert np.array_equal(g_len, want), (len(txt), chunk, general)


# ---------------------------------------------------------------------------------------------------------
# K2: super-k-mer records
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,m", [(31, 0), (31, 15), (21, 9), (61, 0), (33, 16)])
def test_k2_records_hold_exactly_the_kmer_instances(R, orc, hostemu, hooks, example_text, k, m):
    txt = example_text
    ints, counts, c, _ = _oracle_table(orc, txt, k, orc.FASTQ_RUN)
    with R.ReflexivContext(_param(R, kmerSize=k), minimizer_len=m) as ctx:
        ctx.push_fastq(txt)
        ctx.partition(1)
        offs, recs = hooks.records(ctx)
        st = ctx.stats()
        mm = m if m else 11
        n_bins = st["n_bins"]
    nk = (recs[:, 0] >> np.uint64(48)).astype(np.int64)
    assert int(nk.sum()) == c["n_instances"] == st["n_instances"]
    assert offs[0] == 0 and offs[-1] == len(recs) and np.all(np.diff(offs.astype(np.int64)) >= 0)
    bins = np.repeat(np.arange(n_bins, dtype=np.uint32), np.diff(offs.astype(np.int64)))
    bad = C.c_int64(0)
    d = hostemu.emu_count_records(recs.ctypes.data, bins.ctypes.data, len(recs), k, mm, n_bins, C.addressof(bad))
    hi = np.zeros(d, np.uint64); lo = np.zeros(d, np.uint64); cnt = np.zeros(d, np.uint32)
    hostemu.emu_count_fetch(hi.ctypes.data, lo.ctypes.data, cnt.ctypes.data)
    assert bad.value == 0
    assert np.array_equal(hi, c["keys_hi"]) and np.array_equal(lo, c["keys_lo"]) and np.array_equal(cnt, c["counts"])


# ---------------------------------------------------------------------------------------------------------
# K3 + K4: counting + coverage filter
# ---------------------------------------------------------------------------------------------------------
def test_count_table_golden_digests(R, example_text, golden):
    """BASELINE config 1 through the C ABI: the digests of SURVEY 8c / tests/golden."""
    for cov in (1, 2, 3):
        with R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=cov)) as ctx:
            ctx.push_fastq(example_text)
            st = ctx.count()
            csv = ctx.counts_csv()
        g = golden["oracle"]
        assert (st["n_reads"], st["n_instances"], st["n_distinct"]) == (g["n_reads"], g["n_instances"], g["n_distinct"])
        assert st["n_rows"] == g[f"count_ge{cov}"]["rows"]
        rows = sorted(csv.decode().splitlines())
        assert hashlib.sha256(("\n".join(rows) + "\n").encode()).hexdigest() == g[f"count_ge{cov}"]["sha256_sorted_csv"]


@pytest.mark.parametrize("k", [5, 15, 21, 31, 32, 33, 47, 61, 63])
def test_counts_match_oracle_all_k(R, orc, example_text, k):
    txt = example_text[:600_000]
    txt = txt[:txt.rfind(b"\n@NODE")] + b"\n"
    ints, counts, c, _ = _oracle_table(orc, txt, k, orc.FASTQ_RUN)
    with R.ReflexivContext(_param(R, kmerSize=k, minKmerCoverage=1)) as ctx:
        ctx.push_fastq(txt)
        st = ctx.count()
        g_ints, g_counts = _sorted_table(R, ctx, k)
    assert st["n_instances"] == c["n_instances"] and st["n_distinct"] == c["n_distinct"]
    assert g_ints == ints
    assert np.array_equal(g_counts, counts)


@pytest.mark.parametrize("k,cover,bin_target", [(5, 1, 0), (21, 1, 0), (31, 2, 0), (33, 1, 0), (61, 2, 0), (63, 1, 0), (31, 1, 60_000), (61, 1, 30_000)])
def test_sort_based_counting_kernel_matches_oracle(R, orc, example_text, monkeypatch, k, cover, bin_target):
    """The measured alternative of the hash kernel (sort_bins_kernel: expand, bitonic sort, run-length count), forced here;
    bins far larger than its shared-memory array go through hash-class passes (bin_target)."""
    monkeypatch.setenv("RFX_COUNT_VARIANT", "sort")
    noisy = bytes(make_reads(31, 50_000, 5000, read_len=150, err=0.01, frag=400))
    for txt in (example_text, noisy):
        s, l = orc.fastq_reads(txt, orc.FASTQ_RUN)
        c = orc.count_kmers(txt, s, l, k, 0, 0, cover, 10_000_000, 1)
        ints = [(int(h) << 64) | int(lo) for h, lo in zip(c["keys_hi"], c["keys_lo"])]
        with R.ReflexivContext(_param(R, kmerSize=k, minKmerCoverage=cover), bin_target_kmers=bin_target) as ctx:
            ctx.push_fastq(txt)
            st = ctx.count()
            g_ints, g_counts = _sorted_table(R, ctx, k)
        assert st["n_instances"] == c["n_instances"] and st["n_distinct"] == c["n_distinct"]
        assert g_ints == ints and np.array_equal(g_counts, c["counts"])
        if bin_target and txt is noisy:  # (the example is too small to overfill the 64 bins a run has at least)
            assert st["n_bin_splits"] > 0


def test_pilot_can_route_noisy_bins_to_the_sort_kernel(R, orc, monkeypatch):
    """RFX_SORT_RATIO=<x>: the pilot (~300 bins counted without writing) sends a run to the sort kernel when more than x of its
    k-mer instances are k-mers of their own.  Off by default -- the sort kernel lost every measurement -- but the route is
    kept and must give the oracle's table; clean reads stay on the hash kernel under the same setting."""
    monkeypatch.setenv("RFX_SORT_RATIO", "0.35")
    clean = bytes(make_reads(41, 60_000, 6000, read_len=150, err=0.0, frag=400))
    noisy = bytes(make_reads(42, 60_000, 6000, read_len=150, err=0.012, frag=400))
    for txt, k in ((clean, 31), (noisy, 61), (noisy, 31)):
        s, l = orc.fastq_reads(txt, orc.FASTQ_RUN)
        c = orc.count_kmers(txt, s, l, k, 0, 0, 1, 10_000_000, 1)
        ints = [(int(h) << 64) | int(lo) for h, lo in zip(c["keys_hi"], c["keys_lo"])]
        with R.ReflexivContext(_param(R, kmerSize=k, minKmerCoverage=1)) as ctx:
            ctx.push_fastq(txt)
            ctx.count()
            g_ints, g_counts = _sorted_table(R, ctx, k)
        assert g_ints == ints and np.array_equal(g_counts, c["counts"])


@pytest.mark.parametrize("k,m", [(31, 15), (31, 9), (27, 15), (61, 16)])
def test_counts_do_not_depend_on_the_minimiser_length(R, orc, example_text, k, m):
    """m = 15 is what inputs with more than 2^16 bins use (register-resident scan, single-pass slab partition)."""
    ints, counts, c, _ = _oracle_table(orc, example_text, k, orc.FASTQ_RUN)
    with R.ReflexivContext(_param(R, kmerSize=k, minKmerCoverage=1), minimizer_len=m) as ctx:
        ctx.push_fastq(example_text)
        st = ctx.count()
        g_ints, g_counts = _sorted_table(R, ctx, k)
    assert st["n_instances"] == c["n_instances"] and st["n_distinct"] == c["n_distinct"]
    assert g_ints == ints and np.array_equal(g_counts, counts)


@pytest.mark.parametrize("counter_mode,cover,maxcov", [(False, 2, 10_000_000), (False, 3, 20), (True, 1, 10_000_000), (True, 2, 30), (True, 0, 5)])
def test_coverage_filter_rules(R, orc, example_text, counter_mode, cover, maxcov):
    """A4: `run` always applies both bounds; `counter` only applies cover if > 1 and maxcov if < 10^7."""
    if counter_mode:
        lo = cover if cover > 1 else 1
        hi = maxcov if maxcov < 10_000_000 else 2**62
    else:
        lo, hi = cover, maxcov
    mode = orc.FASTQ_COUNTER if counter_mode else orc.FASTQ_RUN
    ints, counts, c, _ = _oracle_table(orc, example_text, 31, mode, minc=max(lo, 1), maxc=hi)
    with R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=cover, maxKmerCoverage=maxcov), counter_mode=counter_mode) as ctx:
        ctx.push_fastq(example_text)
        ctx.count()
        g_ints, g_counts = _sorted_table(R, ctx, 31)
    assert g_ints == ints and np.array_equal(g_counts, counts)


def test_bin_overflow_splitting_is_exact(R, orc):
    """Low coverage + few bins: bins hold far more distinct k-mers than the shared-memory table, so classes are split."""
    txt = make_reads(21, 400_000, 3000, read_len=150, err=0.0, frag=400)
    ints, counts, c, _ = _oracle_table(orc, txt, 31, orc.FASTQ_RUN)
    with R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=1), bin_target_kmers=200_000) as ctx:
        ctx.push_fastq(txt)
        st = ctx.count()
        g_ints, g_counts = _sorted_table(R, ctx, 31)
    assert st["n_bin_splits"] > 0
    assert g_ints == ints and np.array_equal(g_counts, counts)
    txt = make_reads(22, 400_000, 4000, read_len=150, err=0.0, frag=400)
    ints, counts, c, _ = _oracle_table(orc, txt, 61, orc.FASTQ_RUN)
    with R.ReflexivContext(_param(R, kmerSize=61, minKmerCoverage=1), bin_target_kmers=200_000) as ctx:
        ctx.push_fastq(txt)
        st = ctx.count()
        g_ints, g_counts = _sorted_table(R, ctx, 61)
    assert st["n_bin_splits"] > 0
    assert g_ints == ints and np.array_equal(g_counts, counts)


def test_repeated_runs_are_bit_identical(R, orc, monkeypatch):
    """compute-sanitizer is closed on the GPU pool (profiles/r2_sanitizer.txt); a race in the counting kernel's shared-memory
    machinery or in the request / answer exchange of the sharded graph stages would show as a run that differs.  Twenty runs
    of a split-forcing input on one context, twenty sharded runs of two ranks on one device: one digest each."""
    import hashlib
    from reflexiv_b200 import sharded
    from reflexiv_b200.pipeline import keys_to_int
    txt = bytes(make_reads(23, 60_000, 4000, read_len=150, err=0.01, frag=400))
    ref = orc.run_pipeline(txt, k=31, cover=1, min_contig=100)
    want_rows = len(ref["counts"]["counts"])
    want_contigs = sorted(ref["asm"]["contigs"])

    def digest(tables, contigs):
        rows = sorted(kv for keys, cnt in tables for kv in zip(keys_to_int(keys, 31), cnt.tolist()))
        return hashlib.sha256(repr((rows, sorted(contigs))).encode()).hexdigest(), len(rows)

    monkeypatch.setenv("RFX_COUNT_VARIANT", "small")
    seen = set()
    with R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=1, minContig=100), bin_target_kmers=200_000) as ctx:
        for _ in range(20):
            ctx.reset()
            ctx.push_fastq(txt)
            st = ctx.count()
            assert st["n_bin_splits"] > 0
            tab = ctx.counts()
            ctx.assemble()
            d, n = digest([tab], [s for s, _, _ in ctx.contigs()])
            assert n == want_rows
            seen.add(d)
    assert len(seen) == 1
    monkeypatch.delenv("RFX_COUNT_VARIANT")
    cut = txt.find(b"\n@r", len(txt) // 2) + 1
    parts = [txt[:cut], txt[cut:]]
    ctxs = [R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=1, minContig=100)) for _ in range(2)]
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=1 << 30)
        for _ in range(20):
            out = [None, None]

            def body(r, c):
                c.reset()
                c.push_fastq(parts[r])
                c.count_sharded()
                tab = c.counts()
                c.assemble_sharded()
                out[r] = (tab, [s for s, _, _ in c.contigs()])
            grp.run(body)
            d, n = digest([o[0] for o in out], [s for o in out for s in o[1]])
            assert n == want_rows and sorted(s for o in out for s in o[1]) == want_contigs
            seen.add(d)
    finally:
        for c in ctxs:
            c.close()
    assert len(seen) == 1  # ... and the sharded runs give the very digest of the single-context runs


@pytest.mark.parametrize("k", [31, 61])
def test_long_and_ragged_reads(R, orc, k):
    """Reads of up to 11 000 bases (warps of very uneven reads in the register-resident scan), mixed with short and empty
    ones, on the default single-pass partition.  The same reads on the two-pass partition, whose spill pass they reach:
    test_skewed_inputs.test_spill_pass_of_the_two_pass_partition."""
    rng = np.random.default_rng(9)
    g = "".join("ACGT"[i] for i in rng.integers(0, 4, 20_000))
    seqs = [g[a:a + n] for a, n in ((0, 5000), (3000, 4000), (100, k), (200, k + 1), (300, k + 2), (400, 150), (9000, 11000), (0, 0), (5, 3))]
    seqs += [orc.revcomp_str(g[a:a + 700]) for a in range(0, 19000, 450)]
    txt = ("\n".join(seqs) + "\n").encode()
    ints, counts, c, _ = _oracle_table(orc, txt, k, orc.FASTQ_LINE)
    with R.ReflexivContext(_param(R, kmerSize=k, minKmerCoverage=1), fastq_mode=2) as ctx:
        ctx.push_fastq(txt)
        st = ctx.count()
        g_ints, g_counts = _sorted_table(R, ctx, k)
    assert st["n_instances"] == c["n_instances"]
    assert g_ints == ints and np.array_equal(g_counts, counts)


def test_push_reads_and_repeated_push(R, orc, example_text):
    s, l = orc.fastq_reads(example_text, orc.FASTQ_RUN)
    seqs = [example_text[int(a):int(a) + int(b)] for a, b in zip(s, l)]
    ints, counts, c, _ = _oracle_table(orc, example_text, 31, orc.FASTQ_RUN)
    with R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=1)) as ctx:
        half = len(seqs) // 2
        for part in (seqs[:half], seqs[half:]):
            offs = np.concatenate([[0], np.cumsum([len(x) for x in part])]).astype(np.uint64)
            ctx.push_reads(b"".join(part), offs)
        ctx.count()
        g_ints, g_counts = _sorted_table(R, ctx, 31)
        assert g_ints == ints and np.array_equal(g_counts, counts)
        # reset + FASTQ text pushed in two record-aligned pieces
        ctx.reset()
        cut = example_text.find(b"\n@NODE", len(example_text) // 2) + 1
        ctx.push_fastq(example_text[:cut])
        ctx.push_fastq(example_text[cut:])
        ctx.count()
        g_ints, g_counts = _sorted_table(R, ctx, 31)
        assert g_ints == ints and np.array_equal(g_counts, counts)


# ---------------------------------------------------------------------------------------------------------
# K5: fork filters ; K6/K7: extension and contigs
# ---------------------------------------------------------------------------------------------------------
def _oracle_run(orc, txt, k, cover, E=8, min_contig=500):
    return orc.run_pipeline(txt, k=k, cover=cover, min_error_cov=E, min_contig=min_contig)


def _check_assembly(R, orc, txt, k, cover, E=8, min_contig=500):
    ref = _oracle_run(orc, txt, k, cover, E, min_contig)
    with R.ReflexivContext(_param(R, kmerSize=k, minKmerCoverage=cover, minErrorCoverage=E, minContig=min_contig)) as ctx:
        ctx.push_fastq(txt)
        ctx.count()
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
    got = sorted((s, l, r) for s, l, r in contigs)
    exp = sorted(zip(a["contigs"], a["left"].tolist(), a["right"].tolist()))
    assert got == exp
    return ref, st


def test_docs_golden_contig_on_gpu(R, orc, example_text, golden):
    """The reference's documented answer: `reflexiv run -kmer 31 -cover 3` on example/ -> 2 x 4558 bp, documented prefix."""
    ref, st = _check_assembly(R, orc, example_text, 31, 3)
    with R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=3)) as ctx:
        ctx.push_fastq(example_text)
        ctx.count()
        ctx.assemble()
        contigs = [c for c, _, _ in ctx.contigs()]
    assert sorted(len(c) for c in contigs) == [4558, 4558]
    assert sum(c.startswith(golden["documented"]["prefix_1200"]) for c in contigs) == 1
    cs = orc.canonical_contig_set(contigs)
    assert [hashlib.sha256(x.encode()).hexdigest() for x in cs] == golden["oracle"]["contigs_cover3"]["canonical_sha256"]


@pytest.mark.parametrize("k,cover,E,err", [(31, 2, 8, 0.0), (31, 2, 8, 0.01), (31, 2, 0, 0.01), (21, 1, 8, 0.02), (41, 2, 8, 0.01), (61, 2, 8, 0.005), (24, 1, 8, 0.01)])
def test_assembly_matches_oracle(R, orc, k, cover, E, err):
    from workload import synth
    g = synth.genome(30_000, 100 + k)
    g[12000:12800] = g[3000:3800]    # repeat: real forks, budget junctions
    g[20000:20040] = np.frombuffer(b"AT" * 20, np.uint8)  # palindromic low-complexity stretch (cycles for even k)
    txt = synth.fastq(g, 6000, read_len=150, frag_len=400, error_rate=err, seed_reads=5, seed_errors=6)
    ref, st = _check_assembly(R, orc, txt, k, cover, E, min_contig=100)
    assert st["n_contigs"] >= 2


@pytest.mark.parametrize("k,cover,E,err", [(31, 2, 8, 0.01), (61, 2, 8, 0.005), (24, 1, 8, 0.01), (5, 1, 8, 0.0), (12, 2, 0, 0.01), (33, 2, 8, 0.0)])
def test_assembly_with_the_bin_local_index(R, orc, monkeypatch, k, cover, E, err):
    """Tables beyond the L2 use minimiser-bin-local index regions; forced here on small inputs (RFX_GRAPH_INDEX=local)."""
    from workload import synth
    monkeypatch.setenv("RFX_GRAPH_INDEX", "local")
    g = synth.genome(30_000, 200 + k)
    g[12000:12800] = g[3000:3800]
    g[20000:20040] = np.frombuffer(b"AT" * 20, np.uint8)
    txt = synth.fastq(g, 6000, read_len=150, frag_len=400, error_rate=err, seed_reads=7, seed_errors=8)
    _check_assembly(R, orc, txt, k, cover, E, min_contig=100)


def _uniform_table(g: np.ndarray, k: int, seed: int):
    """Canonical k-mer table of a genome with near-equal counts (10..12): every fork is a real one (flag k-1)."""
    code = np.zeros(256, np.uint8)
    for i, ch in enumerate(b"ACGT"):
        code[ch] = i
    c = code[g].astype(object)
    mask = (1 << (2 * k)) - 1
    fwd = rc = 0
    seen = {}
    for i, v in enumerate(c.tolist()):
        fwd = ((fwd << 2) | v) & mask
        rc = (rc >> 2) | ((3 - v) << (2 * (k - 1)))
        if i >= k - 1:
            key = min(fwd, rc)
            seen.setdefault(key, 10 + (hash((key, seed)) % 3))
    keys = np.array(sorted(seen), dtype=np.uint64)
    counts = np.array([seen[int(x)] for x in keys], dtype=np.uint32)
    return keys, counts


@pytest.mark.parametrize("k,glen,seed", [(9, 3000, 1), (10, 2000, 4), (11, 20000, 2), (13, 60000, 3), (12, 40000, 6), (31, 8000, 5)])
def test_budget_walks_on_dense_forks(R, orc, monkeypatch, k, glen, seed):
    """A9 clauses 3 / 4 (ReflexivDSMain.java:3077-3084): fork winners absorb up to k-1 clean k-mers.  Random genomes at small k
    are full of repeated (k-1)-mers, so winners sit within reach of each other, face each other and lie on closed paths;
    the GPU must give the oracle's canonical contigs WITH their header flags, and the canonical closed form must equal
    the reference's four merge clauses applied literally under the same schedule (ORC_ASM_SCHEDULED)."""
    from workload import synth
    g = synth.genome(glen, 300 + seed)
    if k == 31:
        g[5000:5400] = g[1000:1400]
        g[7000:7060] = g[2000:2060]
        g[3000] = ord("A") if g[3000] != ord("A") else ord("C")
    keys, counts = _uniform_table(g, k, seed)
    zero = np.zeros(len(keys), np.uint64)
    ff = orc.fork_filter(zero, keys, counts, k, 8)
    a = orc.assemble(ff["keys_hi"], ff["keys_lo"], ff["left"], ff["right"], k, k, orc.ASM_CANONICAL)
    s = orc.assemble(ff["keys_hi"], ff["keys_lo"], ff["left"], ff["right"], k, k, orc.ASM_SCHEDULED)
    assert a["n_budget_admissible"] > 0 and a["n_budget_junctions"] > 0
    if a["n_cycles"] == 0 and s["n_cycles"] == 0:
        assert sorted(zip(a["contigs"], a["left"].tolist(), a["right"].tolist())) == sorted(zip(s["contigs"], s["left"].tolist(), s["right"].tolist()))
    else:
        assert sorted(a["contigs"]) == sorted(s["contigs"])  # where a closed contig is cut decides its two flags
    for index in ("global", "local"):
        monkeypatch.setenv("RFX_GRAPH_INDEX", index)
        with R.ReflexivContext(_param(R, kmerSize=k, minContig=k)) as ctx:
            ctx.load_counts(keys.reshape(-1, 1), counts)
            st = ctx.assemble()
            hi, lo, le, ri = ctx.oriented()
            contigs = ctx.contigs()
        order = np.lexsort((lo, hi))
        assert np.array_equal(lo[order], ff["keys_lo"]) and np.array_equal(le[order], ff["left"]) and np.array_equal(ri[order], ff["right"])
        assert (st["n_budget_junctions"], st["n_budget_admissible"], st["n_cycles"]) == (a["n_budget_junctions"], a["n_budget_admissible"], a["n_cycles"])
        assert sorted(contigs) == sorted(zip(a["contigs"], a["left"].tolist(), a["right"].tolist()))


def test_cycles_and_tiny_graphs(R, orc, monkeypatch):
    def fq(seqs):
        return "".join(f"@r{i}\n{s}\n+\n{'I' * len(s)}\n" for i, s in enumerate(seqs)).encode()
    rng = np.random.default_rng(3)
    circ = "".join("ACGT"[i] for i in rng.integers(0, 4, 300))
    reads = [(circ + circ)[i:i + 120] for i in range(0, 300, 7)] * 3          # a circular genome: one cycle per strand
    _check_assembly(R, orc, fq(reads), 31, 2, min_contig=50)
    _check_assembly(R, orc, fq(["A" * 100] * 3), 31, 2, min_contig=10)       # homopolymer: 1-cycle
    _check_assembly(R, orc, fq(["ACGT" * 30] * 3), 16, 2, min_contig=10)     # period-4 cycle, even k, palindromes
    _check_assembly(R, orc, fq([circ[:33]] * 2), 31, 2, min_contig=10)       # three k-mers
    monkeypatch.setenv("RFX_GRAPH_INDEX", "local")
    _check_assembly(R, orc, fq(reads), 31, 2, min_contig=50)
    _check_assembly(R, orc, fq(["A" * 100] * 3), 31, 2, min_contig=10)
    _check_assembly(R, orc, fq(["ACGT" * 30] * 3), 16, 2, min_contig=10)


def test_load_counts_seam(R, orc, example_text):
    """-kmerc: assemble from a (k-mer, count) table instead of reads (ReflexivDSMain.assemblyFromKmer)."""
    ref = _oracle_run(orc, example_text, 31, 2)
    c = ref["counts"]
    keys = c["keys_lo"].reshape(-1, 1)
    with R.ReflexivContext(_param(R, kmerSize=31)) as ctx:
        ctx.load_counts(keys, c["counts"])
        ctx.assemble()
        got = sorted(s for s, _, _ in ctx.contigs())
    assert got == sorted(ref["asm"]["contigs"])


@pytest.mark.parametrize("k,E,fold,kmax,cover,err,index", [(31, 8, 1.5, 95, 1, 0.01, None), (31, 6, 2.0, 31, 2, 0.01, "local"), (23, 8, 1.5, 95, 1, 0.02, None),
                                                            (41, 8, 1.5, 95, 1, 0.01, None), (53, 24, 2.0, 95, 1, 0.005, "local"), (12, 3, 1.5, 53, 1, 0.02, None)])
def test_sorted_stage_matches_oracle(R, orc, monkeypatch, k, E, fold, kmax, cover, err, index):
    """SURVEY 8f-2, Count_<k>_sorted: rfx_sort_kmers against the oracle's restatement of ReflexivDSKmerLeftAndRightSorting
    (rows as arrays and as the CSV text the reference writes), with both index layouts and coverages past the 30000
    saturation; the assembly results of the same context stay retrievable only until the stage takes the index over."""
    from workload import synth
    if index:
        monkeypatch.setenv("RFX_GRAPH_INDEX", index)
    g = synth.genome(30_000, 300 + k)
    g[12000:12800] = g[3000:3800]
    g[20000:20040] = np.frombuffer(b"AT" * 20, np.uint8)
    txt = synth.fastq(g, 6000, read_len=150, frag_len=400, error_rate=err, seed_reads=9, seed_errors=10)
    s, l = orc.fastq_reads(txt, orc.FASTQ_RUN)
    c = orc.count_kmers(txt, s, l, k, min_count=cover)
    c["counts"][::131] = 40000 + np.arange(len(c["counts"][::131]), dtype=np.uint32)
    ref = orc.sorted_rows(c["keys_hi"], c["keys_lo"], c["counts"], k, E, fold, kmax)
    ints = [(int(h) << 64) | int(lo) for h, lo in zip(c["keys_hi"], c["keys_lo"])]
    keys = R.pipeline.encode_kmer_rows([orc.decode_kmer(h, lo, k) for h, lo in zip(c["keys_hi"], c["keys_lo"])], k)
    assert R.pipeline.keys_to_int(keys, k) == ints
    with R.ReflexivContext(_param(R, kmerSize=k, minKmerCoverage=1)) as ctx:
        ctx.load_counts(keys, c["counts"])
        n = ctx.sort_kmers(E, fold, kmax)
        hi, lo, le, ri = ctx.sorted_rows()
        csv = ctx.sorted_csv()
        with pytest.raises(R.RfxError) as e:
            ctx.contigs()
        assert e.value.code == R._lib.RFX_E_STATE
    assert n == len(ref["left"]) and n > 0
    order = np.lexsort((lo, hi))
    assert np.array_equal(hi[order], ref["keys_hi"]) and np.array_equal(lo[order], ref["keys_lo"])
    assert np.array_equal(le[order], ref["left"]) and np.array_equal(ri[order], ref["right"])
    assert sorted(csv.decode().splitlines()) == sorted(orc.sorted_rows_text(ref, k).splitlines())
    if k == 31 and index is None:
        assert (le == kmax + 3).any() and (ri == kmax + 3).any()


def test_sorted_stage_pipeline_and_domain(R, orc, example_text, tmp_path):
    """Count_<k> CSV -> Count_<k>_sorted through the host mirror of Pipelines.reflexivLeftAndRightSortingPipe, and the
    inputs the reference itself cannot process."""
    import gzip
    cout = tmp_path / "work"
    from conftest import GOLDEN
    pc = R.ParameterOfCounter(["-fastq", os.path.join(GOLDEN, "paired_dat*.fq.gz"), "-outfile", str(cout), "-kmer", "31", "-cover", "1", "-gzip"]).importCommandLine()
    R.Pipelines(pc).reflexivDSCounterPipe()
    p = R.DefaultParam(kmerSize=31, outputPath=str(cout), inputKmerPath=str(cout / "Count_31" / "part*.csv.gz"), gzip=True, maxKmerCoverage=1_000_000)
    st = R.Pipelines(p).reflexivLeftAndRightSortingPipe()
    d = cout / "Count_31_sorted"
    parts = [f for f in os.listdir(d) if f.startswith("part-")]
    assert len(parts) == 1 and (d / "_SUCCESS").exists()
    rows = sorted(gzip.open(d / parts[0]).read().decode().splitlines())
    s, l = orc.fastq_reads(example_text, orc.FASTQ_COUNTER)
    c = orc.count_kmers(example_text, s, l, 31)
    ref = orc.sorted_rows(c["keys_hi"], c["keys_lo"], c["counts"], 31, 8, 1.5, 95, 1_000_000)
    assert rows == sorted(orc.sorted_rows_text(ref, 31).splitlines()) and st["n_sorted_rows"] == len(rows)
    assert all(r[31:34] == ",1|" for r in rows)
    # the same stage through the C++ driver (`reflexiv sort`, option names of `run`)
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "reflexiv_b200", "reflexiv")
    r = subprocess.run([exe, "sort", "-kmerc", str(cout / "Count_31" / "part*.csv.gz"), "-outfile", str(tmp_path / "cli"), "-kmer", "31", "-maxcov", "1000000"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    dd = tmp_path / "cli" / "Count_31_sorted"
    pp = [f for f in os.listdir(dd) if f.startswith("part-")]
    assert len(pp) == 1 and (dd / "_SUCCESS").exists()
    assert sorted((dd / pp[0]).read_text().splitlines()) == rows
    r = subprocess.run([exe, "sort", "-kmerc", str(cout / "Count_31" / "part*.csv.gz"), "-outfile", str(tmp_path / "cli2"), "-kmer", "31", "-klist", "23,41", "-gzip"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    pp = [f for f in os.listdir(tmp_path / "cli2" / "Count_31_sorted") if f.startswith("part-")]
    assert len(pp) == 1 and gzip.open(tmp_path / "cli2" / "Count_31_sorted" / pp[0]).read() == b""
    r = subprocess.run([exe, "sort", "-kmerc", str(cout / "Count_31" / "part*.csv.gz"), "-outfile", str(tmp_path / "cli3"), "-kmer", "31", "-accurate", "-error", "6"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    pp = [f for f in os.listdir(tmp_path / "cli3" / "Count_31_sorted") if f.startswith("part-")]
    ref2 = orc.sorted_rows(c["keys_hi"], c["keys_lo"], c["counts"], 31, 6, 2.0, 95)
    assert sorted((tmp_path / "cli3" / "Count_31_sorted" / pp[0]).read_text().splitlines()) == sorted(orc.sorted_rows_text(ref2, 31).splitlines())
    # a k outside the k-mer list: the reference's binarizer drops every row
    p2 = R.DefaultParam(kmerSize=31, outputPath=str(tmp_path / "w2"), inputKmerPath=str(cout / "Count_31" / "part*.csv.gz"), kmerList="23,41")
    assert R.Pipelines(p2).reflexivLeftAndRightSortingPipe()["n_sorted_rows"] == 0
    for k, E in [(31, 0), (32, 8), (63, 8)]:
        with R.ReflexivContext(_param(R, kmerSize=k, minKmerCoverage=1)) as ctx:
            ctx.push_fastq(example_text)
            ctx.count()
            with pytest.raises(R.RfxError) as e:
                ctx.sort_kmers(E, 1.5, 95)
            assert e.value.code == R._lib.RFX_E_UNSUPPORTED
    with R.ReflexivContext(_param(R, kmerSize=31)) as ctx:
        with pytest.raises(R.RfxError) as e:
            ctx.sort_kmers()
        assert e.value.code == R._lib.RFX_E_STATE


def test_error_paths(R, example_text):
    with R.ReflexivContext(_param(R, kmerSize=31)) as ctx:
        with pytest.raises(R.RfxError) as e:
            ctx.assemble()
        assert e.value.code == R._lib.RFX_E_STATE
    with R.ReflexivContext(_param(R, kmerSize=31, bubble=False)) as ctx:
        ctx.push_fastq(example_text)
        ctx.count()
        with pytest.raises(R.RfxError) as e:
            ctx.assemble()
        assert e.value.code == R._lib.RFX_E_UNSUPPORTED
    with R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=1), table_capacity=100) as ctx:
        ctx.push_fastq(example_text)
        with pytest.raises(R.RfxError) as e:
            ctx.count()
        assert e.value.code == R._lib.RFX_E_CAPACITY


def test_pipelines_write_reference_output_trees(R, orc, example_text, tmp_path, golden):
    import gzip
    from conftest import GOLDEN
    out = tmp_path / "result"
    p = R.Parameter(["-fastq", os.path.join(GOLDEN, "paired_dat*.fq.gz"), "-outfile", str(out), "-kmer", "31", "-cover", "3"]).importCommandLine()
    R.Pipelines(p).reflexivDSMainPipe()
    text = (out / "part-00000").read_text()
    assert (out / "_SUCCESS").exists()
    recs = text.strip().split(">")[1:]
    assert len(recs) == 2
    for i, r in enumerate(recs):
        head, *lines = r.strip().split("\n")
        assert head == f"Contig-4558-(-4,-4)-{i}"
        assert all(len(x) == 100 for x in lines[:-1]) and len("".join(lines)) == 4558
    with pytest.raises(FileExistsError):
        R.Pipelines(p).reflexivDSMainPipe()
    cout = tmp_path / "counts"
    pc = R.ParameterOfCounter(["-fastq", os.path.join(GOLDEN, "paired_dat*.fq.gz"), "-outfile", str(cout), "-kmer", "31", "-cover", "2", "-gzip"]).importCommandLine()
    R.Pipelines(pc).reflexivDSCounterPipe()
    d = cout / "Count_31"
    parts = [f for f in os.listdir(d) if f.startswith("part-")]
    assert len(parts) == 1 and parts[0].endswith(".csv.gz") and (d / "_SUCCESS").exists()
    rows = sorted(gzip.open(d / parts[0]).read().decode().splitlines())
    assert hashlib.sha256(("\n".join(rows) + "\n").encode()).hexdigest() == golden["oracle"]["count_ge2"]["sha256_sorted_csv"]
    # and back in through -kmerc
    p2 = R.Parameter(["-kmerc", str(d / "part*.csv.gz"), "-outfile", str(tmp_path / "asm"), "-kmer", "31"]).importCommandLine()
    R.Pipelines(p2).reflexivDSMainPipe()
    assert (tmp_path / "asm" / "Assemble_31" / "part-00000").read_text().startswith(">Contig-4575-(-3,-3)-0\n")


def test_full_size_properties_config2_slice(R, orc):
    """Size-independent properties at a larger scale (a 1/8 slice of BASELINE config 2): the sum of counts equals the
    number of k-mer instances, the table has no duplicates, error-free 100x reads reproduce every genome k-mer with
    the right multiplicity bound, and the contigs are substrings of the genome."""
    from workload import synth
    G = 575_000
    g = synth.genome(G)
    n_pairs = synth.n_pairs_for(G, 100.0)
    txt = synth.fastq(g, n_pairs)
    with R.ReflexivContext(_param(R, kmerSize=31, minKmerCoverage=1)) as ctx:
        ctx.push_fastq(txt)
        st = ctx.count()
        keys, cnt = ctx.counts()
        assert st["n_reads"] == 2 * n_pairs and st["n_instances"] == 2 * n_pairs * 120
        assert int(cnt.astype(np.int64).sum()) == st["n_instances"]
        assert len(np.unique(keys[:, 0])) == len(keys) == st["n_distinct"]
        st = ctx.assemble()
        contigs = [c for c, _, _ in ctx.contigs()]
    gs = bytes(g).decode()
    grc = orc.revcomp_str(gs)
    assert st["n_contigs"] >= 2 and sum(len(c) for c in contigs) > 1.9 * 0.99 * G
    for c in contigs[:40]:
        assert c in gs or c in grc


def test_reflexiv_binary_matches_documented_run(R, tmp_path, golden):
    """The C++ `reflexiv` driver (csrc/reflexiv_main.cpp) with the command line of docs/example.html:303, Spark options
    included: same output tree as the reference, contig of the documented length and prefix on both strands."""
    import gzip
    import subprocess
    from conftest import GOLDEN, ROOT
    exe = os.path.join(ROOT, "reflexiv_b200", "reflexiv")
    assert os.path.exists(exe), "build() must produce the reflexiv binary"
    out = tmp_path / "result"
    r = subprocess.run([exe, "run", "--driver-memory", "3G", "--executor-memory", "3G", "-fastq", os.path.join(GOLDEN, "paired_dat*.fq.gz"),
                        "-outfile", str(out), "-kmer", "31", "-cover", "3"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Reflexiv" in r.stdout and (out / "_SUCCESS").exists()
    recs = (out / "part-00000").read_text().strip().split(">")[1:]
    seqs = ["".join(x.strip().split("\n")[1:]) for x in recs]
    assert [x.split("\n")[0] for x in recs] == ["Contig-4558-(-4,-4)-0", "Contig-4558-(-4,-4)-1"]
    assert sum(s.startswith(golden["documented"]["prefix_1200"]) for s in seqs) == 1
    # counter command, gzip output, then assembly from the counts (-kmerc)
    cout = tmp_path / "c"
    r = subprocess.run([exe, "counter", "-fastq", os.path.join(GOLDEN, "paired_dat*.fq.gz"), "-outfile", str(cout), "-kmer", "31", "-cover", "2", "-gzip"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    parts = [f for f in os.listdir(cout / "Count_31") if f.startswith("part-")]
    rows = sorted(gzip.open(cout / "Count_31" / parts[0]).read().decode().splitlines())
    assert hashlib.sha256(("\n".join(rows) + "\n").encode()).hexdigest() == golden["oracle"]["count_ge2"]["sha256_sorted_csv"]
    r = subprocess.run([exe, "run", "-kmerc", str(cout / "Count_31" / "part*"), "-outfile", str(tmp_path / "a"), "-kmer", "31"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "a" / "Assemble_31" / "part-00000").read_text().startswith(">Contig-4575-(-3,-3)-0\n")
    # reference behaviour on bad options: message, exit code 0, nothing written
    r = subprocess.run([exe, "run", "-fastq", "x", "-outfile", str(tmp_path / "z"), "-nosuch"], capture_output=True, text=True)
    assert r.returncode == 0 and "Parameter settings incorrect" in r.stdout and not (tmp_path / "z").exists()


def test_reflexiv_binary_streams_many_input_files(R, example_text, tmp_path, golden):
    """SURVEY 8f-3: the driver inflates / maps the files matching -fastq on a few host threads and pushes them one by one
    (one rfx_push_fastq per file).  Plain, gzip'ed, empty and newline-less files, one reader or many: same table."""
    import gzip
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "reflexiv_b200", "reflexiv")
    lines = example_text.split(b"\n")
    recs = [b"\n".join(lines[i:i + 4]) + b"\n" for i in range(0, len(lines) - 1, 4)]
    assert b"".join(recs) == example_text
    ind = tmp_path / "in"
    ind.mkdir()
    cuts = [0, 300, 301, 900, 1500, 1500, 2000, len(recs)]
    for j in range(len(cuts) - 1):
        blob = b"".join(recs[cuts[j]:cuts[j + 1]])
        if j % 3 == 0:
            (ind / f"part{j}.fq").write_bytes(blob)
        elif j % 3 == 1:
            (ind / f"part{j}.fq").write_bytes(blob[:-1])          # no final newline
        else:
            with gzip.open(ind / f"part{j}.fq.gz", "wb") as f:
                f.write(blob)
    tables = []
    for readers in ("1", "8"):
        out = tmp_path / f"c{readers}"
        r = subprocess.run([exe, "counter", "-fastq", str(ind / "part*"), "-outfile", str(out), "-kmer", "31", "-cover", "2"], capture_output=True, text=True,
                           env=dict(os.environ, REFLEXIV_READERS=readers))
        assert r.returncode == 0, r.stderr
        parts = [f for f in os.listdir(out / "Count_31") if f.startswith("part-")]
        tables.append(sorted((out / "Count_31" / parts[0]).read_text().splitlines()))
    assert tables[0] == tables[1]
    assert hashlib.sha256(("\n".join(tables[0]) + "\n").encode()).hexdigest() == golden["oracle"]["count_ge2"]["sha256_sorted_csv"]
    # the directory itself as input (Spark reads every file in it), run command
    r = subprocess.run([exe, "run", "-fastq", str(ind), "-outfile", str(tmp_path / "asm"), "-kmer", "31", "-cover", "3"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "asm" / "part-00000").read_text().startswith(">Contig-4558-(-4,-4)-0\n")
    r = subprocess.run([exe, "counter", "-fastq", str(tmp_path / "nothing*"), "-outfile", str(tmp_path / "n"), "-kmer", "31"], capture_output=True, text=True)
    assert r.returncode == 1 and "does not exist" in r.stderr
