"""Count_<k> tables parsed on the device (include/reflexiv_cuda.h: rfx_load_counts_csv) against the `reflexiv` binary's host parser
(csrc/reflexiv_main.cpp: parse_counts), which stays in the source as the reference: the row decoder on the host through tests/hostemu,
the call on the GPU (same table row for row, chunking, errors, round trip), the binary's -kmerc paths on one GPU and across ranks."""
import gzip
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

KS = [1, 5, 21, 31, 32, 33, 47, 61, 63]

HARNESS = r'''
#define main reflexiv_real_main
#include "%s"
#undef main
int main(int argc, char** argv) {   // <file> <k> <minc> <maxc>: parse_counts, rows as "hi lo count" (the internal key split in two words)
    std::string text;
    FILE* f = fopen(argv[1], "rb");
    char buf[1 << 16]; size_t got;
    while ((got = fread(buf, 1, sizeof(buf), f)) > 0) text.append(buf, got);
    fclose(f);
    std::vector<uint64_t> keys; std::vector<uint32_t> counts;
    const int k = atoi(argv[2]);
    if (!parse_counts(text.data(), text.size(), k, atoi(argv[3]), atoi(argv[4]), keys, counts)) { fprintf(stderr, "malformed\n"); return 2; }
    const size_t w = k <= 31 ? 1 : k / 32 + 1;
    for (size_t i = 0; i < counts.size(); i++) {
        unsigned __int128 v = keys[i * w];
        if (w == 2) v = (v << (2 * (k %% 32))) | keys[i * w + 1];   // the reference layout back to one 2k-bit integer
        printf("%%llu %%llu %%u\n", (unsigned long long)(v >> 64), (unsigned long long)v, counts[i]);
    }
    return 0;
}
'''


@pytest.fixture(scope="module")
def parse_counts_exe(tmp_path_factory):
    """The binary's parse_counts on its own (host only, no library call)."""
    d = tmp_path_factory.mktemp("parse_counts")
    src = d / "t.cpp"
    src.write_text(HARNESS % os.path.join(ROOT, "reflexiv_b200", "csrc", "reflexiv_main.cpp"))
    exe = d / "t"
    libdir = os.path.join(ROOT, "reflexiv_b200")
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "reflexiv_b200", "csrc"), "../libreflexiv_cuda.so"], check=True)
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", str(exe), str(src), "-L" + libdir, "-lreflexiv_cuda", "-lz", "-pthread", "-Wl,-rpath," + libdir], check=True)
    return str(exe)


@pytest.fixture(scope="module")
def csv_emu(tmp_path_factory):
    """tests/hostemu/counts_csv_emu.cpp: the device row decoder (rfx_counts_csv.cuh) on the host."""
    import ctypes as C
    d = tmp_path_factory.mktemp("csv_emu")
    so = d / "libcsvemu.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas", "-o", str(so),
                    os.path.join(ROOT, "tests", "hostemu", "counts_csv_emu.cpp")], check=True)
    L = C.CDLL(str(so))
    P = C.c_void_p
    L.emu_decode_counts.restype = C.c_int64
    L.emu_decode_counts.argtypes = [P, C.c_int64, C.c_int, C.c_int64, C.c_int64, P, P, P, C.c_int64]
    return L


def reference_rows(exe, tmp_path, text: bytes, k: int, minc: int, maxc: int):
    """parse_counts: (hi, lo, count) rows in text order, or None for a malformed table."""
    p = tmp_path / "t.csv"
    p.write_bytes(text)
    r = subprocess.run([exe, str(p), str(k), str(minc), str(maxc)], capture_output=True, text=True)
    if r.returncode == 2:
        return None
    assert r.returncode == 0, r.stderr
    return [tuple(int(x) for x in line.split()) for line in r.stdout.splitlines()]


def emu_rows(L, text: bytes, k: int, minc: int, maxc: int):
    """(rows, first malformed line or 0)"""
    cap = text.count(b"\n") + 1
    hi, lo, cnt = np.zeros(cap, np.uint64), np.zeros(cap, np.uint64), np.zeros(cap, np.uint32)
    n = L.emu_decode_counts(text, len(text), k, minc, maxc, hi.ctypes.data, lo.ctypes.data, cnt.ctypes.data, cap)
    if n < 0:
        return None, -n
    return [(int(a), int(b), int(c)) for a, b, c in zip(hi[:n], lo[:n], cnt[:n])], 0


def fuzz_table(rng, k: int, n: int, bad_every: int = 0) -> bytes:
    """Every row form KmerBinarizer accepts: `KMER,c` and `(KMER,c)`, CRLF, blank lines, k-mer fields longer than k, 'N' and lower
    case bases, counts of 1 to 11 digits, junk behind the count, empty counts; optionally malformed rows."""
    alpha = np.frombuffer(b"ACGTACGTACGTNacgtn", np.uint8)
    lines = []
    for i in range(n):
        extra = int(rng.integers(0, 4)) if rng.random() < 0.2 else 0
        km = bytes(alpha[rng.integers(0, len(alpha) if rng.random() < 0.3 else 4, k + extra)])
        digits = int(rng.choice([1, 2, 3, 6, 9, 9, 10, 10, 11]))
        cnt = str(int(rng.integers(10 ** (digits - 1) if digits > 1 else 0, 10 ** digits))).encode()
        tail = [b"", b"", b"", b"x", b"3x", b",7", b" "][int(rng.integers(0, 7))]
        if rng.random() < 0.05:
            cnt = b""
        row = km + b"," + cnt + tail
        form = int(rng.integers(0, 6))
        if form == 1:
            row = b"(" + row + b")"
        elif form == 2:
            row = b"(" + row
        elif form == 3:
            row = row + b")"
        end = b"\r\n" if rng.random() < 0.2 else b"\n"
        if bad_every and i % bad_every == bad_every - 1:
            row = [km[:max(k - 1, 0)] + b"," + cnt, km + cnt, b"(", b"()", b"," + km + b",5"][int(rng.integers(0, 5))]
        lines.append(row + end)
        if rng.random() < 0.05:
            lines.append(b"\n" if rng.random() < 0.5 else b"\r\n")
    text = b"".join(lines)
    if rng.random() < 0.5:
        text = text.rstrip(b"\n").rstrip(b"\r")  # no final newline
    return text


@pytest.mark.parametrize("k", KS)
def test_row_decoder_on_the_host_matches_parse_counts(parse_counts_exe, csv_emu, tmp_path, k):
    rng = np.random.default_rng(100 + k)
    for trial in range(6):
        text = fuzz_table(rng, k, 300)
        for minc, maxc in ((2, 10_000_000), (-2**31, 2**31 - 1), (5, 5000)):
            ref = reference_rows(parse_counts_exe, tmp_path, text, k, minc, maxc)
            got, bad = emu_rows(csv_emu, text, k, minc, maxc)
            assert ref is not None and bad == 0 and got == ref, (k, trial, minc, maxc)
    # malformed rows: both parsers refuse the table, the decoder names the first bad line
    for trial in range(6):
        text = fuzz_table(rng, k, 200, bad_every=37 + trial)
        assert reference_rows(parse_counts_exe, tmp_path, text, k, 1, 100) is None
        got, bad = emu_rows(csv_emu, text, k, 1, 100)
        assert got is None and bad > 0
        # the first malformed line by bisection: parse_counts accepts the lines in front of it and refuses it
        lines = text.split(b"\n")
        lo, hi = 0, len(lines)  # the first `lo` lines are accepted, the first `hi` refused
        while hi - lo > 1:
            mid = (lo + hi) // 2
            if reference_rows(parse_counts_exe, tmp_path, b"\n".join(lines[:mid]) + b"\n", k, 1, 100) is None:
                hi = mid
            else:
                lo = mid
        assert bad == hi


def test_row_decoder_edge_rows(parse_counts_exe, csv_emu, tmp_path):
    """Rows one at a time: each field boundary at every offset of a 16-byte block, the 9 / 10 / 11-digit counts, bare brackets."""
    for k in (1, 15, 16, 17, 31, 32, 63):
        km = ("ACGTTGCA" * 8)[:k]
        rows = []
        for lead in range(0, 17):
            pre = "G" * lead
            for cnt in ("0", "7", "123456789", "999999999", "1000000000", "12345678901", "12x", "", "4294967295"):
                rows.append(f"{pre}{km},{cnt}")
                rows.append(f"({km}{pre},{cnt})")
        for row in rows + ["", "\r", "(" + km + ",1", km + ",1)", "(", "()", ")", km[:-1] + ",5", km, "," + km + ",5"]:
            for end in ("\n", "\r\n", ""):
                text = (row + end).encode()
                ref = reference_rows(parse_counts_exe, tmp_path, text, k, -2**31, 2**31 - 1)
                got, bad = emu_rows(csv_emu, text, k, -2**31, 2**31 - 1)
                assert got == ref and (bad == 1) == (ref is None), (k, row, end)


# ---- on the GPU -----------------------------------------------------------------------------------------------------------------
RUN_BOUNDS = (2, 10_000_000)          # `run`: cover..maxcov
SORT_BOUNDS = (-2**31, 10_000_000)    # `sort`: INT32_MIN..maxcov


def ref_layout(rows, k):
    """(hi, lo, count) rows -> (keys in the reference layout rfx_load_counts takes, counts)"""
    w = 1 if k <= 31 else k // 32 + 1
    keys = np.zeros((len(rows), w), np.uint64)
    res = k % 32
    for i, (hi, lo, _) in enumerate(rows):
        v = (hi << 64) | lo
        if w == 1:
            keys[i, 0] = v
        else:
            keys[i, 0] = (v >> (2 * res)) & (2**64 - 1)
            keys[i, 1] = v & ((1 << (2 * res)) - 1)
    return keys, np.array([c for _, _, c in rows], np.uint32)


def ctx_for(k, **kw):
    import reflexiv_b200 as R
    return R.ReflexivContext(R.DefaultParam(kmerSize=k, **kw), device=0)


@pytest.mark.gpu
@pytest.mark.parametrize("k", KS)
def test_same_table_as_parse_counts_and_load_counts(parse_counts_exe, tmp_path, k):
    rng = np.random.default_rng(7 + k)
    text = fuzz_table(rng, k, 3000)
    with ctx_for(k) as a, ctx_for(k) as b:
        for minc, maxc in (RUN_BOUNDS, SORT_BOUNDS):
            ref = reference_rows(parse_counts_exe, tmp_path, text, k, minc, maxc)
            assert ref
            b.load_counts(*ref_layout(ref, k))
            a.load_counts_csv(text, minc, maxc)
            ka, ca = a.counts()
            kb, cb = b.counts()
            assert np.array_equal(ka, kb) and np.array_equal(ca, cb), (k, minc)
            assert a.stats()["n_rows"] == len(ref) and a.stats()["ms_parse"] > 0
        a.load_counts_csv(b"", *RUN_BOUNDS)                      # len 0: an empty table
        assert a.counts()[1].size == 0


@pytest.mark.gpu
@pytest.mark.parametrize("k", [5, 31, 61])
def test_many_chunks_and_appended_calls_equal_one_call(parse_counts_exe, tmp_path, monkeypatch, k):
    rng = np.random.default_rng(70 + k)
    text = fuzz_table(rng, k, 4000).rstrip(b"\r\n") + b"\n"
    ref = reference_rows(parse_counts_exe, tmp_path, text, k, *RUN_BOUNDS)
    with ctx_for(k) as one:
        one.load_counts_csv(text, *RUN_BOUNDS)
        want = one.counts()
    assert np.array_equal(want[1], ref_layout(ref, k)[1])
    lines = text.splitlines(keepends=True)
    for chunk in ("64", "200", "4096"):                          # rows straddle the staging chunks
        monkeypatch.setenv("RFX_CSV_CHUNK_BYTES", chunk)
        with ctx_for(k) as ctx:
            ctx.load_counts_csv(text, *RUN_BOUNDS)
            got = ctx.counts()
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), chunk
            cuts = sorted({0, len(lines)} | set(rng.integers(0, len(lines), 12).tolist()))
            for j, (lo, hi) in enumerate(zip(cuts, cuts[1:])):    # appended calls, some of them empty
                ctx.load_counts_csv(b"".join(lines[lo:hi]), *RUN_BOUNDS, append=j > 0)
                ctx.load_counts_csv(b"", *RUN_BOUNDS, append=True)
            got = ctx.counts()
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), chunk


@pytest.mark.gpu
def test_malformed_row_names_its_line_and_the_context_stays_usable(monkeypatch):
    from reflexiv_b200 import _lib
    km = "ACGT" * 7 + "ACG"
    good = "".join(f"{km},{i + 2}\n" for i in range(500)).encode()
    for chunk in (None, "128"):
        if chunk:
            monkeypatch.setenv("RFX_CSV_CHUNK_BYTES", chunk)
        with ctx_for(31) as ctx:
            kb = km.encode()
            for bad, line in ((good + b"ACGT,3\n" + good, 501), (good + b"\n" + kb + b"\n" + good + kb[:5] + b",1\n", 502), (b"(\n" + good, 1)):
                ctx.load_counts_csv(good, *RUN_BOUNDS)
                with pytest.raises(_lib.RfxError) as e:
                    ctx.load_counts_csv(bad, *RUN_BOUNDS, append=True)
                assert e.value.code == _lib.RFX_E_INVALID and f"line {line}:" in str(e.value), str(e.value)
                with pytest.raises(_lib.RfxError) as e:            # no table after a failure
                    ctx.counts()
                assert e.value.code == _lib.RFX_E_STATE
                ctx.load_counts_csv(good, *RUN_BOUNDS)
                assert ctx.counts()[1].tolist() == list(range(2, 502))


@pytest.mark.gpu
def test_counter_output_round_trip(example_text):
    """`counter -cover 2` of the example back in: the contig of the documented -kmerc run."""
    import reflexiv_b200 as R
    from reflexiv_b200.pipeline import format_contig
    with R.ReflexivContext(R.DefaultParam(kmerSize=31, minKmerCoverage=2), counter_mode=True, device=0) as ctx:
        ctx.push_fastq(example_text)
        ctx.count()
        csv = ctx.counts_csv()
    with ctx_for(31) as ctx:
        ctx.load_counts_csv(csv, *RUN_BOUNDS)
        ctx.assemble()
        seq, left, right = ctx.contigs()[0]
        assert format_contig(seq, left, right, 0).startswith(">Contig-4575-(-3,-3)-0\n")


# ---- the `reflexiv` binary ------------------------------------------------------------------------------------------------------
EXE = os.path.join(ROOT, "reflexiv_b200", "reflexiv")
ENV = dict(os.environ, REFLEXIV_ARENA_MB="768", CUDA_MODULE_LOADING="EAGER", CUDA_DEVICE_MAX_CONNECTIONS="32")


def _part_lines(d):
    out = []
    for f in sorted(os.listdir(d)):
        if f.startswith("part-"):
            data = gzip.open(d / f).read() if f.endswith(".gz") else (d / f).read_bytes()
            out += data.decode().splitlines()
    return out


def _contig_records(d):
    text = "\n".join(_part_lines(d))
    recs = [r.split("\n") for r in text.split(">")[1:]]
    return sorted((r[0].rsplit("-", 1)[0], "".join(r[1:])) for r in recs)   # header without the contig index, sequence


@pytest.fixture(scope="module")
def kmerc_tables(tmp_path_factory):
    """The example's Count_31 (`counter -cover 2`) as part files: plain and gzip, `(KMER,c)` rows and CRLF mixed in, an empty part
    file and one of two lines."""
    d = tmp_path_factory.mktemp("kmerc")
    r = subprocess.run([EXE, "counter", "-fastq", os.path.join(GOLDEN, "paired_dat*.fq.gz"), "-outfile", str(d / "c"), "-kmer", "31", "-cover", "2"],
                       capture_output=True, text=True, env=ENV)
    assert r.returncode == 0, r.stderr
    rows = _part_lines(d / "c" / "Count_31")
    rows = [f"({x})" if i % 5 == 0 else x for i, x in enumerate(rows)]
    n = len(rows)
    t = d / "t"
    t.mkdir()
    (t / "part-00000.csv").write_text("\n".join(rows[:n // 3]) + "\n")
    with gzip.open(t / "part-00001.csv.gz", "wb") as f:
        f.write(("\r\n".join(rows[n // 3:2 * n // 3]) + "\r\n").encode())
    (t / "part-00002.csv").write_text("")
    (t / "part-00003.csv").write_text("\n".join(rows[2 * n // 3:n - 2]))        # no final newline
    (t / "part-00004.csv").write_text("\n".join(rows[n - 2:]) + "\n")           # fewer lines than ranks
    (t / "_SUCCESS").write_text("")
    return t


def _run(cmd, gpus, table, out, extra=()):
    r = subprocess.run([EXE, cmd, "--gpus", str(gpus), "-kmerc", str(table), "-outfile", str(out), "-kmer", "31", *extra], capture_output=True, text=True, env=ENV)
    assert r.returncode == 0, r.stderr + r.stdout
    return r


@pytest.mark.gpu
def test_binary_matches_the_python_mirror(kmerc_tables, tmp_path):
    """`run -kmerc` / `sort -kmerc` on one GPU against Pipelines, which still parses on the host."""
    import reflexiv_b200 as R
    _run("run", 1, kmerc_tables, tmp_path / "b", ["-cover", "3"])
    p = R.Parameter(["-kmerc", str(kmerc_tables), "-outfile", str(tmp_path / "p"), "-kmer", "31", "-cover", "3"]).importCommandLine()
    R.Pipelines(p).reflexivDSMainPipe()
    assert _contig_records(tmp_path / "b" / "Assemble_31") == _contig_records(tmp_path / "p" / "Assemble_31")
    assert len(_contig_records(tmp_path / "b" / "Assemble_31")) >= 2
    _run("sort", 1, kmerc_tables, tmp_path / "b", ["-maxcov", "400"])
    p = R.Parameter(["-kmerc", str(kmerc_tables), "-outfile", str(tmp_path / "p"), "-kmer", "31", "-maxcov", "400"]).importCommandLine()
    R.Pipelines(p).reflexivLeftAndRightSortingPipe()
    got, want = _part_lines(tmp_path / "b" / "Count_31_sorted"), _part_lines(tmp_path / "p" / "Count_31_sorted")
    assert len(got) > 100 and sorted(got) == sorted(want)


@pytest.mark.gpu
@pytest.mark.parametrize("gpus", [2, 3, 4])
def test_binary_across_ranks_equals_one_gpu(kmerc_tables, tmp_path, gpus):
    _run("run", 1, kmerc_tables, tmp_path / "r1")
    _run("run", gpus, kmerc_tables, tmp_path / "rn")
    one, many = _contig_records(tmp_path / "r1" / "Assemble_31"), _contig_records(tmp_path / "rn" / "Assemble_31")
    assert one and one == many
    assert len([f for f in os.listdir(tmp_path / "rn" / "Assemble_31") if f.startswith("part-")]) == gpus
    for klist, expect_rows in (("23,31,41", True), ("23,41", False)):   # k outside -klist: an empty Count_31_sorted
        _run("sort", 1, kmerc_tables, tmp_path / "s1", ["-klist", klist])
        _run("sort", gpus, kmerc_tables, tmp_path / "sn", ["-klist", klist])
        one, many = sorted(_part_lines(tmp_path / "s1" / "Count_31_sorted")), sorted(_part_lines(tmp_path / "sn" / "Count_31_sorted"))
        assert one == many and bool(one) == expect_rows


@pytest.mark.gpu
def test_binary_reports_a_malformed_row(tmp_path):
    (tmp_path / "bad.csv").write_text("ACGTACGTACGTACGTACGTACGTACGTACG,5\nACGT,3\n")
    for gpus in (1, 2):
        r = subprocess.run([EXE, "run", "--gpus", str(gpus), "-kmerc", str(tmp_path / "bad.csv"), "-outfile", str(tmp_path / f"o{gpus}"), "-kmer", "31"],
                           capture_output=True, text=True, env=ENV)
        assert r.returncode == 1 and "malformed" in r.stderr and "line" in r.stderr, r.stderr


@pytest.mark.gpu
def test_ranks_parse_their_slices_then_shard_like_load_counts(parse_counts_exe, tmp_path):
    """Library level: every rank parses a run of whole lines, then rfx_shard_table; each shard equals, as a multiset, the shard
    that rfx_load_counts slices of the same rows give."""
    from reflexiv_b200 import sharded
    k, world = 31, 3
    rng = np.random.default_rng(11)
    text = fuzz_table(rng, k, 6000).rstrip(b"\r\n") + b"\n"
    lines = text.splitlines(keepends=True)
    cuts = [0, 1, len(lines) // 2, len(lines)]                     # one rank gets a single line
    pieces = [b"".join(lines[a:b]) for a, b in zip(cuts, cuts[1:])]
    slices = [ref_layout(reference_rows(parse_counts_exe, tmp_path, p, k, *RUN_BOUNDS), k) for p in pieces]

    def shards(load):
        ctxs = [ctx_for(k) for _ in range(world)]
        out = [None] * world
        try:
            grp = sharded.LocalRanks(ctxs, arena_bytes=256 << 20)

            def body(r, ctx):
                load(r, ctx)
                ctx.shard_table()
                keys, cnt = ctx.counts()
                out[r] = sorted(zip(keys[:, 0].tolist(), cnt.tolist()))
            grp.run(body)
        finally:
            for c in ctxs:
                c.close()
        return out

    got = shards(lambda r, ctx: (ctx.load_counts_csv(b"", *RUN_BOUNDS), ctx.load_counts_csv(pieces[r], *RUN_BOUNDS, append=True)))
    want = shards(lambda r, ctx: ctx.load_counts(*slices[r]))
    assert got == want and sum(len(x) for x in got) == sum(len(s[1]) for s in slices)
