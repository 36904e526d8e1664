"""K5 reads every neighbour set from the stored out-sets N(Y) of the adjacency pass (rfx_graph.cu: adjacency_kernel): the
predecessors, the right-filter group and the left-filter group of a node are all reached through a neighbour's set.
These cases pin what the oracle comparisons of test_gpu_parity reach only by chance: palindromic rows (even k, one node
for two strands), fork groups at chain ends that no stored set names (the direct-probe fallback), a 1-cycle and a
circular genome, and dense forks where the sets hold 3-4 entries.  Fork flags, survivors, budget / cycle statistics
and contigs are compared with the oracle under both index layouts."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

INDEXES = ("global", "local")


@pytest.fixture(scope="module")
def R():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import reflexiv_b200 as R
    R.load_library()
    return R


def _codes(s) -> list:
    table = {ord("A"): 0, ord("C"): 1, ord("G"): 2, ord("T"): 3}
    b = s.encode() if isinstance(s, str) else bytes(s)
    return [table[x] for x in b]


def _rc(x: int, k: int) -> int:
    r = 0
    for _ in range(k):
        r = (r << 2) | (3 - (x & 3))
        x >>= 2
    return r


def _table(seqs, k: int, count_of):
    """Canonical k-mer table (k <= 31) of the sequences; count_of(key, index of the sequence) gives the count of a k-mer
    the first time it is seen."""
    mask = (1 << (2 * k)) - 1
    seen = {}
    for si, s in enumerate(seqs):
        fwd = rc = 0
        for i, v in enumerate(_codes(s)):
            fwd = ((fwd << 2) | v) & mask
            rc = (rc >> 2) | ((3 - v) << (2 * (k - 1)))
            if i >= k - 1:
                key = min(fwd, rc)
                seen.setdefault(key, count_of(key, si))
    keys = np.array(sorted(seen), dtype=np.uint64)
    counts = np.array([seen[int(x)] for x in keys], dtype=np.uint32)
    return keys, counts


def _check_table(R, orc, monkeypatch, keys, counts, k, E=8):
    zero = np.zeros(len(keys), np.uint64)
    ff = orc.fork_filter(zero, keys, counts, k, E)
    a = orc.assemble(ff["keys_hi"], ff["keys_lo"], ff["left"], ff["right"], k, k, orc.ASM_CANONICAL)
    for index in INDEXES:
        monkeypatch.setenv("RFX_GRAPH_INDEX", index)
        with R.ReflexivContext(R.DefaultParam(kmerSize=k, minContig=k, minErrorCoverage=E)) as ctx:
            ctx.load_counts(keys.reshape(-1, 1), counts)
            st = ctx.assemble()
            hi, lo, le, ri = ctx.oriented()
            contigs = ctx.contigs()
        order = np.lexsort((lo, hi))
        assert np.array_equal(lo[order], ff["keys_lo"]), index
        assert np.array_equal(le[order], ff["left"]) and np.array_equal(ri[order], ff["right"]), index
        assert st["n_oriented"] == len(ff["left"]), index
        assert (st["n_budget_junctions"], st["n_budget_admissible"], st["n_cycles"]) == (a["n_budget_junctions"], a["n_budget_admissible"], a["n_cycles"]), index
        assert sorted(contigs) == sorted(zip(a["contigs"], a["left"].tolist(), a["right"].tolist())), index
    return ff, a


def _fq(seqs) -> bytes:
    return "".join(f"@r{i}\n{s}\n+\n{'I' * len(s)}\n" for i, s in enumerate(seqs)).encode()


def _check_reads(R, orc, monkeypatch, txt, k, cover, E=8, min_contig=10):
    ref = orc.run_pipeline(txt, k=k, cover=cover, min_error_cov=E, min_contig=min_contig)
    f, a = ref["forks"], ref["asm"]
    for index in INDEXES:
        monkeypatch.setenv("RFX_GRAPH_INDEX", index)
        with R.ReflexivContext(R.DefaultParam(kmerSize=k, minKmerCoverage=cover, minErrorCoverage=E, minContig=min_contig)) as ctx:
            ctx.push_fastq(txt)
            ctx.count()
            st = ctx.assemble()
            hi, lo, le, ri = ctx.oriented()
            contigs = ctx.contigs()
        order = np.lexsort((lo, hi))
        assert np.array_equal(hi[order], f["keys_hi"]) and np.array_equal(lo[order], f["keys_lo"]), index
        assert np.array_equal(le[order], f["left"]) and np.array_equal(ri[order], f["right"]), index
        assert st["n_oriented"] == len(f["left"]), index
        assert (st["n_budget_junctions"], st["n_budget_admissible"], st["n_cycles"]) == (a["n_budget_junctions"], a["n_budget_admissible"], a["n_cycles"]), index
        assert sorted(contigs) == sorted(zip(a["contigs"], a["left"].tolist(), a["right"].tolist())), index
    return ref


def _palindromes(rng, half: int, n: int) -> list:
    out = []
    for _ in range(n):
        s = "".join("ACGT"[i] for i in rng.integers(0, 4, half))
        out.append(s + s[::-1].translate(str.maketrans("ACGT", "TGCA")))
    return out


def palindromic_table_k12(glen: int, seed: int):
    """k = 12 table: a genome with 40 palindromic 12-mers spliced in, each palindrome again with other flanks."""
    from workload import synth
    k = 12
    rng = np.random.default_rng(seed)
    g = synth.genome(glen, 500 + seed).tobytes().decode()
    pals = _palindromes(rng, k // 2, 40)
    # each palindrome twice, with different flanks: forks on both sides of a palindromic node
    parts, pos = [], 0
    for p in pals:
        parts.append(g[pos:pos + 40] + p)
        pos += 40
    seqs = ["".join(parts) + g[pos:], "".join(p + g[i * 7:i * 7 + 5] for i, p in enumerate(pals))]
    return _table(seqs, k, lambda key, si: 10 + (hash((key, seed)) % 3) if si == 0 else 2 + (key % 15))


@pytest.mark.parametrize("glen,seed", [(3000, 1), (20000, 2)])
def test_palindromic_rows_at_k12(R, orc, monkeypatch, glen, seed):
    """Even k: a palindromic row is one node (find returns its even id, the odd id is dead).  Its predecessors and its
    left group are reached through the other strand of a neighbour; that strand must be mapped back to the even id, or a
    palindromic candidate's count is dropped from a left group.  Palindromes sit inside real forks here (repeated
    11-mers at this genome size)."""
    keys, counts = palindromic_table_k12(glen, seed)
    n_pal = sum(int(x) == _rc(int(x), 12) for x in keys)
    assert n_pal >= 20
    _check_table(R, orc, monkeypatch, keys, counts, 12)


def palindromic_reads_k32(at_stretch: bool = True) -> bytes:
    """Reads (0.5 % errors) of a genome with a palindromic AT stretch (a closed path) and 12 palindromic 32-mers, one of
    them twice."""
    from workload import synth
    rng = np.random.default_rng(7)
    g = synth.genome(30_000, 732)
    if at_stretch:
        g[20000:20060] = np.frombuffer(b"AT" * 30, np.uint8)
    for i, p in enumerate(_palindromes(rng, 16, 12)):
        g[2000 + 1500 * i:2000 + 1500 * i + 32] = np.frombuffer(p.encode(), np.uint8)
    g[25000:25032] = g[2000:2032]  # one palindrome twice: forks around it
    return bytes(synth.fastq(g, 6000, read_len=150, frag_len=400, error_rate=0.005, seed_reads=11, seed_errors=12))


def test_palindromic_rows_at_k32(R, orc, monkeypatch):
    """k = 32 (two-word keys): palindromic stretches and embedded palindromes in a read set, with repeats."""
    _check_reads(R, orc, monkeypatch, palindromic_reads_k32(), 32, 2, min_contig=100)


def chain_end_table(k: int, tip_count: int, seed: int = 0):
    """A 3000-base genome (counts 10..12) with forks at both chain ends and three dead ends inside, the tips at tip_count.
    Returns the sequences (the genome first, then the branches of the head group, the tail group and the dead ends), keys
    and counts."""
    from workload import synth
    rng = np.random.default_rng(100 + k + tip_count + 1000 * seed)
    g = synth.genome(3000, 900 + k + 1000 * seed).tobytes().decode()

    def other(b):
        return "ACGT"[("ACGT".index(b) + 1 + int(rng.integers(0, 3))) % 4]

    def rnd(n):
        return "".join("ACGT"[i] for i in rng.integers(0, 4, n))
    seqs = [g]
    seqs.append(g[:k - 1] + other(g[k - 1]) + rnd(20))        # right group at the head: prefix(first k-mer)·b'
    seqs.append(g[:k - 1] + other(g[k - 1]))                  # one lone k-mer in the same group (no successor either)
    seqs.append(rnd(20) + other(g[-k]) + g[-(k - 1):])        # left group at the tail: a'·suffix(last k-mer)
    for i in (700, 1500, 2200):                               # dead ends inside the genome: a tip k-mer and its left sibling
        y = g[i:i + k - 1] + other(g[i + k - 1])
        seqs.append(y)
        seqs.append(other(y[0]) + y[1:])
    keys, counts = _table(seqs, k, lambda key, si: 10 + (key % 3) if si == 0 else tip_count)
    return seqs, keys, counts


@pytest.mark.parametrize("k", [31, 12])
@pytest.mark.parametrize("tip_count", [2, 11])
def test_fork_groups_at_chain_ends(R, orc, monkeypatch, k, tip_count):
    """Siblings without a predecessor (forks at the first k-mer of a sequence) and without a successor (forks at the
    last one): no stored out-set names their groups, so each node probes its siblings directly.  Tips as errors (count 2
    against 10..12) and as real forks (count 11)."""
    _, keys, counts = chain_end_table(k, tip_count)
    ff, _ = _check_table(R, orc, monkeypatch, keys, counts, k)
    assert (ff["left"] >= 0).any() or (ff["right"] >= 0).any() or tip_count == 2


def test_one_cycle_and_circular_genome(R, orc, monkeypatch):
    """A node that is its own successor (homopolymer), the same with a branch leaving it, and a circular genome (one
    closed path per strand, no head anywhere)."""
    rng = np.random.default_rng(5)
    circ = "".join("ACGT"[i] for i in rng.integers(0, 4, 400))
    _check_reads(R, orc, monkeypatch, _fq([(circ + circ)[i:i + 120] for i in range(0, 400, 7)] * 3), 31, 2, min_contig=50)
    _check_reads(R, orc, monkeypatch, _fq(["A" * 100] * 3), 31, 2)
    _check_reads(R, orc, monkeypatch, _fq(["A" * 60 + circ[:80]] * 3 + ["C" * 50 + "A" * 60] * 3), 31, 2)
    _check_reads(R, orc, monkeypatch, _fq(["ACGT" * 30] * 3), 16, 2)


def hairpin_reads(k: int, seed: int = 0):
    """Odd k: error-free reads (every 5 bases, twice) of a 3000-base genome with six palindromic (k-1)-mers P spliced in.
    The node X = aP (a the base in front of P) has rc(X) = P·comp(a) among its successors: where the genome goes on with
    comp(a) that is its only successor (a straight hairpin), elsewhere a fork against X's own row.  Returns the genome, the
    sites (start of P, straight or not) and the FASTQ text."""
    from workload import synth
    assert k % 2 == 1
    comp = dict(zip("ACGT", "TGCA"))
    rng = np.random.default_rng(60 + k + 1000 * seed)
    g = list(synth.genome(3000, 960 + k + 1000 * seed).tobytes().decode())
    sites = []
    for i, p in enumerate(_palindromes(rng, (k - 1) // 2, 6)):
        at, straight = 200 + 450 * i, i % 2 == 0
        g[at:at + k - 1] = p
        c = comp[g[at - 1]]
        g[at + k - 1] = c if straight else "ACGT"[("ACGT".index(c) + 1 + int(rng.integers(0, 3))) % 4]
        sites.append((at, straight))
    g = "".join(g)
    return g, sites, _fq([g[i:i + 120] for i in range(0, len(g) - 119, 5)] * 2)


@pytest.mark.parametrize("k", [31, 33, 61])
def test_hairpins_at_odd_k(R, orc, monkeypatch, k):
    """A palindromic (k-1)-mer inside a genome: a node whose successor group holds the other strand of its own row, alone
    (straight hairpin) or next to the genome's successor (a fork against the own row).  k = 33 and 61: two-word keys."""
    g, sites, txt = hairpin_reads(k)
    comp = dict(zip("ACGT", "TGCA"))
    for at, straight in sites:
        p = g[at:at + k - 1]
        assert p == p[::-1].translate(str.maketrans("ACGT", "TGCA"))
        assert (g[at + k - 1] == comp[g[at - 1]]) == straight
    assert {s for _, s in sites} == {True, False}
    _check_reads(R, orc, monkeypatch, txt, k, 2, min_contig=k)


@pytest.mark.parametrize("skewed", [False, True])
def test_dense_forks_at_k11(R, orc, monkeypatch, skewed):
    """k = 11 over 200 kb: thousands of (k-1)-mers have 3 or 4 extensions, so many groups of the filters are read from stored
    sets with several entries.  Near-equal counts give real forks, skewed counts error forks."""
    from workload import synth
    k = 11
    g = synth.genome(200_000, 311)
    keys, counts = _table([g.tobytes()], k, (lambda key, si: 1 + (hash((key, 3)) % 40)) if skewed else (lambda key, si: 10 + (hash((key, 3)) % 3)))
    ext = {}
    for x in keys.tolist():
        for y in (x, _rc(x, k)):
            ext.setdefault(y >> 2, set()).add(y & 3)
    assert sum(len(v) >= 3 for v in ext.values()) > 1000 and any(len(v) == 4 for v in ext.values())
    _check_table(R, orc, monkeypatch, keys, counts, k)
