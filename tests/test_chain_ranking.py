"""K6 / K7 on one GPU (rfx_graph.cu: graph_impl): chain lengths, tails, contig selection and contig offsets are worked out
over the splitter list, and one pass over the nodes writes the bases.  Splitters are the heads and the alive nodes whose
oriented id hashes to one (is_random_splitter); load_counts keeps the row order, so the oriented ids -- hence the
splitters -- of these inputs are known here and the cases below are checked to contain what they are meant to: chains
without a random splitter, chains whose tail is one, segments of one node, closed paths with and without splitters.
Contigs with their flags, the counts and the budget / cycle statistics are compared with the oracle under both index
layouts."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

INDEXES = ("global", "local")
STRIDE = 16  # one alive node in STRIDE is a random splitter (rfx_graph.cu: is_random_splitter)
K = 31


@pytest.fixture(scope="module")
def R():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import reflexiv_b200 as R
    R.load_library()
    return R


def _fmix32(h: int) -> int:
    h ^= h >> 16
    h = (h * 0x85EBCA6B) & 0xFFFFFFFF
    h ^= h >> 13
    h = (h * 0xC2B2AE35) & 0xFFFFFFFF
    h ^= h >> 16
    return h


def _random_splitter(oid: int) -> bool:
    return _fmix32(oid ^ 0xA5A5A5A5) % STRIDE == 0


_CODE = {ord("A"): 0, ord("C"): 1, ord("G"): 2, ord("T"): 3}


def _kmers(s: str, k: int) -> list:
    """Oriented k-mers of s, in order, as (forward, reverse complement) integers."""
    mask = (1 << (2 * k)) - 1
    out, fwd, rc = [], 0, 0
    for i, ch in enumerate(s.encode()):
        v = _CODE[ch]
        fwd = ((fwd << 2) | v) & mask
        rc = (rc >> 2) | ((3 - v) << (2 * (k - 1)))
        if i >= k - 1:
            out.append((fwd, rc))
    return out


def _rnd(rng, n: int) -> str:
    return "".join("ACGT"[i] for i in rng.integers(0, 4, n))


class Table:
    """Count table of sequences (linear, or circular: the k-mers wrap around) with every k-mer at count 10, and the
    oriented ids of each sequence's k-mers on both strands."""

    def __init__(self, linear, circular=(), k=K):
        self.k = k
        paths = [(s, False) for s in linear] + [(s, True) for s in circular]
        km = [_kmers(s + s[:k - 1] if circ else s, k) for s, circ in paths]
        keys = sorted({min(f, r) for seq in km for f, r in seq})
        row = {x: i for i, x in enumerate(keys)}
        self.keys = np.array(keys, dtype=np.uint64)
        self.counts = np.full(len(keys), 10, np.uint32)
        # oriented ids along each path, forward strand and reverse strand (in walking order)
        self.paths = []
        for (s, circ), seq in zip(paths, km):
            fwd = [2 * row[min(f, r)] + (0 if f <= r else 1) for f, r in seq]
            self.paths.append((circ, fwd, [x ^ 1 for x in reversed(fwd)]))

    def chains(self):
        for circ, fwd, rev in self.paths:
            if not circ:
                yield fwd
                yield rev

    def cycles(self):
        for circ, fwd, rev in self.paths:
            if circ:
                yield fwd
                yield rev


def _check(R, orc, monkeypatch, t: Table, min_contig: int):
    k = t.k
    zero = np.zeros(len(t.keys), np.uint64)
    ff = orc.fork_filter(zero, t.keys, t.counts, k, 8)
    a = orc.assemble(ff["keys_hi"], ff["keys_lo"], ff["left"], ff["right"], k, min_contig, orc.ASM_CANONICAL)
    want = sorted(zip(a["contigs"], a["left"].tolist(), a["right"].tolist()))
    for index in INDEXES:
        monkeypatch.setenv("RFX_GRAPH_INDEX", index)
        with R.ReflexivContext(R.DefaultParam(kmerSize=k, minContig=min_contig, minErrorCoverage=8)) as ctx:
            ctx.load_counts(t.keys.reshape(-1, 1), t.counts)
            st = ctx.assemble()
            contigs = ctx.contigs()
        assert st["n_oriented"] == len(ff["left"]), index
        assert (st["n_budget_junctions"], st["n_budget_admissible"], st["n_cycles"]) == (a["n_budget_junctions"], a["n_budget_admissible"], a["n_cycles"]), index
        assert st["n_contigs"] == len(want), index
        assert st["n_contig_bases"] == sum(len(c) for c, _, _ in want), index
        assert sorted(contigs) == want, index
    return a


def _lengths_cover_the_stride(rng, per_len=4):
    return [_rnd(rng, n + K - 1) for n in range(1, 3 * STRIDE + 1) for _ in range(per_len)]


def test_linear_chains_of_every_length_up_to_three_strides(R, orc, monkeypatch):
    """Disjoint chains of 1 .. 3 x STRIDE nodes: chains without a random splitter (their head walks the whole chain),
    tails that are random splitters (a segment of one node ends the chain), random splitters right behind the head."""
    t = Table(_lengths_cover_the_stride(np.random.default_rng(11)))
    chains = list(t.chains())
    assert any(not any(_random_splitter(x) for x in c[1:]) and len(c) > STRIDE for c in chains)
    assert any(len(c) > 1 and _random_splitter(c[-1]) for c in chains)
    assert any(len(c) > 1 and _random_splitter(c[1]) for c in chains)
    a = _check(R, orc, monkeypatch, t, K)
    assert len(a["contigs"]) == len(chains)


def test_chains_and_closed_paths_in_one_input(R, orc, monkeypatch):
    """Linear chains next to closed paths: one long enough to hold random splitters, short ones of which at least one
    strand holds none (no walk reaches it), and a 1-cycle (a homopolymer k-mer is its own successor).  The first ranking
    finds them, the cycles are opened at their smallest k-mer, the second ranking takes the path without closed ones."""
    rng = np.random.default_rng(23)
    linear = _lengths_cover_the_stride(rng, per_len=1) + ["A" * (K + 6)]
    ring = _rnd(rng, 400)
    while True:
        t = Table(linear, [ring] + [_rnd(rng, n) for n in (5, 7, 9)])
        cyc = list(t.cycles())
        if any(not any(_random_splitter(x) for x in c) for c in cyc[2:]):
            break
    assert sum(_random_splitter(x) for x in cyc[0]) >= 2 and sum(_random_splitter(x) for x in cyc[1]) >= 2
    a = _check(R, orc, monkeypatch, t, K)
    assert a["n_cycles"] > 0


@pytest.mark.parametrize("above", [0, 1])
def test_min_contig_at_a_chain_length(R, orc, monkeypatch, above):
    """minContig exactly at the length of the contig of one chain (kept) and one base above it (dropped)."""
    rng = np.random.default_rng(31)
    seqs = [_rnd(rng, n) for n in (60, 75, 90, 120)]
    a = _check(R, orc, monkeypatch, Table(seqs), 75 + above)
    assert sorted({len(c) for c in a["contigs"]}) == ([75, 90, 120] if above == 0 else [90, 120])


def test_thousands_of_contigs(R, orc, monkeypatch):
    """Several thousand chains in one call: many blocks of the splitter scan, contig offsets across them."""
    rng = np.random.default_rng(47)
    seqs = [_rnd(rng, int(n)) for n in rng.integers(K, K + 80, 3000)]
    a = _check(R, orc, monkeypatch, Table(seqs), K)
    assert len(a["contigs"]) == 6000
