"""The sharded graph stages (rfx_shard_graph.cuh: K5 request / answer passes, K6 with two levels of splitters and pointer
jumping across ranks, K7 gathering bases into the head owner's buffer) on constructed count tables whose shapes are known
on the host.

Every rank's rows are the keys whose minimiser bin it owns, and that owner is computed here independently of the
library (hostemu.emu_bins_bruteforce, bins shard-major).  counts() returns a rank's rows in the order the graph uses, so
the local oriented id of a node is 2 * row + strand and the level-1 splitters (heads, nodes whose predecessor lives on
another rank, the 1-in-64 sample sg_l1_sample) are known after the run; level-2 splitters hash ids handed out in block
order and show only in n_l2_splitters.  Each case checks that it holds the shape it names, then compares with the oracle
and with one context.  fell_back is asserted on every input: 1 exactly when the oracle finds a closed path of more than one
node, so the whole-table fallback never hides a chain-ranking error.

Ranks are host threads of one process sharing device 0."""
import ctypes as C

import numpy as np
import pytest

from test_chain_ranking import Table, _fmix32, _rnd
from test_graph_adjacency import _fq, _rc, chain_end_table, hairpin_reads, palindromic_reads_k32, palindromic_table_k12
from test_kmerc_sharded import _check_against_oracle, _contiguous, _oracle_table, _ref_layout

pytestmark = pytest.mark.gpu

E, FOLD, KMAX = 8, 1.5, 95
BINS_PER_RANK = 96  # shard_set_bins(96 * world): m = 11 (m = k below 11)
ARENA = 256 << 20
L1_STRIDE = 64      # sg_l1_sample


@pytest.fixture(scope="module")
def R():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import reflexiv_b200 as R
    R.load_library()
    return R


class _Groups:
    """LocalRanks groups (and one-context runs) by (world, k, minContig).  Only the last one stays open: groups of ranks
    that share the device are run one at a time, as everywhere in the suite."""

    def __init__(self, R, keep=1):
        self.R, self.keep, self.live = R, keep, {}

    def _ctx(self, k, min_contig):
        return self.R.ReflexivContext(self.R.DefaultParam(kmerSize=k, minContig=min_contig, minErrorCoverage=E), device=0)

    def _open(self, key, make):
        if key not in self.live:
            while len(self.live) >= self.keep:
                for c in self.live.pop(next(iter(self.live)))[0]:
                    c.close()
            self.live[key] = make()
        return self.live[key]

    def get(self, world, k, min_contig):
        from reflexiv_b200 import sharded

        def make():
            ctxs = [self._ctx(k, min_contig) for _ in range(world)]
            return ctxs, sharded.LocalRanks(ctxs, arena_bytes=ARENA)
        return self._open((world, k, min_contig), make)[1]

    def single(self, k, min_contig):
        return self._open(("one", k, min_contig), lambda: ([self._ctx(k, min_contig)], None))[0][0]

    def close(self):
        for ctxs, _ in self.live.values():
            for c in ctxs:
                c.close()
        self.live = {}


@pytest.fixture(scope="module")
def groups(R):
    g = _Groups(R)
    yield g
    g.close()


# ---- where rows live -------------------------------------------------------------------------------------------------------
def _owners(hostemu, hi, lo, k, world):
    """Owner rank of every key (oracle form: hi / lo words of the right-aligned 2k bits): the keys are packed back to back as
    one read, emu_bins_bruteforce gives the bin of every k-mer position, every k-th is a key."""
    n = len(lo)
    if n == 0:
        return np.zeros(0, np.int64)
    B = BINS_PER_RANK * world
    sh = 2 * (k - 1 - np.arange(k))
    hi = np.asarray(hi, np.uint64)[:, None]
    lo = np.asarray(lo, np.uint64)[:, None]
    from_lo = (lo >> np.minimum(sh, 63).astype(np.uint64)) & np.uint64(3)
    from_hi = (hi >> np.maximum(sh - 64, 0).astype(np.uint64)) & np.uint64(3)
    codes = np.where(sh[None, :] >= 64, from_hi, from_lo).ravel()
    L = len(codes)
    nw = (L + 31) // 32 + 1
    pad = np.zeros(nw * 32, np.uint64)
    pad[:L] = codes
    words = np.ascontiguousarray(np.bitwise_or.reduce(pad.reshape(nw, 32) << (62 - 2 * np.arange(32)).astype(np.uint64), axis=1))
    bins = np.zeros(L - k + 1, np.uint32)
    hostemu.emu_bins_bruteforce(words.ctypes.data, C.c_uint32(L), k, min(k, 11), C.c_uint32(B), bins.ctypes.data)
    return bins[::k].astype(np.int64) // BINS_PER_RANK


def _ints(strs):
    code = {"A": 0, "C": 1, "G": 2, "T": 3}
    out = []
    for s in strs:
        v = 0
        for ch in s:
            v = (v << 2) | code[ch]
        out.append(v)
    return out


def _split(ints):
    return (np.array([x >> 64 for x in ints], np.uint64), np.array([x & ((1 << 64) - 1) for x in ints], np.uint64))


def _owner_of_strs(hostemu, strs, k, world):
    return _owners(hostemu, *_split(_ints(strs)), k, world).tolist()


def _table_of(t: Table):
    return dict(keys_hi=np.zeros(len(t.keys), np.uint64), keys_lo=t.keys, counts=t.counts)


def _key_ints(t):
    return [(int(h) << 64) | int(lo) for h, lo in zip(t["keys_hi"], t["keys_lo"])]


# ---- one sharded run and its checks ---------------------------------------------------------------------------------------
def _body(slices, bins, results, sort):
    def body(rank, ctx):
        ctx.reset()
        ctx.load_counts(*slices[rank])
        ctx.shard_set_bins(bins)
        st = ctx.shard_table()
        keys, cnt = ctx.counts()
        st2 = ctx.assemble_sharded()
        sh = ctx.shard_stats()
        res = dict(keys=keys, cnt=cnt, st=st, st2=st2, sh=sh, ori=None if sh["fell_back"] else ctx.oriented(), contigs=ctx.contigs())
        if sort:
            res["n_sorted"] = ctx.sort_kmers_sharded(E, FOLD, KMAX)
            res["rows"] = ctx.sorted_rows()
        results[rank] = res
    return body


def _lex(hi, lo, *rest):
    o = np.lexsort((lo, hi))
    return [a[o] for a in (hi, lo) + rest]


def _closed_path(orc, t, k, a):
    """The oracle's walk found a closed path of more than one node: n_cycles counts those and the joining 1-cycles
    (a surviving homopolymer k-mer is its own successor)."""
    f = orc.fork_filter(t["keys_hi"], t["keys_lo"], t["counts"], k, E)
    homo = {sum(b << (2 * i) for i in range(k)) for b in range(4)}
    n_self = sum(((int(h) << 64) | int(lo)) in homo and (le < 0) == (ri < 0) for h, lo, le, ri in zip(f["keys_hi"], f["keys_lo"], f["left"], f["right"]))
    return a["n_cycles"] > n_self


def run_case(hostemu, orc, groups, t, k, world, min_contig=None, sort=False, closed=False):
    """Shards the table t (oracle form, sorted keys) over `world` ranks and checks placement, fork filters, contigs and
    statistics against the host, the oracle and one context.  `closed`: whether the table holds a closed path (None: not
    asserted).  Returns (results, key -> owner, oracle assembly)."""
    min_contig = k if min_contig is None else min_contig
    keys, cnt = _ref_layout(t, k), t["counts"].astype(np.uint32)
    grp = groups.get(world, k, min_contig)
    results = [None] * world
    grp.run(_body(_contiguous(keys, cnt, world), BINS_PER_RANK * world, results, sort))
    from reflexiv_b200.pipeline import keys_to_int
    # placement: every rank holds exactly the keys the host assigns it
    ints = _key_ints(t)
    owner = dict(zip(ints, _owners(hostemu, t["keys_hi"], t["keys_lo"], k, world).tolist()))
    for r, res in enumerate(results):
        assert res["st"]["n_bins"] == BINS_PER_RANK * world
        assert sorted(keys_to_int(res["keys"], k)) == sorted(x for x in ints if owner[x] == r), f"rank {r}: rows"
    a, fell_back = _check_against_oracle(orc, t, k, E, min_contig, results)
    is_closed = _closed_path(orc, t, k, a)
    if closed is not None:
        assert is_closed == closed
    assert [r["sh"]["fell_back"] for r in results] == [int(is_closed)] * world
    assert all(r["sh"]["n_contigs_global"] == len(a["contigs"]) for r in results)
    if not is_closed:
        for r, res in enumerate(results):
            assert res["sh"]["n_l1_splitters"] > 0 or len(res["ori"][0]) == 0, r
            for s, _, _ in res["contigs"]:  # a contig lives with the owner of its first k-mer
                x = _ints([s[:k]])[0]
                assert owner[min(x, _rc(x, k))] == r, (r, s)
    # one context on the whole table
    single = groups.single(k, min_contig)
    single.reset()
    single.load_counts(keys, cnt)
    single.assemble()
    assert sorted(x for r in results for x in r["contigs"]) == sorted(single.contigs())
    if not fell_back:
        got = [np.concatenate([r["ori"][i] for r in results]) for i in range(4)]
        assert all(np.array_equal(x, y) for x, y in zip(_lex(*got), _lex(*single.oriented())))
    if sort:
        ref = orc.sorted_rows(t["keys_hi"], t["keys_lo"], t["counts"], k, E, FOLD, KMAX)
        got = _lex(*[np.concatenate([r["rows"][i] for r in results]) for i in range(4)])
        assert all(np.array_equal(x, ref[n]) for x, n in zip(got, ("keys_hi", "keys_lo", "left", "right")))
        assert sum(r["n_sorted"] for r in results) == len(ref["left"])
        single.sort_kmers(E, FOLD, KMAX)
        assert all(np.array_equal(x, y) for x, y in zip(got, _lex(*single.sorted_rows())))
    return results, owner, a


# ---- K6: level-1 segments ---------------------------------------------------------------------------------------------------
def _l1_sample(oid: int) -> bool:
    return (_fmix32(oid ^ 0xA5A5A5A5) & (L1_STRIDE - 1)) == 0


def _local_oids(results, k):
    """canonical key -> (rank, local row) after shard_table: counts() lists the rows in the order the graph numbers them."""
    from reflexiv_b200.pipeline import keys_to_int
    return {x: (r, i) for r, res in enumerate(results) for i, x in enumerate(keys_to_int(res["keys"], k))}


def _chain_nodes(t: Table, owner, where):
    """Per chain of t (both strands of every linear sequence): [(owner rank, level-1 sample?)] of its nodes in walking order."""
    out = []
    for chain in t.chains():
        nodes = []
        for oid in chain:
            key = int(t.keys[oid >> 1])
            rank, row = where[key]
            assert owner[key] == rank
            nodes.append((rank, _l1_sample(2 * row + (oid & 1))))
        out.append(nodes)
    return out


def _one_rank_chains(hostemu, rng, k, world, n, lo=66, hi=72):
    """Chains of lo..hi nodes whose every k-mer holds the same m-mer M (spaced at most w = k - m + 1 apart, random bases
    between), M being the minimiser of all of them: every node in one bin, on one rank."""
    w = k - 11 + 1
    out = []
    while len(out) < n:
        M = _rnd(rng, 11)
        for _ in range(n - len(out)):
            nodes = int(rng.integers(lo, hi + 1))
            s = M
            while len(s) < nodes + k - 1:
                s += _rnd(rng, int(rng.integers(4, w - 11 + 1))) + M
            s = s[:nodes + k - 1]
            if len(set(_owner_of_strs(hostemu, [s[i:i + k] for i in range(nodes)], k, world))) != 1:
                break  # M is not the minimiser everywhere: another M
            out.append(s)
    return out


def _alternating_chains(hostemu, rng, k, world, n, run=8, nodes=30):
    """Chains of `nodes` k-mers whose owner changes at `run` consecutive nodes: one-node level-1 segments on alternating ranks."""
    out = []
    while len(out) < n:
        s = _rnd(rng, k)
        prev = _owner_of_strs(hostemu, [s], k, world)[0]
        while len(s) - k + 1 < nodes:
            cand = [s[len(s) - k + 1:] + b for b in "ACGT"]
            own = _owner_of_strs(hostemu, cand, k, world)
            ok = [i for i in rng.permutation(4) if own[i] != prev] if len(s) - k + 1 <= run else list(rng.permutation(4))
            if not ok:
                break
            s += "ACGT"[ok[0]]
            prev = own[ok[0]]
        else:
            out.append(s)
    return out


@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
def test_level1_segments(R, orc, hostemu, groups, world):
    """k = 31: chains of 1 .. 3 x 64 nodes and chains of more than 64 nodes on one rank (one walk covers those without a
    sample behind the head); heads whose successor lives on another rank and tails that are cross-rank splitters.  k = 12:
    chains whose owner changes at 8 consecutive nodes (segments of one node, every link a cross-rank one)."""
    rng = np.random.default_rng(1000 + world)
    k = 31
    seqs = [_rnd(rng, n + k - 1) for n in range(1, 3 * L1_STRIDE + 1)] + _one_rank_chains(hostemu, rng, k, world, 24)
    t = Table(seqs, k=k)
    results, owner, a = run_case(hostemu, orc, groups, _table_of(t), k, world)
    real = set(a["contigs"])
    chains = [c for c, s in zip(_chain_nodes(t, owner, _local_oids(results, k)), (x for s in seqs for x in (s, orc.revcomp_str(s)))) if s in real]
    assert len(chains) == 2 * len(seqs)  # every sequence is a chain of the graph, on both strands
    assert max(len(c) for c in chains) == 3 * L1_STRIDE
    assert any(len(c) > L1_STRIDE and len({r for r, _ in c}) == 1 and not any(x for _, x in c[1:]) for c in chains)
    if world > 1:
        assert any(len(c) > 1 and c[0][0] != c[1][0] for c in chains)     # a head whose successor lives on another rank
        assert any(len(c) > 1 and c[-1][0] != c[-2][0] for c in chains)   # a tail that is a cross-rank level-1 splitter
        assert all(res["sh"]["n_remote_probes"] > 0 for res in results)
        k = 12
        seqs = _alternating_chains(hostemu, rng, k, world, 8)
        t = Table(seqs, k=k)
        results, owner, a = run_case(hostemu, orc, groups, _table_of(t), k, world)
        real = set(a["contigs"])
        chains = [c for c, s in zip(_chain_nodes(t, owner, _local_oids(results, k)), (x for s in seqs for x in (s, orc.revcomp_str(s)))) if s in real]
        assert any(all(c[i][0] != c[i - 1][0] for i in range(j, j + 8)) for c in chains for j in range(1, len(c) - 7))


# ---- K6: level 2 and pointer jumping ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [3, 8])
def test_level2_walks_and_jumping(R, orc, hostemu, groups, world):
    """Three linear sequences of 20 kb (six chains): their level-1 lists cross ranks at every owner change, and some chain's
    level-2 list has more than 32 entries, so pointer jumping needs at least 6 rounds.  Not one of them may look closed."""
    rng = np.random.default_rng(77 + world)
    k = 31
    seqs = [_rnd(rng, 20_000) for _ in range(3)]
    t = Table(seqs, k=k)
    results, owner, a = run_case(hostemu, orc, groups, _table_of(t), k, world)
    assert sorted(a["contigs"]) == sorted(seqs + [orc.revcomp_str(s) for s in seqs])
    chains = _chain_nodes(t, owner, _local_oids(results, k))
    assert all(sum(c[i][0] != c[i - 1][0] for i in range(1, len(c))) > 500 for c in chains)
    n_l2 = sum(r["sh"]["n_l2_splitters"] for r in results)
    assert n_l2 > 32 * len(chains)  # > the 6 heads, and one list at least 33 long
    assert all(r["sh"]["fell_back"] == 0 for r in results)


# ---- K7: gathering the bases ----------------------------------------------------------------------------------------------
def _shared_words(results, owner, k):
    """Words of 8 bytes of a rank's contig buffer that hold bases of several contigs written by several ranks (a node's
    base comes from the node's owner, the first k - 1 bases of a contig from its head's)."""
    n = 0
    for res in results:
        writers = {}
        pos = 0
        for s, _, _ in res["contigs"]:
            nodes = _ints(s[i:i + k] for i in range(len(s) - k + 1))
            who = [owner[min(x, _rc(x, k))] for x in nodes]
            for j in range(len(s)):
                writers.setdefault((pos + j) >> 3, set()).add((pos, who[max(0, j - (k - 1))]))
            pos += len(s)
        n += sum(len({c for c, _ in v}) > 1 and len({w for _, w in v}) > 1 for v in writers.values())
    return n


@pytest.mark.parametrize("world", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("k", [11, 12])
def test_gather_short_contigs(R, orc, hostemu, groups, monkeypatch, world, k):
    """About 3000 chains of 1 .. 10 nodes (contigs of k .. k + 9 bases): several contigs, written by different ranks, share
    one 8-byte word of the head owner's buffer.  Byte stores (RFX_GATHER=nodes) and packed words OR-ed in per segment
    (=segments)."""
    rng = np.random.default_rng(300 + 10 * world + k)
    n_nodes = np.minimum(rng.geometric(0.3, 3000), 10)
    assert (n_nodes == 1).sum() > 500
    t = Table([_rnd(rng, int(n) + k - 1) for n in n_nodes], k=k)
    for mode in ("nodes", "segments"):
        monkeypatch.setenv("RFX_GATHER", mode)
        results, owner, a = run_case(hostemu, orc, groups, _table_of(t), k, world)
        assert len(a["contigs"]) > 5000
        if world > 1:
            assert _shared_words(results, owner, k) > 100


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("above", [0, 1])
def test_min_contig_at_a_chain_length(R, orc, hostemu, groups, world, above):
    """minContig exactly at the length of some contigs (kept) and one base above it (dropped), across ranks."""
    rng = np.random.default_rng(500 + world)
    k = 12
    t = Table([_rnd(rng, n) for n in range(k, 40) for _ in range(20)], k=k)
    _, _, a = run_case(hostemu, orc, groups, _table_of(t), k, world, min_contig=20 + above)
    lens = {len(c) for c in a["contigs"]}
    assert (20 in lens) == (above == 0) and min(lens) == 20 + above


# ---- K5 shapes across ranks ---------------------------------------------------------------------------------------------------
def _table_from_keys(keys, counts):
    return dict(keys_hi=np.zeros(len(keys), np.uint64), keys_lo=np.asarray(keys, np.uint64), counts=np.asarray(counts, np.uint32))


def _chain_end_split(hostemu, k, tip_count, world):
    """The chain-end table of the first seed whose head group or tail group has its two siblings on different ranks: each
    asks the other's owner for its count (pass 2)."""
    for seed in range(400):
        seqs, keys, counts = chain_end_table(k, tip_count, seed)
        g = seqs[0]
        own = _owner_of_strs(hostemu, [g[:k], seqs[2], g[-k:], seqs[3][-k:]], k, world)
        if own[0] != own[1] or own[2] != own[3]:
            return _table_from_keys(keys, counts)
    raise AssertionError("no seed splits a chain-end group across ranks")


def _read_table(orc, txt, k):
    t = _oracle_table(orc, txt, k, 2)
    return dict(keys_hi=t["keys_hi"], keys_lo=t["keys_lo"], counts=t["counts"])


def _k5_table(orc, hostemu, case, world):
    """(table, k, closed, sort) of a K5 case."""
    name, *arg = case
    if name == "palindromes12":
        glen, seed, closed = arg
        return _table_from_keys(*palindromic_table_k12(glen, seed)), 12, closed, True
    if name == "palindromes32":
        return _read_table(orc, palindromic_reads_k32(at_stretch=arg[0]), 32), 32, arg[0], False  # no sorted stage at k = 32
    if name == "chain_ends":
        k, tip = arg
        return _chain_end_split(hostemu, k, tip, world), k, False, True
    if name == "hairpins":
        return _read_table(orc, hairpin_reads(arg[0])[2], arg[0]), arg[0], None, True
    if name == "homopolymer":
        return _read_table(orc, _fq(["A" * 100] * 3), 31), 31, False, False
    if name == "homopolymer_branch":
        tail = _rnd(np.random.default_rng(5), 80)
        return _read_table(orc, _fq(["A" * 60 + tail] * 3 + ["C" * 50 + "A" * 60] * 3), 31), 31, False, False
    if name == "acgt":
        return _read_table(orc, _fq(["ACGT" * 30] * 3), 16), 16, None, False
    raise KeyError(name)


# the palindrome tables of test_graph_adjacency: (3000, 1) and the AT stretch at k = 32 hold closed paths, the others none
K5_CASES = [("palindromes12", 3000, 1, True), ("palindromes12", 20000, 2, False), ("chain_ends", 12, 2), ("chain_ends", 12, 11),
            ("palindromes32", False), ("palindromes32", True), ("chain_ends", 31, 2), ("chain_ends", 31, 11), ("homopolymer",), ("homopolymer_branch",),
            ("hairpins", 31), ("hairpins", 33), ("hairpins", 61), ("acgt",)]


@pytest.mark.parametrize("case,world", [(c, w) for c in K5_CASES for w in (2, 3)], ids=lambda v: "-".join(map(str, v)) if isinstance(v, tuple) else str(v))
def test_k5_shapes(R, orc, hostemu, groups, case, world):
    """Palindromic rows (even k: one node for two strands), fork groups at chain ends with siblings on different ranks,
    1-cycles with and without a branch, hairpins at odd k (a node whose successor group holds its own row's other strand;
    k = 33, 61: two-word keys) and "ACGT" * 30 at k = 16.  Fork flags and survivors, contigs, and the sorted stage
    (sort_kmers_sharded; it rejects k = 32) against the oracle and one context."""
    t, k, closed, sort = _k5_table(orc, hostemu, case, world)
    results, owner, a = run_case(hostemu, orc, groups, t, k, world, sort=sort, closed=closed)
    if case[0] == "palindromes12":
        assert sum(x == _rc(x, k) for x in owner) >= 20
    if case[0] in ("palindromes12", "palindromes32", "chain_ends"):
        assert sum(r["sh"]["n_remote_probes"] for r in results) > 0
    if case[0].startswith("homopolymer"):
        assert "A" * 31 in {s for r in results for s, _, _ in r["contigs"]}  # a contig of its own
