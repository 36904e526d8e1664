"""rfx_stitch_begin_sharded / rfx_stitch_finish_sharded on the host: the kernels of the sharded stage (and the reused ones) run
thread by thread for W simulated ranks (tests/hostemu/stitch_sharded_emu.cpp), a rank's peer pointers being the other ranks'
host arrays.  For every split of the contigs and of the reads over the ranks, the union of the ranks' records must be the
oracle's stitched set, and the per-rank statistics must add up to (or, for the global ones, equal) the oracle's."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle import orc
from test_stitch import _as_fastq_case, assembled, gap_scenario, hand_cases, random_scenarios, triples

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _EmuOut(C.Structure):
    _fields_ = [("n", C.c_uint64), ("off", C.POINTER(C.c_uint64)), ("bases", C.POINTER(C.c_char)), ("left", C.POINTER(C.c_int32)),
                ("right", C.POINTER(C.c_int32)), ("stats", C.c_uint64 * 6)]


_E = None


def _emu():
    """Compiles the harness into a temporary directory (the source tree is never written) and loads it once per process."""
    global _E
    if _E is None:
        src = os.path.join(ROOT, "tests", "hostemu", "stitch_sharded_emu.cpp")
        out = os.path.join(tempfile.mkdtemp(prefix="stitch_sharded_emu_"), "libstitchshardedemu.so")
        cxx = "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else "g++"
        subprocess.run([cxx, "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas", "-x", "c++", "-o", out, src], check=True)
        E = C.CDLL(out)
        E.emu_stitch_sharded.restype = C.c_int
        E.emu_stitch_sharded.argtypes = [C.c_int] + [C.c_void_p] * 9 + [C.c_int, C.c_int, C.c_uint64, C.c_void_p]
        E.emu_stitch_sharded_free.argtypes = [C.c_void_p, C.c_int]
        _E = E
    return _E


def emu_stitch_sharded(ctg_parts, read_parts, contigs, left, right, txt, k, min_contig, cap0=4):
    """ctg_parts[r]: indices of the contigs rank r holds; read_parts[r]: indices of the reads of `txt` pushed to rank r.
    Returns the records and the six statistics of every rank."""
    E = _emu()
    world = len(ctg_parts)
    a = np.frombuffer(txt, dtype=np.uint8)
    starts, lens = orc.fastq_reads(a, orc.FASTQ_RUN)
    keep = []

    def arr(x, dt):
        x = np.ascontiguousarray(x, dtype=dt)
        keep.append(x)
        return x.ctypes.data

    ns, offs, blobs, ls, rs, nr, ss, ll = [], [], [], [], [], [], [], []
    for r in range(world):
        cs = [contigs[i] for i in ctg_parts[r]]
        o = np.zeros(len(cs) + 1, dtype=np.uint64)
        if cs:
            o[1:] = np.cumsum([len(c) for c in cs])
        ns.append(len(cs))
        offs.append(arr(o, np.uint64))
        blobs.append(arr(np.frombuffer("".join(cs).encode() + b"\0", dtype=np.uint8), np.uint8))
        ls.append(arr([left[i] for i in ctg_parts[r]] + [0], np.int32))
        rs.append(arr([right[i] for i in ctg_parts[r]] + [0], np.int32))
        idx = np.asarray(read_parts[r], dtype=np.int64)
        nr.append(len(idx))
        ss.append(arr(np.append(starts[idx], 0), np.uint64))
        ll.append(arr(np.append(lens[idx], 0), np.uint32))
    P = C.c_void_p * world
    outs = (_EmuOut * world)()
    rc = E.emu_stitch_sharded(world, arr(ns, np.uint64), P(*offs), P(*blobs), P(*ls), P(*rs), a.ctypes.data, arr(nr, np.uint64), P(*ss), P(*ll), k, min_contig, cap0,
                              C.cast(outs, C.c_void_p))
    assert rc == 0, rc
    res = []
    for o in outs:
        n = o.n
        of = np.ctypeslib.as_array(o.off, shape=(n + 1,)).copy()
        b = C.string_at(o.bases, int(of[-1])) if n else b""
        res.append(dict(contigs=[b[int(of[i]):int(of[i + 1])].decode() for i in range(n)], left=[o.left[i] for i in range(n)],
                        right=[o.right[i] for i in range(n)], stats=list(o.stats)))
    E.emu_stitch_sharded_free(C.cast(outs, C.c_void_p), world)
    return res


def union(res):
    return sorted(t for r in res for t in zip(r["contigs"], r["left"], r["right"]))


def check(res, want):
    """Union == the oracle; n_fragments, n_stitched, n_rings add up; n_probes, n_after_pass1, n_joined are global."""
    assert union(res) == triples(want)
    st = list(want["stats"].values())  # probes, fragments, after pass 1, joined, stitched records, rings
    for r in res:
        assert r["stats"][0] == st[0] and r["stats"][2] == st[2] and r["stats"][3] == st[3]
    assert [sum(r["stats"][i] for r in res) for i in (1, 4, 5)] == [st[1], st[4], st[5]]


def splits(n, world, rng):
    """Ways to put n items on `world` ranks: contiguous, round robin, random, all on the last rank, and (world > 1) one rank
    left empty."""
    out = [[list(range(n * r // world, n * (r + 1) // world)) for r in range(world)],
           [list(range(r, n, world)) for r in range(world)]]
    owner = rng.integers(0, world, n)
    out.append([np.flatnonzero(owner == r).tolist() for r in range(world)])
    out.append([[] for _ in range(world - 1)] + [list(range(n))])
    if world > 1:
        owner = rng.integers(1, world, n)
        out.append([np.flatnonzero(owner == r).tolist() for r in range(world)])
    return out


def _cases():
    cases = [(k, *assembled(txt, k), txt) for k, txt in random_scenarios(8)]
    cases += [_as_fastq_case(c) for c in hand_cases().values()]
    txt = gap_scenario(5, 6000, 100, [(2000, 2060), (4000, 4070)])[1]
    cases.append((31, *assembled(txt, 31), txt))
    return cases


def test_sharded_stitch_kernels_on_the_host_match_the_oracle():
    rng = np.random.default_rng(11)
    stitched = rings = cross = 0
    for ci, (k, contigs, left, right, txt) in enumerate(_cases()):
        n_reads = len(orc.fastq_reads(np.frombuffer(txt, dtype=np.uint8), orc.FASTQ_RUN)[0])
        for min_contig in (0, 200):
            want = orc.stitch(contigs, left, right, txt, k, min_contig=min_contig)
            for world in (1, 2, 3, 5):
                cs, rs = splits(len(contigs), world, rng), splits(n_reads, world, rng)
                for j, ctg_parts in enumerate(cs):
                    read_parts = rs[(j + ci) % len(rs)]
                    res = emu_stitch_sharded(ctg_parts, read_parts, contigs, left, right, txt, k, min_contig, cap0=1 + j)
                    check(res, want)
                    if world > 1 and min_contig == 0:
                        # a record whose pieces were held by two ranks
                        owner = {contigs[i]: r for r, p in enumerate(ctg_parts) for i in p}
                        for r in res:
                            for s in r["contigs"]:
                                holders = {o for c, o in owner.items() if len(c) >= k and c in s and c != s}
                                cross += len(holders) > 1
        stitched += want["stats"]["stitched_records"]
        rings += want["stats"]["rings"]
    assert stitched > 10 and rings > 0 and cross > 10


def test_sharded_stitch_on_the_host_rank_extremes():
    """All contigs on one rank and all reads on another; a rank with no contigs and no reads; one rank holding every read."""
    k, txt = 31, gap_scenario(6, 6000, 100, [(2000, 2060), (4000, 4070)], err=0.02)[1]
    contigs, left, right = assembled(txt, k)
    n, m = len(contigs), len(orc.fastq_reads(np.frombuffer(txt, dtype=np.uint8), orc.FASTQ_RUN)[0])
    want = orc.stitch(contigs, left, right, txt, k, min_contig=500)
    assert want["stats"]["stitched_records"] > 0
    every, none = list(range(n)), []
    layouts = [
        ([every, none], [none, list(range(m))]),                                  # contigs on rank 0, reads on rank 1
        ([none, every, none], [list(range(0, m, 2)), none, list(range(1, m, 2))]),  # all contigs on rank 1, rank 1 reads nothing
        ([[i for i in every if i % 2 == 0], [], [i for i in every if i % 2]], [list(range(m)), [], []]),  # rank 1 holds nothing at all
    ]
    for ctg_parts, read_parts in layouts:
        res = emu_stitch_sharded(ctg_parts, read_parts, contigs, left, right, txt, k, 500)
        check(res, want)
        assert all(not r["contigs"] for r, p in zip(res, ctg_parts) if not p)  # a rank without contigs heads no record
