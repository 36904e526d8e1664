"""bench.py --dump-outputs: the arrays are in an order of their own, hold every value exactly and stay under the size cap."""
import os

import numpy as np

import bench


class _Ctx:
    """Stands in for a ReflexivContext after a step: the result in a given row order."""

    def __init__(self, keys, cnts, contigs, order):
        self.keys, self.cnts = keys[order], cnts[order]
        seqs = [contigs[i] for i in order]
        self.bases = np.frombuffer("".join(s for s, _, _ in seqs).encode(), dtype=np.uint8)
        self.offs = np.concatenate(([0], np.cumsum([len(s) for s, _, _ in seqs]))).astype(np.uint64)
        self.left = np.array([l for _, l, _ in seqs], dtype=np.int32)
        self.right = np.array([r for _, _, r in seqs], dtype=np.int32)

    def counts(self):
        return self.keys, self.cnts

    def contigs_raw(self):
        return self.bases, self.offs, self.left, self.right


def test_result_arrays_are_exact_and_independent_of_row_order():
    rng = np.random.default_rng(5)
    keys = rng.integers(0, 2**64, size=(6, 2), dtype=np.uint64)
    keys[0, 0] = 2**64 - 1  # beyond any float mantissa
    cnts = rng.integers(1, 2**32, size=6, dtype=np.uint32)
    contigs = [("ACGTTG", -4, -4), ("CAACGT", -4, -4), ("AC", 1, 2), ("AC", 1, -1), ("GGGAT", 0, 7), ("ATCCC", 7, 0)]
    ctxs = [_Ctx(keys, cnts, contigs, np.arange(6)), _Ctx(keys, cnts, contigs, np.array([3, 5, 0, 4, 1, 2]))]
    for mode in ("counter", "run"):
        a, b = (bench.result_arrays(c, mode) for c in ctxs)
        assert a.keys() == b.keys()
        for name in a:
            assert a[name].dtype in (np.float32, np.float64)
            assert np.array_equal(a[name], b[name]), (mode, name)
    got = bench.result_arrays(ctxs[1], "counter")
    back = got["count_keys"].astype(np.uint32).view(np.uint64)
    order = np.lexsort(keys.T)
    assert np.array_equal(back, keys[order]) and np.array_equal(got["count_values"].astype(np.uint32), cnts[order])
    got = bench.result_arrays(ctxs[1], "run")
    text = got["contig_bases"].astype(np.uint8).tobytes().decode()
    ends = np.cumsum(got["contig_lengths"].astype(int))
    seqs = [text[e - n:e] for e, n in zip(ends, got["contig_lengths"].astype(int))]
    assert list(zip(seqs, got["contig_left"].astype(int), got["contig_right"].astype(int))) == sorted(contigs)


def test_dump_outputs_stays_under_the_cap_with_a_repeatable_sample(tmp_path):
    rng = np.random.default_rng(6)
    arrays = {"big": rng.random(1 << 20).astype(np.float32), "rows": rng.random((1 << 17, 4)), "small": np.arange(10.0)}
    limit = 1 << 20
    for d in ("a", "b"):
        bench.dump_outputs(arrays, str(tmp_path / d), limit)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["big.npy", "rows.npy", "small.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= limit
    a = {f: np.load(tmp_path / "a" / f) for f in files}
    assert np.array_equal(a["small.npy"], arrays["small"])
    assert a["rows.npy"].shape[1] == 4 and 0 < len(a["rows.npy"]) < len(arrays["rows"])
    assert np.isin(a["big.npy"], arrays["big"]).all()
    for f in files:
        assert np.array_equal(a[f], np.load(tmp_path / "b" / f))
