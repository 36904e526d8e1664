"""`reflexiv sort --gpus N` at scale: a Count_31 table re-sharded with rfx_shard_table and run through rfx_sort_kmers_sharded
on N = 1 / 2 / 4 / 8 ranks, against rfx_sort_kmers of the same table on one context.

Tables: configs[1] (4.6 Mbp genome, 100x, k = 31, cover 2: ~4.6 M rows) and a 10x larger one (46 Mbp, 20x), the tables of
kmerc_sharded_scale.py.  Each table is counted once on the GPU from synthetic reads, kept in device memory, and every rank
loads its contiguous slice with rfx_load_counts_device (the host CSV parse of the binary is not part of these numbers).
Times are device events around each library call (rfx_stats: ms_partition for rfx_shard_table, ms_graph for the sort call),
rank 0's view, median of 3 repetitions after one warm-up; host clocks around the same calls are recorded beside them.
With fewer devices than ranks, ranks share devices (the JSON says how many devices there were): such rows measure the
protocol's cost, not a multi-GPU speed-up.
usage: python profiles/sorted_sharded_scale.py > profiles/sorted_sharded_scale.json"""
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ.setdefault("CUDA_MODULE_LOADING", "EAGER")
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
import torch

import reflexiv_b200 as R
from reflexiv_b200 import sharded
from workload import synth

REPS = 3
K, E, FOLD, KMAX = 31, 8, 1.5, 95


def table_on_device(glen, cov):
    g = synth.genome(glen, seed=11)
    txt = synth.fastq(g, synth.n_pairs_for(glen, cov, 150), read_len=150, frag_len=400)
    with R.ReflexivContext(R.DefaultParam(kmerSize=K, minKmerCoverage=2), device=0) as ctx:
        ctx.push_fastq(txt)
        ctx.count()
        pk, pc, n, kb = ctx.counts_device()
        keys = sharded.device_view(torch, pk, n * kb, torch.device("cuda", 0)).clone()
        cnt = sharded.device_view(torch, pc, n * 4, torch.device("cuda", 0)).clone()
    torch.cuda.synchronize()
    return keys, cnt, n, kb


def single(keys, cnt, n):
    ev, host, rows = [], [], 0
    with R.ReflexivContext(R.DefaultParam(kmerSize=K), device=0) as ctx:
        for it in range(REPS + 1):
            ctx.reset()
            ctx.load_counts_device(keys.data_ptr(), cnt.data_ptr(), n)
            t0 = time.perf_counter()
            rows = ctx.sort_kmers(E, FOLD, KMAX)
            t1 = time.perf_counter()
            if it:
                ev.append(ctx.stats()["ms_graph"])
                host.append((t1 - t0) * 1e3)
    return {"ms_sort": statistics.median(ev), "ms_sort_all": ev, "ms_sort_host": statistics.median(host), "n_sorted": rows}


def ranks(keys, cnt, n, kb, world, n_dev):
    per_dev = -(-world // n_dev)
    free = torch.cuda.mem_get_info(0)[0]
    arena = int(free * 0.8 / per_dev) & ~((1 << 20) - 1)
    ctxs = [R.ReflexivContext(R.DefaultParam(kmerSize=K), device=r % n_dev) for r in range(world)]
    rows = [(n * r // world, n * (r + 1) // world) for r in range(world)]
    reps = []
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=arena)

        def body(r, ctx):
            lo, hi = rows[r]
            ctx.reset()
            ctx.load_counts_device(keys.data_ptr() + lo * kb, cnt.data_ptr() + lo * 4, hi - lo)
            t0 = time.perf_counter()
            a = ctx.shard_table()
            t1 = time.perf_counter()
            m = ctx.sort_kmers_sharded(E, FOLD, KMAX)
            t2 = time.perf_counter()
            st, sh = ctx.stats(), ctx.shard_stats()
            return dict(ms_shard_table=a["ms_partition"], ms_sort_sharded=st["ms_graph"], ms_shard_table_host=(t1 - t0) * 1e3,
                        ms_sort_sharded_host=(t2 - t1) * 1e3, ms_comm_sort=sh["ms_comm"], rows=a["n_rows"], n_sorted=m,
                        n_sorted_global=sh["n_oriented_global"], n_remote_probes=sh["n_remote_probes"])
        for it in range(REPS + 1):
            out = grp.run(body)
            if it:
                reps.append(out)
    finally:
        for c in ctxs:
            c.close()
    med = lambda key: statistics.median(rep[0][key] for rep in reps)  # noqa: E731
    last = reps[-1]
    return {"world": world, "devices_used": min(world, n_dev), "ranks_share_a_device": world > n_dev, "arena_bytes_per_rank": arena,
            "ms_shard_table": med("ms_shard_table"), "ms_sort_sharded": med("ms_sort_sharded"),
            "ms_total": med("ms_shard_table") + med("ms_sort_sharded"), "ms_sort_sharded_host": med("ms_sort_sharded_host"),
            "ms_shard_table_host": med("ms_shard_table_host"), "ms_comm_in_sort": med("ms_comm_sort"),
            "rows_per_rank": [x["rows"] for x in last], "n_sorted_global": last[0]["n_sorted_global"],
            "n_sorted_sum": sum(x["n_sorted"] for x in last), "n_remote_probes_per_rank": [x["n_remote_probes"] for x in last]}


def main():
    n_dev = torch.cuda.device_count()
    if n_dev < 1:
        raise SystemExit("no CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    out = {"what": __doc__.split("\n")[0], "devices": smi, "n_devices": n_dev, "k": K, "E": E, "fold": FOLD, "max_kmer_size": KMAX, "tables": []}
    for name, glen, cov in (("configs[1]: 4.6 Mbp, 100x, cover 2", 4_600_000, 100.0), ("10x: 46 Mbp, 20x, cover 2", 46_000_000, 20.0)):
        keys, cnt, n, kb = table_on_device(glen, cov)
        one = single(keys, cnt, n)
        entry = {"table": name, "rows": n, "table_bytes": n * (kb + 4), "one_gpu_rfx_sort_kmers": one, "sharded": []}
        for world in (1, 2, 4, 8):
            s = ranks(keys, cnt, n, kb, world, n_dev)
            s["same_row_count_as_one_gpu"] = s["n_sorted_sum"] == one["n_sorted"] == s["n_sorted_global"]
            s["speedup_vs_one_gpu"] = one["ms_sort"] / s["ms_total"]
            entry["sharded"].append(s)
            print(json.dumps({"table": name, **{k: v for k, v in s.items() if k not in ("rows_per_rank", "n_remote_probes_per_rank")}}), file=sys.stderr, flush=True)
        out["tables"].append(entry)
        del keys, cnt
        torch.cuda.empty_cache()
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
