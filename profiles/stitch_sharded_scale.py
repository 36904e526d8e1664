"""-stitch across ranks (rfx_stitch_begin_sharded / rfx_stitch_finish_sharded) at the read count of configs[1]: the workload of
stitch_scale.py (46 Mbp genome at 10x, 3.07 M x 150 bp reads, k = 31, cover 3, -mincontig 500) on N = 1 / 2 / 4 / 8 ranks, against
rfx_stitch_begin / rfx_stitch_finish on one context.

The table is counted once on one context and kept in device memory; every rank loads a contiguous slice with
rfx_load_counts_device and re-shards it with rfx_shard_table.  The FASTQ is cut into N slices on record boundaries, each slice
device-resident on its rank's GPU, pushed with rfx_push_fastq_device between begin and finish.  Per stage, rank 0 and the
maximum over the ranks: begin (sharded assembly + summary pull + probe table: host clock, ms_stitch after begin), the read scan
(ms_parse delta), finish (ms_stitch delta), ms_comm of the begin and of the finish.  Median of 3 repetitions after one
warm-up.  With fewer devices than ranks, ranks share devices (the JSON says how many there were): such rows measure the
protocol's cost, not a multi-GPU speed-up.
usage: python profiles/stitch_sharded_scale.py > profiles/stitch_sharded_scale.json"""
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ.setdefault("CUDA_MODULE_LOADING", "EAGER")
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
import numpy as np
import torch

import reflexiv_b200 as R
from reflexiv_b200 import sharded
from workload import synth

REPS = 3
K, COVER, MINC = 31, 3, 500


def slices_on_record_boundaries(txt, world):
    """Byte ranges of `world` slices of a 4-line FASTQ, cut just before a record's '@' line."""
    nl = np.flatnonzero(txt == ord("\n"))
    rec_starts = np.concatenate([[0], nl[3::4] + 1])[:-1] if len(nl) >= 4 else np.array([0])
    n_rec = len(rec_starts)
    cuts = [int(rec_starts[n_rec * r // world]) if r < world else len(txt) for r in range(world + 1)]
    cuts[0], cuts[world] = 0, len(txt)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def single(txt_dev, n_bytes):
    reps, out = [], None
    with R.ReflexivContext(R.DefaultParam(kmerSize=K, minKmerCoverage=COVER, minContig=MINC), device=0) as ctx:
        for it in range(REPS + 1):
            ctx.reset()
            ctx.push_fastq_device(txt_dev.data_ptr(), n_bytes)
            ctx.count()
            pk, pc, n, kb = ctx.counts_device()
            if it == 0:
                keys = sharded.device_view(torch, pk, n * kb, torch.device("cuda", 0)).clone()
                cnt = sharded.device_view(torch, pc, n * 4, torch.device("cuda", 0)).clone()
            p0 = ctx.stats()["ms_parse"]
            t0 = time.perf_counter()
            b = ctx.stitch_begin()
            t1 = time.perf_counter()
            ctx.push_fastq_device(txt_dev.data_ptr(), n_bytes)
            p1 = ctx.stats()["ms_parse"]
            f = ctx.stitch_finish()
            t2 = time.perf_counter()
            if it:
                reps.append({"ms_begin_host": (t1 - t0) * 1e3, "ms_begin_probe_table": b["ms_stitch"], "ms_scan": p1 - p0,
                             "ms_finish": f["ms_stitch"] - b["ms_stitch"], "ms_total_host": (t2 - t0) * 1e3})
            out = sorted(ctx.contigs())
            stats = f
    torch.cuda.synchronize()
    med = {key: statistics.median(r[key] for r in reps) for key in reps[0]}
    return med, out, stats, keys, cnt, n, kb


def ranks(keys, cnt, n, kb, txt, world, n_dev):
    per_dev = -(-world // n_dev)
    free = torch.cuda.mem_get_info(0)[0]
    arena = int(free * 0.6 / per_dev) & ~((1 << 20) - 1)
    ctxs = [R.ReflexivContext(R.DefaultParam(kmerSize=K, minKmerCoverage=COVER, minContig=MINC), device=r % n_dev) for r in range(world)]
    rows = [(n * r // world, n * (r + 1) // world) for r in range(world)]
    parts = slices_on_record_boundaries(txt, world)
    d_parts = []
    for r, (a, b) in enumerate(parts):  # each rank's slice of the text, resident on its own GPU
        d = torch.zeros(b - a + 128, dtype=torch.uint8, device=f"cuda:{r % n_dev}")
        d[:b - a] = torch.from_numpy(txt[a:b]).to(d.device)
        d_parts.append((d, b - a))
    torch.cuda.synchronize()
    reps, got, last = [], None, None
    try:
        grp = sharded.LocalRanks(ctxs, arena_bytes=arena)

        def body(r, ctx):
            lo, hi = rows[r]
            ctx.reset()
            ctx.load_counts_device(keys.data_ptr() + lo * kb, cnt.data_ptr() + lo * 4, hi - lo)
            ctx.shard_table()
            p0 = ctx.stats()["ms_parse"]
            t0 = time.perf_counter()
            b = ctx.stitch_begin_sharded()
            t1 = time.perf_counter()
            comm_b = ctx.shard_stats()["ms_comm"]
            d, nb = d_parts[r]
            ctx.push_fastq_device(d.data_ptr(), nb)
            p1 = ctx.stats()["ms_parse"]
            t2 = time.perf_counter()
            f = ctx.stitch_finish_sharded()
            t3 = time.perf_counter()
            sh = ctx.shard_stats()
            return dict(ms_begin_host=(t1 - t0) * 1e3, ms_begin_probe_table=b["ms_stitch"], ms_scan=p1 - p0, ms_scan_host=(t2 - t1) * 1e3,
                        ms_finish=f["ms_stitch"] - b["ms_stitch"], ms_finish_host=(t3 - t2) * 1e3, ms_comm_begin=comm_b, ms_comm_finish=sh["ms_comm"],
                        stats=f, contigs=ctx.contigs(), n_contigs_global=sh["n_contigs_global"], arena_used=sh["arena_used"])
        for it in range(REPS + 1):
            out = grp.run(body)
            if it:
                reps.append(out)
            got, last = sorted(x for o in out for x in o["contigs"]), out
    finally:
        for c in ctxs:
            c.close()
    keys_t = ["ms_begin_host", "ms_begin_probe_table", "ms_scan", "ms_scan_host", "ms_finish", "ms_finish_host", "ms_comm_begin", "ms_comm_finish"]
    res = {"world": world, "devices_used": min(world, n_dev), "ranks_share_a_device": world > n_dev, "arena_bytes_per_rank": arena}
    for key in keys_t:
        res[key] = {"rank0": statistics.median(rep[0][key] for rep in reps), "max_over_ranks": statistics.median(max(x[key] for x in rep) for rep in reps)}
    st = [o["stats"] for o in last]
    res["stats_per_rank"] = [{k: v for k, v in s.items() if k != "ms_stitch"} for s in st]
    res["n_contigs_global"] = last[0]["n_contigs_global"]
    res["arena_used_per_rank"] = [o["arena_used"] for o in last]
    return res, got


def main():
    n_dev = torch.cuda.device_count()
    if n_dev < 1:
        raise SystemExit("no CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    glen = int(sys.argv[1]) if len(sys.argv) > 1 else 46_000_000
    cov = float(sys.argv[2]) if len(sys.argv) > 2 else 10.0
    g = synth.genome(glen, seed=7)
    txt = np.asarray(synth.fastq(g, synth.n_pairs_for(glen, cov, 150), read_len=150, frag_len=400))
    n_bytes = txt.size
    d_text = torch.zeros(n_bytes + 128, dtype=torch.uint8, device="cuda:0")
    d_text[:n_bytes] = torch.from_numpy(txt).cuda()
    torch.cuda.synchronize()
    one, one_contigs, one_stats, keys, cnt, n, kb = single(d_text, n_bytes)
    del d_text
    torch.cuda.empty_cache()
    out = {"what": __doc__.split("\n")[0], "workload": f"{glen} bp genome, {cov:g}x, 150 bp paired reads, k={K}, cover {COVER}, -mincontig {MINC}",
           "devices": smi, "n_devices": n_dev, "fastq_bytes": int(n_bytes), "table_rows": int(n), "repetitions": REPS,
           "one_context": {**one, "stats": {k: v for k, v in one_stats.items() if k != "ms_stitch"}, "n_contigs": len(one_contigs)}, "sharded": []}
    for world in (1, 2, 4, 8):
        s, got = ranks(keys, cnt, n, kb, txt, world, n_dev)
        s["equal_to_one_context"] = got == one_contigs
        s["stats_sum_equal_to_one_context"] = all(sum(p[f] for p in s["stats_per_rank"]) == one_stats[f] for f in ("n_fragments", "n_stitched", "n_rings")) and \
            all(p[f] == one_stats[f] for p in s["stats_per_rank"] for f in ("n_probes", "n_after_pass1", "n_joined"))
        out["sharded"].append(s)
        print(json.dumps({k: v for k, v in s.items() if k not in ("stats_per_rank", "arena_used_per_rank")}), file=sys.stderr, flush=True)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
