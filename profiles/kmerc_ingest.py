"""Count_<k> ingest on the B200: the host parser (`reflexiv`'s parse_counts, all threads) + rfx_load_counts against rfx_load_counts_csv,
the kernels alone, and the wall clock of `reflexiv run -kmerc` at --gpus 1 and 8 for the parent build and this one.

Inputs are synthetic Count_<k> tables generated from a seed: uniform random k-mers (distinct: checked up to 2e7 rows), counts skewed (1 + Zipf(1.6), at most
9 digits), rows `KMER,count\\n`.  Sizes: k = 31 at 4.6e6 rows (a configs[1]-size table), k = 31 at 1.5e8 rows, k = 61 at 5.5e6 rows
(the scaled configs[3] table).  Every time is the median of --reps calls after a warm-up call on the first MB of the table; the kernel
time is summed from one call under torch.profiler (CUDA activities) in the same process.

    python profiles/kmerc_ingest.py [--out profiles/kmerc_ingest.json] [--parent DIR_WITH_PARENT_reflexiv] [--scale 0.01]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HBM_GBS = 6498.7  # measured HBM copy bandwidth the project quotes its kernels against (DESIGN.md section 4)
TABLES = [("k31_4.6e6", 31, 4_600_000, 1), ("k31_1.5e8", 31, 150_000_000, 2), ("k61_5.5e6", 61, 5_500_000, 3)]
BOUNDS = (2, 10_000_000)  # `run -kmerc` defaults: cover..maxcov

HARNESS = r'''
#define main reflexiv_real_main
#include "%s"
#undef main
#include <chrono>
static double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }
int main(int argc, char** argv) {  // <file> <k> <minc> <maxc> <reps>: one JSON line per rep
    std::string text;
    FILE* f = fopen(argv[1], "rb");
    std::vector<char> buf(1 << 24); size_t got;
    while ((got = fread(buf.data(), 1, buf.size(), f)) > 0) text.append(buf.data(), got);
    fclose(f);
    const int k = atoi(argv[2]), minc = atoi(argv[3]), maxc = atoi(argv[4]), reps = atoi(argv[5]);
    rfx_params p; rfx_params_default(&p); p.kmer_size = k;
    rfx_ctx* c = nullptr;
    if (rfx_create(&c, &p) != RFX_OK) { fprintf(stderr, "rfx_create: %%s\n", rfx_last_error(nullptr)); return 1; }
    const size_t warm = text.find('\n', std::min<size_t>(text.size() - 1, 1 << 20)) + 1;
    {
        std::vector<uint64_t> keys; std::vector<uint32_t> counts;
        parse_counts(text.data(), warm, k, minc, maxc, keys, counts);
        rfx_load_counts(c, keys.data(), counts.data(), counts.size());
        rfx_load_counts_csv(c, (const uint8_t*)text.data(), warm, minc, maxc, 0);
    }
    const size_t words = k <= 31 ? 1 : k / 32 + 1;
    for (int r = 0; r < reps; r++) {
        std::vector<uint64_t> keys; std::vector<uint32_t> counts;
        const double t0 = now_ms();
        if (!parse_counts(text.data(), text.size(), k, minc, maxc, keys, counts)) { fprintf(stderr, "malformed\n"); return 1; }
        const double t1 = now_ms();
        if (rfx_load_counts(c, keys.data(), counts.data(), counts.size()) != RFX_OK) { fprintf(stderr, "%%s\n", rfx_last_error(c)); return 1; }
        const double t2 = now_ms();
        int same = -1;
        if (r == 0) {  // the two tables, row for row
            std::vector<uint64_t> k1(counts.size() * words); std::vector<uint32_t> c1(counts.size());
            rfx_counts_copy(c, k1.data(), c1.data());
            if (rfx_load_counts_csv(c, (const uint8_t*)text.data(), text.size(), minc, maxc, 0) != RFX_OK) { fprintf(stderr, "%%s\n", rfx_last_error(c)); return 1; }
            uint64_t n = 0; rfx_counts_size(c, &n, nullptr);
            std::vector<uint64_t> k2(n * words); std::vector<uint32_t> c2(n);
            rfx_counts_copy(c, k2.data(), c2.data());
            same = n == counts.size() && k1 == k2 && c1 == c2 && c1 == counts;
        }
        const double t3 = now_ms();
        if (rfx_load_counts_csv(c, (const uint8_t*)text.data(), text.size(), minc, maxc, 0) != RFX_OK) { fprintf(stderr, "%%s\n", rfx_last_error(c)); return 1; }
        const double t4 = now_ms();
        rfx_stats_t s; rfx_stats(c, &s);
        printf("{\"host_parse_ms\": %%.3f, \"load_counts_ms\": %%.3f, \"csv_pageable_ms\": %%.3f, \"rows\": %%zu, \"same_table\": %%d, \"threads\": %%u}\n",
               t1 - t0, t2 - t1, t4 - t3, counts.size(), same, std::thread::hardware_concurrency());
        fflush(stdout);
    }
    rfx_destroy(c);
    return 0;
}
'''


def write_table(path, seed, k, n, block=10_000_000):
    """Count_<k> text of n random k-mers with skewed counts; returns (bytes, distinct k-mers)."""
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    lut = acgt[(np.arange(256)[:, None] >> np.array([6, 4, 2, 0])[None, :]) & 3].astype(np.uint8)  # byte -> its 4 bases
    words = (k + 31) // 32
    seen = []
    with open(path, "wb") as f:
        for s in range(0, n, block):
            m = min(block, n - s)
            w = rng.integers(0, 2**63, size=(m, words), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=(m, words), dtype=np.uint64)
            bases = lut[w.astype(">u8").view(np.uint8)].reshape(m, 32 * words)[:, 32 * words - k:]  # the last k of 32 * words random bases
            if k <= 32:
                seen.append(w[:, 0] & np.uint64((1 << (2 * k)) - 1))
            else:
                seen.append(np.stack([w[:, 0] & np.uint64((1 << (2 * (k - 32))) - 1), w[:, 1]], 1))
            cnt = np.minimum(1 + rng.zipf(1.6, m), 999_999_999).astype(np.int64)
            nd = np.ones(m, np.int64)
            for d in range(1, 9):
                nd += cnt >= 10 ** d
            width = k + 1 + 9 + 1  # bases, ',', the count right-aligned in 9 columns, '\n'; leading columns masked out
            mat = np.empty((m, width), np.uint8)
            mat[:, :k] = bases
            mat[:, k] = ord(",")
            rest = cnt.copy()
            for j in range(9):
                mat[:, k + 9 - j] = 48 + rest % 10
                rest //= 10
            mat[:, k + 10] = 10
            mask = np.ones((m, width), bool)
            mask[:, k + 1:k + 10] = np.arange(9)[None, :] >= (9 - nd)[:, None]
            f.write(mat[mask].tobytes())
    if n > 20_000_000:  # sorting 1.5e8 keys costs minutes of host time: the expected number of equal pairs instead
        return os.path.getsize(path), f"not checked: {n * (n - 1) / 2 / 4.0 ** k:.2g} equal pairs expected among uniform random {k}-mers"
    keys = np.concatenate(seen)
    return os.path.getsize(path), int(len(np.unique(keys)) if k <= 32 else len(np.unique(keys, axis=0)))


def median(xs):
    return float(np.median(xs)) if xs else None


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()


def pinned_and_kernels(path, k, reps, trace_dir):
    """rfx_load_counts_csv from pinned host memory (wall clock), and the kernels of one call (torch.profiler)."""
    import torch
    import reflexiv_b200 as R
    data = np.fromfile(path, np.uint8)
    pinned = torch.empty(data.size, dtype=torch.uint8, pin_memory=True)
    arr = pinned.numpy()
    arr[:] = data
    del data
    out = {}
    with R.ReflexivContext(R.DefaultParam(kmerSize=k), device=0) as ctx:
        start = min(1 << 20, arr.size - 1)  # the warm-up call: the lines up to the first newline behind 1 MB (the whole of a smaller table)
        warm = int(np.flatnonzero(arr[start:] == 10)[0]) + start + 1
        ctx.load_counts_csv(arr[:warm], *BOUNDS)
        ts, gpu = [], []
        for _ in range(reps):
            before = ctx.stats()["ms_parse"]
            t0 = time.perf_counter()
            ctx.load_counts_csv(arr, *BOUNDS)
            ts.append((time.perf_counter() - t0) * 1e3)
            gpu.append(ctx.stats()["ms_parse"] - before)
        out["csv_pinned_ms"] = median(ts)
        out["csv_pinned_call_gpu_ms"] = median(gpu)
        out["rows"] = int(ctx.stats()["n_rows"])
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            ctx.load_counts_csv(arr, *BOUNDS)
            torch.cuda.synchronize()
        trace = os.path.join(trace_dir, "trace.json")
        prof.export_chrome_trace(trace)
        ev = json.load(open(trace))
        ev = ev["traceEvents"] if isinstance(ev, dict) else ev
        kern = [e for e in ev if e.get("cat") == "kernel"]
        copies = [e for e in ev if e.get("cat") == "gpu_memcpy"]
        by = {}
        for e in kern:
            name = e["name"].split("<")[0].split("(")[0].replace("void ", "")
            by[name] = by.get(name, 0.0) + e["dur"] / 1e3
        out["kernel_ms"] = sum(e["dur"] for e in kern) / 1e3
        out["kernels_ms_by_name"] = {n: round(v, 3) for n, v in sorted(by.items(), key=lambda x: -x[1])}
        out["kernel_launches"] = len(kern)
        out["h2d_copy_ms"] = sum(e["dur"] for e in copies if "HtoD" in e["name"]) / 1e3
    return out


def wall_clock(exe, table, gpus, k, tmp, tag):
    out = os.path.join(tmp, f"o_{tag}_{gpus}_{time.monotonic_ns()}")
    env = dict(os.environ, CUDA_MODULE_LOADING="EAGER", CUDA_DEVICE_MAX_CONNECTIONS="32")
    import torch
    n_dev = torch.cuda.device_count()
    if gpus > n_dev:
        env["REFLEXIV_ARENA_MB"] = str(min(16000, 150_000 // gpus))
    t0 = time.perf_counter()
    r = subprocess.run([exe, "run", "--gpus", str(gpus), "-kmerc", table, "-outfile", out, "-kmer", str(k)], capture_output=True, text=True, env=env)
    t = time.perf_counter() - t0
    shutil.rmtree(out, ignore_errors=True)
    if r.returncode != 0:
        raise RuntimeError(f"{exe} --gpus {gpus}: {r.stderr[-400:]}")
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "kmerc_ingest.json"))
    ap.add_argument("--parent", default=None, help="directory holding the parent commit's reflexiv + libreflexiv_cuda.so")
    ap.add_argument("--scale", type=float, default=1.0, help="row counts times this (rehearsal)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--tables", default=",".join(t[0] for t in TABLES), help="comma-separated subset of " + ", ".join(t[0] for t in TABLES))
    ap.add_argument("--budget-s", type=float, default=900, help="wall clock runs are skipped once the script has run this long")
    a = ap.parse_args()
    t_start = time.monotonic()
    res = {"gpu": gpu_info(), "hbm_gbs_reference": HBM_GBS, "bounds": list(BOUNDS), "reps": a.reps, "tables": {}}
    tmp = tempfile.mkdtemp(prefix="kmerc_ingest_")
    try:
        harness_src = os.path.join(tmp, "h.cpp")
        open(harness_src, "w").write(HARNESS % os.path.join(ROOT, "reflexiv_b200", "csrc", "reflexiv_main.cpp"))
        lib = os.path.join(ROOT, "reflexiv_b200")
        harness = os.path.join(tmp, "h")
        subprocess.run(["g++", "-O2", "-std=c++17", "-o", harness, harness_src, "-L" + lib, "-lreflexiv_cuda", "-lz", "-pthread", "-Wl,-rpath," + lib], check=True)
        exes = {"this": os.path.join(ROOT, "reflexiv_b200", "reflexiv")}
        if a.parent:
            exes["parent"] = os.path.join(a.parent, "reflexiv")
        for name, k, n, seed in TABLES:
            if name not in a.tables.split(","):
                continue
            n = max(1000, int(n * a.scale))
            path = os.path.join(tmp, f"{name}.csv")
            t0 = time.perf_counter()
            nbytes, distinct = write_table(path, seed, k, n)
            entry = {"k": k, "rows": n, "distinct": distinct, "text_bytes": nbytes, "generate_s": round(time.perf_counter() - t0, 1)}
            res["tables"][name] = entry
            try:
                r = subprocess.run([harness, path, str(k), str(BOUNDS[0]), str(BOUNDS[1]), str(a.reps)], capture_output=True, text=True, check=True)
                reps = [json.loads(x) for x in r.stdout.splitlines()]
                entry["host_parse_ms"] = median([x["host_parse_ms"] for x in reps])
                entry["host_load_counts_ms"] = median([x["load_counts_ms"] for x in reps])
                entry["host_parse_plus_load_ms"] = median([x["host_parse_ms"] + x["load_counts_ms"] for x in reps])
                entry["csv_pageable_ms"] = median([x["csv_pageable_ms"] for x in reps])
                entry["kept_rows"] = reps[0]["rows"]
                entry["same_table_row_for_row"] = bool(reps[0]["same_table"] == 1)
                entry["host_threads"] = reps[0]["threads"]
            except Exception as e:  # noqa: BLE001
                entry["host_and_pageable"] = f"not measured: {e}"
            try:
                pk = pinned_and_kernels(path, k, a.reps, tmp)
                entry.update(pk)
                entry["kernel_text_gbs"] = nbytes / (pk["kernel_ms"] * 1e-3) / 1e9
                entry["kernel_share_of_hbm"] = entry["kernel_text_gbs"] / HBM_GBS
            except Exception as e:  # noqa: BLE001
                entry["pinned_and_kernels"] = f"not measured: {e}"
            wc = {}
            for gpus in (1, 8):
                for rep in range(2):
                    for tag, exe in exes.items():  # alternating the two builds
                        key = f"{tag}_gpus{gpus}_s"
                        if time.monotonic() - t_start > a.budget_s:
                            wc.setdefault(key, "not measured: time budget")
                            continue
                        try:
                            t = wall_clock(exe, path, gpus, k, tmp, tag)
                            wc[key] = t if not isinstance(wc.get(key), float) else min(wc[key], t)
                        except Exception as e:  # noqa: BLE001
                            wc[key] = f"not measured: {e}"
            entry["run_kmerc_wall_clock_best_of_2"] = wc
            os.remove(path)
            print(json.dumps({name: entry}), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    import torch
    res["devices"] = torch.cuda.device_count()
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    json.dump(res, open(a.out, "w"), indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
