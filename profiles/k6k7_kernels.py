"""Per-kernel device time of the assembly stages (K5 graph, K6 chain ranking, K7 contigs) on configs[1], from
torch.profiler with CUDA activities.  Only rfx_assemble is profiled: every step pushes and counts the reads outside the
profiler, then assembles inside it.  Prints a table of microseconds per step and launches per step, sorted by time, plus
the stage timers of the same steps (taken under the profiler: read them as shares).

    python profiles/k6k7_kernels.py [--steps 10] [--warmup 3] [--out FILE]
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the table here")
    args = ap.parse_args()

    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile
    import reflexiv_b200 as R
    from bench import Workload

    if not torch.cuda.is_available():
        raise SystemExit("k6k7_kernels.py needs a CUDA device")
    wl = Workload(2, 1)
    txt = wl.text(0)
    d_text = torch.zeros(len(txt) + 64, dtype=torch.uint8, device="cuda")
    d_text[: len(txt)].copy_(torch.from_numpy(np.asarray(txt)))
    torch.cuda.synchronize()
    ctx = R.ReflexivContext(R.DefaultParam(kmerSize=wl.k, minKmerCoverage=wl.cfg["cover"]), device=0)

    def counted():
        ctx.reset()
        ctx.push_fastq_device(d_text.data_ptr(), len(txt))
        ctx.count()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        counted()
        ctx.assemble()
    kern = {}
    stages = {"ms_graph": 0.0, "ms_extend": 0.0, "ms_contigs": 0.0}
    for _ in range(args.steps):
        counted()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            st = ctx.assemble()
            torch.cuda.synchronize()
        for key in stages:
            stages[key] += st[key]
        for e in prof.key_averages():
            us = getattr(e, "self_device_time_total", None)
            if us is None:
                us = e.self_cuda_time_total
            if us <= 0:
                continue
            t, n = kern.get(e.key, (0.0, 0))
            kern[e.key] = (t + us, n + e.count)

    card = torch.cuda.get_device_name(0)
    lines = [f"# {card}; configs[1] ({wl.describe()}); rfx_assemble under torch.profiler, {args.steps} steps after {args.warmup} warm-up",
             "# us/step  launches/step  kernel"]
    total = 0.0
    for name, (t, n) in sorted(kern.items(), key=lambda kv: -kv[1][0]):
        total += t
        short = name if len(name) <= 110 else name[:107] + "..."
        lines.append(f"{t / args.steps:9.1f}  {n / args.steps:6.1f}  {short}")
    lines.append(f"{total / args.steps:9.1f}          total device time per step")
    lines.append("# stage timers under the profiler (ms/step): " + ", ".join(f"{k} {v / args.steps:.3f}" for k, v in stages.items()))
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)
    ctx.close()


if __name__ == "__main__":
    main()
