"""Where the time of a C1 step goes on the device: every kernel's duration and the time the GPU runs no kernel at all.

Runs `steps` (default 8) one-GPU C1 steps (2^24 rows, 1e6 keys, inputs resident in HBM, as bench.py) under torch.profiler
with CUDA activities, after 3 untimed warm-up steps.  A step runs from the start of one k_scatter to the start of the
next.  Per step it prints each kernel (stream, start offset in the step, duration) and the idle time: the part of the
step that no kernel on any stream covers.  Diagnostic only: the profiler adds host overhead, the bench line is the
number to quote.

    python tools/diag_gaps.py [steps] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402  (torch loads its own NCCL before libbwgpu loads the system one)
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from bytewax_b200 import gpu  # noqa: E402

A = 1_640_995_200_000_000
B = 1 << 24
N_KEYS = 1_000_000
WARMUP = 3


def short(name):
    for k in ("k_scatter", "k_segfold", "k_verdict_none", "k_verdict", "k_spill", "k_close_dirty", "k_stream_reset"):
        if k in name:
            return k
    return name.split("(")[0][:40]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("steps", type=int, nargs="?", default=8)
    ap.add_argument("--out", help="also write the per-step table as JSON here")
    args = ap.parse_args()
    ctx = gpu.Context(0)
    fold = gpu.WindowFold(ctx, "count", 60_000_000, None, A, 0, val_dtype="u64", ts_from_value=True,
                          capacity_hint=N_KEYS, max_batch_rows=B, max_emit_rows=1 << 24)
    n = args.steps + WARMUP + 1  # (+1: the last timed step's fold stage is queued by the next ingest)
    bufs = [(ctx.dev_alloc(B * 8), ctx.dev_alloc(B * 8)) for _ in range(n)]
    for s, (dk, dv) in enumerate(bufs):
        fold.gen_c1(dk, dv, s * B, B, N_KEYS)
    fold.sync()
    for s in range(WARMUP):
        fold.ingest_device(*bufs[s], None, B)
    fold.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for s in range(WARMUP, n):
            fold.ingest_device(*bufs[s], None, B)
        fold.sync()
    kern = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and e.time_range.elapsed_us() >= 0
                   and "Memcpy" not in e.name and "Memset" not in e.name), key=lambda e: e.time_range.start)
    starts = [e.time_range.start for e in kern if short(e.name) == "k_scatter"]
    rows = []
    for i in range(min(args.steps, len(starts) - 1)):
        t0, t1 = starts[i], starts[i + 1]
        ks = [e for e in kern if t0 <= e.time_range.start < t1]
        busy, end = 0.0, t0
        for e in ks:  # union of the kernels' intervals (the verdict overlaps the fold on another stream)
            a, b = max(e.time_range.start, end), min(e.time_range.end, t1)
            if b > a:
                busy += b - a
                end = b
        step_us = t1 - t0
        rows.append({"step": i, "step_us": step_us, "idle_us": step_us - busy,
                     "kernels": [{"name": short(e.name), "stream": getattr(e, "device_resource_id", None),
                                  "start_us": e.time_range.start - t0, "dur_us": e.time_range.elapsed_us()} for e in ks]})
    for r in rows:
        print(f"step {r['step']}: {r['step_us']:.1f} us, idle {r['idle_us']:.1f} us")
        for k in r["kernels"]:
            print(f"    {k['name']:<16} stream {k['stream']!s:>4}  at {k['start_us']:7.1f}  {k['dur_us']:7.1f} us")
    if rows:
        med = sorted(rows, key=lambda r: r["idle_us"])[len(rows) // 2]
        print(f"median idle per step: {med['idle_us']:.1f} us of {sorted(r['step_us'] for r in rows)[len(rows) // 2]:.1f} us "
              f"({torch.cuda.get_device_name(0)})")
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"device": torch.cuda.get_device_name(0), "steps": rows}, f, indent=1)
    fold.close()
    for dk, dv in bufs:
        ctx.dev_free(dk)
        ctx.dev_free(dv)
    ctx.close()


if __name__ == "__main__":
    main()
