#!/usr/bin/env python
"""Benchmark of the north-star path: tumbling fold_window count-by-key (config C1).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (SURVEY.md section 8d, BASELINE.json configs[1]): rows (u64 key, u64 val),
key_i = splitmix64(0x5EED ^ i) mod 10^6, val_i = ts_i = i us after 2022-01-01,
EventClock(wait=0), TumblingWindower(60 s), count fold.  One step = one
activation (epoch batch) of 2^24 rows per GPU; the default 60 steps are the
whole 10^9-row job.  Inputs (60 x 256 MiB per GPU) never fit the 126 MB L2.

Printed JSON (one line, rank 0): `value` = events/s with inputs resident in
HBM (CUDA events on the launching stream, max over ranks); `e2e` = the same
job through the C ABI from pinned HOST buffers (H2D of every step and D2H of
every emitted row inside the timed region); `roofline` for the fold kernel;
`cpu_baseline` = the C restatement of the reference path (oracle/) on the
host cores, bounded sample.

`--impl reference` times that CPU restatement alone (the reference's Rust
engine cannot be built here: no cargo, un-vendored timely -- DESIGN.md).

`--dump-outputs DIR` writes, after the timed steps, the rows the timed job hands
its caller: `bw_advance` after the last timed step (every window the K steps
closed) and `bw_eof` (the windows still open), one float64 `DIR/<name>.npy` per
non-empty column (the C1 stream has no late rows, so no late columns).  The
inputs depend only on the arguments, so two builds given the same arguments can
be compared file by file.
"""

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALIGN_US = 1_640_995_200_000_000
N_KEYS = 1_000_000
WINDOW_US = 60_000_000
BATCH_ROWS = 1 << 24
BYTES_PER_EVENT = 16  # SURVEY.md 8(d): one read of the (u64, u64) record
DUMP_BYTES = 60 << 20  # --dump-outputs writes at most this much: a seeded sample of each longer column


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device=0):
        self.device, self.proc, self.lines = device, None, []
        self.nvml_samples, self._stop = [], threading.Event()

    def _nvml_loop(self):
        """NVML polled every ~2 ms beside nvidia-smi's 100 ms loop: the timed region is only tens of milliseconds long."""
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.device)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            bits = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40), ("sw_power_cap", 0x4))
            while not self._stop.is_set():
                try:
                    sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    self.nvml_samples.append((float(sm), float(mx), [n for n, b in bits if r & b]))
                except Exception:
                    pass
                time.sleep(0.002)
        except Exception:
            return

    def start(self):
        try:
            self.tn = threading.Thread(target=self._nvml_loop, daemon=True)
            self.tn.start()
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.device)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        self._stop.set()
        if not self.proc and not self.nvml_samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        for c, m, rs in self.nvml_samples:
            sm.append(c)
            mx.append(m)
            reasons.update(rs)
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # under load == upper half of the samples
        load = sm[len(sm) // 2:] if sm else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n):
    """torch.distributed is plumbing only: rendezvous, barrier, max-over-ranks."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    if world == 1:
        return 0, 1, 0, None
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local, dist


def barrier_max(dist, local, value):
    if dist is None:
        return value
    import torch

    t = torch.tensor([value], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(dist, local):
    if dist is not None:
        import torch

        dist.barrier(device_ids=[local])
        torch.cuda.synchronize(local)


def share_nccl_id(dist, rank, local):
    from bytewax_b200 import gpu
    import torch

    buf = torch.zeros(128, dtype=torch.uint8, device=f"cuda:{local}")
    if rank == 0:
        buf.copy_(torch.frombuffer(bytearray(gpu.Context.new_nccl_id()), dtype=torch.uint8))
    dist.broadcast(buf, 0)
    return bytes(buf.cpu().numpy().tobytes())


def check_counts(em, em_eof, K, B, world, dist, local, ts_stride, late_frac=0.0):
    """Size-independent checks of a whole job (SURVEY 8d C1 (ii)), over ALL ranks: the counts add up to the rows ingested,
    and -- ts_i = i us -- every full 60 s window of the global stream holds exactly 6e7 / ts_stride events."""
    import numpy as np

    wid = np.concatenate([em.closed_window_id, em_eof.closed_window_id])
    acc = np.concatenate([em.closed_acc, em_eof.closed_acc]).astype(np.int64)
    nwin = (K * B * world * ts_stride) // WINDOW_US + 2
    per_window = np.bincount(wid, weights=acc, minlength=nwin).astype(np.int64)[:nwin] if len(wid) else np.zeros(nwin, np.int64)
    if dist is not None:
        import torch

        t = torch.from_numpy(per_window.copy()).to(f"cuda:{local}")
        dist.all_reduce(t)
        per_window = t.cpu().numpy()
    total = int(per_window.sum())
    nfull = (K * B * world * ts_stride) // WINDOW_US
    if late_frac > 0:  # diagnostic stream with late rows: every row is either counted or in the late stream (one window each)
        n_late = len(em.late_key) + len(em_eof.late_key)
        if dist is not None:
            import torch

            t = torch.tensor([n_late], dtype=torch.int64, device=f"cuda:{local}")
            dist.all_reduce(t)
            n_late = int(t.item())
        if total + n_late != K * B * world:
            raise SystemExit(f"bench: WRONG RESULT: counted {total} + late {n_late} != {K * B * world}")
        return total, f"late rows {n_late}"
    ok = bool(total == K * B * world and (per_window[:nfull] == WINDOW_US // ts_stride).all())
    if not ok:
        raise SystemExit(f"bench: WRONG RESULT: sum of counts {total} != {K * B * world} or a full window is not {WINDOW_US // ts_stride}")
    return total, ok


def run_gpu(args):
    if args.ts_stride != 1 or args.late_frac > 0:
        import torch  # noqa: F401  (diagnostic mode only; torch must load its own NCCL before libbwgpu loads the system one)
    from bytewax_b200 import _native as N, gpu

    rank, world, local, dist = dist_setup(args.gpus)
    nccl_id = share_nccl_id(dist, rank, local) if world > 1 else None
    ctx = gpu.Context(local, rank, world, nccl_id)
    K, W, B = args.steps, args.warmup, args.batch_rows
    N_KEYS = args.n_keys

    def make_fold(ring_slots=3, emit_order=N.ORDER_REFERENCE):
        return gpu.WindowFold(
            ctx, "count", WINDOW_US, None, ALIGN_US, 0, val_dtype="u64", ts_from_value=True,
            emit_order=emit_order, capacity_hint=N_KEYS if world == 1 else (N_KEYS * 3) // (2 * world) + 1024,
            max_batch_rows=B, max_emit_rows=max(1 << 20, (K + W + 2) * B // 40),
            max_late_rows=(1 << 16) if args.late_frac <= 0 else int((K + W + 2) * B * args.late_frac * 1.5) + (1 << 16),
            ring_slots=ring_slots, exchange=N.XCHG_NCCL if args.exchange == "nccl" else N.XCHG_P2P)

    # ---- device-resident inputs: step s of this rank = global rows [(s*world+rank)*B, +B) ----
    nbuf = K + W
    fold = make_fold()
    dk = [ctx.dev_alloc(B * 8) for _ in range(nbuf)]
    dv = [ctx.dev_alloc(B * 8) for _ in range(nbuf)]
    for s in range(nbuf):
        fold.gen_c1(dk[s], dv[s], (s * world + rank) * B, B, N_KEYS)
    fold.sync()
    if args.ts_stride != 1:
        # diagnostic: stretch event time (ts = stride * row index) to reproduce on one GPU the
        # activations of an N-rank job, which span N x 2^24 us each
        import torch

        scratch = torch.empty(B, dtype=torch.int64, device=f"cuda:{local}")
        for s in range(nbuf):
            ctx.lib.bw_memcpy(ctx.h, C.c_void_p(scratch.data_ptr()), C.c_void_p(dv[s]), B * 8, 2)
            scratch.mul_(args.ts_stride)
            torch.cuda.synchronize(local)
            ctx.lib.bw_memcpy(ctx.h, C.c_void_p(dv[s]), C.c_void_p(scratch.data_ptr()), B * 8, 2)
        del scratch
    if args.late_frac > 0:
        # diagnostic: every 1/late_frac-th row is sent 120 s into the past (two windows late): its activation cannot be
        # proven clean and takes the exact path
        import torch

        period = max(2, int(round(1.0 / args.late_frac)))
        scratch = torch.empty(B, dtype=torch.int64, device=f"cuda:{local}")
        mask = (torch.arange(B, device=f"cuda:{local}") % period) == (period // 2)
        for s in range(nbuf):
            ctx.lib.bw_memcpy(ctx.h, C.c_void_p(scratch.data_ptr()), C.c_void_p(dv[s]), B * 8, 2)
            scratch[mask] = torch.clamp(scratch[mask] - 120_000_000, min=0)
            torch.cuda.synchronize(local)
            ctx.lib.bw_memcpy(ctx.h, C.c_void_p(dv[s]), C.c_void_p(scratch.data_ptr()), B * 8, 2)
        del scratch, mask
    # warm-up: W untimed steps on a scratch fold (same shapes)
    for s in range(W):
        fold.ingest_device(dk[K + s], dv[K + s], None, B)
    fold.advance()
    fold.close()
    # The timed region is exactly K steps on a fresh fold (created outside it).  --min-timed-s > 0 repeats that K-step job
    # (a fresh fold each time) until that much timed device work has accumulated, so that the clock / throttle sampler
    # sees the GPU under load; ms_per_step is then the MEDIAN repetition.
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    rep_ms, reps_total_ms = [], 0.0
    st0 = st1 = None
    checks = emitted = None
    while True:
        fold = make_fold()
        st0 = fold.stats()
        barrier(dist, local)
        fold.time_begin()
        for s in range(K):
            fold.ingest_device(dk[s], dv[s], None, B)
        ms = fold.time_end()
        barrier(dist, local)
        ms = barrier_max(dist, local, ms)
        rep_ms.append(ms)
        reps_total_ms += ms
        st1 = fold.stats()
        more = reps_total_ms < args.min_timed_s * 1e3 and len(rep_ms) < args.max_repeats
        if not more or checks is None:
            # correctness of what was timed (first and last repetition): every row counted once, in the right window
            em = fold.advance()
            em_eof = fold.eof()
            checks = check_counts(em, em_eof, K, B, world, dist, local, args.ts_stride, args.late_frac)
            emitted = (em, em_eof)
        fold.close()
        if not more:
            break
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"advance": emitted[0], "eof": emitted[1]})
    rep_ms.sort()
    ms = rep_ms[len(rep_ms) // 2]
    total_counts, per_window_ok = checks
    launches = int(st1.kernel_launches - st0.kernel_launches)
    fold_ms_avg = st1.sum_fold_ms / max(1, st1.timed_folds)  # (every 4th activation's kernels are timed: bw_stats.timed_folds)
    scatter_ms_avg = st1.sum_scatter_ms / max(1, st1.scatter_launches)
    verdict_ms_avg = st1.sum_verdict_ms / max(1, st1.scatter_launches)
    # rows per fold launch (an activation may be folded in several sub-range launches); ~B per rank per step after an exchange
    rows_per_fold = st1.fold_rows / max(1, st1.timed_folds) if world == 1 else K * B / max(1, st1.fold_launches)
    combined = int(st1.combined_folds)
    fold_path = "direct" if combined == 0 else ("stream" if combined == st1.fold_launches else "mixed")
    for p in dk + dv:
        ctx.dev_free(p)
    value = K * B * world / (ms / 1e3)

    # ---- end to end: pinned host -> H2D -> kernels -> ordered rows D2H ----
    e2e = None
    if not args.no_e2e:
        try:
            e2e = run_e2e(ctx, make_fold, K if world == 1 else min(K, 16), B, rank, world, dist, local)
        except Exception as ex:  # pinned allocation can fail on small hosts
            e2e = {"value": None, "unit": "events/s", "error": str(ex)[:200]}

    out = None
    if rank == 0:
        peak, peak_src = peaks()
        # Two streaming kernels make the fold stage of the default path; the roofline object is the slower one's
        # (16 algorithmic bytes per event, SURVEY 8d, over its CUDA-event time), `stage` has both and their sum.
        kern = {"k_fold" if fold_path == "direct" else "k_segfold": fold_ms_avg}
        if fold_path != "direct" and scatter_ms_avg > 0:
            kern["k_scatter"] = scatter_ms_avg
            kern["k_verdict"] = verdict_ms_avg
        dom = max(kern, key=kern.get)
        gbs = lambda t: BYTES_PER_EVENT * rows_per_fold / (t / 1e3) / 1e9 if t > 0 else None  # noqa: E731
        achieved = gbs(kern[dom])
        stage_ms = sum(kern.values())
        traffic = None
        tp = os.path.join(ROOT, "profiles", "fold_traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                traffic = json.load(f).get(dom.split()[0], {}).get("dram_bytes_per_launch")
        out = {
            "metric": "events/sec tumbling fold_window count-by-key",
            "value": value, "unit": "events/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": {
                "workload": "C1: tumbling fold_window count-by-key, 2^24-row epochs of (u64 key, u64 val), "
                            "1e6 distinct keys, 60 s windows, EventClock wait=0 (BASELINE.json configs[1])",
                "rows_per_step_per_gpu": B, "total_rows": K * B * world, "n_keys": N_KEYS,
                "l2": "inputs larger than L2 (each step reads a distinct 256 MiB batch; 16 GiB resident)",
                "exchange": ("none" if world == 1 else args.exchange), "emit_order": "reference",
                "sum_of_counts_check": total_counts, "per_window_totals_exact": per_window_ok,
                "checks_cover": "all ranks (all-reduced); the run aborts when they fail",
                "fold_path": fold_path,
                "repeats": len(rep_ms), "timed_region_s": reps_total_ms / 1e3,
                "ms_per_step_min_median_max": [rep_ms[0] / K, ms / K, rep_ms[-1] / K],
            },
            "clocks": clocks,
            "e2e": e2e,
            "gpu_launches": launches,
            "roofline": {
                "bound": "hbm", "kernel": dom,
                "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                "peak_source": peak_src, "algorithmic_bytes_per_event": BYTES_PER_EVENT,
                "avg_launch_ms": kern[dom], "rows_per_launch": rows_per_fold,
                "timed_launches": int(st1.timed_folds), "timed_launches_note": "CUDA events around every 4th activation's kernels (last repetition)",
                "stage": {"kernels_avg_ms": kern, "sum_ms": stage_ms, "achieved": gbs(stage_ms),
                          "frac": (gbs(stage_ms) / peak) if stage_ms > 0 else None,
                          "bytes_moved_per_event": 16 + 16 + 16 + 4,
                          "note": "the design moves ~52 B/event: 16 in + 16 B record out (scatter), 16 B record in + table slice (fold)"},
            },
        }
        if args.late_frac > 0:  # diagnostic line: how the not-clean activations were handled in the last repetition
            out["config"]["late_frac"] = args.late_frac
            out["config"]["late_path"] = {"split_batches": int(st1.split_batches - st0.split_batches),
                                          "sort_batches": int(st1.slow_batches - st0.slow_batches), "steps": K}
        if world == 1 and not args.no_cpu:
            out["cpu_baseline"] = cpu_baseline(sample_rows=1 << 22)
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(out))


def dump_outputs(out_dir, streams):
    """Every non-empty column of every `Emitted` as float64 `out_dir/<stream>_<column>.npy` (the bench's keys, window ids,
    counts and epochs are far below 2^53, so the values are exact).  A column longer than its share of DUMP_BYTES is replaced by the
    rows at a seeded, sorted sample of positions: the same positions for the same row count, so emission order still counts."""
    import dataclasses

    import numpy as np

    cols = {f"{name}_{f.name}": getattr(em, f.name) for name, em in streams.items() for f in dataclasses.fields(em)}
    cols = {name: a for name, a in cols.items() if len(a)}
    cap = DUMP_BYTES // (8 * len(cols))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in cols.items():
        if len(a) > cap:
            a = a[np.sort(np.random.default_rng(0x5EED).choice(len(a), cap, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def run_e2e(ctx, make_fold, K, B, rank, world, dist, local):
    """Same job through the public C-ABI calls with HOST buffers."""
    import numpy as np

    fold = make_fold(ring_slots=K + 1)
    # fill K pinned slots (untimed): generate on the device, copy back into the slot
    dk, dv = ctx.dev_alloc(B * 8), ctx.dev_alloc(B * 8)
    slots = []
    for s in range(K):
        b = fold.acquire(B)
        fold.gen_c1(dk, dv, (s * world + rank) * B, B, 1_000_000)
        fold.sync()
        ctx.lib.bw_memcpy(ctx.h, C.cast(b.keys, C.c_void_p), C.c_void_p(dk), B * 8, 1)
        ctx.lib.bw_memcpy(ctx.h, b.vals, C.c_void_p(dv), B * 8, 1)
        slots.append(b)
    ctx.dev_free(dk)
    ctx.dev_free(dv)
    barrier(dist, local)
    t0 = time.perf_counter()
    fold.time_begin()
    commit_ms = []
    for s in range(K):
        tc = time.perf_counter()
        fold.commit(slots[s], B)
        commit_ms.append((time.perf_counter() - tc) * 1e3)
    # waits, orders, copies every emitted row into the library's pinned host buffers; the rows are consumed
    # in place (the C ABI hands out pointers that stay valid until the next advance / eof)
    ta = time.perf_counter()
    em = fold.advance(copy=False)
    out_rows, acc_sum = len(em.closed_key), int(em.closed_acc.sum())
    te = time.perf_counter()
    em2 = fold.eof(copy=False)
    out_rows, acc_sum = out_rows + len(em2.closed_key), acc_sum + int(em2.closed_acc.sum())
    tz = time.perf_counter()
    dev_ms = fold.time_end()
    wall_ms = (time.perf_counter() - t0) * 1e3
    barrier(dist, local)
    ms = barrier_max(dist, local, max(dev_ms, wall_ms))
    if dist is not None:  # every rank's rows, summed: the whole job's count
        import torch

        t = torch.tensor([acc_sum], dtype=torch.int64, device=f"cuda:{local}")
        dist.all_reduce(t)
        acc_sum = int(t.item())
    assert acc_sum == K * B * world, (acc_sum, K * B * world)
    fold.close()
    return {
        "value": K * B * world / (ms / 1e3), "unit": "events/s", "h2d_bytes_per_step": B * 16,
        "d2h_bytes_per_step": out_rows * 40 // K, "ms_total": ms, "steps": K,
        # where the time went (host clock): one commit == H2D of 16 B/row + lateness verdict; 2^24 rows at 55 GB/s == 4.9 ms
        "commit_ms_median": sorted(commit_ms)[len(commit_ms) // 2], "commit_ms_max": max(commit_ms),
        "advance_ms": (te - ta) * 1e3, "eof_ms": (tz - te) * 1e3,
        "path": "bw_ingest_commit (pinned slot -> async H2D) x steps, bw_advance + bw_eof (ordered rows D2H)",
    }


def cpu_baseline(sample_rows, budget_s=5.0, max_batches=80, threads=None, runs=3):
    """The C restatement of the reference path (oracle/fold_oracle.c) on the host cores: `runs` independent runs (fresh
    state each) of consecutive activations of the C1 stream, about `budget_s` seconds of fold time each; the value is
    the MEDIAN run (the host is shared: single runs of this arm have differed by 2x)."""
    from oracle import coracle

    T = threads or min(os.cpu_count() or 1, 64)
    l = coracle.lib()
    rates, secs, nb_used = [], 0.0, 0
    for _ in range(runs):
        orcs = [coracle.COracle("count", WINDOW_US, align_us=ALIGN_US) for _ in range(T)]
        arr = (C.c_void_p * T)(*[o.h for o in orcs])
        dt, n_batches = 0.0, 0
        while dt < budget_s and n_batches < max_batches:
            keys, ts, _ = coracle.gen_c1(n_batches * sample_rows, sample_rows, N_KEYS, ALIGN_US)  # untimed
            t0 = time.perf_counter()
            l.orc_on_batch_mt(arr, T, keys.ctypes.data_as(C.c_void_p), ts.ctypes.data_as(C.c_void_p), sample_rows)
            dt += time.perf_counter() - t0
            n_batches += 1
        for o in orcs:
            o.close()
        rates.append(sample_rows * n_batches / dt)
        secs += dt
        nb_used = n_batches
    rates.sort()
    return {
        "value": rates[len(rates) // 2], "unit": "events/s", "cores": T, "kind": "port",
        "sample": f"median of {runs} runs, each {nb_used} activations x {sample_rows} rows of C1 from the start of the job, "
                  f"{T} key-sharded worker threads, C restatement of the reference's Python logic + Rust engine order",
        "seconds": secs, "runs": rates,
    }


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the path.

    The Rust/Timely engine is unbuildable here, so this is the oracle port
    (oracle/fold_oracle.c) with all host threads; each step is a bounded sample
    (2^22 rows) of the same workload.  Under torchrun only rank 0 works."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import coracle

    T = min(os.cpu_count() or 1, 64)
    rows = args.batch_rows  # the same step as the GPU arm: one 2^24-row activation
    l = coracle.lib()
    orcs = [coracle.COracle("count", WINDOW_US, align_us=ALIGN_US) for _ in range(T)]
    arr = (C.c_void_p * T)(*[o.h for o in orcs])
    K, W = args.steps, args.warmup
    times = []
    for s in range(W + K):
        keys, ts, _ = coracle.gen_c1(s * rows, rows, N_KEYS, ALIGN_US)
        t0 = time.perf_counter()
        l.orc_on_batch_mt(arr, T, keys.ctypes.data_as(C.c_void_p), ts.ctypes.data_as(C.c_void_p), rows)
        if s >= W:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    value = rows * K / total
    sample = f"{K} steps x {rows} rows of C1 (the GPU arm's step), {T} key-sharded worker threads (oracle/fold_oracle.c)"
    print(json.dumps({
        "impl": "reference", "metric": "events/sec tumbling fold_window count-by-key", "value": value,
        "unit": "events/s", "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": total / K * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "C1: tumbling fold_window count-by-key, 2^24-row epochs of (u64 key, u64 val), 1e6 distinct keys, "
                               "60 s windows, EventClock wait=0 (BASELINE.json configs[1]); the first steps of the job",
                   "rows_per_step_per_gpu": rows, "n_keys": N_KEYS},
        "cpu_baseline": {"value": value, "unit": "events/s", "cores": T, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def run_config(args):
    """Secondary lines for BASELINE.json configs[2..4] (`--config c2|c3|c4`; the headline stays C1).  One GPU, scaled so a
    run takes seconds; inputs are made with numpy on the host (untimed).  c3 goes through the same fold kernels as C1
    (device columns, CUDA-event timing); c2 / c4 time the public call with HOST columns (their C-ABI entry points take
    host arrays), i.e. they are end-to-end numbers."""
    import numpy as np

    from bytewax_b200 import _native as N, gpu

    rank, world, local, dist = (0, 1, 0, None)
    if args.config == "c3":  # the one secondary config whose path shards: same launch contract as the headline
        rank, world, local, dist = dist_setup(args.gpus)
    nccl_id = share_nccl_id(dist, rank, local) if world > 1 else None
    ctx = gpu.Context(local, rank, world, nccl_id)
    K, W = args.steps, args.warmup
    rnd = np.random.default_rng(7 + rank)
    out = {"n_gpus": world, "steps": K, "warmup": W, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "data": "synthetic", "unit": "events/s"}
    if args.config == "c3":
        B = min(args.batch_rows, 1 << 22)
        S = 1_000_000
        mk = lambda emit: gpu.WindowFold(  # noqa: E731
            ctx, "sum", 60 * S, 10 * S, ALIGN_US, 0, val_dtype="f32", capacity_hint=N_KEYS if world == 1 else (N_KEYS * 3) // (2 * world) + 1024,
            max_batch_rows=B, max_emit_rows=emit, max_late_rows=1 << 16, exchange=N.XCHG_NCCL if args.exchange == "nccl" else N.XCHG_P2P)
        fold = mk(1 << 24)
        bufs, tot = [], 0.0
        for s in range(K + W):  # in-order event time, 1 us per row of the global stream; rank r holds the r-th slice of a step
            keys = rnd.integers(0, N_KEYS, B).astype(np.uint64)
            vals = rnd.random(B).astype(np.float32)
            ts = (ALIGN_US + ((s * world + rank) * B + np.arange(B))).astype(np.int64)
            d = [ctx.dev_alloc(B * 8), ctx.dev_alloc(B * 4), ctx.dev_alloc(B * 8)]
            for p_, a in zip(d, (keys, vals, ts)):
                ctx.lib.bw_memcpy(ctx.h, C.c_void_p(p_), a.ctypes.data_as(C.c_void_p), a.nbytes, 0)
            bufs.append(d)
            if s >= W:
                tot += float(vals.astype(np.float64).sum())
        for s in range(W):
            fold.ingest_device(bufs[s][0], bufs[s][1], bufs[s][2], B)
        fold.advance()
        fold.close()
        fold = mk(1 << 25)
        barrier(dist, local)
        fold.time_begin()
        for s in range(W, K + W):
            fold.ingest_device(bufs[s][0], bufs[s][1], bufs[s][2], B)
        ms = fold.time_end()
        barrier(dist, local)
        ms = barrier_max(dist, local, ms)
        em, em2 = fold.advance(), fold.eof()
        got = float(em.closed_acc.astype(np.float64).sum() + em2.closed_acc.astype(np.float64).sum())
        if dist is not None:  # every rank's windows / values, summed
            import torch

            t = torch.tensor([got, tot], dtype=torch.float64, device=f"cuda:{local}")
            dist.all_reduce(t)
            got, tot = float(t[0].item()), float(t[1].item())
        ok = abs(got - 6.0 * tot) <= 1e-5 * 6.0 * tot  # every value lands in exactly length / offset = 6 windows
        if not ok:
            raise SystemExit(f"bench c3: WRONG RESULT: sum over windows {got} != 6 x sum of values {6 * tot}")
        st = fold.stats()
        out.update(metric="events/sec sliding 60s/10s sum (f32) by key", value=K * B * world / (ms / 1e3), ms_per_step=ms / K, dtype="f32",
                   config={"workload": "C3 shape: sliding 60 s / 10 s event-time sum, f32 values, 1e6 keys, in-order (BASELINE.json configs[3], scaled)",
                           "rows_per_step_per_gpu": B, "total_rows": K * B * world, "sum_over_windows_equals_6x_sum_of_values": ok,
                           "checks_cover": "all ranks (all-reduced)", "exchange": "none" if world == 1 else args.exchange,
                           "fold_path": "stream" if st.combined_folds == st.fold_launches else "mixed", "timing": "CUDA events (bw_fold_time_begin/end), max over ranks, inputs resident in HBM"})
        fold.close()
    elif args.config == "c2":
        B = min(args.batch_rows, 1 << 22)
        n_ranks = 100_000
        zm = gpu.ZScoreMap(ctx, 10, 2.0, val_dtype="f32", capacity_hint=n_ranks, max_batch_rows=B)
        steps = []
        for s in range(K + W):
            ranks = np.minimum(rnd.zipf(1.1, B), n_ranks).astype(np.uint64)
            steps.append((ranks, rnd.normal(0.0, 1.0, B).astype(np.float32)))
        for s in range(W):
            zm.apply(*steps[s])
        t0 = time.perf_counter()
        flagged = 0
        for s in range(W, K + W):
            _mu, _sigma, flag = zm.apply(*steps[s])
            flagged += int(flag.sum())
        dt = time.perf_counter() - t0
        out.update(metric="events/sec stateful_map z-score detector (K5)", value=K * B / dt, ms_per_step=dt * 1e3 / K, dtype="f32",
                   config={"workload": "C2 shape: stateful_map rolling z-score (examples/anomaly_detector.py), Zipf-1.1 keys over 1e5 ranks, f32 (BASELINE.json configs[2])",
                           "rows_per_step": B, "total_rows": K * B, "anomalies_flagged": flagged,
                           "timing": "wall clock around bw_smap_apply with HOST columns in and out (end to end; includes pageable H2D / D2H)"})
        zm.close()
    elif args.config == "c4":
        B = min(args.batch_rows, 1 << 21)
        n_keys = 50_000_000
        kj = gpu.KeyedJoin(ctx, "last", "complete", capacity_hint=min(n_keys, 2 * B * (K + W)), max_batch_rows=2 * B, max_emit_rows=4 * B)
        steps = []
        for s in range(K + W):  # both sides of an activation, interleaved arrival
            keys = rnd.integers(0, n_keys if args.n_keys == N_KEYS else args.n_keys, 2 * B).astype(np.uint64)
            sides = (np.arange(2 * B) & 1).astype(np.uint8)
            steps.append((keys, sides, np.arange(2 * B, dtype=np.uint64) + s * 2 * B))
        lib = ctx.lib
        rows = N.BwJoinRows()
        for s in range(W):
            kj.apply(*steps[s])
            N.check(lib.bw_join_advance(kj.h, C.byref(rows)), ctx.h)
        t0 = time.perf_counter()
        emitted = 0
        for s in range(W, K + W):
            kj.apply(*steps[s])
            N.check(lib.bw_join_advance(kj.h, C.byref(rows)), ctx.h)
            emitted += int(rows.n)
        dt = time.perf_counter() - t0
        out.update(metric="events/sec two-stream keyed join (K6)", value=K * 2 * B / dt, ms_per_step=dt * 1e3 / K, dtype="u64",
                   config={"workload": "C4 shape on 1 GPU: two-stream keyed join, u64 keys, insert last / emit complete (BASELINE.json configs[4], scaled)",
                           "rows_per_step_both_sides": 2 * B, "total_rows": K * 2 * B, "pairs_emitted": emitted,
                           "timing": "wall clock around bw_join_apply + bw_join_advance with HOST columns (end to end)"})
        kj.close()
    else:
        raise SystemExit(f"unknown --config {args.config!r} (c2, c3 or c4)")
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(out))


def main():
    # stdout carries exactly one JSON line: NCCL's version banner (NCCL_DEBUG=VERSION in some images) goes to stdout too
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 60 for c1, 8 for c2 | c3 | c4)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--batch-rows", type=int, default=BATCH_ROWS)
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"])
    ap.add_argument("--n-keys", type=int, default=N_KEYS, help="diagnostic: key cardinality (the metric is quoted at the default)")
    ap.add_argument("--ts-stride", type=int, default=1, help="diagnostic: event time advances this many us per row")
    ap.add_argument("--min-timed-s", type=float, default=0.0,
                    help="repeat the K-step job (a fresh fold each time) until this much timed device work; ms_per_step is the median")
    ap.add_argument("--max-repeats", type=int, default=200)
    ap.add_argument("--late-frac", type=float, default=0.0, help="diagnostic: this fraction of the rows arrives 120 s late (exact path)")
    ap.add_argument("--config", default="c1", help="c1 (the headline metric, default); c2 | c3 | c4: secondary lines for BASELINE.json configs[2..4]")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the rows the timed job emits to DIR/<name>.npy (c1 on the GPU only)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.config != "c1"):
        ap.error("--dump-outputs needs the c1 GPU path")
    if args.steps is None:
        args.steps = 60 if args.config == "c1" else 8
    if args.impl == "reference":
        run_reference(args)
    elif args.config != "c1":
        run_config(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
