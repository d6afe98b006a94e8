"""Generate ``tests/golden/*.json`` from the UNMODIFIED reference Python logic.

TEST INFRASTRUCTURE ONLY.  Needs a source checkout of the reference (bytewax v0.21.1):

    BYTEWAX_SRC=<checkout> python oracle/gen_golden.py

For every case it builds a real reference flow (``win.count_window`` /
``win.reduce_window`` / ``win.max_window`` / ``win.min_window`` /
``win.fold_window``), pulls the ``stateful_batch`` core step's ``builder``
out of the step tree (src/worker.rs:447-461) and drives the reference's own
``_WindowLogic`` objects with the engine rules of src/operators.rs:755-806
and :862-894 (ascending key-string order per activation, discard on
``is_complete``, ``on_eof`` at the end).  ``now_getter`` is frozen.

The cases named ``ref_*`` restate inputs of the reference's own tests and are
additionally asserted against the expected lists written in those tests.
"""

import gzip
import json
import math
import os
import random
import sys
from datetime import datetime, timedelta, timezone

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import refstub  # noqa: E402
from oracle.streams import ALIGN_US, gen_random, random_case, spec_, sweep_case  # noqa: E402

win = refstub.load()
import bytewax.operators as op  # noqa: E402  (the reference's)
from bytewax.dataflow import Dataflow  # noqa: E402
from bytewax.testing import TestingSource  # noqa: E402

EPOCH = datetime(1970, 1, 1, tzinfo=timezone.utc)
NOW = datetime(2030, 1, 1, tzinfo=timezone.utc)


def dt(us: int) -> datetime:
    return EPOCH + timedelta(microseconds=us)


def us(d: datetime) -> int:
    delta = d - EPOCH
    return (delta.days * 86400 + delta.seconds) * 1_000_000 + delta.microseconds


def build_logic_builder(spec, now_getter=None):
    """Return the reference ``stateful_batch`` builder for this spec.

    Items are ``(key_str, value, ts_us)``.
    """
    clock = win.EventClock(
        lambda x: dt(x[2]),
        wait_for_system_duration=timedelta(microseconds=spec["wait_us"]),
        now_getter=now_getter or (lambda: NOW),
    )
    offset = spec["offset_us"] or spec["length_us"]
    windower = win.SlidingWindower(
        length=timedelta(microseconds=spec["length_us"]),
        offset=timedelta(microseconds=offset),
        align_to=dt(spec["align_us"]),
    )
    flow = Dataflow("g")
    s = op.input("in", flow, TestingSource([]))
    red, ordered = spec["reduction"], spec["ordered"]
    if red == "count" and not ordered:
        wo = win.count_window("w", s, clock, windower, lambda x: x[0])
        unwrap = lambda acc: acc  # noqa: E731
    else:
        keyed = op.key_on("k", s, lambda x: x[0])
        if red == "count":
            wo = win.fold_window(
                "w", keyed, clock, windower, lambda: 0, lambda a, _x: a + 1, lambda a, b: a + b, ordered=True
            )
            unwrap = lambda acc: acc  # noqa: E731
        elif red == "sum" and not ordered:
            wo = win.reduce_window("w", keyed, clock, windower, lambda a, b: (a[0], a[1] + b[1], b[2]))
            unwrap = lambda acc: acc[1]  # noqa: E731
        elif red == "sum":
            wo = win.fold_window(
                "w",
                keyed,
                clock,
                windower,
                lambda: None,
                lambda a, x: x[1] if a is None else a + x[1],
                lambda a, b: a + b,
                ordered=True,
            )
            unwrap = lambda acc: acc  # noqa: E731
        elif red == "max":
            wo = win.max_window("w", keyed, clock, windower, by=lambda x: x[1])
            unwrap = lambda acc: acc[1]  # noqa: E731
        elif red == "min":
            wo = win.min_window("w", keyed, clock, windower, by=lambda x: x[1])
            unwrap = lambda acc: acc[1]  # noqa: E731
        elif red == "mean":
            wo = win.fold_window(
                "w",
                keyed,
                clock,
                windower,
                lambda: (0.0, 0),
                lambda a, x: (a[0] + float(x[1]), a[1] + 1),
                lambda a, b: (a[0] + b[0], a[1] + b[1]),
                ordered=ordered,
            )
            unwrap = lambda acc: list(acc)  # noqa: E731
        else:
            raise ValueError(red)
    step = refstub.find_stateful_batch(flow)
    return step.builder, unwrap


def run_reference(spec, batches):
    builder, unwrap = build_logic_builder(spec)
    logics = {}
    acts = []

    def conv(k, events):
        rows = []
        for wid, tag, payload in events:
            if tag == "E":
                rows.append([int(k), wid, "E", unwrap(payload)])
            elif tag == "L":
                rows.append([int(k), wid, "L", payload[1]])
            else:
                rows.append([int(k), wid, "M", [us(payload.open_time), us(payload.close_time)]])
        return rows

    for keys, ts, vals in batches:
        grouped = {}
        for k, t, v in zip(keys, ts, vals):
            grouped.setdefault(str(k), []).append((str(k), v, t))
        rows = []
        for ks in sorted(grouped):  # BTreeMap order, src/operators.rs:758-767
            logic = logics.get(ks)
            if logic is None:
                logic = logics[ks] = builder(None)
            events, done = logic.on_batch(grouped[ks])
            rows.extend(conv(ks, list(events)))
            if done:
                del logics[ks]
        acts.append(rows)
    rows = []
    for ks in sorted(logics):  # src/operators.rs:862-894
        events, done = logics[ks].on_eof()
        rows.extend(conv(ks, list(events)))
    acts.append(rows)
    return acts


def main():
    cases = {}

    def add(name, spec, batches, expect_down=None, cite=None):
        acts = run_reference(spec, batches)
        if expect_down is not None:
            down = [[r[0], r[1], r[3]] for act in acts for r in act if r[2] == "E"]
            assert down == expect_down, (name, down, expect_down)
        cases[name] = dict(spec=spec, batches=batches, acts=acts, cite=cite)

    S = 1_000_000
    # --- reference tests restated (keys a,b -> 1,2; "ALL" -> 0) ---------------
    # pytests/operators/windowing/test_count_window.py:10-35
    add(
        "ref_count_window",
        spec_("count", 10 * S),
        [[[1], [ALIGN_US + 0 * S], [1]], [[1], [ALIGN_US + 4 * S], [1]], [[2], [ALIGN_US + 8 * S], [1]],
         [[1], [ALIGN_US + 12 * S], [1]], [[1], [ALIGN_US + 13 * S], [1]]],
        expect_down=[[1, 0, 2], [1, 1, 2], [2, 0, 1]],
        cite="pytests/operators/windowing/test_count_window.py:10-35",
    )
    # pytests/operators/windowing/test_reduce_window.py:10-44
    add(
        "ref_reduce_window",
        spec_("sum", 10 * S),
        [[[1], [ALIGN_US + s * S], [1]] for s in (0, 4, 8, 12, 13)],
        expect_down=[[1, 0, 3], [1, 1, 2]],
        cite="pytests/operators/windowing/test_reduce_window.py:10-44",
    )
    # pytests/operators/windowing/test_fold_window.py:37-88 (per-type counts -> total count)
    add(
        "ref_fold_window_tumbling",
        spec_("count", 10 * S, ordered=True),
        [[[0], [ALIGN_US + s * S], [1]] for s in (0, 4, 8, 16)],
        expect_down=[[0, 0, 3], [0, 1, 1]],
        cite="pytests/operators/windowing/test_fold_window.py:37-88",
    )
    # pytests/operators/windowing/test_fold_window.py:143-197 (list lengths -> counts; "h" is late)
    add(
        "ref_fold_window_sliding",
        spec_("count", 10 * S, 5 * S, ordered=True),
        [[[0], [ALIGN_US + s * S], [1]] for s in (1, 4, 8, 12, 13, 14, 16, 1)],
        expect_down=[[0, -1, 2], [0, 0, 3], [0, 1, 4], [0, 2, 4], [0, 3, 1]],
        cite="pytests/operators/windowing/test_fold_window.py:143-197",
    )
    # pytests/operators/windowing/test_fold_window.py:200-235 shape, shortened:
    # 1 key, 1 s apart, tumbling 1 min, batches of 10 -> one row per minute.
    n = 6000
    add(
        "ref_fold_window_benchmark_shape",
        spec_("count", 60 * S),
        [[[0] * 10, [ALIGN_US + (i + j) * S for j in range(10)], [0] * 10] for i in range(0, n, 10)],
        expect_down=[[0, i, 60] for i in range(n // 60)],
        cite="pytests/operators/windowing/test_fold_window.py:200-235",
    )
    # pytests/operators/windowing/test_max_min_window.py:14-67 shape
    add(
        "ref_max_window",
        spec_("max", 10 * S),
        [[[1], [ALIGN_US + s * S], [v]] for s, v in ((0, 1), (4, 9), (8, 3), (12, 7), (13, 2))],
        expect_down=[[1, 0, 9], [1, 1, 7]],
        cite="pytests/operators/windowing/test_max_min_window.py:14-67",
    )
    add(
        "ref_min_window",
        spec_("min", 10 * S),
        [[[1], [ALIGN_US + s * S], [v]] for s, v in ((0, 4), (4, 9), (8, 3), (12, 7), (13, 2))],
        expect_down=[[1, 0, 3], [1, 1, 2]],
        cite="pytests/operators/windowing/test_max_min_window.py:14-67",
    )

    # --- seeded cases against the reference logic ------------------------------
    add("tumbling_count_inorder", spec_("count", 10 * S),
        gen_random(1, 1500, 23, 95 * S, 0, [1, 7, 64, 200, 13]))
    add("tumbling_count_wait_disorder", spec_("count", 10 * S, wait_us=5 * S),
        gen_random(2, 1500, 17, 80 * S, 3 * S, [50, 3, 111]))
    add("tumbling_count_lates", spec_("count", 10 * S, wait_us=0),
        gen_random(3, 1200, 11, 70 * S, 6 * S, [40, 9, 1, 130]))
    add("tumbling_count_lates_wait", spec_("count", 10 * S, wait_us=2 * S),
        gen_random(4, 1200, 9, 70 * S, 9 * S, [25, 300]))
    add("sliding_sum_lates", spec_("sum", 10 * S, 5 * S, wait_us=1 * S),
        gen_random(5, 1000, 7, 60 * S, 4 * S, [33, 5, 90]))
    add("sliding_count_indivisible_negative", spec_("count", 10 * S, 3 * S, wait_us=2 * S),
        gen_random(6, 900, 5, 50 * S, 2 * S, [20, 77], start_us=ALIGN_US - 25 * S))
    add("sliding_6x_sum_float", spec_("sum", 60 * S, 10 * S, wait_us=0),
        gen_random(7, 1500, 13, 300 * S, 0, [128, 17], fval=True))
    add("tumbling_min_float", spec_("min", 7 * S, wait_us=3 * S),
        gen_random(8, 900, 9, 60 * S, 2 * S, [45, 10], fval=True))
    add("tumbling_max_int_lates", spec_("max", 7 * S, wait_us=0),
        gen_random(9, 900, 9, 60 * S, 5 * S, [45, 10]))
    add("tumbling_mean_float", spec_("mean", 10 * S, wait_us=1 * S),
        gen_random(10, 900, 6, 60 * S, 1 * S, [64]))
    add("ordered_count_wait", spec_("count", 10 * S, wait_us=4 * S, ordered=True),
        gen_random(11, 1200, 8, 70 * S, 6 * S, [30, 200, 2]))
    add("ordered_sum_sliding_wait", spec_("sum", 10 * S, 5 * S, wait_us=3 * S, ordered=True),
        gen_random(12, 1000, 6, 60 * S, 5 * S, [70, 11]))
    add("big_keys_count", spec_("count", 10 * S),
        gen_random(13, 600, 40, 40 * S, 0, [100], key_base=(1 << 64) - 41))
    add("wait_never_closes", spec_("count", 10 * S, wait_us=10**15),
        gen_random(14, 800, 12, 100 * S, 30 * S, [100, 1]))

    # key goes quiet, all its windows close -> logic discarded, watermark resets
    # (windowing.py:1110-1113, src/operators.rs:796-799): an *older* timestamp
    # arriving later is then NOT late and re-opens window 0.
    add(
        "discard_resets_watermark",
        spec_("count", 10 * S),
        [
            [[1, 2], [ALIGN_US + 1 * S, ALIGN_US + 2 * S], [0, 0]],
            [[1, 2], [ALIGN_US + 25 * S, ALIGN_US + 3 * S], [0, 0]],
            [[1], [ALIGN_US + 45 * S], [0]],   # closes window 2 too? no: 45 s is window 4
            [[2, 1], [ALIGN_US + 31 * S, ALIGN_US + 2 * S], [0, 0]],  # key 1: ts 2 s is late
            [[3], [ALIGN_US + 5 * S], [0]],
        ],
    )

    # C1-shaped (SURVEY.md section 8d) scaled down: ts_i = align + i*1000 us, 64 keys.
    def c1(start, n):
        sys.path.insert(0, os.path.dirname(HERE))
        from oracle.pyoracle import splitmix64

        ks = [splitmix64(0x5EED ^ i) % 64 for i in range(start, start + n)]
        return [ks, [ALIGN_US + i * 1000 for i in range(start, start + n)], list(range(start, start + n))]

    add("c1_shape_small", spec_("count", 1 * S), [c1(i, 700) for i in range(0, 4200, 700)])

    out_dir = os.path.join(os.path.dirname(HERE), "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "window_fold_cases.json")
    with open(path, "w") as f:
        json.dump(cases, f, separators=(",", ":"))
    print("wrote", path, os.path.getsize(path), "bytes,", len(cases), "cases")

    # Windower / clock KATs computed by the reference classes themselves.
    kats = {"intersects": [], "clock": []}
    rnd = random.Random(99)
    for _ in range(300):
        length = rnd.choice([1, 3, 7, 10, 60]) * S
        offset = rnd.choice([o for o in (1, 2, 3, 5, 7, 10, 60) if o * S <= length]) * S
        t = ALIGN_US + rnd.randint(-200 * S, 200 * S)
        logic = win._SlidingWindowerLogic(
            timedelta(microseconds=length), timedelta(microseconds=offset), dt(ALIGN_US), win._SlidingWindowerState()
        )
        kats["intersects"].append([length, offset, ALIGN_US, t, logic.intersects(dt(t))])
    for seed in range(20):
        rnd = random.Random(1000 + seed)
        wait = rnd.choice([0, 1, 5, 30]) * S
        now = [NOW]
        logic = win._EventClockLogic(lambda: now[0], lambda x: x, lambda x: x, timedelta(microseconds=wait))
        steps = []
        for _ in range(30):
            if rnd.random() < 0.3:
                adv = rnd.randint(0, 3 * S)
                now[0] = now[0] + timedelta(microseconds=adv)
                logic.before_batch()
                steps.append(["adv", adv])
            t = ALIGN_US + rnd.randint(0, 100 * S)
            _, wm = logic.on_item(dt(t))
            steps.append(["item", t, us(wm)])
        kats["clock"].append(dict(wait_us=wait, now_us=us(NOW), steps=steps))
    path = os.path.join(out_dir, "windower_clock_kats.json")
    with open(path, "w") as f:
        json.dump(kats, f, separators=(",", ":"))
    print("wrote", path, os.path.getsize(path), "bytes")


def run_reference_timed(spec, steps):
    """Moving system clock.  ``steps``: ``["batch", now_us, keys, ts, vals]`` -- one activation's on_batch phase with
    ``now_getter() == now_us`` -- or ``["notify", now_us]`` -- the notify phase (src/operators.rs:808-858): every key whose
    ``notify_at()`` <= now gets ``on_notify()``, ascending key-string order.  Returns the rows of every step + EOF."""
    now = [dt(steps[0][1])]
    builder, unwrap = build_logic_builder(spec, now_getter=lambda: now[0])
    logics, sched, acts = {}, {}, []

    def conv(k, events):
        rows = []
        for wid, tag, payload in events:
            if tag == "E":
                rows.append([int(k), wid, "E", unwrap(payload)])
            elif tag == "L":
                rows.append([int(k), wid, "L", payload[1]])
            else:
                rows.append([int(k), wid, "M", [us(payload.open_time), us(payload.close_time)]])
        return rows

    def resched(ks, logic, done):
        if done:
            del logics[ks]
            sched.pop(ks, None)
            return
        at = logic.notify_at()
        if at is None:
            sched.pop(ks, None)
        else:
            sched[ks] = at

    for step in steps:
        now[0] = dt(step[1])
        rows = []
        if step[0] == "batch":
            _kind, _now, keys, ts, vals = step
            grouped = {}
            for k, t, v in zip(keys, ts, vals):
                grouped.setdefault(str(k), []).append((str(k), v, t))
            for ks in sorted(grouped):
                logic = logics.get(ks)
                if logic is None:
                    logic = logics[ks] = builder(None)
                events, done = logic.on_batch(grouped[ks])
                rows.extend(conv(ks, list(events)))
                resched(ks, logic, done)
        else:
            for ks in sorted(k for k, at in sched.items() if at <= now[0]):
                logic = logics[ks]
                events, done = logic.on_notify()
                rows.extend(conv(ks, list(events)))
                resched(ks, logic, done)
        acts.append(rows)
    rows = []
    for ks in sorted(logics):
        events, done = logics[ks].on_eof()
        rows.extend(conv(ks, list(events)))
    acts.append(rows)
    return acts


def main_timed():
    """tests/golden/system_time_cases.json: `_WindowLogic` + `_EventClockLogic` under a MOVING system clock, by the
    reference's own classes (windowing.py:263-302 watermark drift, :1135-1180 on_notify / notify_at)."""
    S = 1_000_000
    cases = {}

    def add(name, spec, steps, cite=None):
        cases[name] = dict(spec=spec, steps=steps, acts=run_reference_timed(spec, steps), cite=cite)

    A = ALIGN_US
    # an idle key's window closes once the system clock has carried the watermark past it
    add("idle_key_closes_on_notify", spec_("count", 10 * S),
        [["batch", A + 2 * S, [1, 1, 2], [A + 1 * S, A + int(1.5 * S), A + 1 * S], [1, 1, 1]],
         ["notify", A + 5 * S], ["notify", A + 11 * S], ["notify", A + 30 * S]],
        cite="windowing.py:289-298 on_notify; pytests/operators/windowing/test_event_clock.py")
    # the watermark drifts with the system clock: after 20 idle seconds an item 1 s newer than the key's maximum is late
    add("drift_makes_item_late", spec_("sum", 10 * S, wait_us=2 * S),
        [["batch", A + 1 * S, [7, 8], [A + 1 * S, A + 1 * S], [5, 6]],
         ["batch", A + 21 * S, [7], [A + 2 * S], [100]],
         ["batch", A + 22 * S, [8], [A + 25 * S], [7]],
         ["notify", A + 40 * S]],
        cite="windowing.py:263-287")
    # the wait holds the watermark back; due keys (close <= now) whose watermark has not got there yet emit nothing
    add("due_but_watermark_behind", spec_("count", 10 * S, wait_us=5 * S),
        [["batch", A + 9 * S, [3, 4], [A + 8 * S, A + 2 * S], [1, 1]],
         ["notify", A + 12 * S], ["notify", A + 14 * S], ["notify", A + 16 * S]])
    # sliding windows close one by one as the clock advances
    add("sliding_closes_stepwise", spec_("sum", 10 * S, offset_us=5 * S),
        [["batch", A + 8 * S, [1, 1, 2], [A + 3 * S, A + 7 * S, A + 6 * S], [1, 2, 4]],
         ["notify", A + 11 * S], ["notify", A + 16 * S], ["batch", A + 17 * S, [1], [A + 16 * S], [8]], ["notify", A + 40 * S]])
    for seed, (red, length, offset, wait, ordered) in enumerate([
            ("count", 10, None, 0, False), ("sum", 10, 5, 2, False), ("max", 7, None, 3, False), ("min", 10, 5, 0, False),
            ("count", 10, 3, 2, True), ("sum", 6, None, 1, False)]):
        rnd = random.Random(4000 + seed)
        now, steps = A + rnd.randint(0, 3 * S), []
        for _ in range(40):
            now += rnd.randint(0, 4 * S) if rnd.random() < 0.8 else rnd.randint(8 * S, 25 * S)
            if rnd.random() < 0.65:
                n = rnd.randint(1, 12)
                keys = [rnd.randint(1, 5) for _ in range(n)]
                ts = [now - rnd.randint(0, 6 * S) if rnd.random() < 0.9 else now - rnd.randint(10 * S, 40 * S) for _ in range(n)]
                steps.append(["batch", now, keys, ts, [rnd.randint(-9, 9) for _ in range(n)]])
            else:
                steps.append(["notify", now])
        add(f"random_clock_{red}_{seed}", spec_(red, length * S, offset * S if offset else None, wait * S, ordered), steps)
    out_dir = os.path.join(os.path.dirname(HERE), "tests", "golden")
    path = os.path.join(out_dir, "system_time_cases.json")
    with open(path, "w") as f:
        json.dump(cases, f, separators=(",", ":"))
    print("wrote", path, os.path.getsize(path), "bytes,", len(cases), "cases")


def main_keyed():
    """Goldens for config C2 (the reference example's own mapper) and C4 (the reference's `_JoinLogic`)."""
    src = open(os.path.join(refstub.REFERENCE_ROOT, "examples", "anomaly_detector.py")).read()
    ns = {}
    start, end = src.index("@dataclass\nclass DetectorState"), src.index("labeled_metrics =")
    exec("from dataclasses import dataclass, field\nfrom typing import List, Optional\n" + src[start:end], ns)  # examples/anomaly_detector.py:16-48
    rnd = random.Random(77)
    out = {"zscore": [], "join": []}
    for case in range(3):
        n, nkeys = 600, [1, 7, 40][case]
        keys = [rnd.randrange(nkeys) for _ in range(n)]
        vals = [float(rnd.randrange(0, 10)) if case < 2 else round(rnd.uniform(0, 10), 3) for _ in range(n)]
        states, rows = {}, []
        for k, v in zip(keys, vals):
            st, emit = ns["mapper"](states.get(k), v)
            states[k] = st
            rows.append([emit[1], emit[2], emit[3]])
        out["zscore"].append(dict(keys=keys, vals=vals, rows=rows))
    import bytewax.operators as rop

    for im in ("first", "last"):
        for em in ("complete", "running", "final"):
            items = [(rnd.randrange(9), rnd.randrange(2), rnd.randrange(1000)) for _ in range(400)]
            logics, rows = {}, []
            for k, sd, v in items:  # one item per activation (TestingSource batch_size=1)
                lg = logics.get(k)
                if lg is None:
                    lg = logics[k] = rop._JoinLogic(im, em, rop._JoinState.for_side_count(2))
                emitted, discard = lg.on_item((sd, v))
                rows.extend([k, t[0], t[1]] for t in emitted)
                if discard:
                    del logics[k]
            if em == "final":
                for k in sorted(logics, key=str):
                    emitted, _ = logics[k].on_eof()
                    rows.extend([k, t[0], t[1]] for t in emitted)
            out["join"].append(dict(insert_mode=im, emit_mode=em, items=[list(i) for i in items], rows=rows))
    path = os.path.join(os.path.dirname(HERE), "tests", "golden", "keyed_cases.json")
    with open(path, "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print("wrote", path, os.path.getsize(path), "bytes")


def main_sweep():
    """tests/golden/reference_sweep_cases.json.gz: the reference's rows per activation for the seeded specs and streams of
    `oracle.streams.random_case` (seeds 30..35) and `sweep_case` (seeds 100..147); the inputs are regenerated from the seeds."""
    out = {"random": {}, "sweep": {}}
    for name, make, seeds in (("random", random_case, range(30, 36)), ("sweep", sweep_case, range(100, 148))):
        for seed in seeds:
            spec, batches = make(seed)
            out[name][str(seed)] = dict(spec=spec, acts=run_reference(spec, batches))
    path = os.path.join(os.path.dirname(HERE), "tests", "golden", "reference_sweep_cases.json.gz")
    with gzip.GzipFile(path, "wb", mtime=0) as f:
        f.write(json.dumps(out, separators=(",", ":")).encode())
    print("wrote", path, os.path.getsize(path), "bytes")


SNAPSHOT_PARAMS = [("count", 10, None, 0), ("sum", 10, None, 3), ("sum", 10, 5, 2), ("max", 12, 4, 1)]
I64_MIN = -(1 << 63)


def _device_columns(accepted, opened_by_key, max_ts, red, length, offset, closed_upto):
    """What the device table holds at the cut: per key the live panes (those under a still-open window) with the fold of the
    accepted items in them, the first arrival index per pane, the key's running maximum and its `closed_upto`."""
    g = math.gcd(length, offset)
    a, b = offset // g, length // g
    cols = {n: [] for n in ("key", "pane_id", "acc", "count", "open_seq", "max_ts_us", "closed_upto")}
    fold = {"count": lambda x, v: x + 1, "sum": lambda x, v: x + v, "min": min, "max": max}[red]
    for k, opened in opened_by_key.items():
        panes = {}
        for seq, ts, v in accepted[k]:
            q = (ts - ALIGN_US) // g
            w_lo, w_hi = -((-(q - b + 1)) // a), q // a
            if not any(w in opened for w in range(w_lo, w_hi + 1)):
                continue  # every window of this pane has closed: the pane is gone
            cur = panes.get(q)
            if cur is None:
                panes[q] = [(1 if red == "count" else v), seq]
            else:
                cur[0] = fold(cur[0], v)
        for q, (acc, seq) in sorted(panes.items()):
            cols["key"].append(k)
            cols["pane_id"].append(q)
            cols["acc"].append(acc & 0xFFFFFFFFFFFFFFFF)
            cols["count"].append(0)
            cols["open_seq"].append(seq)
            cols["max_ts_us"].append(max_ts[k])
            cols["closed_upto"].append(closed_upto.get(k, I64_MIN))
    return cols


def main_snapshots():
    """tests/golden/snapshot_resume_cases.json: a seeded stream folded by the reference's `_WindowLogic` objects up to a cut;
    the state at the cut written the way the device dumps it (one row per live (key, pane): what `bw_snapshot_take`
    returns), the reference's own `snapshot()` of every key at the cut, and the rows the uninterrupted logics emit after it."""
    S = 1_000_000
    cases = []
    for ci, (red, length, offset, wait) in enumerate(SNAPSHOT_PARAMS):
        spec = spec_(red, length * S, offset * S if offset else None, wait * S, False)
        off = spec["offset_us"] or spec["length_us"]
        rnd = random.Random(7000 + ci)
        batches, t = [], ALIGN_US
        for _ in range(12):
            n = rnd.randint(20, 60)
            keys = [rnd.randint(1, 9) for _ in range(n)]
            ts = [t + rnd.randint(0, 6 * S) - (rnd.randint(0, 8 * S) if rnd.random() < 0.2 else 0) for _ in range(n)]
            t += 5 * S
            batches.append([keys, ts, [rnd.randint(-20, 20) for _ in range(n)]])
        cut = 6
        builder, unwrap = build_logic_builder(spec)

        def drive(logics, chunk, seq0, accepted=None, max_ts=None):
            rows = []
            for bi, (keys, ts, vals) in enumerate(chunk):
                grouped = {}
                for i, (k, tt, v) in enumerate(zip(keys, ts, vals)):
                    grouped.setdefault(str(k), []).append((str(k), v, tt, (seq0 + bi) << 32 | i))
                for ks in sorted(grouped):
                    logic = logics.get(ks)
                    if logic is None:
                        logic = logics[ks] = builder(None)
                    events, done = logic.on_batch([(k, v, tt) for k, v, tt, _s in grouped[ks]])
                    events = list(events)
                    late_vals = [p[1] for _w, tag, p in events if tag == "L"]
                    for k, v, tt, sq in grouped[ks]:
                        if accepted is not None:
                            if late_vals and v in late_vals and any(p[2] == tt for _w, tag, p in events if tag == "L"):
                                continue
                            accepted.setdefault(int(ks), []).append((sq, tt, v))
                            max_ts[int(ks)] = max(max_ts.get(int(ks), I64_MIN), tt)
                    rows.extend([ks, w, tag, (unwrap(p) if tag == "E" else None)] for w, tag, p in events if tag != "M")
                    if done:
                        del logics[ks]
                        if accepted is not None:  # the key's state is gone with its logic (discard resets the watermark)
                            accepted.pop(int(ks), None)
                            max_ts.pop(int(ks), None)
            return rows

        # uninterrupted
        ref_logics = {}
        drive(ref_logics, batches[:cut], 0)
        want = drive(ref_logics, batches[cut:], cut)
        want_eof = [[ks, w, tag, unwrap(p) if tag == "E" else None] for ks in sorted(ref_logics)
                    for w, tag, p in ref_logics[ks].on_eof()[0] if tag != "M"]
        # up to the cut, remembering what the table would hold
        logics, accepted, max_ts = {}, {}, {}
        drive(logics, batches[:cut], 0, accepted, max_ts)
        opened_by_key = {int(ks): dict(lg.windower.state.opened) for ks, lg in logics.items()}
        # sliding windows: every id below the oldest open one that covers a live pane has been emitted
        closed_upto = {k: (min(o) - 1 if (offset and o) else I64_MIN) for k, o in opened_by_key.items()}
        cols = _device_columns(accepted, opened_by_key, max_ts, red, spec["length_us"], off, closed_upto)
        snaps = {}
        for ks, lg in logics.items():
            real = lg.snapshot()
            snaps[ks] = dict(
                opened=[[w, us(m.open_time), us(m.close_time)] for w, m in real.windower_state.opened.items()],
                logic_states=[[w, unwrap(v) if red != "count" else v] for w, v in real.logic_states.items()],
                clock_delta_us=us(real.clock_state.watermark_base) - us(real.clock_state.system_time_of_max_event),
            )
        cases.append(dict(params=[red, length, offset, wait], spec=spec, now_us=us(NOW), cut=cut, batches=batches,
                          columns=cols, snapshots=snaps, want=want, want_eof=want_eof))
    path = os.path.join(os.path.dirname(HERE), "tests", "golden", "snapshot_resume_cases.json")
    with open(path, "w") as f:
        json.dump(cases, f, separators=(",", ":"))
    print("wrote", path, os.path.getsize(path), "bytes,", len(cases), "cases")


if __name__ == "__main__":
    main()
    main_keyed()
    main_timed()
    main_sweep()
    main_snapshots()
