"""`bytewax_b200.snapshot_rows`: the columnar device snapshot turned into the reference's per-key `_WindowSnapshot` objects.

`tests/golden/snapshot_resume_cases.json` (oracle/gen_golden.py) holds, per case, a seeded stream folded by the reference's OWN
`_WindowLogic` objects up to a cut: the state at the cut written the way the device dumps it (one row per live (key, pane): what
`bw_snapshot_take` returns), the reference's own `snapshot()` of every key there, and the rows the uninterrupted logics emit
after the cut.  The columns are converted, must equal the reference's snapshots, are handed to the builder of `count_window` as
`resume_state`, and the resumed logics must emit exactly what the uninterrupted reference logics did."""
import json
import os
import pickle
from datetime import datetime, timedelta, timezone

import numpy as np
import pytest

from oracle.refstub import find_stateful_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

EPOCH = datetime(1970, 1, 1, tzinfo=timezone.utc)
S = 1_000_000


def _us(d):
    delta = d - EPOCH
    return (delta.days * 86400 + delta.seconds) * 1_000_000 + delta.microseconds


def _cases():
    with open(os.path.join(ROOT, "tests", "golden", "snapshot_resume_cases.json")) as f:
        return {tuple(c["params"]): c for c in json.load(f)}


def _count_builder(spec, now_us):
    """The `stateful_batch` builder of this package's `count_window` for the spec (items are `(key_str, value, ts_us)`)."""
    import bytewax_b200.operators as op
    from bytewax_b200.dataflow import Dataflow
    from bytewax_b200.operators import windowing as win
    from bytewax_b200.testing import TestingSource

    dt = lambda us: EPOCH + timedelta(microseconds=us)  # noqa: E731
    clock = win.EventClock(lambda x: dt(x[2]), wait_for_system_duration=timedelta(microseconds=spec["wait_us"]),
                           now_getter=lambda: dt(now_us))
    windower = win.SlidingWindower(length=timedelta(microseconds=spec["length_us"]),
                                   offset=timedelta(microseconds=spec["offset_us"] or spec["length_us"]), align_to=dt(spec["align_us"]))
    flow = Dataflow("g")
    win.count_window("w", op.input("in", flow, TestingSource([])), clock, windower, lambda x: x[0])
    return find_stateful_batch(flow).builder


def _drive(logics, builder, chunk):
    rows = []
    for keys, ts, vals in chunk:
        grouped = {}
        for k, tt, v in zip(keys, ts, vals):
            grouped.setdefault(str(k), []).append((str(k), v, tt))
        for ks in sorted(grouped):
            logic = logics.get(ks)
            if logic is None:
                logic = logics[ks] = builder(None)
            events, done = logic.on_batch(grouped[ks])
            rows.extend([ks, w, tag, (p if tag == "E" else None)] for w, tag, p in events if tag != "M")
            if done:
                del logics[ks]
    return rows


@pytest.mark.parametrize("red,length,offset,wait", [("count", 10, None, 0), ("sum", 10, None, 3), ("sum", 10, 5, 2), ("max", 12, 4, 1)])
def test_resume_on_the_reference_logic(red, length, offset, wait):
    from bytewax_b200 import snapshot_rows
    from bytewax_b200.operators import windowing as win

    case = _cases()[(red, length, offset, wait)]
    spec, now_us = case["spec"], case["now_us"]
    off = spec["offset_us"] or spec["length_us"]
    dt = dict(key=np.uint64, pane_id=np.int64, acc=np.uint64, count=np.uint64, open_seq=np.uint64, max_ts_us=np.int64, closed_upto=np.int64)
    cols = {n: np.array(v, dtype=dt[n]) for n, v in case["columns"].items()}
    assert len(cols["key"]) > 5
    snaps = snapshot_rows.window_snapshots(cols, reduction=red, length_us=spec["length_us"], offset_us=off, align_us=spec["align_us"],
                                           wait_us=wait * S, now_us=now_us, frozen_now_us=now_us)
    real = case["snapshots"]
    assert set(snaps) == set(real)
    for ks, want in real.items():
        mine = snaps[ks]
        # same windows, same (first-opened) order, same bounds
        assert [[w, _us(m.open_time), _us(m.close_time)] for w, m in mine.windower_state.opened.items()] == want["opened"], ks
        assert all(not m.merged_ids for m in mine.windower_state.opened.values())
        assert mine.logic_states == {w: v for w, v in want["logic_states"]}, ks
        assert _us(mine.clock_state.watermark_base) - _us(mine.clock_state.system_time_of_max_event) == want["clock_delta_us"], ks
        assert mine.queue == []
    rows = snapshot_rows.recovery_rows("flow.step", snaps, 7)
    assert all(isinstance(pickle.loads(r[3]), win._WindowSnapshot) for r in rows) and [r[1] for r in rows] == sorted(snaps)
    if red == "count":  # (for reduce / max the reference's accumulator is the ITEM; a number resumes count and numeric folds only)
        builder = _count_builder(spec, now_us)
        resumed = {ks: builder(pickle.loads(pickle.dumps(s))) for ks, s in snaps.items()}
        got = _drive(resumed, builder, case["batches"][case["cut"]:])
        got_eof = [[ks, w, tag, p if tag == "E" else None] for ks in sorted(resumed) for w, tag, p in resumed[ks].on_eof()[0] if tag != "M"]
        assert got == case["want"] and got_eof == case["want_eof"]
