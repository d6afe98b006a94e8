"""The Python oracle (oracle/pyoracle.py) against vectors produced by the
reference's own, unmodified window logic (oracle/gen_golden.py) and against the
expected lists of the reference's tests (cases named ref_*)."""

import gzip
import json
import os

from oracle import pyoracle as po
from oracle import streams


def _load(golden_dir, name):
    with open(os.path.join(golden_dir, name)) as f:
        return json.load(f)


def _norm(rows):
    out = []
    for k, wid, tag, p in rows:
        if isinstance(p, tuple):
            p = list(p)
        out.append([k, wid, tag, p])
    return out


def test_cases_match_reference_logic(golden_dir):
    cases = _load(golden_dir, "window_fold_cases.json")
    assert len(cases) >= 20
    for name, case in cases.items():
        s = case["spec"]
        spec = po.FoldSpec(
            reduction=s["reduction"], length_us=s["length_us"], offset_us=s["offset_us"],
            align_us=s["align_us"], wait_us=s["wait_us"], ordered=s["ordered"],
        )
        acts = po.run_fold(spec, case["batches"])
        assert len(acts) == len(case["acts"]), name
        for i, (got, want) in enumerate(zip(acts, case["acts"])):
            got = _norm(got)
            if s["reduction"] in ("sum", "mean") and any(isinstance(v, float) for b in case["batches"] for v in b[2]):
                # same left-to-right f64 additions -> still exact
                pass
            assert got == want, f"{name} activation {i}"


def test_reference_test_expectations_present(golden_dir):
    cases = _load(golden_dir, "window_fold_cases.json")
    # expected lists copied from the reference's tests (file:line in `cite`)
    want = {
        "ref_count_window": [[1, 0, 2], [1, 1, 2], [2, 0, 1]],
        "ref_reduce_window": [[1, 0, 3], [1, 1, 2]],
        "ref_fold_window_tumbling": [[0, 0, 3], [0, 1, 1]],
        "ref_fold_window_sliding": [[0, -1, 2], [0, 0, 3], [0, 1, 4], [0, 2, 4], [0, 3, 1]],
        "ref_max_window": [[1, 0, 9], [1, 1, 7]],
        "ref_min_window": [[1, 0, 3], [1, 1, 2]],
    }
    for name, down in want.items():
        case = cases[name]
        s = case["spec"]
        spec = po.FoldSpec(s["reduction"], s["length_us"], s["offset_us"], s["align_us"], s["wait_us"], s["ordered"])
        rows = [r for act in po.run_fold(spec, case["batches"]) for r in act]
        assert [[k, w, p] for k, w, t, p in rows if t == "E"] == down, name
        assert case["cite"].startswith("pytests/")


def test_intersects_kats(golden_dir):
    kats = _load(golden_dir, "windower_clock_kats.json")
    for length, offset, align, t, ids in kats["intersects"]:
        assert po.SlidingWindower(length, offset, align).intersects(t) == ids


def test_intersects_reference_test_values():
    # pytests/operators/windowing/test_sliding_windower.py:6-44, 392-510 (sample)
    S = 1_000_000
    w = po.SlidingWindower(10 * S, 5 * S, 0)
    assert w.intersects(13 * S) == [1, 2]
    assert w.intersects(-3 * S) == [-2, -1]
    assert w.intersects(3 * S) == [-1, 0]
    assert w.intersects(10 * S) == [1, 2]
    t = po.SlidingWindower(10 * S, 10 * S, 0)
    assert t.intersects(13 * S) == [1]
    assert t.intersects(-3 * S) == [-1]
    assert t.intersects(0) == [0]
    assert t.intersects(10 * S) == [1]


def test_clock_kats(golden_dir):
    kats = _load(golden_dir, "windower_clock_kats.json")
    for kat in kats["clock"]:
        clock = po.EventClock(kat["wait_us"], kat["now_us"])
        for step in kat["steps"]:
            if step[0] == "adv":
                clock.now_us += step[1]
                clock.before_batch()
            else:
                _, wm = clock.on_item(step[1])
                assert wm == step[2]


def test_clock_reference_test_values():
    # pytests/operators/windowing/test_event_clock.py:11-75
    S = 1_000_000
    c = po.EventClock(5 * S, 0)
    assert c.on_notify() == po.UTC_MIN_US
    c.before_batch()
    assert c.on_item(7 * S)[1] == 2 * S
    c.now_us += 2 * S
    assert c.on_notify() == 4 * S
    c2 = po.EventClock(5 * S, 0)
    c2.before_batch()
    c2.on_item(7 * S)
    assert c2.on_item(10 * S)[1] == 5 * S
    assert c2.on_item(8 * S)[1] == 5 * S  # does not reverse


def _reference_sweep(golden_dir):
    with gzip.open(os.path.join(golden_dir, "reference_sweep_cases.json.gz")) as f:
        return json.load(f)


def _py_rows(spec, batches):
    fs = po.FoldSpec(spec["reduction"], spec["length_us"], spec["offset_us"], spec["align_us"], spec["wait_us"], spec["ordered"])
    return [[[k, w, t, list(p) if isinstance(p, tuple) else p] for k, w, t, p in a] for a in po.run_fold(fs, batches)]


def test_oracle_vs_live_reference_random(golden_dir):
    """Extra seeds against the rows the reference's unmodified `_WindowLogic` produced for them (oracle/gen_golden.py)."""
    cases = _reference_sweep(golden_dir)["random"]
    assert sorted(map(int, cases)) == list(range(30, 36))
    for seed, case in cases.items():
        spec, batches = streams.random_case(int(seed))
        assert spec == case["spec"], seed
        assert _py_rows(spec, batches) == case["acts"], seed


def test_oracles_vs_live_reference_sweep(golden_dir):
    """Wider differential sweep: 48 seeded specs (all five reductions, tumbling / sliding with divisible and indivisible
    offsets, waits from 0 to beyond the data span, ordered and unordered, timestamps on both sides of align_to, bursts of
    late items); the Python oracle and the C oracle against the rows the reference's unmodified `_WindowLogic` produced for
    them (oracle/gen_golden.py): identical per activation."""
    import numpy as np

    from oracle import coracle

    cases = _reference_sweep(golden_dir)["sweep"]
    assert sorted(map(int, cases)) == list(range(100, 148))
    for seed, case in cases.items():
        spec, b = streams.sweep_case(int(seed))
        assert spec == case["spec"], seed
        want = case["acts"]
        assert _py_rows(spec, b) == want, ("py", seed)
        red = spec["reduction"]
        if red == "mean":
            continue
        orc = coracle.COracle(red, spec["length_us"], spec["offset_us"], spec["align_us"], spec["wait_us"], spec["ordered"])
        for keys, ts, vals in b:
            orc.on_batch(np.array(keys, dtype=np.uint64), np.array(ts, dtype=np.int64), np.array(vals, dtype=np.int64))
        orc.on_eof()
        ck, cw, ca, _, cact = orc.closed()
        lk, lw, lv, _, lact = orc.late()
        want_e = [(a, k, w, p) for a, act in enumerate(want) for k, w, t, p in act if t == "E"]
        want_l = [(a, k, w, p) for a, act in enumerate(want) for k, w, t, p in act if t == "L"]
        assert list(zip(cact.tolist(), ck.tolist(), cw.tolist(), ca.tolist())) == want_e, ("c closed", seed)
        assert list(zip(lact.tolist(), lk.tolist(), lw.tolist(), lv.tolist())) == want_l, ("c late", seed)
        orc.close()


def test_keyed_oracles_match_reference_goldens(golden_dir):
    """C2 / C4 restatements against rows produced by the reference's example mapper and `_JoinLogic`."""
    g = _load(golden_dir, "keyed_cases.json")
    for case in g["zscore"]:
        got = po.run_zscore([(case["keys"], case["vals"])])[0]
        assert [[m, s, f] for m, s, f in got] == case["rows"]
    for case in g["join"]:
        items = case["items"]
        acts = po.run_join([([k], [s], [v]) for k, s, v in items], case["insert_mode"], case["emit_mode"])
        assert [list(r) for a in acts for r in a] == case["rows"], (case["insert_mode"], case["emit_mode"])


def run_timed(spec, steps):
    """`steps` of tests/golden/system_time_cases.json through the oracle engine: a moving system clock."""
    eng = po.StatefulBatchEngine(spec)
    acts = []
    for step in steps:
        if step[0] == "batch":
            _kind, now, keys, ts, vals = step
            eng.set_now(now)
            acts.append(eng.on_batch(keys, ts, vals))
        else:
            acts.append(eng.on_notify(step[1]))
    acts.append(eng.on_eof())
    return acts


def test_moving_system_clock_matches_reference_logic(golden_dir):
    """Watermark drift with the system clock (windowing.py:263-302) and the notify phase (windowing.py:1135-1180,
    src/operators.rs:808-858), against rows produced by the reference's own classes under a stepping `now_getter`."""
    cases = _load(golden_dir, "system_time_cases.json")
    assert len(cases) >= 10
    notified = 0
    for name, case in cases.items():
        s = case["spec"]
        spec = po.FoldSpec(s["reduction"], s["length_us"], s["offset_us"], s["align_us"], s["wait_us"], s["ordered"], now_us=case["steps"][0][1])
        acts = run_timed(spec, case["steps"])
        assert len(acts) == len(case["acts"]), name
        for i, (got, want) in enumerate(zip(acts, case["acts"])):
            assert _norm(got) == want, f"{name} step {i}"
            if i < len(case["steps"]) and case["steps"][i][0] == "notify":
                notified += sum(1 for r in want if r[2] == "E")
    assert notified > 20  # windows that closed because the clock moved, not because an item arrived
    # the idle key: nothing at now = align + 5 s, both keys' window 0 at align + 11 s
    c = cases["idle_key_closes_on_notify"]["acts"]
    assert c[1] == [] and [r[:3] for r in c[2] if r[2] == "E"] == [[1, 0, "E"], [2, 0, "E"]]
    # 20 idle seconds carried the watermark past the item that is only 1 s newer than the key's maximum
    assert [r for r in cases["drift_makes_item_late"]["acts"][1] if r[2] == "L"] == [[7, 0, "L", 100]]
