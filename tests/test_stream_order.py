"""Ordering across the streams of the one-GPU streaming path.  Needs a B200: -m gpu.

The lateness verdict of activation b + 1 runs on a stream of its own, beside the fold stage of activation b, and the
fold stage's kernels are launched so that each may start while the one before it finishes.  An activation with late
rows reads the verdict chain (the running maximum event time, `Counters::gmax_ts`) and takes the late-row split;
the activations around it must still fold exactly, and the snapshot must carry the chain's final maximum."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import coracle  # noqa: E402  (checker only)

A = 1_640_995_200_000_000
WINDOW_US = 60_000_000
ROWS = 1 << 18
N_KEYS = 50_000
STRIDE = 64  # us of event time per row: an activation spans 16.8 s, as a 2^24-row C1 activation does
LATE_AT = 8  # this activation sends every 97th row 120 s into the past (two windows late)


def _batches(n_batches):
    for b in range(n_batches):
        keys, _, _ = coracle.gen_c1(b * ROWS, ROWS, N_KEYS, A)
        vals = (np.arange(b * ROWS, (b + 1) * ROWS, dtype=np.uint64) * np.uint64(STRIDE))
        if b == LATE_AT:
            late = np.arange(ROWS) % 97 == 48
            vals[late] -= np.uint64(120_000_000)
        yield keys, vals


def test_late_activation_between_clean_ones_matches_the_oracle():
    from bytewax_b200 import gpu

    ctx = gpu.Context(0)
    fold = gpu.WindowFold(ctx, "count", WINDOW_US, None, A, 0, val_dtype="u64", ts_from_value=True,
                          capacity_hint=1 << 17, max_batch_rows=ROWS, max_emit_rows=1 << 22, max_late_rows=1 << 18)
    orc = coracle.COracle("count", WINDOW_US, align_us=A)
    gmax = None
    for keys, vals in _batches(11):
        ts = (vals.astype(np.int64) + A)
        fold.ingest(keys, vals, None)
        orc.on_batch(keys, ts)
        gmax = int(ts.max()) if gmax is None else max(gmax, int(ts.max()))
    st = fold.stats()
    assert st.split_batches >= 1, "the late activation did not take the late-row split"
    snap = fold.snapshot()
    assert snap["gmax_ts_us"] == gmax
    em = fold.advance()
    em2 = fold.eof()
    orc.on_eof()
    ck, cw, ca, _, _ = orc.closed()
    got_k = np.concatenate([em.closed_key, em2.closed_key])
    got_w = np.concatenate([em.closed_window_id, em2.closed_window_id])
    got_a = np.concatenate([em.closed_acc, em2.closed_acc])
    assert len(got_k) == len(ck)
    assert got_k.tolist() == ck.tolist() and got_w.tolist() == cw.tolist() and got_a.tolist() == ca.tolist()
    lk, lw, _, lts, _ = orc.late()
    assert len(lk) > 0
    got_late = sorted(zip(np.concatenate([em.late_key, em2.late_key]).tolist(),
                          np.concatenate([em.late_window_id, em2.late_window_id]).tolist(),
                          np.concatenate([em.late_ts_us, em2.late_ts_us]).tolist()))
    assert got_late == sorted(zip(lk.tolist(), lw.tolist(), lts.tolist()))
    fold.close()
    ctx.close()
