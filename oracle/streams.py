"""Seeded input streams and fold specs shared by ``oracle/gen_golden.py`` and the tests.  TEST INFRASTRUCTURE ONLY.

Kept apart from ``gen_golden.py`` (which needs the reference's Python sources) so that a test can regenerate the exact
inputs a stored golden was produced from."""

import random

ALIGN_US = 1_640_995_200_000_000  # 2022-01-01T00:00:00Z
S = 1_000_000


def spec_(reduction="count", length_us=10_000_000, offset_us=None, wait_us=0, ordered=False, align_us=ALIGN_US):
    return dict(
        reduction=reduction, length_us=length_us, offset_us=offset_us, wait_us=wait_us, ordered=ordered, align_us=align_us
    )


def gen_random(seed, n, n_keys, span_us, jitter_us, batch_sizes, fval=False, start_us=ALIGN_US, key_base=0):
    rnd = random.Random(seed)
    keys, ts, vals = [], [], []
    for i in range(n):
        base = start_us + (i * span_us) // n
        t = base + rnd.randint(-jitter_us, jitter_us) if jitter_us else base
        keys.append(key_base + rnd.randrange(n_keys))
        ts.append(t)
        vals.append(round(rnd.uniform(-100, 100), 3) if fval else rnd.randint(-1000, 1000))
    batches, i, b = [], 0, 0
    while i < n:
        sz = batch_sizes[b % len(batch_sizes)]
        batches.append([keys[i : i + sz], ts[i : i + sz], vals[i : i + sz]])
        i += sz
        b += 1
    return batches


def random_case(seed):
    """Seeds 30..35: a spec and a 400-item stream of 7 keys with 4 s of jitter."""
    spec = spec_(["count", "sum", "min", "max"][seed % 4], 10 * S, [None, 5 * S, 3 * S][seed % 3], wait_us=(seed % 4) * S,
                 ordered=bool(seed % 2) and (seed % 4) < 2)
    return spec, gen_random(seed, 400, 7, 50 * S, 4 * S, [17, 60])


def sweep_case(seed):
    """Seeds 100..147: all five reductions, tumbling / sliding with divisible and indivisible offsets, waits from 0 to beyond
    the data span, ordered and unordered, timestamps on both sides of align_to, bursts of late items."""
    red = ["count", "sum", "min", "max", "mean"][seed % 5]
    length = [10 * S, 7 * S, 60 * S, 1 * S][seed % 4]
    offset = [None, length // 2 or None, 3 * S if 3 * S < length else None][seed % 3]
    wait = [0, S, 4 * S, 500 * S][(seed // 3) % 4]
    ordered = bool((seed // 5) % 2) and red in ("count", "sum", "mean")  # max/min_window are always unordered (windowing.py:2189, 2236)
    spec = spec_(red, length, offset, wait_us=wait, ordered=ordered)
    return spec, gen_random(seed, 300, 5, 40 * S, [0, 2 * S, 9 * S][seed % 3], [11, 50, 7], start_us=ALIGN_US - 15 * S)
