// bw_close.cuh -- K4: watermark / close scan and compaction of closed rows.
//
// Replaces `_WindowLogic._flush_queue` -> `_handle_closed`
// (pysrc/bytewax/operators/windowing.py:1087-1108), the windower's
// `close_for` (windowing.py:645-654), the discard of an empty logic
// (windowing.py:1110-1113, src/operators.rs:796-799) and, at end of input,
// `on_eof` for every live key (src/operators.rs:862-894).
//
// Runs between fold kernels, one thread per key whose state may have
// changed shape (the dirty list), so it never races with the fold.
#pragma once
#include "bw_common.cuh"
#include "bw_fold.cuh"


__device__ __forceinline__ u64 bw_warp_reserve(unsigned long long* ctr, u32 n) {
  // opportunistic warp aggregation: one atomic per converged group
  unsigned m = __activemask();
  int lane = threadIdx.x & 31;
  // inclusive scan of n over the active lanes
  u32 pre = 0, tot = 0;
  for (int l = 0; l < 32; ++l) {
    if (m & (1u << l)) {
      u32 v = __shfl_sync(m, n, l);
      if (l < lane) pre += v;
      tot += v;
    }
  }
  int leader = __ffs(m) - 1;
  unsigned long long base = 0;
  if (lane == leader) base = atomicAdd(ctr, (unsigned long long)tot);
  base = __shfl_sync(m, base, leader);
  return base + pre;
}

__device__ __forceinline__ void bw_emit_closed(const EmitBufs& e, Counters* c, u64 key, i64 wid, u64 acc, u64 cnt,
                                               u64 seq, u64 epoch) {
  u64 i = bw_warp_reserve(&c->n_closed, 1u);
  if (i >= e.max_closed) {
    bw_raise(c, 3u);
    return;
  }
  e.c_key[i] = key;
  e.c_wid[i] = wid;
  e.c_acc[i] = acc;
  e.c_count[i] = cnt;
  e.c_seq[i] = seq;
  e.c_epoch[i] = epoch;
}

__device__ __forceinline__ u64 bw_combine(int op, u64 a, u64 b) {
  switch (op) {
    case BW_OP_ADD_ONE:
    case BW_OP_ADD_U64: return a + b;
    case BW_OP_ADD_F64:
      return (u64)__double_as_longlong(__longlong_as_double((i64)a) + __longlong_as_double((i64)b));
    case BW_OP_MIN_S64: return (u64)(((i64)a < (i64)b) ? (i64)a : (i64)b);
    case BW_OP_MIN_U64: return a < b ? a : b;
    case BW_OP_MAX_S64: return (u64)(((i64)a > (i64)b) ? (i64)a : (i64)b);
    default: return a > b ? a : b;
  }
}

// accumulator bits -> emitted bits (undo the ordered-float encoding)
__device__ __forceinline__ u64 bw_finish_acc(const FoldParams& p, u64 acc) {
  if (p.val_dtype >= 2 && (p.op == BW_OP_MIN_U64 || p.op == BW_OP_MAX_U64)) return bw_ordered_to_f64(acc);
  return acc;
}

#define BW_MAX_PANES 64  // live panes per key that K4 can re-rank (beyond: BW_ERR_CAPACITY)

struct PaneRec {
  i64 q;
  u64 acc, cnt, seq;
  u32 born;  // 6-bit creation tag, or BW_TAG_STALE
  bool dead;
};

// Tumbling windows, key without an overflow list (the shape of nearly every key of C1): at most
// the two direct panes.  Same result as the general routine below without its 64-entry
// per-thread scratch (which lives in local memory and dominated K4: 0.26 ms for 250 k keys).
__device__ __forceinline__ bool bw_close_key_simple(const Table& t, const FoldParams& p, const EmitBufs& e, u64 s, bool eof,
                                                    u64 epoch, u32 close_batch) {
  if (!(p.panes_per_offset == 1 && p.panes_per_window == 1)) return false;
  AuxSlot* ax = t.aux + s;
  if (ax->spill_head != 0) return false;
  HotSlot* hs = t.hot + s;
  P1Slot* ps = t.p1 + s;
  const i64 tag = hs->wt0;
  if (tag == BW_EMPTY_WIDTAG) return true;
  const u64 key = hs->key;
  i64 wm;
  if (eof) {
    wm = INT64_MAX;
  } else if (!p.track_wm) {
    wm = INT64_MIN;
  } else {
    wm = bw_sub_sat(hs->max_ts, p.wait_us);
    if (wm < BW_UTC_MIN_US_DEV) wm = BW_UTC_MIN_US_DEV;
  }
  const i64 q0 = bw_widtag_q(tag), q1 = bw_widtag_q1(tag);
  const u64 acc0 = hs->acc0, cnt0 = ax->cnt0, seq0 = ax->seq0;
  const u64 acc1 = ps->acc1, cnt1 = ax->cnt1, seq1 = ps->seq1;
  const bool has1 = seq1 != ~0ULL;
  const bool dead0 = wm >= bw_pane_release(q0, p);
  const bool dead1 = has1 && wm >= bw_pane_release(q1, p);
  // seq_by_id: rows of one key are ordered by (closing activation, window id); the id pass is order_rows'
  const bool ordered_seq = p.seq_by_id != 0;
  if (dead0) bw_emit_closed(e, t.ctr, key, q0, bw_finish_acc(p, acc0), cnt0, ordered_seq ? (u64)close_batch : seq0, epoch);
  if (dead1) bw_emit_closed(e, t.ctr, key, q1, bw_finish_acc(p, acc1), cnt1, ordered_seq ? (u64)close_batch : seq1, epoch);
  const bool alive0 = !dead0, alive1 = has1 && !dead1;
  bool keep1 = false;  // pane 1 keeps a survivor (as "the pane before pane 0")
  if (!alive0 && !alive1) {
    // no panes left: the reference discards the whole logic, watermark included
    hs->max_ts = INT64_MIN;
    hs->wt0 = BW_EMPTY_WIDTAG;
    hs->acc0 = p.acc_identity;
    ax->seq0 = ~0ULL;
    ax->cnt0 = 0;
    t.closed_upto[s] = INT64_MIN;
  } else {
    const bool newest_is_1 = alive1 && (!alive0 || q1 > q0);
    const bool both = alive0 && alive1;  // |q1 - q0| == 1: the older one is exactly "newest - 1"
    const i64 rq = newest_is_1 ? q1 : q0;
    hs->wt0 = bw_pack_widtag(rq, both ? 1u : 0u, BW_TAG_STALE, both, both);
    hs->acc0 = newest_is_1 ? acc1 : acc0;
    ax->cnt0 = newest_is_1 ? cnt1 : cnt0;
    ax->seq0 = newest_is_1 ? seq1 : seq0;
    if (both) {
      ps->acc1 = newest_is_1 ? acc0 : acc1;
      ps->seq1 = newest_is_1 ? seq0 : seq1;
      ax->cnt1 = newest_is_1 ? cnt0 : cnt1;
      keep1 = true;
    }
  }
  if (!keep1) {
    ps->acc1 = p.acc_identity;
    ps->seq1 = ~0ULL;
    ax->cnt1 = 0;
  }
  return true;
}

// Close everything the key's watermark allows, then put the newest pane in
// the hot slot; pane 1 becomes the pane right before it when that one is still
// alive (P1_PREV), else it is left empty for the pane right after it; the
// rest goes on the list.
__device__ void bw_close_key(const Table& t, const FoldParams& p, const EmitBufs& e, u64 s, bool eof, u64 epoch, u32 close_batch) {
  if (bw_close_key_simple(t, p, e, s, eof, epoch, close_batch)) return;
  HotSlot* hs = t.hot + s;
  P1Slot* ps = t.p1 + s;
  AuxSlot* ax = t.aux + s;
  if (hs->wt0 == BW_EMPTY_WIDTAG) return;
  const u64 key = hs->key;
  i64 wm;
  if (eof) {
    wm = INT64_MAX;
  } else if (!p.track_wm) {
    wm = INT64_MIN;
  } else {
    wm = bw_sub_sat(hs->max_ts, p.wait_us);
    if (wm < BW_UTC_MIN_US_DEV) wm = BW_UTC_MIN_US_DEV;
  }
  // gather
  PaneRec P[BW_MAX_PANES];
  u32 nodes[BW_MAX_PANES];
  int n = 0, nn = 0;
  P[n++] = PaneRec{bw_widtag_q(hs->wt0), hs->acc0, ax->cnt0, ax->seq0, (u32)hs->wt0 & 0x7Fu, false};
  if (ps->seq1 != ~0ULL) P[n++] = PaneRec{bw_widtag_q1(hs->wt0), ps->acc1, ax->cnt1, ps->seq1, BW_TAG_STALE, false};
  for (u32 nd = ax->spill_head; nd; nd = t.nodes[nd].next) {
    if (n >= BW_MAX_PANES) {
      bw_raise(t.ctr, 3u);
      return;
    }
    nodes[nn++] = nd;
    P[n++] = PaneRec{t.nodes[nd].wid, t.nodes[nd].acc, t.node_acc2[nd], t.nodes[nd].open_seq, BW_TAG_STALE, false};
  }
  const i64 a = p.panes_per_offset, b = p.panes_per_window;
  const bool ordered_seq = p.seq_by_id != 0;
  if (a == 1 && b == 1) {
    // tumbling: window id == pane id; a closed pane is emitted and dropped
    for (int i = 0; i < n; ++i)
      if (wm >= bw_pane_release(P[i].q, p)) {
        bw_emit_closed(e, t.ctr, key, P[i].q, bw_finish_acc(p, P[i].acc), P[i].cnt, ordered_seq ? (u64)close_batch : P[i].seq, epoch);
        P[i].dead = true;
      }
  } else {
    // sliding: window w = panes [w*a, w*a + b); emit each newly closable window
    // once (from its smallest live pane), then drop panes whose last window closed
    i64 c_new;
    if (eof) c_new = INT64_MAX;
    else if (wm == INT64_MIN) c_new = INT64_MIN;
    else c_new = bw_floordiv(wm - p.align_us - p.length_us, p.offset_us);
    const i64 c_prev = t.closed_upto[s];
    if (c_new > c_prev) {
      for (int i = 0; i < n; ++i) {
        i64 w_lo = bw_floordiv(P[i].q - b + a, a);  // ceil((q - b + 1) / a)
        i64 w_hi = bw_floordiv(P[i].q, a);
        if (w_lo <= c_prev) w_lo = c_prev + 1;
        if (w_hi > c_new) w_hi = c_new;
        for (i64 w = w_lo; w <= w_hi; ++w) {
          const i64 q0 = w * a, q1 = w * a + b;
          bool smallest = true;
          u64 acc = p.acc_identity, cnt = 0, seq = ~0ULL;
          for (int j = 0; j < n; ++j) {
            if (P[j].q < q0 || P[j].q >= q1) continue;
            if (P[j].q < P[i].q) {
              smallest = false;
              break;
            }
            acc = bw_combine(p.op, acc, P[j].acc);
            cnt += P[j].cnt;
            seq = P[j].seq < seq ? P[j].seq : seq;
          }
          if (smallest)
            bw_emit_closed(e, t.ctr, key, w, bw_finish_acc(p, acc), cnt, ordered_seq ? (u64)close_batch : seq, epoch);
        }
      }
      t.closed_upto[s] = c_new;
    }
    for (int i = 0; i < n; ++i)
      if (wm >= bw_pane_release(P[i].q, p)) P[i].dead = true;
  }
  // survivors, newest first (insertion sort of indices)
  int idx[BW_MAX_PANES];
  int m = 0;
  for (int i = 0; i < n; ++i) {
    if (P[i].dead) continue;
    int j = m++;
    while (j > 0 && P[idx[j - 1]].q < P[i].q) {
      idx[j] = idx[j - 1];
      --j;
    }
    idx[j] = i;
  }
  int first_listed = 1;  // survivors idx[first_listed..] go to the list
  if (m == 0) {
    // no panes left: the reference discards the whole logic, watermark included
    // (windowing.py:1110-1113 -> src/operators.rs:796-799)
    hs->max_ts = INT64_MIN;
    hs->wt0 = BW_EMPTY_WIDTAG;
    hs->acc0 = p.acc_identity;
    ax->seq0 = ~0ULL;
    ax->cnt0 = 0;
    t.closed_upto[s] = INT64_MIN;
  } else {
    const PaneRec& r0 = P[idx[0]];
    const bool prev = (m >= 2) && (P[idx[1]].q == r0.q - 1);
    // threshold (pane units) of the earliest window still covering the oldest pane,
    // not yet emitted: T = a * max(ceil((q_old - b + 1) / a), closed_upto + 1)
    i64 w_first = bw_floordiv(P[idx[m - 1]].q - b + a, a);
    if (!(a == 1 && b == 1) && t.closed_upto[s] != INT64_MIN && w_first <= t.closed_upto[s]) w_first = t.closed_upto[s] + 1;
    const i64 dq = r0.q - w_first * a;
    const u64 delta = dq < 0 ? 0 : (u64)dq;
    // K4 runs after the batch that created a pane, so its open_seq is final: mark stale
    hs->wt0 = bw_pack_widtag(r0.q, delta > BW_TAG_DELTA_MAX ? BW_TAG_DELTA_MAX : (u32)delta, BW_TAG_STALE, prev, prev, m > (prev ? 2 : 1));
    hs->acc0 = r0.acc;
    ax->cnt0 = r0.cnt;
    ax->seq0 = r0.seq;
    if (prev) {
      const PaneRec& r1 = P[idx[1]];
      ps->acc1 = r1.acc;
      ps->seq1 = r1.seq;
      ax->cnt1 = r1.cnt;
      first_listed = 2;
    }
  }
  if (first_listed == 1) {  // pane 1 empty: reserved for the pane after pane 0
    ps->acc1 = p.acc_identity;
    ps->seq1 = ~0ULL;
    ax->cnt1 = 0;
  }
  // the rest goes back on the list, reusing node storage
  u32 head = 0;
  int used = 0;
  for (int r = m - 1; r >= first_listed; --r) {
    u32 nd;
    if (used < nn) {
      nd = nodes[used++];
    } else {
      // bump-allocate only: other K4 threads are pushing onto the free stack right now,
      // so popping from it here could read a slot that is reserved but not yet written
      nd = atomicAdd(&t.ctr->pool_next, 1u);
      if (nd >= t.pool_cap) {
        bw_raise(t.ctr, 3u);
        break;
      }
    }
    const PaneRec& rr = P[idx[r]];
    PaneNode v;
    v.wid = rr.q;
    v.acc = rr.acc;
    v.open_seq = rr.seq;
    v.next = head;
    v.born = 0xFFFFFFFFu;
    t.nodes[nd] = v;
    t.node_acc2[nd] = rr.cnt;
    head = nd;
  }
  ax->spill_head = head;
  for (; used < nn; ++used) {
    int top = atomicAdd(&t.ctr->free_top, 1);
    t.free_stack[top] = nodes[used];
  }
}

// K4 for the keys on the dirty list.  The last block to finish empties the list and, given the streaming side just
// folded, its spill list and flags (every block has read the list's length before it counts itself done).
__global__ void k_close_dirty(Table t, FoldParams p, EmitBufs e, u64 epoch, u32 close_batch, StreamVerdict* sv) {
  bw_pdl_wait();
  bw_pdl_launch();
  const u32 n = t.ctr->dirty_count;
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    bw_close_key(t, p, e, t.dirty[i], false, epoch, close_batch);
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(&t.ctr->close_done, 1u) == gridDim.x - 1) {
      t.ctr->close_done = 0;
      t.ctr->dirty_count = 0;
      if (sv) {
        sv->n_spill = 0;
        sv->flags = 0;
      }
    }
  }
}
// EOF: every slot (including the BW_EMPTY_KEY alias slot at index capacity)
__global__ void k_close_all(Table t, FoldParams p, EmitBufs e, u64 epoch, u32 close_batch) {
  const u64 n = t.cap + 1;
  for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (u64)gridDim.x * blockDim.x) {
    if (s < t.cap && t.hot[s].key == BW_EMPTY_KEY) continue;
    bw_close_key(t, p, e, s, true, epoch, close_batch);
  }
}
// Notify phase (src/operators.rs:808-858): system time has moved on with no items.  A key is DUE when the close time of
// its earliest open window has been reached by the system clock (`notify_at` = min close of the opened windows,
// windowing.py:656-659, passed through `to_system_utc`'s default identity); a due key closes what its watermark
//   max_j(ts_j - now_j) - wait + now   allows (`on_notify`, windowing.py:1137-1144).  In the kernels' frame the system
// time is 0 (FoldParams::now_us).
__global__ void k_close_wake(Table t, FoldParams p, EmitBufs e, u64 epoch, u32 close_batch) {
  const u64 n = t.cap + 1;
  const i64 a = p.panes_per_offset, b = p.panes_per_window;
  for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (u64)gridDim.x * blockDim.x) {
    const HotSlot h = t.hot[s];
    if (s < t.cap && h.key == BW_EMPTY_KEY) continue;
    if (h.wt0 == BW_EMPTY_WIDTAG) continue;
    i64 q_old = bw_widtag_q(h.wt0);
    if (t.p1[s].seq1 != ~0ULL) q_old = min(q_old, bw_widtag_q1(h.wt0));
    for (u32 nd = t.aux[s].spill_head; nd; nd = t.nodes[nd].next) q_old = min(q_old, t.nodes[nd].wid);
    i64 w_first = bw_floordiv(q_old - b + a, a);  // earliest window over the oldest pane ...
    if (!(a == 1 && b == 1) && t.closed_upto[s] != INT64_MIN && w_first <= t.closed_upto[s]) w_first = t.closed_upto[s] + 1;  // ... not yet emitted
    if (p.align_us + w_first * p.offset_us + p.length_us > 0) continue;  // not due
    bw_close_key(t, p, e, s, false, epoch, close_batch);
  }
}
