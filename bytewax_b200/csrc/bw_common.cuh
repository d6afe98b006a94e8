// bw_common.cuh -- shared types, hashing and PTX helpers for libbwgpu (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

typedef uint64_t u64;
typedef int64_t i64;
typedef uint32_t u32;
typedef int32_t i32;

#define BW_MAX_WORLD 8
#define BW_SM_COUNT_FALLBACK 148

// ---------------------------------------------------------------------------
// Hash / routing.  The reference routes with an un-pinned SipHash
// (src/timely.rs:455-465); any deterministic hash conforms (SURVEY.md 8c).
// ---------------------------------------------------------------------------
__host__ __device__ __forceinline__ u64 bw_mix64(u64 z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ u64 bw_splitmix64(u64 x) {
  return bw_mix64(x + 0x9E3779B97F4A7C15ULL);
}
// Table placement hash: two multiplies and a fold (~10 instructions against mix64's ~30; the fold stage is
// instruction-issue bound).  Independent of the routing hash, so a rank's slice of the key space still
// spreads over its whole table.
__host__ __device__ __forceinline__ u64 bw_khash(u64 k) {
  k *= 0x9E3779B97F4A7C15ULL;
  k ^= k >> 32;
  k *= 0xD6E8FEB86659FD93ULL;
  return k;
}
// home slot of a table hash: high 32 bits scaled into [0, cap) (cap <= 2^31)
__host__ __device__ __forceinline__ u64 bw_slot_of_khash(u64 h, u64 cap) {
#ifdef __CUDA_ARCH__
  return (u64)__umulhi((u32)(h >> 32), (u32)cap);
#else
  return ((h >> 32) * (u64)(u32)cap) >> 32;
#endif
}
// owning rank: high 32 bits scaled into [0, world)
__host__ __device__ __forceinline__ u32 bw_route_hash(u64 h, u32 world) {
  return (u32)(((h >> 32) * (u64)world) >> 32);
}

// ---------------------------------------------------------------------------
// State layout in HBM (DESIGN.md "Data layout").
//
// One 32-byte HOT slot per key == exactly one L2 sector: everything the
// steady-state fold touches (key, running max ts, newest pane).  One 16-byte
// P1 slot per key for the adjacent pane a key is moving into / out of.  One
// 32-byte AUX slot per key for pane 0's open sequence, counts (MEAN) and the
// head of a short linked list of 32-byte nodes for any further live panes.
// ---------------------------------------------------------------------------
struct __align__(32) HotSlot {
  u64 key;      // BW_EMPTY_KEY when free
  i64 max_ts;   // max event ts seen since the key was (re)created; INT64_MIN when none
  i64 wt0;      // pane 0 (newest after K4): pane_id << 18 | has_list << 17 | has_p1 << 16 | p1_prev << 15 | delta << 8 | dirty << 7 | stale << 6 | born & 63
  u64 acc0;     // pane 0 accumulator (bits)
};
// Pane 1 is implicit: the pane right after pane 0 (the one an in-order key moves
// into inside an activation), or right before it when wt0 has P1_PREV (the one
// an out-of-order key is still finishing).  16 bytes per key keeps the working
// set of a window-boundary activation at hot + 16 B/key.  Present iff seq1 != ~0.
struct __align__(16) P1Slot {
  u64 acc1;
  u64 seq1;     // arrival sequence of the event that opened pane 1
};
struct __align__(32) AuxSlot {
  u64 seq0;         // arrival sequence (batch << 32 | index) of the event that opened pane 0
  u64 cnt0, cnt1;   // value counts of panes 0 / 1 (MEAN divisor)
  u32 spill_head;   // further panes: linked list of PaneNode, 0 == none
  u32 lock;         // structural lock for the node list
};
struct __align__(32) PaneNode {
  i64 wid;
  u64 acc;
  u64 open_seq;
  u32 next;
  u32 born;  // batch number (low 32 bits) that created the node
};

#define BW_UTC_MIN_US_DEV (-62135596800000000LL)
#define BW_EMPTY_KEY 0xFFFFFFFFFFFFFFFFULL
#define BW_EMPTY_WIDTAG INT64_MIN
#define BW_WID_SHIFT 18
#define BW_WID_LIMIT (1LL << 44)  // |pane id| must stay below this
#define BW_TAG_DIRTY 0x80LL
#define BW_TAG_BORN_MASK 0x7FLL  // bits 5:0 = creating batch & 63, bit 6 = "not fresh" (set by K4)
#define BW_TAG_STALE 0x40u
#define BW_TAG_DELTA_SHIFT 8
#define BW_TAG_DELTA_MAX 127u     // 7 bits; the maximum means "always re-examine"
#define BW_TAG_P1_PREV 0x8000LL   // pane 1 is pane0 - 1 (else pane0 + 1)
// What the key holds beyond the hot slot, so that a pass that owns the slot (bw_stream.cuh) knows
// without touching the other arrays: HAS_P1 == the P1 slot is present (seq1 != ~0), HAS_LIST ==
// the overflow list is not empty.  Set by whoever creates them, recomputed by K4.
#define BW_TAG_HAS_P1 0x10000LL
#define BW_TAG_HAS_LIST 0x20000LL

__host__ __device__ __forceinline__ i64 bw_pack_widtag(i64 q, u32 delta, u32 born, bool p1_prev = false, bool has_p1 = false,
                                                       bool has_list = false) {
  return (i64)((u64)q << BW_WID_SHIFT) | (p1_prev ? BW_TAG_P1_PREV : 0LL) | (has_p1 ? BW_TAG_HAS_P1 : 0LL) |
         (has_list ? BW_TAG_HAS_LIST : 0LL) |
         ((i64)(delta > BW_TAG_DELTA_MAX ? BW_TAG_DELTA_MAX : delta) << BW_TAG_DELTA_SHIFT) | (i64)(born & 0x7Fu);
}
__host__ __device__ __forceinline__ i64 bw_widtag_q1(i64 tag) {
  return (tag >> BW_WID_SHIFT) + ((tag & BW_TAG_P1_PREV) ? -1 : 1);
}
__host__ __device__ __forceinline__ i64 bw_widtag_q(i64 tag) { return tag >> BW_WID_SHIFT; }
__host__ __device__ __forceinline__ u32 bw_widtag_delta(i64 tag) { return (u32)((tag >> BW_TAG_DELTA_SHIFT) & 0x7F); }

// accumulator op codes (uniform per fold)
enum BwOp : int {
  BW_OP_ADD_ONE = 0,  // count
  BW_OP_ADD_U64 = 1,  // integer sum (wraps mod 2^64, same bits signed/unsigned)
  BW_OP_ADD_F64 = 2,  // float sum in binary64
  BW_OP_MIN_S64 = 3,
  BW_OP_MIN_U64 = 4,  // also floats through the order-preserving encoding
  BW_OP_MAX_S64 = 5,
  BW_OP_MAX_U64 = 6,
};

// order-preserving f64 -> u64 (for min/max by integer atomics)
__host__ __device__ __forceinline__ u64 bw_f64_to_ordered(u64 b) {
  return (b & 0x8000000000000000ULL) ? ~b : (b | 0x8000000000000000ULL);
}
__host__ __device__ __forceinline__ u64 bw_ordered_to_f64(u64 o) {
  return (o & 0x8000000000000000ULL) ? (o & 0x7FFFFFFFFFFFFFFFULL) : ~o;
}

struct FoldParams {
  i64 length_us, offset_us, align_us, wait_us;
  // pane geometry: pane = [align + q*pane_us, align + (q+1)*pane_us);
  // a window w covers panes [w*panes_per_offset, w*panes_per_offset + panes_per_window)
  i64 pane_us;
  i64 panes_per_offset;  // a
  i64 panes_per_window;  // b
  double inv_pane;       // 1.0 / pane_us
  // exact unsigned division by pane_us (round-up multiply-high): see bw_pane_of
  u64 div_magic;
  u32 div_shift;         // L - 1 where L = ceil(log2(pane_us)); pane_us == 1 handled apart
  u32 div_is_one;
  i64 div_bias;          // multiple of pane_us, makes (ts - align + bias) non-negative
  i64 div_bias_q;        // bias / pane_us
  // closability test in pane units: an event at pane q with remainder r proves every
  // window w with w * panes_per_offset <= q - close_back - (r < wait_rem) closable
  i64 close_back;        // length/pane + wait/pane
  i64 wait_rem;          // wait % pane
  int op;                // BwOp of acc
  int reduction;         // bw_reduction
  int val_dtype;
  int ts_from_value;
  int track_wm;          // 0 when wait == forever (nothing is ever late or closed before EOF)
  int ordered;
  int need_count;        // maintain acc2 (MEAN)
  int seq_by_id;         // first-opened order == ascending window id (ordered flush, or wait == 0: a key's accepted
                         // timestamps never decrease), so emission order needs no arrival sequence
  u64 acc_identity;
  // System time (windowing.py:263-302).  The watermark of a key is  max_j(ts_j - now_j) - wait + now  (now_j: system time
  // when item j arrived): everything the kernels do is invariant under shifting all times by -now, so they work in the
  // frame where the current system time is 0: every timestamp is taken as ts - now_us, align_us is
  // spec.align_us - now_us, and a slot's max_ts holds max_j(ts_j - now_j).  now_us == 0 (never set): the frozen clock.
  i64 now_us;
};

struct Table {
  HotSlot* hot;
  P1Slot* p1;
  AuxSlot* aux;
  i64* closed_upto;  // sliding windows: window ids <= this were already emitted for this key incarnation
  PaneNode* nodes;
  u64* node_acc2;
  u32* free_stack;
  u32* dirty;      // list of slot indices with possibly closable panes
  u64 cap;         // number of slots (a multiple of the segment size); slot `cap` is the BW_EMPTY_KEY alias slot
  u32 pool_cap;
  u32 seg_shift;   // log2 of the segment size
  u32 seg_mask;    // segment size - 1 (power of two): linear probing wraps inside the segment of the home slot,
                   // so a block that owns a segment owns every key that hashes into it (bw_stream.cuh)
  // device counters
  struct Counters* ctr;
};

// verdict of one activation of the streaming path (bw_stream.cuh)
struct StreamVerdict {
  u32 clean;   // no row of the activation can be late (prepass rule, bw_prepass.cuh)
  u32 flags;   // BW_SV_*
  i64 tmin, tmax;  // event-time span of the activation
  i64 ts0;     // base of the records' 32-bit relative timestamps (event time of row 0)
  u32 n_spill; // rows in this activation's spill list
  u32 pad;
  i64 gprev;   // running maximum over everything ingested before this activation
};

struct Counters {
  int free_top;          // free_stack fill
  u32 pool_next;         // bump allocator (node 0 is the null node)
  u32 dirty_count;
  u32 err;               // sticky bw_status raised by a kernel
  unsigned long long live_keys;
  unsigned long long n_closed;   // rows in the closed emit buffer
  unsigned long long n_late;     // rows in the late emit buffer
  unsigned long long gmax_ts;    // i64 bits: max event ts over everything ingested (prepass chain)
  u32 batch_clean;       // verdict of the prepass for the batch in flight
  u32 n_spill;           // rows in the partial-spill list (bw_stream.cuh)
  u32 close_done;        // blocks of k_close_dirty that are done (the last one resets; back to 0 after every launch)
  u32 pad;
};

// home slot = high part of (scrambled hash) * capacity (no power-of-two constraint on the table).
// The owning rank is taken from the HIGH bits of the same mix64(key) (bw_route_hash), so the slot
// must not be: a rank only ever sees keys from a 1/world slice of the high bits, and slicing the
// table the same way multiplies the local load factor by `world` (measured: 2.8 s per fold at 4
// GPUs).  One odd multiply moves the low bits up.
__host__ __device__ __forceinline__ u64 bw_slot_of_hash(u64 h, u64 cap) {
  h *= 0x9E3779B97F4A7C15ULL;
  if (cap >> 32) {  // never for the fold tables (capacity <= 2^31); kept exact for any caller
#ifdef __CUDA_ARCH__
    return __umul64hi(h, cap);
#else
    return (u64)(((unsigned __int128)h * cap) >> 64);
#endif
  }
  // 32 x 32 -> high 32: one IMAD.HI instead of the ~10-instruction 64-bit multiply-high
  // (profiles/r01_fold_ncu_final.md: the hash and the pane division were ~20 % of k_fold's instructions)
#ifdef __CUDA_ARCH__
  return (u64)__umulhi((u32)(h >> 32), (u32)cap);
#else
  return ((h >> 32) * (u64)(u32)cap) >> 32;
#endif
}
__device__ __forceinline__ void bw_raise(Counters* c, u32 status) { atomicCAS(&c->err, 0u, status); }

// up to BW_MAX_WORLD column segments forming one activation in arrival order
struct BatchView {
  const u64* keys[BW_MAX_WORLD];
  const void* vals[BW_MAX_WORLD];
  const i64* ts[BW_MAX_WORLD];
  const u64* d_counts;          // device: rows per segment (after an exchange)
  u64 h_counts[BW_MAX_WORLD];   // rows per segment when known on the host
  u64 max_rows;                 // host-known bound on the total
  int nseg;
  int counts_on_device;
};
__device__ __forceinline__ u64 bw_seg_count(const BatchView& bv, int j) {
  return bv.counts_on_device ? bv.d_counts[j] : bv.h_counts[j];
}

struct EmitBufs {
  u64 *c_key, *c_acc, *c_count, *c_seq, *c_epoch;
  i64* c_wid;
  u64 *l_key, *l_val, *l_seq, *l_epoch;
  i64 *l_wid, *l_ts;
  u64 max_closed, max_late;
};

// ---------------------------------------------------------------------------
// PTX helpers
// ---------------------------------------------------------------------------
// One 32-byte sector in one instruction (LDG.E.256), L2-coherent.
__device__ __forceinline__ void bw_ld_slot(const void* p, u64& a, i64& b, i64& c, u64& d) {
  asm volatile("ld.global.relaxed.gpu.v4.u64 {%0,%1,%2,%3}, [%4];"
               : "=l"(a), "=l"(b), "=l"(c), "=l"(d)
               : "l"(p)
               : "memory");
}
// Streaming loads of the input columns: read once, so keep them out of L1 and
// mark them first-to-evict in L2 -- the 126 MB L2 is reserved for the key table.
__device__ __forceinline__ u64 bw_evict_first_policy() {
  u64 pol;
  // not volatile: a pure value, so the compiler creates it once per kernel instead of once per load
  asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ u64 bw_ld_stream_u64(const u64* p) {
  u64 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(bw_evict_first_policy()));
  return v;
}
__device__ __forceinline__ u32 bw_ld_stream_u32(const u32* p) {
  u32 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(bw_evict_first_policy()));
  return v;
}
__device__ __forceinline__ void bw_red_add_u64(u64* p, u64 v) {
  asm volatile("red.global.relaxed.gpu.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void bw_red_add_f64(u64* p, double v) {
  asm volatile("red.global.relaxed.gpu.add.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ void bw_red_max_s64(i64* p, i64 v) {
  asm volatile("red.global.relaxed.gpu.max.s64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void bw_red_min_s64(i64* p, i64 v) {
  asm volatile("red.global.relaxed.gpu.min.s64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void bw_red_max_u64(u64* p, u64 v) {
  asm volatile("red.global.relaxed.gpu.max.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void bw_red_min_u64(u64* p, u64 v) {
  asm volatile("red.global.relaxed.gpu.min.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// ---------------------------------------------------------------------------
// Shared memory by 32-bit shared-window address.  Pointers into `extern __shared__` that travel
// through structs or runtime-sized layouts lose their address space and compile to GENERIC loads
// and atomics (LD.E / ATOM.E: measured 2x the instructions and none of the ATOMS throughput);
// these keep every access an LDS / STS / ATOMS.
// ---------------------------------------------------------------------------
__device__ __forceinline__ u32 bw_smem_addr(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ u64 bw_lds_u64(u32 a) {
  u64 v;
  asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(a) : "memory");
  return v;
}
// for polling a location another warp writes: ptxas may hoist a plain ld.shared out of a spin loop
__device__ __forceinline__ u64 bw_lds_u64_volatile(u32 a) {
  u64 v;
  asm volatile("ld.volatile.shared.u64 %0, [%1];" : "=l"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ u32 bw_lds_u32(u32 a) {
  u32 v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void bw_lds_2u64(u32 a, u64& x, u64& y) {
  asm volatile("ld.shared.v2.u64 {%0,%1}, [%2];" : "=l"(x), "=l"(y) : "r"(a) : "memory");
}
__device__ __forceinline__ void bw_lds_2u32(u32 a, u32& x, u32& y) {
  asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(x), "=r"(y) : "r"(a) : "memory");
}
__device__ __forceinline__ void bw_sts_u64(u32 a, u64 v) { asm volatile("st.shared.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }
__device__ __forceinline__ void bw_sts_u32(u32 a, u32 v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ u64 bw_atoms_cas_u64(u32 a, u64 cmp, u64 val) {
  u64 old;
  asm volatile("atom.shared.cas.b64 %0, [%1], %2, %3;" : "=l"(old) : "r"(a), "l"(cmp), "l"(val) : "memory");
  return old;
}
__device__ __forceinline__ u32 bw_atoms_add_u32(u32 a, u32 v) {
  u32 old;
  asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ void bw_reds_add_u32(u32 a, u32 v) { asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void bw_reds_or_u32(u32 a, u32 v) { asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void bw_reds_max_s32(u32 a, int v) { asm volatile("red.shared.max.s32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void bw_reds_min_u32(u32 a, u32 v) { asm volatile("red.shared.min.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void bw_reds_add_f64(u32 a, double v) { asm volatile("red.shared.add.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ void bw_reds_min_s64(u32 a, i64 v) { asm volatile("red.shared.min.s64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }
__device__ __forceinline__ void bw_reds_max_s64(u32 a, i64 v) { asm volatile("red.shared.max.s64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }
__device__ __forceinline__ void bw_reds_min_u64(u32 a, u64 v) { asm volatile("red.shared.min.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }
__device__ __forceinline__ void bw_reds_max_u64(u32 a, u64 v) { asm volatile("red.shared.max.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }

// Programmatic dependent launch.  A kernel launched with programmatic stream serialization may start while the
// kernel before it on the stream is still running; bw_pdl_wait blocks until that kernel has completed and its
// writes are visible (a no-op for a kernel launched without the attribute).  Every such kernel calls it in every
// block, before its first access to anything an earlier kernel writes, so that completion stays transitive along
// the stream.  bw_pdl_launch lets the next kernel's blocks be placed; it hands on nothing (the next kernel waits
// for this one's completion either way).
__device__ __forceinline__ void bw_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void bw_pdl_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// mbarrier + 1-D bulk async copy (TMA, `cp.async.bulk`): global -> shared, completion counted in
// bytes on an mbarrier.  SASS: UBLKCP / SYNCS.
__device__ __forceinline__ void bw_mbar_init(u32 bar, u32 count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void bw_mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void bw_mbar_expect_tx(u32 bar, u32 bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool bw_mbar_try_wait(u32 bar, u32 parity) {
  u32 ok;
  asm volatile(
      "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void bw_mbar_wait(u32 bar, u32 parity) {
  // a bulk copy that never lands is a bug: trap (an error the host sees) rather than hang the device
  for (u32 spin = 0; !bw_mbar_try_wait(bar, parity); ++spin)
    if (spin > (1u << 26)) __trap();
}
// size: multiple of 16 bytes; src / dst 16-byte aligned; streaming data: evict-first in L2
__device__ __forceinline__ void bw_bulk_g2s(u32 dst, const void* src, u32 bytes, u32 bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar), "l"(bw_evict_first_policy())
               : "memory");
}

__device__ __forceinline__ void bw_apply(int op, u64* acc, u64 operand) {
  switch (op) {
    case BW_OP_ADD_ONE: bw_red_add_u64(acc, 1ULL); break;
    case BW_OP_ADD_U64: bw_red_add_u64(acc, operand); break;
    case BW_OP_ADD_F64: bw_red_add_f64(acc, __longlong_as_double((i64)operand)); break;
    case BW_OP_MIN_S64: bw_red_min_s64((i64*)acc, (i64)operand); break;
    case BW_OP_MIN_U64: bw_red_min_u64(acc, operand); break;
    case BW_OP_MAX_S64: bw_red_max_s64((i64*)acc, (i64)operand); break;
    default: bw_red_max_u64(acc, operand); break;
  }
}

// floor((ts - align) / pane) for any sign, exact, no division: the dividend is
// biased non-negative and divided by the invariant pane with a precomputed
// round-up multiplier (q = (t + ((n - t) >> 1)) >> (L - 1), t = mulhi(n, m)).
__device__ __forceinline__ i64 bw_pane_of_r(i64 ts, const FoldParams& p, i64& rem) {
  const u64 n = (u64)(ts - p.align_us + p.div_bias);
  u64 qq;
  if (p.div_is_one) {
    qq = n;
  } else {
    const u64 t = __umul64hi(n, p.div_magic);
    qq = (t + ((n - t) >> 1)) >> p.div_shift;
  }
  rem = (i64)(n - qq * (u64)p.pane_us);
  return (i64)qq - p.div_bias_q;
}
// Pane of an event through a per-thread one-entry cache: streams are mostly in order, so the next
// event of a thread nearly always falls in the pane of its previous one (two compares instead of
// a 64-bit multiply-high).
struct PaneCache {
  i64 lo;  // start time of pane q; INT64_MAX == empty
  i64 q;
};
__device__ __forceinline__ i64 bw_pane_cached(i64 ts, const FoldParams& p, i64& rem, PaneCache& c) {
  const u64 d = (u64)(ts - c.lo);
  if (d < (u64)p.pane_us) {
    rem = (i64)d;
    return c.q;
  }
  const i64 q = bw_pane_of_r(ts, p, rem);
  c.lo = ts - rem;
  c.q = q;
  return q;
}
__device__ __forceinline__ i64 bw_pane_of(i64 ts, const FoldParams& p) {
  i64 r;
  return bw_pane_of_r(ts, p, r);
}
// host/device exact floor division
__host__ __device__ __forceinline__ i64 bw_floordiv(i64 a, i64 b) {
  i64 q = a / b, r = a % b;
  return (r != 0 && ((r < 0) != (b < 0))) ? q - 1 : q;
}
// Time at which pane q can be dropped == close time of the last window covering it:
// last window = floor(q / a); close = align + w*offset + length.
__device__ __forceinline__ i64 bw_pane_release(i64 q, const FoldParams& p) {
  i64 w = (p.panes_per_offset == 1) ? q : bw_floordiv(q, p.panes_per_offset);
  return p.align_us + w * p.offset_us + p.length_us;
}
// Earliest time any window covering pane q can close == close time of the first
// window covering it: first window = ceil((q - b + 1) / a).
__device__ __forceinline__ i64 bw_pane_first_close(i64 q, const FoldParams& p) {
  i64 w = (p.panes_per_window == 1 && p.panes_per_offset == 1)
              ? q
              : bw_floordiv(q - p.panes_per_window + p.panes_per_offset, p.panes_per_offset);
  return p.align_us + w * p.offset_us + p.length_us;
}
// saturating ts - wait (the reference's OverflowError branch, windowing.py:281-285)
__host__ __device__ __forceinline__ i64 bw_sub_sat(i64 ts, i64 wait) {
  if (ts < INT64_MIN + wait) return INT64_MIN;
  return ts - wait;
}
