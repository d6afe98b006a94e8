// bw_stream.cuh -- K3, streaming form: fused lateness verdict + bucket scatter, then a
// shared-memory-resident segment fold that touches the table once per (key, activation).
//
// Same contract as k_fold (bw_fold.cuh): the per-key `on_batch` loop of
// src/operators.rs:755-806 over `_WindowLogic.on_batch` (windowing.py:1115-1133),
// followed for tumbling windows by `_flush_queue` -> `_handle_closed` / discard
// (windowing.py:1087-1113) for the keys the activation touched.
//
// The direct kernel pays one random 32-byte L2 read and two L2 reductions per EVENT
// (profiles/r01_fold_ncu_final.md: 45 G event/s ceiling).  Here every byte moves in streams:
//
//   k_scatter   one pass over the input columns (128-bit loads): lateness verdict of the
//               activation (what bw_prepass.cuh computed in its own pass) + multisplit of
//               the rows into one region per table SEGMENT (2048 consecutive home slots):
//               rank inside (tile, bucket) with a shared-memory histogram, one global
//               reservation per (tile, bucket), 16-byte records {key, ts - ts0, arrival index}.
//   k_verdict   one block: chains the per-tile (min, max, bad) triples -> clean?, event-time span.
//   k_segfold   one block per segment.  Probing wraps inside a segment (Table::seg_mask), so the
//               block owns every key that hashes into it: it keeps the segment's KEYS in shared
//               memory, claims new keys there, and accumulates per-(slot, local pane) deltas, the
//               newest timestamp and the first-open index with native 32-bit shared-memory atomics
//               (profiles/r02_ubench_smem.txt: a spread ATOMS costs about what an LDS costs).
//               One thread per touched slot then merges the deltas into the table (plain
//               loads / stores: nobody else touches the segment), closes what the key's new
//               watermark allows and re-ranks its panes -- the work of K4 for those keys.
//   k_spill     the few rows / partials that do not fit that scheme (alias key, full region,
//               a third live pane) through the general path of the direct kernel.
#pragma once
#include <type_traits>

#include "bw_close.cuh"
#include "bw_common.cuh"
#include "bw_fold.cuh"

#define BW_SEG_SHIFT_DEFAULT 11            // 2048 slots per segment == per bucket (env BW_SEG_SHIFT: 10..12)
#define BW_STREAM_MAX_NB 8192              // buckets per table (beyond: the direct kernel)

#define BW_SC_THREADS 1024
#define BW_SC_WARPS (BW_SC_THREADS / 32)
#define BW_SC_TILE 2048                    // rows per scatter tile == rows per TMA stage: one 64-row chunk per warp

#define BW_SF_THREADS 512
#define BW_SF_UNROLL 4

struct __align__(8) SpillRec {  // a row, or a pre-combined partial, for the general path
  u64 key;
  i64 ts;      // newest event time it stands for (its pane is the pane of ts)
  u64 acc;     // operand in accumulator representation (ignored for counts of weight 1 rows: acc == weight)
  u64 seq;     // batch << 32 | arrival index of its first row
  u64 weight;  // number of values it stands for
};

// what every rank tells the others about its slice of an activation (multi-GPU verdict: the slices are chained in
// source-rank order, the arrival order at every destination)
struct VerdictGather {
  i64 tmin, tmax;  // span of the rank's rows (tmin > tmax: no rows)
  u32 bad;         // some row of the slice is later than an earlier one by more than `wait`
  u32 flags;       // BW_SV_* of the rank's scatter
  u32 n_spill;     // rows the rank's scatter set aside
  u32 pad;
};
#define BW_SV_RANGE 1u   // a timestamp is further than 2^31 us from row 0: the activation takes the direct kernel
#define BW_SV_LOST 2u    // the spill list overflowed during the scatter: rows were dropped from the buckets

struct StreamSide {    // one of two alternating sets (scatter of b+1 is queued before the fold of b)
  uint4* rec;          // [nb][nlanes][lane_cap] {key lo, key hi, ts - ts0, w}: w = arrival index (folds that need first-open
                       // order), else the key's home slot inside its segment | 7-bit fingerprint << 16 (bw_rec_tag)
  void* val;           // same shape: values (only folds that need them)
  u32* cnt;            // [nb][nlanes] rows each scatter block put in its lane of each bucket (written whole by every scatter)
  SpillRec* spill;
  StreamVerdict* sv;   // device
};
struct StreamBufs {
  StreamSide side[2];
  u32 nb, nlanes, lane_cap, spill_cap;  // every scatter block owns one lane of lane_cap rows in every bucket's region
  int val_bytes;       // value bytes stored beside the records: 0 (counts), 4 or 8
  i64 *tile_min, *tile_max;  // [2 sides][tiles_cap]
  u32* tile_bad;
  i64* chunk_max;            // [2 sides][tiles_cap][32]
  u32 tiles_cap;
};

// ---------------------------------------------------------------------------
// lateness triples: (min, max, some row later than an earlier row by more than `wait`)
// ---------------------------------------------------------------------------
struct Trip {
  i64 mn, mx;
  u32 bad;
};
__device__ __forceinline__ Trip bw_trip_id() { return Trip{INT64_MAX, INT64_MIN, 0u}; }
__device__ __forceinline__ Trip bw_trip_of(i64 ts, bool valid) { return valid ? Trip{ts, ts, 0u} : bw_trip_id(); }
// a precedes b in arrival order
__device__ __forceinline__ Trip bw_trip_cat(const Trip& a, const Trip& b, i64 wait) {
  Trip r;
  r.mn = a.mn < b.mn ? a.mn : b.mn;
  r.mx = a.mx > b.mx ? a.mx : b.mx;
  r.bad = a.bad | b.bad | ((b.mn < bw_sub_sat(a.mx, wait)) ? 1u : 0u);
  return r;
}
__device__ __forceinline__ Trip bw_trip_shfl_up(const Trip& t, int d) {
  Trip r;
  r.mn = __shfl_up_sync(0xffffffffu, t.mn, d);
  r.mx = __shfl_up_sync(0xffffffffu, t.mx, d);
  r.bad = __shfl_up_sync(0xffffffffu, t.bad, d);
  return r;
}
// concatenation over the warp in lane order; the result is valid in lane 31
__device__ __forceinline__ Trip bw_trip_warp(Trip t, i64 wait) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    Trip y = bw_trip_shfl_up(t, d);
    if (lane >= d) t = bw_trip_cat(y, t, wait);
  }
  return t;
}

// 128-bit streaming loads of two consecutive 8-byte column entries (read once: no L1, evict-first in L2)
__device__ __forceinline__ void bw_ld_stream_2u64(const u64* p, u64& a, u64& b) {
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.u64 {%0,%1}, [%2], %3;"
               : "=l"(a), "=l"(b)
               : "l"(p), "l"(bw_evict_first_policy()));
}
__device__ __forceinline__ void bw_ld_stream_2u32(const u32* p, u32& a, u32& b) {
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.u32 {%0,%1}, [%2], %3;"
               : "=r"(a), "=r"(b)
               : "l"(p), "l"(bw_evict_first_policy()));
}
__device__ __forceinline__ uint4 bw_ld_stream_rec(const uint4* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "l"(p), "l"(bw_evict_first_policy()));
  return v;
}

// What a record carries for the segment fold when it does not need the arrival index: the home slot inside the
// segment and a fingerprint (bit 7 set: a zero byte is a free slot) for the byte-parallel probe.
__device__ __forceinline__ u32 bw_fp_of(u64 h) { return ((u32)(h >> 8) & 0x7Fu) | 0x80u; }
__device__ __forceinline__ u32 bw_rec_tag(u64 h, u64 slot, u32 seg_mask) { return ((u32)slot & seg_mask) | (bw_fp_of(h) << 16); }

struct ScatterArgs {
  const u64* keys;
  const void* vals;  // may be NULL (counts with a ts column)
  const i64* ts;     // NULL unless the fold has a ts column
  u64 n;
  StreamSide out;
  u32 nb, nlanes, lane_cap, spill_cap;
  i64 *tile_min, *tile_max;
  u32* tile_bad;
  i64* chunk_max;    // [tiles][32]: maximum of every warp's 64 rows (read again only when the activation has late rows: bw_late.cuh)
  u64 cap;           // table capacity (slots)
  u32 seg_shift;
  u32 batch_no;
  u32 nstage;        // TMA stages in shared memory (2 or 3)
  u32 rec_idx;       // 1: records carry the arrival index; 0: the slot / fingerprint tag
  u32 dbg;           // diagnostics only (env BW_SC_DBG): 1 skip the record stores, 2 skip the position atomics, 4 skip the verdict
  u32 world, nb_local;  // multi-GPU: bucket = owning rank * nb_local + segment of the key in the owner's table
  u32 stg_cap;       // records per bucket assembled in shared memory before they are written out (0: every record straight out)
  u32 stg_every;     // ... every this many tiles
  // second run over an activation that has late rows (bw_late.cuh): rows whose bit is set are left out
  const u32* late_bits;
  u32 ts0_set;       // take ts0 from here instead of row 0 (which may be one of the late rows, far in the past)
  i64 ts0;
};

__device__ __forceinline__ void bw_spill_push(SpillRec* list, u32* n, u32 cap, u32* flags, u32 lost_flag, Counters* ctr, u64 key,
                                              i64 ts, u64 acc, u64 seq, u64 weight) {
  const u32 i = atomicAdd(n, 1u);
  if (i >= cap) {
    if (flags) atomicOr(flags, lost_flag);
    else bw_raise(ctr, 3u);
    return;
  }
  SpillRec r;
  r.key = key;
  r.ts = ts;
  r.acc = acc;
  r.seq = seq;
  r.weight = weight;
  list[i] = r;
}

// shared-memory bytes of one TMA stage: the tile's key column, value column, ts column
__host__ __device__ __forceinline__ u32 bw_scatter_stage_bytes(int tsm, int vb_in) {
  return (u32)BW_SC_TILE * (8u + (u32)vb_in + (tsm == 0 ? 8u : 0u));
}
// barriers + stage-done counters | stages | per bucket: rows this block has put there (u32), rows of those already
// written out (u32), and stg_cap records being assembled
__host__ __device__ __forceinline__ size_t bw_scatter_smem(int tsm, int vb_in, u32 nstage, u32 nb, u32 stg_cap) {
  return 128 + (size_t)nstage * bw_scatter_stage_bytes(tsm, vb_in) + (((size_t)nb * 8 + 15) & ~(size_t)15) + (size_t)nb * stg_cap * 16;
}

// TSM: 0 = ts column, 1 = ts from the (integer) value, 2 = none (the *_final folds).
// VB_IN: bytes per entry of the value column read here (0: not read).  VB_OUT: value bytes stored beside
// the records (0 for counts).
//
// No block barrier in the tile loop.  One thread keeps `nstage` tiles of the input columns in flight with
// bulk async copies (TMA, completion counted on an mbarrier per stage); every WARP then handles its own 64
// rows of the tile that has landed, start to finish: lateness triple of the chunk, and for each row the
// bucket of its key, a position, and the 16-byte record store.  Every block owns a LANE of lane_cap rows in
// every bucket's region, so a position is just a shared-memory counter: no global atomic, nobody to wait for,
// nothing to pad (the fold reads each lane's row count).  A lane that fills up (skewed keys) overflows into
// the spill list.  The last warp to finish with a stage refills it.
//
// Writing every 16-byte record straight to its lane costs the LSU one wavefront per ROW (32 lanes, 32 lines:
// measured 0.21 ms of a 0.34 ms kernel).  So the records of a bucket are first assembled in shared memory,
// stg_cap per bucket, and every stg_every tiles the block writes what it has assembled: eight lanes per bucket,
// one 128-byte line per wavefront.  A bucket that outruns its staging rows writes those straight out.
template <int TSM, int VB_IN, int VB_OUT>
__global__ void __launch_bounds__(BW_SC_THREADS, 1) k_scatter(ScatterArgs A, FoldParams p) {
  extern __shared__ __align__(128) unsigned char sc_raw[];
  constexpr u32 T = BW_SC_TILE;
  constexpr u32 COLB_K = T * 8, COLB_V = T * VB_IN;
  constexpr u32 STAGE = COLB_K + COLB_V + (TSM == 0 ? T * 8 : 0);
  // lateness triples of the tiles in flight: [2 * nstage tiles][one per warp], combined by the tile's last warp
  __shared__ i64 c_min[8][BW_SC_WARPS], c_max[8][BW_SC_WARPS];
  __shared__ u32 c_bad[8][BW_SC_WARPS], c_done[8];
  const u32 sbase = bw_smem_addr(sc_raw);
  const u32 bars = sbase, done = sbase + 64, stage0 = sbase + 128;
  const u32 lcur = stage0 + A.nstage * STAGE;  // u32[nb]: rows this block has put in each bucket
  const u32 fbase = lcur + A.nb * 4;           // u32[nb]: ... of which already written to the lane
  const u32 stg = fbase + (((A.nb * 8 + 15) & ~15u) - A.nb * 4);  // uint4[nb][stg_cap]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const u64 ntiles = (A.n + T - 1) / T;
  u32* flags = &A.out.sv->flags;
  u32* n_spill = &A.out.sv->n_spill;
  const u32 seg_mask = (1u << A.seg_shift) - 1u;
  auto issue = [&](u64 tile, u32 stage) {  // one thread
    const u64 tbase = tile * (u64)T;
    const u32 rows = (u32)((A.n - tbase < (u64)T) ? A.n - tbase : (u64)T);
    const u32 tr = rows & ~3u;  // whole 16-byte units of every column; the (< 4) rows left are read directly
    const u32 bar = bars + 8 * stage, sk = stage0 + stage * STAGE;
    bw_mbar_expect_tx(bar, tr * (8u + (u32)VB_IN + (TSM == 0 ? 8u : 0u)));
    if (tr) {
      bw_bulk_g2s(sk, A.keys + tbase, tr * 8, bar);
      if (VB_IN) bw_bulk_g2s(sk + COLB_K, (const unsigned char*)A.vals + tbase * VB_IN, tr * VB_IN, bar);
      if (TSM == 0) bw_bulk_g2s(sk + COLB_K + COLB_V, A.ts + tbase, tr * 8, bar);
    }
  };
  if (threadIdx.x == 0) {
    for (u32 s = 0; s < A.nstage; ++s) {
      bw_mbar_init(bars + 8 * s, 1);
      bw_sts_u32(done + 4 * s, 0u);
    }
    for (int s = 0; s < 8; ++s) c_done[s] = 0u;
    bw_mbar_fence_init();
  }
  for (u32 d = threadIdx.x; d < A.nb; d += BW_SC_THREADS) {
    bw_sts_u32(lcur + 4 * d, 0u);
    bw_sts_u32(fbase + 4 * d, 0u);
  }
  const u32 my_tiles = (ntiles > blockIdx.x) ? (u32)((ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0u;
  __syncthreads();
  // Up to here the block has touched only its own shared memory, which overlaps the tail of the kernel before it
  // on the stream.  From here on it reads the input columns (which the caller may have written with a kernel of
  // its own on this stream) and writes this side's buckets, counts and verdict fields (read by earlier kernels).
  bw_pdl_wait();
  // base of the relative timestamps: event time of row 0
  i64 ts0 = p.align_us;
  if (TSM == 0) ts0 = A.ts[0] - p.now_us;
  else if (TSM == 1) ts0 = p.align_us + (i64)((const u64*)A.vals)[0];
  if (A.ts0_set) ts0 = A.ts0;
  if (threadIdx.x == 0)
    for (u32 s = 0; s < A.nstage; ++s) {
      const u64 tile = blockIdx.x + (u64)s * gridDim.x;
      if (tile < ntiles) issue(tile, s);
    }
  // (running counters: the tile loop has no division by a run-time value -- each was ~25 instructions per warp and tile)
  u32 it = 0, stage = 0, parity = 0, ring = 0, since_flush = 0;
  const u64 bucket_stride = (u64)A.nlanes * A.lane_cap;    // rows between the regions of consecutive buckets
  const u64 my_lane_off = (u64)blockIdx.x * A.lane_cap;   // this block's lane inside a bucket's region
  for (u64 tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
    const u32 sk = stage0 + stage * STAGE, sv = sk + COLB_K, st = sv + COLB_V;
    const u64 tbase = tile * (u64)T;
    const u32 rows = (u32)((A.n - tbase < (u64)T) ? A.n - tbase : (u64)T);
    const u32 tr = rows & ~3u;
    bw_mbar_wait(bars + 8 * stage, parity);
    const u32 r0 = 2u * threadIdx.x;  // this thread's two rows of the tile
    bool va = r0 < rows, vb = r0 + 1 < rows;
    const bool ina = va, inb = vb;
    u64 ka = 0, kb = 0, xa = 0, xb = 0;
    i64 ta = p.align_us, tb = p.align_us;
    if (r0 + 1 < tr) {
      bw_lds_2u64(sk + r0 * 8, ka, kb);
      if (VB_IN == 8) bw_lds_2u64(sv + r0 * 8, xa, xb);
      if (VB_IN == 4) {
        u32 x, y;
        bw_lds_2u32(sv + r0 * 4, x, y);
        xa = x;
        xb = y;
      }
      if (TSM == 0) {
        u64 a, b;
        bw_lds_2u64(st + r0 * 8, a, b);
        ta = (i64)a;
        tb = (i64)b;
      }
    } else if (ina) {  // the last (< 4) rows of the input
      ka = A.keys[tbase + r0];
      if (inb) kb = A.keys[tbase + r0 + 1];
      if (VB_IN == 8) {
        xa = ((const u64*)A.vals)[tbase + r0];
        if (inb) xb = ((const u64*)A.vals)[tbase + r0 + 1];
      }
      if (VB_IN == 4) {
        xa = ((const u32*)A.vals)[tbase + r0];
        if (inb) xb = ((const u32*)A.vals)[tbase + r0 + 1];
      }
      if (TSM == 0) {
        ta = A.ts[tbase + r0];
        if (inb) tb = A.ts[tbase + r0 + 1];
      }
    }
    if (A.late_bits && ina) {  // (tbase is a multiple of 32 and r0 is even: both bits are in one word)
      const u32 w = A.late_bits[(tbase + r0) >> 5] >> (r0 & 31u);
      va = !(w & 1u);
      vb = inb && !(w & 2u);
    }
    if (TSM == 1) {
      ta = p.align_us + (i64)xa;
      tb = p.align_us + (i64)xb;
    }
    if (TSM == 0) {  // the frame where system time is 0 (FoldParams::now_us; 0 unless the caller moves the clock)
      ta -= p.now_us;
      tb -= p.now_us;
    }
    // the columns are in registers: this warp is done with the stage; the last warp to say so refills it
    __syncwarp();
    if (lane == 0) {
      // (no fence: the loads above and this atomic go down the same shared-memory pipe in order; a fence here
      // would also wait for the thread's record stores of the previous tile to be acknowledged)
      if (bw_atoms_add_u32(done + 4 * stage, 1u) == BW_SC_WARPS - 1) {
        bw_sts_u32(done + 4 * stage, 0u);
        const u64 next = tile + (u64)A.nstage * gridDim.x;
        if (next < ntiles) issue(next, stage);
      }
    }
    // lateness triple of this warp's 64 consecutive rows; the last warp of the tile concatenates the tile's
    if (TSM != 2 && !(A.dbg & 4u)) {
      Trip ct = bw_trip_id();
      if ((u32)warp * 64u < rows) {
        const i64 nxt = __shfl_down_sync(0xffffffffu, ta, 1);
        const bool ordered = va && vb && ta <= tb && (lane == 31 || tb <= nxt);
        if (__all_sync(0xffffffffu, ordered)) {
          ct.mn = __shfl_sync(0xffffffffu, ta, 0);
          ct.mx = __shfl_sync(0xffffffffu, tb, 31);
          ct.bad = 0u;
        } else {
          ct = bw_trip_warp(bw_trip_cat(bw_trip_of(ta, va), bw_trip_of(tb, vb), p.wait_us), p.wait_us);
          ct.mn = __shfl_sync(0xffffffffu, ct.mn, 31);
          ct.mx = __shfl_sync(0xffffffffu, ct.mx, 31);
          ct.bad = __shfl_sync(0xffffffffu, ct.bad, 31);
        }
      }
      // (ring: a warp is never nstage tiles ahead of another, so 2 * nstage slots never collide)
      u32 last = 0;
      if (lane == 0) {
        ((volatile i64*)c_min[ring])[warp] = ct.mn;
        ((volatile i64*)c_max[ring])[warp] = ct.mx;
        ((volatile u32*)c_bad[ring])[warp] = ct.bad;
        last = atomicAdd(&c_done[ring], 1u) == BW_SC_WARPS - 1 ? 1u : 0u;  // same pipe, in order, after the three stores
      }
      last = __shfl_sync(0xffffffffu, last, 0);
      if (last) {
        const i64 cmx = ((volatile i64*)c_max[ring])[lane];
        A.chunk_max[tile * BW_SC_WARPS + (u64)lane] = cmx;  // (one 256-byte line per tile)
        Trip tt = bw_trip_warp(Trip{((volatile i64*)c_min[ring])[lane], cmx, ((volatile u32*)c_bad[ring])[lane]}, p.wait_us);
        if (lane == 31) {
          A.tile_min[tile] = tt.mn;
          A.tile_max[tile] = tt.mx;
          A.tile_bad[tile] = tt.bad;
          c_done[ring] = 0u;
        }
      }
    }
    // bucket of each row and its position in this block's lane there; record out
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const bool v = h ? vb : va;
      if (!v) continue;
      const u64 k = h ? kb : ka;
      const u64 x = h ? xb : xa;
      const i64 t = h ? tb : ta;
      const u64 row = tbase + r0 + h;
      const i64 d = t - ts0;
      const int rel = (int)d;
      if (d != (i64)rel || rel == INT32_MIN || rel == INT32_MAX) atomicOr(flags, BW_SV_RANGE);
      bool stored = false;
      if (k != BW_EMPTY_KEY) {  // (the alias slot lives outside every segment: general path)
        const u64 hh = bw_khash(k);
        const u64 slot = bw_slot_of_khash(hh, A.cap);
        u32 b = (u32)(slot >> A.seg_shift);
        if (A.world > 1) b += bw_route_hash(bw_mix64(k), A.world) * A.nb_local;
        const u32 pos = (A.dbg & 2u) ? (u32)(row & 7u) : bw_atoms_add_u32(lcur + 4 * b, 1u);
        const uint4 rec4 = make_uint4((u32)k, (u32)(k >> 32), (u32)rel, A.rec_idx ? (u32)row : bw_rec_tag(hh, slot, seg_mask));
        const u32 soff = pos - bw_lds_u32(fbase + 4 * b);  // rows of the bucket since the last write-out
        if (A.dbg & 1u) stored = true;
        else if (VB_OUT == 0 && soff < A.stg_cap && pos < A.lane_cap) {
          asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(stg + 16 * (b * A.stg_cap + soff)), "r"(rec4.x), "r"(rec4.y), "r"(rec4.z),
                       "r"(rec4.w)
                       : "memory");
          stored = true;
        } else if (pos < A.lane_cap) {
          const size_t at = (size_t)(b * bucket_stride + my_lane_off + pos);
          A.out.rec[at] = rec4;
          if (VB_OUT == 8) ((u64*)A.out.val)[at] = x;
          else if (VB_OUT == 4) ((u32*)A.out.val)[at] = (u32)x;
          stored = true;
        }
      }
      if (!stored) {
        u64 operand = 1ULL;
        if (VB_IN) bw_operand(p, x, operand);
        bw_spill_push(A.out.spill, n_spill, A.spill_cap, flags, BW_SV_LOST, nullptr, k, t, (p.op == BW_OP_ADD_ONE) ? 1ULL : operand,
                      ((u64)A.batch_no << 32) | row, 1ULL);
      }
    }
    // every stg_every tiles (and after the last): write out what the buckets have assembled
    if (++stage == A.nstage) {
      stage = 0;
      parity ^= 1u;
    }
    if (++ring == 2u * A.nstage) ring = 0;
    if (VB_OUT == 0 && A.stg_cap && (++since_flush == A.stg_every || it + 1 == my_tiles)) {
      since_flush = 0;
      __syncthreads();
      for (u32 bb = (u32)warp * 4; bb < A.nb; bb += BW_SC_WARPS * 4) {  // uniform trip count per warp: four buckets at a time
        const u32 b = bb + ((u32)lane >> 3);
        u32 c = 0;
        if (b < A.nb) {
          const u32 fb = bw_lds_u32(fbase + 4 * b);
          c = bw_lds_u32(lcur + 4 * b);
          const u32 nrec = min(c - fb, A.stg_cap);
          for (u32 r = (u32)lane & 7u; r < nrec && fb + r < A.lane_cap; r += 8) {
            uint4 v;
            asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(stg + 16 * (b * A.stg_cap + r)) : "memory");
            A.out.rec[(size_t)(b * bucket_stride + my_lane_off + fb + r)] = v;
          }
        }
        __syncwarp();
        if (b < A.nb && ((u32)lane & 7u) == 0) bw_sts_u32(fbase + 4 * b, c);
      }
      __syncthreads();
    }
  }
  // rows in each of this block's lanes
  __syncthreads();
  for (u32 b = threadIdx.x; b < A.nb; b += BW_SC_THREADS) {
    const u32 c = bw_lds_u32(lcur + 4 * b);
    A.out.cnt[(size_t)b * A.nlanes + blockIdx.x] = c < A.lane_cap ? c : A.lane_cap;
  }
}

// One block: chain the tiles (and the earlier activations through gmax_ts) as k_prepass_scan does
// for its ranges; publish the verdict, the span and the base timestamp.
__global__ void __launch_bounds__(1024)
k_verdict(const i64* tile_min, const i64* tile_max, const u32* tile_bad, u32 ntiles, FoldParams p, Counters* ctr, StreamVerdict* sv,
          const i64* ts_col, const u64* val_col, VerdictGather* vg) {
  __shared__ i64 s_mn[32], s_mx[32];
  __shared__ u32 s_bad[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // warp w takes a contiguous run of tiles, 32 at a time with coalesced loads: ordered concatenation inside the 32
  // (lane order == arrival order), then across the run
  const u32 nwarps = blockDim.x >> 5;
  const u32 per = ((ntiles + nwarps - 1) / nwarps + 31) & ~31u;
  const u32 lo = (u32)warp * per, hi = (lo + per < ntiles) ? lo + per : ntiles;
  Trip tt = bw_trip_id();
  for (u32 base = lo; base < hi; base += 32) {
    const u32 r = base + (u32)lane;
    Trip x = (r < hi) ? Trip{tile_min[r], tile_max[r], tile_bad[r]} : bw_trip_id();
    x = bw_trip_warp(x, p.wait_us);
    x.mn = __shfl_sync(0xffffffffu, x.mn, 31);
    x.mx = __shfl_sync(0xffffffffu, x.mx, 31);
    x.bad = __shfl_sync(0xffffffffu, x.bad, 31);
    tt = bw_trip_cat(tt, x, p.wait_us);
  }
  if (lane == 31) {
    s_mn[warp] = tt.mn;
    s_mx[warp] = tt.mx;
    s_bad[warp] = tt.bad;
  }
  __syncthreads();
  if (warp == 0) {
    Trip act = bw_trip_warp(Trip{s_mn[lane], s_mx[lane], s_bad[lane]}, p.wait_us);
    if (lane == 31) {
      sv->tmin = act.mn;
      sv->tmax = act.mx;
      sv->ts0 = (ntiles == 0) ? p.align_us : (ts_col ? ts_col[0] - p.now_us : p.align_us + (i64)val_col[0]);
      if (vg) {
        // multi-GPU: this rank's slice only; the slices are chained on the host once gathered
        vg->tmin = act.mn;
        vg->tmax = act.mx;
        vg->bad = act.bad;
        vg->flags = sv->flags;
        vg->n_spill = sv->n_spill;
        sv->clean = 0u;
      } else {
        const i64 gprev = (i64)ctr->gmax_ts;
        sv->gprev = gprev;
        // everything ingested before this activation: only its maximum matters
        const Trip all = bw_trip_cat(Trip{INT64_MAX, gprev, 0u}, act, p.wait_us);
        ctr->gmax_ts = (unsigned long long)all.mx;
        const u32 clean = (!p.track_wm || !all.bad) ? 1u : 0u;
        ctr->batch_clean = clean;
        sv->clean = clean;
      }
    }
  }
}
// the *_final folds have no event time: everything is window 0 at align_to
__global__ void k_verdict_none(FoldParams p, Counters* ctr, StreamVerdict* sv, VerdictGather* vg, u64 rows) {
  ctr->batch_clean = 1u;
  sv->clean = 1u;
  sv->tmin = p.align_us;
  sv->tmax = p.align_us;
  sv->ts0 = p.align_us;
  if (vg) {
    vg->tmin = rows ? p.align_us : INT64_MAX;
    vg->tmax = rows ? p.align_us : INT64_MIN;
    vg->bad = 0u;
    vg->flags = sv->flags;
    vg->n_spill = sv->n_spill;
  }
}
__global__ void k_set_gmax(Counters* ctr, i64 gmax) { ctr->gmax_ts = (unsigned long long)gmax; }

// ---------------------------------------------------------------------------
// segment fold
// ---------------------------------------------------------------------------
// A key's delta over one pane of one activation, as one rank hands it to the rank that owns the key (multi-GPU:
// every rank first combines its own slice, then the partials -- not the rows -- cross NVLink: SURVEY 8e, the
// precedent is `reduce_final`'s pre-reducer, operators/__init__.py:2836-2847).
struct __align__(16) Partial {
  u64 key;
  u64 acc;   // delta in accumulator representation (a count for counts)
  i64 ts;    // a timestamp of the pane; the key's newest one when this is its newest pane
  u32 seq;   // arrival index (at the source) of the first row it stands for
  u32 cnt;   // rows it stands for
};

struct SegArgs {
  StreamSide in;
  u32 nb, nlanes, lane_cap, spill_cap;
  // multi-GPU (MODE 1 / 2 of k_segfold)
  u32 world, rank, nb_local, part_cap;
  Partial* pout[BW_MAX_WORLD];   // MODE 1: rank d's receive region for THIS source: [nb_local][part_cap] (peer memory over NVLink)
  u32* pcnt_out[BW_MAX_WORLD];   // MODE 1: ... and its counts [nb_local]
  const Partial* pin;            // MODE 2: this rank's receive region [world][nb_local][part_cap]
  const u32* pcnt_in;            // MODE 2: [world][nb_local]
  u32 nlanes_used;  // blocks of the scatter that filled this side
  int val_bytes;
  u32 seg_shift;
  i64 ts0;      // base of the records' relative timestamps
  i64 q_lo;     // pane of the activation's earliest timestamp
  u32 npass;    // the activation spans panes [q_lo, q_lo + 2 * npass): folded two panes at a time, closing in
                // between (what the direct path's sub-ranges do; exact because the activation is clean)
  u32 batch_no;
  u64 epoch;
};

// One accumulator op on a shared-memory delta (32-bit shared-window address)
template <int OP>
struct SegOp {
  static constexpr bool narrow = (OP == BW_OP_ADD_ONE);  // < 2^32 rows per activation: 32-bit deltas
  static constexpr u32 DTB = narrow ? 4u : 8u;
  __device__ __forceinline__ static void apply(u32 a, u64 operand) {
    if (OP == BW_OP_ADD_ONE) {
      bw_reds_add_u32(a, 1u);
    } else if (OP == BW_OP_ADD_U64) {
      // exact 64-bit sum from two native 32-bit atomics: each add carries its own overflow up
      const u32 lo = (u32)operand, hi = (u32)(operand >> 32);
      const u32 old = bw_atoms_add_u32(a, lo);
      const u32 carry = ((u32)(old + lo) < old) ? 1u : 0u;
      if (hi | carry) bw_reds_add_u32(a + 4, hi + carry);
    } else if (OP == BW_OP_ADD_F64) {
      bw_reds_add_f64(a, __longlong_as_double((i64)operand));
    } else if (OP == BW_OP_MIN_S64) {
      bw_reds_min_s64(a, (i64)operand);
    } else if (OP == BW_OP_MIN_U64) {
      bw_reds_min_u64(a, operand);
    } else if (OP == BW_OP_MAX_S64) {
      bw_reds_max_s64(a, (i64)operand);
    } else {
      bw_reds_max_u64(a, operand);
    }
  }
  // a pre-combined delta (a partial from another rank)
  __device__ __forceinline__ static void merge(u32 a, u64 d) {
    if (OP == BW_OP_ADD_ONE) bw_reds_add_u32(a, (u32)d);
    else apply(a, d);
  }
  __device__ __forceinline__ static u64 load(u32 a) { return narrow ? (u64)bw_lds_u32(a) : bw_lds_u64(a); }
  __device__ __forceinline__ static void store(u32 a, u64 v) {
    if (narrow) bw_sts_u32(a, (u32)v);
    else bw_sts_u64(a, v);
  }
};

// shared-memory layout of one segment of S slots:
//   keys u64[S] | fingerprints u8[S] | delta pane 0, pane 1 (u32 or u64)[S] | newest relative ts i32[S] | touched bits u32[S/16]
//   | first arrival index u32[S] x 2 (SEQ) | value counts u32[S] x 2 (CNT)
__host__ __device__ __forceinline__ size_t bw_segfold_smem(u32 S, int op, bool seq, bool cnt) {
  size_t b = (size_t)S * 8 + (size_t)S + (size_t)S * 4;
  b += 2 * (size_t)S * (op == BW_OP_ADD_ONE ? 4 : 8);
  if (op != BW_OP_ADD_ONE) b += (size_t)S / 16 * 4;
  if (seq) b += 2 * (size_t)S * 4;
  if (cnt) b += 2 * (size_t)S * 4;
  return b;
}

// pane record used while one thread re-ranks a key
struct MPane {
  i64 q;
  u64 acc, cnt, seq;
};

// The fold kernel proper.  C = FoldCfg<op, -1, cnt> (compile-time op), SEQ: keep first-open indices
// (folds whose emission order is not simply ascending window id).
// MODE 0: one GPU -- rows of the bucket's lanes into the table.
// MODE 1: multi-GPU, at the source -- rows of a (destination rank, bucket) combined from an empty segment; what the
//         merge phase would put in the table goes to the destination's receive region as partials (stores over NVLink).
// MODE 2: multi-GPU, at the destination -- the partials every source left for this bucket into the table.
template <class C, bool SEQ, int MODE>
__global__ void __launch_bounds__(BW_SF_THREADS)
k_segfold(SegArgs A, Table t, FoldParams p, EmitBufs e) {
  constexpr int OP = C::kOp;
  constexpr bool CNT = C::kCnt != 0;
  const bool WM = p.track_wm != 0;
  typedef SegOp<OP> SO;
  constexpr u32 DTB = SO::DTB;
  extern __shared__ __align__(16) unsigned char sf_raw[];
  __shared__ DirtySink sink;
  __shared__ u32 sink_buf[512];
  __shared__ u32 part_n;  // MODE 1: partials written for the bucket
  const u32 S = 1u << A.seg_shift, smask = S - 1;
  const u32 a_key = bw_smem_addr(sf_raw);
  const u32 a_fp = a_key + S * 8;  // one byte per slot: 0 == free, else 0x80 | 7 hash bits of the key in the slot
  const u32 a_d0 = a_fp + S, a_d1 = a_d0 + S * DTB;
  const u32 a_mts = a_d1 + S * DTB;
  const u32 a_tm = a_mts + S * 4;
  const u32 a_sq0 = a_tm + (SO::narrow ? 0u : S / 16 * 4), a_sq1 = a_sq0 + (SEQ ? S * 4 : 0u);
  const u32 a_cn0 = a_sq1 + (SEQ ? S * 4 : 0u), a_cn1 = a_cn0 + (CNT ? S * 4 : 0u);
  if (threadIdx.x == 0) {
    sink.n_dirty = 0;
    sink.n_new_keys = 0;
    sink.cap = 512;
    sink.buf = sink_buf;
  }
  bw_pdl_wait();
  bw_pdl_launch();
  const u64 ident = (OP <= BW_OP_ADD_F64) ? 0ULL : p.acc_identity;
  const bool tumbling = p.panes_per_offset == 1 && p.panes_per_window == 1;
  for (u32 b = blockIdx.x; b < A.nb; b += gridDim.x) {
    const u64 slot_base = (u64)b << A.seg_shift;
    __syncthreads();  // the previous segment's merge is done with shared memory
    if (MODE == 1 && threadIdx.x == 0) part_n = 0u;
    for (u32 i = threadIdx.x; i < S / 4; i += BW_SF_THREADS) {  // four slots per thread: one 32-bit word of fingerprints
      u32 w = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const u64 key = (MODE == 1) ? BW_EMPTY_KEY : t.hot[slot_base + 4 * i + k].key;
        bw_sts_u64(a_key + 8 * (4 * i + k), key);
        if (key != BW_EMPTY_KEY) w |= bw_fp_of(bw_khash(key)) << (8 * k);
      }
      bw_sts_u32(a_fp + 4 * i, w);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (u32 pass = 0; pass < A.npass; ++pass) {
      // relative start of the two local panes of this pass, and of the next pass
      const i64 q_pass = A.q_lo + 2 * (i64)pass;
      const i64 pb0 = p.align_us + q_pass * p.pane_us - A.ts0, pb1 = pb0 + p.pane_us, pb2 = pb1 + p.pane_us;
      // the same bounds clamped into the records' 32-bit range: the per-event tests are 32-bit compares
      const int lo32 = (A.npass > 1 && pb0 > (i64)INT32_MIN) ? (pb0 > (i64)INT32_MAX ? INT32_MAX : (int)pb0) : INT32_MIN;
      const int mid32 = pb1 > (i64)INT32_MAX ? INT32_MAX : (pb1 < (i64)INT32_MIN ? INT32_MIN : (int)pb1);
      const int hi32 = (A.npass > 1 && pb2 < (i64)INT32_MAX) ? (pb2 < (i64)INT32_MIN ? INT32_MIN : (int)pb2) : INT32_MAX;
      __syncthreads();
      for (u32 i = threadIdx.x; i < S; i += BW_SF_THREADS) {
        SO::store(a_d0 + DTB * i, ident);
        SO::store(a_d1 + DTB * i, ident);
        bw_sts_u32(a_mts + 4 * i, (u32)INT32_MIN);
        if (!SO::narrow && i < S / 16) bw_sts_u32(a_tm + 4 * i, 0u);
        if (SEQ) {
          bw_sts_u32(a_sq0 + 4 * i, 0xFFFFFFFFu);
          bw_sts_u32(a_sq1 + 4 * i, 0xFFFFFFFFu);
        }
        if (CNT) {
          bw_sts_u32(a_cn0 + 4 * i, 0u);
          bw_sts_u32(a_cn1 + 4 * i, 0u);
        }
      }
      __syncthreads();
      // One event (a row, or another rank's partial): find or claim the key's slot, update the slot's deltas.
      // Linear probing from the home slot, wrapping inside the segment, is the table's placement rule
      // (bw_find_slot); here it is walked 16 slots at a time: one LDS.128 brings the fingerprint bytes of an aligned
      // window, byte-parallel compares give the candidate and the free positions, and only a candidate's 8-byte key
      // is read.  The loop is warp-uniform (every lane stays until the last one has its slot) so that the
      // accumulator updates issue once per warp.  Call with all 32 lanes.
      auto fold_one = [&](bool valid, u64 key, int rel, u32 ls, u32 fp, u64 operand, u32 seqv, u32 cntv) {
        const u32 fp4 = fp * 0x01010101u;
        // the window starts at the 8-aligned slot at or below the home slot: at least nine positions lie ahead of
        // the home slot, so a second window is rare (a key is seldom displaced that far at load 0.5)
        u32 wb = ls & ~7u;                 // window base
        u32 ahead = 0xFFFFu << (ls & 7u);  // positions of the window at or after the home slot
        bool searching = valid, found = false;
        u32 tries = 0;
        while (__any_sync(0xffffffffu, searching)) {
          if (searching) {
            u32 w0, w1, w2, w3;
            bw_lds_2u32(a_fp + wb, w0, w1);
            bw_lds_2u32(a_fp + ((wb + 8) & smask), w2, w3);
            // free positions: bytes with bit 7 clear; matches: zero bytes of (word ^ fingerprint x 4), exact
            auto zmask = [](u32 x) { return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x | 0x7F7F7F7Fu); };  // 0x80 per zero byte
            auto pack4 = [](u32 m80) { return (m80 * 0x00204081u) >> 28; };                                // -> 4 bits
            const u32 freem = (pack4(~w0 & 0x80808080u) | (pack4(~w1 & 0x80808080u) << 4) | (pack4(~w2 & 0x80808080u) << 8) |
                               (pack4(~w3 & 0x80808080u) << 12)) & ahead;
            u32 cand = (pack4(zmask(w0 ^ fp4)) | (pack4(zmask(w1 ^ fp4)) << 4) | (pack4(zmask(w2 ^ fp4)) << 8) |
                        (pack4(zmask(w3 ^ fp4)) << 12)) & ahead;
            // the key, if present, sits before the first free position of its probe sequence
            if (freem) cand &= (freem & (0u - freem)) - 1u;
            bool hit = false;
            while (cand) {
              const u32 pos = __ffs(cand) - 1;
              cand &= cand - 1;
              if (bw_lds_u64(a_key + 8 * ((wb + pos) & smask)) == key) {
                ls = (wb + pos) & smask;
                hit = true;
                break;
              }
            }
            if (!hit && freem) {
              const u32 pos = (wb + __ffs(freem) - 1) & smask;
              const u64 old = bw_atoms_cas_u64(a_key + 8 * pos, BW_EMPTY_KEY, key);
              if (old == BW_EMPTY_KEY) {
                asm volatile("st.shared.u8 [%0], %1;" ::"r"(a_fp + pos), "r"(fp) : "memory");
                ls = pos;
                hit = true;
              } else if (old == key) {
                ls = pos;
                hit = true;
              }
              // else: another key won the slot (its fingerprint may not be visible yet): look at the window again
            } else if (!hit) {
              wb = (wb + 16) & smask;
              ahead = 0xFFFFu;
              tries += 16;
            }
            if (hit) {
              found = true;
              searching = false;
            } else if (tries > S + 16) {
              searching = false;
            }
          }
        }
        if (valid && !found) bw_raise(t.ctr, 3u);  // segment full: capacity_hint too small
        if (found) {
          const u32 j = (rel >= mid32) ? 1u : 0u;
          if (MODE == 2) SO::merge((j ? a_d1 : a_d0) + DTB * ls, operand);
          else SO::apply((j ? a_d1 : a_d0) + DTB * ls, operand);
          if (!SO::narrow) bw_reds_or_u32(a_tm + 4 * (ls >> 4), 1u << (2 * (ls & 15) + j));
          bw_reds_max_s32(a_mts + 4 * ls, rel);
          if (SEQ) bw_reds_min_u32((j ? a_sq1 : a_sq0) + 4 * ls, seqv);
          if (CNT) bw_reds_add_u32((j ? a_cn1 : a_cn0) + 4 * ls, cntv);
        }
      };
      if (MODE != 2) {
        // ---- rows of the bucket: its lanes (one per scatter block) are dealt to the warps round-robin ----
        for (u32 ln = (u32)warp; ln < A.nlanes_used; ln += BW_SF_THREADS / 32) {
          const size_t lane_base = ((size_t)b * A.nlanes + ln) * A.lane_cap;
          const u32 n = min(A.in.cnt[(size_t)b * A.nlanes + ln], A.lane_cap);
          const uint4* rec = A.in.rec + lane_base;
          for (u32 base = 0; base < n; base += 32 * BW_SF_UNROLL) {
            uint4 r[BW_SF_UNROLL];
            u64 v[BW_SF_UNROLL];
#pragma unroll
            for (int u = 0; u < BW_SF_UNROLL; ++u) {
              const u32 i = base + (u32)u * 32 + (u32)lane;
              r[u] = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0, 0);  // no record: the empty key
              v[u] = 0;
              if (i < n) {
                r[u] = bw_ld_stream_rec(rec + i);
                if (OP != BW_OP_ADD_ONE) {
                  const size_t at = lane_base + i;
                  v[u] = (A.val_bytes == 8) ? bw_ld_stream_u64((const u64*)A.in.val + at) : (u64)bw_ld_stream_u32((const u32*)A.in.val + at);
                }
              }
            }
#pragma unroll
            for (int u = 0; u < BW_SF_UNROLL; ++u) {
              const u64 key = (u64)r[u].x | ((u64)r[u].y << 32);
              const int rel = (int)r[u].z;
              const bool valid = key != BW_EMPTY_KEY && rel >= lo32 && rel < hi32;  // a record, and of this pass
              u32 ls, fp;
              if (SEQ) {  // the 4th word is the arrival index: hash here
                const u64 hh = bw_khash(key);
                ls = (u32)bw_slot_of_khash(hh, t.cap) & smask;
                fp = bw_fp_of(hh);
              } else {
                ls = r[u].w & smask;
                fp = (r[u].w >> 16) & 0xFFu;
              }
              u64 operand = 0;
              if (OP != BW_OP_ADD_ONE) bw_operand(p, v[u], operand);
              fold_one(valid, key, rel, ls, fp, operand, r[u].w, 1u);
            }
          }
        }
      } else {
        // ---- partials every source rank left for this bucket, in source order ----
        for (u32 src = 0; src < A.world; ++src) {
          const u32 n = min(A.pcnt_in[(size_t)src * A.nb_local + b], A.part_cap);
          const Partial* pp = A.pin + ((size_t)src * A.nb_local + b) * A.part_cap;
          for (u32 base = (u32)warp * 32; base < n; base += BW_SF_THREADS) {
            const u32 i = base + (u32)lane;
            Partial pr;
            pr.key = BW_EMPTY_KEY;
            pr.acc = 0;
            pr.ts = 0;
            pr.seq = 0;
            pr.cnt = 0;
            if (i < n) pr = pp[i];
            const i64 d = pr.ts - A.ts0;
            const int rel = (int)d;  // (the host checked the activation's span fits 32 bits)
            const bool valid = i < n && d == (i64)rel && rel >= lo32 && rel < hi32;
            const u64 hh = bw_khash(pr.key);
            fold_one(valid, pr.key, rel, (u32)bw_slot_of_khash(hh, t.cap) & smask, bw_fp_of(hh), pr.acc, (src << 28) | (pr.seq & 0x0FFFFFFFu),
                     pr.cnt);
          }
        }
      }
      if (MODE == 1) {
        // ---- partials out: what the merge would put in the table goes to the owning rank ----
        __syncthreads();
        const u32 d_rank = b / A.nb_local, bl = b % A.nb_local;
        Partial* out = A.pout[d_rank] + (size_t)bl * A.part_cap;
        for (u32 ls = threadIdx.x; ls < S; ls += BW_SF_THREADS) {
          const int m = (int)bw_lds_u32(a_mts + 4 * ls);
          if (m == INT32_MIN) continue;
          const u64 key = bw_lds_u64(a_key + 8 * ls);
          const u64 dvv[2] = {SO::load(a_d0 + DTB * ls), SO::load(a_d1 + DTB * ls)};
          bool tch[2];
          if (SO::narrow) {
            tch[0] = dvv[0] != 0;
            tch[1] = dvv[1] != 0;
          } else {
            const u32 bits = bw_lds_u32(a_tm + 4 * (ls >> 4)) >> (2 * (ls & 15));
            tch[0] = bits & 1u;
            tch[1] = bits & 2u;
          }
          const i64 ts_new = A.ts0 + (i64)m;
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            if (!tch[j]) continue;
            const u32 pos = atomicAdd(&part_n, 1u);
            if (pos >= A.part_cap) continue;  // (raised below)
            Partial pr;
            pr.key = key;
            pr.acc = dvv[j];
            // the key's newest timestamp goes with its newest pane; the older pane just needs a timestamp inside it
            pr.ts = (j == 0 && tch[1]) ? A.ts0 + pb1 - 1 : ts_new;
            pr.seq = SEQ ? bw_lds_u32((j ? a_sq1 : a_sq0) + 4 * ls) : 0u;
            pr.cnt = CNT ? bw_lds_u32((j ? a_cn1 : a_cn0) + 4 * ls) : 0u;
            out[pos] = pr;
          }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
          if (part_n > A.part_cap) bw_raise(t.ctr, 3u);
          A.pcnt_out[d_rank][bl] = min(part_n, A.part_cap);
        }
        continue;  // (npass == 1: next bucket)
      }
      __syncthreads();
      // ---- merge: one thread per touched slot; the block owns the segment ----
      for (u32 ls = threadIdx.x; ls < S; ls += BW_SF_THREADS) {
        const int m = (int)bw_lds_u32(a_mts + 4 * ls);
        if (m == INT32_MIN) continue;
        const u64 s = slot_base + ls;
        const u64 key = bw_lds_u64(a_key + 8 * ls);
        HotSlot h = t.hot[s];
        if (h.key == BW_EMPTY_KEY) {
          atomicAdd(&sink.n_new_keys, 1u);
          h.key = key;
        }
        const u64 dv[2] = {SO::load(a_d0 + DTB * ls), SO::load(a_d1 + DTB * ls)};
        bool touched[2];
        if (SO::narrow) {
          touched[0] = dv[0] != 0;
          touched[1] = dv[1] != 0;
        } else {
          const u32 bits = bw_lds_u32(a_tm + 4 * (ls >> 4)) >> (2 * (ls & 15));
          touched[0] = bits & 1u;
          touched[1] = bits & 2u;
        }
        u64 dcn[2] = {0, 0}, dsq[2] = {0, 0};
        if (CNT) {
          dcn[0] = bw_lds_u32(a_cn0 + 4 * ls);
          dcn[1] = bw_lds_u32(a_cn1 + 4 * ls);
        }
        const u64 seq_hi = (u64)A.batch_no << 32;
        if (SEQ) {
          dsq[0] = seq_hi | bw_lds_u32(a_sq0 + 4 * ls);
          dsq[1] = seq_hi | bw_lds_u32(a_sq1 + 4 * ls);
        }
        const i64 ts_new = A.ts0 + (i64)m;  // newest event of the key in this pass
        if (WM && ts_new > h.max_ts) h.max_ts = ts_new;
        const i64 tag_in = h.wt0;
        if (tumbling && !SEQ && !CNT && touched[0] != touched[1] && tag_in != BW_EMPTY_WIDTAG &&
            !(tag_in & (BW_TAG_HAS_P1 | BW_TAG_HAS_LIST | BW_TAG_DIRTY))) {
          // The steady state of an in-order stream: the key's only pane took more values and stays open.
          const int j = touched[1] ? 1 : 0;
          const i64 q = q_pass + j;
          if (bw_widtag_q(tag_in) == q) {
            bool open = true;
            if (WM) {
              i64 wm = bw_sub_sat(h.max_ts, p.wait_us);
              if (wm < BW_UTC_MIN_US_DEV) wm = BW_UTC_MIN_US_DEV;
              open = wm < p.align_us + (q + 1) * p.length_us;
            }
            if (open) {
              h.acc0 = bw_combine(OP, h.acc0, dv[j]);
              t.hot[s] = h;
              continue;
            }
          }
        }
        const bool had_p1 = (tag_in & BW_TAG_HAS_P1) != 0;
        bool done = false;
        if (tumbling && !(tag_in & (BW_TAG_HAS_LIST | BW_TAG_DIRTY))) {
          // Every pane of the key is at hand: close what the new watermark allows and re-rank,
          // exactly what K4 (bw_close_key_simple) would do for it after the activation.  (A key
          // already on the dirty list stays K4's: its entry there must meet the DIRTY bit again.)
          MPane P[4];
          int np = 0;
          AuxSlot ax;
          const bool need_aux = (SEQ || CNT) && tag_in != BW_EMPTY_WIDTAG;
          if (need_aux) ax = t.aux[s];
          if (tag_in != BW_EMPTY_WIDTAG) {
            P[np++] = MPane{bw_widtag_q(tag_in), h.acc0, CNT ? ax.cnt0 : 0ULL, SEQ ? ax.seq0 : 0ULL};
            if (had_p1) {
              const P1Slot ps = t.p1[s];
              P[np++] = MPane{bw_widtag_q1(tag_in), ps.acc1, CNT ? ax.cnt1 : 0ULL, ps.seq1};
            }
          }
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            if (!touched[j]) continue;
            const i64 q = q_pass + j;
            int at = -1;
            for (int i = 0; i < np; ++i)
              if (P[i].q == q) at = i;
            if (at < 0) {
              P[np++] = MPane{q, bw_combine(OP, p.acc_identity, dv[j]), dcn[j], dsq[j]};
            } else {
              P[at].acc = bw_combine(OP, P[at].acc, dv[j]);
              P[at].cnt += dcn[j];
              if (dsq[j] < P[at].seq) P[at].seq = dsq[j];
            }
          }
          i64 wm = INT64_MIN;
          if (WM) {
            wm = bw_sub_sat(h.max_ts, p.wait_us);
            if (wm < BW_UTC_MIN_US_DEV) wm = BW_UTC_MIN_US_DEV;
          }
          // survivors: newest and second newest
          int i0 = -1, i1 = -1, alive = 0;
          bool range_ok = true;
          for (int i = 0; i < np; ++i) {
            if (P[i].q <= -BW_WID_LIMIT || P[i].q >= BW_WID_LIMIT) range_ok = false;
            if (WM && wm >= bw_pane_release(P[i].q, p)) continue;
            ++alive;
            if (i0 < 0 || P[i].q > P[i0].q) {
              i1 = i0;
              i0 = i;
            } else if (i1 < 0 || P[i].q > P[i1].q) {
              i1 = i;
            }
          }
          if (!range_ok) {
            bw_raise(t.ctr, 6u);
            continue;
          }
          if (alive <= 1 || (alive == 2 && P[i1].q == P[i0].q - 1)) {
            for (int i = 0; i < np; ++i)
              if (WM && wm >= bw_pane_release(P[i].q, p))
                bw_emit_closed(e, t.ctr, key, P[i].q, bw_finish_acc(p, P[i].acc), P[i].cnt, p.seq_by_id ? (u64)A.batch_no : P[i].seq,
                               A.epoch);
            const bool both = alive == 2;
            if (alive == 0) {
              // no panes left: the reference discards the whole logic, watermark included (windowing.py:1110-1113)
              h.max_ts = INT64_MIN;
              h.wt0 = BW_EMPTY_WIDTAG;
              h.acc0 = p.acc_identity;
              if (SEQ || CNT) {
                AuxSlot z = need_aux ? ax : t.aux[s];
                z.seq0 = ~0ULL;
                z.cnt0 = 0;
                z.cnt1 = 0;
                t.aux[s] = z;
              }
            } else {
              h.wt0 = bw_pack_widtag(P[i0].q, both ? 1u : 0u, BW_TAG_STALE, both, both);
              h.acc0 = P[i0].acc;
              if (SEQ || CNT) {
                AuxSlot z = need_aux ? ax : t.aux[s];
                z.seq0 = P[i0].seq;
                z.cnt0 = P[i0].cnt;
                z.cnt1 = both ? P[i1].cnt : 0;
                t.aux[s] = z;
              }
            }
            if (both) {
              P1Slot ps;
              ps.acc1 = P[i1].acc;
              ps.seq1 = SEQ ? P[i1].seq : 0ULL;  // present (any value but ~0)
              t.p1[s] = ps;
            } else if (had_p1) {
              P1Slot ps;
              ps.acc1 = p.acc_identity;
              ps.seq1 = ~0ULL;
              t.p1[s] = ps;
            }
            t.hot[s] = h;
            done = true;
          }
        }
        if (done) continue;
        // General shape (sliding windows, an overflow list, or more survivors than the two direct
        // panes hold): apply the deltas where the direct kernel would have, leave the closing to K4.
        i64 tag0 = tag_in;
        bool created = false;
        AuxSlot ax = t.aux[s];
        bool aux_dirty = false;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if (!touched[j]) continue;
          const i64 q = q_pass + j;
          if (q <= -BW_WID_LIMIT || q >= BW_WID_LIMIT) {
            bw_raise(t.ctr, 6u);
            continue;
          }
          const u64 d = dv[j], dc = dcn[j], ds = SEQ ? dsq[j] : seq_hi;
          if (tag0 == BW_EMPTY_WIDTAG) {
            const i64 a = p.panes_per_offset, bb = p.panes_per_window;
            const i64 d0 = (a == 1) ? (bb - 1) : (q - a * bw_floordiv(q - bb + a, a));
            tag0 = bw_pack_widtag(q, d0 > (i64)BW_TAG_DELTA_MAX ? BW_TAG_DELTA_MAX : (u32)d0, A.batch_no & 63u);
            h.acc0 = p.acc_identity;
            ax.seq0 = ~0ULL;
            created = true;
          }
          if (bw_widtag_q(tag0) == q) {
            h.acc0 = bw_combine(OP, h.acc0, d);
            ax.cnt0 += dc;
            if (((u32)tag0 & 0x7Fu) == (A.batch_no & 63u) && ds < ax.seq0) ax.seq0 = ds;
            aux_dirty = true;
          } else if (bw_widtag_q1(tag0) == q) {
            P1Slot ps = t.p1[s];
            ps.acc1 = bw_combine(OP, ps.acc1, d);
            if (!(tag0 & BW_TAG_P1_PREV) && ds < ps.seq1) ps.seq1 = ds;
            t.p1[s] = ps;
            tag0 |= BW_TAG_HAS_P1;
            ax.cnt1 += dc;
            aux_dirty = true;
          } else {
            // a further pane: the overflow list, through the general path
            const i64 ts_j = (j == 0 && ts_new >= A.ts0 + pb1) ? A.ts0 + pb1 - 1 : ts_new;
            bw_spill_push(A.in.spill, &A.in.sv->n_spill, A.spill_cap, nullptr, 0u, t.ctr, key, ts_j, d, ds, dc);
          }
        }
        // watermark / closability: what bw_after_fold decides per event, once per key
        {
          i64 rem;
          const i64 qn = bw_pane_of_r(ts_new, p, rem);
          bool mark = created || p.now_us != 0;  // (moving system clock: see bw_after_fold)
          if (WM && !mark) {
            const u32 delta = bw_widtag_delta(tag0);
            const i64 qc = qn - p.close_back - ((rem < p.wait_rem) ? 1 : 0);
            mark = (delta == BW_TAG_DELTA_MAX) || (qc >= bw_widtag_q(tag0) - (i64)delta);
          }
          if (mark && !(tag0 & BW_TAG_DIRTY)) {
            tag0 |= BW_TAG_DIRTY;
            const u32 i = atomicAdd(&sink.n_dirty, 1u);
            if (i < sink.cap) {
              sink.buf[i] = (u32)s;
            } else {
              const u32 g = atomicAdd(&t.ctr->dirty_count, 1u);
              t.dirty[g] = (u32)s;
            }
          }
        }
        h.wt0 = tag0;
        if (aux_dirty && (SEQ || CNT || created)) t.aux[s] = ax;
        t.hot[s] = h;
      }
    }  // pass
    __syncthreads();
    if (sink.n_dirty > sink.cap / 2) bw_sinks_flush(&sink, t);  // uniform: read after the barrier
  }
  __syncthreads();
  bw_sinks_flush(&sink, t);
  if (MODE == 1) __threadfence_system();  // the partials are in peer memory before the exchange barrier is entered
}

// Rows / partials that the streaming scheme set aside, through the general path of the direct kernel.
// Entries [lo, min(hi, count)): the rows the scatter set aside are applied BEFORE the segment fold (which closes
// windows on the assumption that it has seen the whole activation), the partials the fold sets aside after it.
__global__ void __launch_bounds__(256) k_spill(Table t, FoldParams p, const SpillRec* list, const StreamVerdict* sv, u32 cap, u32 batch_no,
                                               u32 lo, u32 hi) {
  __shared__ DirtySink sink;
  __shared__ u32 sink_buf[256];
  if (threadIdx.x == 0) {
    sink.n_dirty = 0;
    sink.n_new_keys = 0;
    sink.cap = 256;
    sink.buf = sink_buf;
  }
  bw_pdl_wait();
  bw_pdl_launch();
  __syncthreads();
  const u32 n = min(min(sv->n_spill, cap), hi);
  for (u32 i = lo + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const SpillRec r = list[i];
    bw_fold_event<FoldCfgRuntime, true>(t, p, &sink, r.key, r.ts, r.acc, r.seq, batch_no, BW_NO_SLOT, r.weight);
  }
  __syncthreads();
  bw_sinks_flush(&sink, t);
}
// end of an activation's fold stage: empty dirty list, empty spill list, no flags
__global__ void k_stream_reset(Table t, StreamVerdict* sv) {
  t.ctr->dirty_count = 0;
  if (sv) {
    sv->n_spill = 0;
    sv->flags = 0;
  }
}
