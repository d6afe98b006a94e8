// bwgpu.cu -- libbwgpu.so: C ABI (include/bwgpu.h) over the sm_100a kernels.
//
// Host side of the epoch pump for ONE stateful step: what src/worker.rs:68-83
// (`Worker::run`) + src/operators.rs:667-1024 (one activation of
// `stateful_batch`) do per epoch, restated as stream-ordered kernel launches:
//
//   commit(epoch):  [H2D] -> (world>1: K1 partition + K2 exchange) -> prepass
//                   -> K3 fold (or the exact slow path) -> K4 close
//   advance():      wait, order rows like the reference, D2H
//   eof():          K4 over every key with watermark = UTC_MAX
//
// No torch, no Python: CUDA runtime + NCCL only.
#include <cub/cub.cuh>
#include <cuda_runtime.h>
#include <nccl.h>

#include <algorithm>
#include <cmath>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../include/bwgpu.h"
#include "bw_close.cuh"
#include "bw_common.cuh"
#include "bw_exchange.cuh"
#include "bw_stream.cuh"
#include "bw_snapshot.cuh"
#include "bw_fold.cuh"
#include "bw_keyed.cuh"
#include "bw_prepass.cuh"
#include "bw_slow.cuh"
#include "bw_late.cuh"

static thread_local std::string g_last_error;

// A "world" whose ranks are threads of ONE process on ONE GPU (bw_loopback_create): the collectives become host
// rendezvous + device-to-device copies and peer memory is plain pointers.  Every multi-rank code path -- routing
// hash, partition, exchange, combine / merge -- then runs on a single-GPU box (tests/test_gpu_loopback.py); the
// kernels and their arguments are the very same as over NCCL + CUDA IPC.
struct bw_loopback {
  int world = 0;
  std::mutex mu;
  std::condition_variable cv;
  int arrived = 0;
  unsigned long long generation = 0;
  const void* slot[BW_MAX_WORLD] = {nullptr};  // what each rank published for the collective in flight
  bool broken = false;
  // false when a peer thread never arrives (it failed and left): the world is then unusable, and says so
  bool barrier() {
    std::unique_lock<std::mutex> lk(mu);
    if (broken) return false;
    const unsigned long long g = generation;
    if (++arrived == world) {
      arrived = 0;
      ++generation;
      cv.notify_all();
      return true;
    }
    if (!cv.wait_for(lk, std::chrono::seconds(120), [&] { return generation != g || broken; }) || broken) {
      broken = true;
      cv.notify_all();
      return false;
    }
    return true;
  }
};

struct bw_ctx {
  int device = 0, rank = 0, world = 1, sm_count = BW_SM_COUNT_FALLBACK;
  ncclComm_t comm = nullptr;
  bw_loopback* loop = nullptr;
  std::string err;
  void* flush_buf = nullptr;
  size_t flush_bytes = 0;
};

#define CTX_FAIL(ctx, code, ...)                         \
  do {                                                   \
    char _b[512];                                        \
    snprintf(_b, sizeof _b, __VA_ARGS__);                \
    if (ctx) (ctx)->err = _b; else g_last_error = _b;    \
    return (code);                                       \
  } while (0)

#define CU(ctx, call)                                                                              \
  do {                                                                                             \
    cudaError_t _e = (call);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      CTX_FAIL(ctx, BW_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, \
               __LINE__);                                                                          \
  } while (0)

#define NC(ctx, call)                                                                               \
  do {                                                                                              \
    ncclResult_t _e = (call);                                                                       \
    if (_e != ncclSuccess)                                                                          \
      CTX_FAIL(ctx, BW_ERR_NCCL, "%s failed: %s (%s:%d)", #call, ncclGetErrorString(_e), __FILE__,  \
               __LINE__);                                                                           \
  } while (0)

// ---- collectives: NCCL, or the loopback world's rendezvous ----
// all-gather of `bytes` per rank, device buffers, in stream order on `s`
static bw_status coll_allgather(bw_ctx* ctx, const void* send, void* recv, size_t bytes, cudaStream_t s) {
  if (!ctx->loop) {
    NC(ctx, ncclAllGather(send, recv, bytes, ncclChar, ctx->comm, s));
    return BW_OK;
  }
  bw_loopback* L = ctx->loop;
  CU(ctx, cudaStreamSynchronize(s));  // my contribution is complete
  L->slot[ctx->rank] = send;
  if (!L->barrier()) CTX_FAIL(ctx, BW_ERR_NCCL, "loopback world: a rank did not reach the all-gather");
  for (int r = 0; r < ctx->world; ++r)
    CU(ctx, cudaMemcpyAsync((char*)recv + (size_t)r * bytes, L->slot[r], bytes, cudaMemcpyDeviceToDevice, s));
  CU(ctx, cudaStreamSynchronize(s));
  // everyone has read everyone's buffer: it may be reused
  if (!L->barrier()) CTX_FAIL(ctx, BW_ERR_NCCL, "loopback world: a rank did not leave the all-gather");
  return BW_OK;
}
// barrier in stream order: completes on `s` once every rank's earlier work on its stream is done
static bw_status coll_barrier(bw_ctx* ctx, u32* d_word, cudaStream_t s) {
  if (!ctx->loop) {
    NC(ctx, ncclAllReduce(d_word, d_word, 1, ncclUint32, ncclMax, ctx->comm, s));
    return BW_OK;
  }
  CU(ctx, cudaStreamSynchronize(s));
  if (!ctx->loop->barrier()) CTX_FAIL(ctx, BW_ERR_NCCL, "loopback world: a rank did not reach the barrier");
  return BW_OK;
}
// every rank's `base` pointer as seen from this rank (CUDA IPC mappings, or the pointers themselves)
static bw_status coll_share_base(bw_ctx* ctx, void* base, void** peers, cudaStream_t s) {
  const int W = ctx->world;
  if (ctx->loop) {
    bw_loopback* L = ctx->loop;
    L->slot[ctx->rank] = base;
    if (!L->barrier()) CTX_FAIL(ctx, BW_ERR_NCCL, "loopback world: a rank did not publish its buffer");
    for (int r = 0; r < W; ++r) peers[r] = const_cast<void*>(L->slot[r]);
    if (!L->barrier()) CTX_FAIL(ctx, BW_ERR_NCCL, "loopback world: a rank did not read the buffers");
    return BW_OK;
  }
  cudaIpcMemHandle_t mine;
  CU(ctx, cudaIpcGetMemHandle(&mine, base));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "ipc handle size");
  unsigned char *d_in = nullptr, *d_all = nullptr;
  CU(ctx, cudaMalloc(&d_in, 64));
  CU(ctx, cudaMalloc(&d_all, 64 * W));
  CU(ctx, cudaMemcpy(d_in, &mine, 64, cudaMemcpyHostToDevice));
  NC(ctx, ncclAllGather(d_in, d_all, 64, ncclChar, ctx->comm, s));
  CU(ctx, cudaStreamSynchronize(s));
  std::vector<cudaIpcMemHandle_t> all(W);
  CU(ctx, cudaMemcpy(all.data(), d_all, 64 * W, cudaMemcpyDeviceToHost));
  cudaFree(d_in);
  cudaFree(d_all);
  for (int r = 0; r < W; ++r) {
    if (r == ctx->rank) peers[r] = base;
    else CU(ctx, cudaIpcOpenMemHandle(&peers[r], all[r], cudaIpcMemLazyEnablePeerAccess));
  }
  return BW_OK;
}

struct Slot {
  u64* h_keys = nullptr;
  void* h_vals = nullptr;
  i64* h_ts = nullptr;
  bool acquired = false;
};
struct Stage {  // device staging for host-ingested batches
  u64* d_keys = nullptr;
  void* d_vals = nullptr;
  i64* d_ts = nullptr;
  cudaEvent_t consumed = nullptr;  // recorded after the kernels that read it
  bool used = false;
};

// optional per-phase timing (env BW_TIMING=1): events on the streams, summed at destroy
struct PhaseTimer {
  static const int NPH = 8;
  const char* names[NPH] = {"part_hist+scan+scatter", "barrier", "prepass", "fold", "close", "scatter + verdict", "segfold", "spill + close"};
  std::vector<cudaEvent_t> ev[NPH][2];
  bool on = false;
  void mark(int ph, int which, cudaStream_t s) {
    if (!on) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, s);
    ev[ph][which].push_back(e);
  }
  void report(int rank) {
    if (!on) return;
    for (int p = 0; p < NPH; ++p) {
      size_t n = std::min(ev[p][0].size(), ev[p][1].size());
      if (!n) continue;
      double tot = 0, mn = 1e30, mx = 0;
      std::vector<float> all;
      for (size_t i = 0; i < n; ++i) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, ev[p][0][i], ev[p][1][i]) == cudaSuccess) {
          tot += ms;
          mn = std::min<double>(mn, ms);
          mx = std::max<double>(mx, ms);
          all.push_back(ms);
        }
      }
      std::sort(all.begin(), all.end());
      fprintf(stderr, "[bwgpu rank %d] %-24s n=%zu avg %.3f ms (min %.3f, median %.3f, max %.3f)\n", rank, names[p], n, tot / n, mn,
              all.empty() ? 0.0 : all[all.size() / 2], mx);
    }
  }
};

struct EventPair {
  cudaEvent_t a, b;
  u64 rows;
  int kind;  // 0: fold stage (k_fold / k_segfold), 1: k_scatter, 2: k_verdict
};

typedef void (*scatter_kernel_t)(ScatterArgs, FoldParams);
typedef void (*segfold_kernel_t)(SegArgs, Table, FoldParams, EmitBufs);

struct Stage;
// An activation whose scatter + verdict are queued but whose fold stage is not: the host looks at a
// verdict only after the NEXT activation's scatter is queued, so the device never waits for the host.
struct Deferred {
  bool valid = false;
  int side = 0;
  const u64* d_keys = nullptr;
  const void* d_vals = nullptr;
  const i64* d_ts = nullptr;
  u64 rows = 0, ord = 0;
  u32 batch_no = 0;
  u32 lanes = 0;           // blocks of this activation's scatter
  Stage* stage = nullptr;  // device staging buffer to release once the fold has read it
};

struct bw_fold {
  bw_ctx* ctx = nullptr;
  bw_fold_spec spec{};
  FoldParams p{};
  Table t{};
  EmitBufs e{};
  Counters* d_ctr = nullptr;
  Counters* h_ctr = nullptr;  // pinned mirror
  cudaStream_t s_compute = nullptr, s_copy = nullptr, s_pre = nullptr, s_x = nullptr;  // s_x: partition + exchange
  cudaEvent_t ev_fold_done = nullptr, ev_xchg_done = nullptr, ev_src_ready = nullptr;
  bool fold_recorded = false;
  cudaEvent_t ev_gen = nullptr;      // last bw_gen_c1 (the only producer of device columns this library runs itself)
  cudaEvent_t pre_wait = nullptr;    // what the verdict pass of the activation in flight has to wait for, if anything
  cudaEvent_t ev_in = nullptr, ev_pre = nullptr, ev_h2d = nullptr, ev_t0 = nullptr, ev_t1 = nullptr;
  int val_bytes = 8;
  bool has_vals = true, has_ts = false;
  // ingest
  std::vector<Slot> slots;
  std::vector<Stage> stages;
  u32 stage_next = 0;
  // prepass
  i64 *d_rmin = nullptr, *d_rmax = nullptr;
  u32* d_rbad = nullptr;
  u32* h_verdict = nullptr;  // pinned
  u32* d_verdict = nullptr;
  u64 max_recv_rows = 0;
  // slow path temp (lazy)
  u64 slow_cap = 0;
  u64 *d_kflat = nullptr, *d_ksorted = nullptr;
  i64 *d_tsflat = nullptr, *d_tssorted = nullptr, *d_prefmax = nullptr;
  u32 *d_idx = nullptr, *d_idxsorted = nullptr;
  unsigned char* d_late = nullptr;
  void* d_cub = nullptr;
  size_t cub_bytes = 0;
  // emit sort temp (lazy)
  u64 sort_cap = 0;
  u64 *d_sk = nullptr, *d_sk2 = nullptr, *d_gather = nullptr;
  u32 *d_perm = nullptr, *d_perm2 = nullptr;
  // Rows of CLOSED epochs are ordered and copied to the host while later activations run (side stream s_out, its own
  // sort scratch): bw_advance then only has the newest rows left to do.  One rank, see flush_rows().
  struct OutScratch {
    u64 cap = 0;
    u64 *sk = nullptr, *sk2 = nullptr, *gather = nullptr;
    u32 *perm = nullptr, *perm2 = nullptr;
    void* cub = nullptr;
    size_t cub_bytes = 0;
  } fl;
  struct RowMark {
    u64 epoch = 0, next_epoch = 0;  // next_epoch: 1 + epoch of the activation folded after this one (0: none yet)
    cudaEvent_t ev = nullptr;       // the counts below are on the host once this has happened
    bool live = false;
  } marks[4];
  unsigned long long* h_marks = nullptr;  // pinned [4][2]: n_closed, n_late after the marked activation
  u32 mark_head = 0;                      // marks enqueued so far
  u64 done_c = 0, done_l = 0;             // rows already ordered and on the host
  cudaStream_t s_out = nullptr;
  u32 timer_stride = 4;                   // env BW_TIMER_STRIDE: every n-th activation's kernels are timed with CUDA events
  bool flush_on = true;                   // env BW_FLUSH=0: order and copy everything in bw_advance
  bool host_ingest = false;               // the caller commits HOST batches (PCIe-bound: the device has time to spare between
                                          // activations; a device-resident caller keeps every SM busy and is left alone)
  // host output (pinned, grown on demand)
  u64 hout_cap_c = 0, hout_cap_l = 0;
  u64 *ho_ckey = nullptr, *ho_cacc = nullptr, *ho_ccount = nullptr, *ho_cepoch = nullptr;
  i64* ho_cwid = nullptr;
  u64 *ho_lkey = nullptr, *ho_lval = nullptr, *ho_lepoch = nullptr;
  i64 *ho_lwid = nullptr, *ho_lts = nullptr;
  // bookkeeping
  u32 batch_no = 0;
  u64 last_epoch = 0, min_epoch = 0;  // epochs are non-decreasing; rows carry the user epoch
  bool have_epoch = false, have_pending = false;
  bool eof_done = false;
  int fold_grid = 0, close_grid = 0;
  void (*fold_kernel)(BatchView, Table, FoldParams, u32, u32, u32) = nullptr;
  // streaming fold (bw_stream.cuh): fused verdict + bucket scatter, shared-memory segment fold
  StreamBufs sb{};
  bool stream_ok = false;   // buffers allocated, fold type supported
  int stream_mode = 1;      // env BW_STREAM=0: always take the direct kernel (k_fold)
  int scatter_grid = 0, segfold_grid = 0;
  scatter_kernel_t scatter_kernel = nullptr;
  segfold_kernel_t segfold_kernel = nullptr;
  size_t segfold_smem = 0, scatter_smem = 0;
  int scatter_nstage = 3;
  u32 last_scatter_grid = 0, scatter_stg_cap = 0, scatter_stg_every = 1;
  // multi-GPU streaming path: combine at the source, partials over NVLink, merge at the owner
  segfold_kernel_t combine_kernel = nullptr, merge_kernel = nullptr;
  int combine_grid = 0, merge_grid = 0;
  u32 nb_local = 0, part_cap = 0;
  void* precv_base = nullptr;            // this rank's receive regions (IPC-shared): [side]{cnt[W][nb_local], rec[W][nb_local][part_cap]}
  void* precv_peer[BW_MAX_WORLD] = {nullptr};
  size_t precv_cnt_off[2] = {0, 0}, precv_rec_off[2] = {0, 0};
  VerdictGather* d_vg_local = nullptr;   // [2]
  VerdictGather* d_vg_all = nullptr;     // [2][W]
  VerdictGather* h_vg = nullptr;         // pinned [2][W]
  bool vg_pending[2] = {false, false};   // a side's local verdict is computed but not gathered yet
  cudaEvent_t ev_vg[2] = {nullptr, nullptr};
  i64 h_gmax = INT64_MIN;                // running maximum event time over all ranks (the verdict chain's memory)
  u32* d_barrier_word = nullptr;
  cudaEvent_t ev_sv[2] = {nullptr, nullptr};
  StreamVerdict* h_sv = nullptr;  // pinned mirror of the two sides' verdicts
  // One GPU: the verdict runs on a stream of its own, beside the fold stage of the activation before it (nothing on
  // s_compute reads it; the host does, one activation later).  ev_sv_last: the newest verdict queued there, which
  // s_compute work that reads or writes Counters::gmax_ts / batch_clean (or copies Counters) waits for.
  cudaStream_t s_verdict = nullptr;
  cudaEvent_t ev_scattered = nullptr, ev_sv_last = nullptr;
  // activations with a few late rows (bw_late.cuh); buffers are made on first use
  LateBufs late = {};
  bool late_ready = false;
  bool late_split = true;   // env BW_LATE_SPLIT=0: every not-clean activation takes the sort path
  u32* h_late_ctr = nullptr;  // pinned: suspects seen, table overflow
  i64* late_chunk_pre = nullptr;  // [tiles][32] running maximum before every 64-row chunk
  Deferred dq{};            // the activation whose fold has not been launched yet
  i64* d_span = nullptr;   // [min ts, max ts] of the activation (prepass)
  // snapshot staging (bw_snapshot_take)
  void* snap_dev = nullptr;
  void* snap_host = nullptr;
  unsigned long long* d_snap_ctr = nullptr;
  bool sub_auto = true;     // env BW_SUB_AUTO=0: never split an activation by its event-time span
  u64 sub_rows = ~0ULL;  // optional fold + close granularity inside one activation (env BW_SUB_ROWS); measured slower on C1
  // multi-GPU exchange
  void* xchg_base = nullptr;  // one allocation, IPC-shared
  size_t xchg_bytes = 0;
  void* peer_base[BW_MAX_WORLD] = {nullptr};
  u64 region_cap = 0;
  u32* d_tile_counts = nullptr;
  u64* d_send_counts = nullptr;   // NCCL mode
  u64* d_all_counts = nullptr;    // NCCL mode [world][world]
  u64* h_all_counts = nullptr;    // pinned
  u64 *send_keys = nullptr;       // NCCL mode local send regions
  void* send_vals = nullptr;
  i64* send_ts = nullptr;
  int xbuf = 0;
  // stats
  bw_stats st{};
  std::vector<EventPair> timers;
  size_t timers_used = 0;
  PhaseTimer pt;
};

#define FAIL(f, code, ...) CTX_FAIL((f)->ctx, code, __VA_ARGS__)
static bw_status ensure_sort_cap(bw_fold* f, u64 n);
static bw_status grow_host(bw_fold* f, u64 nc, u64 nl);
static bw_status mark_rows(bw_fold* f, u64 epoch);
static bw_status flush_rows(bw_fold* f);

// ---------------------------------------------------------------------------
// small kernels
// ---------------------------------------------------------------------------
__global__ void k_init_table(Table t, u64 acc_identity) {
  const u64 n = t.cap + 1;
  for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (u64)gridDim.x * blockDim.x) {
    HotSlot h;
    h.key = BW_EMPTY_KEY;
    h.max_ts = INT64_MIN;
    h.wt0 = BW_EMPTY_WIDTAG;
    h.acc0 = acc_identity;
    t.hot[s] = h;
    P1Slot c;
    c.acc1 = acc_identity;
    c.seq1 = ~0ULL;
    t.p1[s] = c;
    AuxSlot x;
    x.seq0 = ~0ULL;
    x.cnt0 = 0;
    x.cnt1 = 0;
    x.spill_head = 0;
    x.lock = 0;
    t.aux[s] = x;
    t.closed_upto[s] = INT64_MIN;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    Counters z;
    memset(&z, 0, sizeof z);
    z.pool_next = 1;  // node 0 is the null node
    z.gmax_ts = (unsigned long long)INT64_MIN;
    *t.ctr = z;
  }
}

__global__ void k_gen_c1(u64* keys, u64* vals, u64 start, u64 rows, u64 n_keys) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < rows; i += (u64)gridDim.x * blockDim.x) {
    u64 g = start + i;
    keys[i] = bw_splitmix64(0x5EEDULL ^ g) % n_keys;
    vals[i] = g;
  }
}

__global__ void k_fill(unsigned char* p, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n / 16; i += (size_t)gridDim.x * blockDim.x)
    ((uint4*)p)[i] = make_uint4(0xA5A5A5A5u, 0xA5A5A5A5u, 0xA5A5A5A5u, 0xA5A5A5A5u);
}

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
// (C linkage comes from the declarations in include/bwgpu.h)

uint32_t bw_abi_version(void) { return BW_ABI_VERSION; }
const char* bw_last_global_error(void) { return g_last_error.c_str(); }
const char* bw_last_error(const bw_ctx* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }

uint32_t bw_route(uint64_t key, uint32_t world) { return bw_route_hash(bw_mix64(key), world); }

bw_status bw_nccl_unique_id(void* out128) {
  ncclUniqueId id;
  ncclResult_t r = ncclGetUniqueId(&id);
  if (r != ncclSuccess) {
    g_last_error = std::string("ncclGetUniqueId failed: ") + ncclGetErrorString(r);
    return BW_ERR_NCCL;
  }
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  memcpy(out128, &id, 128);
  return BW_OK;
}

bw_status bw_ctx_create(int device, int rank, int world, const void* nccl_unique_id, bw_ctx** out) {
  bw_ctx* null_ctx = nullptr;
  if (!out) CTX_FAIL(null_ctx, BW_ERR_SPEC, "bw_ctx_create: out is NULL");
  if (world < 1 || world > BW_MAX_WORLD || rank < 0 || rank >= world)
    CTX_FAIL(null_ctx, BW_ERR_SPEC, "bw_ctx_create: bad rank/world %d/%d (max world %d)", rank, world, BW_MAX_WORLD);
  if (world > 1 && !nccl_unique_id) CTX_FAIL(null_ctx, BW_ERR_SPEC, "bw_ctx_create: world > 1 needs an NCCL id");
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev <= 0)
    CTX_FAIL(null_ctx, BW_ERR_CUDA, "no CUDA device: %s", cudaGetErrorString(ce));
  if (device < 0 || device >= ndev) CTX_FAIL(null_ctx, BW_ERR_SPEC, "device %d out of range (%d devices)", device, ndev);
  CU(null_ctx, cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(null_ctx, cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    CTX_FAIL(null_ctx, BW_ERR_CUDA, "libbwgpu is built for sm_100a only; device %d is sm_%d%d", device, prop.major,
             prop.minor);
  bw_ctx* c = new bw_ctx();
  c->device = device;
  c->rank = rank;
  c->world = world;
  c->sm_count = prop.multiProcessorCount;
  if (world > 1) {
    ncclUniqueId id;
    memcpy(&id, nccl_unique_id, 128);
    ncclResult_t r = ncclCommInitRank(&c->comm, world, id, rank);
    if (r != ncclSuccess) {
      g_last_error = std::string("ncclCommInitRank failed: ") + ncclGetErrorString(r);
      delete c;
      return BW_ERR_NCCL;
    }
  }
  *out = c;
  return BW_OK;
}

bw_status bw_loopback_create(int world, bw_loopback** out) {
  bw_ctx* null_ctx = nullptr;
  if (!out || world < 2 || world > BW_MAX_WORLD) CTX_FAIL(null_ctx, BW_ERR_SPEC, "bw_loopback_create: world must be in 2..%d", BW_MAX_WORLD);
  bw_loopback* L = new bw_loopback();
  L->world = world;
  *out = L;
  return BW_OK;
}
void bw_loopback_destroy(bw_loopback* world) { delete world; }

bw_status bw_ctx_create_loopback(int device, int rank, bw_loopback* world, bw_ctx** out) {
  bw_ctx* null_ctx = nullptr;
  if (!out || !world || rank < 0 || rank >= world->world) CTX_FAIL(null_ctx, BW_ERR_SPEC, "bw_ctx_create_loopback: bad arguments");
  bw_ctx* c = nullptr;
  bw_status st = bw_ctx_create(device, 0, 1, nullptr, &c);  // device checks; no communicator
  if (st != BW_OK) return st;
  c->rank = rank;
  c->world = world->world;
  c->loop = world;
  *out = c;
  return BW_OK;
}

void bw_ctx_destroy(bw_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->comm) ncclCommDestroy(ctx->comm);
  if (ctx->flush_buf) cudaFree(ctx->flush_buf);
  delete ctx;
}

bw_status bw_dev_alloc(bw_ctx* ctx, uint64_t bytes, void** out) {
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaMalloc(out, bytes ? bytes : 16));
  return BW_OK;
}
bw_status bw_dev_free(bw_ctx* ctx, void* ptr) {
  CU(ctx, cudaFree(ptr));
  return BW_OK;
}
bw_status bw_host_alloc(bw_ctx* ctx, uint64_t bytes, void** out) {
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaHostAlloc(out, bytes ? bytes : 16, cudaHostAllocDefault));
  return BW_OK;
}
bw_status bw_host_free(bw_ctx* ctx, void* ptr) {
  CU(ctx, cudaFreeHost(ptr));
  return BW_OK;
}
bw_status bw_memcpy(bw_ctx* ctx, void* dst, const void* src, uint64_t bytes, int kind) {
  cudaMemcpyKind k = kind == 0 ? cudaMemcpyHostToDevice : kind == 1 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  CU(ctx, cudaMemcpy(dst, src, bytes, k));
  return BW_OK;
}
bw_status bw_flush_l2(bw_ctx* ctx) {
  CU(ctx, cudaSetDevice(ctx->device));
  if (!ctx->flush_buf) {
    ctx->flush_bytes = (size_t)256 << 20;  // 256 MiB > 126 MB L2
    CU(ctx, cudaMalloc(&ctx->flush_buf, ctx->flush_bytes));
  }
  k_fill<<<ctx->sm_count * 8, 256>>>((unsigned char*)ctx->flush_buf, ctx->flush_bytes);
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaDeviceSynchronize());
  return BW_OK;
}

// ---------------------------------------------------------------------------
// fold create / destroy
// ---------------------------------------------------------------------------
static i64 gcd_i64(i64 a, i64 b) {
  while (b) {
    i64 t = a % b;
    a = b;
    b = t;
  }
  return a;
}

template <typename T>
static cudaError_t dmalloc(T** p, size_t n) {
  return cudaMalloc((void**)p, (n ? n : 1) * sizeof(T));
}

// k_fold instantiations: accumulator op x watermark tracking (+ MEAN keeps counts)
typedef void (*fold_kernel_t)(BatchView, Table, FoldParams, u32, u32, u32);
template <int OP, int CNT>
static fold_kernel_t pick_wm(bool wm) {
  return wm ? (fold_kernel_t)k_fold<FoldCfg<OP, 1, CNT>> : (fold_kernel_t)k_fold<FoldCfg<OP, 0, CNT>>;
}
static fold_kernel_t pick_fold_kernel(const FoldParams& p) {
  const bool wm = p.track_wm != 0;
  if (p.need_count) return pick_wm<BW_OP_ADD_F64, 1>(wm);
  switch (p.op) {
    case BW_OP_ADD_ONE: return pick_wm<BW_OP_ADD_ONE, 0>(wm);
    case BW_OP_ADD_U64: return pick_wm<BW_OP_ADD_U64, 0>(wm);
    case BW_OP_ADD_F64: return pick_wm<BW_OP_ADD_F64, 0>(wm);
    case BW_OP_MIN_S64: return pick_wm<BW_OP_MIN_S64, 0>(wm);
    case BW_OP_MIN_U64: return pick_wm<BW_OP_MIN_U64, 0>(wm);
    case BW_OP_MAX_S64: return pick_wm<BW_OP_MAX_S64, 0>(wm);
    default: return pick_wm<BW_OP_MAX_U64, 0>(wm);
  }
}

// k_segfold instantiations: accumulator op (+ counts for MEAN) x first-open indices
template <int OP, int CNT, int MODE>
static segfold_kernel_t pick_seq(bool seq) {
  return seq ? (segfold_kernel_t)k_segfold<FoldCfg<OP, -1, CNT>, true, MODE> : (segfold_kernel_t)k_segfold<FoldCfg<OP, -1, CNT>, false, MODE>;
}
// MODE: 0 one GPU, 1 combine at the source rank, 2 merge at the owning rank (bw_stream.cuh)
template <int MODE>
static segfold_kernel_t pick_segfold_kernel(const FoldParams& p) {
  const bool seq = !p.seq_by_id;
  if (p.need_count) return pick_seq<BW_OP_ADD_F64, 1, MODE>(seq);
  switch (p.op) {
    case BW_OP_ADD_ONE: return pick_seq<BW_OP_ADD_ONE, 0, MODE>(seq);
    case BW_OP_ADD_U64: return pick_seq<BW_OP_ADD_U64, 0, MODE>(seq);
    case BW_OP_ADD_F64: return pick_seq<BW_OP_ADD_F64, 0, MODE>(seq);
    case BW_OP_MIN_S64: return pick_seq<BW_OP_MIN_S64, 0, MODE>(seq);
    case BW_OP_MIN_U64: return pick_seq<BW_OP_MIN_U64, 0, MODE>(seq);
    case BW_OP_MAX_S64: return pick_seq<BW_OP_MAX_S64, 0, MODE>(seq);
    default: return pick_seq<BW_OP_MAX_U64, 0, MODE>(seq);
  }
}
// k_scatter instantiations: timestamp source x value bytes read / stored
static scatter_kernel_t pick_scatter_kernel(int tsm, int vb_in, int vb_out) {
  if (tsm == 1) return vb_out ? (scatter_kernel_t)k_scatter<1, 8, 8> : (scatter_kernel_t)k_scatter<1, 8, 0>;
  if (tsm == 0) {
    if (!vb_out) return (scatter_kernel_t)k_scatter<0, 0, 0>;
    return vb_in == 4 ? (scatter_kernel_t)k_scatter<0, 4, 4> : (scatter_kernel_t)k_scatter<0, 8, 8>;
  }
  if (!vb_out) return (scatter_kernel_t)k_scatter<2, 0, 0>;
  return vb_in == 4 ? (scatter_kernel_t)k_scatter<2, 4, 4> : (scatter_kernel_t)k_scatter<2, 8, 8>;
}

static bw_status stream_alloc(bw_fold* f) {
  bw_ctx* ctx = f->ctx;
  StreamBufs& sb = f->sb;
  const u64 rows = f->spec.max_batch_rows;
  const int W = ctx->world;
  f->nb_local = (u32)(f->t.cap >> f->t.seg_shift);
  const u64 nb = (u64)f->nb_local * W;  // buckets of the scatter: (owning rank, segment of its table)
  if (const char* e = getenv("BW_STREAM")) f->stream_mode = atoi(e) ? 1 : 0;
  if (!f->stream_mode || nb > BW_STREAM_MAX_NB || rows >= (1ULL << 28)) return BW_OK;
  if (W > 1 && f->spec.exchange != BW_XCHG_P2P) return BW_OK;  // the partials travel as peer stores
  // wait == forever with event time: nothing closes before EOF, every key grows an overflow list of panes --
  // the shape the direct kernel's general path is for
  if (!f->p.track_wm && f->p.ts_from_value != 2) return BW_OK;
  sb.nb = (u32)nb;
  // Every scatter block owns a lane in every bucket's region.  A lane holds the block's share of the bucket's rows: mean
  // + 6 sigma, where the variance is that of the rows (Poisson) plus that of the bucket's number of distinct keys (a fuller
  // lane overflows into the spill list).
  sb.nlanes = (u32)ctx->sm_count;
  const u64 max_tiles = (rows + BW_SC_TILE - 1) / BW_SC_TILE;
  const double block_rows = (double)((max_tiles + sb.nlanes - 1) / sb.nlanes) * BW_SC_TILE;
  const double mean = block_rows / (double)nb;
  const double keys_per_bucket = std::max(1.0, (double)std::max<u64>(f->spec.capacity_hint, 1) / (double)f->nb_local);
  const double sigma = std::sqrt(mean + mean * mean / keys_per_bucket);
  sb.lane_cap = (u32)std::min<double>(block_rows, mean + 6.0 * sigma + 24.0);
  sb.lane_cap = (sb.lane_cap + 7u) & ~7u;
  // every row can end up there in the worst case (a pane per event beyond a key's two direct panes: sparse sliding folds)
  sb.spill_cap = (u32)std::min<u64>(std::max<u64>(rows + rows / 8, 8192), 1u << 26);
  sb.val_bytes = (f->p.op == BW_OP_ADD_ONE && !f->p.need_count) ? 0 : f->val_bytes;
  const size_t region_rows = (size_t)sb.nb * sb.nlanes * sb.lane_cap;
  for (int i = 0; i < 2; ++i) {
    CU(ctx, dmalloc(&sb.side[i].rec, region_rows));
    if (sb.val_bytes) CU(ctx, cudaMalloc(&sb.side[i].val, region_rows * (size_t)sb.val_bytes));
    CU(ctx, dmalloc(&sb.side[i].cnt, (size_t)sb.nb * sb.nlanes));
    CU(ctx, cudaMemsetAsync(sb.side[i].cnt, 0, sizeof(u32) * sb.nb * sb.nlanes, f->s_compute));
    CU(ctx, dmalloc(&sb.side[i].spill, sb.spill_cap));
    CU(ctx, dmalloc(&sb.side[i].sv, 1));
    CU(ctx, cudaMemsetAsync(sb.side[i].sv, 0, sizeof(StreamVerdict), f->s_compute));
    CU(ctx, cudaEventCreateWithFlags(&f->ev_sv[i], cudaEventDisableTiming));
  }
  CU(ctx, cudaHostAlloc((void**)&f->h_sv, 2 * sizeof(StreamVerdict), cudaHostAllocDefault));
  const int tsm = f->p.ts_from_value ? f->p.ts_from_value : 0;
  const int vb_in = (tsm == 1) ? 8 : (sb.val_bytes ? f->val_bytes : 0);
  f->scatter_kernel = pick_scatter_kernel(tsm, vb_in, sb.val_bytes);
  sb.tiles_cap = (u32)((rows + BW_SC_TILE - 1) / BW_SC_TILE + 1);  // one lateness triple per scatter tile
  // (one set per side: the tile triples of activation b are read again when it turns out to have late rows, after the
  // scatter of b + 1 has run)
  CU(ctx, dmalloc(&sb.tile_min, 2 * (size_t)sb.tiles_cap));
  CU(ctx, dmalloc(&sb.tile_max, 2 * (size_t)sb.tiles_cap));
  CU(ctx, dmalloc(&sb.tile_bad, 2 * (size_t)sb.tiles_cap));
  CU(ctx, dmalloc(&sb.chunk_max, 2 * (size_t)sb.tiles_cap * BW_SC_WARPS));
  if (const char* e = getenv("BW_LATE_SPLIT")) f->late_split = atoi(e) != 0;
  if (const char* e = getenv("BW_FLUSH")) f->flush_on = atoi(e) != 0;
  if (const char* e = getenv("BW_TIMER_STRIDE")) f->timer_stride = (u32)std::max(1, atoi(e));
  // Shared memory of the scatter: up to 8 records per bucket assembled before they are written out (counts only: the
  // value column is not staged), then as many TMA stages of the input tile (2..4) as still fit.
  const size_t smem_budget = 208 * 1024;
  f->scatter_stg_cap = 0;
  if (sb.val_bytes == 0)
    for (u32 c = 8; c >= 4; c -= 2)
      if (bw_scatter_smem(tsm, vb_in, 2, sb.nb, c) <= smem_budget) {
        f->scatter_stg_cap = c;
        break;
      }
  if (const char* e = getenv("BW_SC_STG")) f->scatter_stg_cap = (u32)std::max(0, std::min(16, atoi(e)));
  // write out when an average bucket has assembled ~7/8 of its staging rows (measured on C1: 2 tiles 0.239 ms, 3 0.217, 4 0.213)
  f->scatter_stg_every = (u32)std::max<double>(1.0, std::floor(0.875 * f->scatter_stg_cap * (double)sb.nb / BW_SC_TILE));
  if (const char* e = getenv("BW_SC_EVERY")) f->scatter_stg_every = (u32)std::max(1, atoi(e));
  f->scatter_nstage = 4;
  while (f->scatter_nstage > 2 && bw_scatter_smem(tsm, vb_in, f->scatter_nstage, sb.nb, f->scatter_stg_cap) > smem_budget) --f->scatter_nstage;
  if (const char* e = getenv("BW_SC_STAGES")) f->scatter_nstage = std::max(2, std::min(4, atoi(e)));
  if (bw_scatter_smem(tsm, vb_in, f->scatter_nstage, sb.nb, f->scatter_stg_cap) > 216 * 1024) return BW_OK;  // too many segments
  f->scatter_smem = bw_scatter_smem(tsm, vb_in, f->scatter_nstage, sb.nb, f->scatter_stg_cap);
  // the attribute belongs to the kernel, not to this fold: folds with other table sizes share it
  CU(ctx, cudaFuncSetAttribute((const void*)f->scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
  int occ = 0;
  CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (const void*)f->scatter_kernel, BW_SC_THREADS, f->scatter_smem));
  f->scatter_grid = ctx->sm_count * std::max(occ, 1);
  f->segfold_kernel = pick_segfold_kernel<0>(f->p);
  f->segfold_smem = bw_segfold_smem(1u << f->t.seg_shift, f->p.op, !f->p.seq_by_id, f->p.need_count != 0);
  CU(ctx, cudaFuncSetAttribute((const void*)f->segfold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
  CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (const void*)f->segfold_kernel, BW_SF_THREADS, f->segfold_smem));
  f->segfold_grid = ctx->sm_count * std::max(occ, 1);
  if (W > 1) {
    f->combine_kernel = pick_segfold_kernel<1>(f->p);
    f->merge_kernel = pick_segfold_kernel<2>(f->p);
    for (segfold_kernel_t k : {f->combine_kernel, f->merge_kernel}) {
      CU(ctx, cudaFuncSetAttribute((const void*)k, cudaFuncAttributeMaxDynamicSharedMemorySize, 216 * 1024));
      CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (const void*)k, BW_SF_THREADS, f->segfold_smem));
      (k == f->combine_kernel ? f->combine_grid : f->merge_grid) = ctx->sm_count * std::max(occ, 1);
    }
    // receive regions: a source can leave at most two partials (two panes) per slot of a segment
    f->part_cap = 2u << f->t.seg_shift;
    size_t off = 0;
    auto take = [&](size_t bytes) {
      size_t o = off;
      off += (bytes + 255) & ~(size_t)255;
      return o;
    };
    for (int sd = 0; sd < 2; ++sd) {
      f->precv_cnt_off[sd] = take(sizeof(u32) * (size_t)W * f->nb_local);
      f->precv_rec_off[sd] = take(sizeof(Partial) * (size_t)W * f->nb_local * f->part_cap);
    }
    CU(ctx, cudaMalloc(&f->precv_base, off));
    CU(ctx, cudaMemset(f->precv_base, 0, off));
    {
      bw_status cst = coll_share_base(ctx, f->precv_base, f->precv_peer, f->s_compute);
      if (cst != BW_OK) return cst;
    }
    CU(ctx, dmalloc(&f->d_vg_local, 2));
    CU(ctx, dmalloc(&f->d_vg_all, 2 * (size_t)W));
    CU(ctx, cudaHostAlloc((void**)&f->h_vg, sizeof(VerdictGather) * 2 * W, cudaHostAllocDefault));
    CU(ctx, dmalloc(&f->d_barrier_word, 1));
    CU(ctx, cudaMemset(f->d_barrier_word, 0, 4));
    // the legacy path is now the fallback of single activations: it runs in line with the rest (its own stream only
    // bought overlap between consecutive legacy activations, and its lateness pass must see the maximum set here)
    if (f->s_x && f->s_x != f->s_compute) {
      cudaStreamDestroy(f->s_x);
      f->s_x = f->s_compute;
    }
  }
  f->stream_ok = true;
  return BW_OK;
}

static bw_status fold_alloc(bw_fold* f) {
  bw_ctx* ctx = f->ctx;
  const bw_fold_spec& s = f->spec;
  // table: capacity_hint / load factor slots (load 0.5 by default, env BW_LOAD_PCT), a whole number of
  // segments of BW_SEG_SLOTS slots: linear probing wraps inside a segment (bw_stream.cuh owns whole segments)
  int load_pct = 50;
  if (const char* e = getenv("BW_LOAD_PCT")) {
    int v = atoi(e);
    if (v >= 10 && v <= 90) load_pct = v;
  }
  u32 seg_shift = BW_SEG_SHIFT_DEFAULT;
  {
    // multi-GPU: the scatter buckets by (owning rank, segment): keep world x segments near the one-GPU bucket count
    const u64 want = (std::max<u64>(s.capacity_hint, 1) * 100 + load_pct - 1) / load_pct;
    if (ctx->world > 1 && (u64)ctx->world * ((want >> seg_shift) + 1) > 1024) seg_shift = 12;
  }
  if (const char* e = getenv("BW_SEG_SHIFT")) seg_shift = (u32)std::max(10, std::min(12, atoi(e)));
  const u64 seg_slots = 1ULL << seg_shift;
  u64 cap = std::max<u64>(seg_slots, (std::max<u64>(s.capacity_hint, 1) * 100 + load_pct - 1) / load_pct);
  cap = (cap + seg_slots - 1) & ~(seg_slots - 1);
  if (cap > (1ULL << 31)) FAIL(f, BW_ERR_SPEC, "capacity_hint too large");
  f->t.cap = cap;
  f->t.seg_shift = seg_shift;
  f->t.seg_mask = (u32)seg_slots - 1;
  {
    // overflow pane nodes: panes a key can hold beyond its two direct slots
    const i64 per_window = f->p.panes_per_window;
    u64 expect = 32;  // wait == forever: nothing closes before EOF
    if (f->p.track_wm) expect = (u64)std::min<i64>(per_window + f->p.wait_us / f->p.pane_us + 4, 1 << 20);
    u64 want = std::max<u64>(2 * cap, std::max<u64>(s.capacity_hint, 1024) * expect) + 1024;
    f->t.pool_cap = (u32)std::min<u64>(want, 0x7FFFFFF0ULL);
  }
  CU(ctx, dmalloc(&f->t.hot, cap + 1));
  CU(ctx, dmalloc(&f->t.p1, cap + 1));
  CU(ctx, dmalloc(&f->t.closed_upto, cap + 1));
  CU(ctx, dmalloc(&f->t.aux, cap + 1));
  CU(ctx, dmalloc(&f->t.nodes, f->t.pool_cap));
  CU(ctx, dmalloc(&f->t.node_acc2, f->t.pool_cap));
  CU(ctx, dmalloc(&f->t.free_stack, f->t.pool_cap));
  CU(ctx, dmalloc(&f->t.dirty, cap + 2));
  CU(ctx, dmalloc(&f->d_ctr, 1));
  f->t.ctr = f->d_ctr;
  CU(ctx, cudaHostAlloc((void**)&f->h_ctr, sizeof(Counters), cudaHostAllocDefault));
  // emit buffers
  f->e.max_closed = s.max_emit_rows;
  f->e.max_late = s.max_late_rows;
  CU(ctx, dmalloc(&f->e.c_key, s.max_emit_rows));
  CU(ctx, dmalloc(&f->e.c_wid, s.max_emit_rows));
  CU(ctx, dmalloc(&f->e.c_acc, s.max_emit_rows));
  CU(ctx, dmalloc(&f->e.c_count, s.max_emit_rows));
  CU(ctx, dmalloc(&f->e.c_seq, s.max_emit_rows));
  CU(ctx, dmalloc(&f->e.c_epoch, s.max_emit_rows));
  CU(ctx, dmalloc(&f->e.l_key, s.max_late_rows));
  CU(ctx, dmalloc(&f->e.l_wid, s.max_late_rows));
  CU(ctx, dmalloc(&f->e.l_val, s.max_late_rows));
  CU(ctx, dmalloc(&f->e.l_ts, s.max_late_rows));
  CU(ctx, dmalloc(&f->e.l_seq, s.max_late_rows));
  CU(ctx, dmalloc(&f->e.l_epoch, s.max_late_rows));
  // prepass
  f->max_recv_rows = s.max_batch_rows * (u64)ctx->world;
  u64 nranges = (f->max_recv_rows + BW_RANGE_ROWS - 1) / BW_RANGE_ROWS + 1;
  CU(ctx, dmalloc(&f->d_rmin, nranges));
  CU(ctx, dmalloc(&f->d_rmax, nranges));
  CU(ctx, dmalloc(&f->d_rbad, nranges));
  CU(ctx, dmalloc(&f->d_verdict, 1));
  CU(ctx, dmalloc(&f->d_span, 2));
  CU(ctx, cudaHostAlloc((void**)&f->h_verdict, 64, cudaHostAllocDefault));
  CU(ctx, cudaStreamCreateWithFlags(&f->s_compute, cudaStreamNonBlocking));
  CU(ctx, cudaStreamCreateWithFlags(&f->s_copy, cudaStreamNonBlocking));
  {
    // the verdict pass gates the next fold: let its blocks be placed first whenever an SM has room
    int prio_lo = 0, prio_hi = 0;
    CU(ctx, cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    CU(ctx, cudaStreamCreateWithPriority(&f->s_pre, cudaStreamNonBlocking, prio_hi));
    // the one-block verdict likewise: it runs beside the segment fold and should find room as soon as there is any
    CU(ctx, cudaStreamCreateWithPriority(&f->s_verdict, cudaStreamNonBlocking, prio_hi));
  }
  if (getenv("BW_NO_OVERLAP")) f->s_x = f->s_compute;  // diagnostic: serialise exchange and fold
  else CU(ctx, cudaStreamCreateWithFlags(&f->s_x, cudaStreamNonBlocking));
  CU(ctx, cudaEventCreateWithFlags(&f->ev_fold_done, cudaEventDisableTiming));
  CU(ctx, cudaEventCreateWithFlags(&f->ev_xchg_done, cudaEventDisableTiming));
  CU(ctx, cudaEventCreateWithFlags(&f->ev_src_ready, cudaEventDisableTiming));
  CU(ctx, cudaEventCreateWithFlags(&f->ev_in, cudaEventDisableTiming));
  CU(ctx, cudaEventCreateWithFlags(&f->ev_pre, cudaEventDisableTiming));
  CU(ctx, cudaEventCreateWithFlags(&f->ev_h2d, cudaEventDisableTiming));
  CU(ctx, cudaEventCreateWithFlags(&f->ev_scattered, cudaEventDisableTiming));
  // No persisting-L2 carve-out: measured on this part (profiles/r01_notes.md) a 64 MiB persisting
  // window on the hot slots leaves too little normal L2 for the second-pane array and slows
  // window-boundary activations by 15-30 %; plain LRU + evict_first input loads is faster.
  int occ = 0;
  f->fold_kernel = pick_fold_kernel(f->p);
  f->pt.on = getenv("BW_TIMING") != nullptr;
  if (const char* e = getenv("BW_SUB_AUTO")) f->sub_auto = atoi(e) != 0;
  if (const char* e = getenv("BW_SUB_ROWS")) {
    long long v = atoll(e);
    if (v >= 1024) f->sub_rows = (u64)v;
  }
  CU(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, f->fold_kernel, BW_FOLD_THREADS, 0));
  if (occ < 1) occ = 1;
  f->fold_grid = ctx->sm_count * occ;
  // multi-GPU: leave register-file room on every SM so the next activation's partition/scatter
  // (NVLink-bound, on its own stream) can really run beside the fold instead of queueing behind it
  if (ctx->world > 1 && occ > 2 && !getenv("BW_FOLD_FULL")) f->fold_grid = ctx->sm_count * 2;
  f->close_grid = ctx->sm_count * 8;
  {
    bw_status st = stream_alloc(f);
    if (st != BW_OK) return st;
  }
  k_init_table<<<ctx->sm_count * 8, 256, 0, f->s_compute>>>(f->t, f->p.acc_identity);
  CU(ctx, cudaGetLastError());
  f->st.kernel_launches++;
  f->st.table_capacity = cap;
  return BW_OK;
}

// one IPC-shared allocation per rank holding both receive buffers + count tables
struct XLayout {
  size_t counts_off[2], keys_off[2], vals_off[2], ts_off[2], total;
};
static XLayout xlayout(const bw_fold* f) {
  XLayout L;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off += (bytes + 255) & ~(size_t)255;
    return o;
  };
  const size_t rows = (size_t)f->region_cap * f->ctx->world;
  for (int b = 0; b < 2; ++b) {
    L.counts_off[b] = take(sizeof(u64) * BW_MAX_WORLD);
    L.keys_off[b] = take(rows * 8);
    L.vals_off[b] = f->has_vals ? take(rows * (size_t)f->val_bytes) : 0;
    L.ts_off[b] = f->has_ts ? take(rows * 8) : 0;
  }
  L.total = off;
  return L;
}

static bw_status xchg_setup(bw_fold* f) {
  bw_ctx* ctx = f->ctx;
  const int W = ctx->world;
  f->region_cap = f->spec.max_batch_rows;  // worst case: every row of a source goes to one rank
  XLayout L = xlayout(f);
  f->xchg_bytes = L.total;
  CU(ctx, cudaMalloc(&f->xchg_base, L.total));
  CU(ctx, cudaMemset(f->xchg_base, 0, L.total));
  CU(ctx, cudaFuncSetAttribute(k_part_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, BW_PART_TILE * 24));
  u64 ntiles = (f->spec.max_batch_rows + BW_PART_TILE - 1) / BW_PART_TILE + 1;
  CU(ctx, dmalloc(&f->d_tile_counts, ntiles * BW_MAX_WORLD));
  if (f->spec.exchange == BW_XCHG_P2P) {
    // every peer's receive buffer as seen from here (CUDA IPC mappings exchanged through NCCL)
    bw_status cst = coll_share_base(ctx, f->xchg_base, f->peer_base, f->s_compute);
    if (cst != BW_OK) return cst;
  } else {
    const size_t rows = (size_t)f->region_cap * W;
    CU(ctx, dmalloc(&f->send_keys, rows));
    if (f->has_vals) CU(ctx, cudaMalloc(&f->send_vals, rows * (size_t)f->val_bytes));
    if (f->has_ts) CU(ctx, dmalloc(&f->send_ts, rows));
    CU(ctx, dmalloc(&f->d_send_counts, BW_MAX_WORLD));
    CU(ctx, dmalloc(&f->d_all_counts, (size_t)BW_MAX_WORLD * BW_MAX_WORLD));
    CU(ctx, cudaHostAlloc((void**)&f->h_all_counts, sizeof(u64) * BW_MAX_WORLD * BW_MAX_WORLD, cudaHostAllocDefault));
    for (int r = 0; r < W; ++r) f->peer_base[r] = nullptr;
    f->peer_base[ctx->rank] = f->xchg_base;
  }
  return BW_OK;
}

bw_status bw_fold_create(bw_ctx* ctx, const bw_fold_spec* spec, bw_fold** out) {
  if (!ctx || !spec || !out) CTX_FAIL(ctx, BW_ERR_SPEC, "bw_fold_create: NULL argument");
  if (spec->struct_size != sizeof(bw_fold_spec))
    CTX_FAIL(ctx, BW_ERR_SPEC, "bw_fold_spec.struct_size %u != %zu", spec->struct_size, sizeof(bw_fold_spec));
  if (spec->reduction < 0 || spec->reduction > BW_RED_MEAN) CTX_FAIL(ctx, BW_ERR_SPEC, "bad reduction %d", spec->reduction);
  if (spec->val_dtype < 0 || spec->val_dtype > BW_VAL_F64) CTX_FAIL(ctx, BW_ERR_SPEC, "bad val_dtype %d", spec->val_dtype);
  if (spec->length_us <= 0 || spec->offset_us <= 0 || spec->offset_us > spec->length_us)
    CTX_FAIL(ctx, BW_ERR_SPEC, "need 0 < offset_us <= length_us (windowing.py:880-883)");
  if (spec->wait_us < 0) CTX_FAIL(ctx, BW_ERR_SPEC, "wait_us must be >= 0");
  if (ctx->loop && spec->exchange != BW_XCHG_P2P) CTX_FAIL(ctx, BW_ERR_SPEC, "a loopback world exchanges over peer memory only (BW_XCHG_P2P)");
  if (spec->ts_source < BW_TS_COLUMN || spec->ts_source > BW_TS_NONE) CTX_FAIL(ctx, BW_ERR_SPEC, "bad ts_source %d", spec->ts_source);
  if (spec->ts_source == BW_TS_FROM_VALUE && spec->val_dtype > BW_VAL_I64)
    CTX_FAIL(ctx, BW_ERR_SPEC, "BW_TS_FROM_VALUE needs an integer val_dtype");
  if (spec->ts_source == BW_TS_NONE && spec->wait_us != BW_WAIT_FOREVER)
    CTX_FAIL(ctx, BW_ERR_SPEC, "BW_TS_NONE (the *_final folds) needs wait_us == BW_WAIT_FOREVER: nothing closes before bw_eof");
  if (spec->max_batch_rows == 0 || spec->max_batch_rows >= (1ULL << 32) / (u64)ctx->world)
    CTX_FAIL(ctx, BW_ERR_SPEC, "max_batch_rows * world must be in [1, 2^32)");
  CU(ctx, cudaSetDevice(ctx->device));
  bw_fold* f = new bw_fold();
  f->ctx = ctx;
  f->spec = *spec;
  FoldParams& p = f->p;
  p.length_us = spec->length_us;
  p.offset_us = spec->offset_us;
  p.align_us = spec->align_to_us;
  p.wait_us = spec->wait_us;
  p.pane_us = gcd_i64(spec->length_us, spec->offset_us);
  p.panes_per_offset = spec->offset_us / p.pane_us;
  p.panes_per_window = spec->length_us / p.pane_us;
  p.inv_pane = 1.0 / (double)p.pane_us;
  {
    // round-up multiplier for exact u64 division by pane_us (Granlund-Montgomery / libdivide "algorithm 1")
    const u64 D = (u64)p.pane_us;
    p.div_is_one = (D == 1);
    u32 L = 0;
    while (L < 64 && ((L == 63) ? false : ((1ULL << L) < D))) ++L;
    if ((1ULL << (L >= 64 ? 63 : L)) < D) L = 64;
    if (!p.div_is_one) {
      const unsigned __int128 one = 1;
      const unsigned __int128 num = (one << 64) * (unsigned __int128)(((L >= 64) ? (unsigned __int128)(one << 64) : (unsigned __int128)(one << L)) - D);
      p.div_magic = (u64)(num / D) + 1;
      p.div_shift = L - 1;
    } else {
      p.div_magic = 0;
      p.div_shift = 0;
    }
    // bias: multiple of pane, >= 2^59 (covers |ts - align| for every representable datetime pair)
    const i64 need = (i64)1 << 59;
    p.div_bias_q = (need + p.pane_us - 1) / p.pane_us;
    p.div_bias = p.div_bias_q * p.pane_us;
    const i64 w = p.track_wm ? p.wait_us : 0;
    p.close_back = p.length_us / p.pane_us + w / p.pane_us;
    p.wait_rem = w % p.pane_us;
  }
  p.reduction = spec->reduction;
  p.val_dtype = spec->val_dtype;
  p.ts_from_value = spec->ts_source == BW_TS_FROM_VALUE ? 1 : (spec->ts_source == BW_TS_NONE ? 2 : 0);
  p.track_wm = spec->wait_us != BW_WAIT_FOREVER;
  p.ordered = spec->ordered;
  p.need_count = spec->reduction == BW_RED_MEAN;
  // first-opened order of a key's windows == ascending id when flushes are ordered, when nothing is
  // accepted out of order (wait == 0: an accepted timestamp is never below the key's maximum), or when
  // there is a single window (the *_final folds)
  p.seq_by_id = (spec->ordered || spec->ts_source == BW_TS_NONE || spec->wait_us == 0) ? 1 : 0;
  const bool is_float = spec->val_dtype >= BW_VAL_F32, is_signed = spec->val_dtype == BW_VAL_I64;
  switch (spec->reduction) {
    case BW_RED_COUNT: p.op = BW_OP_ADD_ONE; p.acc_identity = 0; break;
    case BW_RED_SUM: p.op = is_float ? BW_OP_ADD_F64 : BW_OP_ADD_U64; p.acc_identity = 0; break;
    case BW_RED_MEAN: p.op = BW_OP_ADD_F64; p.acc_identity = 0; break;
    case BW_RED_MIN:
      p.op = (is_float || !is_signed) ? BW_OP_MIN_U64 : BW_OP_MIN_S64;
      p.acc_identity = (p.op == BW_OP_MIN_S64) ? (u64)INT64_MAX : ~0ULL;
      break;
    default:
      p.op = (is_float || !is_signed) ? BW_OP_MAX_U64 : BW_OP_MAX_S64;
      p.acc_identity = (p.op == BW_OP_MAX_S64) ? (u64)INT64_MIN : 0ULL;
      break;
  }
  f->val_bytes = spec->val_dtype == BW_VAL_F32 ? 4 : 8;
  f->has_ts = spec->ts_source == BW_TS_COLUMN;
  f->has_vals = true;  // the late stream carries the original value, even for counts
  bw_status st = fold_alloc(f);
  if (st != BW_OK) return st;
  if (ctx->world > 1) {
    st = xchg_setup(f);
    if (st != BW_OK) return st;
  }
  // emission staging is sized once: no allocation on the advance path
  st = ensure_sort_cap(f, std::max<u64>(spec->max_emit_rows, spec->max_late_rows));
  if (st != BW_OK) return st;
  st = grow_host(f, spec->max_emit_rows, spec->max_late_rows);
  if (st != BW_OK) return st;
  CU(ctx, cudaStreamSynchronize(f->s_compute));
  *out = f;
  return BW_OK;
}

static bw_status stream_resolve(bw_fold* f);

void bw_fold_destroy(bw_fold* f) {
  if (!f) return;
  cudaSetDevice(f->ctx->device);
  stream_resolve(f);
  cudaDeviceSynchronize();
  f->pt.report(f->ctx->rank);
  for (int r = 0; r < f->ctx->world; ++r)
    if (r != f->ctx->rank && !f->ctx->loop) {
      if (f->peer_base[r] && f->spec.exchange == BW_XCHG_P2P) cudaIpcCloseMemHandle(f->peer_base[r]);
      if (f->precv_peer[r]) cudaIpcCloseMemHandle(f->precv_peer[r]);
    }
  void* dev[] = {f->t.hot, f->t.p1, f->t.closed_upto, f->t.aux, f->t.nodes, f->t.node_acc2, f->t.free_stack, f->t.dirty, f->d_ctr, f->e.c_key,
                 f->e.c_wid, f->e.c_acc, f->e.c_count, f->e.c_seq, f->e.c_epoch, f->e.l_key, f->e.l_wid, f->e.l_val,
                 f->e.l_ts, f->e.l_seq, f->e.l_epoch, f->d_rmin, f->d_rmax, f->d_rbad, f->d_verdict, f->d_kflat,
                 f->d_ksorted, f->d_tsflat, f->d_tssorted, f->d_prefmax, f->d_idx, f->d_idxsorted, f->d_late, f->d_cub,
                 f->d_sk, f->d_sk2, f->d_gather, f->d_perm, f->d_perm2, f->xchg_base, f->d_tile_counts,
                 f->d_send_counts, f->d_all_counts, f->send_keys, f->send_vals, f->send_ts, f->d_span, f->snap_dev, f->d_snap_ctr};
  for (void* p : dev)
    if (p) cudaFree(p);
  for (int i = 0; i < 2; ++i) {
    void* sp[] = {f->sb.side[i].rec, f->sb.side[i].val, f->sb.side[i].cnt, f->sb.side[i].spill, f->sb.side[i].sv};
    for (void* q : sp)
      if (q) cudaFree(q);
    if (f->ev_sv[i]) cudaEventDestroy(f->ev_sv[i]);
  }
  {
    void* sp[] = {f->sb.tile_min, f->sb.tile_max, f->sb.tile_bad, f->sb.chunk_max};
    for (void* q : sp)
      if (q) cudaFree(q);
    if (f->h_sv) cudaFreeHost(f->h_sv);
    void* lp[] = {f->late.key_bits, f->late.late_bits, f->late.ent, f->late.counters, f->late.gpre, f->late_chunk_pre, f->late.s_key, f->late.s_ts, f->late.s_idx, f->late.s_slot};
    for (void* q : lp)
      if (q) cudaFree(q);
    if (f->h_late_ctr) cudaFreeHost(f->h_late_ctr);
  }
  for (auto& s : f->stages) {
    if (s.d_keys) cudaFree(s.d_keys);
    if (s.d_vals) cudaFree(s.d_vals);
    if (s.d_ts) cudaFree(s.d_ts);
    if (s.consumed) cudaEventDestroy(s.consumed);
  }
  for (auto& s : f->slots) {
    if (s.h_keys) cudaFreeHost(s.h_keys);
    if (s.h_vals) cudaFreeHost(s.h_vals);
    if (s.h_ts) cudaFreeHost(s.h_ts);
  }
  void* host[] = {f->snap_host, f->h_ctr, f->h_verdict, f->h_all_counts, f->ho_ckey, f->ho_cacc, f->ho_ccount, f->ho_cepoch,
                  f->ho_cwid, f->ho_lkey, f->ho_lval, f->ho_lepoch, f->ho_lwid, f->ho_lts};
  for (void* p : host)
    if (p) cudaFreeHost(p);
  for (auto& t : f->timers) {
    cudaEventDestroy(t.a);
    cudaEventDestroy(t.b);
  }
  if (f->s_out) {
    cudaStreamSynchronize(f->s_out);
    cudaStreamDestroy(f->s_out);
    void* q[] = {f->fl.sk, f->fl.sk2, f->fl.gather, f->fl.perm, f->fl.perm2, f->fl.cub};
    for (void* x : q)
      if (x) cudaFree(x);
    for (auto& m : f->marks)
      if (m.ev) cudaEventDestroy(m.ev);
    if (f->h_marks) cudaFreeHost(f->h_marks);
  }
  if (f->s_compute) cudaStreamDestroy(f->s_compute);
  if (f->s_copy) cudaStreamDestroy(f->s_copy);
  if (f->s_pre) cudaStreamDestroy(f->s_pre);
  if (f->s_verdict) cudaStreamDestroy(f->s_verdict);
  if (f->ev_scattered) cudaEventDestroy(f->ev_scattered);
  if (f->s_x && f->s_x != f->s_compute) cudaStreamDestroy(f->s_x);
  if (f->ev_in) cudaEventDestroy(f->ev_in);
  if (f->ev_gen) cudaEventDestroy(f->ev_gen);
  if (f->ev_pre) cudaEventDestroy(f->ev_pre);
  if (f->ev_h2d) cudaEventDestroy(f->ev_h2d);
  delete f;
}

// ---------------------------------------------------------------------------
// ingest
// ---------------------------------------------------------------------------
bw_status bw_ingest_acquire(bw_fold* f, uint64_t max_rows, bw_batch* out) {
  if (!f || !out) return BW_ERR_SPEC;
  bw_ctx* ctx = f->ctx;
  if (max_rows > f->spec.max_batch_rows) FAIL(f, BW_ERR_SPEC, "acquire: %llu rows > max_batch_rows", (unsigned long long)max_rows);
  CU(ctx, cudaSetDevice(ctx->device));
  const u32 nslots = f->spec.ring_slots > 0 ? (u32)f->spec.ring_slots : 3u;
  u32 pick = ~0u;
  for (u32 i = 0; i < f->slots.size(); ++i)
    if (!f->slots[i].acquired) {
      pick = i;
      break;
    }
  if (pick == ~0u) {
    if (f->slots.size() >= nslots) FAIL(f, BW_ERR_STATE, "all %u ingest slots are acquired; commit one first", nslots);
    Slot s;
    const size_t rows = f->spec.max_batch_rows;
    CU(ctx, cudaHostAlloc((void**)&s.h_keys, rows * 8, cudaHostAllocDefault));
    if (f->has_vals) CU(ctx, cudaHostAlloc(&s.h_vals, rows * (size_t)f->val_bytes, cudaHostAllocDefault));
    if (f->has_ts) CU(ctx, cudaHostAlloc((void**)&s.h_ts, rows * 8, cudaHostAllocDefault));
    f->slots.push_back(s);
    pick = (u32)f->slots.size() - 1;
  }
  Slot& s = f->slots[pick];
  s.acquired = true;
  out->keys = s.h_keys;
  out->vals = s.h_vals;
  out->ts_us = s.h_ts;
  out->capacity = f->spec.max_batch_rows;
  out->slot = pick;
  out->reserved = 0;
  return BW_OK;
}

// CUDA-event pair for one kernel launch of activation `batch_no`.  Every record with timing drains the stream for a few
// microseconds, so only every timer_stride-th activation is timed (env BW_TIMER_STRIDE, default 4): the averages in bw_stats
// are over that sample.
static EventPair* next_timer(bw_fold* f, u32 batch_no) {
  if (f->timer_stride > 1 && batch_no % f->timer_stride != 0) return nullptr;
  if (f->timers_used == f->timers.size()) {
    if (f->timers.size() >= 4096) return nullptr;
    EventPair ep;
    if (cudaEventCreate(&ep.a) != cudaSuccess || cudaEventCreate(&ep.b) != cudaSuccess) return nullptr;
    ep.rows = 0;
    ep.kind = 0;
    f->timers.push_back(ep);
  }
  return &f->timers[f->timers_used++];
}


// Partition + exchange of this rank's rows; fills `bv` with the received segments.
static bw_status exchange(bw_fold* f, const u64* d_keys, const void* d_vals, const i64* d_ts, u64 rows, BatchView* bv) {
  bw_ctx* ctx = f->ctx;
  const int W = ctx->world, R = ctx->rank;
  // Partition + exchange run on their own stream so that the scatter of activation b+1 (NVLink-bound)
  // overlaps the fold of activation b.  The producer of the input columns is ordered before it through
  // ev_src_ready; the barrier waits for this rank's fold of the previous activation, which is what makes
  // the double-buffered receive regions safe to overwrite two activations later.
  cudaStream_t s = f->s_x;
  CU(ctx, cudaStreamWaitEvent(s, f->ev_src_ready, 0));
  const int buf = f->xbuf;
  f->xbuf ^= 1;
  XLayout L = xlayout(f);
  PartIn in;
  in.keys = d_keys;
  in.vals = d_vals;
  in.ts = f->has_ts ? d_ts : nullptr;
  in.n = rows;
  in.val_bytes = d_vals ? f->val_bytes : 0;
  in.world = W;
  PartOut po;
  memset(&po, 0, sizeof po);
  po.region_cap = f->region_cap;
  const bool p2p = f->spec.exchange == BW_XCHG_P2P;
  const bool hv = d_vals != nullptr;  // counts may come without a value column
  for (int d = 0; d < W; ++d) {
    if (p2p) {
      char* base = (char*)f->peer_base[d];
      po.keys[d] = (u64*)(base + L.keys_off[buf]) + (size_t)R * f->region_cap;
      po.vals[d] = hv ? (void*)(base + L.vals_off[buf] + (size_t)R * f->region_cap * f->val_bytes) : nullptr;
      po.ts[d] = f->has_ts ? (i64*)(base + L.ts_off[buf]) + (size_t)R * f->region_cap : nullptr;
      po.counts[d] = (u64*)(base + L.counts_off[buf]) + R;
    } else {
      po.keys[d] = f->send_keys + (size_t)d * f->region_cap;
      po.vals[d] = hv ? (void*)((char*)f->send_vals + (size_t)d * f->region_cap * f->val_bytes) : nullptr;
      po.ts[d] = f->has_ts ? f->send_ts + (size_t)d * f->region_cap : nullptr;
      po.counts[d] = f->d_send_counts + d;
    }
  }
  const u64 ntiles = (rows + BW_PART_TILE - 1) / BW_PART_TILE;
  int grid = (int)std::min<u64>(std::max<u64>(ntiles, 1), (u64)ctx->sm_count * 8);
  f->pt.mark(0, 0, s);
  k_part_hist<<<grid, BW_PART_THREADS, 0, s>>>(in, f->d_tile_counts);
  k_part_scan<<<W, 1024, 0, s>>>(rows, W, f->d_tile_counts, po, f->d_ctr);
  const size_t stage_bytes = (size_t)BW_PART_TILE * (8 + (size_t)in.val_bytes + (in.ts ? 8 : 0));
  k_part_scatter<<<grid, BW_PART_THREADS, stage_bytes, s>>>(in, f->d_tile_counts, po);
  CU(ctx, cudaGetLastError());
  f->st.kernel_launches += 3;
  f->pt.mark(0, 1, s);
  char* mine = (char*)f->xchg_base;
  u64* my_counts = (u64*)(mine + L.counts_off[buf]);
  if (f->fold_recorded) CU(ctx, cudaStreamWaitEvent(s, f->ev_fold_done, 0));
  f->pt.mark(1, 0, s);
  if (p2p) {
    // every rank's stores are complete once it enters this collective (stream
    // order); its completion here means all peers have entered it.
    {
      bw_status cst = coll_barrier(ctx, f->d_verdict, s);
      if (cst != BW_OK) return cst;
    }
  } else {
    NC(ctx, ncclAllGather(f->d_send_counts, f->d_all_counts, BW_MAX_WORLD, ncclUint64, ctx->comm, s));
    CU(ctx, cudaMemcpyAsync(f->h_all_counts, f->d_all_counts, sizeof(u64) * BW_MAX_WORLD * W, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
    u64 recv_counts[BW_MAX_WORLD];
    NC(ctx, ncclGroupStart());
    for (int r = 0; r < W; ++r) {
      const u64 nsend = f->h_all_counts[(size_t)R * BW_MAX_WORLD + r];
      const u64 nrecv = f->h_all_counts[(size_t)r * BW_MAX_WORLD + R];
      recv_counts[r] = nrecv;
      u64* rk = (u64*)(mine + L.keys_off[buf]) + (size_t)r * f->region_cap;
      NC(ctx, ncclSend(f->send_keys + (size_t)r * f->region_cap, nsend, ncclUint64, r, ctx->comm, s));
      NC(ctx, ncclRecv(rk, nrecv, ncclUint64, r, ctx->comm, s));
      if (hv) {
        char* rv = mine + L.vals_off[buf] + (size_t)r * f->region_cap * f->val_bytes;
        NC(ctx, ncclSend((char*)f->send_vals + (size_t)r * f->region_cap * f->val_bytes, nsend * f->val_bytes, ncclChar, r,
                         ctx->comm, s));
        NC(ctx, ncclRecv(rv, nrecv * f->val_bytes, ncclChar, r, ctx->comm, s));
      }
      if (f->has_ts) {
        i64* rt = (i64*)(mine + L.ts_off[buf]) + (size_t)r * f->region_cap;
        NC(ctx, ncclSend(f->send_ts + (size_t)r * f->region_cap, nsend, ncclInt64, r, ctx->comm, s));
        NC(ctx, ncclRecv(rt, nrecv, ncclInt64, r, ctx->comm, s));
      }
    }
    NC(ctx, ncclGroupEnd());
    CU(ctx, cudaMemcpyAsync(my_counts, recv_counts, sizeof(u64) * W, cudaMemcpyHostToDevice, s));
    // recv_counts is a stack array: make the copy complete before returning
    CU(ctx, cudaStreamSynchronize(s));
  }
  f->pt.mark(1, 1, s);
  memset(bv, 0, sizeof *bv);
  bv->nseg = W;
  bv->counts_on_device = 1;
  bv->d_counts = my_counts;
  bv->max_rows = f->max_recv_rows;
  for (int r = 0; r < W; ++r) {
    bv->keys[r] = (const u64*)(mine + L.keys_off[buf]) + (size_t)r * f->region_cap;
    bv->vals[r] = hv ? (const void*)(mine + L.vals_off[buf] + (size_t)r * f->region_cap * f->val_bytes) : nullptr;
    bv->ts[r] = f->has_ts ? (const i64*)(mine + L.ts_off[buf]) + (size_t)r * f->region_cap : nullptr;
  }
  return BW_OK;
}

// A kernel that may be placed while the kernel before it on the stream is still running (programmatic dependent
// launch): its launch and its prologue overlap the other's tail.  It must call bw_pdl_wait (bw_common.cuh) in every block.
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// Work queued on `s` after this sees every verdict queued so far (one GPU: they run on s_verdict).
static bw_status verdict_join(bw_fold* f, cudaStream_t s) {
  if (f->ev_sv_last) CU(f->ctx, cudaStreamWaitEvent(s, f->ev_sv_last, 0));
  return BW_OK;
}

// K4 for the keys the fold marked; its last block does the end-of-activation resets
static bw_status close_stage(bw_fold* f, u64 ord, u32 batch_no, StreamVerdict* sv) {
  bw_ctx* ctx = f->ctx;
  f->pt.mark(4, 0, f->s_compute);
  CU(ctx, launch_pdl(k_close_dirty, f->close_grid, 256, 0, f->s_compute, f->t, f->p, f->e, ord, batch_no, sv));
  f->st.kernel_launches++;
  f->pt.mark(4, 1, f->s_compute);
  return BW_OK;
}

// The direct fold kernel over a clean activation, in sub-ranges when it spans several panes.
static bw_status direct_fold(bw_fold* f, const BatchView& bv, u64 known, u32 batch_no, u64 ord, i64 tmin, i64 tmax) {
  bw_ctx* ctx = f->ctx;
  const u64 tile = (u64)BW_FOLD_THREADS * BW_FOLD_UNROLL;
  // Fold + close in sub-ranges of the activation (by arrival index, resolved on the device so
  // that it also works on exchanged rows whose counts the host never sees).  Windows a key has
  // left are closed -- and its newest pane promoted into the hot slot -- between sub-ranges, so
  // an activation that spans several windows (8 ranks x 2^24 rows of C1 = 134 s of event time
  // per activation) keeps hitting the two direct panes instead of the overflow list.  Rows are
  // identical: a pane closed early would also close at the end (the watermark only grows, and
  // the pane holding max_ts never closes).  One sub-range per pane of event-time span, for
  // in-order streams; activations inside one pane (C1 on one GPU) are not split.
  u32 n_sub = 1;
  if (f->sub_rows != ~0ULL) {
    n_sub = (u32)std::min<u64>((known + f->sub_rows - 1) / f->sub_rows, 64);
  } else if (f->sub_auto && f->p.track_wm) {
    if (tmax > tmin) {
      const u64 panes = (u64)(tmax - tmin) / (u64)f->p.pane_us + (((u64)(tmax - tmin) % (u64)f->p.pane_us) ? 1 : 0);
      n_sub = (u32)std::min<u64>(panes, 8);
      n_sub = (u32)std::min<u64>(n_sub, std::max<u64>(known >> 20, 1));  // keep sub-ranges >= 2^20 rows
    }
  }
  if (n_sub < 1) n_sub = 1;
  for (u32 i = 0; i < n_sub; ++i) {
    const u64 n_hi = (known * (i + 1ULL)) / n_sub, n_lo = (known * (u64)i) / n_sub;
    EventPair* ep = next_timer(f, batch_no);
    if (ep) {
      ep->rows = (ctx->world > 1) ? 0 : (n_hi - n_lo);
      ep->kind = 0;
      CU(ctx, cudaEventRecord(ep->a, f->s_compute));
    }
    int grid = (int)std::min<u64>((n_hi - n_lo + tile - 1) / tile + 1, (u64)f->fold_grid);
    f->fold_kernel<<<grid, BW_FOLD_THREADS, 0, f->s_compute>>>(bv, f->t, f->p, batch_no, i, n_sub);
    CU(ctx, cudaGetLastError());
    if (ep) CU(ctx, cudaEventRecord(ep->b, f->s_compute));
    f->st.kernel_launches++;
    f->st.fold_launches++;
    if (f->pt.on && ep) {
      f->pt.ev[3][0].push_back(ep->a);
      f->pt.ev[3][1].push_back(ep->b);
    }
    if (i + 1 < n_sub) {
      k_close_dirty<<<f->close_grid, 256, 0, f->s_compute>>>(f->t, f->p, f->e, ord, batch_no, nullptr);
      f->st.kernel_launches++;
    }
  }
  return BW_OK;
}

// ---- streaming path (bw_stream.cuh): queue scatter + verdict now, the fold stage one activation later ----
static bool stream_usable(const bw_fold* f, const u64* d_keys, const void* d_vals, const i64* d_ts, u64 rows) {
  if (!f->stream_ok || rows == 0 || rows > f->spec.max_batch_rows) return false;
  // 128-bit loads of column pairs
  if (((uintptr_t)d_keys & 15) || ((uintptr_t)d_vals & 15) || ((uintptr_t)d_ts & 15)) return false;
  if (f->p.ts_from_value == 1 && !d_vals) return false;
  if (f->sb.val_bytes && !d_vals) return false;
  return true;
}

static bw_status stream_front(bw_fold* f, const u64* d_keys, const void* d_vals, const i64* d_ts, u64 rows, u32 batch_no, int side,
                              const u32* late_bits = nullptr, i64 ts0 = 0) {
  bw_ctx* ctx = f->ctx;
  const StreamBufs& sb = f->sb;
  cudaStream_t s = f->s_compute;
  ScatterArgs A;
  memset(&A, 0, sizeof A);
  A.keys = d_keys;
  A.vals = d_vals;
  A.ts = f->has_ts ? d_ts : nullptr;
  A.n = rows;
  A.out = sb.side[side];
  A.nb = sb.nb;
  A.nlanes = sb.nlanes;
  A.lane_cap = sb.lane_cap;
  A.spill_cap = sb.spill_cap;
  A.tile_min = sb.tile_min + (size_t)side * sb.tiles_cap;
  A.tile_max = sb.tile_max + (size_t)side * sb.tiles_cap;
  A.tile_bad = sb.tile_bad + (size_t)side * sb.tiles_cap;
  A.chunk_max = sb.chunk_max + (size_t)side * sb.tiles_cap * BW_SC_WARPS;
  A.late_bits = late_bits;  // second run over an activation with late rows: they are left out
  A.ts0_set = late_bits ? 1u : 0u;
  A.ts0 = ts0;
  A.cap = f->t.cap;
  A.seg_shift = f->t.seg_shift;
  A.nstage = (u32)f->scatter_nstage;
  A.rec_idx = f->p.seq_by_id ? 0u : 1u;
  if (const char* e = getenv("BW_SC_DBG")) A.dbg = (u32)atoi(e);
  A.stg_cap = f->scatter_stg_cap;
  A.stg_every = f->scatter_stg_every;
  A.batch_no = batch_no;
  A.world = (u32)ctx->world;
  A.nb_local = f->nb_local;
  const bool multi = ctx->world > 1;
  // multi-GPU: every rank goes through here for every activation (the verdicts are gathered collectively); a rank
  // whose columns the scatter cannot read (no rows, unaligned) sends no rows / asks everyone for the legacy path
  const bool usable = stream_usable(f, d_keys, d_vals, d_ts, rows);
  VerdictGather* vg = multi ? f->d_vg_local + side : nullptr;
  const u64 T = BW_SC_TILE;
  const u64 ntiles = usable ? (rows + T - 1) / T : 0;
  const int grid = (int)std::min<u64>(ntiles, (u64)std::min<u32>((u32)f->scatter_grid, sb.nlanes));
  f->last_scatter_grid = (u32)grid;
  if (multi && !usable && rows) CU(ctx, cudaMemsetAsync(&sb.side[side].sv->flags, 0xFF, sizeof(u32), s));  // every flag: legacy path
  EventPair* ep = next_timer(f, batch_no);
  if (ep) {
    ep->rows = rows;
    ep->kind = 1;
    CU(ctx, cudaEventRecord(ep->a, s));
  }
  f->pt.mark(5, 0, s);
  if (grid) CU(ctx, launch_pdl(f->scatter_kernel, grid, BW_SC_THREADS, f->scatter_smem, s, A, f->p));
  if (ep) CU(ctx, cudaEventRecord(ep->b, s));  // (the scatter kernel alone: the one-block verdict is timed apart)
  // One GPU: the verdict goes to its own stream once the scatter is done, and s_compute goes straight on to the fold
  // stage of the activation before.  Multi-GPU: it stays on s_compute (the gather behind it is a collective there).
  cudaStream_t vs = s;
  if (!multi) {
    vs = f->s_verdict;
    CU(ctx, cudaEventRecord(f->ev_scattered, s));
    CU(ctx, cudaStreamWaitEvent(vs, f->ev_scattered, 0));
  }
  EventPair* ev = next_timer(f, batch_no);
  if (ev) {
    ev->rows = 0;
    ev->kind = 2;
    CU(ctx, cudaEventRecord(ev->a, vs));
  }
  if (f->p.ts_from_value == 2) k_verdict_none<<<1, 1, 0, vs>>>(f->p, f->d_ctr, sb.side[side].sv, vg, rows);
  else
    k_verdict<<<1, 1024, 0, vs>>>(A.tile_min, A.tile_max, A.tile_bad, (u32)ntiles, f->p, f->d_ctr, sb.side[side].sv,
                                  f->has_ts ? d_ts : nullptr, (const u64*)d_vals, vg);
  CU(ctx, cudaGetLastError());
  f->pt.mark(5, 1, vs);
  if (ev) CU(ctx, cudaEventRecord(ev->b, vs));
  f->st.kernel_launches += 2;
  CU(ctx, cudaMemcpyAsync(&f->h_sv[side], sb.side[side].sv, sizeof(StreamVerdict), cudaMemcpyDeviceToHost, vs));
  if (multi) f->vg_pending[side] = true;  // gathered by the next collective on the stream (gather_verdict)
  CU(ctx, cudaEventRecord(f->ev_sv[side], vs));
  if (!multi) f->ev_sv_last = f->ev_sv[side];
  return BW_OK;
}

static bw_status slow_path(bw_fold* f, const BatchView& bv, u64 total, u64 epoch_ord, u32 batch_no);

static bw_status slow_path(bw_fold* f, const BatchView& bv, u64 total, u64 epoch_ord, u32 batch_no);

// The direct path of one activation, start to finish: (world > 1: partition + exchange of the rows) -> lateness pass ->
// k_fold or the exact path -> K4.
static bw_status legacy_batch(bw_fold* f, const u64* d_keys, const void* d_vals, const i64* d_ts, u64 rows, u32 batch_no, u64 ord, Stage* stage) {
  bw_ctx* ctx = f->ctx;
  BatchView bv;
  memset(&bv, 0, sizeof bv);
  u64 max_total = rows;
  cudaStream_t pre_stream = f->s_pre;
  if (ctx->world > 1) {
    bw_status st = exchange(f, d_keys, d_vals, d_ts, rows, &bv);
    if (st != BW_OK) return st;
    max_total = f->max_recv_rows;
    pre_stream = f->s_x;  // the verdict is computed right behind the exchange, beside the previous fold
  } else {
    bv.nseg = 1;
    bv.keys[0] = d_keys;
    bv.vals[0] = d_vals;
    bv.ts[0] = f->has_ts ? d_ts : nullptr;
    bv.h_counts[0] = rows;
    bv.max_rows = rows;
    f->st.rows_received += rows;
  }
  bool clean = true;
  if (f->p.track_wm && max_total > 0) {
    if (pre_stream != f->s_compute && ctx->world == 1 && f->pre_wait) CU(ctx, cudaStreamWaitEvent(pre_stream, f->pre_wait, 0));
    {  // (k_prepass_scan chains from Counters::gmax_ts)
      bw_status vst = verdict_join(f, pre_stream);
      if (vst != BW_OK) return vst;
    }
    const u64 nranges = (max_total + BW_RANGE_ROWS - 1) / BW_RANGE_ROWS;
    // one warp per 2048-row range; cap at 64 warps per SM in total (the block size is small so that a block fits beside the fold)
    int grid = (int)std::min<u64>((nranges * 32 + BW_PRE_THREADS - 1) / BW_PRE_THREADS, (u64)ctx->sm_count * (2048 / BW_PRE_THREADS));
    if (grid < 1) grid = 1;
    f->pt.mark(2, 0, pre_stream);
    k_prepass_ranges<<<grid, BW_PRE_THREADS, 0, pre_stream>>>(bv, f->p, f->d_rmin, f->d_rmax, f->d_rbad);
    k_prepass_scan<<<1, 1024, 0, pre_stream>>>(bv, f->p, f->d_rmin, f->d_rmax, f->d_rbad, f->d_ctr, f->d_verdict, f->d_span);
    CU(ctx, cudaGetLastError());
    f->st.kernel_launches += 2;
    f->pt.mark(2, 1, pre_stream);
    CU(ctx, cudaMemcpyAsync(f->h_verdict, f->d_verdict, sizeof(u32), cudaMemcpyDeviceToHost, pre_stream));
    CU(ctx, cudaMemcpyAsync(f->h_verdict + 4, f->d_span, 2 * sizeof(i64), cudaMemcpyDeviceToHost, pre_stream));
    CU(ctx, cudaEventRecord(f->ev_pre, pre_stream));
    CU(ctx, cudaEventSynchronize(f->ev_pre));
    clean = (*f->h_verdict != 0);
    if (pre_stream != f->s_compute) CU(ctx, cudaStreamWaitEvent(f->s_compute, f->ev_pre, 0));
  }
  if (ctx->world > 1) {  // the fold may start once the exchange (and the verdict pass behind it) is done
    CU(ctx, cudaEventRecord(f->ev_xchg_done, f->s_x));
    CU(ctx, cudaStreamWaitEvent(f->s_compute, f->ev_xchg_done, 0));
  }
  if (max_total > 0) {
    if (clean) {
      const u64 known = (ctx->world == 1) ? rows : max_total;
      const i64 tmin = ((const i64*)(f->h_verdict + 4))[0], tmax = ((const i64*)(f->h_verdict + 4))[1];
      bw_status st = direct_fold(f, bv, known, batch_no, ord, f->p.track_wm ? tmin : 0, f->p.track_wm ? tmax : 0);
      if (st != BW_OK) return st;
    } else {
      u64 total = rows;
      if (ctx->world > 1) {
        u64 hc[BW_MAX_WORLD];
        CU(ctx, cudaMemcpyAsync(hc, bv.d_counts, sizeof(u64) * ctx->world, cudaMemcpyDeviceToHost, f->s_compute));
        CU(ctx, cudaStreamSynchronize(f->s_compute));
        total = 0;
        for (int r = 0; r < ctx->world; ++r) total += hc[r];
      }
      bw_status st = slow_path(f, bv, total, ord, batch_no);
      if (st != BW_OK) return st;
      f->st.slow_batches++;
    }
    bw_status st = close_stage(f, ord, batch_no, nullptr);
    if (st != BW_OK) return st;
  }
  if (ctx->world > 1) {
    CU(ctx, cudaEventRecord(f->ev_fold_done, f->s_compute));
    f->fold_recorded = true;
  } else {
    bw_status mst = mark_rows(f, ord);
    if (mst != BW_OK) return mst;
  }
  if (stage) {
    CU(ctx, cudaEventRecord(stage->consumed, f->s_compute));
    stage->used = true;
  }
  return BW_OK;
}


// One collective per activation: the all-gather that brings every rank's verdict of the activation just scattered is
// also the barrier behind the previous activation's combine (a rank enters it after its peer stores, in stream order).
static bw_status gather_verdict(bw_fold* f, int side) {
  bw_ctx* ctx = f->ctx;
  cudaStream_t s = f->s_compute;
  const int W = ctx->world;
  VerdictGather* all = f->d_vg_all + (size_t)side * W;
  {
    bw_status cst = coll_allgather(ctx, f->d_vg_local + side, all, sizeof(VerdictGather), s);
    if (cst != BW_OK) return cst;
  }
  CU(ctx, cudaMemcpyAsync(f->h_vg + (size_t)side * W, all, sizeof(VerdictGather) * W, cudaMemcpyDeviceToHost, s));
  if (!f->ev_vg[side]) CU(ctx, cudaEventCreateWithFlags(&f->ev_vg[side], cudaEventDisableTiming));
  CU(ctx, cudaEventRecord(f->ev_vg[side], s));
  f->vg_pending[side] = false;
  return BW_OK;
}

// Multi-GPU fold stage of the deferred activation.  Every rank has the same gathered verdicts, so every rank takes
// the same branch (the collectives below line up): either combine -> partials over NVLink -> barrier -> merge, or
// the legacy path (partition + exchange of the raw rows, direct / exact fold).
static bw_status stream_resolve_multi(bw_fold* f, const Deferred& d) {
  bw_ctx* ctx = f->ctx;
  const StreamBufs& sb = f->sb;
  const FoldParams& p = f->p;
  cudaStream_t s = f->s_compute;
  const int W = ctx->world, R = ctx->rank;
  const StreamVerdict sv = f->h_sv[d.side];
  // this activation's verdicts: gathered by the previous activation's exchange barrier, else (first activation, or
  // after a flush) by a collective of their own
  if (f->vg_pending[d.side]) {
    bw_status gst = gather_verdict(f, d.side);
    if (gst != BW_OK) return gst;
  }
  CU(ctx, cudaEventSynchronize(f->ev_vg[d.side]));
  const int next_side = d.side ^ 1;  // the activation scattered after this one (if any) waits for its gather
  const VerdictGather* vg = f->h_vg + (size_t)d.side * W;
  // chain the ranks' slices in source order: the arrival order at every destination (bw_prepass.cuh's rule)
  i64 running = f->h_gmax, gmin = INT64_MAX, gmax = INT64_MIN;
  bool bad = false, unfit = false;
  for (int r = 0; r < W; ++r) {
    if (vg[r].flags || vg[r].n_spill) unfit = true;  // a row some scatter set aside belongs to another rank's table
    if (vg[r].tmax < vg[r].tmin) continue;            // no rows on that rank
    if (vg[r].bad || vg[r].tmin < bw_sub_sat(running, p.wait_us)) bad = true;
    running = std::max(running, vg[r].tmax);
    gmin = std::min(gmin, vg[r].tmin);
    gmax = std::max(gmax, vg[r].tmax);
    // the combine folds a rank's slice in one pass: two panes
    if (bw_floordiv(vg[r].tmax - p.align_us, p.pane_us) - bw_floordiv(vg[r].tmin - p.align_us, p.pane_us) > 1) unfit = true;
  }
  const bool any_rows = gmax >= gmin;
  const bool clean = !p.track_wm || !bad;
  i64 q_lo = 0, q_hi = 0;
  if (any_rows) {
    q_lo = bw_floordiv(gmin - p.align_us, p.pane_us);
    q_hi = bw_floordiv(gmax - p.align_us, p.pane_us);
    if ((u64)(gmax - gmin) >= 0x7FFFFFF0ULL || q_hi - q_lo >= 2 * 64) unfit = true;
  }
  f->h_gmax = running;
  k_set_gmax<<<1, 1, 0, s>>>(f->d_ctr, running);  // (the legacy path's lateness pass chains from the same maximum)
  f->st.kernel_launches++;
  if (!clean || unfit) {
    if (f->vg_pending[next_side]) {
      bw_status gst = gather_verdict(f, next_side);
      if (gst != BW_OK) return gst;
    }
    bw_status st = legacy_batch(f, d.d_keys, d.d_vals, d.d_ts, d.rows, d.batch_no, d.ord, d.stage);
    if (st != BW_OK) return st;
    k_stream_reset<<<1, 1, 0, s>>>(f->t, sb.side[d.side].sv);
    k_set_gmax<<<1, 1, 0, s>>>(f->d_ctr, running);
    return BW_OK;
  }
  f->st.rows_received += d.rows;  // (this rank's share of the rows arrives as partials)
  SegArgs A;
  memset(&A, 0, sizeof A);
  A.in = sb.side[d.side];
  A.nb = sb.nb;
  A.nlanes = sb.nlanes;
  A.lane_cap = sb.lane_cap;
  A.nlanes_used = d.lanes;
  A.spill_cap = sb.spill_cap;
  A.val_bytes = sb.val_bytes;
  A.seg_shift = f->t.seg_shift;
  A.world = (u32)W;
  A.rank = (u32)R;
  A.nb_local = f->nb_local;
  A.part_cap = f->part_cap;
  A.batch_no = d.batch_no;
  A.epoch = d.ord;
  for (int r = 0; r < W; ++r) {
    char* base = (char*)f->precv_peer[r];
    A.pcnt_out[r] = (u32*)(base + f->precv_cnt_off[d.side]) + (size_t)R * f->nb_local;
    A.pout[r] = (Partial*)(base + f->precv_rec_off[d.side]) + (size_t)R * f->nb_local * f->part_cap;
  }
  A.pcnt_in = (const u32*)((char*)f->precv_base + f->precv_cnt_off[d.side]);
  A.pin = (const Partial*)((char*)f->precv_base + f->precv_rec_off[d.side]);
  EventPair* ep = next_timer(f, d.batch_no);
  if (ep) {
    ep->rows = d.rows;
    ep->kind = 0;
    CU(ctx, cudaEventRecord(ep->a, s));
  }
  // combine this rank's slice (one pass over its own two panes) and store the partials in their owners' regions
  A.ts0 = sv.ts0;
  A.q_lo = (sv.tmax >= sv.tmin) ? bw_floordiv(sv.tmin - p.align_us, p.pane_us) : 0;
  A.npass = 1;
  f->pt.mark(6, 0, s);
  f->combine_kernel<<<(int)std::min<u32>(sb.nb, (u32)f->combine_grid), BW_SF_THREADS, f->segfold_smem, s>>>(A, f->t, f->p, f->e);
  CU(ctx, cudaGetLastError());
  // every rank's partials are in place once every rank has entered this collective -- which also carries the verdicts
  // of the activation scattered after this one
  f->pt.mark(1, 0, s);
  if (f->vg_pending[next_side]) {
    bw_status gst = gather_verdict(f, next_side);
    if (gst != BW_OK) return gst;
  } else {
    bw_status cst = coll_barrier(ctx, f->d_barrier_word, s);
    if (cst != BW_OK) return cst;
  }
  f->pt.mark(1, 1, s);
  // merge what every source left for this rank's segments, in source order, over the activation's whole span
  A.nb = f->nb_local;
  A.ts0 = any_rows ? gmin : p.align_us;
  A.q_lo = q_lo;
  A.npass = (u32)((q_hi - q_lo) / 2 + 1);
  f->merge_kernel<<<(int)std::min<u32>(f->nb_local, (u32)f->merge_grid), BW_SF_THREADS, f->segfold_smem, s>>>(A, f->t, f->p, f->e);
  CU(ctx, cudaGetLastError());
  f->pt.mark(6, 1, s);
  if (ep) CU(ctx, cudaEventRecord(ep->b, s));
  f->pt.mark(7, 0, s);
  k_spill<<<ctx->sm_count, 256, 0, s>>>(f->t, f->p, sb.side[d.side].spill, sb.side[d.side].sv, sb.spill_cap, d.batch_no, 0u, 0xFFFFFFFFu);
  f->st.kernel_launches += 3;
  f->st.fold_launches++;
  f->st.combined_folds++;
  bw_status st = close_stage(f, d.ord, d.batch_no, sb.side[d.side].sv);
  f->pt.mark(7, 1, s);
  if (d.stage) {
    CU(ctx, cudaEventRecord(d.stage->consumed, s));
    d.stage->used = true;
  }
  return st;
}

// The fold stage of the deferred activation: the segment fold when its verdict allows, else what the
// direct path would have done (its scatter output is dropped; the input columns are still there).
// An activation the verdict could not prove clean (one GPU): find its late rows without sorting it (bw_late.cuh), then
// scatter it again without them.  *ok: *sv is now the verdict of the rows that are left -- none of them late, so the
// streaming fold is exact for them -- and the late rows wait in f->late for k_late_emit.  Not ok (more suspects than
// the table takes, or the second scatter raised a flag): nothing has been folded or emitted, take the sort path.
static bw_status late_split(bw_fold* f, const Deferred& d, const BatchView& bv, StreamVerdict* sv, bool* ok) {
  bw_ctx* ctx = f->ctx;
  const StreamBufs& sb = f->sb;
  cudaStream_t s = f->s_compute;
  *ok = false;
  {
    bw_status vst = verdict_join(f, s);
    if (vst != BW_OK) return vst;
  }
  LateBufs& L = f->late;
  if (!f->late_ready) {
    const u64 maxr = f->spec.max_batch_rows;
    L.cap = (u32)std::max<u64>(1024, maxr / 16);
    u32 M = 2048;
    while (M < 2 * L.cap) M <<= 1;
    L.m_mask = M - 1;
    u32 kb = 1u << 16;
    while (kb < 16 * L.cap && kb < (1u << 27)) kb <<= 1;
    L.kb_mask = kb - 1;
    CU(ctx, dmalloc(&L.key_bits, kb / 32));
    CU(ctx, dmalloc(&L.late_bits, maxr / 32 + 2));
    CU(ctx, dmalloc(&L.ent, M));
    CU(ctx, cudaMemsetAsync(L.ent, 0, (size_t)M * sizeof(LateEnt), s));  // generation 0: every entry free, once
    CU(ctx, dmalloc(&L.counters, 2));
    CU(ctx, dmalloc(&L.s_key, L.cap));
    CU(ctx, dmalloc(&L.s_ts, L.cap));
    CU(ctx, dmalloc(&L.s_idx, L.cap));
    CU(ctx, dmalloc(&L.s_slot, L.cap));
    CU(ctx, dmalloc(&L.gpre, sb.tiles_cap));
    CU(ctx, dmalloc(&f->late_chunk_pre, (size_t)sb.tiles_cap * BW_SC_WARPS));
    CU(ctx, cudaHostAlloc((void**)&f->h_late_ctr, 2 * sizeof(u32), cudaHostAllocDefault));
    f->late_ready = true;
  }
  const u64 rows = d.rows;
  const u32 ntiles = (u32)((rows + BW_SC_TILE - 1) / BW_SC_TILE);
  CU(ctx, cudaMemsetAsync(L.key_bits, 0, ((size_t)L.kb_mask + 1) / 8, s));
  CU(ctx, cudaMemsetAsync(L.late_bits, 0, (rows / 32 + 2) * sizeof(u32), s));
  L.gen = d.batch_no + 1u;  // (batch numbers of a fold never repeat)
  CU(ctx, cudaMemsetAsync(L.counters, 0, 2 * sizeof(u32), s));
  const size_t toff = (size_t)d.side * sb.tiles_cap;
  const int wide = ctx->sm_count * 8;
  k_late_gpre<<<1, 1024, 0, s>>>(sb.tile_max + toff, ntiles, sv->gprev, L.gpre);
  k_late_chunkpre<<<(int)std::min<u32>((ntiles + 7u) / 8u, (u32)wide), 256, 0, s>>>(sb.chunk_max + toff * BW_SC_WARPS, L.gpre, ntiles, f->late_chunk_pre);
  k_late_suspect<<<wide, 256, 0, s>>>(bv, f->p, rows, f->late_chunk_pre, L);
  k_late_build<<<wide, 256, 0, s>>>(L);
  k_late_prefmax<<<wide, 256, 0, s>>>(bv, f->p, rows, L);
  k_late_classify<<<wide, 256, 0, s>>>(f->t, f->p, L);
  k_stream_reset<<<1, 1, 0, s>>>(f->t, sb.side[d.side].sv);  // what the first scatter set aside / flagged is void
  CU(ctx, cudaGetLastError());
  f->st.kernel_launches += 7;
  CU(ctx, cudaMemcpyAsync(f->h_late_ctr, L.counters, 2 * sizeof(u32), cudaMemcpyDeviceToHost, s));
  // base of the records' 32-bit relative timestamps: row 0 may be a late row from far back, so count from the
  // activation's newest timestamp instead
  i64 ts0 = sv->tmin;
  if (sv->tmax - (i64)0x7FFFFFF0 > ts0) ts0 = sv->tmax - (i64)0x7FFFFFF0;
  bw_status st = stream_front(f, d.d_keys, d.d_vals, d.d_ts, rows, d.batch_no, d.side, L.late_bits, ts0);
  if (st != BW_OK) return st;
  CU(ctx, cudaEventSynchronize(f->ev_sv[d.side]));
  if (f->h_late_ctr[0] > L.cap || f->h_late_ctr[1]) return BW_OK;
  const StreamVerdict sv2 = f->h_sv[d.side];
  if (sv2.flags) return BW_OK;
  *sv = sv2;
  sv->clean = 1u;
  sv->ts0 = ts0;
  *ok = true;
  return BW_OK;
}

static bw_status stream_resolve(bw_fold* f) {
  bw_ctx* ctx = f->ctx;
  Deferred d = f->dq;
  if (!d.valid) return BW_OK;
  f->dq.valid = false;
  const StreamBufs& sb = f->sb;
  cudaStream_t s = f->s_compute;
  CU(ctx, cudaEventSynchronize(f->ev_sv[d.side]));
  if (ctx->world > 1) return stream_resolve_multi(f, d);
  StreamVerdict sv = f->h_sv[d.side];
  const FoldParams& p = f->p;
  BatchView bv;
  memset(&bv, 0, sizeof bv);
  bv.nseg = 1;
  bv.keys[0] = d.d_keys;
  bv.vals[0] = d.d_vals;
  bv.ts[0] = f->has_ts ? d.d_ts : nullptr;
  bv.h_counts[0] = d.rows;
  bv.max_rows = d.rows;
  bool split = false;
  if (!sv.clean && p.track_wm && f->late_split) {
    bw_status lst = late_split(f, d, bv, &sv, &split);
    if (lst != BW_OK) return lst;
  }
  i64 q_lo = 0, q_hi = 0;
  if (sv.tmax >= sv.tmin) {
    q_lo = bw_floordiv(sv.tmin - p.align_us, p.pane_us);
    q_hi = bw_floordiv(sv.tmax - p.align_us, p.pane_us);
  }
  const bool fits = sv.clean && !sv.flags && (q_hi - q_lo) < 2 * 64;
  bw_status st = BW_OK;
  if (fits) {
    SegArgs A;
    memset(&A, 0, sizeof A);
    A.in = sb.side[d.side];
    A.nb = sb.nb;
    A.nlanes = sb.nlanes;
    A.lane_cap = sb.lane_cap;
    A.nlanes_used = d.lanes;
    A.spill_cap = sb.spill_cap;
    A.val_bytes = sb.val_bytes;
    A.seg_shift = f->t.seg_shift;
    A.ts0 = sv.ts0;
    A.q_lo = q_lo;
    A.npass = (u32)((q_hi - q_lo) / 2 + 1);
    A.batch_no = d.batch_no;
    A.epoch = d.ord;
    EventPair* ep = next_timer(f, d.batch_no);
    if (ep) {
      ep->rows = d.rows;
      ep->kind = 0;
      CU(ctx, cudaEventRecord(ep->a, s));
    }
    if (getenv("BW_DEBUG_CURSOR")) {
      std::vector<u32> hc((size_t)sb.nb * sb.nlanes);
      cudaMemcpy(hc.data(), sb.side[d.side].cnt, sizeof(u32) * hc.size(), cudaMemcpyDeviceToHost);
      u64 sum = 0;
      u32 mx = 0;
      for (u32 bb = 0; bb < sb.nb; ++bb)
        for (u32 l = 0; l < d.lanes; ++l) {
          sum += hc[(size_t)bb * sb.nlanes + l];
          mx = std::max(mx, hc[(size_t)bb * sb.nlanes + l]);
        }
      fprintf(stderr, "[bwgpu] batch %u: nb %u lanes %u lane_cap %u rows %llu in lanes %llu max %u spill %u flags %u span [%lld, %lld]\n", d.batch_no,
              sb.nb, d.lanes, sb.lane_cap, (unsigned long long)d.rows, (unsigned long long)sum, mx, sv.n_spill, sv.flags, (long long)sv.tmin,
              (long long)sv.tmax);
    }
    if (split) {
      k_late_emit<<<ctx->sm_count * 4, 256, 0, s>>>(bv, f->t, f->p, f->e, f->late, d.batch_no,
                                                                                                            d.ord);
      f->st.kernel_launches++;
      f->st.split_batches++;
    }
    const u32 n_pre = std::min<u32>(sv.n_spill, sb.spill_cap);  // rows the scatter set aside: fold them first
    if (n_pre) {
      k_spill<<<(int)std::min<u32>((n_pre + 255) / 256, (u32)ctx->sm_count * 4), 256, 0, s>>>(f->t, f->p, sb.side[d.side].spill, sb.side[d.side].sv,
                                                                                           sb.spill_cap, d.batch_no, 0u, n_pre);
      f->st.kernel_launches++;
    }
    f->pt.mark(6, 0, s);
    const int grid = (int)std::min<u32>(sb.nb, (u32)f->segfold_grid);
    CU(ctx, launch_pdl(f->segfold_kernel, grid, BW_SF_THREADS, f->segfold_smem, s, A, f->t, f->p, f->e));
    f->pt.mark(6, 1, s);
    if (ep) CU(ctx, cudaEventRecord(ep->b, s));
    f->pt.mark(7, 0, s);
    // (what the segment fold set aside; nearly always nothing, and only the device knows: the launch overlaps the
    // fold's tail and the kernel finds the list empty)
    CU(ctx, launch_pdl(k_spill, ctx->sm_count, 256, 0, s, f->t, f->p, (const SpillRec*)sb.side[d.side].spill,
                       (const StreamVerdict*)sb.side[d.side].sv, sb.spill_cap, d.batch_no, n_pre, 0xFFFFFFFFu));
    f->st.kernel_launches += 2;
    f->st.fold_launches++;
    f->st.combined_folds++;
    st = close_stage(f, d.ord, d.batch_no, sb.side[d.side].sv);
    f->pt.mark(7, 1, s);
  } else {
    // (the scatter output of this activation is simply not read)
    {  // the direct and sort paths' kernels see the verdict chain as it stood on s_compute before
      bw_status vst = verdict_join(f, s);
      if (vst != BW_OK) return vst;
    }
    if (split) sv = f->h_sv[d.side], sv.clean = 0u;  // (split, but too many panes for the segment fold: the sort path; nothing was emitted)
    if (sv.clean) {
      st = direct_fold(f, bv, d.rows, d.batch_no, d.ord, sv.tmin, sv.tmax);
    } else {
      st = slow_path(f, bv, d.rows, d.ord, d.batch_no);
      f->st.slow_batches++;
    }
    if (st == BW_OK) st = close_stage(f, d.ord, d.batch_no, sb.side[d.side].sv);
  }
  if (st == BW_OK) st = mark_rows(f, d.ord);
  if (d.stage) {
    CU(ctx, cudaEventRecord(d.stage->consumed, s));
    d.stage->used = true;
  }
  return st;
}

// Everything after the columns are on the device (on s_compute's dependency chain).
static bw_status run_batch(bw_fold* f, const u64* d_keys, const void* d_vals, const i64* d_ts, u64 rows, u64 epoch, Stage* stage) {
  bw_ctx* ctx = f->ctx;
  if (f->have_epoch && epoch < f->last_epoch) FAIL(f, BW_ERR_STATE, "epochs must not decrease (got %llu after %llu)", (unsigned long long)epoch, (unsigned long long)f->last_epoch);
  const u32 batch_no = f->batch_no++;
  if (!f->have_pending) { f->min_epoch = epoch; f->have_pending = true; }
  f->last_epoch = epoch;
  f->have_epoch = true;
  const u64 ord = epoch;
  f->st.rows_ingested += rows;
  if (ctx->world > 1 ? f->stream_ok : stream_usable(f, d_keys, d_vals, d_ts, rows)) {
    // queue this activation's scatter + verdict BEFORE looking at the previous verdict: the device
    // always has the next stage waiting while the host decides
    const int side = (int)(batch_no & 1u);
    if (ctx->world == 1) f->st.rows_received += rows;
    bw_status st = stream_front(f, d_keys, d_vals, d_ts, rows, batch_no, side);
    if (st != BW_OK) return st;
    const u32 lanes = f->last_scatter_grid;  // (resolving the previous activation may scatter it a second time)
    st = stream_resolve(f);
    if (st != BW_OK) return st;
    Deferred& d = f->dq;
    d.valid = true;
    d.side = side;
    d.d_keys = d_keys;
    d.d_vals = d_vals;
    d.d_ts = d_ts;
    d.rows = rows;
    d.ord = ord;
    d.batch_no = batch_no;
    d.lanes = lanes;
    d.stage = stage;
    return flush_rows(f);
  }
  {  // activations fold in order
    bw_status st = stream_resolve(f);
    if (st != BW_OK) return st;
  }
  bw_status st = legacy_batch(f, d_keys, d_vals, d_ts, rows, batch_no, ord, stage);
  return st == BW_OK ? flush_rows(f) : st;
}

bw_status bw_ingest_commit(bw_fold* f, const bw_batch* batch, uint64_t rows, uint64_t epoch) {
  if (!f || !batch) return BW_ERR_SPEC;
  bw_ctx* ctx = f->ctx;
  if (f->eof_done) FAIL(f, BW_ERR_STATE, "commit after eof");
  f->host_ingest = true;
  if (batch->slot >= f->slots.size() || !f->slots[batch->slot].acquired) FAIL(f, BW_ERR_STATE, "commit of a slot that is not acquired");
  if (rows > f->spec.max_batch_rows) FAIL(f, BW_ERR_SPEC, "commit: rows > max_batch_rows");
  CU(ctx, cudaSetDevice(ctx->device));
  Slot& sl = f->slots[batch->slot];
  // device staging: 3 buffers, reused once the kernels that read them are done
  if (f->stages.empty()) f->stages.resize(3);
  Stage& sg = f->stages[f->stage_next];
  f->stage_next = (f->stage_next + 1) % (u32)f->stages.size();
  if (!sg.d_keys) {
    const size_t cap = f->spec.max_batch_rows;
    CU(ctx, dmalloc(&sg.d_keys, cap));
    if (f->has_vals) CU(ctx, cudaMalloc(&sg.d_vals, cap * (size_t)f->val_bytes));
    if (f->has_ts) CU(ctx, dmalloc(&sg.d_ts, cap));
    CU(ctx, cudaEventCreateWithFlags(&sg.consumed, cudaEventDisableTiming));
  }
  if (sg.used) CU(ctx, cudaStreamWaitEvent(f->s_copy, sg.consumed, 0));
  if (rows) {
    CU(ctx, cudaMemcpyAsync(sg.d_keys, sl.h_keys, rows * 8, cudaMemcpyHostToDevice, f->s_copy));
    if (f->has_vals) CU(ctx, cudaMemcpyAsync(sg.d_vals, sl.h_vals, rows * (size_t)f->val_bytes, cudaMemcpyHostToDevice, f->s_copy));
    if (f->has_ts) CU(ctx, cudaMemcpyAsync(sg.d_ts, sl.h_ts, rows * 8, cudaMemcpyHostToDevice, f->s_copy));
  }
  CU(ctx, cudaEventRecord(f->ev_h2d, f->s_copy));
  CU(ctx, cudaStreamWaitEvent(f->s_compute, f->ev_h2d, 0));
  CU(ctx, cudaEventRecord(f->ev_in, f->s_copy));
  f->pre_wait = f->ev_in;
  CU(ctx, cudaEventRecord(f->ev_src_ready, f->s_copy));
  bw_status st = run_batch(f, sg.d_keys, sg.d_vals, sg.d_ts, rows, epoch, &sg);
  if (st != BW_OK) {  // (the slot goes back to the ring on the error paths too: repeated failures must not use it up)
    cudaEventSynchronize(f->ev_h2d);
    sl.acquired = false;
    return st;
  }
  // the pinned slot may be refilled once its H2D is done
  CU(ctx, cudaEventSynchronize(f->ev_h2d));
  sl.acquired = false;
  return BW_OK;
}

bw_status bw_ingest_device(bw_fold* f, const uint64_t* d_keys, const void* d_vals, const int64_t* d_ts_us, uint64_t rows,
                           uint64_t epoch) {
  if (!f) return BW_ERR_SPEC;
  bw_ctx* ctx = f->ctx;
  if (f->eof_done) FAIL(f, BW_ERR_STATE, "ingest after eof");
  if (rows > f->spec.max_batch_rows) FAIL(f, BW_ERR_SPEC, "ingest: rows > max_batch_rows");
  if (rows && (!d_keys || (!d_vals && (f->spec.reduction != BW_RED_COUNT || f->spec.ts_source == BW_TS_FROM_VALUE)) || (f->has_ts && !d_ts_us)))
    FAIL(f, BW_ERR_SPEC, "ingest: missing column");
  CU(ctx, cudaSetDevice(ctx->device));
  // The caller's columns are complete (bwgpu.h): the verdict pass takes no ordering from the fold's stream, so
  // it runs beside the previous activation's fold instead of behind it.  Columns written by this library's own
  // generator are ordered through its event.
  f->pre_wait = f->ev_gen;
  // multi-GPU: the caller's columns must already be complete (see bwgpu.h); no ordering with the fold's
  // stream is taken, so that this activation's exchange can overlap the previous activation's fold
  CU(ctx, cudaEventRecord(f->ev_src_ready, f->s_x));
  return run_batch(f, d_keys, d_vals, d_ts_us, rows, epoch, nullptr);
}

// ---------------------------------------------------------------------------
// exact path for an activation with possible late items
// ---------------------------------------------------------------------------
struct MaxI64 {
  __host__ __device__ __forceinline__ i64 operator()(const i64& a, const i64& b) const { return a > b ? a : b; }
};

static bw_status slow_path(bw_fold* f, const BatchView& bv, u64 total, u64 epoch_ord, u32 batch_no) {
  bw_ctx* ctx = f->ctx;
  cudaStream_t s = f->s_compute;
  if (total == 0) return BW_OK;
  if (total > f->slow_cap) {
    void* old[] = {f->d_kflat, f->d_ksorted, f->d_tsflat, f->d_tssorted, f->d_prefmax, f->d_idx, f->d_idxsorted, f->d_late};
    CU(ctx, cudaStreamSynchronize(s));
    for (void* p : old)
      if (p) cudaFree(p);
    u64 cap = std::max<u64>(total, 1024);
    CU(ctx, dmalloc(&f->d_kflat, cap));
    CU(ctx, dmalloc(&f->d_ksorted, cap));
    CU(ctx, dmalloc(&f->d_tsflat, cap));
    CU(ctx, dmalloc(&f->d_tssorted, cap));
    CU(ctx, dmalloc(&f->d_prefmax, cap));
    CU(ctx, dmalloc(&f->d_idx, cap));
    CU(ctx, dmalloc(&f->d_idxsorted, cap));
    CU(ctx, dmalloc(&f->d_late, cap));
    size_t b1 = 0, b2 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, b1, f->d_kflat, f->d_ksorted, f->d_idx, f->d_idxsorted, (int)cap, 0, 64, s);
    cub::DeviceScan::ExclusiveScanByKey(nullptr, b2, f->d_ksorted, f->d_tssorted, f->d_prefmax, MaxI64(), (i64)INT64_MIN,
                                        (int)cap, ::cuda::std::equal_to<>(), s);
    if (std::max(b1, b2) + 256 > f->cub_bytes) {  // the scratch is shared with the emission sort: only ever grow it
      if (f->d_cub) cudaFree(f->d_cub);
      f->cub_bytes = std::max(b1, b2) + 256;
      CU(ctx, cudaMalloc(&f->d_cub, f->cub_bytes));
    }
    f->slow_cap = cap;
  }
  const int grid = ctx->sm_count * 8;
  k_slow_flatten<<<grid, 256, 0, s>>>(bv, f->p, f->d_kflat, f->d_tsflat, f->d_idx);
  size_t tb = f->cub_bytes;
  CU(ctx, cub::DeviceRadixSort::SortPairs(f->d_cub, tb, f->d_kflat, f->d_ksorted, f->d_idx, f->d_idxsorted, (int)total, 0, 64, s));
  k_gather_i64<<<grid, 256, 0, s>>>(f->d_tsflat, f->d_idxsorted, f->d_tssorted, total);
  tb = f->cub_bytes;
  CU(ctx, cub::DeviceScan::ExclusiveScanByKey(f->d_cub, tb, f->d_ksorted, f->d_tssorted, f->d_prefmax, MaxI64(),
                                              (i64)INT64_MIN, (int)total, ::cuda::std::equal_to<>(), s));
  k_slow_classify<<<grid, 256, 0, s>>>(f->t, f->p, f->d_ksorted, f->d_idxsorted, f->d_tssorted, f->d_prefmax, f->d_late, total);
  k_slow_fold<<<f->fold_grid, BW_FOLD_THREADS, 0, s>>>(bv, f->t, f->p, f->e, f->d_late, batch_no, epoch_ord);
  CU(ctx, cudaGetLastError());
  f->st.kernel_launches += 4;  // ours; CUB's launches are not counted
  return BW_OK;
}

// ---------------------------------------------------------------------------
// advance / eof
// ---------------------------------------------------------------------------
static bw_status ensure_sort_cap(bw_fold* f, u64 n) {
  bw_ctx* ctx = f->ctx;
  if (n <= f->sort_cap) return BW_OK;
  void* old[] = {f->d_sk, f->d_sk2, f->d_gather, f->d_perm, f->d_perm2};
  for (void* p : old)
    if (p) cudaFree(p);
  u64 cap = std::max<u64>(n, 4096);
  CU(ctx, dmalloc(&f->d_sk, cap));
  CU(ctx, dmalloc(&f->d_sk2, cap));
  CU(ctx, dmalloc(&f->d_gather, cap));
  CU(ctx, dmalloc(&f->d_perm, cap));
  CU(ctx, dmalloc(&f->d_perm2, cap));
  size_t b = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, b, f->d_sk, f->d_sk2, f->d_perm, f->d_perm2, (int)cap, 0, 64, f->s_compute);
  if (b + 256 > f->cub_bytes) {
    if (f->d_cub) cudaFree(f->d_cub);
    f->cub_bytes = b + 256;
    CU(ctx, cudaMalloc(&f->d_cub, f->cub_bytes));
  }
  f->sort_cap = cap;
  return BW_OK;
}

// Build the reference-order permutation of n rows (LSD passes of stable radix sorts).
static bw_status order_rows(bw_fold* f, u64 n, const u64* key, const u64* seq, const u64* epoch, const i64* wid,
                            bool wid_pass, u64 n_ordinals, bool side = false) {
  bw_ctx* ctx = f->ctx;
  cudaStream_t s = side ? f->s_out : f->s_compute;
  // (the side stream sorts in its own scratch: the main one is shared with the sort path of not-clean activations)
  u64 *&d_sk = side ? f->fl.sk : f->d_sk, *&d_sk2 = side ? f->fl.sk2 : f->d_sk2;
  u32 *&d_perm = side ? f->fl.perm : f->d_perm, *&d_perm2 = side ? f->fl.perm2 : f->d_perm2;
  void* d_cub = side ? f->fl.cub : f->d_cub;
  const size_t cub_bytes = side ? f->fl.cub_bytes : f->cub_bytes;
  const int grid = ctx->sm_count * 4;
  k_iota<<<grid, 256, 0, s>>>(d_perm, n);
  f->st.kernel_launches++;
  struct Pass {
    int kind, bits;
  };
  int ebits = 1;
  while ((1ULL << ebits) < n_ordinals + 1) ++ebits;
  std::vector<Pass> passes;
  if (wid_pass) passes.push_back({BW_SK_WID, 64});
  passes.push_back({BW_SK_SEQ, 64});
  passes.push_back({BW_SK_DIGITS, 16});
  passes.push_back({BW_SK_ALIGNED, 64});
  if (n_ordinals > 1) passes.push_back({BW_SK_EPOCH, ebits});
  for (const Pass& ps : passes) {
    k_sortkey<<<grid, 256, 0, s>>>(ps.kind, key, seq, epoch, wid, d_perm, d_sk, n, f->min_epoch);
    size_t tb = cub_bytes;
    CU(ctx, cub::DeviceRadixSort::SortPairs(d_cub, tb, d_sk, d_sk2, d_perm, d_perm2, (int)n, 0, ps.bits, s));
    std::swap(d_perm, d_perm2);
    f->st.kernel_launches++;
  }
  CU(ctx, cudaGetLastError());
  return BW_OK;
}

static bw_status grow_host(bw_fold* f, u64 nc, u64 nl) {
  bw_ctx* ctx = f->ctx;
  if (nc > f->hout_cap_c) {
    void* old[] = {f->ho_ckey, f->ho_cacc, f->ho_ccount, f->ho_cepoch, f->ho_cwid};
    for (void* p : old)
      if (p) cudaFreeHost(p);
    u64 cap = std::max<u64>(nc, 4096);
    CU(ctx, cudaHostAlloc((void**)&f->ho_ckey, cap * 8, cudaHostAllocDefault));
    CU(ctx, cudaHostAlloc((void**)&f->ho_cacc, cap * 8, cudaHostAllocDefault));
    CU(ctx, cudaHostAlloc((void**)&f->ho_ccount, cap * 8, cudaHostAllocDefault));
    CU(ctx, cudaHostAlloc((void**)&f->ho_cepoch, cap * 8, cudaHostAllocDefault));
    CU(ctx, cudaHostAlloc((void**)&f->ho_cwid, cap * 8, cudaHostAllocDefault));
    f->hout_cap_c = cap;
  }
  if (nl > f->hout_cap_l) {
    void* old[] = {f->ho_lkey, f->ho_lval, f->ho_lepoch, f->ho_lwid, f->ho_lts};
    for (void* p : old)
      if (p) cudaFreeHost(p);
    u64 cap = std::max<u64>(nl, 4096);
    CU(ctx, cudaHostAlloc((void**)&f->ho_lkey, cap * 8, cudaHostAllocDefault));
    CU(ctx, cudaHostAlloc((void**)&f->ho_lval, cap * 8, cudaHostAllocDefault));
    CU(ctx, cudaHostAlloc((void**)&f->ho_lepoch, cap * 8, cudaHostAllocDefault));
    CU(ctx, cudaHostAlloc((void**)&f->ho_lwid, cap * 8, cudaHostAllocDefault));
    CU(ctx, cudaHostAlloc((void**)&f->ho_lts, cap * 8, cudaHostAllocDefault));
    f->hout_cap_l = cap;
  }
  return BW_OK;
}

static const char* status_name(u32 s) {
  switch (s) {
    case BW_ERR_CAPACITY: return "capacity exhausted (key table, pane pool, exchange region or emit buffer): raise capacity_hint / max_emit_rows / max_late_rows";
    case BW_ERR_RANGE: return "window id out of range (timestamp too far from align_to for this window length)";
    default: return "device-side failure";
  }
}

// Order rows [lo, hi) of the closed or late columns and copy them to the same positions of the host arrays.
static bw_status ship_rows(bw_fold* f, bool late, u64 lo, u64 hi, bool side) {
  bw_ctx* ctx = f->ctx;
  if (hi <= lo) return BW_OK;
  cudaStream_t s = side ? f->s_out : f->s_compute;
  const u64 n = hi - lo;
  const bool ordered = f->spec.emit_order == BW_ORDER_REFERENCE;
  const int grid = ctx->sm_count * 4;
  const u64 n_ord = f->have_pending ? (f->last_epoch - f->min_epoch + 1) : 1;
  // the window-id pass orders a key's rows where the sequence column ties: sliding windows emitted from one
  // pane, and folds whose sequence is just the closing activation (FoldParams::seq_by_id)
  const bool sliding = f->p.panes_per_window > 1 || f->p.panes_per_offset > 1 || f->p.seq_by_id;
  const EmitBufs& e = f->e;
  if (ordered) {
    if (side && n > f->fl.cap) {  // (grow the side scratch: nothing is in flight on it once the stream is idle)
      CU(ctx, cudaStreamSynchronize(s));
      void* old[] = {f->fl.sk, f->fl.sk2, f->fl.gather, f->fl.perm, f->fl.perm2, f->fl.cub};
      for (void* q : old)
        if (q) cudaFree(q);
      const u64 cap = std::max<u64>(2 * n, 1 << 16);
      CU(ctx, dmalloc(&f->fl.sk, cap));
      CU(ctx, dmalloc(&f->fl.sk2, cap));
      CU(ctx, dmalloc(&f->fl.gather, cap));
      CU(ctx, dmalloc(&f->fl.perm, cap));
      CU(ctx, dmalloc(&f->fl.perm2, cap));
      size_t b = 0;
      cub::DeviceRadixSort::SortPairs(nullptr, b, f->fl.sk, f->fl.sk2, f->fl.perm, f->fl.perm2, (int)cap, 0, 64, s);
      f->fl.cub_bytes = b + 256;
      CU(ctx, cudaMalloc(&f->fl.cub, f->fl.cub_bytes));
      f->fl.cap = cap;
    }
    bw_status st;
    if (!late) st = order_rows(f, n, e.c_key + lo, e.c_seq + lo, e.c_epoch + lo, e.c_wid + lo, sliding, n_ord, side);
    else  // rows of one late item were reserved contiguously in ascending window id; stable sorts keep that
      st = order_rows(f, n, e.l_key + lo, e.l_seq + lo, e.l_epoch + lo, e.l_wid + lo, false, n_ord, side);
    if (st != BW_OK) return st;
  }
  const u32* perm = side ? f->fl.perm : f->d_perm;
  u64* gather = side ? f->fl.gather : f->d_gather;
  auto ship = [&](const u64* src, u64* dst) -> bw_status {
    if (ordered) {
      k_gather_u64<<<grid, 256, 0, s>>>(src + lo, perm, gather, n);
      f->st.kernel_launches++;
      CU(ctx, cudaMemcpyAsync(dst + lo, gather, n * 8, cudaMemcpyDeviceToHost, s));
    } else {
      CU(ctx, cudaMemcpyAsync(dst + lo, src + lo, n * 8, cudaMemcpyDeviceToHost, s));
    }
    return BW_OK;
  };
  bw_status st;
  if (!late) {
    if ((st = ship(e.c_key, f->ho_ckey))) return st;
    if ((st = ship((const u64*)e.c_wid, (u64*)f->ho_cwid))) return st;
    if ((st = ship(e.c_acc, f->ho_cacc))) return st;
    if ((st = ship(e.c_count, f->ho_ccount))) return st;
    if ((st = ship(e.c_epoch, f->ho_cepoch))) return st;
  } else {
    if ((st = ship(e.l_key, f->ho_lkey))) return st;
    if ((st = ship((const u64*)e.l_wid, (u64*)f->ho_lwid))) return st;
    if ((st = ship(e.l_val, f->ho_lval))) return st;
    if ((st = ship((const u64*)e.l_ts, (u64*)f->ho_lts))) return st;
    if ((st = ship(e.l_epoch, f->ho_lepoch))) return st;
  }
  return BW_OK;
}

// After an activation's fold stage has been queued: remember how many rows exist once it is done.
static bw_status mark_rows(bw_fold* f, u64 epoch) {
  bw_ctx* ctx = f->ctx;
  if (!f->flush_on || ctx->world > 1 || !f->host_ingest) return BW_OK;
  if (!f->s_out) {
    CU(ctx, cudaStreamCreateWithFlags(&f->s_out, cudaStreamNonBlocking));
    CU(ctx, cudaHostAlloc((void**)&f->h_marks, 4 * 2 * sizeof(unsigned long long), cudaHostAllocDefault));
    for (auto& m : f->marks) CU(ctx, cudaEventCreateWithFlags(&m.ev, cudaEventDisableTiming));
  }
  if (f->mark_head) f->marks[(f->mark_head - 1) & 3].next_epoch = epoch + 1;  // (+1: 0 means "none yet")
  bw_fold::RowMark& m = f->marks[f->mark_head & 3];
  m.epoch = epoch;
  m.next_epoch = 0;
  m.live = true;
  CU(ctx, cudaMemcpyAsync(f->h_marks + 2 * (f->mark_head & 3), &f->d_ctr->n_closed, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                          f->s_compute));
  CU(ctx, cudaEventRecord(m.ev, f->s_compute));
  ++f->mark_head;
  return BW_OK;
}

// Rows of epochs that are closed -- a later activation with a larger epoch has been folded -- and whose counts have
// reached the host: order them and copy them out now, on the side stream, beside whatever the fold stream is doing.
// Segments end on epoch boundaries and are shipped in epoch order, so the host arrays end up exactly as one sort of
// everything would leave them (the order is epoch-major).
static bw_status flush_rows(bw_fold* f) {
  bw_ctx* ctx = f->ctx;
  if (!f->flush_on || !f->s_out) return BW_OK;
  for (u32 k = 0; k < 4 && k < f->mark_head; ++k) {  // newest first
    const u32 at = (f->mark_head - 1 - k) & 3;
    bw_fold::RowMark& m = f->marks[at];
    if (!m.live) break;
    if (!m.next_epoch || m.next_epoch - 1 <= m.epoch) continue;  // its epoch may still get rows
    if (cudaEventQuery(m.ev) != cudaSuccess) continue;
    const u64 nc = std::min<u64>(f->h_marks[2 * at], f->e.max_closed), nl = std::min<u64>(f->h_marks[2 * at + 1], f->e.max_late);
    bw_status st = ship_rows(f, false, f->done_c, nc, true);
    if (st != BW_OK) return st;
    st = ship_rows(f, true, f->done_l, nl, true);
    if (st != BW_OK) return st;
    if (nc > f->done_c) f->done_c = nc;
    if (nl > f->done_l) f->done_l = nl;
    for (u32 j = k; j < 4 && j < f->mark_head; ++j) f->marks[(f->mark_head - 1 - j) & 3].live = false;  // this one and the older ones: done
    CU(ctx, cudaGetLastError());
    break;
  }
  return BW_OK;
}

static bw_status collect(bw_fold* f, bw_emit* out) {
  bw_ctx* ctx = f->ctx;
  cudaStream_t s = f->s_compute;
  {
    bw_status vst = verdict_join(f, s);
    if (vst != BW_OK) return vst;
  }
  CU(ctx, cudaMemcpyAsync(f->h_ctr, f->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, s));
  CU(ctx, cudaStreamSynchronize(s));
  if (f->s_out) CU(ctx, cudaStreamSynchronize(f->s_out));

  if (f->h_ctr->err) FAIL(f, (bw_status)f->h_ctr->err, "kernel raised status %u: %s", f->h_ctr->err, status_name(f->h_ctr->err));
  const u64 nc = std::min<u64>(f->h_ctr->n_closed, f->e.max_closed);
  const u64 nl = std::min<u64>(f->h_ctr->n_late, f->e.max_late);
  f->st.live_keys = f->h_ctr->live_keys;
  f->st.pane_nodes_used = f->h_ctr->pool_next - 1;
  bw_status st = grow_host(f, nc, nl);
  if (st != BW_OK) return st;
  // what the side stream has not already ordered and copied (everything, when nothing was flushed early)
  if ((st = ship_rows(f, false, std::min(f->done_c, nc), nc, false))) return st;
  if ((st = ship_rows(f, true, std::min(f->done_l, nl), nl, false))) return st;
  f->done_c = f->done_l = 0;
  for (auto& m : f->marks) m.live = false;
  // reset the row counters for the next round
  CU(ctx, cudaMemsetAsync(&f->d_ctr->n_closed, 0, sizeof(unsigned long long) * 2, s));
  CU(ctx, cudaStreamSynchronize(s));
  f->have_pending = false;
  out->n_closed = nc;
  out->closed_key = f->ho_ckey;
  out->closed_window_id = f->ho_cwid;
  out->closed_acc = f->ho_cacc;
  out->closed_count = f->ho_ccount;
  out->closed_epoch = f->ho_cepoch;
  out->n_late = nl;
  out->late_key = f->ho_lkey;
  out->late_window_id = f->ho_lwid;
  out->late_val = f->ho_lval;
  out->late_ts_us = f->ho_lts;
  out->late_epoch = f->ho_lepoch;
  return BW_OK;
}

bw_status bw_fold_set_system_now(bw_fold* f, int64_t system_now_us) {
  if (!f) return BW_ERR_SPEC;
  if (f->ctx->world > 1) FAIL(f, BW_ERR_SPEC, "bw_fold_set_system_now: one rank only (every rank would need the same clock)");
  CU(f->ctx, cudaSetDevice(f->ctx->device));
  if (!f->p.track_wm || f->p.ts_from_value == 2) return BW_OK;  // no watermark to move
  if (system_now_us <= f->p.now_us) return BW_OK;              // "don't let now go backwards" (windowing.py:250-261)
  bw_status st = stream_resolve(f);  // the activation in flight was scattered in the old frame: fold it there
  if (st != BW_OK) return st;
  f->p.now_us = system_now_us;
  f->p.align_us = f->spec.align_to_us - system_now_us;
  return BW_OK;
}

bw_status bw_advance(bw_fold* f, uint64_t closed_epoch, int64_t system_now_us, bw_emit* out) {
  (void)closed_epoch;
  if (!f || !out) return BW_ERR_SPEC;
  bw_ctx* ctx = f->ctx;
  CU(ctx, cudaSetDevice(ctx->device));
  bw_status st = stream_resolve(f);
  if (st != BW_OK) return st;
  if (system_now_us > 0 && ctx->world == 1 && f->p.track_wm && f->p.ts_from_value != 2 && !f->eof_done) {
    // the notify phase at this system time: due keys close what their watermark now allows
    st = bw_fold_set_system_now(f, system_now_us);
    if (st != BW_OK) return st;
    if (!f->have_pending) { f->min_epoch = f->last_epoch; f->have_pending = true; }
    k_close_wake<<<f->close_grid, 256, 0, f->s_compute>>>(f->t, f->p, f->e, f->last_epoch, f->batch_no);
    CU(ctx, cudaGetLastError());
    f->st.kernel_launches++;
  }
  return collect(f, out);
}

bw_status bw_eof(bw_fold* f, bw_emit* out) {
  if (!f || !out) return BW_ERR_SPEC;
  bw_ctx* ctx = f->ctx;
  CU(ctx, cudaSetDevice(ctx->device));
  if (f->eof_done) FAIL(f, BW_ERR_STATE, "eof called twice");
  {
    bw_status st = stream_resolve(f);
    if (st != BW_OK) return st;
  }
  const u64 ord = f->last_epoch;
  if (!f->have_pending) { f->min_epoch = f->last_epoch; f->have_pending = true; }
  k_close_all<<<f->close_grid, 256, 0, f->s_compute>>>(f->t, f->p, f->e, ord, f->batch_no);
  CU(ctx, cudaGetLastError());
  f->st.kernel_launches++;
  f->eof_done = true;
  return collect(f, out);
}

// ---------------------------------------------------------------------------
// snapshot / restore
// ---------------------------------------------------------------------------
static SnapCols snap_cols(void* base, u64 n) {
  SnapCols c;
  u64* b = (u64*)base;
  c.key = b;
  c.pane = (i64*)(b + n);
  c.acc = b + 2 * n;
  c.cnt = b + 3 * n;
  c.seq = b + 4 * n;
  c.max_ts = (i64*)(b + 5 * n);
  c.closed_upto = (i64*)(b + 6 * n);
  c.cap = n;
  return c;
}

bw_status bw_snapshot_take(bw_fold* f, bw_snapshot* out) {
  if (!f || !out) return BW_ERR_SPEC;
  bw_ctx* ctx = f->ctx;
  CU(ctx, cudaSetDevice(ctx->device));
  if (f->eof_done) FAIL(f, BW_ERR_STATE, "snapshot after eof");
  {
    bw_status st = stream_resolve(f);
    if (st != BW_OK) return st;
  }
  cudaStream_t s = f->s_compute;
  if (f->s_x) CU(ctx, cudaStreamSynchronize(f->s_x));
  {
    bw_status vst = verdict_join(f, s);
    if (vst != BW_OK) return vst;
  }
  if (!f->d_snap_ctr) CU(ctx, dmalloc(&f->d_snap_ctr, 2));
  CU(ctx, cudaMemsetAsync(f->d_snap_ctr, 0, 2 * sizeof(unsigned long long), s));
  k_snap_count<<<f->close_grid, 256, 0, s>>>(f->t, f->d_snap_ctr);
  unsigned long long n = 0;
  CU(ctx, cudaMemcpyAsync(&n, f->d_snap_ctr, sizeof n, cudaMemcpyDeviceToHost, s));
  CU(ctx, cudaMemcpyAsync(f->h_ctr, f->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, s));
  CU(ctx, cudaStreamSynchronize(s));
  if (f->h_ctr->err) FAIL(f, (bw_status)f->h_ctr->err, "a kernel reported status %u before the snapshot", f->h_ctr->err);
  if (f->snap_dev) { cudaFree(f->snap_dev); f->snap_dev = nullptr; }
  if (f->snap_host) { cudaFreeHost(f->snap_host); f->snap_host = nullptr; }
  const u64 rows = n ? n : 1;
  CU(ctx, cudaMalloc(&f->snap_dev, rows * 7 * 8));
  CU(ctx, cudaHostAlloc(&f->snap_host, rows * 7 * 8, cudaHostAllocDefault));
  SnapCols dc = snap_cols(f->snap_dev, rows), hc = snap_cols(f->snap_host, rows);
  if (n) {
    k_snap_fill<<<f->close_grid, 256, 0, s>>>(f->t, dc, f->d_snap_ctr + 1);
    CU(ctx, cudaGetLastError());
    CU(ctx, cudaMemcpyAsync(f->snap_host, f->snap_dev, rows * 7 * 8, cudaMemcpyDeviceToHost, s));
    CU(ctx, cudaStreamSynchronize(s));
  }
  f->st.kernel_launches += n ? 2 : 1;
  memset(out, 0, sizeof *out);
  out->n = n;
  out->key = hc.key;
  out->pane_id = hc.pane;
  out->acc = hc.acc;
  out->count = hc.cnt;
  out->open_seq = hc.seq;
  out->max_ts_us = hc.max_ts;
  out->closed_upto = hc.closed_upto;
  out->batch_no = f->batch_no;
  out->gmax_ts_us = (i64)f->h_ctr->gmax_ts;
  out->last_epoch = f->last_epoch;
  return BW_OK;
}

bw_status bw_snapshot_load(bw_fold* f, const bw_snapshot* in) {
  if (!f || !in) return BW_ERR_SPEC;
  bw_ctx* ctx = f->ctx;
  CU(ctx, cudaSetDevice(ctx->device));
  if (f->batch_no != 0 || f->eof_done) FAIL(f, BW_ERR_STATE, "bw_snapshot_load needs a freshly created fold");
  if (in->n && (!in->key || !in->pane_id || !in->acc || !in->count || !in->open_seq || !in->max_ts_us || !in->closed_upto))
    FAIL(f, BW_ERR_SPEC, "bw_snapshot_load: missing column");
  if (in->batch_no >= (1ULL << 32)) FAIL(f, BW_ERR_SPEC, "bw_snapshot_load: bad batch_no");
  cudaStream_t s = f->s_compute;
  const u64 n = in->n;
  if (n) {
    void* dev = nullptr;
    CU(ctx, cudaMalloc(&dev, n * 7 * 8));
    SnapCols dc = snap_cols(dev, n);
    const void* src[7] = {in->key, in->pane_id, in->acc, in->count, in->open_seq, in->max_ts_us, in->closed_upto};
    void* dst[7] = {dc.key, dc.pane, dc.acc, dc.cnt, dc.seq, dc.max_ts, dc.closed_upto};
    for (int c = 0; c < 7; ++c) CU(ctx, cudaMemcpyAsync(dst[c], src[c], n * 8, cudaMemcpyHostToDevice, s));
    k_snap_load<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(f->t, f->p, dc, n, (u32)in->batch_no, ctx->world, ctx->rank);
    CU(ctx, cudaGetLastError());
    // re-rank every restored key (newest pane into the hot slot); nothing is closable in a state dumped after an advance
    k_close_dirty<<<f->close_grid, 256, 0, s>>>(f->t, f->p, f->e, in->last_epoch, (u32)in->batch_no, nullptr);
    f->st.kernel_launches += 2;
    CU(ctx, cudaStreamSynchronize(s));
    cudaFree(dev);
  }
  {
    bw_status vst = verdict_join(f, s);
    if (vst != BW_OK) return vst;
  }
  k_snap_set_gmax<<<1, 1, 0, s>>>(f->d_ctr, (i64)in->gmax_ts_us);
  CU(ctx, cudaMemcpyAsync(f->h_ctr, f->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, s));
  CU(ctx, cudaStreamSynchronize(s));
  if (f->h_ctr->err) FAIL(f, (bw_status)f->h_ctr->err, "restore failed on the device with status %u (capacity_hint too small?)", f->h_ctr->err);
  f->batch_no = (u32)in->batch_no;
  f->h_gmax = std::max<i64>(f->h_gmax, (i64)in->gmax_ts_us);
  f->last_epoch = in->last_epoch;
  f->have_epoch = in->last_epoch != 0;
  return BW_OK;
}

void bw_window_bounds(const bw_fold_spec* spec, int64_t window_id, int64_t* open_us, int64_t* close_us) {
  const int64_t o = spec->align_to_us + spec->offset_us * window_id;
  if (open_us) *open_us = o;
  if (close_us) *close_us = o + spec->length_us;
}

static void drain_timers(bw_fold* f) {
  for (size_t i = 0; i < f->timers_used; ++i) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, f->timers[i].a, f->timers[i].b) == cudaSuccess) {
      if (f->timers[i].kind == 1) {
        f->st.sum_scatter_ms += ms;
        f->st.scatter_launches++;
      } else if (f->timers[i].kind == 2) {
        f->st.sum_verdict_ms += ms;
      } else {
        f->st.last_fold_ms = ms;
        f->st.sum_fold_ms += ms;
        f->st.fold_rows += f->timers[i].rows;
        f->st.timed_folds++;
      }
    }
  }
  f->timers_used = 0;
}

bw_status bw_fold_stats(bw_fold* f, bw_stats* out) {
  if (!f || !out) return BW_ERR_SPEC;
  CU(f->ctx, cudaSetDevice(f->ctx->device));
  {
    bw_status st = stream_resolve(f);
    if (st != BW_OK) return st;
  }
  CU(f->ctx, cudaStreamSynchronize(f->s_verdict));
  CU(f->ctx, cudaStreamSynchronize(f->s_compute));
  drain_timers(f);
  *out = f->st;
  return BW_OK;
}
bw_status bw_fold_reset_timers(bw_fold* f) {
  if (!f) return BW_ERR_SPEC;
  {
    bw_status st = stream_resolve(f);
    if (st != BW_OK) return st;
  }
  CU(f->ctx, cudaStreamSynchronize(f->s_verdict));
  CU(f->ctx, cudaStreamSynchronize(f->s_compute));
  drain_timers(f);
  f->st.sum_scatter_ms = 0;
  f->st.sum_verdict_ms = 0;
  f->st.scatter_launches = 0;
  f->st.sum_fold_ms = 0;
  f->st.last_fold_ms = 0;
  f->st.fold_rows = 0;
  f->st.timed_folds = 0;
  f->st.fold_launches = 0;
  f->st.combined_folds = 0;
  f->st.split_batches = 0;
  return BW_OK;
}
bw_status bw_fold_sync(bw_fold* f) {
  if (!f) return BW_ERR_SPEC;
  CU(f->ctx, cudaSetDevice(f->ctx->device));
  {
    bw_status st = stream_resolve(f);
    if (st != BW_OK) return st;
  }
  CU(f->ctx, cudaStreamSynchronize(f->s_copy));
  CU(f->ctx, cudaStreamSynchronize(f->s_pre));
  CU(f->ctx, cudaStreamSynchronize(f->s_x));
  CU(f->ctx, cudaStreamSynchronize(f->s_verdict));
  CU(f->ctx, cudaStreamSynchronize(f->s_compute));
  return BW_OK;
}
bw_status bw_fold_time_begin(bw_fold* f) {
  if (!f) return BW_ERR_SPEC;
  bw_ctx* ctx = f->ctx;
  CU(ctx, cudaSetDevice(ctx->device));
  if (!f->ev_t0) {
    CU(ctx, cudaEventCreate(&f->ev_t0));
    CU(ctx, cudaEventCreate(&f->ev_t1));
  }
  // everything submitted so far (copies, prepass) must be done before the clock starts
  {
    bw_status st = stream_resolve(f);
    if (st != BW_OK) return st;
  }
  CU(ctx, cudaStreamSynchronize(f->s_copy));
  CU(ctx, cudaStreamSynchronize(f->s_pre));
  CU(ctx, cudaStreamSynchronize(f->s_x));
  CU(ctx, cudaStreamSynchronize(f->s_verdict));
  CU(ctx, cudaStreamSynchronize(f->s_compute));
  CU(ctx, cudaEventRecord(f->ev_t0, f->s_compute));
  return BW_OK;
}
bw_status bw_fold_time_end(bw_fold* f, float* ms) {
  if (!f || !ms || !f->ev_t0) return BW_ERR_SPEC;
  bw_ctx* ctx = f->ctx;
  {
    bw_status st = stream_resolve(f);
    if (st != BW_OK) return st;
  }
  CU(ctx, cudaStreamSynchronize(f->s_copy));
  CU(ctx, cudaStreamSynchronize(f->s_pre));
  CU(ctx, cudaStreamSynchronize(f->s_x));
  {  // (every verdict is done by now: stream_resolve has waited for the newest; the stop event is behind them anyway)
    bw_status vst = verdict_join(f, f->s_compute);
    if (vst != BW_OK) return vst;
  }
  CU(ctx, cudaEventRecord(f->ev_t1, f->s_compute));
  CU(ctx, cudaEventSynchronize(f->ev_t1));
  CU(ctx, cudaEventElapsedTime(ms, f->ev_t0, f->ev_t1));
  return BW_OK;
}
void* bw_fold_stream(bw_fold* f) { return f ? (void*)f->s_compute : nullptr; }

bw_status bw_gen_c1(bw_fold* f, uint64_t* d_keys, uint64_t* d_vals, uint64_t start, uint64_t rows, uint64_t n_keys) {
  if (!f || !n_keys) return BW_ERR_SPEC;
  CU(f->ctx, cudaSetDevice(f->ctx->device));
  k_gen_c1<<<f->ctx->sm_count * 8, 256, 0, f->s_compute>>>(d_keys, d_vals, start, rows, n_keys);
  CU(f->ctx, cudaGetLastError());
  if (!f->ev_gen) CU(f->ctx, cudaEventCreateWithFlags(&f->ev_gen, cudaEventDisableTiming));
  CU(f->ctx, cudaEventRecord(f->ev_gen, f->s_compute));
  f->st.kernel_launches++;
  return BW_OK;
}


// ===========================================================================
// K5 / K6 host side
// ===========================================================================
struct MaxU32 {
  __host__ __device__ __forceinline__ u32 operator()(const u32& a, const u32& b) const { return a > b ? a : b; }
};

struct KeyedScratch {  // grouping of one activation by key (stable)
  u64 cap = 0;
  u64 *d_keys = nullptr, *d_ksorted = nullptr, *d_slot = nullptr;
  u32 *d_idx = nullptr, *d_isorted = nullptr, *d_head = nullptr;
  void* d_cub = nullptr;
  size_t cub_bytes = 0;
};

static bw_status keyed_alloc(bw_ctx* ctx, KeyedScratch& k, u64 cap, cudaStream_t s) {
  k.cap = cap;
  CU(ctx, dmalloc(&k.d_keys, cap));
  CU(ctx, dmalloc(&k.d_ksorted, cap));
  CU(ctx, dmalloc(&k.d_slot, cap));
  CU(ctx, dmalloc(&k.d_idx, cap));
  CU(ctx, dmalloc(&k.d_isorted, cap));
  CU(ctx, dmalloc(&k.d_head, cap));
  size_t b1 = 0, b2 = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, b1, k.d_keys, k.d_ksorted, k.d_idx, k.d_isorted, (int)cap, 0, 64, s);
  cub::DeviceScan::InclusiveScan(nullptr, b2, k.d_head, k.d_head, MaxU32(), (int)cap, s);
  k.cub_bytes = std::max(b1, b2) + 256;
  CU(ctx, cudaMalloc(&k.d_cub, k.cub_bytes));
  return BW_OK;
}
static void keyed_free(KeyedScratch& k) {
  void* p[] = {k.d_keys, k.d_ksorted, k.d_slot, k.d_idx, k.d_isorted, k.d_head, k.d_cub};
  for (void* q : p)
    if (q) cudaFree(q);
}
// stable group-by-key of n device keys: ksorted / isorted / head positions
static bw_status keyed_group(bw_ctx* ctx, KeyedScratch& k, const u64* d_keys, u64 n, cudaStream_t s) {
  const int grid = ctx->sm_count * 4;
  k_iota<<<grid, 256, 0, s>>>(k.d_idx, n);
  size_t tb = k.cub_bytes;
  CU(ctx, cub::DeviceRadixSort::SortPairs(k.d_cub, tb, d_keys, k.d_ksorted, k.d_idx, k.d_isorted, (int)n, 0, 64, s));
  k_keyed_heads<<<grid, 256, 0, s>>>(k.d_ksorted, k.d_head, n);
  tb = k.cub_bytes;
  CU(ctx, cub::DeviceScan::InclusiveScan(k.d_cub, tb, k.d_head, k.d_head, MaxU32(), (int)n, s));
  CU(ctx, cudaGetLastError());
  return BW_OK;
}

struct bw_smap {
  bw_ctx* ctx = nullptr;
  bw_smap_spec spec{};
  SmapTable t{};
  KeyedScratch k;
  cudaStream_t s = nullptr;
  u32* h_err = nullptr;
  void* d_vals = nullptr;
  double *d_mu = nullptr, *d_sigma = nullptr;
  unsigned char* d_flag = nullptr;
};

bw_status bw_smap_create(bw_ctx* ctx, const bw_smap_spec* spec, bw_smap** out) {
  if (!ctx || !spec || !out) CTX_FAIL(ctx, BW_ERR_SPEC, "bw_smap_create: NULL argument");
  if (spec->struct_size != sizeof(bw_smap_spec)) CTX_FAIL(ctx, BW_ERR_SPEC, "bw_smap_spec.struct_size mismatch");
  if (spec->window < 1 || spec->window > BW_SMAP_MAXW) CTX_FAIL(ctx, BW_ERR_SPEC, "window must be in 1..%d", BW_SMAP_MAXW);
  if (spec->val_dtype != BW_VAL_F32 && spec->val_dtype != BW_VAL_F64) CTX_FAIL(ctx, BW_ERR_SPEC, "val_dtype must be F32 or F64");
  if (spec->max_batch_rows == 0 || spec->max_batch_rows >= (1ULL << 31)) CTX_FAIL(ctx, BW_ERR_SPEC, "bad max_batch_rows");
  CU(ctx, cudaSetDevice(ctx->device));
  bw_smap* m = new bw_smap();
  m->ctx = ctx;
  m->spec = *spec;
  u64 cap = std::max<u64>(1024, 2 * std::max<u64>(spec->capacity_hint, 1));
  m->t.cap = cap;
  m->t.window = spec->window;
  CU(ctx, cudaStreamCreateWithFlags(&m->s, cudaStreamNonBlocking));
  CU(ctx, dmalloc(&m->t.keys, cap + 1));
  CU(ctx, dmalloc(&m->t.cnt, cap + 1));
  CU(ctx, dmalloc(&m->t.ring, (cap + 1) * (u64)spec->window));
  CU(ctx, dmalloc(&m->t.err, 1));
  CU(ctx, cudaMemsetAsync(m->t.err, 0, 4, m->s));
  CU(ctx, cudaHostAlloc((void**)&m->h_err, 64, cudaHostAllocDefault));
  const u64 n = spec->max_batch_rows;
  bw_status st = keyed_alloc(ctx, m->k, n, m->s);
  if (st != BW_OK) return st;
  CU(ctx, cudaMalloc(&m->d_vals, n * 8));
  CU(ctx, dmalloc(&m->d_mu, n));
  CU(ctx, dmalloc(&m->d_sigma, n));
  CU(ctx, dmalloc(&m->d_flag, n));
  k_smap_init<<<ctx->sm_count * 4, 256, 0, m->s>>>(m->t);
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaStreamSynchronize(m->s));
  *out = m;
  return BW_OK;
}

void bw_smap_destroy(bw_smap* m) {
  if (!m) return;
  cudaSetDevice(m->ctx->device);
  cudaStreamSynchronize(m->s);
  void* p[] = {m->t.keys, m->t.cnt, m->t.ring, m->t.err, m->d_vals, m->d_mu, m->d_sigma, m->d_flag};
  for (void* q : p)
    if (q) cudaFree(q);
  keyed_free(m->k);
  if (m->h_err) cudaFreeHost(m->h_err);
  cudaStreamDestroy(m->s);
  delete m;
}

bw_status bw_smap_apply_device(bw_smap* m, const uint64_t* d_keys, const void* d_vals, uint64_t rows, double* d_mu,
                               double* d_sigma, uint8_t* d_flag) {
  if (!m) return BW_ERR_SPEC;
  bw_ctx* ctx = m->ctx;
  if (rows > m->spec.max_batch_rows) CTX_FAIL(ctx, BW_ERR_SPEC, "smap: rows > max_batch_rows");
  if (rows == 0) return BW_OK;
  CU(ctx, cudaSetDevice(ctx->device));
  bw_status st = keyed_group(ctx, m->k, d_keys, rows, m->s);
  if (st != BW_OK) return st;
  const int grid = ctx->sm_count * 8;
  const int is_f32 = m->spec.val_dtype == BW_VAL_F32;
  k_smap_slots<<<grid, 256, 0, m->s>>>(m->t, m->k.d_ksorted, m->k.d_head, m->k.d_slot, rows);
  k_smap_eval<<<grid, 256, 0, m->s>>>(m->t, m->k.d_isorted, m->k.d_head, m->k.d_slot, d_vals, is_f32, m->spec.threshold, d_mu, d_sigma,
                                       d_flag, rows);
  k_smap_update<<<grid, 256, 0, m->s>>>(m->t, m->k.d_ksorted, m->k.d_isorted, m->k.d_head, m->k.d_slot, d_vals, is_f32, rows);
  CU(ctx, cudaGetLastError());
  return BW_OK;
}

bw_status bw_smap_sync(bw_smap* m) {
  if (!m) return BW_ERR_SPEC;
  bw_ctx* ctx = m->ctx;
  CU(ctx, cudaMemcpyAsync(m->h_err, m->t.err, 4, cudaMemcpyDeviceToHost, m->s));
  CU(ctx, cudaStreamSynchronize(m->s));
  if (*m->h_err) CTX_FAIL(ctx, (bw_status)*m->h_err, "smap kernel raised status %u: key table full (raise capacity_hint)", *m->h_err);
  return BW_OK;
}

bw_status bw_smap_apply(bw_smap* m, const uint64_t* keys, const void* vals, uint64_t rows, double* out_mu, double* out_sigma,
                        uint8_t* out_flag) {
  if (!m) return BW_ERR_SPEC;
  bw_ctx* ctx = m->ctx;
  if (rows > m->spec.max_batch_rows) CTX_FAIL(ctx, BW_ERR_SPEC, "smap: rows > max_batch_rows");
  if (rows == 0) return BW_OK;
  CU(ctx, cudaSetDevice(ctx->device));
  const size_t vb = m->spec.val_dtype == BW_VAL_F32 ? 4 : 8;
  CU(ctx, cudaMemcpyAsync(m->k.d_keys, keys, rows * 8, cudaMemcpyHostToDevice, m->s));
  CU(ctx, cudaMemcpyAsync(m->d_vals, vals, rows * vb, cudaMemcpyHostToDevice, m->s));
  bw_status st = bw_smap_apply_device(m, m->k.d_keys, m->d_vals, rows, m->d_mu, m->d_sigma, m->d_flag);
  if (st != BW_OK) return st;
  CU(ctx, cudaMemcpyAsync(out_mu, m->d_mu, rows * 8, cudaMemcpyDeviceToHost, m->s));
  CU(ctx, cudaMemcpyAsync(out_sigma, m->d_sigma, rows * 8, cudaMemcpyDeviceToHost, m->s));
  CU(ctx, cudaMemcpyAsync(out_flag, m->d_flag, rows, cudaMemcpyDeviceToHost, m->s));
  return bw_smap_sync(m);
}

struct bw_join {
  bw_ctx* ctx = nullptr;
  bw_join_spec spec{};
  JoinSlot* slots = nullptr;
  u64 cap = 0;
  KeyedScratch k;
  cudaStream_t s = nullptr;
  u32 *d_err = nullptr, *h_err = nullptr;
  unsigned long long *d_nrows = nullptr, *h_nrows = nullptr;
  unsigned char* d_side = nullptr;
  u64* d_vals = nullptr;
  JoinEmit e{};
  // ordering scratch + host output
  u64 *d_sk = nullptr, *d_sk2 = nullptr, *d_gather = nullptr;
  u32 *d_perm = nullptr, *d_perm2 = nullptr;
  void* d_cub = nullptr;
  size_t cub_bytes = 0;
  u64 *h_key = nullptr, *h_l = nullptr, *h_r = nullptr, *h_mask = nullptr, *h_epoch = nullptr;
  u32 batch_no = 0;
  u64 min_epoch = 0, last_epoch = 0;
  bool pending = false;
};

bw_status bw_join_create(bw_ctx* ctx, const bw_join_spec* spec, bw_join** out) {
  if (!ctx || !spec || !out) CTX_FAIL(ctx, BW_ERR_SPEC, "bw_join_create: NULL argument");
  if (spec->struct_size != sizeof(bw_join_spec)) CTX_FAIL(ctx, BW_ERR_SPEC, "bw_join_spec.struct_size mismatch");
  if (spec->insert_mode < 0 || spec->insert_mode > 1) CTX_FAIL(ctx, BW_ERR_SPEC, "insert_mode must be first or last (product: host path)");
  if (spec->emit_mode < 0 || spec->emit_mode > 2) CTX_FAIL(ctx, BW_ERR_SPEC, "bad emit_mode");
  if (spec->max_batch_rows == 0 || spec->max_batch_rows >= (1ULL << 31)) CTX_FAIL(ctx, BW_ERR_SPEC, "bad max_batch_rows");
  CU(ctx, cudaSetDevice(ctx->device));
  bw_join* j = new bw_join();
  j->ctx = ctx;
  j->spec = *spec;
  j->cap = std::max<u64>(1024, 2 * std::max<u64>(spec->capacity_hint, 1));
  CU(ctx, cudaStreamCreateWithFlags(&j->s, cudaStreamNonBlocking));
  CU(ctx, dmalloc(&j->slots, j->cap + 1));
  CU(ctx, dmalloc(&j->d_err, 1));
  CU(ctx, dmalloc(&j->d_nrows, 1));
  CU(ctx, cudaMemsetAsync(j->d_err, 0, 4, j->s));
  CU(ctx, cudaMemsetAsync(j->d_nrows, 0, 8, j->s));
  CU(ctx, cudaHostAlloc((void**)&j->h_err, 64, cudaHostAllocDefault));
  CU(ctx, cudaHostAlloc((void**)&j->h_nrows, 64, cudaHostAllocDefault));
  const u64 n = spec->max_batch_rows, m = std::max<u64>(spec->max_emit_rows, 1024);
  bw_status st = keyed_alloc(ctx, j->k, n, j->s);
  if (st != BW_OK) return st;
  CU(ctx, dmalloc(&j->d_side, n));
  CU(ctx, dmalloc(&j->d_vals, n));
  u64** cols[] = {&j->e.key, &j->e.l, &j->e.r, &j->e.mask, &j->e.seq, &j->e.epoch, &j->d_sk, &j->d_sk2, &j->d_gather};
  for (u64** c : cols) CU(ctx, dmalloc(c, m));
  CU(ctx, dmalloc(&j->d_perm, m));
  CU(ctx, dmalloc(&j->d_perm2, m));
  j->e.max_rows = spec->max_emit_rows;
  j->e.n_rows = j->d_nrows;
  size_t b = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, b, j->d_sk, j->d_sk2, j->d_perm, j->d_perm2, (int)m, 0, 64, j->s);
  j->cub_bytes = b + 256;
  CU(ctx, cudaMalloc(&j->d_cub, j->cub_bytes));
  u64** hcols[] = {&j->h_key, &j->h_l, &j->h_r, &j->h_mask, &j->h_epoch};
  for (u64** c : hcols) CU(ctx, cudaHostAlloc((void**)c, m * 8, cudaHostAllocDefault));
  k_join_init<<<ctx->sm_count * 4, 256, 0, j->s>>>(j->slots, j->cap);
  CU(ctx, cudaGetLastError());
  CU(ctx, cudaStreamSynchronize(j->s));
  *out = j;
  return BW_OK;
}

void bw_join_destroy(bw_join* j) {
  if (!j) return;
  cudaSetDevice(j->ctx->device);
  cudaStreamSynchronize(j->s);
  void* p[] = {j->slots, j->d_err, j->d_nrows, j->d_side, j->d_vals, j->e.key, j->e.l, j->e.r, j->e.mask, j->e.seq, j->e.epoch,
               j->d_sk, j->d_sk2, j->d_gather, j->d_perm, j->d_perm2, j->d_cub};
  for (void* q : p)
    if (q) cudaFree(q);
  keyed_free(j->k);
  void* h[] = {j->h_err, j->h_nrows, j->h_key, j->h_l, j->h_r, j->h_mask, j->h_epoch};
  for (void* q : h)
    if (q) cudaFreeHost(q);
  cudaStreamDestroy(j->s);
  delete j;
}

bw_status bw_join_apply(bw_join* j, const uint64_t* keys, const uint8_t* side, const uint64_t* vals, uint64_t rows, uint64_t epoch) {
  if (!j) return BW_ERR_SPEC;
  bw_ctx* ctx = j->ctx;
  if (rows > j->spec.max_batch_rows) CTX_FAIL(ctx, BW_ERR_SPEC, "join: rows > max_batch_rows");
  if (j->pending && epoch < j->last_epoch) CTX_FAIL(ctx, BW_ERR_STATE, "join: epochs must not decrease");
  if (!j->pending) {
    j->min_epoch = epoch;
    j->pending = true;
  }
  j->last_epoch = epoch;
  const u32 batch_no = j->batch_no++;
  if (rows == 0) return BW_OK;
  CU(ctx, cudaSetDevice(ctx->device));
  CU(ctx, cudaMemcpyAsync(j->k.d_keys, keys, rows * 8, cudaMemcpyHostToDevice, j->s));
  CU(ctx, cudaMemcpyAsync(j->d_side, side, rows, cudaMemcpyHostToDevice, j->s));
  CU(ctx, cudaMemcpyAsync(j->d_vals, vals, rows * 8, cudaMemcpyHostToDevice, j->s));
  bw_status st = keyed_group(ctx, j->k, j->k.d_keys, rows, j->s);
  if (st != BW_OK) return st;
  k_join_apply<<<ctx->sm_count * 8, 256, 0, j->s>>>(j->slots, j->cap, j->d_err, j->k.d_ksorted, j->k.d_isorted, j->k.d_head, j->d_side,
                                                      j->d_vals, rows, j->spec.insert_mode, j->spec.emit_mode, j->e, batch_no, epoch);
  CU(ctx, cudaGetLastError());
  // the host columns may be reused by the caller once this returns
  CU(ctx, cudaStreamSynchronize(j->s));
  return BW_OK;
}

static bw_status join_collect(bw_join* j, bw_join_rows* out) {
  bw_ctx* ctx = j->ctx;
  cudaStream_t s = j->s;
  CU(ctx, cudaMemcpyAsync(j->h_err, j->d_err, 4, cudaMemcpyDeviceToHost, s));
  CU(ctx, cudaMemcpyAsync(j->h_nrows, j->d_nrows, 8, cudaMemcpyDeviceToHost, s));
  CU(ctx, cudaStreamSynchronize(s));
  if (*j->h_err) CTX_FAIL(ctx, (bw_status)*j->h_err, "join kernel raised status %u: key table or emit buffer full", *j->h_err);
  const u64 n = std::min<u64>(*j->h_nrows, j->e.max_rows);
  if (n) {
    const int grid = ctx->sm_count * 4;
    k_iota<<<grid, 256, 0, s>>>(j->d_perm, n);
    const u64 n_ord = j->last_epoch - j->min_epoch + 1;
    int ebits = 1;
    while ((1ULL << ebits) < n_ord + 1) ++ebits;
    struct Pass { int kind, bits; };
    std::vector<Pass> passes = {{BW_SK_SEQ, 64}, {BW_SK_DIGITS, 16}, {BW_SK_ALIGNED, 64}};
    if (n_ord > 1) passes.push_back({BW_SK_EPOCH, ebits});
    for (const Pass& ps : passes) {
      k_sortkey<<<grid, 256, 0, s>>>(ps.kind, j->e.key, j->e.seq, j->e.epoch, nullptr, j->d_perm, j->d_sk, n, j->min_epoch);
      size_t tb = j->cub_bytes;
      CU(ctx, cub::DeviceRadixSort::SortPairs(j->d_cub, tb, j->d_sk, j->d_sk2, j->d_perm, j->d_perm2, (int)n, 0, ps.bits, s));
      std::swap(j->d_perm, j->d_perm2);
    }
    const u64* src[] = {j->e.key, j->e.l, j->e.r, j->e.mask, j->e.epoch};
    u64* dst[] = {j->h_key, j->h_l, j->h_r, j->h_mask, j->h_epoch};
    for (int c = 0; c < 5; ++c) {
      k_gather_u64<<<grid, 256, 0, s>>>(src[c], j->d_perm, j->d_gather, n);
      CU(ctx, cudaMemcpyAsync(dst[c], j->d_gather, n * 8, cudaMemcpyDeviceToHost, s));
    }
    CU(ctx, cudaGetLastError());
  }
  CU(ctx, cudaMemsetAsync(j->d_nrows, 0, 8, s));
  CU(ctx, cudaStreamSynchronize(s));
  j->pending = false;
  out->n = n;
  out->key = j->h_key;
  out->left = j->h_l;
  out->right = j->h_r;
  out->mask = j->h_mask;
  out->epoch = j->h_epoch;
  return BW_OK;
}

bw_status bw_join_advance(bw_join* j, bw_join_rows* out) {
  if (!j || !out) return BW_ERR_SPEC;
  CU(j->ctx, cudaSetDevice(j->ctx->device));
  return join_collect(j, out);
}

bw_status bw_join_eof(bw_join* j, bw_join_rows* out) {
  if (!j || !out) return BW_ERR_SPEC;
  bw_ctx* ctx = j->ctx;
  CU(ctx, cudaSetDevice(ctx->device));
  if (!j->pending) {
    j->min_epoch = j->last_epoch;
    j->pending = true;
  }
  k_join_eof<<<ctx->sm_count * 8, 256, 0, j->s>>>(j->slots, j->cap, j->d_err, j->spec.emit_mode, j->e, j->last_epoch);
  CU(ctx, cudaGetLastError());
  return join_collect(j, out);
}
