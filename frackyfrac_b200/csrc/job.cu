// Host side of libfrcfrc_cuda: the C ABI of include/frcfrc_cuda.h.
//
// A job is one unifrac() call (frcfrc/unifrac.go:97-124).  It is made of PARTS, one per GPU this
// process drives (one part unless opts.n_devices > 1):
//
//   frc_create   validate the options and the table header                  (this thread)
//                stage: check + copy the CSR entries and walk the tree       (worker pool, once per job
//                       into ONE portable pinned buffer every device reads    whatever the device count)
//                plan:  operand columns, bands, owners  -> csrc/plan.cpp     (this thread, meanwhile)
//                prepare(part): tiles, device buffers, ring slots, upload    (one pool task per device)
//                       of the plan, tensor maps, length quantisation
//                launch(part): upload the inputs, embedding (+ exchange of   (one pool task per device)
//                       the sample shards between the devices), first bands
//   frc_next*    bands of consecutive rows are contiguous flat ranges; every part computes the bands it
//                owns on two alternating streams, each followed by its own D2H into a pinned ring slot,
//                and the job hands them out strictly in flat-index order (the ordered iter.Seq of
//                unifrac.go:209-228) from whichever part owns the next one.
//
// Fast-path kernels store fp32 (wire.cu); frc_next_f32 hands the pinned slot out as it is, frc_next
// widens it on the host.  The exact path is fp64 end to end.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include "../../include/frcfrc_cuda.h"
#include "frc_internal.h"
#include "host_pool.h"
#include "plan.h"

using namespace frc;
using frc_host::Pool;

namespace {

thread_local std::string g_create_error;

// ------------------------------------------------------------------ arenas
struct Arena {
  struct Block { char* p; size_t cap, off; };
  std::vector<Block> blocks;
  bool pinned = false;
  size_t min_block = 0;

  void* alloc(size_t bytes, cudaError_t* err) {
    bytes = (bytes + 255) & ~size_t(255);
    if (bytes == 0) bytes = 256;
    for (auto& b : blocks)
      if (b.cap - b.off >= bytes) { void* r = b.p + b.off; b.off += bytes; return r; }
    size_t cap = std::max(bytes, min_block);
    char* p = nullptr;
    // portable: one staging buffer feeds the uploads of every device of a multi-GPU job
    cudaError_t e = pinned ? cudaHostAlloc(reinterpret_cast<void**>(&p), cap, cudaHostAllocPortable)
                           : cudaMalloc(reinterpret_cast<void**>(&p), cap);
    if (e != cudaSuccess && cap > bytes) {  // retry without the rounding-up
      cudaGetLastError();
      cap = bytes;
      e = pinned ? cudaHostAlloc(reinterpret_cast<void**>(&p), cap, cudaHostAllocPortable)
                 : cudaMalloc(reinterpret_cast<void**>(&p), cap);
    }
    if (e != cudaSuccess) { cudaGetLastError(); *err = e; return nullptr; }
    blocks.push_back({p, cap, bytes});
    return p;
  }
  void reset() { for (auto& b : blocks) b.off = 0; }
  void release() {
    for (auto& b : blocks) { if (pinned) cudaFreeHost(b.p); else cudaFree(b.p); }
    blocks.clear();
  }
};

uint16_t bf16_rn(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7F800000u) == 0x7F800000u) return static_cast<uint16_t>((u >> 16) | ((u & 0xFFFFu) ? 0x40u : 0u));
  u += 0x7FFFu + ((u >> 16) & 1u);
  return static_cast<uint16_t>(u >> 16);
}
float bf16_to_float(uint16_t h) {
  uint32_t u = static_cast<uint32_t>(h) << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

constexpr int64_t kWidePiece = 2LL << 20;        // frc_next on a fast path: pairs widened per call (16 MB of doubles: cache-resident)
constexpr int kSlots = 12;                      // output ring: a part's 8 bands all fit, so nothing is launched while the stream is read
constexpr int kMinSlots = 3;
constexpr int64_t kSlotBytesBudget = 1LL << 30;  // bytes the output ring may take beyond kMinSlots (pinned allocation is slow: ~0.4 s per GB)
constexpr double kFlagBelow = 0.125;            // fast unweighted (fp64 / bf16 modes): recompute d below this exactly
constexpr double kFlagBelowW = 0.03125;         // fast weighted: fp32 error is ~6e-8 / d -> 2e-6 at this d
constexpr int64_t kExactWorkLimit = 1LL << 28;  // AUTO: pairs * nodes at or below this -> exact
constexpr int kMaxExceptions = 4096;            // per band: distances fp32 cannot carry (wire.cuh)
constexpr int kFixupCtas = 32;                  // weighted fix-up: CTAs (one int64[B] workspace each, per stream)
constexpr int kMaxParts = 8;                    // devices per job (PeerPtrs holds 8)

// The calling thread's current device is restored when an entry point returns (a job may drive several).
struct DeviceGuard {
  int prev = -1;
  DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); } }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace

// One GPU of a context: streams + reusable memory.
struct DevCtx {
  int device = 0;
  int num_sms = 0;
  cudaStream_t stream[4] = {nullptr, nullptr, nullptr, nullptr};  // two compute streams, one D2H stream, one device-to-device (visiting shards) stream
  Arena dev, pin, sym;
};

struct frc_ctx {
  std::vector<DevCtx*> devs;
  Arena pin;  // staging of a job's inputs and plan: portable pinned memory, read by every device's upload
  std::unique_ptr<Pool> pool;
  std::vector<std::vector<int64_t>> stamps;  // per-worker duplicate-detection scratch
  int64_t stamp_epoch = 0;
  bool in_use = false;
  bool peer_ok = false;   // every device of the context can address every other's memory (NVLink / PCIe P2P)
  Comm* comm = nullptr;   // NCCL communicator over the PROCESSES of a multi-process run (frc_ctx_comm_init)
  // multi-process "symmetric heap": buffers every rank allocates identically (devs[0]->sym), so block index +
  // offset name the same buffer on every rank; each block is mapped from the peers with CUDA IPC
  std::vector<std::vector<char*>> sym_peer;  // [block][rank] mapped base (own rank: the local base)
};

namespace {

// What the pair stage of a fast path writes: fp32 distances, the pairs flagged for the fix-up, their count (mapped
// pinned, published by the fix-up) and the distances fp32 cannot carry.  A ring slot owns one for its band; in
// capacity mode a row-shard group owns one for all of its bands.
struct PairOut {
  float* dev32 = nullptr;
  uint32_t* flagged = nullptr;
  unsigned long long* n_flagged_host = nullptr;
  Exceptions ex;          // mapped pinned
  bool counted = false;   // its counts have been added to the part's info on this pass
};

struct Slot {
  double* dev64 = nullptr;   // exact path: the band in HBM / its pinned landing buffer
  double* host64 = nullptr;
  float* host32 = nullptr;   // fast paths: the pinned landing buffer
  PairOut own;               // fast paths outside capacity mode
  PairOut* out = nullptr;    // fast paths: the record the slot's band lives in (`own` or its group's), from out_off on
  int64_t out_off = 0;
  cudaEvent_t k0 = nullptr, k1 = nullptr, k2 = nullptr, done = nullptr;
};

struct Seg { size_t off = 0, bytes = 0; };
struct SegAlloc {
  size_t total = 0;
  Seg operator()(size_t bytes) { Seg s{total, bytes}; total += (bytes + 255) & ~size_t(255); return s; }
};

// What the parts of a job share: options, sizes, the plan and the pinned staging buffers (read-only
// once frc_create's staging phase has joined).
struct Shared {
  frc_opts_t opts{};
  Knobs knobs;
  int64_t N = 0, np = 0, nnz = 0;
  int32_t B = 0, kp = 0, nw = 0;
  bool exact = false, weighted = false, prescale = true, need_val = false;
  bool unsorted_l = false;    // normalize == 0 on the exact path: the reference's -l as coded (post-order lists, exact.cu)
  bool keyed = false;         // normalize == 0 on the FP32 tiles (FRC_FLAG_L_TILES): key panels next to the values
  bool node_mult = false;     // FRC_FLAG_PRUNE, fast weighted, normalize == 1: the totals weigh node v by mult[v]
  bool d2h = true;
  Geometry geo;               // frc_create_cross: the query x reference block of the staged table (n_q = N - geo.q0)
  int n_parts = 1;
  int world = 1, rank0 = 0;   // band ownership: `world` owners; part p owns owner id rank0 + p
  Variant variant;            // which variant of the fast path runs (csrc/plan.cpp)
  ShardPlan shards;           // which samples each owner builds (np = shards.np)
  ColumnPlan cols;
  std::vector<Band> bands;   // every band of the job (owners filled in)
  std::vector<int32_t> level_ptr;
  int32_t tree_height = 0;
  // inputs: [row_ptr | tree arrays ... | col | val] in one pinned buffer, same layout on every device
  char* stage_in = nullptr;
  Seg in_rowptr, in_parent, in_len, in_cptr, in_cidx, in_lvl, in_lpar, in_lptr, in_lenf, in_post, in_mult, in_col, in_val;
  size_t in_bytes = 0;
  // plan: operand columns, chunks
  char* stage_plan = nullptr;
  Seg pl_q0, pl_hi, pl_lo, pl_lenq, pl_order, pl_cexp, pl_lcol, pl_cend, pl_cscale, pl_cshift;
  size_t plan_bytes = 0;

  int owners() const { return n_parts > 1 ? n_parts : world; }
  // rows of the staged table whose CSR entries owner `owner` reads (set once plan_exchange has run)
  std::pair<int64_t, int64_t> rows_read(int owner) const {
    return frc::rows_read(N, owners(), owner, variant.sharded_fast_uw);
  }
};

}  // namespace

struct frc_job;

namespace {

// One device's share of a job.
struct Part {
  frc_job* job = nullptr;
  const Shared* sh = nullptr;
  DevCtx* dc = nullptr;
  int index = 0;   // position in job->parts
  int owner = 0;   // band owner id of this part
  int rc = FRC_OK;
  std::string err;
  frc_info_t info{};

  std::vector<int> mine;    // indices into sh->bands, ascending
  std::vector<Band> bands;  // copies of the bands in `mine` with this part's tile offsets
  std::vector<Tile> tiles;

  // first sample shard of the embedding this part builds (word columns of 32 samples; everything unless sharded)
  int32_t shard_w0 = 0, shard_nw = 0;
  int64_t csr_k0 = 0, csr_k1 = 0;  // CSR entries this part uploads
  PanelMap pm;
  // capacity mode: the rows of each of this part's (two) shards form one GROUP with one output buffer for the whole
  // pass (the column shards visit one at a time, so all rows advance together) and ONE launch per visiting shard:
  // thousands of tiles each -- per-band launches of 50-100 tiles left two thirds of the SMs idle at cfg5 sizes,
  // where the 48 MB band cap makes a band one or two tile rows thin.  Bands are sub-ranges of their group's
  // buffer; the pinned ring slots only carry the D2H.
  struct CapGroup {
    int shard = 0;                 // row shard (also the last column shard its tiles need)
    int64_t first = 0, count = 0;  // flat range of the group's rows
    int32_t tile_off = 0;          // into the part's tile list
    std::vector<int32_t> coff;     // tile offset (inside the group's list) of every column shard, + end
    PairOut out;
    cudaEvent_t done = nullptr;
  };
  std::vector<CapGroup> cap;
  std::vector<int> band_group;     // per band of this part: index into cap
  float* d_V[2] = {nullptr, nullptr};          // visiting buffers: one shard of panels each
  std::vector<cudaEvent_t> ev_fetch, ev_used;  // per column shard: "has arrived" / "no launch reads it any more"

  DevTree dtree;
  DevCsr dcsr;
  char* d_in = nullptr;
  char* d_plan = nullptr;
  Tile* d_tiles = nullptr;
  int32_t* d_level_ptr = nullptr;
  int32_t* d_post = nullptr;
  unsigned long long* d_flag_counts = nullptr;  // one per band of this part (capacity mode: per group)
  int64_t ws_slab = 0;
  bool peer_push = false;     // multi-process sharding: the bits kernel stores into every rank's bitsT over IPC mappings
  uint32_t* d_bits2[2] = {nullptr, nullptr};  // (double-buffered by run parity: a rank may be one pass ahead)
  PeerPtrs peers[2];
  int64_t run_count = 0;
  void *d_q0 = nullptr, *d_q1 = nullptr, *d_q2 = nullptr;
  int32_t *d_order = nullptr, *d_col_exp = nullptr;
  uint32_t* d_qam = nullptr;
  uint32_t* d_bitsS = nullptr;
  long long* d_r_int = nullptr;
  long long* d_fix_ws[2] = {nullptr, nullptr};  // weighted fix-up: one zeroed int64[B] per CTA, per compute stream
  uint8_t* d_need = nullptr;
  double *d_lenq = nullptr, *d_len_col = nullptr, *d_flag_u = nullptr, *d_qerr = nullptr;
  TcChunks d_chunks;
  float* d_lenf = nullptr;
  const double* d_mult = nullptr;  // FRC_FLAG_PRUNE: original nodes per node of the merged tree (Shared::node_mult)
  double *d_E = nullptr, *d_total = nullptr, *d_W = nullptr, *d_r = nullptr, *d_scratch = nullptr;
  float* d_A = nullptr;
  int32_t* d_K = nullptr;     // keyed -l tiles: key panels, same layout as d_A (resident only)
  uint32_t *d_bits = nullptr, *d_node_scratch = nullptr;
  void *d_P = nullptr, *d_Bh = nullptr, *d_Bl = nullptr;
  TcOperands* tc = nullptr;
  // -l as coded: per-sample post-order lists
  int64_t* d_list_ptr = nullptr;
  int32_t* d_list_id = nullptr;
  double* d_list_val = nullptr;
  int64_t list_cap = 0;

  Slot slots[kSlots];
  int n_slots = 0;
  int64_t max_band = 1;
  size_t next_enqueue = 0, next_deliver = 0;
  cudaEvent_t ev_h2d0 = nullptr, ev_h2d1 = nullptr, ev_embed0 = nullptr, ev_embed1 = nullptr;
  cudaEvent_t ev_run1 = nullptr, ev_join = nullptr, ev_bits = nullptr, ev_rsum = nullptr;
  cudaEvent_t ev_shard = nullptr;  // in-process exchange: this part's shard has been stored into every device
  bool run_timed = false, embed_timed = false;
  std::chrono::steady_clock::time_point t_host0;
};

}  // namespace

struct frc_job {
  frc_ctx* ctx = nullptr;
  bool own_ctx = false;
  Shared sh;
  std::vector<std::unique_ptr<Part>> parts;
  std::string err;
  frc_info_t info{};
  // delivery: the bands this process yields, in flat-index order
  struct Item { int part, idx; };
  std::vector<Item> order;
  size_t next_item = 0;
  int held_part = -1;   // part whose slot the caller currently reads
  int held_slot = -1;
  int64_t held_first = 0, held_count = 0;  // flat range of the run handed out last
  std::vector<int64_t> ex_index;           // frc_chunk_exceptions: the entries inside that range
  std::vector<double> ex_value;
  int read_mode = 0;    // 0 = not decided, 1 = frc_next (float64), 2 = frc_next_f32
  double* wide = nullptr;  // frc_next on a fast path: the one double buffer handed out (<= kWidePiece values)
  int64_t piece_first = 0, piece_off = 0, piece_end = 0;
  double create_ms = 0;
};

namespace {

#define PART_CUDA(p, expr)                                                                   \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      (p)->err = std::string(#expr) + ": " + cudaGetErrorString(_e);                         \
      cudaGetLastError();                                                                    \
      return (p)->rc = (_e == cudaErrorMemoryAllocation ? FRC_ERR_OOM : FRC_ERR_CUDA);       \
    }                                                                                        \
  } while (0)

int pfail(Part* p, int code, const std::string& msg) { p->err = msg; return p->rc = code; }
int fail(frc_job* j, int code, const std::string& msg) { j->err = msg; return code; }

template <class T>
T* dev_alloc(Part* p, size_t n) {
  cudaError_t e = cudaSuccess;
  void* q = p->dc->dev.alloc(n * sizeof(T), &e);
  if (!q) {
    p->err = "device allocation of " + std::to_string(n * sizeof(T)) + " bytes failed: " + cudaGetErrorString(e);
    p->rc = FRC_ERR_OOM;
  }
  return static_cast<T*>(q);
}
template <class T>
T* pin_alloc(Part* p, size_t n) {
  cudaError_t e = cudaSuccess;
  void* q = p->dc->pin.alloc(n * sizeof(T), &e);
  if (!q) {
    p->err = "pinned host allocation of " + std::to_string(n * sizeof(T)) + " bytes failed: " + cudaGetErrorString(e);
    p->rc = FRC_ERR_OOM;
  }
  return static_cast<T*>(q);
}

// A PairOut for n pairs.
int alloc_pair_out(Part* p, PairOut& o, int64_t n) {
  if (!(o.dev32 = dev_alloc<float>(p, n))) return p->rc;
  if (!(o.flagged = dev_alloc<uint32_t>(p, n))) return p->rc;
  if (!(o.n_flagged_host = pin_alloc<unsigned long long>(p, 1))) return p->rc;
  *o.n_flagged_host = 0;
  if (!(o.ex.count = pin_alloc<unsigned long long>(p, 1))) return p->rc;
  if (!(o.ex.index = pin_alloc<int64_t>(p, kMaxExceptions))) return p->rc;
  if (!(o.ex.value = pin_alloc<double>(p, kMaxExceptions))) return p->rc;
  o.ex.cap = kMaxExceptions;
  *o.ex.count = 0;
  return FRC_OK;
}

// Runs fn(part index) for every part: on the pool when there are several (each task binds its own
// device), inline otherwise.  Returns the first failing part's status.
int for_parts(frc_job* j, const std::function<int(Part*)>& fn) {
  const int n = static_cast<int>(j->parts.size());
  if (n == 1) {
    cudaSetDevice(j->parts[0]->dc->device);
    fn(j->parts[0].get());
  } else {
    Pool* pool = j->ctx->pool.get();
    const int T = std::min(n, pool->size());
    std::atomic<int> next{0};
    pool->run(T, [&](int) {
      for (int k = next.fetch_add(1); k < n; k = next.fetch_add(1)) {
        cudaSetDevice(j->parts[k]->dc->device);
        fn(j->parts[k].get());
      }
    });
  }
  for (auto& p : j->parts)
    if (p->rc) { j->err = p->err; return p->rc; }
  return FRC_OK;
}

// Multi-process sharding: maps the blocks of the symmetric heap that the peers have not seen yet (collective:
// every rank allocates the same sequence, so every rank gains the same blocks at the same time).
// *usable = false when SOME rank could not map a peer's block (no P2P between the GPUs, IPC unavailable in a
// container): the ranks agree on that with one more tiny exchange, and the caller falls back to the NCCL
// all-gather of the bit columns on every rank -- the decision has to be collective.
int sym_sync(Part* p, bool* usable) {
  frc_ctx* c = p->job->ctx;
  DevCtx* dc = p->dc;
  const int world = comm_world(c->comm), rank = comm_rank(c->comm);
  char failed = 0;
  while (c->sym_peer.size() < dc->sym.blocks.size()) {
    const size_t b = c->sym_peer.size();
    cudaIpcMemHandle_t mine;
    memset(&mine, 0, sizeof(mine));
    if (cudaIpcGetMemHandle(&mine, dc->sym.blocks[b].p) != cudaSuccess) { cudaGetLastError(); failed = 1; }
    std::vector<cudaIpcMemHandle_t> all(world);
    std::string cerr;
    if (!comm_all_gather_host(c->comm, &mine, sizeof(mine), all.data(), dc->stream[0], &cerr))
      return pfail(p, FRC_ERR_CUDA, cerr);
    std::vector<char*> bases(world, nullptr);
    for (int r = 0; r < world; ++r) {
      if (r == rank) { bases[r] = dc->sym.blocks[b].p; continue; }
      void* q = nullptr;
      if (failed || cudaIpcOpenMemHandle(&q, all[r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError();
        failed = 1;
        q = nullptr;
      }
      bases[r] = static_cast<char*>(q);
    }
    c->sym_peer.push_back(bases);
  }
  for (auto& blk : c->sym_peer)
    for (char* base : blk)
      if (!base) failed = 1;  // (a block that could not be mapped for an earlier job)
  std::vector<char> flags(world, 0);
  std::string cerr;
  if (!comm_all_gather_host(c->comm, &failed, 1, flags.data(), dc->stream[0], &cerr)) return pfail(p, FRC_ERR_CUDA, cerr);
  *usable = true;
  for (char f : flags) if (f) *usable = false;
  return FRC_OK;
}

// ------------------------------------------------------------------ embedding
// A per-sample array of the embedding that every part reads for ALL samples, at the same sample offsets everywhere.
struct ShardArray {
  void* (*on)(const Part*);  // the array on a part
  size_t sample_bytes;
  bool copy = true;  // false: the producing kernel stored the shard into every part itself (counted, not copied)
};
template <auto M> void* part_array(const Part* q) { return q->*M; }

// Makes the samples [rg.s0, rg.s1) of every array in `arrs`, built by this part, visible to the other parts (stream s)
// and adds the bytes that reach them to info.gather_bytes.  kNccl: one in-place all-gather group (rank r's slice is the
// r-th: the sharded plan puts shard r there), a barrier when nothing is copied; kInProcess: copies over NVLink.
int exchange_shard(Part* p, const std::vector<ShardArray>& arrs, const Range& rg, cudaStream_t s) {
  const Shared& sh = *p->sh;
  if (sh.variant.exchange == Variant::kNone) return FRC_OK;
  const size_t n = static_cast<size_t>(rg.s1 - rg.s0);
  const int others = (sh.variant.exchange == Variant::kNccl ? sh.world : sh.n_parts) - 1;
  std::vector<void*> bufs;
  std::vector<size_t> bytes;
  for (const ShardArray& a : arrs) {
    p->info.gather_bytes += static_cast<int64_t>(n * a.sample_bytes) * others;
    if (a.copy) { bufs.push_back(a.on(p)); bytes.push_back(n * a.sample_bytes); }
  }
  if (sh.variant.exchange == Variant::kNccl) {
    Comm* comm = p->job->ctx->comm;
    std::string cerr;
    const bool ok = bufs.empty() ? comm_barrier(comm, s, &cerr)
                                 : comm_all_gather_inplace(comm, bufs.data(), bytes.data(), static_cast<int>(bufs.size()), s, &cerr);
    return ok ? FRC_OK : pfail(p, FRC_ERR_CUDA, cerr);
  }
  for (int q = 0; q < sh.n_parts; ++q) {
    if (q == p->index) continue;
    const Part* o = p->job->parts[q].get();
    for (const ShardArray& a : arrs) {
      if (!a.copy) continue;
      const size_t off = rg.s0 * a.sample_bytes;
      PART_CUDA(p, cudaMemcpyPeerAsync(static_cast<char*>(a.on(o)) + off, o->dc->device, static_cast<char*>(a.on(p)) + off,
                                       p->dc->device, n * a.sample_bytes, s));
    }
  }
  return FRC_OK;
}

// Stage 1 of the embedding on stream 0 of the part: everything up to (and including) the point where this
// part's sample shard has been made visible to the other devices.  Unsharded jobs run the whole embedding here.
int embed_stage1(Part* p) {
  const Shared& sh = *p->sh;
  const Variant& v = sh.variant;
  DevCtx* dc = p->dc;
  frc_ctx* c = p->job->ctx;
  cudaStream_t s = dc->stream[0];
  int launches = 0;
  p->t_host0 = std::chrono::steady_clock::now();
  if (p->d_flag_counts)
    PART_CUDA(p, cudaMemsetAsync(p->d_flag_counts, 0, sizeof(unsigned long long) * (p->mine.size() + 1), s));
  PART_CUDA(p, cudaEventRecord(p->ev_embed0, s));
  p->info.gather_bytes = 0;
  if (sh.exact) {
    launches += launch_embed_f64(p->dtree, sh.level_ptr.data(), p->dcsr, p->d_E, sh.np, 0, s);
    // (normalisation cannot change membership, which is all the unweighted kernel reads -- and a
    // proportion that underflows to 0 would drop a node the reference keeps)
    if (sh.opts.normalize == 1 && sh.weighted) {
      launches += launch_totals_f64(p->d_E, sh.B, sh.np, sh.N, p->d_total, s);
      launches += launch_normalize_f64(p->d_E, sh.B, sh.np, sh.N, p->d_total, s);
    }
    if (sh.unsorted_l) {
      // per-sample lists in post-order; their total size is only known after the counting pass
      launches += launch_postorder_lists(p->d_E, p->d_post, sh.B, sh.np, sh.N, p->d_list_ptr, nullptr, nullptr, s);
      int64_t total = 0;
      PART_CUDA(p, cudaMemcpyAsync(&total, p->d_list_ptr + sh.N, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
      PART_CUDA(p, cudaStreamSynchronize(s));
      if (total > p->list_cap) {
        p->list_cap = total;
        if (!(p->d_list_id = dev_alloc<int32_t>(p, static_cast<size_t>(total) + 1))) return p->rc;
        if (!(p->d_list_val = dev_alloc<double>(p, static_cast<size_t>(total) + 1))) return p->rc;
      }
      launches += launch_postorder_lists(p->d_E, p->d_post, sh.B, sh.np, sh.N, p->d_list_ptr, p->d_list_id,
                                         p->d_list_val, s);
    }
    p->info.embed_bytes = 2LL * sh.B * sh.np * 8 + 12LL * sh.nnz;
  } else if (sh.weighted) {
    // fast weighted: the fp64 embedding is built one slab of samples at a time (E[B][slab] stays
    // <= 2 GB whatever the sample count) and leaves as the fp32 tile-panel operand + denominators;
    // a part of a sharded job only builds the slabs of its own sample shard
    const bool norm = sh.opts.normalize == 1;
    // what the other devices read of a shard, in the order of the NCCL group: panels (unless they stay sharded:
    // capacity mode), denominators, normalisers, key panels
    std::vector<ShardArray> arrs;
    if (!v.capacity) arrs.push_back({part_array<&Part::d_A>, sizeof(float) * sh.kp});
    arrs.push_back({part_array<&Part::d_W>, sizeof(double)});
    if (norm) arrs.push_back({part_array<&Part::d_total>, sizeof(double)});
    if (sh.keyed) arrs.push_back({part_array<&Part::d_K>, sizeof(int32_t) * sh.kp});
    int64_t built = 0;
    for (const Range& rg : sh.shards.ranges[p->owner]) {
      built += rg.s1 - rg.s0;
      // panels are addressed by GLOBAL sample inside the kernel: shift the base so that the range lands in its
      // local slot (resident: the slot is the range's global place, no shift)
      const int64_t shift = (rg.slot * sh.shards.shard_rows - rg.s0) * sh.kp;
      float* Ap = p->d_A + shift;
      int32_t* Kp = sh.keyed ? p->d_K + shift : nullptr;
      for (int64_t sb = rg.s0; sb < rg.s1; sb += p->ws_slab) {
        const int64_t ld = std::min<int64_t>(p->ws_slab, rg.s1 - sb);
        // (keyed: the key panels of the slab are built by the same scatter + level passes)
        launches += launch_embed_f64(p->dtree, sh.level_ptr.data(), p->dcsr, p->d_E, ld, sb, s, Kp, sh.kp);
        if (norm) launches += launch_totals_fast_f64(p->d_E, sh.B, ld, p->d_mult, p->d_total + sb, p->d_scratch, s);
        launches += launch_weighted_operand_panels(p->d_E, p->dtree.length, sh.B, sh.kp, ld, sb,
                                                   norm ? p->d_total + sb : nullptr, sh.prescale, Ap, p->d_W,
                                                   p->d_scratch, s);
      }
      if (exchange_shard(p, arrs, rg, s)) return p->rc;
    }
    p->pm = PanelMap{};
    if (v.capacity) {
      // own shards in their slots; the visiting shards are filled in by the rotation (start_pairs_capacity)
      p->pm.n_shards = sh.shards.n_shards;
      p->pm.tiles_per_shard = static_cast<int32_t>(sh.shards.shard_rows / kTile);
      for (int k = 0; k < sh.shards.n_shards; ++k)
        if (sh.shards.owner[k] == p->owner) p->pm.shard[k] = p->d_A + sh.shards.slot[k] * sh.shards.shard_rows * sh.kp;
    } else {
      p->pm.shard[0] = p->d_A;
    }
    // write each element once, read it once when folded into its parent (+ CSR; keyed: + the int32 keys)
    p->info.embed_bytes = 2LL * sh.B * built * (sh.keyed ? 12 : 8) + 12LL * (p->csr_k1 - p->csr_k0);
  } else if (v.fused_embed) {
    const int cur = static_cast<int>(p->run_count & 1);
    if (p->peer_push) {
      p->d_bits = p->d_bits2[cur];
      if (p->run_count == 0) {  // nobody may still be reading these buffers for an earlier job
        std::string cerr;
        if (!comm_barrier(c->comm, s, &cerr)) return pfail(p, FRC_ERR_CUDA, cerr);
      }
    }
    ++p->run_count;
    PeerPtrs peers;  // n = 0: local stores only
    if (p->peer_push) peers = p->peers[cur];
    else if (v.peer_store) {
      // in-process sharding: the kernel stores its finished bit columns straight into every device's
      // bitsT (peer access over NVLink): the all-gather is fused into the producing kernel
      peers.n = sh.n_parts; peers.self = p->index;
      for (int q = 0; q < sh.n_parts; ++q) peers.p[q] = p->job->parts[q]->d_bits;
    }
    launches += launch_embed_presence_fused(p->dtree, p->d_level_ptr, p->dcsr, sh.nw, p->shard_w0, p->shard_nw,
                                            sh.kp, p->d_order, p->d_node_scratch, p->d_bits, p->d_bitsS, peers, s);
    // Row sums: made by the operand expansion of stage 2 (integer mode with materialised operands: nothing to
    // exchange but the bit columns), or by a pass over this part's shard here (Variant::rowsum_split: beside the
    // expansion on the second compute stream).
    cudaStream_t rs = v.rowsum_split ? dc->stream[1] : s;
    if (v.rowsum_split) {
      PART_CUDA(p, cudaEventRecord(p->ev_bits, s));
      PART_CUDA(p, cudaStreamWaitEvent(rs, p->ev_bits, 0));
    }
    if (!v.rowsum_in_expand)
      launches += launch_presence_rowsum_t(p->d_bits, sh.B, sh.nw, p->shard_w0, p->shard_nw, sh.kp, p->d_lenq,
                                           sh.cols.i8 ? p->d_qam : nullptr, p->d_col_exp, p->d_scratch, p->d_r,
                                           sh.cols.e_min, sh.cols.intacc ? p->d_r_int : nullptr, rs);
    // what the other parts read of the shard: row sums (unless the expansion makes them) and bit columns (2.5 GB at
    // cfg4 instead of 120 GB of operands; bits-fed: the bit rows, same size), unless the kernel above stored them.
    std::vector<ShardArray> arrs;
    if (!v.rowsum_in_expand)
      arrs.push_back({sh.cols.intacc ? part_array<&Part::d_r_int> : part_array<&Part::d_r>, sizeof(double)});
    arrs.push_back({v.bits_feed ? part_array<&Part::d_bitsS> : part_array<&Part::d_bits>, sizeof(uint32_t) * sh.kp / 32,
                    peers.n == 0});
    if (exchange_shard(p, arrs, sh.shards.ranges[p->owner][0], s)) return p->rc;
    if (v.exchange != Variant::kNone) {
      // bits written + read once per level pass (+ CSR cols): this part's shard
      p->info.embed_bytes = 2LL * sh.B * p->shard_nw * 4 + 4LL * (p->csr_k1 - p->csr_k0);
    }
  }
  PART_CUDA(p, cudaGetLastError());
  if (v.exchange == Variant::kInProcess) PART_CUDA(p, cudaEventRecord(p->ev_shard, s));
  p->info.kernel_launches += launches;
  return FRC_OK;
}

// Stage 2: wait for the other devices' shards, then whatever every device does for ALL samples.
int embed_stage2(Part* p) {
  const Shared& sh = *p->sh;
  DevCtx* dc = p->dc;
  cudaStream_t s = dc->stream[0];
  int launches = 0;
  const Variant& v = sh.variant;
  if (v.exchange == Variant::kInProcess)
    for (auto& o : p->job->parts)
      if (o.get() != p) PART_CUDA(p, cudaStreamWaitEvent(s, o->ev_shard, 0));
  if (!sh.exact && !sh.weighted) {
    if (v.fused_embed) {
      if (!v.bits_feed)
        launches += launch_expand_operands_t(p->d_bits, sh.nw, sh.kp, sh.np, sh.cols.i8, p->d_q0, p->d_q1, p->d_q2,
                                             p->d_P, p->d_Bh, p->d_Bl, p->d_need, p->d_qam, p->d_col_exp, sh.cols.e_min,
                                             v.rowsum_in_expand ? p->d_r_int : nullptr, s);
      if (v.rowsum_split) {
        PART_CUDA(p, cudaEventRecord(p->ev_rsum, dc->stream[1]));
        PART_CUDA(p, cudaStreamWaitEvent(s, p->ev_rsum, 0));
      }
      if (v.exchange == Variant::kNone) p->info.embed_bytes = 2LL * sh.B * sh.nw * 4 + 4LL * sh.nnz;
      // + three operands written once, the bit columns read once more
      if (!v.bits_feed) p->info.embed_bytes += 3LL * sh.np * sh.kp * (sh.cols.i8 ? 1 : 2) + 4LL * sh.nw * sh.kp;
    } else {
      launches += launch_embed_bits(p->dtree, sh.level_ptr.data(), p->dcsr, p->d_bits, sh.nw, s);
      launches += launch_presence_rowsum(p->d_bits, sh.B, sh.nw, p->d_lenq, p->d_r, p->d_scratch, s);
      launches += launch_expand_operands(p->d_bits, sh.B, sh.nw, sh.kp, sh.np,
                                         static_cast<const uint16_t*>(p->d_q1), static_cast<const uint16_t*>(p->d_q2),
                                         static_cast<uint16_t*>(p->d_P), static_cast<uint16_t*>(p->d_Bh),
                                         static_cast<uint16_t*>(p->d_Bl), s);
      p->info.embed_bytes = 2LL * sh.B * sh.nw * 4 + 3LL * sh.np * sh.kp * 2 + 4LL * sh.nnz;
    }
  }
  PART_CUDA(p, cudaGetLastError());
  PART_CUDA(p, cudaEventRecord(p->ev_embed1, s));
  PART_CUDA(p, cudaStreamWaitEvent(dc->stream[1], p->ev_embed1, 0));
  p->info.kernel_launches += launches;
  p->embed_timed = false;
  return FRC_OK;
}

// Fast paths: the tile kernel over n tiles into record o, whose first pair has flat index `first`; *cnt counts the
// flagged pairs.  (pm: where the weighted panels are; the capacity mode passes the visiting shards.)
int launch_tiles(Part* p, const PanelMap& pm, const Tile* tiles, int32_t n, int64_t first, const PairOut& o,
                 unsigned long long* cnt, cudaStream_t s) {
  const Shared& sh = *p->sh;
  if (sh.weighted)
    return launch_weighted_tiles(pm, sh.np, sh.kp, p->d_lenf, sh.prescale, p->d_W, tiles, n, sh.N, first, sh.geo, o.dev32,
                                 kFlagBelowW, o.flagged, cnt, p->dc->num_sms, s, p->d_K);
  return launch_unweighted_tc(p->tc, p->d_r, tiles, n, sh.N, first, sh.geo, o.dev32, kFlagBelow, o.flagged, cnt,
                              p->dc->num_sms, s);
}

// ... and the fix-up of the pairs it flagged (ws: the weighted fix-up's workspace).
int launch_fixup(Part* p, const PairOut& o, const unsigned long long* cnt, int64_t first, long long* ws, cudaStream_t s) {
  const Shared& sh = *p->sh;
  if (sh.weighted)
    return launch_weighted_fixup(p->dcsr, p->dtree, sh.opts.normalize == 1 ? p->d_total : nullptr, p->d_W, o.flagged, cnt,
                                 o.n_flagged_host, first, sh.geo, ws, kFixupCtas, o.dev32, o.ex, s, p->d_K, sh.kp);
  return launch_unweighted_fixup(p->tc, o.flagged, cnt, o.n_flagged_host, first, sh.geo, o.dev32, o.ex, p->dc->num_sms, s);
}

// Queue the way of band mine[idx] to the host on stream s, after `ready` unless that is null: the D2H into its slot,
// the slot's `done` event and, after the part's last band, the join of the streams and the end-of-run stamp.
int hand_off_band(Part* p, size_t idx, cudaEvent_t ready, cudaStream_t s) {
  const Shared& sh = *p->sh;
  DevCtx* dc = p->dc;
  const Slot& sl = p->slots[idx % p->n_slots];
  if (ready) PART_CUDA(p, cudaStreamWaitEvent(s, ready, 0));
  if (sh.d2h) {
    const int64_t bytes = (sh.exact ? sizeof(double) : sizeof(float)) * p->bands[idx].count;
    if (sh.exact) PART_CUDA(p, cudaMemcpyAsync(sl.host64, sl.dev64, bytes, cudaMemcpyDeviceToHost, s));
    else PART_CUDA(p, cudaMemcpyAsync(sl.host32, sl.out->dev32 + sl.out_off, bytes, cudaMemcpyDeviceToHost, s));
    p->info.d2h_bytes += bytes;
  }
  PART_CUDA(p, cudaEventRecord(sl.done, s));
  if (idx + 1 == p->mine.size()) {
    // last band queued: join all streams and stamp the end of the run on stream 0
    PART_CUDA(p, cudaEventRecord(p->ev_join, dc->stream[1]));
    PART_CUDA(p, cudaStreamWaitEvent(dc->stream[0], p->ev_join, 0));
    PART_CUDA(p, cudaStreamWaitEvent(dc->stream[0], sl.done, 0));
    PART_CUDA(p, cudaEventRecord(p->ev_run1, dc->stream[0]));
  }
  return FRC_OK;
}

// Queue band mine[idx] of the part into its slot.
int enqueue_band(Part* p, size_t idx) {
  const Shared& sh = *p->sh;
  DevCtx* dc = p->dc;
  if (sh.knobs.trace)
    fprintf(stderr, "[host] dev %d enqueue band %zu at %.3f ms\n", dc->device, idx,
            std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - p->t_host0).count());
  const Band& b = p->bands[idx];
  Slot& sl = p->slots[idx % p->n_slots];
  const int si = static_cast<int>(idx % 2);
  cudaStream_t s = dc->stream[si];
  int launches = 0;
  if (sh.variant.capacity) {
    // the band was (or is being) computed by the rotation into its group's record
    Part::CapGroup& cb = p->cap[p->band_group[idx]];
    sl.out = &cb.out;
    sl.out_off = b.first - cb.first;
    return hand_off_band(p, idx, cb.done, dc->stream[2]);
  }
  PART_CUDA(p, cudaEventRecord(sl.k0, s));
  if (sh.exact) {
    if (sh.unsorted_l)
      launches += launch_unsorted_pairs(p->d_list_ptr, p->d_list_id, p->d_list_val, p->dtree.length, b.first, sh.geo,
                                        b.count, sl.dev64, s);
    else
      launches += launch_exact_pairs(p->d_E, p->dtree.length, sh.B, sh.np, sh.weighted, b.first, sh.geo, b.count,
                                     sl.dev64, s);
    PART_CUDA(p, cudaEventRecord(sl.k1, s));
  } else {
    // no copy-engine work between the kernels: a memset or an 8-byte D2H would queue behind the
    // previous band's bulk D2H and stall this band (measured).  Counters are per band, zeroed once
    // per run; the fix-up kernel publishes the count through mapped pinned memory.
    unsigned long long* cnt = p->d_flag_counts + idx;
    sl.out = &sl.own;      // (at offset 0)
    *sl.own.ex.count = 0;  // (the slot's previous band has been delivered)
    sl.own.counted = false;
    launches += launch_tiles(p, p->pm, p->d_tiles + b.tile_off, b.n_tiles, b.first, sl.own, cnt, s);
    PART_CUDA(p, cudaEventRecord(sl.k1, s));
    // (one weighted workspace per compute stream: consecutive bands run their fix-ups concurrently)
    launches += launch_fixup(p, sl.own, cnt, b.first, p->d_fix_ws[si], s);
  }
  PART_CUDA(p, cudaGetLastError());
  PART_CUDA(p, cudaEventRecord(sl.k2, s));
  p->info.kernel_launches += launches;
  // bulk D2H runs on its own stream so the compute streams never hold copy-engine work
  // (a kernel queued behind a copy in the same stream cannot overlap that copy)
  return sh.d2h ? hand_off_band(p, idx, sl.k2, dc->stream[2]) : hand_off_band(p, idx, nullptr, s);
}

// Capacity mode of the fast weighted path: queue the WHOLE pair stage of this part.  The column shards
// 0, 1, ... visit the device one at a time: a shard of another device is copied into one of two visiting buffers
// by the copy engines (device-to-device over NVLink, on its own stream, while the previous shard is in use), and
// for every visiting shard c one launch per band covers the tiles (rows of the band) x (columns of shard c).  A
// band is complete -- fix-up, then its `done` event -- once the shard of its own rows has passed.  Every remote
// shard crosses NVLink exactly once per device and pass; the tile kernel itself only ever reads local HBM.
int start_pairs_capacity(Part* p) {
  const Shared& sh = *p->sh;
  DevCtx* dc = p->dc;
  cudaStream_t s = dc->stream[0], cin = dc->stream[3];
  const ShardPlan& sp = sh.shards;
  const size_t shard_floats = static_cast<size_t>(sp.shard_rows) * sh.kp;
  int launches = 0, n_remote = 0, last_c = 0;
  for (const Part::CapGroup& cb : p->cap) last_c = std::max(last_c, cb.shard);
  PanelMap pm = p->pm;  // own shards set by the embedding stage
  int prev_user[2] = {-1, -1};
  int64_t fetched = 0;
  for (Part::CapGroup& cb : p->cap) { *cb.out.ex.count = 0; cb.out.counted = false; }
  for (int c = 0; c <= last_c; ++c) {
    const bool remote = sp.owner[c] != p->index;
    if (remote) {
      const int buf = n_remote++ & 1;
      Part* o = p->job->parts[sp.owner[c]].get();
      const float* src = o->d_A + sp.slot[c] * shard_floats;
      if (prev_user[buf] >= 0) PART_CUDA(p, cudaStreamWaitEvent(cin, p->ev_used[prev_user[buf]], 0));
      PART_CUDA(p, cudaStreamWaitEvent(cin, o->ev_shard, 0));  // the owner has built it
      PART_CUDA(p, cudaMemcpyPeerAsync(p->d_V[buf], dc->device, src, o->dc->device, shard_floats * sizeof(float), cin));
      PART_CUDA(p, cudaEventRecord(p->ev_fetch[c], cin));
      PART_CUDA(p, cudaStreamWaitEvent(s, p->ev_fetch[c], 0));
      pm.shard[c] = p->d_V[buf];
      prev_user[buf] = c;
      fetched += static_cast<int64_t>(shard_floats * sizeof(float));
    }
    for (size_t k = 0; k < p->cap.size(); ++k) {
      const Part::CapGroup& cb = p->cap[k];
      if (cb.shard < c) continue;
      unsigned long long* cnt = p->d_flag_counts + k;  // (zeroed with the bands' counters: a part has no fewer bands)
      const int32_t t0 = cb.coff[c], n = cb.coff[c + 1] - cb.coff[c];
      launches += launch_tiles(p, pm, p->d_tiles + cb.tile_off + t0, n, cb.first, cb.out, cnt, s);
      if (cb.shard == c) {
        launches += launch_fixup(p, cb.out, cnt, cb.first, p->d_fix_ws[0], s);
        PART_CUDA(p, cudaEventRecord(cb.done, s));
      }
    }
    PART_CUDA(p, cudaGetLastError());
    if (remote) PART_CUDA(p, cudaEventRecord(p->ev_used[c], s));
  }
  p->info.gather_bytes += fetched;
  p->info.kernel_launches += launches;
  return FRC_OK;
}

int start_pairs(Part* p) {
  p->next_enqueue = p->next_deliver = 0;
  p->info.pairs_ms = 0;
  p->info.fixup_ms = 0;
  p->info.run_ms = 0;
  p->run_timed = false;
  p->info.flagged_pairs = 0;
  p->info.exceptions = 0;
  p->info.d2h_bytes = 0;
  if (p->mine.empty()) {  // nothing to compute: the run ends with the embedding
    PART_CUDA(p, cudaEventRecord(p->ev_run1, p->dc->stream[0]));
    return FRC_OK;
  }
  if (p->sh->variant.capacity && start_pairs_capacity(p)) return p->rc;
  // keep one slot free for the band the caller is still reading
  while (p->next_enqueue < p->mine.size() && p->next_enqueue < static_cast<size_t>(p->n_slots - 1)) {
    if (enqueue_band(p, p->next_enqueue)) return p->rc;
    ++p->next_enqueue;
  }
  return FRC_OK;
}

void destroy_part(Part* p) {
  if (!p) return;
  if (p->dc) {
    cudaSetDevice(p->dc->device);
    for (auto s : p->dc->stream) if (s) cudaStreamSynchronize(s);
    cudaGetLastError();
  }
  for (auto& sl : p->slots) {
    if (sl.k0) cudaEventDestroy(sl.k0);
    if (sl.k1) cudaEventDestroy(sl.k1);
    if (sl.k2) cudaEventDestroy(sl.k2);
    if (sl.done) cudaEventDestroy(sl.done);
  }
  for (cudaEvent_t e : {p->ev_h2d0, p->ev_h2d1, p->ev_embed0, p->ev_embed1, p->ev_run1, p->ev_join, p->ev_bits,
                        p->ev_rsum, p->ev_shard})
    if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : p->ev_fetch) if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : p->ev_used) if (e) cudaEventDestroy(e);
  for (auto& cb : p->cap) if (cb.done) cudaEventDestroy(cb.done);
  tc_operands_destroy(p->tc);
  if (p->dc) {
    p->dc->dev.reset();
    p->dc->pin.reset();
    p->dc->sym.reset();
  }
}

void destroy_job(frc_job* j) {
  if (!j) return;
  // every device must be idle before any part's memory is recycled (peers store into each other's buffers)
  for (auto& p : j->parts)
    if (p->dc) {
      cudaSetDevice(p->dc->device);
      for (auto s : p->dc->stream) if (s) cudaStreamSynchronize(s);
    }
  cudaGetLastError();
  for (auto& p : j->parts) destroy_part(p.get());
  if (j->ctx) {
    j->ctx->pin.reset();
    j->ctx->in_use = false;
    if (j->own_ctx) frc_ctx_destroy(j->ctx);
  }
  delete j;
}

int make_dev_ctx(int device, DevCtx** out) {
  cudaError_t e;
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    g_create_error = std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e);
    return FRC_ERR_CUDA;
  }
  if (prop.major != 10) {
    g_create_error = "libfrcfrc_cuda is built for sm_100a (B200) only; device " + std::to_string(device) +
                     " is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) + " (" + prop.name + ")";
    return FRC_ERR_UNSUPPORTED;
  }
  if ((e = cudaSetDevice(device)) != cudaSuccess) {
    g_create_error = std::string("cudaSetDevice: ") + cudaGetErrorString(e);
    return FRC_ERR_CUDA;
  }
  DevCtx* d = new DevCtx();
  d->device = device;
  d->num_sms = prop.multiProcessorCount;
  d->dev.pinned = false; d->dev.min_block = 64u << 20;
  d->sym.pinned = false; d->sym.min_block = 32u << 20;
  d->pin.pinned = true;  d->pin.min_block = 8u << 20;
  *out = d;
  for (auto& s : d->stream)
    if ((e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking)) != cudaSuccess) {
      g_create_error = std::string("cudaStreamCreate: ") + cudaGetErrorString(e);
      return FRC_ERR_CUDA;
    }
  // function attributes live in the device's context: once per device, not once per process
  std::string terr;
  if (!tc_setup(&terr)) { g_create_error = terr; return FRC_ERR_CUDA; }
  weighted_setup();
  embed_setup();
  if ((e = cudaGetLastError()) != cudaSuccess) {
    g_create_error = std::string("kernel attribute setup: ") + cudaGetErrorString(e);
    return FRC_ERR_CUDA;
  }
  return FRC_OK;
}

}  // namespace

extern "C" {

int frc_abi_version(void) { return FRC_ABI_VERSION; }

const char* frc_last_error(const frc_job_t* job) { return job ? job->err.c_str() : g_create_error.c_str(); }

int frc_ctx_create_multi(int32_t n_devices, const int32_t* devices, frc_ctx_t** out) {
  if (!out) { g_create_error = "frc_ctx_create: out is NULL"; return FRC_ERR_ARG; }
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    cudaGetLastError();
    g_create_error = std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count is 0");
    return FRC_ERR_CUDA;
  }
  DeviceGuard guard;
  std::vector<int> ids;
  if (n_devices < 0) {  // every visible sm_100 device
    for (int d = 0; d < count && static_cast<int>(ids.size()) < kMaxParts; ++d) {
      cudaDeviceProp prop;
      if (cudaGetDeviceProperties(&prop, d) == cudaSuccess && prop.major == 10) ids.push_back(d);
    }
    if (ids.empty()) { g_create_error = "no sm_100 device visible (libfrcfrc_cuda is built for B200 only)"; return FRC_ERR_UNSUPPORTED; }
  } else {
    if (n_devices == 0) n_devices = 1;
    if (n_devices > kMaxParts) { g_create_error = "at most 8 devices per job"; return FRC_ERR_UNSUPPORTED; }
    for (int k = 0; k < n_devices; ++k) {
      int d = devices ? devices[k] : k;
      if (n_devices == 1 && d < 0) { if (guard.prev >= 0) d = guard.prev; else d = 0; }
      if (d < 0 || d >= count) { g_create_error = "device ordinal out of range"; return FRC_ERR_ARG; }
      for (int x : ids) if (x == d) { g_create_error = "device listed twice"; return FRC_ERR_ARG; }
      ids.push_back(d);
    }
  }
  frc_ctx* c = new frc_ctx();
  c->pin.pinned = true; c->pin.min_block = 8u << 20;
  for (int d : ids) {
    DevCtx* dc = nullptr;
    int rc = make_dev_ctx(d, &dc);
    if (dc) c->devs.push_back(dc);
    if (rc) { frc_ctx_destroy(c); return rc; }
  }
  if (c->devs.size() > 1) {
    // peer access between every pair (NVLink on an HGX board): lets the embedding kernel of one device store
    // into the others' HBM.  Without it the devices work independently (each rebuilds the embedding).
    bool ok = true;
    for (DevCtx* a : c->devs)
      for (DevCtx* b : c->devs) {
        if (a == b) continue;
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, a->device, b->device) != cudaSuccess || !can) { ok = false; continue; }
        cudaSetDevice(a->device);
        cudaError_t pe = cudaDeviceEnablePeerAccess(b->device, 0);
        if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) ok = false;
        cudaGetLastError();
      }
    c->peer_ok = ok;
  }
  {
    int hw = static_cast<int>(std::thread::hardware_concurrency());
    int n = std::max(1, std::min(16, hw));
    if (c->devs.size() > 1) n = std::max(n, std::min(hw, 32));  // several rings to serve
    if (const char* ev = getenv("FRC_HOST_THREADS")) n = std::max(1, atoi(ev));
    c->pool.reset(new Pool(n - 1));
    c->stamps.resize(n);
  }
  *out = c;
  return FRC_OK;
}

int frc_ctx_create(int32_t device, frc_ctx_t** out) { return frc_ctx_create_multi(1, &device, out); }

void frc_ctx_destroy(frc_ctx_t* c) {
  if (!c) return;
  DeviceGuard guard;
  c->pool.reset();
  for (DevCtx* d : c->devs) {
    cudaSetDevice(d->device);
    for (auto s : d->stream) if (s) cudaStreamSynchronize(s);
  }
  if (!c->devs.empty()) {
    DevCtx* d0 = c->devs[0];
    cudaSetDevice(d0->device);
    for (size_t b = 0; b < c->sym_peer.size(); ++b)
      for (size_t r = 0; r < c->sym_peer[b].size(); ++r)
        if (c->sym_peer[b][r] && c->sym_peer[b][r] != d0->sym.blocks[b].p) cudaIpcCloseMemHandle(c->sym_peer[b][r]);
    c->sym_peer.clear();
    comm_destroy(c->comm);
    c->comm = nullptr;
  }
  for (DevCtx* d : c->devs) {
    cudaSetDevice(d->device);
    d->sym.release();
    for (auto s : d->stream) if (s) cudaStreamDestroy(s);
    d->dev.release();
    d->pin.release();
    delete d;
  }
  c->pin.release();
  cudaGetLastError();
  delete c;
}

int frc_comm_unique_id(char* id) {
  if (!id) { g_create_error = "frc_comm_unique_id: id is NULL"; return FRC_ERR_ARG; }
  std::string err;
  if (!comm_unique_id(id, &err)) { g_create_error = err; return FRC_ERR_UNSUPPORTED; }
  return FRC_OK;
}

int frc_ctx_comm_init(frc_ctx_t* ctx, const char* id, int32_t rank, int32_t world) {
  if (!ctx || !id || world < 1 || rank < 0 || rank >= world) {
    g_create_error = "frc_ctx_comm_init: bad argument";
    return FRC_ERR_ARG;
  }
  if (ctx->in_use) { g_create_error = "context has a live job"; return FRC_ERR_STATE; }
  if (ctx->devs.size() != 1) { g_create_error = "a communicator joins one-device contexts (one process per GPU)"; return FRC_ERR_STATE; }
  DeviceGuard guard;
  cudaSetDevice(ctx->devs[0]->device);
  comm_destroy(ctx->comm);
  ctx->comm = nullptr;
  std::string err;
  ctx->comm = comm_create(id, rank, world, &err);
  if (!ctx->comm) { g_create_error = err; return FRC_ERR_CUDA; }
  return FRC_OK;
}

}  // extern "C"

namespace {

// ------------------------------------------------------------------ frc_create, unit by unit
// The shape checks of one table; `name` is null for frc_create's table, "reference" / "query" for the two tables of
// frc_create_cross (their messages then name the table and the row within it).
int check_table(frc_job* j, const frc_csr_t* t, const char* name) {
  const std::string pre = name ? std::string(name) + " table: " : "";
  const int64_t N = t->n_samples;
  if (N < 0 || (N > 0 && !t->row_ptr)) return fail(j, FRC_ERR_ARG, pre + "bad abundance table");
  if (N > (1LL << 31) - 256) return fail(j, FRC_ERR_UNSUPPORTED, pre + "too many samples");
  const int64_t nnz = N > 0 ? t->row_ptr[N] : 0;
  if (N > 0 && t->row_ptr[0] != 0) return fail(j, FRC_ERR_ARG, pre + "row_ptr[0] != 0");
  if (nnz < 0 || (nnz > 0 && (!t->col || !t->val))) return fail(j, FRC_ERR_ARG, pre + "bad abundance table");
  for (int64_t s = 0; s < N; ++s)
    if (t->row_ptr[s + 1] < t->row_ptr[s] || t->row_ptr[s + 1] > nnz)
      return fail(j, FRC_ERR_ARG, name ? pre + "row_ptr is not monotone at " + name + " sample #" + std::to_string(s + 1)
                                       : std::string("row_ptr is not monotone"));
  return FRC_OK;
}

// (1) options and table header; fills the sizes of `sh`.  No CUDA call.  query != null: frc_create_cross, abnd is
// the reference table and the job stages [reference rows; empty rows up to q0; query rows] (Geometry).
int validate_header(frc_job* j, const frc_tree_t* tree, const frc_csr_t* abnd, const frc_csr_t* query,
                    const frc_opts_t* opts) {
  Shared& sh = j->sh;
  if (opts->mode != FRC_UNWEIGHTED && opts->mode != FRC_WEIGHTED) return fail(j, FRC_ERR_ARG, "bad mode");
  if (opts->path < FRC_PATH_AUTO || opts->path > FRC_PATH_EXACT) return fail(j, FRC_ERR_ARG, "bad path");
  if (opts->normalize < 0 || opts->normalize > 2) return fail(j, FRC_ERR_ARG, "bad normalize");
  if (opts->normalize != 1 && opts->mode != FRC_WEIGHTED)  // frcfrc.go:84-86
    return fail(j, FRC_ERR_ARG, "-l can only be used with weighted unifrac");
  // normalize = 0 runs the exact list walk unless the caller accepts the key-matched tiles (within 1e-5 instead of
  // bit-exact); the flag means nothing for the other modes
  const bool l_tiles = opts->normalize == 0 && (opts->flags & FRC_FLAG_L_TILES) != 0;
  if (opts->normalize == 0 && opts->path == FRC_PATH_FAST && !l_tiles)
    return fail(j, FRC_ERR_UNSUPPORTED, "normalize = 0 (flag -l as coded in the reference: unsorted merge-join) only "
                                        "exists on the exact path unless FRC_FLAG_L_TILES selects the key-matched FP32 "
                                        "tiles; normalize = 2 is the documented -l");
  const int world = opts->world <= 0 ? 1 : opts->world;
  const int rank = opts->world <= 0 ? 0 : opts->rank;
  if (rank < 0 || rank >= world) return fail(j, FRC_ERR_ARG, "rank outside [0, world)");
  if (opts->band_rows < 0) return fail(j, FRC_ERR_ARG, "band_rows < 0");
  if (query) {
    // one process, one ordered stream of the block: the multi-process forms (band sharding over ranks, the sharded
    // embedding) are triangle-only
    if (opts->world > 1)
      return fail(j, FRC_ERR_UNSUPPORTED, "frc_create_cross runs in one process (world <= 1); opts.n_devices spreads "
                                          "it over several GPUs");
    if (opts->flags & FRC_FLAG_SHARD_EMBED)
      return fail(j, FRC_ERR_UNSUPPORTED, "FRC_FLAG_SHARD_EMBED (one process per GPU) is not supported by "
                                          "frc_create_cross");
  }
  const int32_t B = tree->n_nodes;
  if (B < 1 || !tree->parent || !tree->length) return fail(j, FRC_ERR_ARG, "empty tree");
  if (tree->parent[0] != -1) return fail(j, FRC_ERR_ARG, "parent[0] must be -1 (root has pre-order id 0)");
  if (int rc = check_table(j, abnd, query ? "reference" : nullptr)) return rc;
  if (query)
    if (int rc = check_table(j, query, "query")) return rc;
  // (entries are validated while they are copied into the pinned staging buffer)
  int64_t N = abnd->n_samples;
  int64_t nnz = N > 0 ? abnd->row_ptr[N] : 0;
  int64_t n_pairs = N >= 2 ? tri(N) : 0;
  if (query) {
    const int64_t n_ref = N, n_q = query->n_samples;
    sh.geo.rect = true;
    sh.geo.n_ref = n_ref;
    sh.geo.q0 = round_up(n_ref, 2 * kTile);
    N = sh.geo.q0 + n_q;
    if (N > (1LL << 31) - 256) return fail(j, FRC_ERR_UNSUPPORTED, "too many samples");
    nnz += n_q > 0 ? query->row_ptr[n_q] : 0;
    n_pairs = n_q * n_ref;
  }
  sh.opts = *opts;
  sh.opts.devices = nullptr;  // (borrowed pointer: not kept)
  sh.weighted = opts->mode == FRC_WEIGHTED;
  sh.N = N; sh.B = B; sh.nnz = nnz;
  sh.world = world; sh.rank0 = rank;
  sh.d2h = !(opts->flags & FRC_FLAG_NO_D2H);
  if (opts->path == FRC_PATH_EXACT || (opts->normalize == 0 && !l_tiles)) sh.exact = true;
  else if (opts->path == FRC_PATH_FAST) sh.exact = false;
  else sh.exact = n_pairs == 0 || (static_cast<double>(n_pairs) * B <= static_cast<double>(kExactWorkLimit));
  sh.unsorted_l = opts->normalize == 0 && sh.exact;
  sh.keyed = opts->normalize == 0 && !sh.exact;
  sh.need_val = sh.exact || sh.weighted;
  return FRC_OK;
}

// (2) layout of the staged inputs.
void layout_inputs(Shared& sh) {
  SegAlloc seg;
  const int32_t B = sh.B;
  const int32_t kp_pad = static_cast<int32_t>(round_up(B, kKBlock));
  sh.in_rowptr = seg(sizeof(int64_t) * (sh.N + 1));
  sh.in_parent = seg(sizeof(int32_t) * B);
  sh.in_len = seg(sizeof(double) * B);
  sh.in_cptr = seg(sizeof(int32_t) * (B + 1));
  sh.in_cidx = seg(sizeof(int32_t) * B);
  sh.in_lvl = seg(sizeof(int32_t) * B);
  sh.in_lpar = seg(sizeof(int32_t) * B);
  sh.in_lptr = seg(sizeof(int32_t) * (static_cast<size_t>(B) + 2));
  sh.in_lenf = seg(sizeof(float) * kp_pad);
  sh.in_post = seg(sh.unsorted_l ? sizeof(int32_t) * B : 0);
  sh.in_mult = seg(sh.node_mult ? sizeof(double) * B : 0);
  sh.in_col = seg(sizeof(int32_t) * sh.nnz);   // the two bulk arrays last: a sharded part uploads a slice of them
  sh.in_val = seg(sh.need_val ? sizeof(double) * sh.nnz : 0);
  sh.in_bytes = seg.total;
}

// FRC_FLAG_PRUNE: the subtree the staged table observes, from the leaves listed in ANY of its rows, so that every
// rank of a sharded multi-process job derives the same tree.  Everything from the layout on runs on the pruned tree;
// the entries are still checked against the caller's tree (same checks, same node ids in the messages) and staged
// with their new ids.  A tree that fails the pre-order check is not pruned (false): the tree walks report it as they
// do without the flag.
bool prune_to_table(Shared& sh, Pool& pool, const frc_tree_t* tree, const StagedTable& table, PrunedTree* out) {
  const int32_t B = tree->n_nodes;
  std::vector<int32_t> depth(B);
  int32_t bad_parent = 0, bad_order = 0;
  if (!check_preorder(tree->parent, B, depth.data(), &bad_parent, &bad_order)) return false;
  std::vector<uint8_t> marks(B, 0);
  const int64_t nnz = sh.nnz;
  const int T = nnz >= 65536 ? pool.size() : 1;
  pool.run(T, [&](int t) { mark_table_leaves(table, nnz * t / T, nnz * (t + 1) / T, B, marks.data()); });
  // merging reorders the fp64 sums of the exact path: it is only pruned
  *out = prune_tree(tree->parent, tree->length, B, marks.data(), !sh.exact);
  sh.B = out->n_nodes;
  sh.node_mult = !sh.exact && sh.weighted && sh.opts.normalize == 1;
  return true;
}

// The two tree tasks of the staging (pool workers, while the entries are staged), on the tree the kernels use.
// Level order and level_ptr.
TreeLevels stage_tree_levels(const Shared& sh, const frc_tree_t* tree) {
  char* const st = sh.stage_in;
  TreeLevels levels = tree_levels(tree->parent, sh.B, reinterpret_cast<int32_t*>(st + sh.in_lvl.off),
                                  reinterpret_cast<int32_t*>(st + sh.in_lpar.off));
  if (levels.height >= 0) memcpy(st + sh.in_lptr.off, levels.level_ptr.data(), sizeof(int32_t) * (levels.height + 2));
  return levels;
}
// Children lists, parent / length, fp32 lengths, post-order (-l as coded), node multiplicities (mult: FRC_FLAG_PRUNE).
// false when a parent id is out of range.
bool stage_tree_children(const Shared& sh, const frc_tree_t* tree, const int32_t* mult) {
  char* const st = sh.stage_in;
  const int32_t B = sh.B;
  if (!tree_children(tree->parent, B, reinterpret_cast<int32_t*>(st + sh.in_cptr.off),
                     reinterpret_cast<int32_t*>(st + sh.in_cidx.off))) return false;
  memcpy(st + sh.in_parent.off, tree->parent, sizeof(int32_t) * B);
  memcpy(st + sh.in_len.off, tree->length, sizeof(double) * B);
  float* lf = reinterpret_cast<float*>(st + sh.in_lenf.off);
  const int32_t kp_pad = static_cast<int32_t>(round_up(B, kKBlock));
  for (int32_t v = 0; v < kp_pad; ++v) lf[v] = v < B ? static_cast<float>(tree->length[v]) : 0.f;
  if (sh.unsorted_l) tree_post_order(tree->parent, B, reinterpret_cast<int32_t*>(st + sh.in_post.off));
  if (sh.node_mult) {
    double* m = reinterpret_cast<double*>(st + sh.in_mult.off);
    for (int32_t v = 0; v < B; ++v) m[v] = mult[v];
  }
  return true;
}

// Branch lengths: bad = a non-finite one in the caller's tree (only the exact path handles it), neg = a negative
// finite one in the tree the kernels use.
void scan_lengths(const frc_tree_t* caller, const frc_tree_t* tree, bool* bad, bool* neg) {
  bool b = false, n = false;
  for (int32_t v = 0; v < caller->n_nodes; ++v) {
    const double l = caller->length[v];
    if (!(l == l) || std::isinf(l)) b = true;
  }
  for (int32_t v = 0; v < tree->n_nodes; ++v) {
    const double l = tree->length[v];
    if (l < 0 && !std::isinf(l)) n = true;
  }
  *bad = b; *neg = n;
}

// What the variant of the job depends on (plan_exchange, plan_variant).
VariantIn variant_in(const Shared& sh, const frc_ctx* c) {
  VariantIn in;
  in.exact = sh.exact; in.weighted = sh.weighted; in.keyed = sh.keyed; in.rect = sh.geo.rect;
  in.flags = sh.opts.flags; in.world = sh.world; in.rank = sh.rank0; in.N = sh.N;
  in.n_parts = sh.n_parts; in.peer_ok = c->peer_ok;
  if (c->comm) { in.comm_world = comm_world(c->comm); in.comm_rank = comm_rank(c->comm); }
  return in;
}

// (3) the plan that does not depend on the table: the variant and the operand columns; then bands + owners.
int plan_job(frc_job* j, const frc_tree_t* tree, bool neg_len) {
  Shared& sh = j->sh;
  frc_ctx* c = j->ctx;
  auto free_hbm = [c](size_t* free_b) {
    size_t total_b = 0;
    cudaSetDevice(c->devs[0]->device);
    const bool ok = cudaMemGetInfo(free_b, &total_b) == cudaSuccess;
    cudaGetLastError();
    return ok;
  };
  std::string err;
  if (int rc = plan_variant(sh.variant, variant_in(sh, c), sh.knobs, neg_len, tree->length, sh.B, tc_chunk_kblocks(),
                            free_hbm, &sh.cols, &err))
    return fail(j, rc, err);
  const int owners = sh.owners();
  sh.shards = plan_shards(sh.N, owners, sh.variant.shard_mode);
  sh.np = sh.shards.np;
  sh.nw = static_cast<int32_t>(sh.np / 32);
  sh.kp = !sh.exact && !sh.weighted ? sh.cols.kp : static_cast<int32_t>(round_up(sh.B, kKBlock));
  sh.prescale = !neg_len;
  if (sh.geo.rect)
    sh.bands = make_bands_cross(sh.geo.q0, sh.N - sh.geo.q0, sh.geo.n_ref, sh.opts.band_rows, owners, sh.d2h,
                                sh.knobs.bands_per_rank, 8);
  else
    sh.bands = sh.variant.capacity ? make_bands_capacity(sh.N, sh.shards, sh.opts.band_rows, sh.d2h)
                                   : make_bands(sh.N, sh.opts.band_rows, owners, sh.d2h, sh.knobs.bands_per_rank, 8);
  for (const Band& b : sh.bands)
    if (b.count >= (1LL << 32)) return fail(j, FRC_ERR_UNSUPPORTED, "band too large; lower band_rows");
  return FRC_OK;
}

// (4) the plan arrays every device receives, into pinned staging memory.
int stage_plan(frc_job* j, const frc_tree_t* tree) {
  Shared& sh = j->sh;
  const ColumnPlan& cp = sh.cols;
  SegAlloc seg;
  sh.pl_q0 = seg(sh.kp); sh.pl_hi = seg(sizeof(uint16_t) * sh.kp); sh.pl_lo = seg(sizeof(uint16_t) * sh.kp);
  sh.pl_lenq = seg(sizeof(double) * sh.kp);
  sh.pl_order = seg(sizeof(int32_t) * cp.col_order.size()); sh.pl_cexp = seg(sizeof(int32_t) * cp.col_exp.size());
  sh.pl_lcol = seg(sizeof(double) * cp.len_col.size()); sh.pl_cend = seg(sizeof(int32_t) * cp.chunk_end.size());
  sh.pl_cscale = seg(sizeof(double) * cp.chunk_scale.size()); sh.pl_cshift = seg(sizeof(int32_t) * cp.chunk_shift.size());
  sh.plan_bytes = seg.total;
  cudaError_t e = cudaSuccess;
  sh.stage_plan = static_cast<char*>(j->ctx->pin.alloc(sh.plan_bytes, &e));
  if (!sh.stage_plan) return fail(j, FRC_ERR_OOM, std::string("pinned staging: ") + cudaGetErrorString(e));
  char* st = sh.stage_plan;
  if (!sh.exact && !sh.weighted && !cp.i8) {  // (u8: k_quantize_lengths fills q0/q1/q2 and lenq on the device)
    uint16_t* hi = reinterpret_cast<uint16_t*>(st + sh.pl_hi.off);
    uint16_t* lo = reinterpret_cast<uint16_t*>(st + sh.pl_lo.off);
    double* lq = reinterpret_cast<double*>(st + sh.pl_lenq.off);
    for (int32_t v = 0; v < sh.B; ++v) {
      const double l = tree->length[v];
      hi[v] = bf16_rn(static_cast<float>(l));
      const double res = l - static_cast<double>(bf16_to_float(hi[v]));
      lo[v] = (l == l && !std::isinf(l)) ? bf16_rn(static_cast<float>(res)) : 0;
      lq[v] = static_cast<double>(bf16_to_float(hi[v])) + static_cast<double>(bf16_to_float(lo[v]));
    }
    for (int32_t v = sh.B; v < sh.kp; ++v) { hi[v] = 0; lo[v] = 0; lq[v] = 0.0; }
  }
  auto put = [&](const Seg& s, const void* src) { if (s.bytes) memcpy(st + s.off, src, s.bytes); };
  put(sh.pl_order, cp.col_order.data()); put(sh.pl_cexp, cp.col_exp.data()); put(sh.pl_lcol, cp.len_col.data());
  put(sh.pl_cend, cp.chunk_end.data()); put(sh.pl_cscale, cp.chunk_scale.data()); put(sh.pl_cshift, cp.chunk_shift.data());
  return FRC_OK;
}

// (5) per device: tiles of its bands, device buffers, ring slots, upload of the plan, tensor maps.
int prepare_part(Part* p) {
  const Shared& sh = *p->sh;
  DevCtx* dc = p->dc;
  frc_ctx* c = p->job->ctx;
  const int32_t B = sh.B;
  PART_CUDA(p, cudaSetDevice(dc->device));
  // ---- bands + tiles of this owner
  p->max_band = 1;
  for (size_t k = 0; k < sh.bands.size(); ++k)
    if (sh.bands[k].owner == p->owner) {
      p->mine.push_back(static_cast<int>(k));
      p->bands.push_back(sh.bands[k]);
      p->info.n_pairs_mine += sh.bands[k].count;
      p->max_band = std::max(p->max_band, sh.bands[k].count);
    }
  if (sh.variant.capacity) {
    // one group per row shard of this part (csrc/plan.cpp): its bands, and its tiles grouped by COLUMN SHARD (the
    // order the shards visit in), column-major inside a column shard (the CTAs of a wave share a column panel)
    const std::vector<CapGroupPlan> groups =
        plan_capacity_groups(p->bands, sh.N, sh.shards.shard_rows, sh.shards.n_shards, p->tiles, p->band_group);
    for (const CapGroupPlan& gp : groups) {
      if (gp.count >= (1LL << 32)) return pfail(p, FRC_ERR_UNSUPPORTED, "capacity mode: a row shard holds 2^32 pairs or more");
      Part::CapGroup g;
      g.shard = gp.shard; g.first = gp.first; g.count = gp.count; g.tile_off = gp.tile_off; g.coff = gp.coff;
      p->cap.push_back(g);
    }
  } else if (!sh.exact) {
    const int32_t col_tiles = sh.geo.rect ? static_cast<int32_t>((sh.geo.n_ref + kTile - 1) / kTile) : 0;
    for (Band& b : p->bands) append_band_tiles(b, !sh.weighted, p->tiles, col_tiles);
  }
  std::vector<uint8_t> need;
  if (sh.variant.need_blocks) need = operand_need_blocks(p->tiles, sh.np, true);
  // ---- sample shard: the first range of this owner (capacity: the second one is as large)
  const Range& own = sh.shards.ranges[p->owner][0];
  p->shard_w0 = static_cast<int32_t>(own.s0 / 32);
  p->shard_nw = static_cast<int32_t>((own.s1 - own.s0) / 32);
  // CSR entries this part uploads (row_ptr is copied into the staging buffer before any task starts)
  {
    const int64_t* rp = reinterpret_cast<const int64_t*>(sh.stage_in + sh.in_rowptr.off);
    const std::pair<int64_t, int64_t> rows = sh.rows_read(p->owner);
    p->csr_k0 = rp[rows.first]; p->csr_k1 = rp[rows.second];
  }
  // ---- per-part staging: tiles + need blocks
  SegAlloc seg;
  const Seg s_tiles = seg(sizeof(Tile) * p->tiles.size()), s_need = seg(need.size());
  char* st = pin_alloc<char>(p, seg.total);
  if (!st) return p->rc;
  char* d_small = dev_alloc<char>(p, seg.total);
  if (!d_small) return p->rc;
  if (!p->tiles.empty()) memcpy(st + s_tiles.off, p->tiles.data(), s_tiles.bytes);
  if (!need.empty()) memcpy(st + s_need.off, need.data(), s_need.bytes);
  if (!(p->d_plan = dev_alloc<char>(p, sh.plan_bytes))) return p->rc;
  if (!(p->d_in = dev_alloc<char>(p, sh.in_bytes))) return p->rc;
  for (cudaEvent_t* e : {&p->ev_h2d0, &p->ev_h2d1, &p->ev_embed0, &p->ev_embed1, &p->ev_run1})
    PART_CUDA(p, cudaEventCreate(e));
  for (cudaEvent_t* e : {&p->ev_join, &p->ev_bits, &p->ev_rsum, &p->ev_shard})
    PART_CUDA(p, cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  cudaStream_t s0 = dc->stream[0];
  PART_CUDA(p, cudaEventRecord(p->ev_h2d0, s0));
  PART_CUDA(p, cudaMemcpyAsync(p->d_plan, sh.stage_plan, sh.plan_bytes, cudaMemcpyHostToDevice, s0));
  if (seg.total) PART_CUDA(p, cudaMemcpyAsync(d_small, st, seg.total, cudaMemcpyHostToDevice, s0));
  p->info.h2d_bytes = static_cast<int64_t>(sh.plan_bytes + seg.total);
  // ---- device views
  char* d = p->d_plan;
  char* di = p->d_in;
  p->dcsr.n_samples = sh.N; p->dcsr.nnz = sh.nnz;
  p->dcsr.row_ptr = reinterpret_cast<int64_t*>(di + sh.in_rowptr.off);
  p->dcsr.col = reinterpret_cast<int32_t*>(di + sh.in_col.off);
  p->dcsr.val = sh.need_val ? reinterpret_cast<double*>(di + sh.in_val.off) : nullptr;
  p->dtree.n_nodes = B; p->dtree.height = 0;  // (height: set when the tree walk has joined)
  p->dtree.parent = reinterpret_cast<int32_t*>(di + sh.in_parent.off);
  p->dtree.length = reinterpret_cast<double*>(di + sh.in_len.off);
  p->dtree.child_ptr = reinterpret_cast<int32_t*>(di + sh.in_cptr.off);
  p->dtree.child_idx = reinterpret_cast<int32_t*>(di + sh.in_cidx.off);
  p->dtree.level_nodes = reinterpret_cast<int32_t*>(di + sh.in_lvl.off);
  p->dtree.level_parent = reinterpret_cast<int32_t*>(di + sh.in_lpar.off);
  p->d_level_ptr = reinterpret_cast<int32_t*>(di + sh.in_lptr.off);
  p->d_lenf = reinterpret_cast<float*>(di + sh.in_lenf.off);
  p->d_post = sh.unsorted_l ? reinterpret_cast<int32_t*>(di + sh.in_post.off) : nullptr;
  p->d_mult = sh.node_mult ? reinterpret_cast<const double*>(di + sh.in_mult.off) : nullptr;
  p->d_q0 = d + sh.pl_q0.off;
  p->d_q1 = d + sh.pl_hi.off;
  p->d_q2 = d + sh.pl_lo.off;
  p->d_lenq = reinterpret_cast<double*>(d + sh.pl_lenq.off);
  p->d_order = reinterpret_cast<int32_t*>(d + sh.pl_order.off);
  p->d_col_exp = reinterpret_cast<int32_t*>(d + sh.pl_cexp.off);
  p->d_len_col = reinterpret_cast<double*>(d + sh.pl_lcol.off);
  p->d_chunks.end = reinterpret_cast<int32_t*>(d + sh.pl_cend.off);
  p->d_chunks.scale = reinterpret_cast<double*>(d + sh.pl_cscale.off);
  p->d_chunks.n = static_cast<int32_t>(sh.cols.chunk_end.size());
  p->d_chunks.shift = sh.cols.chunk_shift.empty() ? nullptr : reinterpret_cast<int32_t*>(d + sh.pl_cshift.off);
  p->d_chunks.biased = sh.cols.i8 && sh.cols.biased;
  p->d_tiles = reinterpret_cast<Tile*>(d_small + s_tiles.off);
  p->d_need = need.empty() ? nullptr : reinterpret_cast<uint8_t*>(d_small + s_need.off);

  // ---- device buffers
  const int chunks = weighted_scratch_chunks(B);
  const bool i8 = sh.cols.i8, intacc = sh.cols.intacc;
  if (sh.exact || sh.weighted) {
    // exact: the whole fp64 embedding; fast weighted: one slab of samples at a time, <= 2 GB
    const int64_t per = static_cast<int64_t>(p->shard_nw) * 32;
    p->ws_slab = sh.exact ? sh.np : std::min<int64_t>(per, std::max<int64_t>(kTile, (2LL << 30) / (8LL * B) / kTile * kTile));
    if (!sh.exact && sh.knobs.ws_slab > 0)  // tests: force several slabs on a small problem
      p->ws_slab = std::min<int64_t>(per, round_up(sh.knobs.ws_slab, kTile));
    if (!(p->d_E = dev_alloc<double>(p, static_cast<size_t>(B) * p->ws_slab))) return p->rc;
    if (!(p->d_total = dev_alloc<double>(p, sh.np))) return p->rc;
    if (sh.unsorted_l && !(p->d_list_ptr = dev_alloc<int64_t>(p, sh.N + 2))) return p->rc;
    if (!sh.exact) {
      // resident: the panels of all samples; capacity: of this device's two shards only
      const size_t a_samples =
          sh.variant.capacity ? static_cast<size_t>(2 * sh.shards.shard_rows) : static_cast<size_t>(sh.np);
      if (!(p->d_A = dev_alloc<float>(p, static_cast<size_t>(sh.kp) * a_samples))) return p->rc;
      if (sh.keyed && !(p->d_K = dev_alloc<int32_t>(p, static_cast<size_t>(sh.kp) * a_samples))) return p->rc;
      if (sh.variant.capacity) {
        for (int k = 0; k < 2; ++k)
          if (!(p->d_V[k] = dev_alloc<float>(p, static_cast<size_t>(sh.kp) * sh.shards.shard_rows))) return p->rc;
        p->ev_fetch.assign(sh.shards.n_shards, nullptr);
        p->ev_used.assign(sh.shards.n_shards, nullptr);
        for (int k = 0; k < sh.shards.n_shards; ++k) {
          PART_CUDA(p, cudaEventCreateWithFlags(&p->ev_fetch[k], cudaEventDisableTiming));
          PART_CUDA(p, cudaEventCreateWithFlags(&p->ev_used[k], cudaEventDisableTiming));
        }
        for (Part::CapGroup& cb : p->cap) {
          if (alloc_pair_out(p, cb.out, cb.count)) return p->rc;
          PART_CUDA(p, cudaEventCreateWithFlags(&cb.done, cudaEventDisableTiming));
        }
      }
      if (!(p->d_W = dev_alloc<double>(p, sh.np))) return p->rc;
      if (!(p->d_scratch = dev_alloc<double>(p, static_cast<size_t>(chunks) * sh.np))) return p->rc;
      if (!(p->d_flag_counts = dev_alloc<unsigned long long>(p, p->mine.size() + 1))) return p->rc;
      const size_t ws_words = static_cast<size_t>(kFixupCtas) * B * (sh.keyed ? 2 : 1);  // (keyed: diff + sum)
      for (int k = 0; k < 2; ++k) {
        if (!(p->d_fix_ws[k] = dev_alloc<long long>(p, ws_words))) return p->rc;
        PART_CUDA(p, cudaMemsetAsync(p->d_fix_ws[k], 0, sizeof(long long) * ws_words, s0));
      }
    }
  } else {
    // fused: published columns bitsT[nw][kp] (+ node-indexed scratch for trees beyond shared memory);
    // FRC_EMBED_LEVELS=1: node-major bits[B][nw], one launch per tree level
    const size_t words = sh.variant.fused_embed ? static_cast<size_t>(sh.kp) * sh.nw : static_cast<size_t>(B) * sh.nw;
    p->peer_push = sh.variant.peer_push;
    if (p->peer_push) {
      // two buffers from the symmetric heap (same block + offset on every rank), mapped from the peers
      for (int k = 0; k < 2; ++k) {
        cudaError_t e = cudaSuccess;
        p->d_bits2[k] = static_cast<uint32_t*>(dc->sym.alloc(words * sizeof(uint32_t), &e));
        if (!p->d_bits2[k]) return pfail(p, FRC_ERR_OOM, std::string("symmetric heap: ") + cudaGetErrorString(e));
      }
      bool usable = true;
      if (sym_sync(p, &usable) != FRC_OK) return p->rc;
      if (!usable) p->peer_push = false;  // every rank takes the NCCL all-gather of the bit columns instead
    }
    if (p->peer_push) {
      for (int k = 0; k < 2; ++k) {
        size_t blk = 0;
        for (; blk < dc->sym.blocks.size(); ++blk) {
          char* base = dc->sym.blocks[blk].p;
          if (reinterpret_cast<char*>(p->d_bits2[k]) >= base &&
              reinterpret_cast<char*>(p->d_bits2[k]) < base + dc->sym.blocks[blk].cap) break;
        }
        const size_t off = reinterpret_cast<char*>(p->d_bits2[k]) - dc->sym.blocks[blk].p;
        p->peers[k].n = sh.world; p->peers[k].self = sh.rank0;
        for (int r = 0; r < sh.world; ++r) p->peers[k].p[r] = reinterpret_cast<uint32_t*>(c->sym_peer[blk][r] + off);
      }
      p->d_bits = p->d_bits2[0];
    } else if (!(p->d_bits = dev_alloc<uint32_t>(p, std::max<size_t>(words, 64)))) return p->rc;
    const size_t ns = sh.variant.fused_embed ? static_cast<size_t>(presence_node_scratch_words(B, p->shard_nw)) : 0;
    if (ns && !(p->d_node_scratch = dev_alloc<uint32_t>(p, ns))) return p->rc;
    const size_t opsz = sh.variant.bits_feed ? 256 : static_cast<size_t>(sh.np) * sh.kp * (i8 ? 1 : 2);
    if (!(p->d_P = dev_alloc<char>(p, opsz))) return p->rc;
    if (!(p->d_Bh = dev_alloc<char>(p, opsz))) return p->rc;
    if (!(p->d_Bl = dev_alloc<char>(p, opsz))) return p->rc;
    if (sh.variant.bits_feed && !(p->d_bitsS = dev_alloc<uint32_t>(p, static_cast<size_t>(sh.np) * (sh.kp / 32)))) return p->rc;
    if (!(p->d_r = dev_alloc<double>(p, sh.np))) return p->rc;
    if (!(p->d_scratch = dev_alloc<double>(p, static_cast<size_t>(chunks) * sh.np))) return p->rc;
    if (!(p->d_flag_counts = dev_alloc<unsigned long long>(p, p->mine.size() + 1))) return p->rc;
    if (i8 && !(p->d_flag_u = dev_alloc<double>(p, 1))) return p->rc;
    if (i8 && !(p->d_qerr = dev_alloc<double>(p, sh.kp))) return p->rc;
    if (i8 && !(p->d_qam = dev_alloc<uint32_t>(p, sh.kp))) return p->rc;
    if (intacc && !(p->d_r_int = dev_alloc<long long>(p, sh.np))) return p->rc;
    std::string terr;
    if (sh.variant.bits_feed) {
      p->tc = tc_operands_create_bits(p->d_bitsS, sh.np, sh.kp, static_cast<const uint8_t*>(p->d_q0),
                                      static_cast<const uint8_t*>(p->d_q1), static_cast<const uint8_t*>(p->d_q2),
                                      p->d_chunks, p->d_len_col, p->d_flag_u, p->d_r_int,
                                      std::ldexp(1.0, sh.cols.e_min), &terr);
    } else {
      p->tc = tc_operands_create(p->d_P, p->d_Bh, p->d_Bl, sh.np, sh.kp, i8, p->d_chunks, p->d_len_col, p->d_flag_u, &terr);
      if (p->tc && intacc) tc_operands_set_int(p->tc, p->d_r_int, std::ldexp(1.0, sh.cols.e_min));
    }
    if (!p->tc) return pfail(p, FRC_ERR_CUDA, terr);
    if (i8) {  // a function of the tree only: once per job, not per restart
      p->info.kernel_launches += launch_quantize_lengths(
          p->d_len_col, p->d_col_exp, sh.kp, static_cast<uint8_t*>(p->d_q0), static_cast<uint8_t*>(p->d_q1),
          static_cast<uint8_t*>(p->d_q2), p->d_qam, p->d_lenq, p->d_qerr, p->d_flag_u, s0);
      PART_CUDA(p, cudaGetLastError());
    }
  }
  // ---- output ring
  {
    const int vb = sh.exact ? 8 : 4;
    const int64_t want = std::max<int64_t>(kMinSlots, std::min<int64_t>(kSlots, kSlotBytesBudget / (p->max_band * vb)));
    p->n_slots = static_cast<int>(std::min<int64_t>(want, std::max<int64_t>(2, static_cast<int64_t>(p->mine.size()) + 1)));
  }
  if (p->mine.empty()) p->n_slots = 0;
  for (int k = 0; k < p->n_slots; ++k) {
    Slot& sl = p->slots[k];
    if (sh.exact) {
      if (!(sl.dev64 = dev_alloc<double>(p, p->max_band))) return p->rc;
      if (sh.d2h && !(sl.host64 = pin_alloc<double>(p, p->max_band))) return p->rc;
    } else {
      if (sh.d2h && !(sl.host32 = pin_alloc<float>(p, p->max_band))) return p->rc;
      // (capacity mode: a band lives in its row-shard group's record, Part::CapGroup)
      if (!sh.variant.capacity && alloc_pair_out(p, sl.own, p->max_band)) return p->rc;
    }
    for (cudaEvent_t* e : {&sl.k0, &sl.k1, &sl.k2, &sl.done}) PART_CUDA(p, cudaEventCreate(e));
  }
  return FRC_OK;
}

// (6a) per device: upload the staged inputs, first stage of the embedding.
int launch_part_stage1(Part* p) {
  const Shared& sh = *p->sh;
  DevCtx* dc = p->dc;
  cudaStream_t s0 = dc->stream[0];
  p->dtree.height = sh.tree_height;
  p->info.tree_height = sh.tree_height;
  // row_ptr + tree arrays, then this part's slice of the entries
  PART_CUDA(p, cudaMemcpyAsync(p->d_in, sh.stage_in, sh.in_col.off, cudaMemcpyHostToDevice, s0));
  int64_t up = static_cast<int64_t>(sh.in_col.off);
  const int64_t k0 = p->csr_k0, n = p->csr_k1 - p->csr_k0;
  if (n > 0) {
    PART_CUDA(p, cudaMemcpyAsync(p->d_in + sh.in_col.off + 4 * k0, sh.stage_in + sh.in_col.off + 4 * k0, 4 * n,
                                 cudaMemcpyHostToDevice, s0));
    up += 4 * n;
    if (sh.need_val) {
      PART_CUDA(p, cudaMemcpyAsync(p->d_in + sh.in_val.off + 8 * k0, sh.stage_in + sh.in_val.off + 8 * k0, 8 * n,
                                   cudaMemcpyHostToDevice, s0));
      up += 8 * n;
    }
  }
  p->info.h2d_bytes += up;
  PART_CUDA(p, cudaEventRecord(p->ev_h2d1, s0));
  return embed_stage1(p);
}
int launch_part_stage2(Part* p) {
  if (embed_stage2(p)) return p->rc;
  return start_pairs(p);
}

void aggregate_info(frc_job* j) {
  frc_info_t& a = j->info;
  const Shared& sh = j->sh;
  a = frc_info_t{};
  a.path_taken = sh.exact ? FRC_PATH_EXACT : FRC_PATH_FAST;
  a.n_bands_total = static_cast<int32_t>(sh.bands.size());
  a.tree_height = sh.tree_height;
  a.n_pairs_total = sh.geo.rect ? (sh.N - sh.geo.q0) * sh.geo.n_ref : sh.N >= 2 ? tri(sh.N) : 0;
  a.n_nodes_padded = sh.exact ? sh.B : sh.kp;
  a.operand_kind = sh.variant.operand_kind;
  a.n_devices = static_cast<int32_t>(j->parts.size());
  a.value_bytes = sh.exact ? 8 : 4;
  a.create_ms = j->create_ms;
  for (auto& p : j->parts) {
    const frc_info_t& i = p->info;
    a.n_bands_mine += static_cast<int32_t>(p->mine.size());
    a.n_pairs_mine += i.n_pairs_mine;
    a.kernel_launches += i.kernel_launches;
    a.h2d_ms = std::max(a.h2d_ms, i.h2d_ms);
    a.embed_ms = std::max(a.embed_ms, i.embed_ms);
    a.pairs_ms += i.pairs_ms;
    a.fixup_ms += i.fixup_ms;
    a.run_ms = std::max(a.run_ms, i.run_ms);
    a.h2d_bytes += i.h2d_bytes;
    a.d2h_bytes += i.d2h_bytes;
    a.embed_bytes += i.embed_bytes;
    a.flagged_pairs += i.flagged_pairs;
    a.gather_bytes += i.gather_bytes;
    a.exceptions += i.exceptions;
  }
}

// The job's context (the caller's, or one of its own from opts), one part per device, and how the parts' sample
// shards meet.
int attach_context(frc_job* j, frc_ctx_t* ctx, const frc_opts_t* opts) {
  Shared& sh = j->sh;
  if (ctx) {
    if (ctx->in_use) return fail(j, FRC_ERR_STATE, "context already has a live job");
    j->ctx = ctx;
  } else {
    const int rc = opts->n_devices > 1 || opts->n_devices < 0
                       ? frc_ctx_create_multi(opts->n_devices, opts->devices, &j->ctx)
                       : frc_ctx_create(opts->n_devices == 1 && opts->devices ? opts->devices[0] : opts->device, &j->ctx);
    if (rc) { j->err = g_create_error; j->ctx = nullptr; return rc; }
    j->own_ctx = true;
  }
  frc_ctx* c = j->ctx;
  c->in_use = true;
  sh.n_parts = static_cast<int>(c->devs.size());
  if (sh.n_parts > 1 && sh.world > 1)
    return fail(j, FRC_ERR_UNSUPPORTED, "a multi-device job cannot also be a rank of a multi-process run (world > 1)");
  for (int k = 0; k < sh.n_parts; ++k) {
    j->parts.emplace_back(new Part());
    Part* p = j->parts.back().get();
    p->job = j; p->sh = &sh; p->dc = c->devs[k]; p->index = k;
    p->owner = sh.n_parts > 1 ? k : sh.rank0;
  }
  sh.variant = plan_exchange(variant_in(sh, c), sh.knobs);
  return FRC_OK;
}

// frc_create (query == null) and frc_create_cross (abnd = the reference table).  A cross job stages ONE table of
// q0 + n_q rows -- the reference rows, empty rows up to q0, the query rows (Shared::geo) -- and everything up to the
// pair stage runs on it as on any table; only the bands, the tiles and the pair kernels' geometry differ.
int create_job(frc_ctx_t* ctx, const frc_tree_t* tree, const frc_csr_t* abnd, const frc_csr_t* query,
               const frc_opts_t* opts, frc_job_t** out) {
  DeviceGuard guard;
  const auto t_create0 = std::chrono::steady_clock::now();
  frc_job* j = new frc_job();
  Shared& sh = j->sh;
  bool workers_busy = false;  // the table is validated + staged by the pool while this thread plans
  auto bail = [&](int rc) {
    if (workers_busy) { j->ctx->pool->wait(); workers_busy = false; }
    g_create_error = j->err; destroy_job(j); return rc;
  };
  sh.knobs = Knobs::read();
  const bool trace = sh.knobs.trace;
  auto tp0 = t_create0;
  auto mark = [&](const char* what) {
    if (!trace) return;
    auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[frc_create] %-32s %8.1f us\n", what, std::chrono::duration<double, std::micro>(now - tp0).count());
    tp0 = now;
  };

  // ------------------------------------------------------------ (1) options, table header
  int rc = validate_header(j, tree, abnd, query, opts);
  if (rc) return bail(rc);
  const frc_tree_t* const tree0 = tree;  // the caller's tree (FRC_FLAG_PRUNE: `tree` becomes the pruned one)
  const StagedTable table{abnd, query, sh.geo.q0};
  const int64_t N = sh.N, nnz = sh.nnz;

  // ------------------------------------------------------------ context
  if ((rc = attach_context(j, ctx, opts)) != FRC_OK) return bail(rc);
  frc_ctx* c = j->ctx;

  PrunedTree pruned;
  frc_tree_t ptree{};
  if ((opts->flags & FRC_FLAG_PRUNE) && prune_to_table(sh, *c->pool, tree0, table, &pruned)) {
    ptree = frc_tree_t{pruned.n_nodes, pruned.parent.data(), pruned.length.data()};
    tree = &ptree;
  }

  // ------------------------------------------------------------ (2) staging buffer; row_ptr right away
  layout_inputs(sh);
  {
    cudaError_t e = cudaSuccess;
    sh.stage_in = static_cast<char*>(c->pin.alloc(sh.in_bytes, &e));
    if (!sh.stage_in) return bail(fail(j, FRC_ERR_OOM, std::string("pinned staging of the inputs: ") + cudaGetErrorString(e)));
  }
  int64_t* const staged_rp = reinterpret_cast<int64_t*>(sh.stage_in + sh.in_rowptr.off);
  table.fill_row_ptr(staged_rp);

  // One task list for the pool: the tree walks, the preparation of devices 1.. (they wait for the plan),
  // then the CSR entries in chunks, all handed out through one counter; the calling thread plans, prepares
  // device 0 and then joins in, so the split adapts to any pool size.
  TreeLevels levels;
  bool children_ok = false;
  std::atomic<int> plan_ready{0};  // 1 = planned, -1 = planning failed
  // The entries are cut into many more chunks than workers and handed out through a counter: a worker
  // on a busy or slow core (the slowest static share took 1.5-2.4x the median) just takes fewer.
  // The one part of a process stages the rows it reads; several parts of one process stage every row once.
  const std::pair<int64_t, int64_t> rows = sh.n_parts == 1 ? sh.rows_read(sh.rank0) : std::pair<int64_t, int64_t>{0, N};
  const int64_t stage_k0 = staged_rp[rows.first], stage_k1 = staged_rp[rows.second];
  const int csr_chunks = nnz >= 65536 ? static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(c->pool->size() * 8LL, nnz / 8192))) : 1;
  const int n_prep = sh.n_parts - 1;
  const int n_tasks = 2 + n_prep + csr_chunks;
  std::atomic<int> task_next{0};
  std::vector<std::string> csr_errs(csr_chunks);
  std::vector<double> csr_us(c->pool->size(), 0.0);
  // duplicate detection: stamp[leaf] = epoch-tagged sample id; the arrays persist in the
  // context, so nothing is cleared between jobs
  const int64_t stamp_tag = c->stamp_epoch;
  c->stamp_epoch += N + 1;
  int32_t* const dcol = reinterpret_cast<int32_t*>(sh.stage_in + sh.in_col.off);
  double* const dval = sh.need_val ? reinterpret_cast<double*>(sh.stage_in + sh.in_val.off) : nullptr;
  const int32_t* const new_of_old = pruned.new_of_old.empty() ? nullptr : pruned.new_of_old.data();
  const std::function<void(int)> work = [&](int t) {
    const auto w0 = std::chrono::steady_clock::now();
    std::vector<int64_t>& stamp = c->stamps[t];
    if (dval && static_cast<int32_t>(stamp.size()) < tree0->n_nodes) stamp.assign(tree0->n_nodes, -1);
    for (int task = task_next.fetch_add(1, std::memory_order_relaxed); task < n_tasks;
         task = task_next.fetch_add(1, std::memory_order_relaxed)) {
      if (task == 0) { levels = stage_tree_levels(sh, tree); continue; }
      if (task == 1) { children_ok = stage_tree_children(sh, tree, pruned.mult.data()); continue; }
      if (task < 2 + n_prep) {
        int ready;
        while ((ready = plan_ready.load(std::memory_order_acquire)) == 0) std::this_thread::yield();
        if (ready > 0) prepare_part(j->parts[task - 1].get());
        continue;
      }
      const int ch = task - 2 - n_prep;
      const std::pair<int64_t, int64_t> r = chunk_rows(staged_rp, N, stage_k0, stage_k1, ch, csr_chunks);
      // (checked against the caller's tree, staged with the pruned tree's ids)
      csr_errs[ch] = stage_entries(table, staged_rp, r.first, r.second, tree0->parent, tree0->n_nodes, new_of_old,
                                   stamp.data(), stamp_tag, dcol, dval);
    }
    csr_us[t] += std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - w0).count();
  };
  const int n_workers = c->pool->size() - 1;
  if (n_workers > 0) {
    workers_busy = true;
    c->pool->start(n_workers, work);
  }
  mark("header checks, context, workers started");

  // ------------------------------------------------------------ (3) plan (the walks and the staging run in the pool)
  // (refused on the caller's lengths; the sign test is on the lengths the kernels use)
  bool bad_len = false, neg_len = false;
  scan_lengths(tree0, tree, &bad_len, &neg_len);
  auto plan_failed = [&](int code) { plan_ready.store(-1, std::memory_order_release); return bail(code); };
  if (!sh.exact && bad_len)
    return plan_failed(fail(j, FRC_ERR_UNSUPPORTED, "non-finite branch length: only the exact path handles it"));
  if ((rc = plan_job(j, tree, neg_len)) != FRC_OK) return plan_failed(rc);
  if ((rc = stage_plan(j, tree)) != FRC_OK) return plan_failed(rc);
  mark("column plan + bands");
  plan_ready.store(1, std::memory_order_release);
  // ------------------------------------------------------------ (5) device 0 on this thread
  prepare_part(j->parts[0].get());
  mark("device 0 prepared");
  work(n_workers);  // whatever is left of the task list (everything, without workers)
  if (workers_busy) { c->pool->wait(); workers_busy = false; }
  if (trace) { fprintf(stderr, "[frc_create] share times (us):"); for (double u : csr_us) fprintf(stderr, " %.0f", u); fprintf(stderr, "\n"); }
  if (levels.bad_parent) return bail(fail(j, FRC_ERR_ARG, "parent[" + std::to_string(levels.bad_parent) + "] is not a smaller node id"));
  if (levels.bad_order) return bail(fail(j, FRC_ERR_ARG, "node ids are not a pre-order numbering (node " + std::to_string(levels.bad_order) + ")"));
  const std::string& csr_err = first_error(csr_errs);
  if (!csr_err.empty()) return bail(fail(j, FRC_ERR_ARG, csr_err));
  if (levels.height < 0 || !children_ok) return bail(fail(j, FRC_ERR_ARG, "tree topology could not be prepared"));  // (unreachable)
  for (auto& p : j->parts)
    if (p->rc) { j->err = p->err; return bail(p->rc); }
  sh.level_ptr = levels.level_ptr;
  sh.tree_height = levels.height;
  // the delivery order: bands of this process in flat-index order
  {
    std::vector<int> cursor(sh.n_parts, 0);
    for (const Band& b : sh.bands)
      for (int k = 0; k < sh.n_parts; ++k)
        if (j->parts[k]->owner == b.owner) { j->order.push_back({k, cursor[k]++}); break; }
  }
  if (!sh.exact && sh.d2h) {
    int64_t mb = 1;
    for (auto& p : j->parts) mb = std::max(mb, p->max_band);
    cudaError_t e = cudaSuccess;
    j->wide = static_cast<double*>(c->pin.alloc(sizeof(double) * std::min(mb, kWidePiece), &e));
    if (!j->wide) return bail(fail(j, FRC_ERR_OOM, std::string("pinned widening buffer: ") + cudaGetErrorString(e)));
  }
  mark("workers joined");
  // ------------------------------------------------------------ (6) go
  if ((rc = for_parts(j, launch_part_stage1)) != FRC_OK) return bail(rc);
  if ((rc = for_parts(j, launch_part_stage2)) != FRC_OK) return bail(rc);
  mark("uploads, embedding, first bands queued");
  j->create_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_create0).count();
  *out = j;
  return FRC_OK;
}

}  // namespace

extern "C" {

int frc_create(frc_ctx_t* ctx, const frc_tree_t* tree, const frc_csr_t* abnd, const frc_opts_t* opts,
               frc_job_t** out) {
  g_create_error.clear();
  if (!out) { g_create_error = "frc_create: out is NULL"; return FRC_ERR_ARG; }
  *out = nullptr;
  if (!tree || !abnd || !opts) { g_create_error = "frc_create: NULL argument"; return FRC_ERR_ARG; }
  return create_job(ctx, tree, abnd, nullptr, opts, out);
}

int frc_create_cross(frc_ctx_t* ctx, const frc_tree_t* tree, const frc_csr_t* ref, const frc_csr_t* query,
                     const frc_opts_t* opts, frc_job_t** out) {
  g_create_error.clear();
  if (!out) { g_create_error = "frc_create_cross: out is NULL"; return FRC_ERR_ARG; }
  *out = nullptr;
  if (!tree || !ref || !opts) { g_create_error = "frc_create_cross: NULL argument"; return FRC_ERR_ARG; }
  if (!query) { g_create_error = "frc_create_cross: the query table is NULL"; return FRC_ERR_ARG; }
  return create_job(ctx, tree, ref, query, opts, out);
}

}  // extern "C"

namespace {

// Waits for band idx of the part and does the per-band bookkeeping.
int part_wait_band(Part* p, size_t idx, Slot** out) {
  const Shared& sh = *p->sh;
  PART_CUDA(p, cudaSetDevice(p->dc->device));
  if (idx >= p->next_enqueue) {  // only when the ring has 2 slots and this is the first call
    if (enqueue_band(p, p->next_enqueue)) return p->rc;
    ++p->next_enqueue;
  }
  Slot& sl = p->slots[idx % p->n_slots];
  const auto tn0 = std::chrono::steady_clock::now();
  PART_CUDA(p, cudaEventSynchronize(sl.done));
  float ms = 0.f;
  const bool spans = !sh.variant.capacity;  // (capacity mode: a group's kernels serve all of its bands; no per-band span)
  if (spans && (p->mine.size() <= 2 || sh.knobs.trace)) {
    // per-band kernel spans (info.pairs_ms / fixup_ms): meaningful for a job of one or two bands (bench.py's
    // roofline leg); a many-band stream skips the four driver calls per band on the consumer's thread
    PART_CUDA(p, cudaEventElapsedTime(&ms, sl.k0, sl.k1));
    p->info.pairs_ms += ms;
    PART_CUDA(p, cudaEventElapsedTime(&ms, sl.k1, sl.k2));
    p->info.fixup_ms += ms;
  }
  if (idx + 1 == p->mine.size() && !p->run_timed) {
    PART_CUDA(p, cudaEventSynchronize(p->ev_run1));
    PART_CUDA(p, cudaEventElapsedTime(&ms, p->ev_embed0, p->ev_run1));
    p->info.run_ms = ms;
    p->run_timed = true;
  }
  if (sl.out && !sl.out->counted) {  // (the record's work has completed; a group's record holds several bands)
    PairOut& o = *sl.out;
    o.counted = true;
    p->info.flagged_pairs += static_cast<int64_t>(*o.n_flagged_host);
    const unsigned long long n = *o.ex.count;
    if (n > static_cast<unsigned long long>(o.ex.cap))
      return pfail(p, FRC_ERR_UNSUPPORTED, "more than " + std::to_string(o.ex.cap) + " distances of one band lie below "
                                           "fp32's range (|d| < 1.2e-38): run this input with path = FRC_PATH_EXACT");
    p->info.exceptions += static_cast<int64_t>(n);
  }
  if (sh.knobs.trace) {
    float a = 0, b = 0, c2 = 0, d = 0;
    if (spans) {
      cudaEventElapsedTime(&a, p->ev_embed0, sl.k0);
      cudaEventElapsedTime(&b, p->ev_embed0, sl.k1);
      cudaEventElapsedTime(&c2, p->ev_embed0, sl.k2);
    }
    cudaEventElapsedTime(&d, p->ev_embed0, sl.done);
    fprintf(stderr, "[dev %d band %3zu] host: deliver at %.3f ms after waiting %.1f us; device: start %.3f kernel_end %.3f "
                    "fixup_end %.3f d2h_end %.3f ms (pairs %lld)\n", p->dc->device, idx,
            std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - p->t_host0).count(),
            std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - tn0).count(), a, b, c2, d,
            static_cast<long long>(p->bands[idx].count));
  }
  *out = &sl;
  return FRC_OK;
}

// frc_next on a fast path: widens pairs [off, off + n) of the held band into j->wide (wire.cu) and patches the
// exceptions that fall into the piece.
void widen_piece(frc_job* j, const Slot& sl, int64_t band_first, int64_t off, int64_t n) {
  const bool trace = j->sh.knobs.trace;
  const auto t0 = std::chrono::steady_clock::now();
  Pool* pool = j->ctx->pool.get();
  int T = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(std::min(pool->size(), 16), n / 65536)));
  if (j->sh.knobs.widen_threads > 0) T = std::max(1, std::min(T, j->sh.knobs.widen_threads));
  const float* src = sl.host32 + off;
  double* dst = j->wide;
  // chunks handed out through a counter (a worker on a busy core takes fewer); the first round is
  // static so that thread t starts where it started last time and finds its destination lines in its L2
  constexpr int64_t kChunk = 16384;
  const int64_t n_chunks = (n + kChunk - 1) / kChunk;
  std::atomic<int64_t> next{0};
  std::atomic<int64_t>* nx = &next;
  pool->run(T, [=](int t) {
    for (int64_t ch = t < n_chunks ? t : n_chunks; ch < n_chunks;) {
      const int64_t lo = ch * kChunk, hi = std::min(n, lo + kChunk);
      widen_band(src + lo, dst + lo, hi - lo, /*stream_stores=*/false);
      ch = T + nx->fetch_add(1, std::memory_order_relaxed);
    }
  });
  const Exceptions& ex = sl.out->ex;
  const int64_t n_ex = std::min<int64_t>(static_cast<int64_t>(*ex.count), ex.cap);
  for (int64_t k = 0; k < n_ex; ++k) {
    const int64_t at = ex.index[k] - band_first - off;
    if (at >= 0 && at < n) dst[at] = ex.value[k];
  }
  if (trace)
    fprintf(stderr, "[host] widened %lld pairs on %d threads in %.0f us\n", static_cast<long long>(n), T,
            std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count());
}

// Common body of frc_next / frc_next_f32.  mode 1: float64 out, mode 2: float32 out.
int next_chunk(frc_job* j, int mode, const void** data, int64_t* first_index, int64_t* count) {
  const Shared& sh = j->sh;
  *data = nullptr; *first_index = 0; *count = 0;
  if (j->read_mode == 0) j->read_mode = mode;
  if (j->read_mode != mode) return fail(j, FRC_ERR_STATE, "frc_next and frc_next_f32 cannot be mixed on one pass of a job");
  if (mode == 2 && sh.exact)
    return fail(j, FRC_ERR_STATE, "this job took the exact path (bit-exact float64): read it with frc_next");
  if (mode == 1 && !sh.exact && !sh.d2h)
    return fail(j, FRC_ERR_STATE, "FRC_FLAG_NO_D2H on a fast path keeps fp32 in HBM: read it with frc_next_f32");
  DeviceGuard guard;
  // a band larger than the widening buffer is handed out piece by piece
  if (mode == 1 && j->held_part >= 0 && !sh.exact && j->piece_off < j->piece_end) {
    const int64_t n = std::min(kWidePiece, j->piece_end - j->piece_off);
    widen_piece(j, j->parts[j->held_part]->slots[j->held_slot], j->piece_first, j->piece_off, n);
    *data = j->wide;
    *first_index = j->piece_first + j->piece_off;
    *count = n;
    j->piece_off += n;
    return FRC_OK;
  }
  // the band handed out by the previous call is released now: its slot takes the part's next band
  if (j->held_part >= 0) {
    Part* hp = j->parts[j->held_part].get();
    j->held_part = -1; j->held_slot = -1;
    if (hp->next_enqueue < hp->mine.size()) {
      cudaSetDevice(hp->dc->device);
      if (enqueue_band(hp, hp->next_enqueue)) return fail(j, hp->rc, hp->err);
      ++hp->next_enqueue;
    }
  }
  if (j->next_item >= j->order.size()) return FRC_OK;  // end of stream
  const frc_job::Item it = j->order[j->next_item];
  Part* p = j->parts[it.part].get();
  Slot* sl = nullptr;
  if (part_wait_band(p, static_cast<size_t>(it.idx), &sl)) return fail(j, p->rc, p->err);
  const Band& b = p->bands[it.idx];
  int64_t deliver_n = b.count;
  if (sh.exact) {
    *data = sh.d2h ? sl->host64 : sl->dev64;
  } else if (mode == 2) {
    *data = sh.d2h ? sl->host32 : sl->out->dev32 + sl->out_off;
  } else {
    deliver_n = std::min(kWidePiece, b.count);
    j->piece_first = b.first; j->piece_off = deliver_n; j->piece_end = b.count;
    widen_piece(j, *sl, b.first, 0, deliver_n);
    *data = j->wide;
  }
  *first_index = b.first;
  *count = deliver_n;
  j->held_first = b.first; j->held_count = b.count;
  j->held_part = it.part;
  j->held_slot = static_cast<int>(it.idx % p->n_slots);
  ++p->next_deliver;
  ++j->next_item;
  return FRC_OK;
}

}  // namespace

extern "C" {

int frc_next(frc_job_t* j, const double** data, int64_t* first_index, int64_t* count) {
  if (!j || !data || !first_index || !count) return FRC_ERR_ARG;
  const void* d = nullptr;
  const int rc = next_chunk(j, 1, &d, first_index, count);
  *data = static_cast<const double*>(d);
  return rc;
}

int frc_next_f32(frc_job_t* j, const float** data, int64_t* first_index, int64_t* count) {
  if (!j || !data || !first_index || !count) return FRC_ERR_ARG;
  const void* d = nullptr;
  const int rc = next_chunk(j, 2, &d, first_index, count);
  *data = static_cast<const float*>(d);
  return rc;
}

int frc_chunk_exceptions(frc_job_t* j, const int64_t** index, const double** value, int64_t* count) {
  if (!j || !index || !value || !count) return FRC_ERR_ARG;
  *index = nullptr; *value = nullptr; *count = 0;
  if (j->held_part < 0 || j->sh.exact) return FRC_OK;
  const Exceptions& ex = j->parts[j->held_part]->slots[j->held_slot].out->ex;
  const int64_t n = std::min<int64_t>(static_cast<int64_t>(*ex.count), ex.cap);
  if (n == 0) return FRC_OK;
  // (a list may cover more than this run: the capacity mode keeps one per row shard)
  j->ex_index.clear(); j->ex_value.clear();
  for (int64_t k = 0; k < n; ++k)
    if (ex.index[k] >= j->held_first && ex.index[k] < j->held_first + j->held_count) {
      j->ex_index.push_back(ex.index[k]);
      j->ex_value.push_back(ex.value[k]);
    }
  *index = j->ex_index.data();
  *value = j->ex_value.data();
  *count = static_cast<int64_t>(j->ex_index.size());
  return FRC_OK;
}

int frc_restart(frc_job_t* j) {
  if (!j) return FRC_ERR_ARG;
  DeviceGuard guard;
  // every stream of every device idle before the buffers are rewritten (peers store into each other's memory)
  for (auto& p : j->parts) {
    cudaSetDevice(p->dc->device);
    for (auto s : p->dc->stream)
      if (cudaStreamSynchronize(s) != cudaSuccess) return fail(j, FRC_ERR_CUDA, std::string("cudaStreamSynchronize: ") + cudaGetErrorString(cudaGetLastError()));
    p->info.kernel_launches = 0;
  }
  j->next_item = 0;
  j->held_part = j->held_slot = -1;
  j->read_mode = 0;
  j->piece_off = j->piece_end = 0;
  int rc = for_parts(j, embed_stage1);
  if (rc) return rc;
  return for_parts(j, launch_part_stage2);
}

int frc_job_info(const frc_job_t* cj, frc_info_t* info) {
  if (!cj || !info) return FRC_ERR_ARG;
  frc_job* j = const_cast<frc_job*>(cj);
  DeviceGuard guard;
  for (auto& p : j->parts) {
    if (!p->embed_timed && p->ev_embed1) {
      cudaSetDevice(p->dc->device);
      if (cudaEventSynchronize(p->ev_embed1) == cudaSuccess) {
        float a = 0.f, b = 0.f;
        if (cudaEventElapsedTime(&a, p->ev_h2d0, p->ev_h2d1) == cudaSuccess) p->info.h2d_ms = a;
        if (cudaEventElapsedTime(&b, p->ev_embed0, p->ev_embed1) == cudaSuccess) p->info.embed_ms = b;
        p->embed_timed = true;
      }
      cudaGetLastError();
    }
  }
  aggregate_info(j);
  *info = j->info;
  return FRC_OK;
}

void frc_destroy(frc_job_t* j) {
  DeviceGuard guard;
  destroy_job(j);
}

int64_t frc_plan_bands(int64_t n_samples, int64_t band_rows, int32_t rank, int32_t world, uint32_t flags,
                       int64_t* first_index, int64_t* count, int64_t cap) {
  if (world <= 0) { world = 1; rank = 0; }
  if (n_samples < 0 || band_rows < 0 || rank < 0 || rank >= world) return -FRC_ERR_ARG;
  const Knobs knobs = Knobs::read();
  const std::vector<Band> bands = make_bands(n_samples, band_rows, world, !(flags & FRC_FLAG_NO_D2H), knobs.bands_per_rank, 8);
  int64_t n = 0;
  for (const Band& b : bands)
    if (b.owner == rank) {
      if (n < cap && first_index && count) { first_index[n] = b.first; count[n] = b.count; }
      ++n;
    }
  return n;
}

}  // extern "C"
