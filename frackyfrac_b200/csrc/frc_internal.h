// Internal interfaces between the translation units of libfrcfrc_cuda.
// Nothing here is part of the C ABI (include/frcfrc_cuda.h).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <string>

namespace frc {

constexpr int kTile = 128;   // samples per tile edge (pair tiles are kTile x kTile)
constexpr int kKBlock = 64;  // nodes per contraction block (128 B of bf16)

inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
// Flat index of the first pair of row i in the lower triangle (common/common.go:21-31).
inline int64_t tri(int64_t i) { return i * (i - 1) / 2; }

// Tree arrays resident on the device.
struct DevTree {
  int32_t n_nodes = 0;
  int32_t height = 0;                  // number of levels above the leaves
  const int32_t* parent = nullptr;     // [B]
  const double* length = nullptr;      // [B]
  const int32_t* child_ptr = nullptr;  // [B+1]
  const int32_t* child_idx = nullptr;  // [B-1], ascending id within a parent = file order
  const int32_t* level_nodes = nullptr;// [B] nodes grouped by height (leaves first), ascending id
  const int32_t* level_parent = nullptr;// [B] parent of level_nodes[k] (root: 0)
};

struct DevCsr {
  int64_t n_samples = 0;
  int64_t nnz = 0;
  const int64_t* row_ptr = nullptr;
  const int32_t* col = nullptr;
  const double* val = nullptr;  // may be null for the presence-only path
};

// The same buffer in every rank's HBM (CUDA IPC mappings over NVLink); p[self] is the local one.
struct PeerPtrs {
  uint32_t* p[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int n = 0;     // ranks (0: no peers, local stores only)
  int self = 0;
};

// One tile of the lower triangle: rows [128*ti, +128) x cols [128*tj, +128), tj <= ti.
struct Tile { int32_t ti, tj; };

// Which pairs a job computes.  Triangle (rect == false): (i, j), j < i, of the whole table, flat index
// i(i-1)/2 + j.  Rectangle (frc_create_cross): the table is [reference rows; empty rows up to q0; query rows]
// with q0 a multiple of 256 (a CTA-pair tile), and the pairs are (i, j) for every query row i >= q0 and
// reference row j < n_ref, flat index (i - q0) * n_ref + j.  The kernels take it as a compile-time choice
// (Tri / Rect instantiations) plus this argument; the launchers below pick the instantiation from `rect`.
struct Geometry {
  bool rect = false;
  int64_t q0 = 0, n_ref = 0;
};

// The fast paths store fp32 distances.  A fix-up kernel that meets a value fp32 cannot carry to 2^-23
// relative (|d| < 1.2e-38: pathological trees only) also reports it here, in mapped pinned host memory:
// frc_next patches it into the widened doubles, frc_chunk_exceptions hands it to fp32 consumers.
struct Exceptions {
  unsigned long long* count = nullptr;  // entries appended (may exceed cap: the host then fails the call)
  int64_t* index = nullptr;             // flat pair index
  double* value = nullptr;
  int32_t cap = 0;
};

// ---- embed.cu ---------------------------------------------------------------
// fp64 branch embedding, node-major E[B][ld] (unifrac.go:32-53): leaf rows
// scattered from the CSR, then one pass per tree level, children summed in
// child order starting from 0.0.  Returns launches.
// E holds the ld samples starting at sample s_base (the whole table: s_base = 0, ld = np).
// K (keyed -l tiles only, else null): also the int32 key panels of the same samples, in the tile-panel layout
// K[np/128][kp][128] of the weighted operand (addressed by global sample tile): key = the largest present leaf
// id in the node's subtree, -1 where the node is absent (E == 0) and in the padding rows [n_nodes, kp).
int launch_embed_f64(const DevTree& t, const int32_t* level_ptr_host, const DevCsr& a, double* E,
                     int64_t ld, int64_t s_base, cudaStream_t s, int32_t* K = nullptr, int32_t kp = 0);
// total[s] = sum over ALL nodes in ascending id order (unifrac.go:60-63).
int launch_totals_f64(const double* E, int32_t n_nodes, int64_t ld, int64_t n_samples,
                      double* total, cudaStream_t s);
// Same totals for the fast path (chunked partial sums, any order; scratch as for launch_weighted_operand).
// mult (merged tree, FRC_FLAG_PRUNE; else nullptr): total[s] = sum of mult[v] * E[v][s].
int launch_totals_fast_f64(const double* E, int32_t n_nodes, int64_t ld, const double* mult, double* total,
                           double* scratch, cudaStream_t s);
// E[v][s] /= total[s] for non-zero entries (unifrac.go:64-66).
int launch_normalize_f64(double* E, int32_t n_nodes, int64_t ld, int64_t n_samples,
                         const double* total, cudaStream_t s);
// Weighted operand: A[v][s] = float(len[v] * E[v][s] / total[s]) (prescale) or
// float(E[v][s] / total[s]); rows [n_nodes, kp) zero.  total == nullptr: no division (-l).
// Also W[s] = sum_v len[v] * a[v][s] in fp64 (denominator, separable).
int launch_weighted_operand(const double* E, const double* length, int32_t n_nodes, int32_t kp,
                            int64_t ld, int64_t n_samples, const double* total, bool prescale,
                            float* A, double* W, double* scratch, cudaStream_t s);
// Fast weighted path: the same operand in tile-panel layout Ap[np/128][kp][128] (a pair tile reads
// 32-node x 128-sample slabs that are contiguous 16 KB, and sample shards of a multi-GPU run are
// contiguous byte ranges), from a slab E[B][ld] of the samples [s_base, s_base + ld); total is the
// slab's (ld entries), W the global array.
int launch_weighted_operand_panels(const double* E, const double* length, int32_t n_nodes, int32_t kp,
                                   int64_t ld, int64_t s_base, const double* total, bool prescale, float* Ap,
                                   double* W, double* scratch, cudaStream_t s);
// Rows of scratch (each ld doubles) the two partial-sum reductions need.
int weighted_scratch_chunks(int32_t n_nodes);

// Presence bits, node-major bits[B][nw] (bit s%32 of word s/32).
int launch_embed_bits(const DevTree& t, const int32_t* level_ptr_host, const DevCsr& a,
                      uint32_t* bits, int32_t nw, cudaStream_t s);
// r[s] = sum_v lenq[v] * present(v, s) in fp64.
int launch_presence_rowsum(const uint32_t* bits, int32_t n_nodes, int32_t nw, const double* lenq,
                           double* r, double* scratch, cudaStream_t s);
// Expand bits into the three K-major bf16 operands [np][kp]:
// P = 0/1, Bh = P * len_hi, Bl = P * len_lo.
int launch_expand_operands(const uint32_t* bits, int32_t n_nodes, int32_t nw, int32_t kp,
                           int64_t np, const uint16_t* len_hi, const uint16_t* len_lo,
                           uint16_t* P, uint16_t* Bh, uint16_t* Bl, cudaStream_t s);

// The unweighted embedding stage of the fast path: one CTA per 32 samples runs the whole
// bottom-up presence pass in shared memory (scatter, one block barrier per tree level) and
// publishes its word column in OPERAND COLUMN order: bitsT[w][k] = presence word of node
// order[k] (0 where order[k] < 0); then the row sums r[s] = sum_k lenq[k] * present(k, s)
// (fp64, fixed order) and the expansion into the three K-major operands [np][kp]:
//   bf16: P = 0/1, Bh = P * len_hi, Bl = P * len_lo          (len_hi / len_lo per column)
//   u8  : A = P * qa, Bh = P * qh, Bl = P * ql               (see k_quantize_lengths)
// `node_scratch` holds the per-CTA node-indexed column when the tree is too large for shared
// memory (presence_node_scratch_words(n_nodes, nw) words, 0 when shared memory is used).
int64_t presence_node_scratch_words(int32_t n_nodes, int32_t nw);
void embed_setup();  // cudaFuncSetAttribute calls for the CURRENT device (once per device context)
// qam / col_exp non-null (u8): integer row sums from q[k] = a*m and the per-column exponents.
// Only the word columns [w0, w0 + w_count) (32 samples each) are built: the sample shard of this rank.
// bitsS != null: also the sample-major form bitsS[np][kp / 32] that the bits-fed pair kernel reads.
// peers.n > 0: the kernel stores its bit columns into bitsT of EVERY rank (peer memory over NVLink): the
// all-gather of the sharded embedding is fused into the kernel that produces it.
int launch_embed_presence_fused(const DevTree& t, const int32_t* level_ptr_dev, const DevCsr& a,
                                int32_t nw, int32_t w0, int32_t w_count, int32_t kp, const int32_t* order,
                                uint32_t* node_scratch, uint32_t* bitsT, uint32_t* bitsS, const PeerPtrs& peers,
                                cudaStream_t s);
// r[s] for the same word columns from bitsT (qam / col_exp non-null: integer row sums of the u8 path).
// Independent of the operand expansion, so the job runs the two on different streams.
// r_int != null (u8 integer mode): INSTEAD of r, the exact integer row sums in units of 2^e_min.
int launch_presence_rowsum_t(const uint32_t* bitsT, int32_t n_nodes, int32_t nw, int32_t w0, int32_t w_count,
                             int32_t kp, const double* lenq, const uint32_t* qam, const int32_t* col_exp,
                             double* partial, double* r, int32_t e_min, long long* r_int, cudaStream_t s);
// need[np / 256] (device, may be null = everything): bit 0 = write the A rows of that block of 256
// samples, bit 1 = write its Bh / Bl rows.
// r_int != null (u8 integer mode): the expansion also produces the exact integer row sums (units of 2^e_min) of
// every sample block it touches, from the words it already holds -- no separate row-sum pass over bitsT.
int launch_expand_operands_t(const uint32_t* bitsT, int32_t nw, int32_t kp, int64_t np, bool i8,
                             const void* q0, const void* q1, const void* q2, void* P, void* Bh, void* Bl,
                             const uint8_t* need, const uint32_t* qam, const int32_t* col_exp, int32_t e_min,
                             long long* r_int, cudaStream_t s);
// u8 block floating point: for operand column k with true length len_col[k] >= 0 and chunk
// exponent col_exp[k], find the 8-bit a and 16-bit m = 256*qh + ql minimising
// |a * m * 2^e - len| ; lenq[k] = a * m * 2^e (exact in fp64).
// flag_u[0] = 1e6 * sum of |lenq - len| over the columns whose relative quantisation error
// exceeds 2e-6 (pairs with a unique length below that are recomputed exactly), summed in a fixed
// order through qerr[kp] (device scratch): the same bits on every run, rank and device.
int launch_quantize_lengths(const double* len_col, const int32_t* col_exp, int32_t kp, uint8_t* qa,
                            uint8_t* qh, uint8_t* ql, uint32_t* qam, double* lenq, double* qerr, double* flag_u,
                            cudaStream_t s);

// ---- comm.cu ----------------------------------------------------------------
struct Comm;  // one NCCL communicator (dlopen-bound)
bool comm_unique_id(char* id128, std::string* err);
Comm* comm_create(const char* id128, int rank, int world, std::string* err);  // collective
void comm_destroy(Comm* c);
int comm_rank(const Comm* c);
int comm_world(const Comm* c);
// In-place all-gathers (rank r owns bytes [r*bytes_per_rank, (r+1)*bytes_per_rank) of each buffer),
// issued as one NCCL group on stream s.
bool comm_all_gather_inplace(Comm* c, void* const* bufs, const size_t* bytes_per_rank, int n, cudaStream_t s,
                             std::string* err);

bool comm_all_gather_host(Comm* c, const void* mine, size_t bytes, void* all, cudaStream_t s, std::string* err);
bool comm_barrier(Comm* c, cudaStream_t s, std::string* err);

// ---- exact.cu ---------------------------------------------------------------
// fp64 reference-order distances for pairs [first, first+count) of the job's geometry.
int launch_exact_pairs(const double* E, const double* length, int32_t n_nodes, int64_t ld,
                       bool weighted, int64_t first, const Geometry& geo, int64_t count, double* out, cudaStream_t s);
// Flag -l AS CODED in the reference (normalize = 0): without normalizeFlatNodes the per-sample lists stay in
// the order abundanceToFlatNodes appended them (post-order, unifrac.go:32-53) and unifracDistWeighted's
// merge-join (:174-205) compares ids of lists that are not sorted.  Reproduced literally here; the fast form of
// the same distances (FRC_FLAG_L_TILES) is the keyed variant of the weighted tiles (weighted.cu):
//   launch_postorder_lists  per sample, the (id, raw subtree sum) entries with sum > 0 in post-order, from the
//                           fp64 embedding E[B][ld] (two passes: count -> host prefix is avoided by a device
//                           scan over samples; list_ptr has n_samples + 1 entries)
//   launch_unsorted_pairs   one thread per pair runs the reference's two-pointer walk over the two lists.
int launch_postorder_lists(const double* E, const int32_t* post_order, int32_t n_nodes, int64_t ld, int64_t n_samples,
                           int64_t* list_ptr, int32_t* list_id, double* list_val, cudaStream_t s);
int launch_unsorted_pairs(const int64_t* list_ptr, const int32_t* list_id, const double* list_val,
                          const double* length, int64_t first, const Geometry& geo, int64_t count, double* out,
                          cudaStream_t s);

// ---- wire.cu ----------------------------------------------------------------
// fp32 on PCIe for the fast paths: the pair kernels store fp32, frc_next widens on the host.
void widen_band(const float* src, double* dst, int64_t n, bool stream_stores);  // host

// ---- weighted.cu ------------------------------------------------------------
// Where the fp32 tile panels of the weighted operand live.  Resident (n_shards == 0): one array
// Ap[np/128][kp][128] in this device's HBM (shard[0]).  Capacity mode (the panels of all samples exceed one
// GPU's HBM -- BASELINE config 5 is 320 GB): the samples are cut into 2G shards of `tiles_per_shard` tiles,
// device d builds and keeps the panels of shards d and 2G-1-d, and the OTHER shards visit it one at a time:
// shard[s] points at wherever shard s currently sits in THIS device's HBM (its own slot, or one of two visiting
// buffers that the copy engines fill from the owner over NVLink while the previous shard is being used).  A
// launch only touches the shards of its tiles' rows (own) and of its one column shard.
struct PanelMap {
  const float* shard[16] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                            nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int32_t n_shards = 0;
  int32_t tiles_per_shard = 0;
};
// A is the tile-panel operand (see PanelMap; resident: Ap[np/128][kp][128]).
// Pairs with d < flag_below are appended to flagged[] for the fix-up pass (as the unweighted kernel).
// K non-null: normalize = 0 (-l as coded) on the keyed tiles: K are the resident key panels (launch_embed_f64) and
// node v only counts as matched, |a - b|, where the two samples' keys agree; everywhere else a + b.
int launch_weighted_tiles(const PanelMap& A, int64_t ld, int32_t kp, const float* lenf, bool prescaled,
                          const double* W, const Tile* tiles, int32_t n_tiles, int64_t n_samples,
                          int64_t first, const Geometry& geo, float* out, double flag_below, uint32_t* flagged,
                          unsigned long long* n_flagged, int num_sms, cudaStream_t s, const int32_t* K = nullptr);
// fp64 / fixed-point recompute of the flagged pairs from the CSR rows (total: per-sample normaliser,
// null for -l); ws = ws_ctas zeroed int64 arrays of n_nodes entries (2 * n_nodes with K), left zeroed.
// K non-null: the keyed -l numerator, with the match decision read from the key panels K[np/128][kp][128].
int launch_weighted_fixup(const DevCsr& a, const DevTree& t, const double* total, const double* W,
                          const uint32_t* flagged, const unsigned long long* n_flagged,
                          unsigned long long* count_host, int64_t first, const Geometry& geo, long long* ws,
                          int ws_ctas, float* out, const Exceptions& ex, cudaStream_t s, const int32_t* K = nullptr,
                          int32_t kp = 0);
void weighted_setup();  // cudaFuncSetAttribute calls for the CURRENT device (once per device context)

// ---- unweighted_tc.cu -------------------------------------------------------
// The unweighted pair stage has two operand feeds; the handle records which one a job uses, and the launches
// below dispatch on it.
struct TcOperands;  // opaque: operand feed, tensor maps, chunk table
// Runs of 128-byte K blocks that accumulate uninterrupted in TMEM; device arrays.
struct TcChunks {
  const int32_t* end = nullptr;
  const double* scale = nullptr;
  const int32_t* shift = nullptr;  // u8 integer mode: log2(scale / smallest scale) per chunk
  int32_t n = 0;
  bool biased = false;  // u8 fp64 mode: all scales within 2^8 -> single-instruction biased accumulation
};
// Materialised feed: the three K-major operands [np][kp] (bf16 or u8) in HBM.
// flag_u: device scalar; pairs with unique length below it are recomputed exactly (null: none).
TcOperands* tc_operands_create(const void* P, const void* Bh, const void* Bl, int64_t np, int32_t kp,
                               bool i8, const TcChunks& chunks, const double* len_col, const double* flag_u,
                               std::string* err);
// Bits feed (u8 integer mode only): the u8 operand tiles are expanded inside the pair kernel from the bit rows
// bitsS[np][kp / 32] and the per-column factors qa / qh / ql: no operand arrays in HBM.
TcOperands* tc_operands_create_bits(const uint32_t* bitsS, int64_t np, int32_t kp, const uint8_t* qa,
                                    const uint8_t* qh, const uint8_t* ql, const TcChunks& chunks,
                                    const double* len_col, const double* flag_u, const long long* r_int,
                                    double unit, std::string* err);
// u8 integer mode (chunk scales within 2^16): row sums as integers in units of `unit` = the smallest scale.
void tc_operands_set_int(TcOperands* o, const long long* r_int, double unit);
void tc_operands_destroy(TcOperands* o);
int tc_chunk_kblocks();  // bf16: K blocks per fp32 accumulation run (FRC_TC_CHUNK_KBLOCKS)
// Distances of the tiles in `tiles` into out[index - first]; the band offset of
// every pair with d < flag_below is appended to flagged[] (count in *n_flagged;
// capacity = pairs of the band, so it cannot overflow) for the fix-up pass.
// Integer mode (either feed) flags by flag_u alone; the bits feed does not read r or flag_below.
int launch_unweighted_tc(const TcOperands* ops, const double* r, const Tile* tiles, int32_t n_tiles,
                         int64_t n_samples, int64_t first, const Geometry& geo, float* out, double flag_below,
                         uint32_t* flagged, unsigned long long* n_flagged, int num_sms, cudaStream_t s);
// fp64 recompute of the flagged pairs from the feed's presence rows and true lengths.
int launch_unweighted_fixup(const TcOperands* ops, const uint32_t* flagged,
                            const unsigned long long* n_flagged, unsigned long long* count_host,
                            int64_t first, const Geometry& geo, float* out, const Exceptions& ex, int num_sms,
                            cudaStream_t s);
bool tc_setup(std::string* err);  // driver entry point (once per process) + smem attributes for the CURRENT device

}  // namespace frc
