// Host-only planning of a job (no CUDA calls, no device memory): the pieces of frc_create that decide
// WHAT runs where.  Kept free of the runtime so that the CPU test-suite can drive them through the
// frc_debug_* entry points at the bottom of plan.cpp (tests/test_plan.py) without a GPU.
//
//   band plan      rows of the lower triangle (common/common.go:21-31) -> contiguous flat ranges, owners
//   column plan    fast unweighted: node -> operand column, u8 block-floating-point chunks
//   tile lists     per band: the 128 x 128 sample tiles (CTA-pair tiles for the tensor-core kernel)
//   tree walk      pre-order check, children lists, level order (what enumerateNodes' numbering implies,
//                  frcfrc/unifrac.go:127-133)
//   table staging  the caller's CSR entries checked and copied into the staged table (tests/test_stage.py)
//   variant        which variant of the fast path a job runs (tests/test_variant.py)
#pragma once
#include <cstdint>
#include <functional>
#include <string>
#include <utility>
#include <vector>

#include "../../include/frcfrc_cuda.h"
#include "frc_internal.h"

namespace frc {

// Environment knobs (tests and experiments; DESIGN.md has the table).  Read ONCE per frc_create: nothing
// on the per-band path calls getenv.
struct Knobs {
  bool trace = false;
  int bands_per_rank = 0;     // FRC_BANDS
  int widen_threads = 0;      // FRC_WIDEN_THREADS
  int ws_slab = 0;            // FRC_WS_SLAB
  bool uw_bf16 = false;       // FRC_UW_KERNEL=bf16
  bool u8_acc_f64 = false;    // FRC_U8_ACC=f64
  bool feed_bits = false;     // FRC_UW_FEED=bits
  bool embed_levels = false;  // FRC_EMBED_LEVELS=1
  int peer_push = -1;         // FRC_PEER_PUSH (multi-process sharding: 0 = NCCL all-gather of the bits)
  int group_binades = 3;      // FRC_U8_GROUP_BINADES
  int shard = -1;             // FRC_SHARD (in-process multi-GPU: 0 = every device rebuilds the embedding)
  int capacity = -1;          // FRC_CAPACITY (in-process multi-GPU, fast weighted: 1 / 0 = force / forbid the sharded-panel mode)
  static Knobs read();
};

struct Band {
  int64_t row0 = 0, row1 = 0;   // rows [row0, row1) of the triangle
  int64_t first = 0, count = 0; // flat index of the first pair, number of pairs
  int32_t tile_off = 0, n_tiles = 0;  // into the owner's tile list
  int owner = 0;                // rank (process) or device that computes it
};

// Row boundaries of the bands (multiples of the tile size, first 0, last N).
//   requested > 0 : uniform bands of that many rows (rounded up to whole tiles);
//   otherwise     : bands of (nearly) EQUAL PAIR COUNT, boundaries at N * sqrt(k / n): about
//                   `per_rank` bands per rank when streamed to the host (copies overlap kernels),
//                   one or two per rank when the distances stay in HBM; more when a band would exceed
//                   96 MB (streamed) / 1.5 GB (kept in HBM).
std::vector<int64_t> band_boundaries(int64_t N, int64_t requested, int world, bool d2h, int per_rank, int value_bytes);
// Owners of bands with these pair counts: one band per owner in every round of G consecutive bands, greedily
// balanced (deterministic; the same in every process).
std::vector<int> band_owners(const std::vector<int64_t>& counts, int world);
// Every non-empty band of the triangle, in flat-index order, with its owner.
std::vector<Band> make_bands(int64_t N, int64_t requested, int world, bool d2h, int per_rank, int value_bytes);
// The query x reference block (Geometry in frc_internal.h): bands of whole 128-row query tiles, rows [row0, row1)
// of the staged table (query rows from q0 on) and flat range [(row0 - q0) * n_ref, (row1 - q0) * n_ref).
// `requested` counts query rows; the band count and byte caps follow band_boundaries, the owners band_owners.
// Empty when n_q or n_ref is 0.
std::vector<Band> make_bands_cross(int64_t q0, int64_t n_q, int64_t n_ref, int64_t requested, int world, bool d2h,
                                   int per_rank, int value_bytes);

// Sample shards of the embedding: the padded samples [0, np) in n_shards shards of shard_rows samples (whole tiles).
// A shard sits in its owner's per-sample arrays at [slot * shard_rows, +shard_rows).
//   kWhole    one shard, built by every owner;
//   kSharded  shard r on owner r at its global place (slot r), as the in-place all-gather needs it;
//   kCapacity 2G shards, device d holds shards d and 2G-1-d in slots 0 and 1: row r has r columns, so the two
//             shards of every device add up to the same pair count.
struct Range { int64_t s0, s1, slot; };  // samples [s0, s1) in slot `slot` of their owner
struct ShardPlan {
  enum Mode { kWhole, kSharded, kCapacity };
  int64_t np = 0, shard_rows = 0;
  int n_shards = 1;
  std::vector<int> owner, slot;            // per shard (owner -1: every owner)
  std::vector<std::vector<Range>> ranges;  // per owner, in slot order
};
ShardPlan plan_shards(int64_t N, int owners, ShardPlan::Mode mode);
// Rows [first, second) of the staged table whose CSR entries `owner` reads.  With a sharded embedding on the fast
// unweighted path only the embedding reads the table, and an owner builds its own kSharded shard; otherwise every row
// (the weighted fix-up walks the rows of any flagged pair, and the capacity mode is weighted only).
std::pair<int64_t, int64_t> rows_read(int64_t N, int owners, int owner, bool sharded_fast_uw);

// Capacity mode of the fast weighted path (PanelMap in frc_internal.h): the bands of every shard of `sp`, owned by
// the shard's device.  Bands never straddle a shard.
std::vector<Band> make_bands_capacity(int64_t N, const ShardPlan& sp, int64_t requested, bool d2h);

// Capacity mode, one device: its bands (in row order) grouped by row shard, and per group the tile list ordered by
// the COLUMN shard the tiles read (the order the shards visit in), column-major inside a column shard.
struct CapGroupPlan {
  int shard = 0;                 // row shard (also the last column shard its tiles need)
  int64_t first = 0, count = 0;  // flat range of the group's rows
  int32_t tile_off = 0;          // into `tiles`
  std::vector<int32_t> coff;     // [n_shards + 1] tile offset (inside the group's list) of every column shard
};
// `bands`: the device's bands; appends the groups' tiles to `tiles`; band_group[k] = group of bands[k].
std::vector<CapGroupPlan> plan_capacity_groups(const std::vector<Band>& bands, int64_t N, int64_t shard_rows, int n_shards,
                                               std::vector<Tile>& tiles, std::vector<int>& band_group);

// Fast unweighted path: which node sits in which column of the K-major operands and how the
// columns group into TMEM accumulation chunks.
struct ColumnPlan {
  bool i8 = false;       // u8 block floating point (kind::i8) / bf16 hi-lo planes (kind::f16)
  bool intacc = false;   // u8: all chunk scales within 2^16 -> 64-bit integer accumulation
  bool biased = false;   // u8 fp64 accumulation: all scales within 2^8 (single-instruction form)
  int32_t kp = 0;        // operand columns (multiple of 128 for u8, of 64 for bf16)
  int32_t e_min = 0;     // u8: smallest chunk exponent (integer unit = 2^e_min)
  std::vector<int32_t> col_order;  // [kp] node of column k, -1 = padding
  std::vector<int32_t> col_exp;    // [kp] u8: exponent of the column's chunk
  std::vector<double> len_col;     // [kp] true length of the column's node (0 in padding)
  std::vector<int32_t> chunk_end;  // K blocks (128 B of every operand row) where each chunk ends
  std::vector<double> chunk_scale;
  std::vector<int32_t> chunk_shift;  // u8: log2(scale / smallest scale)
};
ColumnPlan plan_columns(const double* length, int32_t n_nodes, bool want_i8, int group_binades, bool force_f64_acc,
                        int bf16_chunk_kblocks);

// Which variant of the fast path a job runs.  plan_exchange fills the first three fields before the staging starts
// (the staging needs rows_read); plan_variant the rest once the branch lengths are known.  Every stage reads it.
struct Variant {
  enum Exchange { kNone, kInProcess, kNccl };
  Exchange exchange = kNone;     // how the sample shards of the embedding meet
  bool fused_embed = true;       // unweighted embedding: one fused kernel (FRC_EMBED_LEVELS=1: one launch per level)
  bool sharded_fast_uw = false;  // rows_read: an owner reads only its own shard's rows
  bool capacity = false;         // fast weighted over several devices: panels stay sharded (PanelMap), tiles read peers' HBM
  ShardPlan::Mode shard_mode = ShardPlan::kWhole;
  // fast unweighted only (false / 0 otherwise)
  bool want_i8 = false;          // u8 operands (plan_columns) rather than bf16
  bool bits_feed = false;        // integer mode: the pair kernel expands its tiles from the bit rows
  bool rowsum_in_expand = false; // the operand expansion makes the integer row sums
  bool rowsum_split = false;     // fused, no exchange: the row-sum pass runs on the second compute stream
  bool peer_store = false;       // kInProcess: the embedding kernel stores its bit columns into every device
  bool peer_push = false;        // kNccl: the same into every rank over IPC (wanted; prepare_part may fall back)
  bool need_blocks = false;      // several owners: the expansion fills only the operand rows this owner's tiles read
  int operand_kind = 0;          // frc_info_t::operand_kind: 0 none, 1 bf16, 2 u8, 3 u8 from the bits
};
// What the variant depends on: the options, the path taken, the context.
struct VariantIn {
  bool exact = false, weighted = false, keyed = false, rect = false;
  uint32_t flags = 0;
  int world = 1, rank = 0;              // opts (world <= 0: 1)
  int64_t N = 0;
  int n_parts = 1;                      // devices of the context
  bool peer_ok = false;
  int comm_world = -1, comm_rank = -1;  // the context's communicator (-1: none)
  int owners() const { return n_parts > 1 ? n_parts : world; }
};
Variant plan_exchange(const VariantIn& in, const Knobs& k);
// The rest of `v` (from plan_exchange), and for the fast unweighted path the column plan of length[B] into *cols.
// free_hbm(&bytes) gives device 0's free HBM (false: the query failed, which chooses neither mode); it is asked at
// most once, and only when the panels or the u8 operands are large enough for the answer to matter.  Returns FRC_OK
// or an error code with its message in *err.
int plan_variant(Variant& v, const VariantIn& in, const Knobs& k, bool neg_len, const double* length, int32_t B,
                 int bf16_chunk_kblocks, const std::function<bool(size_t*)>& free_hbm, ColumnPlan* cols,
                 std::string* err);

// Tiles of one band, appended to `tiles`: pair tiles (ti, tj) + (ti, tj + 1), tj even, walked in
// super-tiles of ~9 tile rows x ~8 tile-pair columns when `pair_tiles` (tensor-core kernel), plain
// column-major 128 x 128 tiles otherwise (FP32 tile kernel).  Triangle (col_tiles == 0): tj <= ti;
// rectangle: every tj < col_tiles (the reference tiles), no diagonal.
void append_band_tiles(Band& b, bool pair_tiles, std::vector<Tile>& tiles, int32_t col_tiles = 0);
// Per block of 256 samples: bit 0 = some tile reads its A rows (column samples), bit 1 = its Bh / Bl rows.
std::vector<uint8_t> operand_need_blocks(const std::vector<Tile>& tiles, int64_t np, bool pair_tiles);

// The tree walk.  Outputs go to caller-provided arrays (pinned staging memory in frc_create).
struct TreeLevels {
  int32_t height = -1;             // levels above the leaves; -1 = failed
  int32_t bad_parent = 0, bad_order = 0;  // first offending node ids
  std::vector<int32_t> level_ptr;  // [height + 2]
};
// Pre-order check: parent[v] must be a smaller id (else *bad_parent = the first v that breaks it) and the node of its
// depth on the current root-to-(v-1) path (else *bad_order = the first such v).  depth[n_nodes] receives the depths.
bool check_preorder(const int32_t* parent, int32_t n_nodes, int32_t* depth, int32_t* bad_parent, int32_t* bad_order);
// check_preorder, then the level order: level_nodes[B] grouped by height (leaves first), level_parent[k] = parent of
// level_nodes[k].
TreeLevels tree_levels(const int32_t* parent, int32_t n_nodes, int32_t* level_nodes, int32_t* level_parent);
// Children lists in ascending id (= file order).  false when a parent id is out of range.
bool tree_children(const int32_t* parent, int32_t n_nodes, int32_t* child_ptr, int32_t* child_idx);
// post_order[k] = node visited k-th by abundanceToFlatNodes' recursion (children first, in file order,
// then the node: unifrac.go:32-53).
void tree_post_order(const int32_t* parent, int32_t n_nodes, int32_t* post_order);

// FRC_FLAG_PRUNE (DESIGN.md, "Pruning to the table's support").  The support S is the root and every node with a
// marked node in its subtree; the survivors keep their order, which is again a pre-order numbering.  With `merge`, a
// non-root survivor with exactly one surviving child is dropped as well: the lowest node of such a chain takes the
// parent above the chain, the chain's lengths summed top-down in fp64, and mult = the number of original nodes it
// stands for (the mults add up to |S|).  parent[] must satisfy 0 <= parent[v] < v for v > 0 (check_preorder).
struct PrunedTree {
  int32_t n_nodes = 0;
  std::vector<int32_t> parent, new_of_old;  // new_of_old[v] = id in the pruned tree, -1 if v was dropped
  std::vector<double> length;
  std::vector<int32_t> mult;
};
PrunedTree prune_tree(const int32_t* parent, const double* length, int32_t n_nodes, const uint8_t* marks, bool merge);

// The table frc_create stages: the caller's table, or for frc_create_cross the reference rows, empty rows up to q0
// (Geometry), then the query rows, whose entries follow the reference entries.  The one place that maps staged rows
// and entries back to the caller's tables.  The tables' headers have been checked (validate_header).
struct StagedTable {
  const frc_csr_t* ref = nullptr;    // frc_create: the table; frc_create_cross: the reference table
  const frc_csr_t* query = nullptr;  // frc_create_cross: the query table
  int64_t q0 = 0;                    // staged row of query row 0

  int64_t ref_nnz() const { return ref->n_samples > 0 ? ref->row_ptr[ref->n_samples] : 0; }
  bool in_query(int64_t s) const { return query && s >= q0; }
  // the caller's entries of staged row s (not for the empty rows below q0)
  const int32_t* col(int64_t s) const {
    return in_query(s) ? query->col + query->row_ptr[s - q0] : ref->col + ref->row_ptr[s];
  }
  const double* val(int64_t s) const {
    return in_query(s) ? query->val + query->row_ptr[s - q0] : ref->val + ref->row_ptr[s];
  }
  // "sample #k", "reference sample #k" or "query sample #k" (k from 1, within the caller's table)
  std::string row_name(int64_t s) const;
  // the staged row_ptr: q0 + n_q + 1 entries (frc_create: n_samples + 1)
  void fill_row_ptr(int64_t* rp) const;
};

// Checks the entries of staged rows [s0, s1) against the caller's tree parent[n_nodes] and copies them into the
// staged col / val (rp: the staged row_ptr) with streaming stores, node ids mapped through new_of_old (null: kept).
// The checks, in this order, on every entry: node id in range, a leaf (pre-order ids: a node's first child is the next
// id), value positive and finite, and -- only when values are used (val != null) -- not listed twice in its row.  The
// duplicate test marks stamp[node] = stamp_tag + row: stamp[n_nodes] persists across jobs, and each job's tag lies
// past every mark of the previous ones.  Stops at the first bad entry and returns its message (empty: none).
std::string stage_entries(const StagedTable& t, const int64_t* rp, int64_t s0, int64_t s1, const int32_t* parent,
                          int32_t n_nodes, const int32_t* new_of_old, int64_t* stamp, int64_t stamp_tag, int32_t* col,
                          double* val);
// The staged entries [k0, k1) are checked and copied in n_chunks chunks of whole rows and about equal entry counts:
// rows [first, second) of chunk ch (rp: the staged row_ptr of N rows).
std::pair<int64_t, int64_t> chunk_rows(const int64_t* rp, int64_t N, int64_t k0, int64_t k1, int ch, int n_chunks);
// The error frc_create reports from its chunks' messages: the first bad entry in row order (empty: none).
const std::string& first_error(const std::vector<std::string>& chunk_errors);
// FRC_FLAG_PRUNE: marks[node] = 1 for every node listed in the staged entries [k0, k1) of either table (ids outside
// [0, n_nodes) are left to stage_entries).  Relaxed atomic stores: several threads mark disjoint entry ranges.
void mark_table_leaves(const StagedTable& t, int64_t k0, int64_t k1, int32_t n_nodes, uint8_t* marks);

}  // namespace frc
