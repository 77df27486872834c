// Host-only planning of a job (no CUDA calls, no device memory): the pieces of frc_create that decide
// WHAT runs where.  Kept free of the runtime so that the CPU test-suite can drive them through the
// frc_debug_* entry points at the bottom of plan.cpp (tests/test_plan.py) without a GPU.
//
//   band plan      rows of the lower triangle (common/common.go:21-31) -> contiguous flat ranges, owners
//   column plan    fast unweighted: node -> operand column, u8 block-floating-point chunks
//   tile lists     per band: the 128 x 128 sample tiles (CTA-pair tiles for the tensor-core kernel)
//   tree walk      pre-order check, children lists, level order (what enumerateNodes' numbering implies,
//                  frcfrc/unifrac.go:127-133)
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "frc_internal.h"

namespace frc {

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

}  // namespace frc
