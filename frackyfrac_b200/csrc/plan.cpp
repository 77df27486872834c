// Host-only planning (see plan.h).  No CUDA runtime call in this file.
#include "plan.h"

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#if defined(__x86_64__)
#include <immintrin.h>
#endif

namespace frc {

// Largest-first onto the least loaded owner: the best balance, any order.
static std::vector<int> band_owners_lpt(const std::vector<int64_t>& cnt, int world) {
  const size_t n = cnt.size();
  std::vector<int> owner(n, 0);
  std::vector<size_t> order(n);
  for (size_t k = 0; k < n; ++k) order[k] = k;
  std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return cnt[a] > cnt[b]; });
  std::vector<int64_t> load(world, 0);
  for (size_t k : order) {
    int best = 0;
    for (int r = 1; r < world; ++r)
      if (load[r] < load[best]) best = r;
    owner[k] = best;
    load[best] += cnt[k];
  }
  return owner;
}

std::vector<int> band_owners(const std::vector<int64_t>& counts, int world) {
  // Few bands (at most 8 per owner: the automatic plan of a triangle that fits the rings): every owner queues
  // ALL its bands at once, so the order in which the consumer reads them cannot stall anybody and the
  // assignment only has to balance: largest first onto the least loaded owner (within ~1 %).
  if (world > 1 && counts.size() <= 8 * static_cast<size_t>(world)) return band_owners_lpt(counts, world);
  // More bands than the rings hold: dealt in ROUNDS of G consecutive bands, every owner exactly one band per round: a consumer reading the
  // stream in flat-index order then drains every owner's ring (and PCIe link) at the same pace, whatever the
  // ring size (a largest-first assignment over all bands balances better but hands one owner runs of
  // consecutive bands: the others' rings fill up and their GPUs idle until the consumer gets to them).
  // Inside a round the largest band goes to the owner with the smallest load so far (tile-row rounding makes
  // band sizes differ by ~10 % on small triangles; the greedy match keeps the owners within ~2 %).
  const size_t n = counts.size();
  std::vector<int> owner(n, 0);
  if (world <= 1) return owner;
  std::vector<int64_t> load(world, 0);
  std::vector<int> who(world);
  std::vector<size_t> idx;
  for (size_t k0 = 0; k0 < n; k0 += world) {
    const size_t k1 = std::min(n, k0 + world);
    idx.clear();
    for (size_t k = k0; k < k1; ++k) idx.push_back(k);
    auto cnt = [&](size_t k) { return counts[k]; };
    std::stable_sort(idx.begin(), idx.end(), [&](size_t a, size_t b) { return cnt(a) > cnt(b); });
    for (int r = 0; r < world; ++r) who[r] = r;
    std::stable_sort(who.begin(), who.end(), [&](int a, int b) { return load[a] < load[b]; });
    for (size_t t = 0; t < idx.size(); ++t) {
      owner[idx[t]] = who[t];
      load[who[t]] += cnt(idx[t]);
    }
  }
  return owner;
}

std::vector<int64_t> band_boundaries(int64_t N, int64_t requested, int world, bool d2h, int per_rank, int value_bytes) {
  std::vector<int64_t> rows;
  rows.push_back(0);
  if (N <= 0) return rows;
  if (world < 1) world = 1;
  if (requested > 0) {
    const int64_t step = round_up(requested, kTile);
    for (int64_t r = step; r < N; r += step) rows.push_back(r);
    rows.push_back(N);
    return rows;
  }
  const int64_t tile_rows = (N + kTile - 1) / kTile;
  int64_t n = d2h ? 8LL * world : (world == 1 ? 1 : 2LL * world);
  if (d2h && per_rank > 0) n = static_cast<int64_t>(per_rank) * world;
  const double total_bytes = static_cast<double>(value_bytes) * static_cast<double>(N) * static_cast<double>(N - 1) / 2.0;
  // streamed to the host: bands of <= 96 MB keep the pinned ring small (pinning memory costs ~0.4 s
  // per GB, paid by the first job of a context) and are still several waves of tiles each
  const double band_cap = d2h ? 96.0 * 1024 * 1024 : 1536.0 * 1024 * 1024;
  const int64_t by_size = static_cast<int64_t>(std::ceil(total_bytes / band_cap));
  if (by_size > n) n = round_up(by_size, 2LL * world);
  n = std::max<int64_t>(1, std::min(n, std::max<int64_t>(world, tile_rows / 2)));
  for (int64_t k = 1; k < n; ++k) {
    int64_t r = static_cast<int64_t>(std::llround(static_cast<double>(N) * std::sqrt(static_cast<double>(k) / n) / kTile)) * kTile;
    r = std::max(r, rows.back() + kTile);
    if (r >= N) break;
    rows.push_back(r);
  }
  rows.push_back(N);
  if (d2h && world == 1 && rows.size() > 2) {
    // one device, streamed: the D2H chain (the bound of an end-to-end call) can only start when the FIRST band
    // is done, so that one is cut again: a quarter of a band first, the rest of it second
    const int64_t r = static_cast<int64_t>(std::llround(static_cast<double>(N) * std::sqrt(0.25 / static_cast<double>(n)) / kTile)) * kTile;
    if (r >= kTile && r < rows[1]) rows.insert(rows.begin() + 1, r);
  }
  return rows;
}

std::vector<Band> make_bands(int64_t N, int64_t requested, int world, bool d2h, int per_rank, int value_bytes) {
  const std::vector<int64_t> rows = band_boundaries(N, requested, world, d2h, per_rank, value_bytes);
  std::vector<int64_t> counts;
  for (size_t k = 0; k + 1 < rows.size(); ++k) counts.push_back(tri(rows[k + 1]) - (rows[k] >= 2 ? tri(rows[k]) : 0));
  const std::vector<int> owners = band_owners(counts, world);
  std::vector<Band> bands;
  for (size_t k = 0; k + 1 < rows.size(); ++k) {
    Band b;
    b.row0 = rows[k]; b.row1 = rows[k + 1];
    b.first = b.row0 >= 2 ? tri(b.row0) : 0;
    b.count = tri(b.row1) - b.first;
    b.owner = owners[k];
    if (b.count > 0) bands.push_back(b);
  }
  return bands;
}

std::vector<Band> make_bands_cross(int64_t q0, int64_t n_q, int64_t n_ref, int64_t requested, int world, bool d2h,
                                   int per_rank, int value_bytes) {
  // query rows [0, n_q) relative to q0; every row holds n_ref pairs, so equal pair counts are equal row counts
  std::vector<int64_t> rows{0};
  if (n_q > 0 && n_ref > 0) {
    if (world < 1) world = 1;
    if (requested > 0) {
      const int64_t step = round_up(requested, kTile);
      for (int64_t r = step; r < n_q; r += step) rows.push_back(r);
    } else {
      // the policy of band_boundaries: band count per owner, the same byte caps per band, whole tiles
      const int64_t tile_rows = (n_q + kTile - 1) / kTile;
      int64_t n = d2h ? 8LL * world : (world == 1 ? 1 : 2LL * world);
      if (d2h && per_rank > 0) n = static_cast<int64_t>(per_rank) * world;
      const double total_bytes = static_cast<double>(value_bytes) * static_cast<double>(n_q) * static_cast<double>(n_ref);
      const double band_cap = d2h ? 96.0 * 1024 * 1024 : 1536.0 * 1024 * 1024;
      const int64_t by_size = static_cast<int64_t>(std::ceil(total_bytes / band_cap));
      if (by_size > n) n = round_up(by_size, 2LL * world);
      n = std::max<int64_t>(1, std::min(n, tile_rows));
      for (int64_t k = 1; k < n; ++k) {
        int64_t r = static_cast<int64_t>(std::llround(static_cast<double>(n_q) * k / n / kTile)) * kTile;
        r = std::max(r, rows.back() + kTile);
        if (r >= n_q) break;
        rows.push_back(r);
      }
      if (d2h && world == 1 && rows.size() > 1) {
        // (as for the triangle: the first band is cut again so that the D2H chain starts early)
        const int64_t r = static_cast<int64_t>(std::llround(static_cast<double>(n_q) * 0.25 / n / kTile)) * kTile;
        if (r >= kTile && r < rows[1]) rows.insert(rows.begin() + 1, r);
      }
    }
    rows.push_back(n_q);
  }
  std::vector<int64_t> counts;
  for (size_t k = 0; k + 1 < rows.size(); ++k) counts.push_back((rows[k + 1] - rows[k]) * n_ref);
  const std::vector<int> owners = band_owners(counts, world);
  std::vector<Band> bands;
  for (size_t k = 0; k + 1 < rows.size(); ++k) {
    Band b;
    b.row0 = q0 + rows[k]; b.row1 = q0 + rows[k + 1];
    b.first = rows[k] * n_ref;
    b.count = counts[k];
    b.owner = owners[k];
    bands.push_back(b);
  }
  return bands;
}

ShardPlan plan_shards(int64_t N, int owners, ShardPlan::Mode mode) {
  ShardPlan sp;
  owners = std::max(1, owners);
  sp.n_shards = mode == ShardPlan::kWhole ? 1 : mode == ShardPlan::kCapacity ? 2 * owners : owners;
  sp.np = std::max<int64_t>(kTile, round_up(N, kTile * static_cast<int64_t>(sp.n_shards)));
  sp.shard_rows = sp.np / sp.n_shards;
  sp.ranges.resize(owners);
  for (int s = 0; s < sp.n_shards; ++s) {
    const int owner = mode == ShardPlan::kWhole ? -1 : s < owners ? s : sp.n_shards - 1 - s;
    const int slot = mode == ShardPlan::kCapacity ? (s < owners ? 0 : 1) : s;
    sp.owner.push_back(owner);
    sp.slot.push_back(slot);
    const Range rg{s * sp.shard_rows, (s + 1) * sp.shard_rows, slot};  // (ascending s: every owner's in slot order)
    if (owner >= 0) sp.ranges[owner].push_back(rg);
    else for (std::vector<Range>& r : sp.ranges) r.push_back(rg);
  }
  return sp;
}

std::pair<int64_t, int64_t> rows_read(int64_t N, int owners, int owner, bool sharded_fast_uw) {
  if (!sharded_fast_uw || N <= 0) return {0, N};
  const Range own = plan_shards(N, owners, ShardPlan::kSharded).ranges[owner][0];
  return {std::min(N, own.s0), std::min(N, own.s1)};
}

std::vector<Band> make_bands_capacity(int64_t N, const ShardPlan& sp, int64_t requested, bool d2h) {
  std::vector<Band> bands;
  if (N < 2) return bands;
  const int64_t R = sp.shard_rows;
  const double band_cap = (d2h ? 96.0 : 1536.0) * 1024 * 1024 / 8.0;  // pairs per band, as in band_boundaries
  for (int s = 0; s < sp.n_shards; ++s) {
    const int64_t r0 = s * R, r1 = std::min<int64_t>(N, (s + 1) * R);
    if (r0 >= r1) break;
    const int owner = sp.owner[s];
    std::vector<int64_t> rows;
    rows.push_back(r0);
    if (requested > 0) {
      const int64_t step = round_up(requested, kTile);
      for (int64_t r = r0 + step; r < r1; r += step) rows.push_back(r);
    } else {
      const int64_t t0 = r0 >= 2 ? tri(r0) : 0, pairs = tri(r1) - t0;
      const int64_t tile_rows = (r1 - r0 + kTile - 1) / kTile;
      int64_t nb = std::max<int64_t>(d2h ? 4 : 1, static_cast<int64_t>(std::ceil(static_cast<double>(pairs) / band_cap)));
      nb = std::max<int64_t>(1, std::min(nb, tile_rows));
      for (int64_t k = 1; k < nb; ++k) {
        // row r with tri(r) = t0 + pairs * k / nb
        const double target = static_cast<double>(t0) + static_cast<double>(pairs) * k / nb;
        int64_t r = static_cast<int64_t>(std::llround((0.5 + std::sqrt(0.25 + 2.0 * target)) / kTile)) * kTile;
        r = std::max(r, rows.back() + kTile);
        if (r >= r1) break;
        rows.push_back(r);
      }
    }
    rows.push_back(r1);
    for (size_t k = 0; k + 1 < rows.size(); ++k) {
      Band b;
      b.row0 = rows[k]; b.row1 = rows[k + 1];
      b.first = b.row0 >= 2 ? tri(b.row0) : 0;
      b.count = tri(b.row1) - b.first;
      b.owner = owner;
      if (b.count > 0) bands.push_back(b);
    }
  }
  return bands;
}

std::vector<CapGroupPlan> plan_capacity_groups(const std::vector<Band>& bands, int64_t N, int64_t shard_rows, int n_shards,
                                               std::vector<Tile>& tiles, std::vector<int>& band_group) {
  std::vector<CapGroupPlan> groups;
  band_group.clear();
  const int64_t T = shard_rows / kTile;
  for (const Band& b : bands) {
    const int shard = static_cast<int>(b.row0 / shard_rows);
    if (groups.empty() || groups.back().shard != shard) {
      CapGroupPlan g;
      g.shard = shard;
      g.first = b.first;
      groups.push_back(g);
    }
    groups.back().count = b.first + b.count - groups.back().first;
    band_group.push_back(static_cast<int>(groups.size()) - 1);
  }
  for (CapGroupPlan& g : groups) {
    const int64_t r0 = static_cast<int64_t>(g.shard) * shard_rows, r1 = std::min<int64_t>(N, r0 + shard_rows);
    const int32_t t0 = static_cast<int32_t>(r0 / kTile), t1 = static_cast<int32_t>((r1 - 1) / kTile);
    g.tile_off = static_cast<int32_t>(tiles.size());
    g.coff.assign(n_shards + 1, 0);
    for (int c = 0; c <= g.shard; ++c) {
      g.coff[c] = static_cast<int32_t>(tiles.size()) - g.tile_off;
      for (int32_t tj = static_cast<int32_t>(c * T); tj < static_cast<int32_t>((c + 1) * T) && tj <= t1; ++tj)
        for (int32_t ti = std::max(tj, t0); ti <= t1; ++ti) tiles.push_back({ti, tj});
    }
    for (int c = g.shard + 1; c <= n_shards; ++c) g.coff[c] = static_cast<int32_t>(tiles.size()) - g.tile_off;
  }
  return groups;
}

// Column k of the K-major operands holds node col_order[k] (-1: padding).  bf16: identity order,
// uniform accumulation chunks.  u8: nodes grouped by binade triples of their length so that one
// power-of-two scale per chunk leaves every length a 21..24-bit integer a * m (zero-length nodes
// contribute nothing and get no column).
ColumnPlan plan_columns(const double* length, int32_t B, bool want_i8, int gb, bool force_f64_acc,
                        int bf16_chunk_kblocks) {
  ColumnPlan p;
  p.i8 = want_i8;
  if (!want_i8) {
    p.kp = static_cast<int32_t>(round_up(B, kKBlock));
    p.col_order.assign(p.kp, -1);
    p.len_col.assign(p.kp, 0.0);
    for (int32_t v = 0; v < B; ++v) { p.col_order[v] = v; p.len_col[v] = length[v]; }
    const int32_t nkb = p.kp / kKBlock, per = std::max(1, bf16_chunk_kblocks);
    for (int32_t kb = 0; kb < nkb;) { kb = std::min(nkb, kb + per); p.chunk_end.push_back(kb); p.chunk_scale.push_back(1.0); }
    return p;
  }
  constexpr int kGroups = 24, kBlockCols = 128, kMaxChunkBlocks = 128;
  gb = std::max(1, std::min(16, gb));
  // floor(log2(l)) of a positive finite double straight from its exponent field (denormals: -1023,
  // they all land in the last group)
  auto ilog = [](double l) {
    uint64_t u;
    memcpy(&u, &l, 8);
    return static_cast<int>((u >> 52) & 0x7FF) - 1023;
  };
  int e_max = INT32_MIN;
  for (int32_t v = 0; v < B; ++v)
    if (length[v] > 0) e_max = std::max(e_max, ilog(length[v]));
  // group of every node, through a table over the exponent distance; 255 = no column (length 0)
  uint8_t group_tab[2112];
  for (int d = 0; d < 2112; ++d) group_tab[d] = static_cast<uint8_t>(std::min(kGroups - 1, d / gb));
  std::vector<uint8_t> grp(B);
  int32_t cnt[kGroups + 1] = {0};
  for (int32_t v = 0; v < B; ++v) {
    const double l = length[v];
    const uint8_t g = l > 0 ? group_tab[e_max - ilog(l)] : static_cast<uint8_t>(kGroups);
    grp[v] = g;
    cnt[g]++;
  }
  // Groups -> accumulation chunks.  Every chunk costs a TMEM drain (>= 2k cycles: 128 KB at
  // 64 B/clk) that only hides behind a long enough MMA run, so a group opens a chunk of its own
  // only when it is large; smaller groups below it join the current chunk at that chunk's
  // (larger) scale.  Their lengths then keep fewer significant bits; k_quantize_lengths sums the
  // absolute error of every column that misses 2e-6 relative, and pairs whose unique length is
  // too small for that sum to be harmless are recomputed exactly (flag_u).
  constexpr int32_t kMinChunkCols = 1024;
  int chunk_of[kGroups], chunk_exp[kGroups], n_ch = 0;
  int32_t ch_cols[kGroups] = {0};
  for (int g = 0; g < kGroups; ++g) {
    if (cnt[g] == 0) { chunk_of[g] = -1; continue; }
    if (n_ch == 0 || cnt[g] >= kMinChunkCols) {
      chunk_exp[n_ch] = e_max - gb * g - 22;  // top of the group: len < 2^(e_max-gb*g+1) -> x < 2^23
      ++n_ch;
    }
    chunk_of[g] = n_ch - 1;
    ch_cols[n_ch - 1] += cnt[g];
  }
  // Chunks are laid out along K from the largest to the smallest (the order is free): the MMA
  // run of a large chunk then covers the ratio epilogue of the previous tile plus the drain of
  // the small chunk before it.
  int ch_order[kGroups];
  for (int c = 0; c < n_ch; ++c) ch_order[c] = c;
  std::stable_sort(ch_order, ch_order + n_ch, [&](int a, int b) { return ch_cols[a] > ch_cols[b]; });
  int32_t ch_off[kGroups + 1] = {0}, ch_at[kGroups], fill[kGroups];
  for (int k = 0; k < n_ch; ++k) {
    ch_at[ch_order[k]] = ch_off[k];
    ch_off[k + 1] = ch_off[k] + static_cast<int32_t>(round_up(ch_cols[ch_order[k]], kBlockCols));
  }
  p.kp = std::max<int32_t>(ch_off[n_ch], kBlockCols);
  p.col_order.assign(p.kp, -1); p.col_exp.assign(p.kp, 0); p.len_col.assign(p.kp, 0.0);
  {  // columns of a chunk: its groups from large to small lengths, node id order inside a group
    int32_t next[kGroups];
    for (int c = 0; c < n_ch; ++c) next[c] = ch_at[c];
    for (int g = 0; g < kGroups; ++g)
      if (chunk_of[g] >= 0) { fill[g] = next[chunk_of[g]]; next[chunk_of[g]] += cnt[g]; }
  }
  for (int32_t v = 0; v < B; ++v) {
    if (grp[v] == kGroups) continue;
    const int32_t k = fill[grp[v]]++;
    p.col_order[k] = v; p.len_col[k] = length[v];
  }
  for (int k = 0; k < n_ch; ++k) {
    const int c = ch_order[k];
    for (int32_t q = ch_off[k]; q < ch_off[k + 1]; ++q) p.col_exp[q] = chunk_exp[c];
    for (int32_t kb = ch_off[k] / kBlockCols; kb < ch_off[k + 1] / kBlockCols;) {
      kb = std::min(ch_off[k + 1] / kBlockCols, kb + kMaxChunkBlocks);  // plane sums stay < 2^31
      p.chunk_end.push_back(kb);
      p.chunk_scale.push_back(std::ldexp(1.0, chunk_exp[c]));
    }
  }
  if (p.chunk_end.empty()) { p.chunk_end.push_back(1); p.chunk_scale.push_back(1.0); }
  // integer mode when all chunk scales lie within 2^16 (sums then stay below 2^60)
  int lo = INT32_MAX, hi = INT32_MIN;
  for (double sc : p.chunk_scale) { const int e = std::ilogb(sc); lo = std::min(lo, e); hi = std::max(hi, e); }
  p.intacc = hi - lo <= 16 && !force_f64_acc;
  p.biased = hi - lo <= 8;
  p.e_min = lo;
  for (double sc : p.chunk_scale) p.chunk_shift.push_back(std::ilogb(sc) - lo);
  return p;
}

Knobs Knobs::read() {
  Knobs k;
  auto num = [](const char* name, int dflt) { const char* e = getenv(name); return e && *e ? atoi(e) : dflt; };
  auto is = [](const char* name, const char* v) { const char* e = getenv(name); return e && !strcmp(e, v); };
  k.trace = getenv("FRC_TRACE") != nullptr;
  k.bands_per_rank = std::max(0, num("FRC_BANDS", 0));
  k.widen_threads = std::max(0, num("FRC_WIDEN_THREADS", 0));
  k.ws_slab = std::max(0, num("FRC_WS_SLAB", 0));
  k.uw_bf16 = is("FRC_UW_KERNEL", "bf16");
  k.u8_acc_f64 = is("FRC_U8_ACC", "f64");
  k.feed_bits = is("FRC_UW_FEED", "bits");
  k.embed_levels = num("FRC_EMBED_LEVELS", 0) == 1;
  k.peer_push = num("FRC_PEER_PUSH", -1);
  k.group_binades = num("FRC_U8_GROUP_BINADES", 3);
  k.shard = num("FRC_SHARD", -1);
  k.capacity = num("FRC_CAPACITY", -1);
  return k;
}

Variant plan_exchange(const VariantIn& in, const Knobs& k) {
  Variant v;
  v.fused_embed = !k.embed_levels;
  if (in.exact) return v;
  if (in.n_parts > 1 && in.peer_ok && k.shard != 0 && (in.weighted || v.fused_embed)) v.exchange = Variant::kInProcess;
  if (in.n_parts == 1 && in.world > 1 && (in.flags & FRC_FLAG_SHARD_EMBED)) v.exchange = Variant::kNccl;
  v.sharded_fast_uw = v.exchange != Variant::kNone && !in.weighted;
  return v;
}

int plan_variant(Variant& v, const VariantIn& in, const Knobs& k, bool neg_len, const double* length, int32_t B,
                 int bf16_chunk_kblocks, const std::function<bool(size_t*)>& free_hbm, ColumnPlan* cols,
                 std::string* err) {
  const bool fast_uw = !in.exact && !in.weighted;
  auto refuse = [&](int code, const char* msg) { *err = msg; return code; };
  if (v.exchange == Variant::kNccl) {
    if (in.comm_world != in.world || in.comm_rank != in.rank)
      return refuse(FRC_ERR_STATE, "FRC_FLAG_SHARD_EMBED needs a context whose communicator "
                                   "(frc_ctx_comm_init) matches opts->rank / opts->world");
    if (fast_uw && !v.fused_embed) return refuse(FRC_ERR_UNSUPPORTED, "FRC_EMBED_LEVELS=1 cannot build a sample shard");
  }
  v.shard_mode = v.exchange == Variant::kNone ? ShardPlan::kWhole : ShardPlan::kSharded;
  // (free_hbm costs milliseconds, a cudaMemGetInfo: only asked when it can matter)
  size_t free_b = 0;
  // Capacity mode of the fast weighted path: the fp32 panels of ALL samples (kp x np x 4 bytes: 320 GB at
  // BASELINE config 5) would not fit one device -> they stay sharded where they are built (two shards per
  // device) and the pair tiles read remote column panels over NVLink (PanelMap, weighted.cu).
  if (v.exchange == Variant::kInProcess && in.weighted && k.capacity != 0 && in.N >= 2) {
    bool want = k.capacity == 1;
    if (!want) {
      // (keyed -l tiles: an int32 key next to every fp32 value)
      const double panels = (in.keyed ? 8.0 : 4.0) * static_cast<double>(round_up(B, kKBlock)) *
                            static_cast<double>(plan_shards(in.N, in.n_parts, ShardPlan::kCapacity).np);
      if (panels > 24.0 * (1 << 30) && free_hbm(&free_b) && panels > 0.55 * static_cast<double>(free_b)) want = true;
    }
    if (want && in.rect)
      return refuse(FRC_ERR_UNSUPPORTED, "frc_create_cross keeps the weighted panels of all samples on every device; the "
                                         "capacity mode, which shards them over the devices when they exceed about half "
                                         "of one device's free HBM (or with FRC_CAPACITY=1), only runs triangle jobs");
    if (want && in.keyed)
      return refuse(FRC_ERR_UNSUPPORTED, "the key-matched tiles of -l as coded (FRC_FLAG_L_TILES) keep the value and key "
                                         "panels of all samples on every device; the capacity mode, which shards them "
                                         "over the devices when they exceed about half of one device's free HBM (or with "
                                         "FRC_CAPACITY=1), does not carry keys");
    v.capacity = want;
    if (want) v.shard_mode = ShardPlan::kCapacity;
  }
  if (!fast_uw) return FRC_OK;
  v.want_i8 = v.fused_embed && !neg_len && !(in.flags & FRC_FLAG_UW_BF16) && !k.uw_bf16;
  *cols = plan_columns(length, B, v.want_i8, k.group_binades, k.u8_acc_f64, bf16_chunk_kblocks);
  v.bits_feed = cols->intacc && ((in.flags & FRC_FLAG_UW_BITS) != 0 || k.feed_bits);
  if (cols->intacc && !v.bits_feed) {
    // capacity: when the three u8 operand arrays would not fit the free HBM (with room for the
    // output ring), the pair kernel expands its tiles from the bit rows instead (8x less memory,
    // about half the speed: DESIGN.md)
    const double need = 3.0 * static_cast<double>(plan_shards(in.N, in.owners(), v.shard_mode).np) * cols->kp;
    if (need > 32.0 * (1 << 30) && free_hbm(&free_b) && need > 0.80 * static_cast<double>(free_b)) v.bits_feed = true;
  }
  // Row sums.  Integer mode with materialised operands: the operand expansion produces them for every sample from
  // the words it holds anyway.  Otherwise a separate pass over this part's shard, beside the expansion on the second
  // compute stream unless an exchange sits between.
  v.rowsum_in_expand = cols->intacc && !v.bits_feed;
  v.rowsum_split = v.fused_embed && v.exchange == Variant::kNone && !v.rowsum_in_expand;
  v.peer_store = v.exchange == Variant::kInProcess && !v.bits_feed;
  v.peer_push = v.exchange == Variant::kNccl && !v.bits_feed && in.world <= 8 && k.peer_push != 0;
  v.need_blocks = v.fused_embed && in.owners() > 1;
  v.operand_kind = cols->i8 ? (v.bits_feed ? 3 : 2) : 1;
  return FRC_OK;
}

void append_band_tiles(Band& b, bool pair_tiles, std::vector<Tile>& tiles, int32_t col_tiles) {
  b.tile_off = static_cast<int32_t>(tiles.size());
  const int32_t t0 = static_cast<int32_t>(b.row0 / kTile), t1 = static_cast<int32_t>((b.row1 - 1) / kTile);
  const bool rect = col_tiles > 0;
  if (pair_tiles) {
    // pair tiles: (ti, tj) and (ti, tj+1) with tj even; needed when tj <= ti (rectangle: tj < col_tiles).
    // The clusters that run together (74 on a B200) take consecutive list entries, so the list walks
    // compact super-tiles of ~9 tile rows x ~8 tile-pair columns: the wave then shares
    // 9 + 8 operand panels instead of 2 + 37 and its working set fits the 126 MB L2.
    const int32_t rows_blk = std::min<int32_t>(9, t1 - t0 + 1);
    const int32_t cols_blk = std::max<int32_t>(1, 74 / rows_blk);  // in tile pairs
    for (int32_t tb = t0; tb <= t1; tb += rows_blk) {
      const int32_t te = std::min(t1, tb + rows_blk - 1);
      const int32_t tp_end = rect ? (col_tiles + 1) / 2 : te / 2 + 1;  // tile pairs of the super-tile row
      for (int32_t pb = 0; pb < tp_end; pb += cols_blk)
        for (int32_t tp = pb; tp < pb + cols_blk && tp < tp_end; ++tp)
          for (int32_t ti = rect ? tb : std::max(2 * tp, tb); ti <= te; ++ti) tiles.push_back({ti, 2 * tp});
    }
  } else {
    // column-major inside the band: CTAs running together share the few i-tiles of the band and
    // neighbouring j-tiles (L2 reuse of both operands)
    for (int32_t tj = 0; tj < (rect ? col_tiles : t1 + 1); ++tj)
      for (int32_t ti = rect ? t0 : std::max(tj, t0); ti <= t1; ++ti) tiles.push_back({ti, tj});
  }
  b.n_tiles = static_cast<int32_t>(tiles.size()) - b.tile_off;
}

std::vector<uint8_t> operand_need_blocks(const std::vector<Tile>& tiles, int64_t np, bool pair_tiles) {
  std::vector<uint8_t> need(static_cast<size_t>((np + 255) / 256), 0);
  const int32_t pairw = pair_tiles ? 2 : 1;
  for (const Tile& t : tiles) {
    need[t.ti / 2] |= 2;
    for (int32_t c = 0; c < pairw; ++c)
      if ((static_cast<int64_t>(t.tj) + c) * kTile < np) need[(t.tj + c) / 2] |= 1;
  }
  return need;
}

bool check_preorder(const int32_t* parent, int32_t B, int32_t* depth, int32_t* bad_parent, int32_t* bad_order) {
  *bad_parent = 0; *bad_order = 0;
  // Branch-free per node (the stack-popping form cost 14 ns per node in mispredictions).
  std::vector<int32_t> on_path(B + 1, 0);  // on_path[d] = node at depth d of the current path
  depth[0] = 0;
  for (int32_t v = 1; v < B; ++v) {
    const int32_t p = parent[v];
    if (p < 0 || p >= v) { *bad_parent = v; return false; }
    const int32_t d = depth[p];
    if ((d > depth[v - 1] || on_path[d] != p) && !*bad_order) *bad_order = v;
    depth[v] = d + 1;
    on_path[d + 1] = v;
  }
  return !*bad_order;
}

TreeLevels tree_levels(const int32_t* parent, int32_t B, int32_t* lvl, int32_t* lpar) {
  TreeLevels out;
  std::vector<int32_t> depth(B, 0), height(B, 0);
  if (!check_preorder(parent, B, depth.data(), &out.bad_parent, &out.bad_order)) return out;
  for (int32_t v = B - 1; v >= 1; --v) height[parent[v]] = std::max(height[parent[v]], height[v] + 1);
  const int32_t H = height[0];
  out.level_ptr.assign(H + 2, 0);
  for (int32_t v = 0; v < B; ++v) out.level_ptr[height[v] + 1]++;
  for (int32_t h = 0; h <= H; ++h) out.level_ptr[h + 1] += out.level_ptr[h];
  std::vector<int32_t>& lfill = depth;  // reused: next free slot of every level
  for (int32_t h = 0; h <= H; ++h) lfill[h] = out.level_ptr[h];
  for (int32_t v = 0; v < B; ++v) lvl[lfill[height[v]]++] = v;
  for (int32_t k = 0; k < B; ++k) lpar[k] = lvl[k] ? parent[lvl[k]] : 0;
  out.height = H;
  return out;
}

bool tree_children(const int32_t* parent, int32_t B, int32_t* cptr, int32_t* cidx) {
  std::vector<int32_t> child_cnt(B, 0);
  for (int32_t v = 1; v < B; ++v) {
    const int32_t p = parent[v];
    if (p < 0 || p >= v) return false;  // (reported by tree_levels)
    child_cnt[p]++;
  }
  cptr[0] = 0;
  for (int32_t v = 0; v < B; ++v) cptr[v + 1] = cptr[v] + child_cnt[v];
  std::vector<int32_t>& fill = child_cnt;  // reused: next free slot of every node's child list
  for (int32_t v = 0; v < B; ++v) fill[v] = cptr[v];
  for (int32_t v = 1; v < B; ++v) cidx[fill[parent[v]]++] = v;  // ascending id = file order
  return true;
}

void tree_post_order(const int32_t* parent, int32_t B, int32_t* post_order) {
  // pre-order ids: the subtree of v is [v, v + size[v]); everything in it except v, and nothing
  // of v's ancestors, is emitted before v: position = v + size[v] - 1 - depth[v]
  std::vector<int32_t> size(B, 1), depth(B, 0);
  for (int32_t v = B - 1; v >= 1; --v) size[parent[v]] += size[v];
  for (int32_t v = 1; v < B; ++v) depth[v] = depth[parent[v]] + 1;
  for (int32_t v = 0; v < B; ++v) post_order[v + size[v] - 1 - depth[v]] = v;
}

PrunedTree prune_tree(const int32_t* parent, const double* length, int32_t B, const uint8_t* marks, bool merge) {
  // keep: 0 = outside the support, 1 = survives, 2 = in the support but merged into the chain below it
  std::vector<uint8_t> keep(B);
  std::vector<int32_t> kids(B, 0);  // surviving children
  for (int32_t v = 0; v < B; ++v) keep[v] = marks[v] ? 1 : 0;
  if (B > 0) keep[0] = 1;
  for (int32_t v = B - 1; v >= 1; --v)
    if (keep[v]) { keep[parent[v]] = 1; kids[parent[v]]++; }
  if (merge)
    for (int32_t v = 1; v < B; ++v)
      if (keep[v] && kids[v] == 1) keep[v] = 2;
  // pre-order: a merged node's chain state (lengths summed from its top, node count, the survivor above the chain)
  // is complete before its child is visited
  PrunedTree t;
  t.new_of_old.assign(B, -1);
  std::vector<double> acc(merge ? B : 0);
  std::vector<int32_t> cnt(merge ? B : 0), up(merge ? B : 0);
  for (int32_t v = 0; v < B; ++v) {
    if (!keep[v]) continue;
    const int32_t p = v ? parent[v] : -1;
    const bool chain = p >= 0 && keep[p] == 2;
    if (keep[v] == 2) {
      acc[v] = chain ? acc[p] + length[v] : length[v];
      cnt[v] = (chain ? cnt[p] : 0) + 1;
      up[v] = chain ? up[p] : p;
      continue;
    }
    t.new_of_old[v] = t.n_nodes++;
    t.parent.push_back(p < 0 ? -1 : t.new_of_old[chain ? up[p] : p]);
    t.length.push_back(chain ? acc[p] + length[v] : length[v]);  // (verbatim unless merged)
    t.mult.push_back((chain ? cnt[p] : 0) + 1);
  }
  return t;
}

std::string StagedTable::row_name(int64_t s) const {
  if (!query) return "sample #" + std::to_string(s + 1);
  return s < q0 ? "reference sample #" + std::to_string(s + 1) : "query sample #" + std::to_string(s - q0 + 1);
}

void StagedTable::fill_row_ptr(int64_t* rp) const {
  const int64_t n_a = ref->n_samples;
  if (n_a > 0) memcpy(rp, ref->row_ptr, sizeof(int64_t) * (n_a + 1)); else rp[0] = 0;
  if (!query) return;
  const int64_t nnz_a = rp[n_a];
  for (int64_t s = n_a + 1; s <= q0; ++s) rp[s] = nnz_a;
  for (int64_t s = 1; s <= query->n_samples; ++s) rp[q0 + s] = nnz_a + query->row_ptr[s];
}

std::string stage_entries(const StagedTable& t, const int64_t* rp, int64_t s0, int64_t s1, const int32_t* parent,
                          int32_t B, const int32_t* new_of_old, int64_t* stamp, int64_t stamp_tag, int32_t* dcol,
                          double* dval) {
  // a leaf listed twice in a row only matters when values are used (presence is an OR)
  const bool check_dup = dval != nullptr;
  std::string err;
  for (int64_t s = s0; s < s1 && err.empty(); ++s) {
    const int64_t b = rp[s], e = rp[s + 1];
    if (b == e) continue;
    const int64_t mark_s = stamp_tag + s;
    const int32_t* scol = t.col(s);
    const double* sval = t.val(s);
    for (int64_t k = b; k < e; ++k) {
      const int32_t cc = scol[k - b];
      const double v = sval[k - b];
      const char* what = nullptr;
      if (cc < 0 || cc >= B) what = "node id out of range";
      // pre-order ids: the first child of a node is the next id (in frc_create the numbering itself is being
      // checked by another task at this moment; a bad tree fails the call before this result counts)
      else if (cc + 1 < B && parent[cc + 1] == cc) what = "node is not a leaf";
      else if (!(v > 0) || std::isinf(v)) what = "bad value";
      else if (check_dup && stamp[cc] == mark_s) what = "leaf listed twice";
      if (what) {
        err = t.row_name(s) + ": entry " + std::to_string(k - b + 1) + " (node " + std::to_string(cc) + "): " + what;
        break;
      }
      if (check_dup) stamp[cc] = mark_s;
      const int32_t id = new_of_old ? new_of_old[cc] : cc;
#if defined(__x86_64__)
      // streaming stores: the staging buffer is read next by the DMA engines, not by a core
      _mm_stream_si32(dcol + k, id);
      if (dval) _mm_stream_si64(reinterpret_cast<long long*>(dval + k), static_cast<long long>(__builtin_bit_cast(int64_t, v)));
#else
      dcol[k] = id;
      if (dval) dval[k] = v;
#endif
    }
  }
#if defined(__x86_64__)
  _mm_sfence();
#endif
  return err;
}

std::pair<int64_t, int64_t> chunk_rows(const int64_t* rp, int64_t N, int64_t k0, int64_t k1, int ch, int n_chunks) {
  auto row_at = [&](int64_t target) { return static_cast<int64_t>(std::lower_bound(rp, rp + N, target) - rp); };
  const int64_t span = k1 - k0;
  return {row_at(k0 + span * ch / n_chunks), row_at(k0 + span * (ch + 1) / n_chunks)};
}

const std::string& first_error(const std::vector<std::string>& chunk_errors) {
  static const std::string none;
  for (const std::string& e : chunk_errors)
    if (!e.empty()) return e;
  return none;
}

void mark_table_leaves(const StagedTable& t, int64_t k0, int64_t k1, int32_t B, uint8_t* marks) {
  auto mark = [&](const int32_t* col, int64_t a, int64_t b) {
    for (int64_t k = a; k < b; ++k) {
      const int32_t cc = col[k];
      // (read first: storing into lines that are already marked would bounce them between the cores)
      if (cc >= 0 && cc < B && !__atomic_load_n(&marks[cc], __ATOMIC_RELAXED))
        __atomic_store_n(&marks[cc], uint8_t{1}, __ATOMIC_RELAXED);
    }
  };
  const int64_t nnz_a = t.ref_nnz();
  if (k0 < nnz_a) mark(t.ref->col, k0, std::min(k1, nnz_a));
  if (t.query && k1 > nnz_a) mark(t.query->col, std::max(k0, nnz_a) - nnz_a, k1 - nnz_a);
}

}  // namespace frc

// ---------------------------------------------------------------- CPU test entry points
// Not part of the C ABI (include/frcfrc_cuda.h): they let tests/test_plan.py, test_prune.py and test_stage.py
// exercise the planning and staging units on the CPU-only box.
static int64_t write_bands(const std::vector<frc::Band>& bands, int64_t* out5, int64_t cap) {
  for (size_t k = 0; k < bands.size() && static_cast<int64_t>(k) < cap; ++k) {
    out5[5 * k] = bands[k].row0; out5[5 * k + 1] = bands[k].row1; out5[5 * k + 2] = bands[k].first;
    out5[5 * k + 3] = bands[k].count; out5[5 * k + 4] = bands[k].owner;
  }
  return static_cast<int64_t>(bands.size());
}

extern "C" {

// Bands of the whole triangle: writes up to `cap` (row0, row1, first, count, owner) quintuples; returns the count.
int64_t frc_debug_bands(int64_t n_samples, int64_t band_rows, int32_t world, int32_t d2h, int32_t per_rank,
                        int32_t value_bytes, int64_t* out5, int64_t cap) {
  return write_bands(frc::make_bands(n_samples, band_rows, world, d2h != 0, per_rank, value_bytes), out5, cap);
}

// Sample shards (plan_shards; mode 0 whole, 1 sharded, 2 capacity): info = {np, n_shards, shard_rows}, (owner, slot)
// per shard into out2 (cap_shards of them), (owner, s0, s1, slot) per range of every owner in turn into out4 (cap of
// them).  Returns the number of ranges (negative: a cap was too small).
int64_t frc_debug_shards(int64_t n_samples, int32_t owners, int32_t mode, int64_t* info, int32_t* out2, int64_t cap_shards,
                         int64_t* out4, int64_t cap) {
  const frc::ShardPlan sp = frc::plan_shards(n_samples, owners, static_cast<frc::ShardPlan::Mode>(mode));
  info[0] = sp.np; info[1] = sp.n_shards; info[2] = sp.shard_rows;
  if (sp.n_shards > cap_shards) return -1;
  for (int s = 0; s < sp.n_shards; ++s) { out2[2 * s] = sp.owner[s]; out2[2 * s + 1] = sp.slot[s]; }
  int64_t k = 0;
  for (size_t r = 0; r < sp.ranges.size(); ++r)
    for (const frc::Range& rg : sp.ranges[r]) {
      if (k == cap) return -1;
      out4[4 * k] = static_cast<int64_t>(r); out4[4 * k + 1] = rg.s0; out4[4 * k + 2] = rg.s1; out4[4 * k + 3] = rg.slot;
      ++k;
    }
  return k;
}

// Capacity-mode bands (the capacity shards of n_dev devices): same output layout as frc_debug_bands (-1: np is not theirs).
int64_t frc_debug_bands_capacity(int64_t n_samples, int64_t np, int32_t n_dev, int64_t band_rows, int32_t d2h,
                                 int64_t* out5, int64_t cap) {
  const frc::ShardPlan sp = frc::plan_shards(n_samples, n_dev, frc::ShardPlan::kCapacity);
  if (sp.np != np) return -1;
  return write_bands(frc::make_bands_capacity(n_samples, sp, band_rows, d2h != 0), out5, cap);
}

// Capacity-mode groups of device `dev`: out_groups holds (shard, first, count, tile_off) quadruples, out_coff
// (n_shards + 1) offsets per group, out_tiles (ti, tj) pairs; returns the number of groups, *n_tiles the tile count
// (negative: a cap was too small, or np is not the plan's padded sample count).
int64_t frc_debug_capacity_groups(int64_t n_samples, int64_t np, int32_t n_dev, int32_t dev, int64_t band_rows, int32_t d2h,
                                  int64_t* out_groups, int32_t* out_coff, int64_t cap_groups, int32_t* out_tiles,
                                  int64_t cap_tiles, int64_t* n_tiles) {
  const frc::ShardPlan sp = frc::plan_shards(n_samples, n_dev, frc::ShardPlan::kCapacity);
  if (sp.np != np) return -1;
  const std::vector<frc::Band> all = frc::make_bands_capacity(n_samples, sp, band_rows, d2h != 0);
  std::vector<frc::Band> mine;
  for (const frc::Band& b : all)
    if (b.owner == dev) mine.push_back(b);
  std::vector<frc::Tile> tiles;
  std::vector<int> band_group;
  const std::vector<frc::CapGroupPlan> g = frc::plan_capacity_groups(mine, n_samples, sp.shard_rows, sp.n_shards, tiles, band_group);
  *n_tiles = static_cast<int64_t>(tiles.size());
  if (static_cast<int64_t>(g.size()) > cap_groups || static_cast<int64_t>(tiles.size()) > cap_tiles) return -1;
  for (size_t k = 0; k < g.size(); ++k) {
    out_groups[4 * k] = g[k].shard; out_groups[4 * k + 1] = g[k].first; out_groups[4 * k + 2] = g[k].count; out_groups[4 * k + 3] = g[k].tile_off;
    for (int c = 0; c <= sp.n_shards; ++c) out_coff[k * (sp.n_shards + 1) + c] = g[k].coff[c];
  }
  for (size_t k = 0; k < tiles.size(); ++k) { out_tiles[2 * k] = tiles[k].ti; out_tiles[2 * k + 1] = tiles[k].tj; }
  return static_cast<int64_t>(g.size());
}

// Bands of the query x reference block (frc_create_cross; q0 = n_ref rounded up to 256): same output layout as
// frc_debug_bands, rows in the staged table (the query rows start at q0).
int64_t frc_debug_cross_bands(int64_t n_ref, int64_t n_q, int64_t band_rows, int32_t world, int32_t d2h, int32_t per_rank,
                              int32_t value_bytes, int64_t* out5, int64_t cap) {
  return write_bands(frc::make_bands_cross(frc::round_up(n_ref, 2 * frc::kTile), n_q, n_ref, band_rows, world, d2h != 0,
                                           per_rank, value_bytes), out5, cap);
}

// Tiles of the cross band [row0, row1) (staged rows) against n_ref reference samples: as frc_debug_band_tiles.
int64_t frc_debug_cross_tiles(int64_t row0, int64_t row1, int64_t n_ref, int32_t pair_tiles, int32_t* out2, int64_t cap) {
  frc::Band b;
  b.row0 = row0; b.row1 = row1;
  std::vector<frc::Tile> tiles;
  frc::append_band_tiles(b, pair_tiles != 0, tiles, static_cast<int32_t>((n_ref + frc::kTile - 1) / frc::kTile));
  for (size_t k = 0; k < tiles.size() && static_cast<int64_t>(k) < cap; ++k) { out2[2 * k] = tiles[k].ti; out2[2 * k + 1] = tiles[k].tj; }
  return static_cast<int64_t>(tiles.size());
}

// Tiles of the band [row0, row1): writes up to `cap` (ti, tj) pairs; returns the count.
int64_t frc_debug_band_tiles(int64_t row0, int64_t row1, int32_t pair_tiles, int32_t* out2, int64_t cap) {
  frc::Band b;
  b.row0 = row0; b.row1 = row1;
  std::vector<frc::Tile> tiles;
  frc::append_band_tiles(b, pair_tiles != 0, tiles);
  for (size_t k = 0; k < tiles.size() && static_cast<int64_t>(k) < cap; ++k) { out2[2 * k] = tiles[k].ti; out2[2 * k + 1] = tiles[k].tj; }
  return static_cast<int64_t>(tiles.size());
}

// Column plan of the fast unweighted path.  col_order / col_exp / len_col hold `cap` entries; chunk arrays 64.
// Returns kp (negative: cap too small); *info = {i8, intacc, biased, e_min, n_chunks}.
int32_t frc_debug_plan_columns(const double* length, int32_t n_nodes, int32_t want_i8, int32_t group_binades,
                               int32_t force_f64, int32_t* col_order, int32_t* col_exp, double* len_col, int32_t cap,
                               int32_t* chunk_end, double* chunk_scale, int32_t* chunk_shift, int32_t* info) {
  const frc::ColumnPlan p = frc::plan_columns(length, n_nodes, want_i8 != 0, group_binades, force_f64 != 0, 64);
  if (p.kp > cap || p.chunk_end.size() > 64) return -p.kp;
  for (int32_t k = 0; k < p.kp; ++k) {
    col_order[k] = p.col_order[k];
    col_exp[k] = p.col_exp.empty() ? 0 : p.col_exp[k];
    len_col[k] = p.len_col[k];
  }
  for (size_t c = 0; c < p.chunk_end.size(); ++c) {
    chunk_end[c] = p.chunk_end[c];
    chunk_scale[c] = p.chunk_scale[c];
    chunk_shift[c] = p.chunk_shift.empty() ? 0 : p.chunk_shift[c];
  }
  info[0] = p.i8; info[1] = p.intacc; info[2] = p.biased; info[3] = p.e_min; info[4] = static_cast<int32_t>(p.chunk_end.size());
  return p.kp;
}

// Tree walk: level_nodes / level_parent / child_idx / post_order hold n_nodes entries, child_ptr n_nodes + 1,
// level_ptr n_nodes + 2.  Returns the height, or -1 - (offending node) for a bad parent / non-pre-order id.
int32_t frc_debug_tree(const int32_t* parent, int32_t n_nodes, int32_t* level_nodes, int32_t* level_parent,
                       int32_t* level_ptr, int32_t* child_ptr, int32_t* child_idx, int32_t* post_order) {
  const frc::TreeLevels t = frc::tree_levels(parent, n_nodes, level_nodes, level_parent);
  if (t.bad_parent) return -1 - t.bad_parent;
  if (t.bad_order) return -1 - t.bad_order;
  for (size_t k = 0; k < t.level_ptr.size(); ++k) level_ptr[k] = t.level_ptr[k];
  if (!frc::tree_children(parent, n_nodes, child_ptr, child_idx)) return -1;
  frc::tree_post_order(parent, n_nodes, post_order);
  return t.height;
}

// Pruned tree (prune_tree; marks[n_nodes] = 1 on the listed leaves): out_parent / out_length / out_mult hold n_nodes
// entries (the pruned tree is never larger), new_of_old n_nodes.  Returns the pruned node count, or -1 - (offending
// node) when parent[] is not a pre-order numbering (frc_create then prunes nothing).
int32_t frc_debug_prune(const int32_t* parent, const double* length, int32_t n_nodes, const uint8_t* marks, int32_t merge,
                        int32_t* out_parent, double* out_length, int32_t* out_mult, int32_t* new_of_old) {
  std::vector<int32_t> depth(n_nodes);
  int32_t bad_parent = 0, bad_order = 0;
  if (!frc::check_preorder(parent, n_nodes, depth.data(), &bad_parent, &bad_order)) return -1 - (bad_parent ? bad_parent : bad_order);
  const frc::PrunedTree t = frc::prune_tree(parent, length, n_nodes, marks, merge != 0);
  for (int32_t v = 0; v < t.n_nodes; ++v) { out_parent[v] = t.parent[v]; out_length[v] = t.length[v]; out_mult[v] = t.mult[v]; }
  for (int32_t v = 0; v < n_nodes; ++v) new_of_old[v] = t.new_of_old[v];
  return t.n_nodes;
}

// Table staging as frc_create does it: the table (n_q < 0) or the reference + query pair of frc_create_cross
// (q0 = n_ref rounded up to 256), checked against parent[n_nodes], its entries cut into n_chunks chunks.  out_rp holds
// the staged rows + 1 entries, out_col / out_val (null: presence only) the entries; new_of_old may be null, stamp
// [n_nodes] is needed with out_val.  Writes the reported message (NUL-terminated, cut to msg_cap) into msg; returns the
// staged row count.  PRUNE marks of the same entries go to marks[n_nodes] unless it is null.
int64_t frc_debug_stage(const int32_t* parent, int32_t n_nodes, int64_t n_ref, const int64_t* ref_rp,
                        const int32_t* ref_col, const double* ref_val, int64_t n_q, const int64_t* q_rp,
                        const int32_t* q_col, const double* q_val, const int32_t* new_of_old, int32_t n_chunks,
                        int64_t* stamp, int64_t stamp_tag, int64_t* out_rp, int32_t* out_col, double* out_val,
                        uint8_t* marks, char* msg, int64_t msg_cap) {
  const frc_csr_t ref{n_ref, ref_rp, ref_col, ref_val}, query{n_q, q_rp, q_col, q_val};
  frc::StagedTable t{&ref, n_q >= 0 ? &query : nullptr, 0};
  int64_t N = n_ref;
  if (t.query) {
    t.q0 = frc::round_up(n_ref, 2 * frc::kTile);
    N = t.q0 + n_q;
  }
  t.fill_row_ptr(out_rp);
  const int64_t nnz = out_rp[N];
  if (marks) frc::mark_table_leaves(t, 0, nnz, n_nodes, marks);
  std::vector<std::string> errs(n_chunks);
  for (int ch = n_chunks - 1; ch >= 0; --ch) {  // (backwards: the report must not depend on which chunk ends first)
    const std::pair<int64_t, int64_t> rows = frc::chunk_rows(out_rp, N, 0, nnz, ch, n_chunks);
    errs[ch] = frc::stage_entries(t, out_rp, rows.first, rows.second, parent, n_nodes, new_of_old, stamp, stamp_tag,
                                  out_col, out_val);
  }
  const std::string& e = frc::first_error(errs);
  snprintf(msg, static_cast<size_t>(msg_cap), "%s", e.c_str());
  return N;
}

// Rows [out2[0], out2[1]) of the staged table whose entries `owner` reads (rows_read).
void frc_debug_rows_read(int64_t n_samples, int32_t owners, int32_t owner, int32_t sharded_fast_uw, int64_t* out2) {
  const std::pair<int64_t, int64_t> r = frc::rows_read(n_samples, owners, owner, sharded_fast_uw != 0);
  out2[0] = r.first; out2[1] = r.second;
}

// The variant frc_create plans (plan_exchange, then plan_variant), with the knobs read from the environment and
// free_hbm as device 0's free HBM (negative: the query fails).  out16 = {exchange, fused_embed, sharded_fast_uw,
// capacity, shard_mode, want_i8, bits_feed, rowsum_in_expand, rowsum_split, peer_store, peer_push, need_blocks,
// operand_kind, columns' intacc, columns' kp, free-HBM queries}.  Returns the error code and writes its message
// (NUL-terminated, cut to msg_cap) into msg.
int32_t frc_debug_plan_variant(int32_t weighted, int32_t exact, int32_t keyed, int32_t rect, uint32_t flags, int32_t world,
                               int32_t rank, int64_t n_samples, const double* length, int32_t n_nodes, int32_t n_parts,
                               int32_t peer_ok, int32_t comm_world, int32_t comm_rank, int32_t neg_len, int64_t free_hbm,
                               int64_t* out16, char* msg, int64_t msg_cap) {
  frc::VariantIn in;
  in.exact = exact != 0; in.weighted = weighted != 0; in.keyed = keyed != 0; in.rect = rect != 0;
  in.flags = flags; in.world = world; in.rank = rank; in.N = n_samples;
  in.n_parts = n_parts; in.peer_ok = peer_ok != 0; in.comm_world = comm_world; in.comm_rank = comm_rank;
  const frc::Knobs k = frc::Knobs::read();
  int64_t asked = 0;
  auto query = [&](size_t* bytes) {
    ++asked;
    *bytes = free_hbm < 0 ? 0 : static_cast<size_t>(free_hbm);
    return free_hbm >= 0;
  };
  frc::Variant v = frc::plan_exchange(in, k);
  frc::ColumnPlan cols;
  std::string err;
  const int rc = frc::plan_variant(v, in, k, neg_len != 0, length, n_nodes, 64, query, &cols, &err);
  const int64_t f[16] = {v.exchange, v.fused_embed, v.sharded_fast_uw, v.capacity, v.shard_mode, v.want_i8, v.bits_feed,
                         v.rowsum_in_expand, v.rowsum_split, v.peer_store, v.peer_push, v.need_blocks, v.operand_kind,
                         cols.intacc, cols.kp, asked};
  memcpy(out16, f, sizeof(f));
  snprintf(msg, static_cast<size_t>(msg_cap), "%s", err.c_str());
  return rc;
}

}  // extern "C"
