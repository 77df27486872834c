// Weighted UniFrac pair tiles on the FP32 CUDA cores (replaces
// unifracDistWeighted, frcfrc/unifrac.go:174-205, for 128 x 128 sample pairs
// per CTA).
//
//   d(i,j) = sum_k len_k |a_ik - a_jk|  /  sum_k len_k (a_ik + a_jk)
//
// The denominator is separable (W_i + W_j, computed once per sample in fp64 by
// the embedding stage), so the pair kernel only accumulates the numerator: an
// L1 distance between two sample columns of the operand, stored as tile panels Ap[np/128][kp][128].  With
// non-negative branch lengths the operand is pre-scaled (A = len * a), so the
// inner loop is exactly two FP32 instructions per (pair, node): FADD d = a - b,
// FADD acc = acc + |d| (|.| is a free source modifier).  Negative lengths use
// the FFMA form with len staged next to the tile.
//
// Tiling: CTA = 128 x 128 pairs, 256 threads, each an 8 x 8 register block
// (two 4-wide groups per side, so every shared-memory read is a conflict-free
// LDS.128).  The contraction is staged through shared memory in slabs of 32 nodes (16 keyed)
// with a 3-deep ring of TMA bulk copies (one copy per operand slab).  Accumulation is two-level: fp32 running
// sums over 256 nodes, flushed into fp64 per-pair totals that live in shared memory (128 KB per CTA:
// they would not fit the registers beside the running sums).  Only the 256-term fp32 level rounds the way a
// regular input (equal lengths and counts) drives every rounding in one direction: at most 4e-6 relative
// for constant terms, against the 1e-5 budget, whatever the number of nodes (tests/test_weighted_accuracy.py
// models this arithmetic).  An fp32 total grew that error with every flush (1.45e-5 at 2^18 nodes).
//
// Keyed variant (normalize = 0, flag -l as the reference codes it, FRC_FLAG_L_TILES).  Without the id-sort the
// reference's merge-join walks post-order lists and pairs nodes up by accident; the outcome has a closed form
// (DESIGN.md, "-l as coded"): with key_s(v) = the largest present leaf id under v (-1 when v is absent),
//   numer = sum_v len_v * (key_i(v) == key_j(v) ? |a - b| : a + b),   denom = W_i + W_j.
// Since a, b >= 0, both branches are |a - (match ? b : -b)|: the kernel sums that term directly -- ISETP + FSEL
// + FADD + FADD, 4 instructions per (pair, node) against the 2 of the L1 loop -- so the numerator never comes from
// a cancellation (W_i + W_j - 2 * sum of the matched min(a, b) multiplied the error of the sum by (1 - d) / d,
// about 30 just above the fix-up threshold).  The int32 key panels K[np/128][kp][128] ride in the same TMA ring as
// the values; a keyed slab is 16 nodes so that its stage (32 KB) leaves room for the fp64 totals.
#include <type_traits>

#include "frc_internal.h"
#include "ptx.cuh"
#include "wire.cuh"

namespace frc {
namespace {

constexpr int kFlushNodes = 256;  // nodes per fp32 running sum, between two flushes into the fp64 totals
template <bool kKeyed> constexpr int kKT = kKeyed ? 16 : 32;       // nodes per smem slab
template <bool kKeyed> constexpr int kSlabFloats = kKT<kKeyed> * kTile;
// ring depth: 2 slabs in flight cover the HBM latency (every panel the kernel reads is in local HBM: the
// capacity mode rotates the remote shards in with the copy engines)
constexpr int kStages = 3;
// per stage: the two value slabs, per-node lengths, keyed: the two key slabs
template <bool kKeyed> constexpr int kStageFloats = (kKeyed ? 4 : 2) * kSlabFloats<kKeyed> + kKT<kKeyed>;
constexpr int kTotBytes = 64 * 256 * 8;  // fp64 totals: 64 pairs per thread
template <bool kKeyed> constexpr int kSmemBytes = kTotBytes + kStages * kStageFloats<kKeyed> * 4 + kStages * 8 + 128;
static_assert(kSmemBytes<false> <= 227 * 1024 && kSmemBytes<true> <= 227 * 1024, "shared memory per CTA");

// Panel of sample tile t (PanelMap in frc_internal.h): the one local array, or the place its shard currently
// occupies in this device's HBM.
__device__ __forceinline__ const float* panel_of(const PanelMap& m, int32_t t, int32_t kp) {
  if (m.n_shards == 0) return m.shard[0] + static_cast<int64_t>(t) * kp * kTile;
  const int32_t s = t / m.tiles_per_shard, r = t - s * m.tiles_per_shard;
  return m.shard[s] + static_cast<int64_t>(r) * kp * kTile;
}

// Operand staging: one thread issues TMA bulk copies (cp.async.bulk, 16 KB per operand slab: the tile-panel
// layout makes a slab of 32 nodes x 128 samples contiguous) that complete on an mbarrier per stage.  The
// FP32-issue-bound inner loop spends no slot on copies and the copy engine keeps the whole ring in flight.
template <bool kPrescaled, bool kKeyed, bool kRect>
__global__ void __launch_bounds__(256, 1)
k_weighted_tiles(const PanelMap A, int64_t ld, int32_t kp, const float* __restrict__ lenf,
                 const double* __restrict__ W, const Tile* __restrict__ tiles, int64_t n_samples,
                 int64_t first, float* __restrict__ out, double flag_below, uint32_t* __restrict__ flagged,
                 unsigned long long* __restrict__ n_flagged, const int32_t* __restrict__ K, const Geometry geo) {
  constexpr int STAGES = kStages;
  constexpr int STAGE_FLOATS = kStageFloats<kKeyed>;
  constexpr int KT = kKT<kKeyed>;
  constexpr int SLAB_FLOATS = kSlabFloats<kKeyed>;
  constexpr int FLUSH = kFlushNodes / KT;  // slabs between flushes
  extern __shared__ __align__(128) float smem[];
  // the fp64 totals of this thread's 64 pairs: tot[e * 256 + tid] (a warp's loads and stores are contiguous),
  // then the ring
  double* const tot = reinterpret_cast<double*>(smem);
  float* const ring = smem + kTotBytes / 4;
  const Tile tile = tiles[blockIdx.x];
  const int64_t i0 = static_cast<int64_t>(tile.ti) * kTile;
  const int64_t j0 = static_cast<int64_t>(tile.tj) * kTile;
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int n_slabs = kp / KT;
  const uint32_t bar0 = ptx::smem_u32(ring + STAGES * STAGE_FLOATS);
  (void)ld;

  // tile-panel layout [kp][128] per sample tile
  const float* const pa = panel_of(A, tile.ti, kp);  // row samples: this device's own shard
  const float* const pb = panel_of(A, tile.tj, kp);  // column samples: own shard or the visiting one
  // keyed: the key panels of the same tiles (resident only: global tile index)
  const int32_t* const ka_g = kKeyed ? K + static_cast<int64_t>(tile.ti) * kp * kTile : nullptr;
  const int32_t* const kb_g = kKeyed ? K + static_cast<int64_t>(tile.tj) * kp * kTile : nullptr;
  auto issue = [&](int slab) {  // thread 0 only
    const int stage = slab % STAGES;
    float* sa = ring + stage * STAGE_FLOATS;
    const uint32_t bar = bar0 + 8u * stage;
    constexpr uint32_t kSlabBytes = SLAB_FLOATS * 4;
    ptx::mbar_expect_tx(bar, (kKeyed ? 4 : 2) * kSlabBytes + (kPrescaled ? 0u : KT * 4u));
    ptx::bulk_load_1d(ptx::smem_u32(sa), pa + static_cast<int64_t>(slab) * SLAB_FLOATS, kSlabBytes, bar);
    ptx::bulk_load_1d(ptx::smem_u32(sa + SLAB_FLOATS), pb + static_cast<int64_t>(slab) * SLAB_FLOATS, kSlabBytes, bar);
    if (!kPrescaled) ptx::bulk_load_1d(ptx::smem_u32(sa + 2 * SLAB_FLOATS), lenf + slab * KT, KT * 4u, bar);
    if (kKeyed) {
      float* sk = sa + 2 * SLAB_FLOATS + KT;
      ptx::bulk_load_1d(ptx::smem_u32(sk), ka_g + static_cast<int64_t>(slab) * SLAB_FLOATS, kSlabBytes, bar);
      ptx::bulk_load_1d(ptx::smem_u32(sk + SLAB_FLOATS), kb_g + static_cast<int64_t>(slab) * SLAB_FLOATS, kSlabBytes, bar);
    }
  };
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) ptx::mbar_init(bar0 + 8u * s, 1);
    ptx::fence_barrier_init();
  }
  __syncthreads();
  if (tid == 0)
    for (int p = 0; p < STAGES - 1 && p < n_slabs; ++p) issue(p);

  float acc[8][8];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) { acc[a][b] = 0.f; tot[(a * 8 + b) * 256 + tid] = 0.0; }

  for (int slab = 0; slab < n_slabs; ++slab) {
    // the stage that slab + STAGES - 1 goes to was read in the previous iteration (barrier at its end)
    if (tid == 0 && slab + STAGES - 1 < n_slabs) issue(slab + STAGES - 1);
    const int stage = slab % STAGES;
    ptx::mbar_wait(bar0 + 8u * stage, static_cast<uint32_t>((slab / STAGES) & 1));
    const float* sa = ring + stage * STAGE_FLOATS;
    const float* sb = sa + SLAB_FLOATS;
    const float* sl = sb + SLAB_FLOATS;
    const int32_t* ska = reinterpret_cast<const int32_t*>(sl + KT);
    const int32_t* skb = ska + SLAB_FLOATS;
#pragma unroll 4
    for (int kk = 0; kk < KT; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(sa + kk * kTile + ty * 4);
      const float4 a1 = *reinterpret_cast<const float4*>(sa + kk * kTile + 64 + ty * 4);
      const float4 b0 = *reinterpret_cast<const float4*>(sb + kk * kTile + tx * 4);
      const float4 b1 = *reinterpret_cast<const float4*>(sb + kk * kTile + 64 + tx * 4);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      if (kKeyed) {
        const int4 p0 = *reinterpret_cast<const int4*>(ska + kk * kTile + ty * 4);
        const int4 p1 = *reinterpret_cast<const int4*>(ska + kk * kTile + 64 + ty * 4);
        const int4 q0 = *reinterpret_cast<const int4*>(skb + kk * kTile + tx * 4);
        const int4 q1 = *reinterpret_cast<const int4*>(skb + kk * kTile + 64 + tx * 4);
        const int32_t ka[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
        const int32_t kb[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
        const float l = kPrescaled ? 1.f : sl[kk];
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = 0; b < 8; ++b) {
            // matched: |a - b|; otherwise a + b = |a - (-b)| (a, b >= 0)
            const float t = fabsf(av[a] - (ka[a] == kb[b] ? bv[b] : -bv[b]));
            if (kPrescaled) acc[a][b] += t;
            else acc[a][b] = fmaf(l, t, acc[a][b]);
          }
      } else if (kPrescaled) {
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = 0; b < 8; ++b) acc[a][b] += fabsf(av[a] - bv[b]);
      } else {
        const float l = sl[kk];
#pragma unroll
        for (int a = 0; a < 8; ++a)
#pragma unroll
          for (int b = 0; b < 8; ++b) acc[a][b] = fmaf(l, fabsf(av[a] - bv[b]), acc[a][b]);
      }
    }
    if ((slab % FLUSH) == FLUSH - 1) {
#pragma unroll
      for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) {
          tot[(a * 8 + b) * 256 + tid] += static_cast<double>(acc[a][b]);
          acc[a][b] = 0.f;
        }
    }
    __syncthreads();  // every thread is done with this stage: it may be refilled
  }

#pragma unroll
  for (int a = 0; a < 8; ++a) {
    const int64_t i = i0 + (a < 4 ? ty * 4 + a : 64 + ty * 4 + (a - 4));
    if (i >= n_samples) continue;
    const double wi = W[i];
    float* orow = kRect ? out + ((i - geo.q0) * geo.n_ref - first) : out + (i * (i - 1) / 2 - first);
#pragma unroll
    for (int b = 0; b < 8; ++b) {
      const int64_t j = j0 + (b < 4 ? tx * 4 + b : 64 + tx * 4 + (b - 4));
      if (kRect ? j < geo.n_ref : j < i) {
        const double num = tot[(a * 8 + b) * 256 + tid] + static_cast<double>(acc[a][b]);
        const double d = num / (wi + W[j]);
        orow[j] = static_cast<float>(d);  // fp32 numerator: fp32 is what the value carries (wire.cu)
        // fp32 operands carry 6e-8 relative error each, so the numerator (L1 or keyed) is off by up to
        // 6e-8 * (W_i + W_j) = 6e-8 / d relative: small distances are recomputed (k_weighted_fixup)
        if (d < flag_below) {
          unsigned long long slot = atomicAdd(n_flagged, 1ULL);
          flagged[slot] = static_cast<uint32_t>(orow + j - out);
        }
      }
    }
  }
}

// Recompute of the flagged pairs from the CSR rows themselves, one CTA per pair at a time:
//   diff[v] = a_i(v) - a_j(v) for every node on a leaf-to-root path of either sample, accumulated as
//   62-bit fixed point with integer atomics (order-independent: deterministic, and identical samples
//   cancel to exactly 0), then numerator = sum_v len_v * |diff[v]| in fp64 over the touched nodes (the
//   second walk takes each node's value with an atomic exchange, which also restores the zeros).
// ws is one zeroed int64 array of n_nodes entries per CTA.
// Keyed (-l as coded): a second array per CTA accumulates sum[v] = a_i(v) + a_j(v) the same way, and a touched
// node adds len * |diff| where the key panels say the two samples match at v, len * sum where they do not.
template <bool kKeyed, bool kRect>
__global__ void __launch_bounds__(256)
k_weighted_fixup(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                 const double* __restrict__ val, const int32_t* __restrict__ parent,
                 const double* __restrict__ length, int32_t n_nodes, const double* __restrict__ total,
                 const double* __restrict__ W, const uint32_t* __restrict__ flagged,
                 const unsigned long long* __restrict__ n_flagged, unsigned long long* __restrict__ count_host,
                 int64_t first, long long* __restrict__ ws, float* __restrict__ out, const Exceptions ex,
                 const int32_t* __restrict__ K, int32_t kp, const Geometry geo) {
  __shared__ double red[8];
  const unsigned long long n = *n_flagged;
  if (blockIdx.x == 0 && threadIdx.x == 0) *count_host = n;  // mapped pinned memory
  long long* diff = ws + static_cast<int64_t>(blockIdx.x) * n_nodes * (kKeyed ? 2 : 1);
  long long* sum = diff + n_nodes;  // (keyed only)
  constexpr double kFix = 1152921504606846976.0;  // 2^60: proportions are <= 1, a node sums <= 1
  for (unsigned long long w = blockIdx.x; w < n; w += gridDim.x) {
    const uint32_t off = flagged[w];
    int64_t i, j;
    pair_at<kRect>(first + off, geo, i, j);
    const int64_t smp[2] = {i, j};
    // without normalisation (-l) raw values are summed: scale them into the fixed-point range
    double inv[2];
#pragma unroll
    for (int side = 0; side < 2; ++side) {
      const double t = total ? total[smp[side]] : 0.0;
      inv[side] = total ? (t > 0.0 ? 1.0 / t : 0.0) : 0.0;
    }
    double unscale = 1.0 / kFix;
    if (!total) {  // common power-of-two scale from the two raw sums (exact)
      double big = 0.0;
      for (int side = 0; side < 2; ++side)
        for (int64_t k = row_ptr[smp[side]]; k < row_ptr[smp[side] + 1]; ++k) big += val[k];
      int e;
      frexp(big > 0.0 ? big : 1.0, &e);
      inv[0] = inv[1] = ldexp(1.0, -e);
      unscale = ldexp(1.0, e) / kFix;
    }
#pragma unroll
    for (int side = 0; side < 2; ++side) {
      const int64_t b = row_ptr[smp[side]], e = row_ptr[smp[side] + 1];
      for (int64_t k = b + threadIdx.x; k < e; k += blockDim.x) {
        const long long x = __double2ll_rn(val[k] * inv[side] * kFix);
        const long long add = side == 0 ? x : -x;
        for (int32_t v = col[k]; v >= 0; v = parent[v]) {
          atomicAdd(reinterpret_cast<unsigned long long*>(diff + v), static_cast<unsigned long long>(add));
          if (kKeyed) atomicAdd(reinterpret_cast<unsigned long long*>(sum + v), static_cast<unsigned long long>(x));
        }
      }
    }
    __syncthreads();
    const int32_t* const ki = kKeyed ? K + (i >> 7) * kp * 128 + (i & 127) : nullptr;
    const int32_t* const kj = kKeyed ? K + (j >> 7) * kp * 128 + (j & 127) : nullptr;
    double num = 0.0;
#pragma unroll
    for (int side = 0; side < 2; ++side) {
      const int64_t b = row_ptr[smp[side]], e = row_ptr[smp[side] + 1];
      for (int64_t k = b + threadIdx.x; k < e; k += blockDim.x)
        for (int32_t v = col[k]; v >= 0; v = parent[v]) {
          const long long x = static_cast<long long>(atomicExch(reinterpret_cast<unsigned long long*>(diff + v), 0ULL));
          if (kKeyed) {
            // (whichever thread takes a node's value adds its term: only one of the two arrays counts per node)
            const long long y = static_cast<long long>(atomicExch(reinterpret_cast<unsigned long long*>(sum + v), 0ULL));
            const long long t = ki[static_cast<int64_t>(v) * 128] == kj[static_cast<int64_t>(v) * 128] ? (x < 0 ? -x : x) : y;
            if (t != 0) num += length[v] * (static_cast<double>(t) * unscale);
          } else if (x != 0) {
            num += length[v] * (fabs(static_cast<double>(x)) * unscale);
          }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) num += __shfl_xor_sync(0xffffffffu, num, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = num;
    __syncthreads();
    if (threadIdx.x == 0) {
      double tot = 0.0;
      for (int k = 0; k < 8; ++k) tot += red[k];
      store_fixed(out, off, tot / (W[i] + W[j]), first, ex);
    }
    __syncthreads();
  }
}

}  // namespace

int launch_weighted_fixup(const DevCsr& a, const DevTree& t, const double* total, const double* W,
                          const uint32_t* flagged, const unsigned long long* n_flagged,
                          unsigned long long* count_host, int64_t first, const Geometry& geo, long long* ws,
                          int ws_ctas, float* out, const Exceptions& ex, cudaStream_t s, const int32_t* K, int32_t kp) {
  const auto kernel = K ? (geo.rect ? k_weighted_fixup<true, true> : k_weighted_fixup<true, false>)
                        : (geo.rect ? k_weighted_fixup<false, true> : k_weighted_fixup<false, false>);
  kernel<<<ws_ctas, 256, 0, s>>>(a.row_ptr, a.col, a.val, t.parent, t.length, t.n_nodes, total, W, flagged, n_flagged,
                                 count_host, first, ws, out, ex, K, K ? kp : 0, geo);
  return 1;
}

void weighted_setup() {
  auto smem = [](auto kernel, int bytes) { cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); };
  smem(k_weighted_tiles<true, false, false>, kSmemBytes<false>);
  smem(k_weighted_tiles<false, false, false>, kSmemBytes<false>);
  smem(k_weighted_tiles<true, true, false>, kSmemBytes<true>);
  smem(k_weighted_tiles<false, true, false>, kSmemBytes<true>);
  smem(k_weighted_tiles<true, false, true>, kSmemBytes<false>);
  smem(k_weighted_tiles<false, false, true>, kSmemBytes<false>);
  smem(k_weighted_tiles<true, true, true>, kSmemBytes<true>);
  smem(k_weighted_tiles<false, true, true>, kSmemBytes<true>);
}

int launch_weighted_tiles(const PanelMap& A, int64_t ld, int32_t kp, const float* lenf, bool prescaled,
                          const double* W, const Tile* tiles, int32_t n_tiles, int64_t n_samples,
                          int64_t first, const Geometry& geo, float* out, double flag_below, uint32_t* flagged,
                          unsigned long long* n_flagged, int num_sms, cudaStream_t s, const int32_t* K) {
  (void)num_sms;
  if (n_tiles <= 0) return 0;
  auto go = [&](auto kernel, int smem) {
    kernel<<<n_tiles, 256, smem, s>>>(A, ld, kp, lenf, W, tiles, n_samples, first, out, flag_below, flagged, n_flagged, K,
                                      geo);
  };
  // (the capacity mode, which shards the panels, only runs triangle jobs)
  auto pick = [&](auto prescaled_c, auto keyed_c) {
    constexpr bool kP = decltype(prescaled_c)::value, kK = decltype(keyed_c)::value;
    if (geo.rect) go(k_weighted_tiles<kP, kK, true>, kSmemBytes<kK>);
    else go(k_weighted_tiles<kP, kK, false>, kSmemBytes<kK>);
  };
  if (K) {
    if (prescaled) pick(std::true_type{}, std::true_type{});
    else pick(std::false_type{}, std::true_type{});
  } else {
    if (prescaled) pick(std::true_type{}, std::false_type{});
    else pick(std::false_type{}, std::false_type{});
  }
  return 1;
}

}  // namespace frc
