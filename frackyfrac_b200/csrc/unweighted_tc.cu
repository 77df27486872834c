// Unweighted UniFrac pair tiles on the tcgen05 tensor cores (replaces
// unifracDistUnweighted, frcfrc/unifrac.go:144-171, for 128 x 128 sample pairs
// per output tile).
//
// For presence P (0/1) and branch lengths len:
//     shared(i,j) = sum_k len_k P_ik P_jk          (the reference's `common`)
//     r_i         = sum_k len_k P_ik
//     unique(i,j) = r_i + r_j - 2 shared           (the reference's `result`)
//     d(i,j)      = unique / (unique + shared) = (R - 2s) / (R - s),  R = r_i + r_j
// so the pairwise part is the dense contraction S = P diag(len) P^T: a GEMM.
//
// Kernels in this file (DESIGN.md, "Pair stage, unweighted"), two operand feeds of one pair stage
// (TcOperands says which):
//   k_unweighted_tc2<2>  default.  CTA pairs (cta_group::2), u8 block-floating-point operands
//                        (len ~= a * m * 2^e), tcgen05 kind::i8 M256 x N256 x K32, exact int32
//                        accumulation in TMEM, 64-bit integer chunk accumulation and an integer / fp32
//                        ratio epilogue (no fp64 instruction).
//   k_unweighted_tc2<1>  the same operands with fp64 chunk accumulation, for trees whose chunk
//                        scales span more than 2^16.
//   k_unweighted_tc2<0>  bf16 operands (P exact, len = hi + lo planes), kind::f16 K16, fp32
//                        accumulators restarted every K-chunk (FRC_FLAG_UW_BF16; negative lengths).
//   k_unweighted_bits2   the integer mode of k_unweighted_tc2<2> with the u8 operand tiles expanded
//                        inside the kernel from the presence bits (capacity mode, FRC_FLAG_UW_BITS):
//                        no operand arrays in HBM.
//   k_unweighted_fixup   exact fp64 recompute of the pairs the epilogues flag, from either feed's rows.
//
// bf16: why two accumulator halves and K-chunks: the tensor core's fp32 accumulate
// loses the addend bits below the accumulator's ulp (measured: a bias, not
// noise).  hi-plane addends are 8-bit significands, so they add EXACTLY while the
// running sum stays within 2^16 of them; keeping the 2^-9-smaller lo plane out of
// that sum and restarting it every K-chunk keeps it so.  The chunk sums are then
// added in registers with round-to-nearest.  r is computed in fp64 from the SAME
// quantised lengths so that R - 2s cancels consistently, and pairs with a small
// distance (where the subtraction loses relative accuracy) go to k_unweighted_fixup.
// Two TMEM buffers (2 x 256 columns = all of TMEM) let the MMAs of chunk c+1
// overlap the drain of chunk c, and the next tile's mainloop this tile's epilogue.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include "frc_internal.h"
#include "ptx.cuh"
#include "wire.cuh"

namespace frc {

namespace {

constexpr int BM = 128, BN = 128, BK = 64, UK = 16;
constexpr int A_BYTES = BM * BK * 2;
constexpr int B_BYTES = BN * BK * 2;
constexpr int EPI_WARP0 = 2;                // warp 0: TMA producer, warp 1: MMA issuer
constexpr int DN = 2 * BN;                 // accumulator columns: [hi | lo]
constexpr uint32_t TMEM_COLS = 2 * DN;    // two buffers: all 512 columns

// ----------------------------------------------------------------------------
// CTA-pair variant (cta_group::2): two CTAs of a cluster (one TPC) compute two
// horizontally adjacent 128 x 128 tiles (ti, tj) and (ti, tj+1) with ONE MMA
// stream of shape M256 x N256 issued by the leader CTA.  The MMA's M side is the
// COLUMN sample of the output (S is symmetric, so the roles are free) because a TMEM
// lane is a thread of the epilogue and consecutive columns j are what is contiguous
// in the flat lower triangle: stores come out coalesced without any transpose
// (with rows on the lanes every store hit 32 different sectors and the epilogue,
// not the tensor pipe, bounded the kernel).
//   A (256 rows)  = each CTA's own P[j-tile] in its own shared memory,
//   B (256 rows)  = [Bh; Bl] of the i-tile, split across the pair: the leader
//                   holds Bh, the peer holds Bl (same offset in both CTAs),
//   D             = each CTA's TMEM: 128 lanes (its j samples) x [hi | lo] columns (i samples).
// Per SM this halves the B-side shared-memory reads and the L2 -> SM operand
// traffic (32 KB per 128-byte K block per SM instead of 48 KB), which is what bounds
// the single-CTA kernel (shared memory: 96 + 96 B/clk demanded of 128 B/clk).
// Barrier protocol: both producers' TMA bytes land on the LEADER's full barrier;
// tcgen05.commit multicasts to both CTAs' empty / accumulator-full barriers; both
// CTAs' epilogue warps arrive on the leader's accumulator-empty barrier.
//
// Two operand encodings share this kernel (template kI8):
//   bf16 (north-star form)  P in {0,1}, Bh = P*len_hi, Bl = P*len_lo as bf16, kind::f16,
//        K = 16 per MMA, fp32 accumulators; chunk sums added in fp32 registers.
//   u8 block floating point  every branch length is quantised to a * m * 2^e with an
//        8-bit factor a, a 16-bit factor m = 256*mh + ml and a per-chunk exponent e
//        (nodes are grouped by binade pairs along K): A = P*a, Bh = P*mh, Bl = P*ml as
//        unsigned bytes, kind::i8, K = 32 per MMA (twice the nodes per instruction and
//        per operand byte), int32 accumulators -- the contraction is EXACT integer
//        arithmetic; chunk sums are scaled by 2^e and added in fp64 registers.
// A K block is 128 bytes of every operand row either way (64 bf16 / 128 u8 nodes);
// chunks are runs of K blocks [chunk_end[c-1], chunk_end[c]) with scale chunk_scale[c].
constexpr int STAGES2 = 6;
constexpr int STAGE2_BYTES = A_BYTES + B_BYTES;
constexpr int NUM_BARS2 = 2 * STAGES2 + 4;
constexpr int SMEM2_BYTES = STAGES2 * STAGE2_BYTES + NUM_BARS2 * 8 + 16 + 1024;
constexpr int BKB = 128;  // bytes of K per block and operand row
// 16 epilogue warps = 4 TMEM lane quarters x 4 groups of 32 columns per plane: with the u8
// operands the mainloop of a tile takes ~82k cycles, and 8 warps holding 64 fp64 accumulators
// each (no registers left for instruction-level parallelism) needed longer than that for the
// chunk drains + the ratio epilogue (ncu: stall_math on dependent DADD/DFMA chains).
// Timeline counters for FRC_TC_DEBUG & 8 (cycles, per CTA): [0] MMA thread waiting for a free
// TMEM buffer, [1] MMA thread waiting for operands, [2] MMA thread total, [3] producer waiting
// for a free stage, [4] epilogue warp 2 waiting for an accumulator, [5] its drains, [6] its
// ratio epilogue + stores, [7] its total.
// Built only with -DFRC_TC_TIMELINE (scripts/exp_timeline.py); FRC_TC_DEBUG then also accepts
// 1 = do not load B, 2 = do not load A, 4 = no ratio epilogue (timing attribution; garbage results).
// k_unweighted_bits2 accumulates its own counters into g_bits_dbg (scripts/exp_bits_timeline.py).
#ifdef FRC_TC_TIMELINE
__device__ unsigned long long g_tc_dbg[512 * 8];
__device__ unsigned long long g_bits_dbg[512 * 8];
#define TL(x) x
#define TL_ON(mask) ((dbg & (mask)) != 0)
#else
#define TL(x)
#define TL_ON(mask) false
#endif
constexpr int EPI2_WARPS = 16;
constexpr int EPI2_COLS = 128 / (EPI2_WARPS / 4);  // accumulator columns per thread and plane
constexpr int THREADS2 = 32 * (EPI_WARP0 + EPI2_WARPS);

// ---- integer-mode epilogue, shared by k_unweighted_tc2<2> and k_unweighted_bits2
// One chunk's accumulators into acc: exact 64-bit accumulation in units of the smallest chunk scale, two
// 32x32+64 integer multiply-adds per element, (256*hi + lo) << shift with shift <= 16 (host-checked range).
// taddr is this thread's first hi-plane column; the lo plane is BN columns on.  Two register sets: the
// tcgen05.ld of batch c+1 is in flight while batch c is folded in.
__device__ __forceinline__ void drain_int(uint32_t taddr, uint32_t shift, unsigned long long (&acc)[EPI2_COLS]) {
  const uint32_t m0 = 1u << shift, m1 = 256u << shift;
  uint32_t v[2][8], w[2][8];
  ptx::tmem_ld_32x8(taddr, v[0]);
  ptx::tmem_ld_32x8(taddr + BN, w[0]);
#pragma unroll
  for (int cc = 0; cc < EPI2_COLS / 8; ++cc) {
    ptx::tmem_ld_wait();
    if (cc + 1 < EPI2_COLS / 8) {
      ptx::tmem_ld_32x8(taddr + (cc + 1) * 8, v[(cc + 1) & 1]);
      ptx::tmem_ld_32x8(taddr + BN + (cc + 1) * 8, w[(cc + 1) & 1]);
    }
#pragma unroll
    for (int x = 0; x < 8; ++x)
      acc[cc * 8 + x] += static_cast<unsigned long long>(v[cc & 1][x]) * m1 +
                         static_cast<unsigned long long>(w[cc & 1][x]) * m0;
  }
}

// The exact ratios of column sample j (this thread's TMEM lane) and row samples i0 + [0, EPI2_COLS) (its
// registers), stored from out[off] on (off: band offset of (i0, j)); pairs with U below flag_u_int are flagged.
template <bool kRect>
__device__ __forceinline__ void ratio_int(const unsigned long long (&acc)[EPI2_COLS], const long long* __restrict__ r_int,
                                          int64_t i0, int64_t j, int lane, int64_t n_samples, int64_t off,
                                          long long flag_u_int, float* __restrict__ out, uint32_t* __restrict__ flagged,
                                          unsigned long long* __restrict__ n_flagged, const Geometry& geo) {
  const long long rj = j < n_samples ? r_int[j] : 0;
  const long long ri_lane = r_int[i0 + lane];
#pragma unroll
  for (int n0 = 0; n0 < EPI2_COLS; n0 += 8) {
    float dv[8];
    bool fu[8];
#pragma unroll
    for (int x = 0; x < 8; ++x) {
      const long long ri = __shfl_sync(0xffffffffu, ri_lane, n0 + x);
      const long long sh = static_cast<long long>(acc[n0 + x]);
      // exact: U = (r_i - s) + (r_j - s) >= 0 (the reference's `result`), V = U + common
      const unsigned long long U = static_cast<unsigned long long>(ri + rj - 2 * sh);
      const unsigned long long V = U + static_cast<unsigned long long>(sh);
      const float Uf = fmaf(__uint2float_rn(static_cast<uint32_t>(U >> 32)), 4294967296.f,
                            __uint2float_rn(static_cast<uint32_t>(U)));
      const float Vf = fmaf(__uint2float_rn(static_cast<uint32_t>(V >> 32)), 4294967296.f,
                            __uint2float_rn(static_cast<uint32_t>(V)));
      dv[x] = __fdividef(Uf, Vf);  // unifrac.go:169; 0/0 -> NaN (A8)
      fu[x] = static_cast<long long>(U) < flag_u_int;
    }
#pragma unroll
    for (int x = 0; x < 8; ++x) {
      const int64_t i = i0 + n0 + x;
      if (i < n_samples && (kRect ? j < geo.n_ref : j < i)) {
        out[off] = dv[x];  // fp32 is what the ratio is; the host widens (wire.cu)
        // U and V are exact integer sums of the quantised lengths: no cancellation error, so a small d
        // needs no recompute here (identical samples give U = 0 exactly); only the absolute-error rule of
        // the merged small-length columns applies
        if (fu[x]) {
          unsigned long long slot = atomicAdd(n_flagged, 1ULL);
          flagged[slot] = static_cast<uint32_t>(off);
        }
      }
      off += kRect ? geo.n_ref : i;  // row i+1 starts i (rectangle: n_ref) entries later
    }
  }
}

// kMode: 0 = bf16 planes (fp32 accumulators), 1 = u8 planes with fp64 chunk accumulation (chunk scales
// spanning more than 2^16), 2 = u8 planes with 64-bit INTEGER accumulation and an integer / fp32 ratio
// epilogue: no fp64 instruction at all (every DADD/DFMA stalls its warp for tens of cycles on B200:
// ncu showed half of the epilogue warps' samples in stall_math on them at 4.5 % fp64-pipe utilisation).
template <int kMode, bool kRect>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS2, 1)
k_unweighted_tc2(const __grid_constant__ CUtensorMap mapP, const __grid_constant__ CUtensorMap mapBh,
                 const __grid_constant__ CUtensorMap mapBl, const int32_t* __restrict__ chunk_end,
                 const double* __restrict__ chunk_scale, const int32_t* __restrict__ chunk_shift,
                 int32_t n_chunks, int32_t biased, const double* __restrict__ r,
                 const long long* __restrict__ r_int, double unit, const Tile* __restrict__ tiles, int32_t n_tiles,
                 int64_t n_samples, int64_t first, float* __restrict__ out, double flag_below,
                 const double* __restrict__ flag_u_ptr, uint32_t* __restrict__ flagged,
                 unsigned long long* __restrict__ n_flagged, int dbg, const Geometry geo) {
  (void)dbg;
  constexpr bool kI8 = kMode != 0;
  constexpr bool kInt = kMode == 2;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = ptx::smem_u32(smem_raw);
  const uint32_t pad = ((raw + 1023u) & ~1023u) - raw;
  uint8_t* smem = smem_raw + pad;
  const uint32_t smem_base = raw + pad;
  const uint32_t bar_base = smem_base + STAGES2 * STAGE2_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES2 + s); };
  auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * STAGES2 + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * STAGES2 + 2 + b); };
  volatile uint32_t* tmem_slot =
      reinterpret_cast<volatile uint32_t*>(smem + STAGES2 * STAGE2_BYTES + NUM_BARS2 * 8);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta = ptx::cluster_ctarank();  // 0 = leader
  const int pair = blockIdx.x >> 1;
  const int n_pairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&mapP);
    ptx::prefetch_tensormap(cta == 0 ? &mapBh : &mapBl);
    for (int s = 0; s < STAGES2; ++s) {
      ptx::mbar_init(full_bar(s), 1);   // leader's producer arms it; both CTAs' TMA bytes complete it
      ptx::mbar_init(empty_bar(s), 1);  // multicast tcgen05.commit
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(tfull_bar(b), 1);
      ptx::mbar_init(tempty_bar(b), 2 * EPI2_WARPS);  // epilogue warps of both CTAs
    }
    ptx::fence_barrier_init();
    ptx::fence_proxy_async();
  }
  if (warp == 1) {
    ptx::tmem_alloc<2>(ptx::smem_u32(const_cast<uint32_t*>(tmem_slot)), TMEM_COLS);
    ptx::tmem_relinquish<2>();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();  // barriers of both CTAs initialised before any remote arrive / TMA
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int n_kblocks = chunk_end[n_chunks - 1];

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const void* mapB = cta == 0 ? static_cast<const void*>(&mapBh) : static_cast<const void*>(&mapBl);
      constexpr int kElems = kI8 ? BKB : BKB / 2;  // tensor-map elements per K block
      TL(long long w_empty = 0;)
      for (int t = pair; t < n_tiles; t += n_pairs) {
        const Tile tile = tiles[t];
        const int row_a = (tile.tj + static_cast<int>(cta)) * BM, row_b = tile.ti * BN;
        for (int kb = 0; kb < n_kblocks; ++kb) {
          TL(const long long c0 = clock64();)
          ptx::mbar_wait(empty_bar(stage), phase ^ 1u);
          TL(w_empty += clock64() - c0;)
          const uint32_t sa = smem_base + stage * STAGE2_BYTES;
          // bytes of BOTH CTAs complete the leader's barrier
          if (cta == 0)
            ptx::mbar_expect_tx(full_bar(stage), 2 * ((TL_ON(2) ? 0 : A_BYTES) + (TL_ON(1) ? 0 : B_BYTES)));
          const uint32_t lead_bar = ptx::mapa_u32(full_bar(stage), 0);
          if (!TL_ON(2)) ptx::tma_load_2d_2sm(sa, &mapP, lead_bar, kb * kElems, row_a);
          if (!TL_ON(1)) ptx::tma_load_2d_2sm(sa + A_BYTES, mapB, lead_bar, kb * kElems, row_b);
          if (++stage == STAGES2) { stage = 0; phase ^= 1u; }
        }
      }
      TL(g_tc_dbg[blockIdx.x * 8 + 3] = w_empty;)
    }
    __syncwarp();
  } else if (warp == 1) {
    // -------------------------------------------------- MMA issuer (leader only)
    if (lane == 0 && cta == 0) {
      constexpr uint32_t idesc = kI8 ? ptx::umma_idesc_u8(2 * BM, DN) : ptx::umma_idesc_bf16(2 * BM, DN);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t chunk = 0;
      TL(long long w_tempty = 0; long long w_full = 0; const long long c_start = clock64();)
      for (int t = pair; t < n_tiles; t += n_pairs) {
        int kb = 0;
        for (int ch = 0; ch < n_chunks; ++ch, ++chunk) {
          const uint32_t buf = chunk & 1u;
          TL(const long long c0 = clock64();)
          ptx::mbar_wait(tempty_bar(buf), ((chunk >> 1) & 1u) ^ 1u);
          TL(w_tempty += clock64() - c0;)
          ptx::tc_fence_after();
          const uint32_t d_tmem = tmem_base + buf * DN;
          const int kb_begin = kb, kb_end = chunk_end[ch];
          for (; kb < kb_end; ++kb) {
            TL(const long long c1 = clock64();)
            ptx::mbar_wait(full_bar(stage), phase);
            TL(w_full += clock64() - c1;)
            ptx::tc_fence_after();
            const uint32_t sa = smem_base + stage * STAGE2_BYTES;
            const uint64_t da = ptx::umma_desc_k_sw128(sa);
            const uint64_t db = ptx::umma_desc_k_sw128(sa + A_BYTES);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              // one MMA consumes 32 B of K per row (16 bf16 / 32 u8): +2 in the (>>4) start-address field
              const uint32_t accum = (kb > kb_begin || k > 0) ? 1u : 0u;
              if constexpr (kI8) ptx::umma_i8<2>(d_tmem, da + 2u * k, db + 2u * k, idesc, accum);
              else ptx::umma_bf16<2>(d_tmem, da + 2u * k, db + 2u * k, idesc, accum);
            }
            ptx::umma_commit_2sm(empty_bar(stage), 3);  // frees the stage in both CTAs
            if (++stage == STAGES2) { stage = 0; phase ^= 1u; }
          }
          ptx::umma_commit_2sm(tfull_bar(buf), 3);  // accumulators of both CTAs complete
        }
      }
      TL(g_tc_dbg[blockIdx.x * 8 + 0] = w_tempty; g_tc_dbg[blockIdx.x * 8 + 1] = w_full;
         g_tc_dbg[blockIdx.x * 8 + 2] = clock64() - c_start;)
    }
    __syncwarp();
  } else {
    // ---------------------------------------------------------------- epilogue
    const int q = warp & 3;                      // TMEM lane quarter this warp may read
    const int cg = (warp - EPI_WARP0) >> 2;      // which EPI2_COLS columns of each plane it owns
    using Acc = typename std::conditional<kInt, unsigned long long,
                                          typename std::conditional<kI8, double, float>::type>::type;
    // pairs whose unique length U is below this are recomputed exactly as well: the summed absolute
    // error of the imprecisely quantised branch lengths could exceed 2e-6 of U (k_quantize_lengths)
    const float flag_u = flag_u_ptr ? static_cast<float>(*flag_u_ptr) : 0.f;
    const float flag_d = static_cast<float>(flag_below);
    // integer mode: lengths, row sums and accumulators are integers in units of `unit` = the smallest chunk scale
    const long long flag_u_int = (kInt && flag_u_ptr) ? static_cast<long long>(*flag_u_ptr / unit) : 0;
    double acc0 = 0.0;  // u8 fp64 mode, biased accumulation: minus the 2^52-bias of every chunk
    if constexpr (kI8 && !kInt)
      if (biased) for (int ch = 0; ch < n_chunks; ++ch) acc0 -= 4503599627370496.0 * chunk_scale[ch];
    uint32_t chunk = 0;
    TL(long long w_tfull = 0; long long t_drain = 0; long long t_ratio = 0; const long long e_start = clock64();)
    for (int t = pair; t < n_tiles; t += n_pairs) {
      const Tile tile = tiles[t];
      Acc acc[EPI2_COLS];
#pragma unroll
      for (int n = 0; n < EPI2_COLS; ++n) acc[n] = static_cast<Acc>(acc0);
      for (int ch = 0; ch < n_chunks; ++ch, ++chunk) {
        const uint32_t buf = chunk & 1u;
        const double scale = (kI8 && !kInt) ? chunk_scale[ch] : 1.0;
        const uint32_t shift = kInt ? static_cast<uint32_t>(chunk_shift[ch]) : 0u;
        TL(const long long c0 = clock64();)
        ptx::mbar_wait(tfull_bar(buf), (chunk >> 1) & 1u);
        TL(const long long c1 = clock64();)
        ptx::tc_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + buf * DN + cg * EPI2_COLS;
        if constexpr (kInt) {
          drain_int(taddr, shift, acc);
        } else if constexpr (kI8) {
          // both plane sums are in [0, 2^31): S = 256*hi + lo < 2^40 comes from one 32x32->64 integer
          // multiply-add; OR-ing it into the mantissa of 2^52 gives the double 2^52 + S without any
          // conversion instruction.  biased: ONE fp64 instruction per element accumulates
          // scale * (2^52 + S); the offsets 2^52 * scale were pre-subtracted (acc0), and the rounding
          // (to multiples of the largest chunk scale) is ~2^-28 of a sum because the host only sets
          // `biased` when all chunk scales lie within 2^8.  Otherwise 2^52 is subtracted first (exact).
          auto drain = [&](auto kBiased) {
            // two register sets: the tcgen05.ld of batch c+1 is in flight while batch c is folded in
            uint32_t v[2][8], w[2][8];
            ptx::tmem_ld_32x8(taddr, v[0]);
            ptx::tmem_ld_32x8(taddr + BN, w[0]);
#pragma unroll
            for (int cc = 0; cc < EPI2_COLS / 8; ++cc) {
              ptx::tmem_ld_wait();
              if (cc + 1 < EPI2_COLS / 8) {
                ptx::tmem_ld_32x8(taddr + (cc + 1) * 8, v[(cc + 1) & 1]);
                ptx::tmem_ld_32x8(taddr + BN + (cc + 1) * 8, w[(cc + 1) & 1]);
              }
#pragma unroll
              for (int x = 0; x < 8; ++x) {
                const unsigned long long S = static_cast<unsigned long long>(v[cc & 1][x]) * 256ull + w[cc & 1][x];
                double D = __longlong_as_double(static_cast<long long>(S | 0x4330000000000000ull));
                if (!decltype(kBiased)::value) D -= 4503599627370496.0;
                acc[cc * 8 + x] = fma(scale, D, acc[cc * 8 + x]);
              }
            }
          };
          if (biased) drain(std::true_type{}); else drain(std::false_type{});
        } else {
#pragma unroll
          for (int cc = 0; cc < EPI2_COLS / 16; ++cc) {
            uint32_t v[16], w[16];
            ptx::tmem_ld_32x16(taddr + cc * 16, v);
            ptx::tmem_ld_32x16(taddr + BN + cc * 16, w);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int x = 0; x < 16; ++x) acc[cc * 16 + x] += __uint_as_float(v[x]) + __uint_as_float(w[x]);
          }
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_cluster(tempty_bar(buf), 0);  // the leader's barrier
        TL(w_tfull += c1 - c0; t_drain += clock64() - c1;)
      }
      TL(const long long c2 = clock64();)
      // this thread's TMEM lane is a COLUMN sample j of the output; its registers run over
      // EPI2_COLS ROW samples i.  For a fixed register the 32 lanes of the warp therefore write
      // 32 consecutive floats of one row of the flat triangle: fully coalesced 128-byte stores.
      const int64_t j = static_cast<int64_t>(tile.tj + static_cast<int>(cta)) * BM + q * 32 + lane;
      const int64_t i0 = static_cast<int64_t>(tile.ti) * BN + cg * EPI2_COLS;
      static_assert(EPI2_COLS == 32, "r[i] is broadcast from lane n");
      if (TL_ON(4)) {
        if (acc[0] == static_cast<Acc>(-1.5)) out[0] = 0.f;
      } else if (kRect || static_cast<int64_t>(tile.tj + static_cast<int>(cta)) * BM + q * 32 < i0 + EPI2_COLS) {  // warp-uniform
        // flat index of (i0, j) relative to the band
        int64_t off = kRect ? (i0 - geo.q0) * geo.n_ref - first + j : i0 * (i0 - 1) / 2 - first + j;
        // r is padded to a multiple of the tile size: the loads are in range and coalesced.
        // Batches of 8 row samples: first the arithmetic of all 8 (independent chains the scheduler can
        // interleave), then the stores and the (rare) fix-up flags.
        if constexpr (kInt) {
          ratio_int<kRect>(acc, r_int, i0, j, lane, n_samples, off, flag_u_int, out, flagged, n_flagged, geo);
        } else {
          const double rj = j < n_samples ? r[j] : 0.0;
          const double ri_lane = r[i0 + lane];
#pragma unroll
          for (int n0 = 0; n0 < EPI2_COLS; n0 += 8) {
            float dv[8], uv[8];
#pragma unroll
            for (int x = 0; x < 8; ++x) {
              const double ri = __shfl_sync(0xffffffffu, ri_lane, n0 + x);
              // fp64 only where cancellation needs it: U = R - 2s (the reference's `result`)
              const double sd = static_cast<double>(acc[n0 + x]);
              const double U = fma(-2.0, sd, ri + rj);
              uv[x] = static_cast<float>(U);
              dv[x] = __fdividef(uv[x], uv[x] + static_cast<float>(sd));  // U / (U + common), unifrac.go:169
            }
#pragma unroll
            for (int x = 0; x < 8; ++x) {
              const int64_t i = i0 + n0 + x;
              if (i < n_samples && (kRect ? j < geo.n_ref : j < i)) {
                out[off] = dv[x];  // fp32 is what the ratio is; the host widens (wire.cu)
                if (dv[x] < flag_d || uv[x] < flag_u) {
                  unsigned long long slot = atomicAdd(n_flagged, 1ULL);
                  flagged[slot] = static_cast<uint32_t>(off);
                }
              }
              off += kRect ? geo.n_ref : i;  // row i+1 starts i (rectangle: n_ref) entries later
            }
          }
        }
      }
      TL(t_ratio += clock64() - c2;)
    }
    TL(if (warp == EPI_WARP0 && lane == 0) {
      g_tc_dbg[blockIdx.x * 8 + 4] = w_tfull;
      g_tc_dbg[blockIdx.x * 8 + 5] = t_drain;
      g_tc_dbg[blockIdx.x * 8 + 6] = t_ratio;
      g_tc_dbg[blockIdx.x * 8 + 7] = clock64() - e_start;
    })
  }

  ptx::tc_fence_before();
  ptx::cluster_sync_all();  // the peer may still read our shared memory / signal our barriers
  if (warp == 1) {
    __syncwarp();
    ptx::tmem_dealloc<2>(tmem_base, TMEM_COLS);
  }
}

// ----------------------------------------------------------------------------
// Bits feed (capacity mode): the CTA-pair kind::i8 GEMM and integer epilogue of k_unweighted_tc2<2>, but the
// u8 operand tiles are never materialised in HBM.  Producer warps expand them straight into the 128-byte
// swizzled shared-memory layout the MMA reads (the same A and B stage tiles of 128 rows x BKB bytes):
//     A[j][k]  = bit(j, k) ? qa[k] : 0      (this CTA's 128 column samples)
//     B[i][k]  = bit(i, k) ? qh[k] | ql[k]  (the 128 row samples; leader: high plane, peer: low plane)
// from sample-major bit rows bitsS[np][kp / 8] (1 bit per (sample, operand column); column k is bit
// k % 8 of byte k / 8) and the per-column quantised factors.  Per 128-column K block a CTA reads
// 4 KB of bits + 256 B of factors instead of 32 KB of operand bytes: the operand expansion kernel,
// its HBM traffic (3 bytes per (sample, column): 60 GB at cfg4) and the per-rank expansion of every
// sample in a multi-GPU run disappear.
//
// Warps: 0 = TMA loader of bit tiles, 1 = MMA issuer, 4..11 = producers (expansion), 12..27 =
// epilogue.  Registers move from the control / producer warp groups to the epilogue ones
// (setmaxnreg), which keep the 96 they have in k_unweighted_tc2.
namespace bits {
constexpr int OSTAGES = 5;                     // operand ring (written by the producers)
constexpr int OSTAGE_BYTES = A_BYTES + B_BYTES;
constexpr int BSTAGES = 8;                     // bit-tile ring (written by TMA)
constexpr int BITS_TILE = 128 * 16;            // 128 samples x 128 columns / 8
constexpr int BSTAGE_BYTES = 2 * BITS_TILE + 2 * BKB;  // A bits, B bits, qa, q(h|l)
constexpr int NUM_BARS = 3 * OSTAGES + 2 * BSTAGES + 4;
constexpr int SMEM_BYTES = OSTAGES * OSTAGE_BYTES + BSTAGES * BSTAGE_BYTES + NUM_BARS * 8 + 16 + 1024;
constexpr int PROD_WARP0 = 4, PROD_WARPS = 8;
constexpr int EPI_WARP0 = 12;                  // EPI2_WARPS epilogue warps, as in k_unweighted_tc2
constexpr int THREADS = 32 * (EPI_WARP0 + EPI2_WARPS);  // 896

// 4 bits (b0..b3 of `nib`, other bits must be zero) -> byte masks 0xFF / 0x00: one multiply puts bit g
// into the sign of byte g, one PRMT replicates the signs.
__device__ __forceinline__ uint32_t mask4(uint32_t nib) {
  uint32_t m;
  asm("prmt.b32 %0, %1, 0, 0xBA98;" : "=r"(m) : "r"(nib * 0x10204080u));
  return m;
}
}  // namespace bits

template <bool kRect>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(bits::THREADS, 1)
k_unweighted_bits2(const __grid_constant__ CUtensorMap mapBits, const uint8_t* __restrict__ qa,
                   const uint8_t* __restrict__ qh, const uint8_t* __restrict__ ql,
                   const int32_t* __restrict__ chunk_end, const int32_t* __restrict__ chunk_shift,
                   int32_t n_chunks, const long long* __restrict__ r_int, double unit,
                   const Tile* __restrict__ tiles, int32_t n_tiles, int64_t n_samples, int64_t first,
                   float* __restrict__ out, const double* __restrict__ flag_u_ptr,
                   uint32_t* __restrict__ flagged, unsigned long long* __restrict__ n_flagged, const Geometry geo) {
  using namespace bits;  // (EPI_WARP0 is written bits::EPI_WARP0: k_unweighted_tc2 has its own)
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = ptx::smem_u32(smem_raw);
  const uint32_t pad = ((raw + 1023u) & ~1023u) - raw;
  uint8_t* smem = smem_raw + pad;
  const uint32_t smem_base = raw + pad;                               // operand ring (1024-aligned)
  const uint32_t bits_base = smem_base + OSTAGES * OSTAGE_BYTES;      // bit-tile ring
  const uint32_t bar_base = bits_base + BSTAGES * BSTAGE_BYTES;
  auto ofull_bar = [&](int s) { return bar_base + 8u * s; };
  auto oempty_bar = [&](int s) { return bar_base + 8u * (OSTAGES + s); };
  auto bfull_bar = [&](int s) { return bar_base + 8u * (2 * OSTAGES + s); };
  auto bempty_bar = [&](int s) { return bar_base + 8u * (2 * OSTAGES + BSTAGES + s); };
  auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * OSTAGES + 2 * BSTAGES + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * OSTAGES + 2 * BSTAGES + 2 + b); };
  // peer CTA only: its producer warps arrive here (CTA scope); one forwarder thread then tells the leader
  auto pfull_bar = [&](int s) { return bar_base + 8u * (2 * OSTAGES + 2 * BSTAGES + 4 + s); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(
      smem + OSTAGES * OSTAGE_BYTES + BSTAGES * BSTAGE_BYTES + NUM_BARS * 8);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta = ptx::cluster_ctarank();  // 0 = leader
  const int pair = blockIdx.x >> 1;
  const int n_pairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&mapBits);
    for (int s = 0; s < OSTAGES; ++s) {
      ptx::mbar_init(ofull_bar(s), PROD_WARPS + 1);  // leader: its producer warps + the peer's forwarder
      ptx::mbar_init(oempty_bar(s), 1);              // multicast tcgen05.commit
      ptx::mbar_init(pfull_bar(s), PROD_WARPS);
    }
    for (int s = 0; s < BSTAGES; ++s) {
      ptx::mbar_init(bfull_bar(s), 1);
      ptx::mbar_init(bempty_bar(s), PROD_WARPS);
    }
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(tfull_bar(b), 1);
      ptx::mbar_init(tempty_bar(b), 2 * EPI2_WARPS);
    }
    ptx::fence_barrier_init();
    ptx::fence_proxy_async();
  }
  if (warp == 1) {
    ptx::tmem_alloc<2>(ptx::smem_u32(const_cast<uint32_t*>(tmem_slot)), TMEM_COLS);
    ptx::tmem_relinquish<2>();
  }
  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_kblocks = chunk_end[n_chunks - 1];

  if (warp == 0) {
    ptx::setmaxnreg_dec<24>();
    // ------------------------------------------------ TMA loader: bit tiles + factors of each K block
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const uint8_t* qb = cta == 0 ? qh : ql;
      for (int t = pair; t < n_tiles; t += n_pairs) {
        const Tile tile = tiles[t];
        const int row_a = (tile.tj + static_cast<int>(cta)) * BM, row_b = tile.ti * BN;
        for (int kb = 0; kb < n_kblocks; ++kb) {
          TL(const long long c0 = clock64();)
          ptx::mbar_wait(bempty_bar(stage), phase ^ 1u);
          TL(g_bits_dbg[blockIdx.x * 8 + 0] += clock64() - c0;)
          const uint32_t sb = bits_base + stage * BSTAGE_BYTES;
          ptx::mbar_expect_tx(bfull_bar(stage), BSTAGE_BYTES);
          ptx::tma_load_2d(sb, &mapBits, bfull_bar(stage), kb * 16, row_a);
          ptx::tma_load_2d(sb + BITS_TILE, &mapBits, bfull_bar(stage), kb * 16, row_b);
          ptx::bulk_load_1d(sb + 2 * BITS_TILE, qa + static_cast<int64_t>(kb) * BKB, BKB, bfull_bar(stage));
          ptx::bulk_load_1d(sb + 2 * BITS_TILE + BKB, qb + static_cast<int64_t>(kb) * BKB, BKB, bfull_bar(stage));
          if (++stage == BSTAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    ptx::setmaxnreg_dec<24>();
    // -------------------------------------------------- MMA issuer (leader only)
    if (lane == 0 && cta == 0) {
      constexpr uint32_t idesc = ptx::umma_idesc_u8(2 * BM, DN);
      int stage = 0;
      uint32_t phase = 0;
      uint32_t chunk = 0;
      for (int t = pair; t < n_tiles; t += n_pairs) {
        int kb = 0;
        for (int ch = 0; ch < n_chunks; ++ch, ++chunk) {
          const uint32_t buf = chunk & 1u;
          TL(const long long c0 = clock64();)
          ptx::mbar_wait(tempty_bar(buf), ((chunk >> 1) & 1u) ^ 1u);
          TL(g_bits_dbg[blockIdx.x * 8 + 1] += clock64() - c0;)
          ptx::tc_fence_after();
          const uint32_t d_tmem = tmem_base + buf * DN;
          const int kb_begin = kb, kb_end = chunk_end[ch];
          for (; kb < kb_end; ++kb) {
            TL(const long long c1 = clock64();)
            ptx::mbar_wait(ofull_bar(stage), phase);
            TL(g_bits_dbg[blockIdx.x * 8 + 2] += clock64() - c1;)
            ptx::tc_fence_after();
            const uint32_t sa = smem_base + stage * OSTAGE_BYTES;
            const uint64_t da = ptx::umma_desc_k_sw128(sa);
            const uint64_t db = ptx::umma_desc_k_sw128(sa + A_BYTES);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              ptx::umma_i8<2>(d_tmem, da + 2u * k, db + 2u * k, idesc, (kb > kb_begin || k > 0) ? 1u : 0u);
            ptx::umma_commit_2sm(oempty_bar(stage), 3);
            if (++stage == OSTAGES) { stage = 0; phase ^= 1u; }
          }
          ptx::umma_commit_2sm(tfull_bar(buf), 3);
        }
      }
    }
    __syncwarp();
  } else if (warp < PROD_WARP0) {
    ptx::setmaxnreg_dec<24>();
    // warp 2 of the PEER forwards "my half of the stage is written" to the leader: one cluster-scope
    // release per K block instead of one per producer warp (a remote arrive with release.cluster
    // semantics costs ~1 us; eight of them per K block made the producers 4x too slow)
    if (warp == 2 && cta == 1 && lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = pair; t < n_tiles; t += n_pairs)
        for (int kb = 0; kb < n_kblocks; ++kb) {
          ptx::mbar_wait(pfull_bar(stage), phase);
          ptx::mbar_arrive_cluster_relaxed(ofull_bar(stage), 0);
          if (++stage == OSTAGES) { stage = 0; phase ^= 1u; }
        }
    }
    __syncwarp();
  } else if (warp < PROD_WARP0 + PROD_WARPS) {
    ptx::setmaxnreg_dec<48>();
    // ---------------------------------------------------------------- producers
    // thread -> 16-byte chunk c of the K block (16 columns) and rows base, base + 32, ... of both tiles
    const int pt = threadIdx.x - PROD_WARP0 * 32;  // 0..255
    const int c = pt & 7;
    const int rbase = pt >> 3;                     // 0..31
    int ostage = 0, bstage = 0;
    uint32_t ophase = 0, bphase = 0;
    for (int t = pair; t < n_tiles; t += n_pairs) {
      for (int kb = 0; kb < n_kblocks; ++kb) {
        TL(const long long c0 = clock64();)
        ptx::mbar_wait(bfull_bar(bstage), bphase);
        TL(const long long c1 = clock64();)
        ptx::mbar_wait(oempty_bar(ostage), ophase ^ 1u);
        TL(const long long c2 = clock64();)
        const uint8_t* sb = smem + OSTAGES * OSTAGE_BYTES + bstage * BSTAGE_BYTES;
        uint8_t* so = smem + ostage * OSTAGE_BYTES;
        const uint4 qA = *reinterpret_cast<const uint4*>(sb + 2 * BITS_TILE + c * 16);
        const uint4 qB = *reinterpret_cast<const uint4*>(sb + 2 * BITS_TILE + BKB + c * 16);
#pragma unroll
        for (int tile_sel = 0; tile_sel < 2; ++tile_sel) {
          const uint4 q = tile_sel == 0 ? qA : qB;
          const uint8_t* tile_bits = sb + tile_sel * BITS_TILE;
          uint8_t* dst = so + tile_sel * A_BYTES;
#pragma unroll
          for (int m = 0; m < 4; ++m) {
            const int r = rbase + 32 * m;
            const uint32_t b16 = *reinterpret_cast<const uint16_t*>(tile_bits + r * 16 + c * 2);
            const uint32_t lo8 = b16 & 0xFFu, hi8 = b16 >> 8;
            uint4 v;
            v.x = q.x & mask4(lo8 & 0xFu);
            v.y = q.y & mask4(lo8 >> 4);
            v.z = q.z & mask4(hi8 & 0xFu);
            v.w = q.w & mask4(hi8 >> 4);
            // SWIZZLE_128B K-major: row r at (r / 8) * 1024 + (r % 8) * 128, 16-byte chunk c at c ^ (r % 8)
            *reinterpret_cast<uint4*>(dst + (r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4)) = v;
          }
        }
        ptx::fence_proxy_async();  // generic-proxy stores -> visible to the tensor core's async proxy
        __syncwarp();
        if (lane == 0) {
          ptx::mbar_arrive(cta == 0 ? ofull_bar(ostage) : pfull_bar(ostage));
          ptx::mbar_arrive(bempty_bar(bstage));
        }
        TL(if (pt == 0) {
          g_bits_dbg[blockIdx.x * 8 + 3] += c1 - c0;             // waiting for bits
          g_bits_dbg[blockIdx.x * 8 + 4] += c2 - c1;             // waiting for a free operand stage
          g_bits_dbg[blockIdx.x * 8 + 5] += clock64() - c2;      // expanding + fence + arrive
        })
        if (++ostage == OSTAGES) { ostage = 0; ophase ^= 1u; }
        if (++bstage == BSTAGES) { bstage = 0; bphase ^= 1u; }
      }
    }
  } else {
    ptx::setmaxnreg_inc<96>();
    // ---------------------------------------------------------------- epilogue (integer mode)
    const int q = warp & 3;
    const int cg = (warp - bits::EPI_WARP0) >> 2;
    const long long flag_u_int = flag_u_ptr ? static_cast<long long>(*flag_u_ptr / unit) : 0;
    uint32_t chunk = 0;
    for (int t = pair; t < n_tiles; t += n_pairs) {
      const Tile tile = tiles[t];
      unsigned long long acc[EPI2_COLS];
#pragma unroll
      for (int n = 0; n < EPI2_COLS; ++n) acc[n] = 0;
      for (int ch = 0; ch < n_chunks; ++ch, ++chunk) {
        const uint32_t buf = chunk & 1u;
        const uint32_t shift = static_cast<uint32_t>(chunk_shift[ch]);
        ptx::mbar_wait(tfull_bar(buf), (chunk >> 1) & 1u);
        ptx::tc_fence_after();
        drain_int(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + buf * DN + cg * EPI2_COLS, shift, acc);
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_cluster(tempty_bar(buf), 0);
      }
      const int64_t j = static_cast<int64_t>(tile.tj + static_cast<int>(cta)) * BM + q * 32 + lane;
      const int64_t i0 = static_cast<int64_t>(tile.ti) * BN + cg * EPI2_COLS;
      if (kRect || static_cast<int64_t>(tile.tj + static_cast<int>(cta)) * BM + q * 32 < i0 + EPI2_COLS)  // warp-uniform
        ratio_int<kRect>(acc, r_int, i0, j, lane, n_samples,
                         kRect ? (i0 - geo.q0) * geo.n_ref - first + j : i0 * (i0 - 1) / 2 - first + j, flag_u_int,
                         out, flagged, n_flagged, geo);
    }
  }

  ptx::tc_fence_before();
  ptx::cluster_sync_all();
  if (warp == 1) {
    __syncwarp();
    ptx::tmem_dealloc<2>(tmem_base, TMEM_COLS);
  }
}

// Exact recompute of flagged pairs: one warp per pair, fp64, TRUE branch lengths (len_col[k] = length of the
// node in operand column k, 0 in padding columns).  Identical samples give exactly 0.  The presence of a node
// is read from `rows`, in one of three formats:
enum class Rows {
  kBf16,  // the A operand [np][kp] of the materialised bf16 feed: P
  kU8,    // the A operand [np][kp] of the materialised u8 feed: P*a, non-zero exactly where the node is present
          // and has a non-zero length
  kBits,  // the bit rows bitsS[np][kp / 32] of the bits feed
};
template <Rows kRows, bool kRect>
__global__ void __launch_bounds__(256)
k_unweighted_fixup(const void* __restrict__ rows, int32_t kp, const double* __restrict__ len_col,
                   const uint32_t* __restrict__ flagged, const unsigned long long* __restrict__ n_flagged,
                   unsigned long long* __restrict__ count_host, int64_t first, float* __restrict__ out,
                   const Exceptions ex, const Geometry geo) {
  const unsigned long long total = *n_flagged;
  if (blockIdx.x == 0 && threadIdx.x == 0) *count_host = total;  // mapped pinned memory
  const int lane = threadIdx.x & 31;
  const unsigned long long warps = (static_cast<unsigned long long>(gridDim.x) * blockDim.x) >> 5;
  const int32_t words = kp / 32;  // (kBits: 32-bit words per row)
  for (unsigned long long w = (static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
       w < total; w += warps) {
    const uint32_t off = flagged[w];
    int64_t i, j;
    pair_at<kRect>(first + off, geo, i, j);
    double uniq = 0.0, comm = 0.0;
    if constexpr (kRows == Rows::kBits) {
      const uint32_t* bi = static_cast<const uint32_t*>(rows) + i * words;
      const uint32_t* bj = static_cast<const uint32_t*>(rows) + j * words;
      for (int32_t c = lane; c < words; c += 32) {
        const uint32_t a = bi[c], b = bj[c];
        uint32_t x = a ^ b, y = a & b;
        while (x) { const int k = __ffs(x) - 1; uniq += len_col[c * 32 + k]; x &= x - 1; }
        while (y) { const int k = __ffs(y) - 1; comm += len_col[c * 32 + k]; y &= y - 1; }
      }
    } else {
      constexpr bool kI8 = kRows == Rows::kU8;
      constexpr int kPer = kI8 ? 16 : 8;  // operand columns per 16-byte load
      const int64_t row_bytes = static_cast<int64_t>(kp) * (kI8 ? 1 : 2);
      const uint4* pi = reinterpret_cast<const uint4*>(static_cast<const uint8_t*>(rows) + i * row_bytes);
      const uint4* pj = reinterpret_cast<const uint4*>(static_cast<const uint8_t*>(rows) + j * row_bytes);
      for (int32_t c = lane; c * kPer < kp; c += 32) {
        const uint4 a = pi[c], b = pj[c];
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int h = 0; h < kPer; ++h) {
          const int32_t k = c * kPer + h;
          bool pa, pb;
          if constexpr (kI8) {
            pa = ((aw[h >> 2] >> ((h & 3) * 8)) & 0xFFu) != 0;
            pb = ((bw[h >> 2] >> ((h & 3) * 8)) & 0xFFu) != 0;
          } else {
            pa = ((aw[h >> 1] >> ((h & 1) * 16)) & 0xFFFFu) != 0;
            pb = ((bw[h >> 1] >> ((h & 1) * 16)) & 0xFFFFu) != 0;
          }
          if (pa && pb) comm += len_col[k];
          else if (pa || pb) uniq += len_col[k];
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      uniq += __shfl_xor_sync(0xffffffffu, uniq, o);
      comm += __shfl_xor_sync(0xffffffffu, comm, o);
    }
    if (lane == 0) store_fixed(out, off, uniq / (uniq + comm), first, ex);
  }
}

typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                        const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                        const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_tmapEncodeTiled g_encode = nullptr;

// K-major operand [rows][kp]; a box is 128 bytes of K x box_rows rows.
bool make_map(CUtensorMap* m, const void* base, int64_t rows, int32_t kp, int box_rows, bool i8,
              std::string* err) {
  const int esz = i8 ? 1 : 2;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(kp), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(kp) * esz};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(BKB / esz), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult rc = g_encode(m, i8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                         const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) {
    if (err) *err = "cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(rc));
    return false;
  }
  return true;
}

}  // namespace

struct TcOperands {
  bool from_bits = false;  // the operand feed: false = materialised (k_unweighted_tc2), true = bits (k_unweighted_bits2)
  CUtensorMap mapP, mapBh, mapBl;  // materialised: the three K-major operands
  const void* P = nullptr;         // materialised: the A operand (the fix-up reads presence from it)
  CUtensorMap mapBits;             // bits: 128-sample x 16-byte tiles of bitsS
  const uint32_t* bitsS = nullptr; // bits: the bit rows [np][kp / 32] (the fix-up reads presence from them)
  const uint8_t *qa = nullptr, *qh = nullptr, *ql = nullptr;  // bits: per-column u8 factors (k_quantize_lengths)
  bool i8;
  int32_t kp;
  TcChunks chunks;
  const double* len_col;
  const double* flag_u;  // device scalar (u8) or null
  const long long* r_int = nullptr;  // u8 integer mode: row sums in units of `unit`
  double unit = 1.0;
  int dbg = 0;  // FRC_TC_DEBUG (timeline builds), read once per job
};

bool tc_setup(std::string* err) {
  if (!g_encode) {  // process-wide: the driver entry point
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) {
      if (err) *err = "cuTensorMapEncodeTiled is not available from the driver";
      return false;
    }
    g_encode = reinterpret_cast<PFN_tmapEncodeTiled>(fn);
  }
  // per device (function attributes live in the device's context): called once per device context
  cudaError_t e = cudaSuccess;
  for (auto kernel : {k_unweighted_tc2<0, false>, k_unweighted_tc2<1, false>, k_unweighted_tc2<2, false>,
                      k_unweighted_tc2<0, true>, k_unweighted_tc2<1, true>, k_unweighted_tc2<2, true>})
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM2_BYTES);
  if (e != cudaSuccess) {
    if (err) *err = std::string("cudaFuncSetAttribute(k_unweighted_tc2): ") + cudaGetErrorString(e);
    return false;
  }
  for (auto kernel : {k_unweighted_bits2<false>, k_unweighted_bits2<true>})
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bits::SMEM_BYTES);
  if (e != cudaSuccess) {
    if (err) *err = std::string("cudaFuncSetAttribute(k_unweighted_bits2): ") + cudaGetErrorString(e);
    return false;
  }
  return true;
}

TcOperands* tc_operands_create(const void* P, const void* Bh, const void* Bl, int64_t np, int32_t kp,
                               bool i8, const TcChunks& chunks, const double* len_col, const double* flag_u,
                               std::string* err) {
  if (!g_encode) { if (err) *err = "tc_setup has not run on this device context"; return nullptr; }
  TcOperands* o = new TcOperands();
  if (const char* de = getenv("FRC_TC_DEBUG")) o->dbg = atoi(de);
  o->P = P;
  o->i8 = i8;
  o->kp = kp;
  o->chunks = chunks;
  o->len_col = len_col;
  o->flag_u = flag_u;
  if (!make_map(&o->mapP, P, np, kp, BM, i8, err) || !make_map(&o->mapBh, Bh, np, kp, BN, i8, err) ||
      !make_map(&o->mapBl, Bl, np, kp, BN, i8, err)) {
    delete o;
    return nullptr;
  }
  return o;
}
TcOperands* tc_operands_create_bits(const uint32_t* bitsS, int64_t np, int32_t kp, const uint8_t* qa,
                                    const uint8_t* qh, const uint8_t* ql, const TcChunks& chunks,
                                    const double* len_col, const double* flag_u, const long long* r_int,
                                    double unit, std::string* err) {
  if (!g_encode) { if (err) *err = "tc_setup has not run on this device context"; return nullptr; }
  TcOperands* o = new TcOperands();
  o->from_bits = true;
  o->bitsS = bitsS; o->qa = qa; o->qh = qh; o->ql = ql;
  o->i8 = true; o->kp = kp; o->chunks = chunks;
  o->len_col = len_col; o->flag_u = flag_u; o->r_int = r_int; o->unit = unit;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(kp / 8), static_cast<cuuint64_t>(np)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(kp / 8)};
  cuuint32_t box[2] = {16, 128};
  cuuint32_t estr[2] = {1, 1};
  CUresult rc = g_encode(&o->mapBits, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint32_t*>(bitsS), dims, strides,
                         box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (rc != CUDA_SUCCESS) {
    if (err) *err = "cuTensorMapEncodeTiled(bits) failed with CUresult " + std::to_string(static_cast<int>(rc));
    delete o;
    return nullptr;
  }
  return o;
}
void tc_operands_set_int(TcOperands* o, const long long* r_int, double unit) { o->r_int = r_int; o->unit = unit; }
void tc_operands_destroy(TcOperands* o) { delete o; }

}  // namespace frc
// Debug helpers (not part of the C ABI): copy the timeline counters of k_unweighted_tc2 (FRC_TC_DEBUG=8) and
// of k_unweighted_bits2 (always accumulated; clear != 0 zeroes them after the copy).
extern "C" int frc_debug_tc_counters(unsigned long long* out, int n) {
#ifdef FRC_TC_TIMELINE
  if (n > 512 * 8) n = 512 * 8;
  return static_cast<int>(cudaMemcpyFromSymbol(out, frc::g_tc_dbg, sizeof(unsigned long long) * n));
#else
  (void)out; (void)n;
  return -1;  // built without -DFRC_TC_TIMELINE
#endif
}
extern "C" int frc_debug_bits_counters(unsigned long long* out, int n, int clear) {
#ifdef FRC_TC_TIMELINE
  if (n > 512 * 8) n = 512 * 8;
  int rc = static_cast<int>(cudaMemcpyFromSymbol(out, frc::g_bits_dbg, sizeof(unsigned long long) * n));
  if (clear) { static unsigned long long z[512 * 8] = {0}; cudaMemcpyToSymbol(frc::g_bits_dbg, z, sizeof(z)); }
  return rc;
#else
  (void)out; (void)n; (void)clear;
  return -1;
#endif
}
namespace frc {

int tc_chunk_kblocks() {
  // bf16: 64 blocks = 4096 nodes per uninterrupted fp32 TMEM accumulation run
  const char* e = getenv("FRC_TC_CHUNK_KBLOCKS");
  int x = e ? atoi(e) : 64;
  return x < 1 ? 1 : x;
}

int launch_unweighted_tc(const TcOperands* ops, const double* r, const Tile* tiles, int32_t n_tiles,
                         int64_t n_samples, int64_t first, const Geometry& geo, float* out, double flag_below,
                         uint32_t* flagged, unsigned long long* n_flagged, int num_sms, cudaStream_t s) {
  if (n_tiles <= 0) return 0;
  // `tiles` lists pair tiles (tj even): one cluster of two CTAs each
  const int pairs = num_sms / 2;
  const int grid = 2 * (n_tiles < pairs ? n_tiles : pairs);
  const TcChunks& c = ops->chunks;
  if (ops->from_bits) {  // integer mode: U and V are exact, so r and flag_below play no part
    const auto kernel = geo.rect ? k_unweighted_bits2<true> : k_unweighted_bits2<false>;
    kernel<<<grid, bits::THREADS, bits::SMEM_BYTES, s>>>(
        ops->mapBits, ops->qa, ops->qh, ops->ql, c.end, c.shift, c.n, ops->r_int, ops->unit, tiles, n_tiles, n_samples,
        first, out, ops->flag_u, flagged, n_flagged, geo);
    return 1;
  }
  const int mode = ops->i8 && ops->r_int ? 2 : ops->i8 ? 1 : 0;
  const auto kernel = geo.rect ? (mode == 2 ? k_unweighted_tc2<2, true> : mode == 1 ? k_unweighted_tc2<1, true>
                                                                                   : k_unweighted_tc2<0, true>)
                               : (mode == 2 ? k_unweighted_tc2<2, false> : mode == 1 ? k_unweighted_tc2<1, false>
                                                                                    : k_unweighted_tc2<0, false>);
  kernel<<<grid, THREADS2, SMEM2_BYTES, s>>>(ops->mapP, ops->mapBh, ops->mapBl, c.end, c.scale, c.shift, c.n,
                                             c.biased ? 1 : 0, r, ops->r_int, ops->unit, tiles, n_tiles, n_samples, first,
                                             out, flag_below, ops->flag_u, flagged, n_flagged, ops->dbg, geo);
  return 1;
}

int launch_unweighted_fixup(const TcOperands* ops, const uint32_t* flagged, const unsigned long long* n_flagged,
                            unsigned long long* count_host, int64_t first, const Geometry& geo, float* out,
                            const Exceptions& ex, int num_sms, cudaStream_t s) {
  const auto kernel = ops->from_bits ? (geo.rect ? k_unweighted_fixup<Rows::kBits, true> : k_unweighted_fixup<Rows::kBits, false>)
                      : ops->i8      ? (geo.rect ? k_unweighted_fixup<Rows::kU8, true> : k_unweighted_fixup<Rows::kU8, false>)
                                     : (geo.rect ? k_unweighted_fixup<Rows::kBf16, true> : k_unweighted_fixup<Rows::kBf16, false>);
  const void* rows = ops->from_bits ? static_cast<const void*>(ops->bitsS) : ops->P;
  kernel<<<num_sms * 4, 256, 0, s>>>(rows, ops->kp, ops->len_col, flagged, n_flagged, count_host, first, out, ex, geo);
  return 1;
}

}  // namespace frc
