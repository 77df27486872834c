// Bottom-up branch embedding on the device (replaces abundanceToFlatNodes +
// normalizeFlatNodes, frcfrc/unifrac.go:32-67, for all samples at once).
//
// Layout: node-major.  Row v of the embedding holds node v for every sample,
// samples contiguous, so every kernel here reads and writes fully coalesced
// rows and a parent row is the sum (or OR) of its child rows.  Node ids are
// pre-order, so parent < child and "children in ascending id" is file order.
//
// Two embeddings:
//   fp64  E[B][ld]    exact subtree sums in the reference's order (child order
//                     from 0.0; totals ascending id) — feeds the exact pair
//                     kernel and, rounded once to fp32, the weighted kernel.
//   bits  P[B][nw]    presence only (unweighted): 1 bit per (node, sample),
//                     parent = OR of children.  32x less traffic than bytes.
// All of it is HBM-bound streaming; the level passes touch each element once
// as a write and once as a read (DESIGN.md, "embedding roofline").
#include "frc_internal.h"

namespace frc {

namespace {

constexpr int kThreads = 256;

// ---------------------------------------------------------------- fp64 path
// One warp per sample: scatter its CSR row into the leaf rows.
// Samples [s_base, s_end) go to columns [0, s_end - s_base) of E (a slab of the sample range).
// K (may be null): the key panels of the keyed -l tiles (launch_embed_f64 in frc_internal.h): a present leaf's key is its id.
__global__ void k_scatter_f64(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                              const double* __restrict__ val, int64_t s_base, int64_t s_end, double* E,
                              int64_t ld, int32_t* __restrict__ K, int32_t kp) {
  int64_t s = s_base + ((static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5);
  int lane = threadIdx.x & 31;
  if (s >= s_end) return;
  int64_t b = row_ptr[s], e = row_ptr[s + 1];
  for (int64_t k = b + lane; k < e; k += 32) {
    E[static_cast<int64_t>(col[k]) * ld + (s - s_base)] = val[k];
    if (K) K[((s >> 7) * kp + col[k]) * 128 + (s & 127)] = col[k];
  }
}

// One tree level: E[v] = ((0 + E[c1]) + E[c2]) + ... in child order.
// grid.x = nodes of the level, grid.y * blockDim.x * 2 covers the samples.
// K (may be null): key[v] = max over the children's keys (-1 = absent): the largest present leaf id under v.
__global__ void k_level_sum_f64(const int32_t* __restrict__ nodes, const int32_t* __restrict__ child_ptr,
                                const int32_t* __restrict__ child_idx, double* E, int64_t ld,
                                int32_t* __restrict__ K, int32_t kp, int64_t s_base) {
  int32_t v = nodes[blockIdx.x];
  int64_t s = (static_cast<int64_t>(blockIdx.y) * blockDim.x + threadIdx.x) * 2;
  if (s >= ld) return;  // ld is even (multiple of 128)
  int32_t cb = child_ptr[v], ce = child_ptr[v + 1];
  double2 acc = make_double2(0.0, 0.0);
  for (int32_t c = cb; c < ce; ++c) {
    const double2 x = *reinterpret_cast<const double2*>(E + static_cast<int64_t>(child_idx[c]) * ld + s);
    acc.x = __dadd_rn(acc.x, x.x);
    acc.y = __dadd_rn(acc.y, x.y);
  }
  *reinterpret_cast<double2*>(E + static_cast<int64_t>(v) * ld + s) = acc;
  if (K) {  // (s_base and s are even: the two samples sit side by side in one tile)
    const int64_t g = s_base + s;
    int32_t* const kt = K + (g >> 7) * kp * 128 + (g & 127);
    int2 key = make_int2(-1, -1);
    for (int32_t c = cb; c < ce; ++c) {
      const int2 x = *reinterpret_cast<const int2*>(kt + static_cast<int64_t>(child_idx[c]) * 128);
      key.x = max(key.x, x.x);
      key.y = max(key.y, x.y);
    }
    *reinterpret_cast<int2*>(kt + static_cast<int64_t>(v) * 128) = key;
  }
}

// total[s] = sum of E[v][s] over all v ascending (zeros add exactly nothing, so
// this equals the reference's sum over its id-sorted non-zero list).
__global__ void k_totals_f64(const double* __restrict__ E, int32_t n_nodes, int64_t ld,
                             int64_t n_samples, double* __restrict__ total) {
  int64_t s = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (s >= n_samples) return;
  double acc = 0.0;
  int32_t v = 0;
  for (; v + 8 <= n_nodes; v += 8) {
    double x[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) x[u] = E[static_cast<int64_t>(v + u) * ld + s];
#pragma unroll
    for (int u = 0; u < 8; ++u) acc = __dadd_rn(acc, x[u]);
  }
  for (; v < n_nodes; ++v) acc = __dadd_rn(acc, E[static_cast<int64_t>(v) * ld + s]);
  total[s] = acc;
}

__global__ void k_normalize_f64(double* E, int32_t n_nodes, int64_t ld, int64_t n_samples,
                                const double* __restrict__ total) {
  int64_t s = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (s >= n_samples) return;
  const double t = total[s];
  for (int32_t v = blockIdx.y; v < n_nodes; v += gridDim.y) {
    double x = E[static_cast<int64_t>(v) * ld + s];
    if (x != 0.0) E[static_cast<int64_t>(v) * ld + s] = __ddiv_rn(x, t);
  }
}

// Fast-path totals: partial[c][s] = sum of E[v][s] over the nodes of chunk c (any order will do off
// the exact path; the sequential ascending-id loop of k_totals_f64 is one dependent fp64 chain per
// sample and was latency-bound).  kMult (pruned tree, FRC_FLAG_PRUNE): node v stands for mult[v] original nodes
// that all hold E[v][s], and the default normaliser counts each of them.
template <bool kMult>
__global__ void k_totals_partial_f64(const double* __restrict__ E, int32_t n_nodes, int64_t ld,
                                     const double* __restrict__ mult, double* __restrict__ partial) {
  int64_t s = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (s >= ld) return;
  int32_t per = (n_nodes + gridDim.y - 1) / gridDim.y;
  int32_t v0 = blockIdx.y * per, v1 = min(n_nodes, v0 + per);
  auto term = [&](int32_t u) {
    const double x = E[static_cast<int64_t>(u) * ld + s];
    if constexpr (kMult) return mult[u] * x;
    else return x;
  };
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  int32_t v = v0;
  for (; v + 4 <= v1; v += 4) {
    a0 += term(v);
    a1 += term(v + 1);
    a2 += term(v + 2);
    a3 += term(v + 3);
  }
  for (; v < v1; ++v) a0 += term(v);
  partial[static_cast<int64_t>(blockIdx.y) * ld + s] = (a0 + a1) + (a2 + a3);
}

// Weighted operand + per-chunk partial denominators.
// grid.x covers samples, grid.y = node chunks; partial[chunk][s].  The proportion is x * (1/T) (one
// fp64 multiply; the exact path divides): fp64-pipe instructions are the scarce resource on B200
// and a division is ~30 of them.
__global__ void k_weighted_operand(const double* __restrict__ E, const double* __restrict__ length,
                                   int32_t n_nodes, int64_t ld, const double* __restrict__ total,
                                   int prescale, float* __restrict__ A, double* __restrict__ partial) {
  int64_t s = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (s >= ld) return;
  int32_t per = (n_nodes + gridDim.y - 1) / gridDim.y;
  int32_t v0 = blockIdx.y * per, v1 = min(n_nodes, v0 + per);
  const double t = total ? total[s] : 1.0;
  const double inv = t > 0.0 ? 1.0 / t : 0.0;  // empty sample: every x is 0
  double w = 0.0;
  for (int32_t v = v0; v < v1; ++v) {
    const double x = E[static_cast<int64_t>(v) * ld + s];
    const double a = total ? x * inv : x;
    const double la = length[v] * a;
    w += la;
    A[static_cast<int64_t>(v) * ld + s] = static_cast<float>(prescale ? la : a);
  }
  partial[static_cast<int64_t>(blockIdx.y) * ld + s] = w;
}

// Same, writing the tile-panel layout of the fast weighted path: Ap[tile][kp][128] (tile = 128
// consecutive samples), E being a slab of S = ld samples starting at sample s_base (a multiple of 128).
// Rows [n_nodes, kp) of the panels are zeroed by the last chunk.
__global__ void k_weighted_operand_panels(const double* __restrict__ E, const double* __restrict__ length,
                                          int32_t n_nodes, int32_t kp, int64_t ld, int64_t s_base,
                                          const double* __restrict__ total, int prescale,
                                          float* __restrict__ Ap, double* __restrict__ partial) {
  int64_t ls = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (ls >= ld) return;
  int32_t per = (n_nodes + gridDim.y - 1) / gridDim.y;
  int32_t v0 = blockIdx.y * per, v1 = min(n_nodes, v0 + per);
  const int64_t s = s_base + ls;
  float* dst = Ap + ((s >> 7) * kp) * 128 + (s & 127);
  const double t = total ? total[ls] : 1.0;
  const double inv = t > 0.0 ? 1.0 / t : 0.0;
  double w = 0.0;
  for (int32_t v = v0; v < v1; ++v) {
    const double x = E[static_cast<int64_t>(v) * ld + ls];
    const double a = total ? x * inv : x;
    const double la = length[v] * a;
    w += la;
    dst[static_cast<int64_t>(v) * 128] = static_cast<float>(prescale ? la : a);
  }
  if (blockIdx.y == gridDim.y - 1)
    for (int32_t v = n_nodes; v < kp; ++v) dst[static_cast<int64_t>(v) * 128] = 0.f;
  partial[static_cast<int64_t>(blockIdx.y) * ld + ls] = w;
}

__global__ void k_reduce_partials(const double* __restrict__ partial, int n_chunks, int64_t ld,
                                  int64_t n, double* __restrict__ out) {
  int64_t s = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (s >= n) return;
  double acc = 0.0;
  for (int c = 0; c < n_chunks; ++c) acc += partial[static_cast<int64_t>(c) * ld + s];
  out[s] = acc;
}

// ---------------------------------------------------------------- bits path
__global__ void k_scatter_bits(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                               int64_t n_samples, uint32_t* bits, int32_t nw) {
  int64_t s = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (s >= n_samples) return;
  int64_t b = row_ptr[s], e = row_ptr[s + 1];
  const uint32_t m = 1u << (s & 31);
  for (int64_t k = b + lane; k < e; k += 32)
    atomicOr(bits + static_cast<int64_t>(col[k]) * nw + (s >> 5), m);
}

__global__ void k_level_or(const int32_t* __restrict__ nodes, const int32_t* __restrict__ child_ptr,
                           const int32_t* __restrict__ child_idx, uint32_t* bits, int32_t nw) {
  int32_t v = nodes[blockIdx.x];
  int32_t w = blockIdx.y * blockDim.x + threadIdx.x;
  if (w >= nw) return;
  int32_t cb = child_ptr[v], ce = child_ptr[v + 1];
  uint32_t acc = 0;
  for (int32_t c = cb; c < ce; ++c) acc |= bits[static_cast<int64_t>(child_idx[c]) * nw + w];
  bits[static_cast<int64_t>(v) * nw + w] = acc;
}

// One warp per (word column, node chunk); lane = sample bit.
__global__ void k_presence_rowsum(const uint32_t* __restrict__ bits, int32_t n_nodes, int32_t nw,
                                  const double* __restrict__ lenq, double* __restrict__ partial) {
  int32_t w = blockIdx.x;
  int lane = threadIdx.x;
  int32_t per = (n_nodes + gridDim.y - 1) / gridDim.y;
  int32_t v0 = blockIdx.y * per, v1 = min(n_nodes, v0 + per);
  double acc = 0.0;
  for (int32_t v = v0; v < v1; ++v) {
    uint32_t word = bits[static_cast<int64_t>(v) * nw + w];
    if ((word >> lane) & 1u) acc += lenq[v];
  }
  partial[static_cast<int64_t>(blockIdx.y) * (static_cast<int64_t>(nw) * 32) + w * 32 + lane] = acc;
}

// bits -> three K-major bf16 operands.  Block = 64 nodes x 256 samples.
__global__ void __launch_bounds__(256)
k_expand_operands(const uint32_t* __restrict__ bits, int32_t n_nodes, int32_t nw, int32_t kp,
                  int64_t np, const uint16_t* __restrict__ len_hi, const uint16_t* __restrict__ len_lo,
                  uint16_t* __restrict__ P, uint16_t* __restrict__ Bh, uint16_t* __restrict__ Bl) {
  __shared__ uint32_t words[64][9];
  const int32_t v0 = blockIdx.x * 64;
  const int32_t w0 = blockIdx.y * 8;
  for (int idx = threadIdx.x; idx < 512; idx += 256) {
    int node = idx >> 3, word = idx & 7;
    uint32_t x = 0;
    if (v0 + node < n_nodes && w0 + word < nw)
      x = bits[static_cast<int64_t>(v0 + node) * nw + w0 + word];
    words[node][word] = x;
  }
  __syncthreads();
  const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int32_t va = v0 + 2 * lane, vb = va + 1;
  const uint32_t wa = words[2 * lane][wi], wb = words[2 * lane + 1][wi];
  const uint32_t ha = va < n_nodes ? len_hi[va] : 0, hb = vb < n_nodes ? len_hi[vb] : 0;
  const uint32_t la = va < n_nodes ? len_lo[va] : 0, lb = vb < n_nodes ? len_lo[vb] : 0;
  const int64_t s0 = (static_cast<int64_t>(w0) + wi) * 32;
#pragma unroll 4
  for (int it = 0; it < 32; ++it) {
    const int64_t s = s0 + it;
    if (s >= np) break;
    const uint32_t ba = (wa >> it) & 1u, bb = (wb >> it) & 1u;
    const int64_t o = s * kp + va;
    const uint32_t ma = 0u - ba, mb = 0u - bb;  // all-ones masks
    *reinterpret_cast<uint32_t*>(P + o) = (0x3F80u & ma) | ((0x3F80u & mb) << 16);
    *reinterpret_cast<uint32_t*>(Bh + o) = (ha & ma) | ((hb & mb) << 16);
    *reinterpret_cast<uint32_t*>(Bl + o) = (la & ma) | ((lb & mb) << 16);
  }
}


// ------------------------------------------------- fused presence embedding
// Samples are independent, so a CTA that owns one word column (32 samples) can run the
// entire bottom-up pass for them with block-level barriers only: its column of the
// presence matrix (one 32-bit word per node) lives in shared memory (or in a private
// global scratch column when the tree is too large for that).
//   phase 1  scatter the 32 CSR rows into leaf words (shared-memory atomics)
//   phase 2  per tree level: every node ORs its word into its parent
//   phase 3  publish the column in operand-column order: bitsT[w][k] = word(order[k])
// k_presence_rowsum_t and k_expand_operands_t then run with thousands of CTAs (writing the
// operands from these few hundred CTAs reached only 2.3 TB/s).
template <bool kSmem>
__global__ void __launch_bounds__(512)
k_embed_presence_fused(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                       int64_t n_samples, const int32_t* __restrict__ level_nodes,
                       const int32_t* __restrict__ level_parent, const int32_t* __restrict__ level_ptr,
                       int32_t height, int32_t n_nodes, int32_t kp, const int32_t* __restrict__ order,
                       uint32_t* __restrict__ node_scratch, uint32_t* __restrict__ bitsT, int32_t w0,
                       uint32_t* __restrict__ bitsS, const PeerPtrs peers) {
  extern __shared__ __align__(16) uint32_t smem_words[];
  __shared__ int32_t lptr[128];
  const int w = blockIdx.x + w0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t* colw = kSmem ? smem_words : node_scratch + static_cast<int64_t>(blockIdx.x) * n_nodes;

  for (int32_t v = tid; v < n_nodes; v += 512) colw[v] = 0u;
  if (tid < 128 && tid <= height + 1) lptr[tid] = level_ptr[tid];
  __syncthreads();
  // phase 1: two CSR rows per warp; both rows' bounds are fetched before either row's entries
  {
    int64_t rb[2], re[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int64_t s = static_cast<int64_t>(w) * 32 + warp + 16 * u;
      rb[u] = s < n_samples ? row_ptr[s] : 0;
      re[u] = s < n_samples ? row_ptr[s + 1] : 0;
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const uint32_t bit = 1u << (warp + 16 * u);
      for (int64_t k = rb[u] + lane; k < re[u]; k += 256) {  // eight loads in flight per lane
        int32_t c[8];
#pragma unroll
        for (int x = 0; x < 8; ++x) c[x] = k + 32 * x < re[u] ? col[k + 32 * x] : -1;
#pragma unroll
        for (int x = 0; x < 8; ++x)
          if (c[x] >= 0) atomicOr(colw + c[x], bit);
      }
    }
  }
  __syncthreads();
  // phase 2: every node ORs its (final) word into its parent, one tree level at a time from the
  // leaves up.  The kernel is latency-bound (157 CTAs at cfg2, DRAM 1.4 %): what a level costs is the
  // round trip of its index loads (level_nodes / level_parent, L2), so the loads are batched:
  //   wide levels (near the leaves): eight independent index pairs in flight per thread;
  //   narrow levels (<= 512 nodes, one per thread; level sizes never grow towards the root): the
  //   indices of EIGHT levels are fetched at once, then the eight levels run on shared memory alone
  //   (read, atomicOr, barrier) -- one load round trip per eight levels instead of one per level.
  auto lp = [&](int32_t h) { return h < 128 ? lptr[h] : level_ptr[h]; };
  int32_t h = 0;
  for (; h < height; ++h) {
    const int32_t b = lp(h), e = lp(h + 1);
    if (e - b <= 512) break;
    for (int32_t idx = b + tid; idx < e; idx += 4096) {
      int32_t n[8], p[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int32_t k = idx + u * 512;
        n[u] = k < e ? level_nodes[k] : -1;
        p[u] = k < e ? level_parent[k] : 0;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (n[u] >= 0) {
          const uint32_t x = colw[n[u]];
          if (x) atomicOr(colw + p[u], x);
        }
    }
    __syncthreads();
  }
  for (; h < height; h += 8) {
    int32_t n[8], p[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      n[u] = -1; p[u] = 0;
      if (h + u < height) {
        const int32_t k = lp(h + u) + tid;
        if (k < lp(h + u + 1)) { n[u] = level_nodes[k]; p[u] = level_parent[k]; }
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      if (h + u < height) {  // (block-uniform)
        if (n[u] >= 0) {
          const uint32_t x = colw[n[u]];
          if (x) atomicOr(colw + p[u], x);
        }
        __syncthreads();
      }
    }
  }
  // phase 3
  uint32_t* dst = bitsT + static_cast<int64_t>(w) * kp;
  if (peers.n > 0) {
    // fused all-gather: this CTA's column goes to the same place in every rank's bitsT, the remote
    // ones as plain stores over NVLink (visible to the peers once this kernel has completed; the
    // ranks meet at the small NCCL all-gather of the row sums before anyone reads bitsT)
    const int64_t at = static_cast<int64_t>(w) * kp;
#pragma unroll 4
    for (int32_t k = tid; k < kp; k += 512) {
      const int32_t v = order[k];
      const uint32_t x = v >= 0 ? colw[v] : 0u;
#pragma unroll
      for (int pr = 0; pr < 8; ++pr)
        if (pr < peers.n) peers.p[pr][at + k] = x;
    }
  } else {
#pragma unroll 8
    for (int32_t k = tid; k < kp; k += 512) {
      const int32_t v = order[k];
      dst[k] = v >= 0 ? colw[v] : 0u;
    }
  }
  // phase 3b (bits-fed pair kernel): the same bits sample-major, bitsS[s][kp / 32] (bit k % 32 of word
  // k / 32 = operand column k).  A warp transposes 128 columns x 32 samples with ballots; lane b then
  // holds the four words of sample b and stores them as one 16-byte piece of its row.
  if (bitsS != nullptr) {
    const int32_t words = kp >> 5;
    for (int32_t g = warp; g * 128 < kp; g += 16) {
      uint32_t wout[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int32_t v = order[g * 128 + u * 32 + lane];
        const uint32_t wv = v >= 0 ? colw[v] : 0u;
        uint32_t mine = 0;
#pragma unroll
        for (int b = 0; b < 32; ++b) {
          const uint32_t bal = __ballot_sync(0xffffffffu, (wv >> b) & 1u);
          if (lane == b) mine = bal;
        }
        wout[u] = mine;
      }
      const int64_t srow = static_cast<int64_t>(w) * 32 + lane;
      *reinterpret_cast<uint4*>(bitsS + srow * words + g * 4) = make_uint4(wout[0], wout[1], wout[2], wout[3]);
    }
  }
}

// partial[c][s] = sum over the columns of chunk c of lenq[k] * present(k, s): one warp per
// (word column, column chunk), lane = sample; words and lengths are read as 16-byte broadcasts.
__global__ void __launch_bounds__(32)
k_presence_rowsum_t(const uint32_t* __restrict__ bitsT, int32_t kp, int32_t per,
                    const double* __restrict__ lenq8, double* __restrict__ partial, int64_t ld, int32_t w0) {
  const int32_t w = blockIdx.x + w0, lane = threadIdx.x;
  const int32_t v0 = blockIdx.y * per, v1 = min(kp, v0 + per);  // per is a multiple of 8
  const uint32_t* col = bitsT + static_cast<int64_t>(w) * kp;
  double a0 = 0.0, a1 = 0.0;
  for (int32_t v = v0; v < v1; v += 8) {
    const uint4 wa = *reinterpret_cast<const uint4*>(col + v), wb = *reinterpret_cast<const uint4*>(col + v + 4);
    const double2 l0 = *reinterpret_cast<const double2*>(lenq8 + v), l1 = *reinterpret_cast<const double2*>(lenq8 + v + 2);
    const double2 l2 = *reinterpret_cast<const double2*>(lenq8 + v + 4), l3 = *reinterpret_cast<const double2*>(lenq8 + v + 6);
    a0 += ((wa.x >> lane) & 1u) ? l0.x : 0.0;
    a1 += ((wa.y >> lane) & 1u) ? l0.y : 0.0;
    a0 += ((wa.z >> lane) & 1u) ? l1.x : 0.0;
    a1 += ((wa.w >> lane) & 1u) ? l1.y : 0.0;
    a0 += ((wb.x >> lane) & 1u) ? l2.x : 0.0;
    a1 += ((wb.y >> lane) & 1u) ? l2.y : 0.0;
    a0 += ((wb.z >> lane) & 1u) ? l3.x : 0.0;
    a1 += ((wb.w >> lane) & 1u) ? l3.y : 0.0;
  }
  partial[static_cast<int64_t>(blockIdx.y) * ld + w * 32 + lane] = a0 + a1;
}

// u8 block floating point: the same row sums in integers.  q[k] = a*m < 2^24 and every aligned
// block of 128 columns has one power-of-two scale 2^col_exp, so a block sums exactly in 32 bits
// (128 * 2^24 = 2^31) and costs one integer add per (sample, column) instead of an fp64 add
// (fp64 instructions run at ~1/8 of the integer rate on B200); one fp64 multiply-add per block.
__global__ void __launch_bounds__(32)
k_presence_rowsum_u8(const uint32_t* __restrict__ bitsT, int32_t kp, int32_t per,
                     const uint32_t* __restrict__ qam, const int32_t* __restrict__ col_exp,
                     double* __restrict__ partial, int64_t ld, int32_t w0, int32_t e_min,
                     long long* __restrict__ r_int) {
  const int32_t w = blockIdx.x + w0, lane = threadIdx.x;
  const int32_t v0 = blockIdx.y * per, v1 = min(kp, v0 + per);  // per is a multiple of 128
  const uint32_t* col = bitsT + static_cast<int64_t>(w) * kp;
  const uint32_t m = 1u << lane;
  double tot = 0.0;
  unsigned long long tot_int = 0;  // the same sum, exact, in units of 2^e_min (integer mode of the pair kernel)
  for (int32_t blk = v0; blk < v1; blk += 128) {
    uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll 4
    for (int32_t v = blk; v < blk + 128; v += 8) {
      const uint4 wa = *reinterpret_cast<const uint4*>(col + v), wb = *reinterpret_cast<const uint4*>(col + v + 4);
      const uint4 qa = *reinterpret_cast<const uint4*>(qam + v), qb = *reinterpret_cast<const uint4*>(qam + v + 4);
      if (wa.x & m) a0 += qa.x;
      if (wa.y & m) a1 += qa.y;
      if (wa.z & m) a2 += qa.z;
      if (wa.w & m) a3 += qa.w;
      if (wb.x & m) a0 += qb.x;
      if (wb.y & m) a1 += qb.y;
      if (wb.z & m) a2 += qb.z;
      if (wb.w & m) a3 += qb.w;
    }
    const uint32_t sum = (a0 + a1) + (a2 + a3);  // < 2^31
    const int32_t e = col_exp[blk];
    if (r_int) tot_int += static_cast<unsigned long long>(sum) << (e - e_min);
    else tot = fma(ldexp(1.0, e), static_cast<double>(sum), tot);
  }
  // integer mode: straight into r_int with a 64-bit integer atomic (order-independent, so still
  // deterministic) -- no partial buffer, no reduce launch, no fp64
  if (r_int) atomicAdd(reinterpret_cast<unsigned long long*>(r_int) + w * 32 + lane, tot_int);
  else partial[static_cast<int64_t>(blockIdx.y) * ld + w * 32 + lane] = tot;
}

// Presence columns bitsT[nw][kp] (word w holds samples 32w..32w+31 of one operand column) -> the
// three K-major bf16 operands [np][kp].  Block = 64 columns x 256 samples; the only HBM-heavy kernel
// of the embedding stage: 3 * np * kp * 2 bytes written, each warp store covers 128 contiguous bytes.
__global__ void __launch_bounds__(256)
k_expand_operands_t(const uint32_t* __restrict__ bitsT, int32_t nw, int32_t kp,
                    int64_t np, const uint16_t* __restrict__ len_hi, const uint16_t* __restrict__ len_lo,
                    uint16_t* __restrict__ P, uint16_t* __restrict__ Bh, uint16_t* __restrict__ Bl,
                    const uint8_t* __restrict__ need) {
  __shared__ uint32_t words[8][64];
  const int32_t v0 = blockIdx.x * 64;
  const int32_t w0 = blockIdx.y * 8;
  const uint32_t nd = need ? need[blockIdx.y] : 3u;  // see k_expand_operands_u8
  if (nd == 0u) return;
  for (int idx = threadIdx.x; idx < 512; idx += 256) {
    int word = idx >> 6, node = idx & 63;
    uint32_t x = 0;
    if (w0 + word < nw) x = bitsT[static_cast<int64_t>(w0 + word) * kp + v0 + node];  // kp is padded: in range
    words[word][node] = x;
  }
  __syncthreads();
  const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int32_t va = v0 + 2 * lane;
  const uint2 wab = *reinterpret_cast<const uint2*>(&words[wi][2 * lane]);
  const uint32_t wa = wab.x, wb = wab.y;
  const uint32_t hab = *reinterpret_cast<const uint32_t*>(len_hi + va);  // len arrays are padded to kp
  const uint32_t lab = *reinterpret_cast<const uint32_t*>(len_lo + va);
  const int64_t s0 = (static_cast<int64_t>(w0) + wi) * 32;
#pragma unroll 4
  for (int it = 0; it < 32; ++it) {
    const int64_t s = s0 + it;
    if (s >= np) break;
    const uint32_t m = (0xFFFFu & (0u - ((wa >> it) & 1u))) | (0xFFFF0000u & (0u - ((wb >> it) & 1u)));
    const int64_t o = s * kp + va;
    if (nd & 1u) *reinterpret_cast<uint32_t*>(P + o) = 0x3F803F80u & m;
    if (nd & 2u) {
      *reinterpret_cast<uint32_t*>(Bh + o) = hab & m;
      *reinterpret_cast<uint32_t*>(Bl + o) = lab & m;
    }
  }
}

// Same for the u8 operands: block = 128 columns x 256 samples, 4 columns (one 32-bit store per
// operand) per thread and sample; 3 * np * kp bytes written.
// r_int != null (integer mode): the block also adds its share of the row sums r_s = sum_k q_k P_ks -- the
// words are in shared memory anyway, so bitsT is read ONCE by the whole stage (the separate row-sum pass
// cost 35 us at cfg2, a third of the stage).  Thread = sample for that part: q[k] = a*m < 2^24, 128 columns
// sum exactly in 32 bits, the block's one power-of-two scale becomes a shift and the partial sum goes to
// r_int with a 64-bit integer atomic (order-independent: deterministic).
__global__ void __launch_bounds__(256)
k_expand_operands_u8(const uint32_t* __restrict__ bitsT, int32_t nw, int32_t kp, int64_t np,
                     const uint8_t* __restrict__ qa, const uint8_t* __restrict__ qh,
                     const uint8_t* __restrict__ ql, uint8_t* __restrict__ A, uint8_t* __restrict__ Bh,
                     uint8_t* __restrict__ Bl, const uint8_t* __restrict__ need,
                     const uint32_t* __restrict__ qam, const int32_t* __restrict__ col_exp, int32_t e_min,
                     long long* __restrict__ r_int) {
  __shared__ __align__(16) uint32_t words[8][128];
  __shared__ __align__(16) uint32_t sq[128];
  const int32_t v0 = blockIdx.x * 128;
  const int32_t w0 = blockIdx.y * 8;
  // need[block of 256 samples]: bit 0 = these samples occur as columns (A), bit 1 = as rows (Bh, Bl)
  // of a tile of this rank's bands; a rank of a multi-GPU run skips the operands it never reads
  const uint32_t nd = need ? need[blockIdx.y] : 3u;
  if (nd == 0u) return;
  for (int idx = threadIdx.x; idx < 1024; idx += 256) {
    int word = idx >> 7, node = idx & 127;
    uint32_t x = 0;
    if (w0 + word < nw) x = bitsT[static_cast<int64_t>(w0 + word) * kp + v0 + node];
    words[word][node] = x;
  }
  if (r_int != nullptr && threadIdx.x < 128) sq[threadIdx.x] = qam[v0 + threadIdx.x];
  __syncthreads();
  const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int32_t va = v0 + 4 * lane;
  const uint4 w4 = *reinterpret_cast<const uint4*>(&words[wi][4 * lane]);
  const uint32_t a4 = *reinterpret_cast<const uint32_t*>(qa + va);
  const uint32_t h4 = *reinterpret_cast<const uint32_t*>(qh + va);
  const uint32_t l4 = *reinterpret_cast<const uint32_t*>(ql + va);
  const int64_t s0 = (static_cast<int64_t>(w0) + wi) * 32;
#pragma unroll 4
  for (int it = 0; it < 32; ++it) {
    const int64_t s = s0 + it;
    if (s >= np) break;
    const uint32_t bits = ((w4.x >> it) & 1u) | (((w4.y >> it) & 1u) << 8) | (((w4.z >> it) & 1u) << 16) |
                          (((w4.w >> it) & 1u) << 24);
    const uint32_t m = bits * 0xFFu;  // 0x01 -> 0xFF per byte
    const int64_t o = s * kp + va;
    if (nd & 1u) *reinterpret_cast<uint32_t*>(A + o) = a4 & m;
    if (nd & 2u) {
      *reinterpret_cast<uint32_t*>(Bh + o) = h4 & m;
      *reinterpret_cast<uint32_t*>(Bl + o) = l4 & m;
    }
  }
  if (r_int != nullptr) {
    // lane = sample of word wi; every read below is a shared-memory broadcast
    const uint32_t m = 1u << lane;
    uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
#pragma unroll 8
    for (int k = 0; k < 128; k += 4) {
      const uint4 w = *reinterpret_cast<const uint4*>(&words[wi][k]);
      const uint4 q = *reinterpret_cast<const uint4*>(&sq[k]);
      a0 += (w.x & m) ? q.x : 0u;
      a1 += (w.y & m) ? q.y : 0u;
      a2 += (w.z & m) ? q.z : 0u;
      a3 += (w.w & m) ? q.w : 0u;
    }
    const uint32_t sum = (a0 + a1) + (a2 + a3);  // < 2^31
    const int64_t s = s0 + lane;
    if (sum != 0u && s < np)
      atomicAdd(reinterpret_cast<unsigned long long*>(r_int) + s,
                static_cast<unsigned long long>(sum) << (col_exp[v0] - e_min));
  }
}

// One thread per operand column: x = len * 2^-e in [0, 2^24); search the 8-bit factor a for
// the 16-bit m = round(x / a) that brings a * m closest to x.
__global__ void k_quantize_lengths(const double* __restrict__ len_col, const int32_t* __restrict__ col_exp,
                                   int32_t kp, uint8_t* __restrict__ qa, uint8_t* __restrict__ qh,
                                   uint8_t* __restrict__ ql, uint32_t* __restrict__ qam,
                                   double* __restrict__ lenq, double* __restrict__ qerr) {
  const int32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= kp) return;
  const double len = len_col[k];
  const int e = col_exp[k];
  const double x = ldexp(len, -e);
  int best_a = 0, best_m = 0;
  if (len > 0.0) {
    double best = 1e300;
    int a0 = static_cast<int>(ceil(x / 65535.0));
    if (a0 < 1) a0 = 1;
    for (int a = a0; a <= 255; ++a) {
      double m = rint(x / static_cast<double>(a));
      if (m > 65535.0) continue;
      if (m < 1.0) m = 1.0;
      const double err = fabs(static_cast<double>(a) * m - x);
      if (err < best) { best = err; best_a = a; best_m = static_cast<int>(m); }
    }
    if (best_a == 0) { best_a = 255; best_m = 65535; }  // x beyond the representable range: saturate
  }
  qa[k] = static_cast<uint8_t>(best_a);
  qh[k] = static_cast<uint8_t>(best_m >> 8);
  ql[k] = static_cast<uint8_t>(best_m & 255);
  qam[k] = static_cast<uint32_t>(best_a) * static_cast<uint32_t>(best_m);
  const double q = ldexp(static_cast<double>(best_a) * static_cast<double>(best_m), e);
  lenq[k] = q;
  // Error budget of a distance d = U / V (U, V exact integer sums of quantised lengths): columns kept
  // to 2e-6 relative bound the error of U and of V by 2e-6 each; the absolute errors of the other
  // columns (small lengths merged into a chunk of larger ones, or an unlucky search) are summed
  // into A, and a pair with U < 1e6 * A (A could exceed 1e-6 of U, hence of V) is recomputed
  // exactly: |rel err d| <= 2 * (2e-6 + 1e-6) = 6e-6 for every pair that is not.
  // (summed in a FIXED order by k_sum_flag_u: the threshold must be the same bits on every run, rank and
  // device, or a pair sitting on it could take different routes and break "same bytes for any world")
  const double err = fabs(q - len);
  qerr[k] = err > 2e-6 * len ? 1e6 * err : 0.0;
}

// flag_u[0] = sum of qerr[0..kp) in a fixed order: thread t adds its strided columns in ascending order,
// then a fixed binary tree over the 1024 partial sums.
__global__ void __launch_bounds__(1024) k_sum_flag_u(const double* __restrict__ qerr, int32_t kp,
                                                     double* __restrict__ flag_u) {
  __shared__ double part[1024];
  double acc = 0.0;
  for (int32_t k = threadIdx.x; k < kp; k += 1024) acc += qerr[k];
  part[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (threadIdx.x < o) part[threadIdx.x] += part[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) flag_u[0] = part[0];
}

}  // namespace

// ------------------------------------------------------------------ launchers
int launch_embed_f64(const DevTree& t, const int32_t* level_ptr, const DevCsr& a, double* E,
                     int64_t ld, int64_t s_base, cudaStream_t s, int32_t* K, int32_t kp) {
  int launches = 0;
  cudaMemsetAsync(E, 0, sizeof(double) * ld * t.n_nodes, s);
  // the slab's key panels are one contiguous range (s_base and ld are multiples of 128): all absent
  if (K) cudaMemsetAsync(K + (s_base >> 7) * kp * 128, 0xFF, sizeof(int32_t) * ld * kp, s);
  const int64_t s_end = s_base + ld < a.n_samples ? s_base + ld : a.n_samples;
  if (s_end > s_base && a.nnz > 0) {
    int64_t threads = (s_end - s_base) * 32;
    k_scatter_f64<<<static_cast<unsigned>((threads + kThreads - 1) / kThreads), kThreads, 0, s>>>(
        a.row_ptr, a.col, a.val, s_base, s_end, E, ld, K, kp);
    ++launches;
  }
  for (int32_t h = 1; h <= t.height; ++h) {
    int32_t b = level_ptr[h], e = level_ptr[h + 1];
    if (e == b) continue;
    dim3 grid(static_cast<unsigned>(e - b), static_cast<unsigned>((ld / 2 + kThreads - 1) / kThreads));
    k_level_sum_f64<<<grid, kThreads, 0, s>>>(t.level_nodes + b, t.child_ptr, t.child_idx, E, ld, K, kp, s_base);
    ++launches;
  }
  return launches;
}

static int pick_chunks(int32_t n_nodes) {
  int c = n_nodes / 256;
  return c < 1 ? 1 : (c > 64 ? 64 : c);
}

int launch_totals_fast_f64(const double* E, int32_t n_nodes, int64_t ld, const double* mult, double* total,
                           double* scratch, cudaStream_t s) {
  const int chunks = pick_chunks(n_nodes);
  dim3 grid(static_cast<unsigned>((ld + kThreads - 1) / kThreads), chunks);
  if (mult) k_totals_partial_f64<true><<<grid, kThreads, 0, s>>>(E, n_nodes, ld, mult, scratch);
  else k_totals_partial_f64<false><<<grid, kThreads, 0, s>>>(E, n_nodes, ld, nullptr, scratch);
  k_reduce_partials<<<static_cast<unsigned>((ld + kThreads - 1) / kThreads), kThreads, 0, s>>>(scratch, chunks, ld, ld,
                                                                                             total);
  return 2;
}

int launch_totals_f64(const double* E, int32_t n_nodes, int64_t ld, int64_t n_samples, double* total,
                      cudaStream_t s) {
  if (n_samples == 0) return 0;
  k_totals_f64<<<static_cast<unsigned>((n_samples + 127) / 128), 128, 0, s>>>(E, n_nodes, ld,
                                                                               n_samples, total);
  return 1;
}

int launch_normalize_f64(double* E, int32_t n_nodes, int64_t ld, int64_t n_samples,
                         const double* total, cudaStream_t s) {
  if (n_samples == 0) return 0;
  dim3 grid(static_cast<unsigned>((n_samples + kThreads - 1) / kThreads),
            static_cast<unsigned>(min(n_nodes, 512)));
  k_normalize_f64<<<grid, kThreads, 0, s>>>(E, n_nodes, ld, n_samples, total);
  return 1;
}


int launch_weighted_operand(const double* E, const double* length, int32_t n_nodes, int32_t kp,
                            int64_t ld, int64_t n_samples, const double* total, bool prescale,
                            float* A, double* W, double* scratch, cudaStream_t s) {
  int chunks = pick_chunks(n_nodes);
  if (kp > n_nodes)
    cudaMemsetAsync(A + static_cast<int64_t>(n_nodes) * ld, 0, sizeof(float) * ld * (kp - n_nodes), s);
  dim3 grid(static_cast<unsigned>((ld + kThreads - 1) / kThreads), chunks);
  k_weighted_operand<<<grid, kThreads, 0, s>>>(E, length, n_nodes, ld, total, prescale ? 1 : 0, A,
                                               scratch);
  k_reduce_partials<<<static_cast<unsigned>((ld + kThreads - 1) / kThreads), kThreads, 0, s>>>(
      scratch, chunks, ld, ld, W);
  (void)n_samples;
  return 2;
}
int launch_weighted_operand_panels(const double* E, const double* length, int32_t n_nodes, int32_t kp,
                                   int64_t ld, int64_t s_base, const double* total, bool prescale, float* Ap,
                                   double* W, double* scratch, cudaStream_t s) {
  int chunks = pick_chunks(n_nodes);
  dim3 grid(static_cast<unsigned>((ld + kThreads - 1) / kThreads), chunks);
  k_weighted_operand_panels<<<grid, kThreads, 0, s>>>(E, length, n_nodes, kp, ld, s_base, total, prescale ? 1 : 0,
                                                      Ap, scratch);
  k_reduce_partials<<<static_cast<unsigned>((ld + kThreads - 1) / kThreads), kThreads, 0, s>>>(
      scratch, chunks, ld, ld, W + s_base);
  return 2;
}
int weighted_scratch_chunks(int32_t n_nodes) { return pick_chunks(n_nodes); }

int launch_embed_bits(const DevTree& t, const int32_t* level_ptr, const DevCsr& a, uint32_t* bits,
                      int32_t nw, cudaStream_t s) {
  int launches = 0;
  cudaMemsetAsync(bits, 0, sizeof(uint32_t) * static_cast<int64_t>(nw) * t.n_nodes, s);
  if (a.n_samples > 0 && a.nnz > 0) {
    int64_t threads = a.n_samples * 32;
    k_scatter_bits<<<static_cast<unsigned>((threads + kThreads - 1) / kThreads), kThreads, 0, s>>>(
        a.row_ptr, a.col, a.n_samples, bits, nw);
    ++launches;
  }
  for (int32_t h = 1; h <= t.height; ++h) {
    int32_t b = level_ptr[h], e = level_ptr[h + 1];
    if (e == b) continue;
    dim3 grid(static_cast<unsigned>(e - b), static_cast<unsigned>((nw + 127) / 128));
    k_level_or<<<grid, 128, 0, s>>>(t.level_nodes + b, t.child_ptr, t.child_idx, bits, nw);
    ++launches;
  }
  return launches;
}

int launch_presence_rowsum(const uint32_t* bits, int32_t n_nodes, int32_t nw, const double* lenq,
                           double* r, double* scratch, cudaStream_t s) {
  int chunks = pick_chunks(n_nodes);
  dim3 grid(nw, chunks);
  k_presence_rowsum<<<grid, 32, 0, s>>>(bits, n_nodes, nw, lenq, scratch);
  int64_t ld = static_cast<int64_t>(nw) * 32;
  k_reduce_partials<<<static_cast<unsigned>((ld + kThreads - 1) / kThreads), kThreads, 0, s>>>(
      scratch, chunks, ld, ld, r);
  return 2;
}

int launch_expand_operands(const uint32_t* bits, int32_t n_nodes, int32_t nw, int32_t kp, int64_t np,
                           const uint16_t* len_hi, const uint16_t* len_lo, uint16_t* P, uint16_t* Bh,
                           uint16_t* Bl, cudaStream_t s) {
  dim3 grid(kp / 64, static_cast<unsigned>((np + 255) / 256));
  k_expand_operands<<<grid, 256, 0, s>>>(bits, n_nodes, nw, kp, np, len_hi, len_lo, P, Bh, Bl);
  return 1;
}


// (nw = word columns this rank builds)
void embed_setup() {
  cudaFuncSetAttribute(k_embed_presence_fused<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
}

int64_t presence_node_scratch_words(int32_t n_nodes, int32_t nw) {
  return static_cast<size_t>(n_nodes) * 4 <= 200 * 1024 ? 0 : static_cast<int64_t>(n_nodes) * nw;
}

int launch_embed_presence_fused(const DevTree& t, const int32_t* level_ptr_dev, const DevCsr& a,
                                int32_t nw, int32_t w0, int32_t w_count, int32_t kp, const int32_t* order,
                                uint32_t* node_scratch, uint32_t* bitsT, uint32_t* bitsS, const PeerPtrs& peers,
                                cudaStream_t s) {
  (void)nw;
  const size_t smem = (static_cast<size_t>(t.n_nodes) * 4 + 15) & ~size_t(15);
  if (smem <= 200 * 1024) {  // (shared-memory attribute: embed_setup, once per device context)
    k_embed_presence_fused<true><<<w_count, 512, smem, s>>>(a.row_ptr, a.col, a.n_samples, t.level_nodes,
                                                            t.level_parent, level_ptr_dev, t.height, t.n_nodes, kp,
                                                            order, node_scratch, bitsT, w0, bitsS, peers);
  } else {
    k_embed_presence_fused<false><<<w_count, 512, 0, s>>>(a.row_ptr, a.col, a.n_samples, t.level_nodes,
                                                          t.level_parent, level_ptr_dev, t.height, t.n_nodes, kp,
                                                          order, node_scratch, bitsT, w0, bitsS, peers);
  }
  return 1;
}

int launch_presence_rowsum_t(const uint32_t* bitsT, int32_t n_nodes, int32_t nw, int32_t w0, int32_t w_count,
                             int32_t kp, const double* lenq, const uint32_t* qam, const int32_t* col_exp,
                             double* partial, double* r, int32_t e_min, long long* r_int, cudaStream_t s) {
  const int64_t np = static_cast<int64_t>(nw) * 32;
  const int chunks = pick_chunks(n_nodes);
  dim3 g(w_count, chunks);
  const int64_t s0 = static_cast<int64_t>(w0) * 32, ns = static_cast<int64_t>(w_count) * 32;
  if (qam) {
    const int32_t per = static_cast<int32_t>(round_up((kp + chunks - 1) / chunks, 128));
    if (r_int) cudaMemsetAsync(r_int + s0, 0, sizeof(long long) * ns, s);
    k_presence_rowsum_u8<<<g, 32, 0, s>>>(bitsT, kp, per, qam, col_exp, partial, np, w0, e_min, r_int);
    if (r_int) return 1;
  } else {
    const int32_t per = static_cast<int32_t>(round_up((kp + chunks - 1) / chunks, 8));
    k_presence_rowsum_t<<<g, 32, 0, s>>>(bitsT, kp, per, lenq, partial, np, w0);
  }
  k_reduce_partials<<<static_cast<unsigned>((ns + kThreads - 1) / kThreads), kThreads, 0, s>>>(partial + s0, chunks, np,
                                                                                              ns, r + s0);
  return 2;
}

int launch_expand_operands_t(const uint32_t* bitsT, int32_t nw, int32_t kp, int64_t np, bool i8,
                             const void* q0, const void* q1, const void* q2, void* P, void* Bh, void* Bl,
                             const uint8_t* need, const uint32_t* qam, const int32_t* col_exp, int32_t e_min,
                             long long* r_int, cudaStream_t s) {
  if (i8) {
    if (r_int) cudaMemsetAsync(r_int, 0, sizeof(long long) * np, s);
    dim3 grid(kp / 128, static_cast<unsigned>((np + 255) / 256));
    k_expand_operands_u8<<<grid, 256, 0, s>>>(bitsT, nw, kp, np, static_cast<const uint8_t*>(q0),
                                              static_cast<const uint8_t*>(q1), static_cast<const uint8_t*>(q2),
                                              static_cast<uint8_t*>(P), static_cast<uint8_t*>(Bh),
                                              static_cast<uint8_t*>(Bl), need, qam, col_exp, e_min, r_int);
  } else {
    (void)q0;
    dim3 grid(kp / 64, static_cast<unsigned>((np + 255) / 256));
    k_expand_operands_t<<<grid, 256, 0, s>>>(bitsT, nw, kp, np, static_cast<const uint16_t*>(q1),
                                             static_cast<const uint16_t*>(q2), static_cast<uint16_t*>(P),
                                             static_cast<uint16_t*>(Bh), static_cast<uint16_t*>(Bl), need);
  }
  return 1;
}

int launch_quantize_lengths(const double* len_col, const int32_t* col_exp, int32_t kp, uint8_t* qa,
                            uint8_t* qh, uint8_t* ql, uint32_t* qam, double* lenq, double* qerr, double* flag_u,
                            cudaStream_t s) {
  k_quantize_lengths<<<(kp + 127) / 128, 128, 0, s>>>(len_col, col_exp, kp, qa, qh, ql, qam, lenq, qerr);
  k_sum_flag_u<<<1, 1024, 0, s>>>(qerr, kp, flag_u);
  return 2;
}

}  // namespace frc
