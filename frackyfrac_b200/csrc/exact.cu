// Exact pair kernel: fp64, the reference's own arithmetic sequence.
//
// One thread per sample pair walks ALL node ids in ascending order over the
// dense fp64 embedding.  The reference (frcfrc/unifrac.go:144-205) walks the
// two id-sorted sparse lists with a merge-join; visiting the absent nodes as
// well changes nothing because they are skipped by the same membership tests,
// and every product and sum below is a separate IEEE operation (__dmul_rn /
// __dadd_rn: no FMA contraction, matching Go on amd64).  The result is
// bit-identical to the reference for any input, which is how the byte-exact
// testdata/*.want files pass through the GPU.  This is a device kernel, not a
// CPU fallback; it is selected for small problems (or on request) because it
// does O(pairs * nodes) fp64 work without tensor cores.
#include "frc_internal.h"
#include "wire.cuh"

namespace frc {
namespace {

template <bool kWeighted, bool kRect>
__global__ void k_exact_pairs(const double* __restrict__ E, const double* __restrict__ length,
                              int32_t n_nodes, int64_t ld, int64_t first, int64_t count,
                              double* __restrict__ out, const Geometry geo) {
  int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= count) return;
  int64_t i, j;
  pair_at<kRect>(first + t, geo, i, j);
  const double* ea = E + i;  // a = sample i (first of the pair, common.go:25)
  const double* eb = E + j;
  if (kWeighted) {
    double numer = 0.0, denom = 0.0;
    for (int32_t k = 0; k < n_nodes; ++k) {
      const double a = ea[static_cast<int64_t>(k) * ld];
      const double b = eb[static_cast<int64_t>(k) * ld];
      const bool pa = a > 0.0, pb = b > 0.0;
      if (!(pa || pb)) continue;
      const double l = length[k];
      if (pa && pb) {
        numer = __dadd_rn(numer, __dmul_rn(l, fabs(__dsub_rn(a, b))));
        denom = __dadd_rn(denom, __dmul_rn(l, __dadd_rn(a, b)));
      } else {
        const double x = __dmul_rn(l, pa ? a : b);
        numer = __dadd_rn(numer, x);
        denom = __dadd_rn(denom, x);
      }
    }
    out[t] = __ddiv_rn(numer, denom);
  } else {
    double result = 0.0, common = 0.0;
    for (int32_t k = 0; k < n_nodes; ++k) {
      const bool pa = ea[static_cast<int64_t>(k) * ld] > 0.0;
      const bool pb = eb[static_cast<int64_t>(k) * ld] > 0.0;
      if (pa && pb) common = __dadd_rn(common, length[k]);
      else if (pa || pb) result = __dadd_rn(result, length[k]);
    }
    out[t] = __ddiv_rn(result, __dadd_rn(result, common));
  }
}

// ---------------------------------------------------------------- flag -l as coded in the reference
// unifrac.go:108-110 skips normalizeFlatNodes when -l is given, and the id-sort lives inside it (:57): the
// lists then reach unifracDistWeighted (:174-205) in the order abundanceToFlatNodes appended them
// (post-order) and the merge-join compares ids of unsorted lists.  No reference test exercises it, but it
// is what `frcfrc -w -l` prints, so normalize = 0 reproduces it literally (normalize = 2 is the documented
// behaviour: sorted lists, raw values).
__global__ void k_list_counts(const double* __restrict__ E, int32_t n_nodes, int64_t ld, int64_t n_samples,
                              int64_t* __restrict__ list_ptr) {
  const int64_t s = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (s >= n_samples) return;
  int64_t c = 0;
  for (int32_t v = 0; v < n_nodes; ++v) c += E[static_cast<int64_t>(v) * ld + s] > 0.0 ? 1 : 0;
  list_ptr[s + 1] = c;
  if (s == 0) list_ptr[0] = 0;
}

// In-place inclusive scan of list_ptr[1..n] by one block (n is a sample count: <= 2^31).
__global__ void __launch_bounds__(1024) k_list_scan(int64_t* __restrict__ list_ptr, int64_t n) {
  __shared__ int64_t part[1024];
  const int64_t per = (n + 1023) / 1024;
  const int64_t b = 1 + threadIdx.x * per, e = min(n + 1, b + per);
  int64_t acc = 0;
  for (int64_t k = b; k < e; ++k) acc += list_ptr[k];
  part[threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    int64_t run = 0;
    for (int t = 0; t < 1024; ++t) { const int64_t x = part[t]; part[t] = run; run += x; }
  }
  __syncthreads();
  acc = part[threadIdx.x];
  for (int64_t k = b; k < e; ++k) { acc += list_ptr[k]; list_ptr[k] = acc; }
}

__global__ void k_list_fill(const double* __restrict__ E, const int32_t* __restrict__ post_order, int32_t n_nodes,
                            int64_t ld, int64_t n_samples, const int64_t* __restrict__ list_ptr,
                            int32_t* __restrict__ list_id, double* __restrict__ list_val) {
  const int64_t s = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (s >= n_samples) return;
  int64_t p = list_ptr[s];
  for (int32_t k = 0; k < n_nodes; ++k) {
    const int32_t v = post_order[k];
    const double x = E[static_cast<int64_t>(v) * ld + s];
    if (x > 0.0) { list_id[p] = v; list_val[p] = x; ++p; }  // unifrac.go:49-51
  }
}

// One thread per pair: the two-pointer walk of unifrac.go:178-203 over lists that are NOT id-sorted,
// every product and sum a separate IEEE operation.
template <bool kRect>
__global__ void k_unsorted_pairs(const int64_t* __restrict__ list_ptr, const int32_t* __restrict__ list_id,
                                 const double* __restrict__ list_val, const double* __restrict__ length,
                                 int64_t first, int64_t count, double* __restrict__ out, const Geometry geo) {
  const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (t >= count) return;
  int64_t si, sj;
  pair_at<kRect>(first + t, geo, si, sj);
  int64_t i = list_ptr[si], j = list_ptr[sj];
  const int64_t ie = list_ptr[si + 1], je = list_ptr[sj + 1];
  double numer = 0.0, denom = 0.0;
  while (i < ie && j < je) {
    const int32_t ia = list_id[i], ib = list_id[j];
    if (ia < ib) {
      const double x = __dmul_rn(length[ia], list_val[i]);
      numer = __dadd_rn(numer, x);
      denom = __dadd_rn(denom, x);
      ++i;
    } else if (ia > ib) {
      const double x = __dmul_rn(length[ib], list_val[j]);
      numer = __dadd_rn(numer, x);
      denom = __dadd_rn(denom, x);
      ++j;
    } else {
      const double l = length[ia], a = list_val[i], b = list_val[j];
      numer = __dadd_rn(numer, __dmul_rn(l, fabs(__dsub_rn(a, b))));
      denom = __dadd_rn(denom, __dmul_rn(l, __dadd_rn(a, b)));
      ++i;
      ++j;
    }
  }
  for (; i < ie; ++i) {
    const double x = __dmul_rn(length[list_id[i]], list_val[i]);
    numer = __dadd_rn(numer, x);
    denom = __dadd_rn(denom, x);
  }
  for (; j < je; ++j) {
    const double x = __dmul_rn(length[list_id[j]], list_val[j]);
    numer = __dadd_rn(numer, x);
    denom = __dadd_rn(denom, x);
  }
  out[t] = __ddiv_rn(numer, denom);
}

}  // namespace

// Pass 1 (list_id == nullptr): the list sizes, scanned into list_ptr[n_samples + 1]; the caller reads
// list_ptr[n_samples], allocates, and calls again with the arrays for pass 2.
int launch_postorder_lists(const double* E, const int32_t* post_order, int32_t n_nodes, int64_t ld, int64_t n_samples,
                           int64_t* list_ptr, int32_t* list_id, double* list_val, cudaStream_t s) {
  if (n_samples <= 0) return 0;
  const unsigned grid = static_cast<unsigned>((n_samples + 127) / 128);
  if (!list_id) {
    k_list_counts<<<grid, 128, 0, s>>>(E, n_nodes, ld, n_samples, list_ptr);
    k_list_scan<<<1, 1024, 0, s>>>(list_ptr, n_samples);
    return 2;
  }
  k_list_fill<<<grid, 128, 0, s>>>(E, post_order, n_nodes, ld, n_samples, list_ptr, list_id, list_val);
  return 1;
}

int launch_unsorted_pairs(const int64_t* list_ptr, const int32_t* list_id, const double* list_val,
                          const double* length, int64_t first, const Geometry& geo, int64_t count, double* out,
                          cudaStream_t s) {
  if (count <= 0) return 0;
  const auto kernel = geo.rect ? k_unsorted_pairs<true> : k_unsorted_pairs<false>;
  kernel<<<static_cast<unsigned>((count + 127) / 128), 128, 0, s>>>(list_ptr, list_id, list_val, length, first, count,
                                                                    out, geo);
  return 1;
}

int launch_exact_pairs(const double* E, const double* length, int32_t n_nodes, int64_t ld,
                       bool weighted, int64_t first, const Geometry& geo, int64_t count, double* out, cudaStream_t s) {
  if (count <= 0) return 0;
  unsigned grid = static_cast<unsigned>((count + 127) / 128);
  const auto kernel = weighted ? (geo.rect ? k_exact_pairs<true, true> : k_exact_pairs<true, false>)
                               : (geo.rect ? k_exact_pairs<false, true> : k_exact_pairs<false, false>);
  kernel<<<grid, 128, 0, s>>>(E, length, n_nodes, ld, first, count, out, geo);
  return 1;
}

}  // namespace frc
