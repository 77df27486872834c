// Device side of the flat pair index and of the fp32 output format (see wire.cu): how a pair kernel
// finds the samples of a flat pair index, and how the exact fix-up kernels store a recomputed distance
// into an fp32 band.
#pragma once
#include "frc_internal.h"

namespace frc {

// Flat pair index p -> samples (i, j), j < i, p = i(i-1)/2 + j (the inverse of tri()).  The fp64 square
// root is only a first guess; the two integer loops make the result exact for every p.
__device__ __forceinline__ void pair_of(int64_t p, int64_t& i, int64_t& j) {
  // largest i with i(i-1)/2 <= p
  int64_t g = static_cast<int64_t>((1.0 + sqrt(1.0 + 8.0 * static_cast<double>(p))) * 0.5);
  while (g * (g - 1) / 2 > p) --g;
  while ((g + 1) * g / 2 <= p) ++g;
  i = g;
  j = p - g * (g - 1) / 2;
}

// Flat pair index p -> samples (i, j) in the job's geometry (Geometry in frc_internal.h): the triangle's pair_of, or
// the query x reference block, p = (i - q0) * n_ref + j (query-major).
template <bool kRect>
__device__ __forceinline__ void pair_at(int64_t p, const Geometry& g, int64_t& i, int64_t& j) {
  if constexpr (kRect) {
    const int64_t q = p / g.n_ref;
    i = g.q0 + q;
    j = p - q * g.n_ref;
  } else {
    pair_of(p, i, j);
  }
}

// out[off] = float(d).  A value fp32 cannot carry to 2^-23 relative (underflow: |d| < 1.2e-38) is also
// appended to the band's exception list in mapped pinned host memory (rare: a system-scope atomic and two
// stores over PCIe).  0, NaN and infinities round-trip and are never exceptions.
__device__ __forceinline__ void store_fixed(float* __restrict__ out, uint32_t off, double d, int64_t first,
                                            const Exceptions& ex) {
  const float f = static_cast<float>(d);
  out[off] = f;
  if (fabs(static_cast<double>(f) - d) > fabs(d) * 0x1p-23) {
    const unsigned long long k = atomicAdd_system(ex.count, 1ULL);
    if (k < static_cast<unsigned long long>(ex.cap)) {
      ex.index[k] = first + off;
      ex.value[k] = d;
    }
  }
}

}  // namespace frc
