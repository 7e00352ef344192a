// -*- C++ -*-
// oracle/shim_avx/packet8_sum.h — companion of the stand-in Eigen headers in oracle/shim (test infrastructure, NOT the
// product, NOT Eigen): DenseBase::sum() and norm() of dynamic-size float vectors on 8-float AVX packets, which is what
// Eigen >= 3.3 runs when the code is compiled with -mavx (Core/Redux.h, LinearVectorizedTraversal / NoUnrolling,
// Packet8f: two packet accumulators, packet_res0 + packet_res1, one odd packet, predux<Packet8f> = predux(lo + hi) with
// predux<Packet4f> = (a0+a2)+(a1+a3), scalar tail).  The stand-in's own sums use 4-float SSE packets.
//
// Used as a FORCED include ahead of every translation unit (g++ -include oracle/shim_avx/packet8_sum.h; recipe:
// oracle/shim_avx/ref_avx.mk), so that it is seen before the reference's sources include <Eigen/...>.  It includes
// the stand-in's Core with its SSE reduction template renamed, after declaring non-template overloads for the two
// loaders the stand-in's Lin<float>::sum() and norm() call it with: overload resolution prefers those, so every
// dynamic-size .sum() / .norm() takes the 8-float path and nothing else of the stand-in changes.  Fixed-size
// reductions (lpNorm<1> of the 6-vector, FullPivLU) do not go through redux_sum and keep their Packet4f form, as in
// Eigen (find_best_packet falls back to Packet4f for size 6).
#ifndef ICT_SHIM_PACKET8_SUM
#define ICT_SHIM_PACKET8_SUM

#include <cstddef>
#include <immintrin.h>

namespace Eigen {
namespace shim {
struct LoadPlain;
struct LoadProd;
inline float ict_redux_sum_p8(const LoadPlain& ld, std::ptrdiff_t size);
inline float ict_redux_sum_p8(const LoadProd& ld, std::ptrdiff_t size);
}  // namespace shim
}  // namespace Eigen

#define redux_sum ict_redux_sum_p8
#include "../shim/Eigen/Core"
#undef redux_sum

namespace Eigen {
namespace shim {

struct Load8Plain { const float* a; __m256 operator()(Index i) const { return _mm256_loadu_ps(a + i); } };
struct Load8Prod { const float* a; const float* b;
  __m256 operator()(Index i) const { return _mm256_mul_ps(_mm256_loadu_ps(a + i), _mm256_loadu_ps(b + i)); } };

inline float predux8(__m256 a) { return predux4(_mm_add_ps(_mm256_castps256_ps128(a), _mm256_extractf128_ps(a, 1))); }

// ld8: 8-float packet at index i; ld.s(i): the scalar element (tail, and sums shorter than one packet)
template <typename L8, typename L> inline float redux_sum_p8(const L8& ld8, const L& ld, Index size) {
  if (size == 0) return 0.0f;
  const Index packetSize = 8;
  const Index alignedSize2 = (size / (2 * packetSize)) * (2 * packetSize);
  const Index alignedSize = (size / packetSize) * packetSize;
  float res;
  if (alignedSize) {
    __m256 p0 = ld8(0);
    if (alignedSize > packetSize) {
      __m256 p1 = ld8(packetSize);
      for (Index index = 2 * packetSize; index < alignedSize2; index += 2 * packetSize) {
        p0 = _mm256_add_ps(p0, ld8(index));
        p1 = _mm256_add_ps(p1, ld8(index + packetSize));
      }
      p0 = _mm256_add_ps(p0, p1);
      if (alignedSize > alignedSize2) p0 = _mm256_add_ps(p0, ld8(alignedSize2));
    }
    res = predux8(p0);
    for (Index index = alignedSize; index < size; ++index) res = res + ld.s(index);
  } else {
    res = ld.s(0);
    for (Index index = 1; index < size; ++index) res = res + ld.s(index);
  }
  return res;
}

inline float ict_redux_sum_p8(const LoadPlain& ld, std::ptrdiff_t size) {
  const Load8Plain l8 = {ld.a};
  return redux_sum_p8(l8, ld, size);
}
inline float ict_redux_sum_p8(const LoadProd& ld, std::ptrdiff_t size) {
  const Load8Prod l8 = {ld.a, ld.b};
  return redux_sum_p8(l8, ld, size);
}

}  // namespace shim
}  // namespace Eigen

#endif  // ICT_SHIM_PACKET8_SUM
