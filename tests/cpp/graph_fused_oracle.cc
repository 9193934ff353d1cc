// The reference's inlier graph (computeTIMs + ScaleInliersSelector::solveForScale + Graph::addEdge,
// registration.cc:427-443, :512-551, :614-619) without materialising the n(n-1)/2 TIMs, which take 65 B per pair in
// orc_build_graph_bits (140 GB at n = 65 536).  For every pair i < j the same IEEE double sequence is evaluated in place:
// v_j - v_i, (x^2 + y^2) + z^2, sqrt, |d1 - d2| <= beta.  Rows run in parallel; the transposed bit and the degree of the
// later vertex are updated atomically.  Build with -ffp-contract=off (no FMA contraction), as the oracle is.
// TEST INFRASTRUCTURE ONLY (tests/oracle_fused.py compiles and loads it).
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

namespace {

inline double tim_norm(const double* v, int i, int j) {
  const double dx = v[3 * (size_t)j + 0] - v[3 * (size_t)i + 0];
  const double dy = v[3 * (size_t)j + 1] - v[3 * (size_t)i + 1];
  const double dz = v[3 * (size_t)j + 2] - v[3 * (size_t)i + 2];
  const double xx = dx * dx, yy = dy * dy, zz = dz * dz;
  double s = xx + yy;
  s = s + zz;
  return std::sqrt(s);
}

}  // namespace

extern "C" {

// bits (nullable, n * words_per_row uint64) must be zeroed by the caller; degree (nullable) is overwritten.
// Returns the edge count.
int64_t graph_bits_fused(const double* src, const double* dst, int n, double noise_bound, double cbar2, uint64_t* bits,
                         int words_per_row, int32_t* degree) {
  const double beta = 2 * noise_bound * std::sqrt(cbar2);
  std::vector<int32_t> deg((size_t)(n > 0 ? n : 1), 0);
  long long e = 0;
#pragma omp parallel for schedule(dynamic, 16) reduction(+ : e)
  for (int i = 0; i < n; ++i) {
    int32_t d = 0;
    for (int j = i + 1; j < n; ++j) {
      if (std::fabs(tim_norm(src, i, j) - tim_norm(dst, i, j)) <= beta) {
        ++d;
        __atomic_fetch_add(&deg[j], 1, __ATOMIC_RELAXED);
        if (bits) {
          __atomic_fetch_or(&bits[(size_t)i * words_per_row + (j >> 6)], 1ull << (j & 63), __ATOMIC_RELAXED);
          __atomic_fetch_or(&bits[(size_t)j * words_per_row + (i >> 6)], 1ull << (i & 63), __ATOMIC_RELAXED);
        }
      }
    }
    __atomic_fetch_add(&deg[i], d, __ATOMIC_RELAXED);
    e += d;
  }
  if (degree) std::memcpy(degree, deg.data(), sizeof(int32_t) * (size_t)n);
  return e;
}

}  // extern "C"
