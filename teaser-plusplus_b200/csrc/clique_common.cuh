// Device helpers shared by the clique kernels of max_clique.cu (n <= kMaxN) and clique_large.cu (the front end of
// larger problems): adjacency rows, in-set degrees, block reductions.
#pragma once

#include "tzr_internal.cuh"

namespace tzr {
namespace {

__device__ __forceinline__ const uint32_t* adj_row32(const Batch& bt, int b, int v) {
  return reinterpret_cast<const uint32_t*>(bt.adj) + ((size_t)b * bt.n + v) * pitch32(bt.n);
}

// |N(u_k) ∩ S| for up to four vertices at once (k < cnt; unused slots alias u[0]): the row loads of the four
// vertices are independent, so one warp keeps 4x the memory-level parallelism of a one-vertex-at-a-time loop
// (these kernels are latency-bound on the L2/HBM-resident bitset, not bandwidth-bound).
__device__ __forceinline__ void inset_degree4(const Batch& bt, int b, const int u[4], int cnt, const uint32_t* S,
                                              int W, int lane, int d[4], int xlo = 0) {
  const uint32_t* r0 = adj_row32(bt, b, u[0]);
  const uint32_t* r1 = adj_row32(bt, b, cnt > 1 ? u[1] : u[0]);
  const uint32_t* r2 = adj_row32(bt, b, cnt > 2 ? u[2] : u[0]);
  const uint32_t* r3 = adj_row32(bt, b, cnt > 3 ? u[3] : u[0]);
  int d0 = 0, d1 = 0, d2 = 0, d3 = 0;
  for (int y = xlo + lane; y < W; y += 32) {  // words below xlo are known to be empty in S
    const uint32_t sw = S[y];
    const uint32_t a0 = r0[y], a1 = r1[y], a2 = r2[y], a3 = r3[y];
    d0 += __popc(a0 & sw);
    d1 += __popc(a1 & sw);
    d2 += __popc(a2 & sw);
    d3 += __popc(a3 & sw);
  }
  d[0] = __reduce_add_sync(0xffffffffu, d0);
  d[1] = __reduce_add_sync(0xffffffffu, d1);
  d[2] = __reduce_add_sync(0xffffffffu, d2);
  d[3] = __reduce_add_sync(0xffffffffu, d3);
}

// ---- block-level helpers ----------------------------------------------------------------------
// max-reduce a 64-bit key over the block; result valid in all threads. s_tmp: >= 33 entries.
__device__ unsigned long long block_max_u64(unsigned long long v, unsigned long long* s_tmp) {
  for (int o = 16; o; o >>= 1) {
    unsigned long long t = __shfl_xor_sync(0xffffffffu, v, o);
    v = t > v ? t : v;
  }
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (lane == 0) s_tmp[w] = v;
  __syncthreads();
  if (w == 0) {
    unsigned long long x = lane < nw ? s_tmp[lane] : 0ull;
    for (int o = 16; o; o >>= 1) {
      unsigned long long t = __shfl_xor_sync(0xffffffffu, x, o);
      x = t > x ? t : x;
    }
    if (lane == 0) s_tmp[32] = x;
  }
  __syncthreads();
  return s_tmp[32];
}

// exclusive scan of one int per thread over the block; returns exclusive prefix, *total = sum.
__device__ int block_excl_scan(int v, int* s_tmp /* >= 34 */, int* total) {
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  int inc = v;
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  __syncthreads();
  if (lane == 31) s_tmp[w] = inc;
  __syncthreads();
  if (w == 0) {
    int x = lane < nw ? s_tmp[lane] : 0;
    int xi = x;
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, xi, o);
      if (lane >= o) xi += t;
    }
    s_tmp[lane] = xi - x;  // exclusive warp offsets
    if (lane == 31) s_tmp[33] = xi;
  }
  __syncthreads();
  *total = s_tmp[33];
  return s_tmp[w] + inc - v;
}

}  // namespace
}  // namespace tzr
