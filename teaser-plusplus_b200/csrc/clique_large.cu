// Front end of the clique stage for problems with kMaxN < n <= kMaxNGraph correspondences.
//
// The clique kernels of max_clique.cu keep per-problem vertex sets of n bits (and, in the heuristic, 16-bit vertex
// lists) in shared memory, which limits them to n <= kMaxN.  Every clique of size >= L lies in the (L-1)-core of the
// graph (each member has L-1 neighbours inside it), so a large problem is reduced on the device to an ordinary one:
//
//   1 clique_heur_large_kernel  the greedy heuristic of clique_heur_kernel on the full graph (candidate set P in shared
//        memory, n/8 bytes; member list and in-P degrees in global scratch) -> L, the best of kHeurRoots greedy cliques
//   2 core_peel_kernel          level-synchronous peel of the HBM-resident bitset to the k-core: in every round each
//        surviving vertex with fewer than k surviving neighbours is removed and every removed vertex's row is read once
//        to decrement its neighbours' degrees (at most one pass over the bitset in total).  A persistent grid
//        (cooperative launch: every CTA resident) with a grid barrier per phase: no host round trip per round.
//   3 survivor_list_kernel      survivors in ascending order (block scan of the alive bitset)
//   4 compact_adj_kernel        the induced sub-graph, one warp per compacted row (one __ballot_sync per 32 columns)
//   5 launch_clique (max_clique.cu, unchanged) on the compacted batch, then clique_map_back_kernel
//
// Relabelling in ascending order preserves the lexicographic order of index sets, so the canonical maximum clique of
// the compacted graph is the canonical maximum clique of the full graph.
#include "clique_common.cuh"

namespace tzr {

namespace {

constexpr int kLargeHeurThreads = 512;
constexpr int kLargeThreads = 1024;   // one CTA per problem: selection, bisection steps, survivor lists, map back
constexpr int kPeelGridThreads = 256;

// valid-vertex mask of bitset word x of an n-vertex problem
__device__ __forceinline__ uint32_t valid_word(int x, int n) {
  const int base = x * 32;
  if (base >= n) return 0u;
  return base + 32 > n ? (1u << (n - base)) - 1u : 0xffffffffu;
}

// Barrier over every CTA of a cooperative launch.  bar[0] counts arrivals and is back to 0 when the barrier opens;
// bar[1] is the generation the waiting CTAs watch.  The fences order each CTA's global writes before its arrival and
// the other CTAs' writes before its departure.
__device__ __forceinline__ void grid_barrier(unsigned int* bar) {
  __syncthreads();
  if (threadIdx.x == 0) {
    volatile unsigned int* vb = bar;
    const unsigned int gen = vb[1];
    __threadfence();
    if (atomicAdd(bar, 1u) == gridDim.x - 1) {
      vb[0] = 0u;
      __threadfence();
      atomicAdd(bar + 1, 1u);
    } else {
      while (vb[1] == gen) __nanosleep(64);
    }
    __threadfence();
  }
  __syncthreads();
}

}  // namespace

size_t large_scratch_bytes(int B, int n) {
  const size_t Bn = (size_t)B * n, W32 = (size_t)pitch32(n);
  return (Bn * kHeurRoots * 2 + Bn + Bn) * 4 + (size_t)B * W32 * 4 + (size_t)B * 5 * 4 + 64 + 8 * 256;
}

LargeScratch large_scratch_carve(void* base, int B, int n) {
  const size_t Bn = (size_t)B * n, W32 = (size_t)pitch32(n);
  char* p = (char*)base;
  auto take = [&](size_t bytes) {
    char* q = p;
    p += (bytes + 255) & ~(size_t)255;
    return q;
  };
  LargeScratch s;
  s.hl = (int32_t*)take(Bn * kHeurRoots * 2 * 4);
  s.dcur = (int32_t*)take(Bn * 4);
  s.surv = (int32_t*)take(Bn * 4);
  s.dying = (uint32_t*)take((size_t)B * W32 * 4);
  s.k = (int32_t*)take((size_t)B * 4);
  s.lo = (int32_t*)take((size_t)B * 4);
  s.hi = (int32_t*)take((size_t)B * 4);
  s.nsurv = (int32_t*)take((size_t)B * 4);
  s.total = (unsigned int*)take(64);
  return s;
}

// =================================================================================================
// 1: greedy heuristic clique from the r-th highest-degree vertex (clique_heur_kernel's rules: universal vertices join
// together, candidates below half the best in-P degree are thinned out, otherwise the max-degree pivot joins).
// dynamic smem: P[W32] u32
// =================================================================================================
__global__ void __launch_bounds__(kLargeHeurThreads) clique_heur_large_kernel(Batch bt, LargeScratch ls) {
  const int r = blockIdx.x, b = blockIdx.y;
  const int n = bt.n, W = pitch32(n);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* P = reinterpret_cast<uint32_t*>(smem_raw);
  int32_t* list = ls.hl + ((size_t)b * kHeurRoots + r) * 2 * (size_t)n;
  int32_t* dl = list + n;
  __shared__ unsigned long long s_key[34];
  __shared__ int s_scan[34];
  __shared__ int s_chosen[kHeurRoots];
  __shared__ int s_csz, s_nuni;

  if (bt.kcore_final && bt.kcore_final[b]) return;  // KCORE_HEU: the innermost core is the answer
  const int32_t* deg = bt.deg + (size_t)b * n;
  int32_t* C = bt.hclq + ((size_t)b * kHeurRoots + r) * n;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;

  int root = -1;
  for (int round = 0; round <= r; ++round) {
    unsigned long long best = 0ull;
    for (int v = tid; v < n; v += blockDim.x) {
      bool excl = false;
      for (int q = 0; q < round; ++q) excl |= (s_chosen[q] == v);
      if (excl) continue;
      const unsigned long long key = ((unsigned long long)(unsigned)deg[v] << 32) | (unsigned)(0xffffffffu - (unsigned)v);
      best = key > best ? key : best;
    }
    best = block_max_u64(best, s_key);
    const int v = (int)(0xffffffffu - (unsigned)(best & 0xffffffffull));
    const int d = (int)(best >> 32);
    if (tid == 0) s_chosen[round] = (best == 0ull || d == 0) ? -1 : v;
    __syncthreads();
    root = s_chosen[round];
    if (root < 0) break;
  }
  if (root < 0) {
    if (tid == 0) bt.hsize[b * kHeurRoots + r] = 0;
    return;
  }
  if (tid == 0) {
    C[0] = root;
    s_csz = 1;
  }
  {
    const uint32_t* rr = adj_row32(bt, b, root);
    for (int x = tid; x < W; x += blockDim.x) P[x] = rr[x];
  }
  __syncthreads();

  for (int iter = 0; iter < n; ++iter) {
    // members of P in ascending order
    int cnt = 0;
    for (int x0 = 0; x0 < W; x0 += blockDim.x) {
      const int x = x0 + tid;
      const uint32_t wv = x < W ? P[x] : 0u;
      int tot = 0;
      int pos = cnt + block_excl_scan(__popc(wv), s_scan, &tot);
      for (uint32_t m = wv; m; m &= m - 1) list[pos++] = x * 32 + (__ffs(m) - 1);
      cnt += tot;
    }
    __syncthreads();
    if (cnt == 0) break;
    for (int k0 = wid * 4; k0 < cnt; k0 += nw * 4) {
      const int kc = min(4, cnt - k0);
      int u[4], d[4];
      for (int q = 0; q < 4; ++q) u[q] = list[k0 + (q < kc ? q : 0)];
      inset_degree4(bt, b, u, kc, P, W, lane, d);
      if (lane < kc) dl[k0 + lane] = lane == 0 ? d[0] : lane == 1 ? d[1] : lane == 2 ? d[2] : d[3];
    }
    if (tid == 0) s_nuni = 0;
    __syncthreads();
    unsigned long long best = 0ull;
    for (int k = tid; k < cnt; k += blockDim.x) {
      const int u = list[k], d = dl[k];
      if (d == cnt - 1) {
        C[atomicAdd(&s_csz, 1)] = u;
        atomicAdd(&s_nuni, 1);
        atomicAnd(&P[u >> 5], ~(1u << (u & 31)));
      } else {
        const unsigned long long key = ((unsigned long long)(unsigned)(d + 1) << 32) | (unsigned)(0xffffffffu - (unsigned)u);
        best = key > best ? key : best;
      }
    }
    best = block_max_u64(best, s_key);  // contains __syncthreads
    if (s_nuni == cnt) break;           // P was a clique
    const int thr = (int)(best >> 32) / 2;  // (pivot's in-P degree + 1) / 2
    __syncthreads();
    if (tid == 0) s_nuni = 0;
    __syncthreads();
    for (int k = tid; k < cnt; k += blockDim.x) {
      const int d = dl[k];
      if (d != cnt - 1 && d < thr) {
        const int u = list[k];
        atomicAnd(&P[u >> 5], ~(1u << (u & 31)));
        s_nuni = 1;
      }
    }
    __syncthreads();
    if (*(volatile int*)&s_nuni) continue;
    const int u = (int)(0xffffffffu - (unsigned)(best & 0xffffffffull));
    if (tid == 0) {
      const int pos = s_csz;
      C[pos] = u;
      s_csz = pos + 1;
    }
    const uint32_t* ru = adj_row32(bt, b, u);
    for (int x = tid; x < W; x += blockDim.x) P[x] &= ru[x];
    __syncthreads();
  }
  __syncthreads();
  if (tid == 0) bt.hsize[b * kHeurRoots + r] = s_csz;
}

// The best greedy clique (first root on ties, as clique_peel_kernel) becomes the incumbent L / clq of the full batch.
// PMC_EXACT peels to the (L-1)-core next (k = L-1); L <= 1 (no edge) needs no search: the solution is invalid either way.
__global__ void __launch_bounds__(kLargeThreads) clique_select_large_kernel(Batch bt, LargeScratch ls, int exact) {
  const int b = blockIdx.x, n = bt.n;
  if (bt.kcore_final && bt.kcore_final[b]) {
    if (threadIdx.x == 0) ls.k[b] = -1;
    return;
  }
  int L = 0, win = 0;
  for (int r = 0; r < kHeurRoots; ++r) {
    const int s = bt.hsize[b * kHeurRoots + r];
    if (s > L) {
      L = s;
      win = r;
    }
  }
  const int32_t* src = bt.hclq + ((size_t)b * kHeurRoots + win) * n;
  int32_t* dst = bt.clq + (size_t)b * n;
  for (int i = threadIdx.x; i < L; i += blockDim.x) dst[i] = src[i];
  if (threadIdx.x == 0) {
    bt.L[b] = L;
    bt.flags[b] = 0;
    ls.k[b] = (exact && L >= 2) ? L - 1 : -1;
  }
}

// =================================================================================================
// 2: peel every problem with k[b] >= 0 from the full vertex set to its k-core.  Cooperative launch (grid barrier).
// Output: bt.alive (survivors), ls.nsurv[b].
// =================================================================================================
__global__ void __launch_bounds__(kPeelGridThreads) core_peel_kernel(Batch bt, LargeScratch ls) {
  const int n = bt.n, W = pitch32(n), B = bt.B;
  const size_t nwords = (size_t)B * W;
  const size_t gtid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, gsz = (size_t)gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31;
  const size_t gwarp = gtid >> 5, nwarps = gsz >> 5;
  for (size_t i = gtid; i < nwords; i += gsz) {
    const int b = (int)(i / W);
    ls.dying[i] = 0u;
    if (ls.k[b] >= 0) bt.alive[i] = valid_word((int)(i - (size_t)b * W), n);
  }
  for (size_t i = gtid; i < (size_t)B * n; i += gsz)
    if (ls.k[i / n] >= 0) ls.dcur[i] = bt.deg[i];
  if (gtid < (size_t)B) ls.nsurv[gtid] = 0;
  grid_barrier(ls.total + 1);
  unsigned int removed = 0u;
  for (;;) {
    // phase A: survivors with fewer than k surviving neighbours are removed
    unsigned int cnt = 0u;
    for (size_t i = gtid; i < nwords; i += gsz) {
      const int b = (int)(i / W);
      const int k = ls.k[b];
      const uint32_t a = __ldcg(bt.alive + i);
      if (k < 0 || !a) continue;
      const int32_t* dc = ls.dcur + (size_t)b * n + (i - (size_t)b * W) * 32;
      uint32_t out = 0u;
      for (uint32_t m = a; m; m &= m - 1) {
        const int bit = __ffs(m) - 1;
        if (__ldcg(dc + bit) < k) out |= 1u << bit;
      }
      if (out) {
        bt.alive[i] = a & ~out;
        ls.dying[i] = out;
        cnt += __popc(out);
      }
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0 && cnt) atomicAdd(ls.total, cnt);
    grid_barrier(ls.total + 1);
    const unsigned int t = *(volatile unsigned int*)ls.total;
    if (t == removed) break;  // uniform: every thread reads the counter between the same two barriers
    removed = t;
    // phase B: one warp per word of removed vertices; each removed row is read once
    for (size_t i = gwarp; i < nwords; i += nwarps) {
      uint32_t m = __ldcg(ls.dying + i);
      if (!m) continue;
      const int b = (int)(i / W);
      const int x = (int)(i - (size_t)b * W);
      int32_t* dc = ls.dcur + (size_t)b * n;
      for (; m; m &= m - 1) {
        const uint32_t* row = adj_row32(bt, b, x * 32 + (__ffs(m) - 1));
        for (int y = lane; y < W; y += 32)
          for (uint32_t e = row[y]; e; e &= e - 1) atomicSub(dc + y * 32 + (__ffs(e) - 1), 1);
      }
      if (lane == 0) ls.dying[i] = 0u;
    }
    grid_barrier(ls.total + 1);
  }
  for (size_t i = gtid; i < nwords; i += gsz) {
    const int b = (int)(i / W);
    const int c = ls.k[b] >= 0 ? __popc(__ldcg(bt.alive + i)) : 0;
    if (c) atomicAdd(ls.nsurv + b, c);
  }
}

// =================================================================================================
// KCORE_HEU: maximum core number by bisection on k (graph.cc:66-81).  Each probe peels the full graph to the k-core.
// =================================================================================================
__global__ void __launch_bounds__(kLargeThreads) kcore_bisect_init_kernel(Batch bt, LargeScratch ls) {
  const int b = blockIdx.x, n = bt.n;
  __shared__ unsigned long long s_key[34];
  unsigned long long md = 0ull;
  for (int v = threadIdx.x; v < n; v += blockDim.x) md = max(md, (unsigned long long)(unsigned)bt.deg[(size_t)b * n + v]);
  const int maxdeg = (int)block_max_u64(md, s_key);
  if (threadIdx.x == 0) {
    const int lo = 0, hi = maxdeg + 1;  // the 0-core (every vertex) is non-empty, the (maxdeg+1)-core is empty
    ls.lo[b] = lo;
    ls.hi[b] = hi;
    ls.k[b] = hi - lo > 1 ? (lo + hi) >> 1 : -1;
  }
}

// after a probe: move the bound, pick the next probe; when the interval is closed the last step peels to lo (the
// innermost core, listed by survivor_list_kernel)
__global__ void kcore_bisect_step_kernel(LargeScratch ls, int B, int last) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  int lo = ls.lo[b], hi = ls.hi[b];
  const int k = ls.k[b];
  if (k >= 0) {
    if (ls.nsurv[b] > 0) lo = k;
    else hi = k;
  }
  ls.lo[b] = lo;
  ls.hi[b] = hi;
  ls.k[b] = last ? lo : (hi - lo > 1 ? (lo + hi) >> 1 : -1);
}

// graph.cc:66-69: threshold 1 disables the shortcut; otherwise max_core > int(thr * |V|) makes the innermost core the
// answer (ascending order)
__global__ void __launch_bounds__(kLargeThreads) kcore_finish_kernel(Batch bt, LargeScratch ls, double kcore_thr) {
  const int b = blockIdx.x, n = bt.n;
  const bool shortcut = (kcore_thr != 1.0) && (ls.lo[b] > (int)(kcore_thr * (double)n));
  if (!shortcut) {
    if (threadIdx.x == 0) bt.kcore_final[b] = 0;
    return;
  }
  const int cnt = ls.nsurv[b];
  const int32_t* src = ls.surv + (size_t)b * n;
  int32_t* dst = bt.clq + (size_t)b * n;
  for (int i = threadIdx.x; i < cnt; i += blockDim.x) dst[i] = src[i];
  if (threadIdx.x == 0) {
    bt.L[b] = cnt;
    bt.flags[b] = 0;
    bt.kcore_final[b] = 1;
  }
}

// =================================================================================================
// 3: survivors of the last peel in ascending order; problems with k[b] < 0 have none
// =================================================================================================
__global__ void __launch_bounds__(kLargeThreads) survivor_list_kernel(Batch bt, LargeScratch ls) {
  const int b = blockIdx.x, n = bt.n, W = pitch32(n);
  __shared__ int s_scan[34];
  if (ls.k[b] < 0) {
    if (threadIdx.x == 0) ls.nsurv[b] = 0;
    return;
  }
  const uint32_t* A = bt.alive + (size_t)b * W;
  int32_t* out = ls.surv + (size_t)b * n;
  int cnt = 0;
  for (int x0 = 0; x0 < W; x0 += blockDim.x) {
    const int x = x0 + threadIdx.x;
    const uint32_t wv = x < W ? A[x] : 0u;
    int tot = 0;
    int pos = cnt + block_excl_scan(__popc(wv), s_scan, &tot);
    for (uint32_t m = wv; m; m &= m - 1) out[pos++] = x * 32 + (__ffs(m) - 1);
    cnt += tot;
  }
  if (threadIdx.x == 0) ls.nsurv[b] = cnt;
}

// =================================================================================================
// 4: induced sub-graph of the survivors.  One warp per compacted row u': the bit of row surv[u'] at column surv[j'] for
// 32 survivors j' at a time becomes one compacted word (__ballot_sync); lane q keeps word 32t+q for a coalesced store.
// Rows and columns past the problem's survivor count are zero (isolated padding vertices).
// =================================================================================================
__global__ void __launch_bounds__(256) compact_adj_kernel(Batch bt, LargeScratch ls, Batch cb) {
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  const int u = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int nc = cb.n, Wc = pitch32(nc);
  if (u >= nc) return;
  const int cnt = ls.nsurv[b];
  const int32_t* sv = ls.surv + (size_t)b * bt.n;
  uint32_t* dst = reinterpret_cast<uint32_t*>(cb.adj) + ((size_t)b * nc + u) * Wc;
  const uint32_t* row = u < cnt ? adj_row32(bt, b, sv[u]) : nullptr;
  for (int x0 = 0; x0 < Wc; x0 += 32) {
    uint32_t mine = 0u;
    for (int q = 0; q < 32 && x0 + q < Wc; ++q) {
      const int j = (x0 + q) * 32 + lane;
      bool bit = false;
      if (row && j < cnt) {
        const int v = sv[j];
        bit = (row[v >> 5] >> (v & 31)) & 1u;
      }
      const uint32_t w = __ballot_sync(0xffffffffu, bit);
      if (lane == q) mine = w;
    }
    if (x0 + lane < Wc) dst[x0 + lane] = mine;
  }
}

// 5: the compacted search's clique in full indices; problems without survivors keep the greedy result (L <= 1)
__global__ void __launch_bounds__(kLargeThreads) clique_map_back_kernel(Batch bt, LargeScratch ls, Batch cb) {
  const int b = blockIdx.x;
  const int cnt = ls.nsurv[b];
  if (cnt == 0) return;
  const int L = cb.L[b];
  const int32_t* sv = ls.surv + (size_t)b * bt.n;
  const int32_t* cq = cb.clq + (size_t)b * cb.n;
  int32_t* dst = bt.clq + (size_t)b * bt.n;
  for (int i = threadIdx.x; i < L; i += blockDim.x) dst[i] = sv[cq[i]];
  if (threadIdx.x == 0) {
    bt.L[b] = L;
    bt.flags[b] = cb.flags[b];
    if (bt.rechecks) atomicMax(bt.mismatches + 15, (unsigned long long)cnt);  // debug counter 15 (flag 4)
  }
}

namespace {

int launch_core_peel(const Batch& bt, const LargeScratch& ls, cudaStream_t st, int num_sms) {
  static int occ_dev[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  int& occ = occ_dev[dev & 63];
  if (occ == 0 &&
      (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, core_peel_kernel, kPeelGridThreads, 0) != cudaSuccess ||
       occ < 1))
    return -1;
  if (cudaMemsetAsync(ls.total, 0, 3 * sizeof(unsigned int), st) != cudaSuccess) return -1;
  Batch a = bt;
  LargeScratch b = ls;
  void* args[] = {&a, &b};
  const unsigned grid = (unsigned)(occ * num_sms);
  return cudaLaunchCooperativeKernel((const void*)core_peel_kernel, dim3(grid), dim3(kPeelGridThreads), args, 0, st) ==
                 cudaSuccess
             ? 1
             : -1;
}

}  // namespace

int launch_clique_large_front(const Batch& bt, const LargeScratch& ls, int mode, double kcore_thr, cudaStream_t st,
                              int num_sms) {
  const int n = bt.n, B = bt.B;
  int launches = 0, rc;
  Batch hb = bt;
  if (mode == 2) {  // KCORE_HEU: max core by bisection; n < 2^17 needs at most 17 probes
    int probes = 0;
    while ((1 << probes) < n + 1) ++probes;
    kcore_bisect_init_kernel<<<B, kLargeThreads, 0, st>>>(bt, ls);
    ++launches;
    for (int i = 0; i <= probes; ++i) {
      if ((rc = launch_core_peel(bt, ls, st, num_sms)) < 0) return -1;
      kcore_bisect_step_kernel<<<(B + 127) / 128, 128, 0, st>>>(ls, B, i == probes ? 1 : 0);
      launches += rc + 1;
    }
    if ((rc = launch_core_peel(bt, ls, st, num_sms)) < 0) return -1;  // the innermost core
    survivor_list_kernel<<<B, kLargeThreads, 0, st>>>(bt, ls);
    kcore_finish_kernel<<<B, kLargeThreads, 0, st>>>(bt, ls, kcore_thr);
    launches += rc + 2;
  } else {
    hb.kcore_final = nullptr;
  }
  clique_heur_large_kernel<<<dim3(kHeurRoots, (unsigned)B), kLargeHeurThreads, (size_t)pitch32(n) * 4 + 16, st>>>(hb, ls);
  clique_select_large_kernel<<<B, kLargeThreads, 0, st>>>(hb, ls, mode == 0 ? 1 : 0);
  launches += 2;
  if (mode == 0) {
    if ((rc = launch_core_peel(bt, ls, st, num_sms)) < 0) return -1;
    survivor_list_kernel<<<B, kLargeThreads, 0, st>>>(bt, ls);
    launches += rc + 1;
  }
  return cudaPeekAtLastError() == cudaSuccess ? launches : -1;
}

void launch_clique_compact(const Batch& bt, const LargeScratch& ls, const Batch& cb, cudaStream_t st) {
  compact_adj_kernel<<<dim3((unsigned)((cb.n + 7) / 8), (unsigned)cb.B), 256, 0, st>>>(bt, ls, cb);
}

void launch_clique_map_back(const Batch& bt, const LargeScratch& ls, const Batch& cb, cudaStream_t st) {
  clique_map_back_kernel<<<bt.B, kLargeThreads, 0, st>>>(bt, ls, cb);
}

}  // namespace tzr
