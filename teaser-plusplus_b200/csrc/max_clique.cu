// Stage 2 of solve(): maximum clique of the inlier graph, on the packed adjacency bitset.
//
// Replaces teaser::MaxCliqueSolver::findMaxClique (teaser/src/graph.cc:12-125) and the PMC library
// calls behind it (pmc::pmc_graph::compute_cores, pmc::pmc_heu::search, pmc::pmcx_maxclique::
// search_dense — an un-vendored, un-pinned dependency, see DESIGN.md).  The result contract
// is the reference's: a maximum clique (PMC_EXACT), returned to solve() which sorts it
// (registration.cc:636).  The algorithm is a GPU re-design, not PMC's:
//
//   K1 clique_heur   (kHeurRoots CTAs / problem)  greedy lower bound from the top-degree vertices:
//        candidate set P = N(root); repeat { in-P degrees by bitset AND+popcount; all "universal"
//        vertices (adjacent to every other candidate) join the clique at once; otherwise the vertex
//        of largest in-P degree joins and P &= N(u) }.
//   K2 clique_peel   (1 CTA / problem)  picks the best heuristic clique (size L), then peels the
//        graph to its (L-1)-core (a member of a clique of size >= L has L-1 neighbours).  For
//        TEASER-style inlier graphs only the clique itself survives — the situation in which the
//        reference's `lb == ub` early-out (graph.cc:100-102) fires through PMC's k-core bound.
//   K3 clique_exact  (G CTAs / problem, one warp per root vertex)  branch and bound over the
//        survivors: root v owns the cliques whose smallest index is v (P = N(v) ∩ alive ∩ {u>v});
//        every node is reduced by in-P degree rules (universal vertices join at once, vertices that
//        cannot reach size L leave), bounded by greedy sequential colouring (branch only on vertices
//        whose colour reaches L - |C|), and expanded depth-first with an explicit stack in global
//        memory.  Branches are cut only when they cannot even TIE the incumbent, so every maximum
//        clique is enumerated and the lexicographically smallest index set is returned: the answer
//        is deterministic and independent of warp scheduling (when the maximum clique is unique —
//        the normal case — it is the reference's answer; PMC returns an unspecified one on ties).
//        The incumbent is shared through L[b] (atomic) + a spin lock for the vertex list/bitset.
//
// Bit-parallel integer work, L2-resident bitset: no tensor cores, no meaningful HBM roofline.
#include "clique_common.cuh"

namespace tzr {

namespace {

constexpr int kHeurThreads = 512;
constexpr int kPeelThreads = 1024;
constexpr int kExactThreads = 256;
#ifndef TZR_EXACT_MIN_BLOCKS
#define TZR_EXACT_MIN_BLOCKS 3  // CTAs per SM the exact kernel is compiled for (80 registers; 2 -> 128)
#endif
constexpr int kExactWarps = kExactThreads / 32;
#ifdef TZR_BLOCK_BOUND
constexpr int kBlkBatch = 16; // block colour bound: row words in flight per lane (x2, ping-pong)
#endif
constexpr int kYU = 2;        // colouring: bitset words per lane whose row loads are issued together
constexpr int kSpecCand = 8;  // colouring: candidates resolved per round trip to the bitset (see node_colour)

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

}  // namespace

// =================================================================================================
// K1: greedy heuristic clique from the r-th highest-degree vertex.
// dynamic smem: P[W32] u32 | list[n] u16 | dl[n] u16
// =================================================================================================
size_t clique_heur_smem(int n) { return (size_t)pitch32(n) * 4 + (size_t)n * 2 * 2 + 16; }

__global__ void __launch_bounds__(kHeurThreads) clique_heur_kernel(Batch bt) {
  const int r = blockIdx.x, b = blockIdx.y;
  const int n = bt.n, W = pitch32(n);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* P = reinterpret_cast<uint32_t*>(smem_raw);
  uint16_t* list = reinterpret_cast<uint16_t*>(P + W);
  uint16_t* dl = list + n;
  __shared__ unsigned long long s_key[34];
  __shared__ int s_scan[34];
  __shared__ int s_chosen[kHeurRoots];
  __shared__ int s_csz, s_nuni;

  if (bt.kcore_final && bt.kcore_final[b]) return;  // KCORE_HEU shortcut already produced the answer
  const int32_t* deg = bt.deg + (size_t)b * n;
  int32_t* C = bt.hclq + ((size_t)b * kHeurRoots + r) * n;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;

  // ---- root = (r+1)-th largest (degree, lowest index)
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
  if (root < 0) {  // fewer than r+1 non-isolated vertices
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
    // ---- enumerate members of P (ordered) into list[]
    int total = 0;
    {
      // each thread owns words tid, tid+T, ... ; W <= 1024 and T = 512 -> at most 2 words; generic loop
      int cnt_local = 0;
      for (int x = tid; x < W; x += blockDim.x) cnt_local += __popc(P[x]);
      // ordered enumeration needs word-major order: do it per "pass" of blockDim words
      int base_total = 0;
      for (int x0 = 0; x0 < W; x0 += blockDim.x) {
        const int x = x0 + tid;
        const uint32_t wv = x < W ? P[x] : 0u;
        int tot = 0;
        int off = block_excl_scan(__popc(wv), s_scan, &tot);
        uint32_t m = wv;
        int pos = base_total + off;
        while (m) {
          const int bit = __ffs(m) - 1;
          m &= m - 1;
          list[pos++] = (uint16_t)(x * 32 + bit);
        }
        base_total += tot;
      }
      total = base_total;
      (void)cnt_local;
    }
    __syncthreads();
    const int cnt = total;
    if (cnt == 0) break;
    // ---- in-P degrees: one warp per four members
    for (int k0 = wid * 4; k0 < cnt; k0 += nw * 4) {
      const int kc = min(4, cnt - k0);
      int u[4], d[4];
      for (int q = 0; q < 4; ++q) u[q] = list[k0 + (q < kc ? q : 0)];
      inset_degree4(bt, b, u, kc, P, W, lane, d);
      if (lane < kc) dl[k0 + lane] = (uint16_t)(lane == 0 ? d[0] : lane == 1 ? d[1] : lane == 2 ? d[2] : d[3]);
    }
    if (tid == 0) s_nuni = 0;
    __syncthreads();
    // ---- universal vertices join the clique together; best non-universal vertex is the pivot
    unsigned long long best = 0ull;
    for (int k = tid; k < cnt; k += blockDim.x) {
      const int u = list[k], d = dl[k];
      if (d == cnt - 1) {
        const int pos = atomicAdd(&s_csz, 1);
        C[pos] = u;
        atomicAdd(&s_nuni, 1);
        atomicAnd(&P[u >> 5], ~(1u << (u & 31)));
      } else {
        const unsigned long long key = ((unsigned long long)(unsigned)(d + 1) << 32) | (unsigned)(0xffffffffu - (unsigned)u);
        best = key > best ? key : best;
      }
    }
    best = block_max_u64(best, s_key);  // contains __syncthreads
    if (s_nuni == cnt) break;           // P was a clique
    // ---- thinning: candidates whose in-P degree is below half of the best one are dropped at once (they
    // linger otherwise, because the max-degree pivot rule favours vertices adjacent to them); only when
    // nothing can be dropped does the pivot join and P shrink to its neighbourhood.
    const int maxd = (int)(best >> 32) - 1;  // in-P degree of the pivot
    const int thr = (maxd + 1) / 2;
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
    // volatile: keeps the compiler from fusing this load with the adjacent s_csz into one LDS.64 executed by all
    // threads (harmless, but racecheck flags it against thread 0's s_csz store below)
    if (*(volatile int*)&s_nuni) continue;  // thinned: recompute degrees on the smaller P
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

// =================================================================================================
// K2: select the best heuristic clique, peel to the L-core.
// dynamic smem: A[W32] | Anew[W32]
// mode: 0 exact, 1 heuristic only
// =================================================================================================
size_t clique_peel_smem(int n) { return (size_t)pitch32(n) * 4 * 3 + 16; }

namespace {

// One peeling round over the vertices of S (shared-memory bitset): in-set degrees by AND+popcount (one warp per
// four vertices), optionally stored in dg[]; vertices with degree < thr are cleared in Sn.  Returns via shared
// counters: s_changed.  Block-wide; contains __syncthreads.
__device__ void peel_round(const Batch& bt, int b, const uint32_t* S, uint32_t* Sn, int W, int thr, int32_t* dg,
                           int* s_changed) {
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
  if (tid == 0) *s_changed = 0;
  __syncthreads();
  for (int x = wid; x < W; x += nw) {
    uint32_t m = S[x];  // warp-uniform
    while (m) {
      int u[4], bits[4], d[4], kc = 0;
      while (m && kc < 4) {
        bits[kc] = __ffs(m) - 1;
        m &= m - 1;
        u[kc] = x * 32 + bits[kc];
        ++kc;
      }
      for (int q = kc; q < 4; ++q) u[q] = u[0];
      inset_degree4(bt, b, u, kc, S, W, lane, d);
      if (lane == 0) {
        uint32_t clr = 0u;
        for (int q = 0; q < kc; ++q) {
          if (dg) dg[u[q]] = d[q];
          if (d[q] < thr) clr |= 1u << bits[q];
        }
        if (clr) {
          atomicAnd(&Sn[x], ~clr);
          *s_changed = 1;
        }
      }
    }
  }
  __syncthreads();
}

__device__ int block_popcount(const uint32_t* S, int W, int* s_cnt) {
  const int tid = threadIdx.x;
  if (tid == 0) *s_cnt = 0;
  __syncthreads();
  int c = 0;
  for (int x = tid; x < W; x += blockDim.x) c += __popc(S[x]);
  c = __reduce_add_sync(0xffffffffu, c);
  if ((tid & 31) == 0 && c) atomicAdd(s_cnt, c);
  __syncthreads();
  return *s_cnt;
}

// Peel S in place to its k-core (vertices with >= k neighbours inside the set).  Sn: scratch of W words.
__device__ void peel_to_core(const Batch& bt, int b, uint32_t* S, uint32_t* Sn, int W, int k, int* s_changed) {
  for (int x = threadIdx.x; x < W; x += blockDim.x) Sn[x] = S[x];
  __syncthreads();
  for (int round = 0; round < 256; ++round) {
    peel_round(bt, b, S, Sn, W, k, nullptr, s_changed);
    const int ch = *s_changed;
    for (int x = threadIdx.x; x < W; x += blockDim.x) S[x] = Sn[x];
    __syncthreads();
    if (!ch) break;
  }
}

}  // namespace

__global__ void __launch_bounds__(kPeelThreads) clique_peel_kernel(Batch bt, int mode) {
  const int b = blockIdx.x;
  const int n = bt.n, W = pitch32(n);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* A = reinterpret_cast<uint32_t*>(smem_raw);
  uint32_t* An = A + W;
  uint32_t* S = An + W;
  __shared__ int s_changed, s_cnt;
  __shared__ unsigned long long s_sum;
  __shared__ unsigned int s_min;
  const int tid = threadIdx.x;

  if (bt.kcore_final && bt.kcore_final[b]) {  // clq / L already hold the max-core vertex set (graph.cc:66-81)
    uint32_t* ag = bt.alive + (size_t)b * W;
    for (int x = tid; x < W; x += blockDim.x) ag[x] = 0u;
    if (tid == 0) {
      bt.root_ctr[b] = 0;
      bt.lock[b] = 0;
      bt.flags[b] = 0;
      bt.alive_cnt[b] = 0;
    }
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
  {
    const int32_t* src = bt.hclq + ((size_t)b * kHeurRoots + win) * n;
    int32_t* dst = bt.clq + (size_t)b * n;
    for (int i = tid; i < L; i += blockDim.x) dst[i] = src[i];
  }
  if (tid == 0) {
    bt.L[b] = L;
    bt.root_ctr[b] = 0;
    bt.lock[b] = 0;
    bt.flags[b] = 0;
    bt.t_start[b] = 0ull;
  }
  // incumbent as a bitset (canonical tie-break in the exact phase compares bitsets)
  uint32_t* bb = bt.best_bits + (size_t)b * W;
  {
    for (int x = tid; x < W; x += blockDim.x) A[x] = 0u;
    __syncthreads();
    const int32_t* srcq = bt.hclq + ((size_t)b * kHeurRoots + win) * n;
    for (int i = tid; i < L; i += blockDim.x) atomicOr(&A[srcq[i] >> 5], 1u << (srcq[i] & 31));
    __syncthreads();
    for (int x = tid; x < W; x += blockDim.x) bb[x] = A[x];
    __syncthreads();
  }
  uint32_t* alive_g = bt.alive + (size_t)b * W;
  if (mode != 0 || L == 0) {
    for (int x = tid; x < W; x += blockDim.x) alive_g[x] = 0u;
    if (tid == 0) bt.alive_cnt[b] = 0;
    return;
  }
  const int32_t* deg = bt.deg + (size_t)b * n;
  for (int x = tid; x < W; x += blockDim.x) {
    uint32_t m = 0;
    for (int k = 0; k < 32; ++k) {
      const int v = x * 32 + k;
      if (v < n && deg[v] >= L - 1) m |= 1u << k;
    }
    A[x] = m;
  }
  __syncthreads();
  peel_to_core(bt, b, A, An, W, L - 1, &s_changed);
  int alive = block_popcount(A, W, &s_cnt);

  // ---- second-chance heuristic.  If far more than the incumbent survives its own core bound, the root-based
  // greedy probably missed the dense part (e.g. a clique of ~1 % of the vertices planted in a 15 %-dense random
  // graph: no top-degree vertex belongs to it).  Global peeling: repeatedly drop every vertex whose degree inside
  // the surviving set is below the set's mean until the set is a clique.  A larger clique replaces the incumbent
  // and the core bound is re-applied; the exact phase then starts from a strong lower bound.
  if (alive > 4 * L + 64) {
    int32_t* dg = bt.hclq + (size_t)b * kHeurRoots * n;  // the heuristic candidates are no longer needed
    for (int x = tid; x < W; x += blockDim.x) {
      S[x] = A[x];
      An[x] = A[x];
    }
    __syncthreads();
    int cnt = alive;
    bool is_clique = false;
    for (int round = 0; round < 4096 && cnt > L; ++round) {
      peel_round(bt, b, S, An, W, -1, dg, &s_changed);  // degrees only (threshold -1 removes nothing)
      unsigned long long sum = 0ull, mn = ~0ull;
      for (int x = tid; x < W; x += blockDim.x) {
        uint32_t m = S[x];
        while (m) {
          const int v = x * 32 + (__ffs(m) - 1);
          m &= m - 1;
          sum += (unsigned)dg[v];
          mn = min(mn, (unsigned long long)(unsigned)dg[v]);
        }
      }
      // block reductions of the degree sum and minimum
      if (tid == 0) {
        s_sum = 0ull;
        s_min = 0xffffffffu;
      }
      __syncthreads();
      sum = __reduce_add_sync(0xffffffffu, (unsigned)(sum & 0xffffffffu)) +
            ((unsigned long long)__reduce_add_sync(0xffffffffu, (unsigned)(sum >> 32)) << 32);
      const unsigned mnw = __reduce_min_sync(0xffffffffu, (unsigned)min(mn, 0xffffffffull));
      if ((tid & 31) == 0) {
        atomicAdd(&s_sum, sum);
        atomicMin(&s_min, mnw);
      }
      __syncthreads();
      const unsigned long long tot = s_sum;
      const int dmin = (int)s_min;
      if (dmin == cnt - 1) {
        is_clique = true;
        break;
      }
      // far from a clique (mean degree < 3/4 of cnt-1): drop every vertex below the mean degree; close to one:
      // drop only the minimum-degree vertices (the mean rule would start cutting clique members).
      const bool coarse = tot * 4ull < 3ull * (unsigned long long)cnt * (unsigned long long)(cnt - 1);
      int removed_any = 0;
      for (int x = tid; x < W; x += blockDim.x) {
        uint32_t m = S[x], keep = m;
        while (m) {
          const int bit = __ffs(m) - 1;
          m &= m - 1;
          const unsigned dv = (unsigned)dg[x * 32 + bit];
          const bool drop = coarse ? ((unsigned long long)dv * (unsigned long long)cnt < tot) : ((int)dv == dmin);
          if (drop) keep &= ~(1u << bit);
        }
        if (keep != S[x]) removed_any = 1;
        An[x] = keep;
      }
      removed_any = __syncthreads_or(removed_any);
      if (!removed_any) {
        if (tid == 0) {
          for (int x = 0; x < W; ++x)
            if (An[x]) {
              An[x] &= An[x] - 1;  // clear the lowest set bit
              break;
            }
        }
        __syncthreads();
      }
      for (int x = tid; x < W; x += blockDim.x) S[x] = An[x];
      __syncthreads();
      cnt = block_popcount(S, W, &s_cnt);
    }
    if (is_clique) {
      // greedy extension: every alive vertex adjacent to ALL of S may still join (the peeling above is lossy);
      // CN = A ∩ (∩_{s∈S} N(s)); then repeatedly take the lowest vertex of CN and intersect with its row.
      for (int x = tid; x < W; x += blockDim.x) An[x] = A[x] & ~S[x];
      __syncthreads();
      for (int x0 = 0; x0 < W; ++x0) {
        uint32_t m = S[x0];  // uniform
        while (m) {
          const int sv = x0 * 32 + (__ffs(m) - 1);
          m &= m - 1;
          const uint32_t* rs = adj_row32(bt, b, sv);
          for (int x = tid; x < W; x += blockDim.x) An[x] &= rs[x];
        }
      }
      __syncthreads();
      __shared__ int s_pick;
      for (int it = 0; it < n; ++it) {
        if (tid == 0) {
          s_pick = -1;
          for (int x = 0; x < W; ++x)
            if (An[x]) {
              s_pick = x * 32 + (__ffs(An[x]) - 1);
              break;
            }
        }
        __syncthreads();
        const int v = s_pick;
        if (v < 0) break;
        const uint32_t* rv = adj_row32(bt, b, v);
        for (int x = tid; x < W; x += blockDim.x) An[x] &= rv[x];
        if (tid == 0) S[v >> 5] |= 1u << (v & 31);
        __syncthreads();
      }
      cnt = block_popcount(S, W, &s_cnt);
    }
    if (is_clique && cnt > L) {
      // new incumbent: S
      L = cnt;
      if (tid == 0) {
        int32_t* dst = bt.clq + (size_t)b * n;
        int k = 0;
        for (int x = 0; x < W; ++x) {
          uint32_t m = S[x];
          while (m) {
            dst[k++] = x * 32 + (__ffs(m) - 1);
            m &= m - 1;
          }
        }
        bt.L[b] = L;
      }
      for (int x = tid; x < W; x += blockDim.x) bb[x] = S[x];
      __syncthreads();
      // re-apply the (L-1)-core bound with the stronger L (A is still a superset of the new core)
      for (int x = tid; x < W; x += blockDim.x) {
        uint32_t m = A[x], keep = m;
        while (m) {
          const int bit = __ffs(m) - 1;
          m &= m - 1;
          if (deg[x * 32 + bit] < L - 1) keep &= ~(1u << bit);
        }
        A[x] = keep;
      }
      __syncthreads();
      peel_to_core(bt, b, A, An, W, L - 1, &s_changed);
      alive = block_popcount(A, W, &s_cnt);
    }
  }
  // If exactly L vertices survive the (L-1)-core bound they ARE the incumbent clique (its members always survive):
  // no other clique of size >= L can exist, the maximum clique is unique and proven — the exact phase is skipped.
  // This is the GPU counterpart of the reference's `lb == ub` early return (graph.cc:100-102).
  if (alive == L) alive = 0;
  for (int x = tid; x < W; x += blockDim.x) alive_g[x] = alive ? A[x] : 0u;
  if (tid == 0) bt.alive_cnt[b] = alive;
}

// =================================================================================================
// K0 (KCORE_HEU mode only): maximum core number by bisection on k, each probe peeling the current core to its
// k-core with in-set degrees (k-cores are nested, so a probe above `lo` starts from the lo-core).  If
// max_core > threshold * n the vertices of the innermost core are the answer (graph.cc:66-81: "remove all nodes
// with core number less than max core number"); otherwise the heuristic kernels run as in PMC_HEU mode.
// dynamic smem: A[W] | T[W] | Tn[W]
// =================================================================================================
size_t clique_kcore_smem(int n) { return (size_t)pitch32(n) * 4 * 3 + 16; }

__global__ void __launch_bounds__(kPeelThreads) clique_kcore_kernel(Batch bt, double kcore_thr) {
  const int b = blockIdx.x;
  const int n = bt.n, W = pitch32(n);
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* A = reinterpret_cast<uint32_t*>(smem_raw);
  uint32_t* T = A + W;
  uint32_t* Tn = T + W;
  __shared__ unsigned long long s_key[34];
  __shared__ int s_changed, s_cnt;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
  const int32_t* deg = bt.deg + (size_t)b * n;
  unsigned long long md = 0ull;
  for (int v = tid; v < n; v += blockDim.x) md = max(md, (unsigned long long)(unsigned)deg[v]);
  const int maxdeg = (int)block_max_u64(md, s_key);
  for (int x = tid; x < W; x += blockDim.x) {
    uint32_t m = 0xffffffffu;
    const int base = x * 32;
    if (base >= n) m = 0u;
    else if (base + 32 > n) m = (1u << (n - base)) - 1u;
    A[x] = m;
  }
  __syncthreads();
  int lo = 0, hi = maxdeg + 1;  // lo-core (= A) is non-empty, hi-core is empty
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    for (int x = tid; x < W; x += blockDim.x) {
      T[x] = A[x];
      Tn[x] = A[x];
    }
    __syncthreads();
    for (int round = 0; round < n + 1; ++round) {
      if (tid == 0) s_changed = 0;
      __syncthreads();
      for (int x = wid; x < W; x += nw) {
        uint32_t m = T[x];
        while (m) {
          int u[4], bits[4], d[4], kc = 0;
          while (m && kc < 4) {
            bits[kc] = __ffs(m) - 1;
            m &= m - 1;
            u[kc] = x * 32 + bits[kc];
            ++kc;
          }
          for (int q = kc; q < 4; ++q) u[q] = u[0];
          inset_degree4(bt, b, u, kc, T, W, lane, d);
          if (lane == 0) {
            uint32_t clr = 0u;
            for (int q = 0; q < kc; ++q)
              if (d[q] < mid) clr |= 1u << bits[q];
            if (clr) {
              atomicAnd(&Tn[x], ~clr);
              s_changed = 1;
            }
          }
        }
      }
      __syncthreads();
      const int ch = s_changed;
      for (int x = tid; x < W; x += blockDim.x) T[x] = Tn[x];
      __syncthreads();
      if (!ch) break;
    }
    if (tid == 0) s_cnt = 0;
    __syncthreads();
    int c = 0;
    for (int x = tid; x < W; x += blockDim.x) c += __popc(T[x]);
    c = __reduce_add_sync(0xffffffffu, c);
    if (lane == 0 && c) atomicAdd(&s_cnt, c);
    __syncthreads();
    if (s_cnt > 0) {
      lo = mid;
      for (int x = tid; x < W; x += blockDim.x) A[x] = T[x];
    } else {
      hi = mid;
    }
    __syncthreads();
  }
  const int max_core = lo;
  // graph.cc:66-69: threshold != 1 short-circuits; compare against int(thr * |V|)
  const bool shortcut = (kcore_thr != 1.0) && (max_core > (int)(kcore_thr * (double)n));
  if (!shortcut) {
    if (tid == 0) bt.kcore_final[b] = 0;
    return;
  }
  // emit the innermost core's vertices in ascending order (one thread: n <= 32768, off the hot path)
  if (tid == 0) {
    int32_t* dst = bt.clq + (size_t)b * n;
    int cnt = 0;
    for (int x = 0; x < W; ++x) {
      uint32_t m = A[x];
      while (m) {
        const int bit = __ffs(m) - 1;
        m &= m - 1;
        dst[cnt++] = x * 32 + bit;
      }
    }
    bt.L[b] = cnt;
    bt.kcore_final[b] = 1;
  }
}

// =================================================================================================
// K3: exact branch and bound, one warp per root.
// dynamic smem per warp: Pc[W] | Q[W] | R[W] | Bs[W]
// =================================================================================================
size_t clique_exact_smem(int n) { return ((size_t)pitch32(n) * 4 + kSpecCand) * 4 * kExactWarps + 16; }

namespace {

__device__ __forceinline__ int warp_popc(const uint32_t* bits, int W, int lane, int xlo = 0) {
  int c = 0;
  for (int x = xlo + lane; x < W; x += 32) c += __popc(bits[x]);
  return __reduce_add_sync(0xffffffffu, c);
}

// lowest set bit at word index >= xstart, or -1.  *xfound = word index.
__device__ __forceinline__ int warp_first_bit(const uint32_t* bits, int W, int lane, int xstart, int* xfound) {
  for (int base = xstart & ~31; base < W; base += 32) {
    const int x = base + lane;
    const uint32_t w = (x < W && x >= xstart) ? bits[x] : 0u;
    const unsigned nz = __ballot_sync(0xffffffffu, w != 0u);
    if (nz) {
      const int srcl = __ffs(nz) - 1;
      const uint32_t ww = __shfl_sync(0xffffffffu, w, srcl);
      *xfound = base + srcl;
      return (base + srcl) * 32 + (__ffs(ww) - 1);
    }
  }
  *xfound = W;
  return -1;
}

struct WarpCtx {
  unsigned long long* cnt;  // debug counters (nullptr unless debug flag 4): see tzr_ctx_debug_counters
  const Batch* bt;
  int b, n, W, lane;
  uint32_t *Pc, *Q, *R, *Bs;     // shared memory (this warp); words below xlo are never read nor written
  int* cand;                     // shared memory (this warp): kSpecCand candidate vertices of the colouring
  int blk;                       // vertices per block of the block colour bound (0: W too small for it)
  int bb_col, bb_vtx;            // colours / vertices of the blocks coloured so far in this problem (predicts the bound)
  uint32_t* stack;               // global: level d -> P at stack + d*2W, B at stack + d*2W + W
  int32_t* cv;                   // global: current clique
  int32_t* centry;               // global: clique size at entry of level d
  volatile int32_t* Lp;
  int strict;                    // 1 after a Nemhauser-Trotter reduction: only cliques that BEAT the incumbent matter (the
                                 // canonical tie-break is already forfeited, and dense graphs have astronomically many ties)
  int xlo;                       // word index of the current root: every candidate set is empty below it
};

// Reduce the node in Pc.  Returns: 0 pruned, 1 leaf (Pc empty, csz >= incumbent size), 2 continue.
__device__ int node_reduce(WarpCtx& c, int& csz) {
  const int W = c.W, lane = c.lane;
  for (int round = 0; round < 8; ++round) {
    const int cnt = warp_popc(c.Pc, W, lane, c.xlo);
    if (c.cnt && lane == 0) {
      atomicAdd(c.cnt + 3, 1ull);
      atomicAdd(c.cnt + 4, (unsigned long long)cnt);
    }
    const int Lc = *c.Lp + c.strict;
    if (csz + cnt < Lc) return 0;  // cannot even tie the incumbent (ties are enumerated: canonical result)
    if (cnt == 0) return 1;
    const int need = Lc - csz - 1;  // a candidate must have >= need neighbours inside P to reach size Lc
    for (int x = c.xlo + lane; x < W; x += 32) c.Q[x] = c.Pc[x];
    __syncwarp();
    int removed = 0;
    int added = 0;
    {
      int x = c.xlo;
      uint32_t m = c.Pc[x];  // warp-uniform (shared memory broadcast)
      while (true) {
        int u[4], d[4], kc = 0;
        while (kc < 4) {
          while (!m && ++x < W) m = c.Pc[x];
          if (!m) break;
          const int bit = __ffs(m) - 1;
          m &= m - 1;
          u[kc++] = x * 32 + bit;
        }
        if (kc == 0) break;
        for (int q = kc; q < 4; ++q) u[q] = u[0];
        inset_degree4(*c.bt, c.b, u, kc, c.Pc, W, lane, d, c.xlo);
        for (int q = 0; q < kc; ++q) {
          if (d[q] == cnt - 1) {  // universal: belongs to every maximal clique of this node
            if (lane == 0) {
              c.Q[u[q] >> 5] &= ~(1u << (u[q] & 31));
              c.cv[csz + added] = u[q];
            }
            ++added;
          } else if (d[q] < need) {
            if (lane == 0) c.Q[u[q] >> 5] &= ~(1u << (u[q] & 31));
            ++removed;
          }
        }
        if (kc < 4) break;
      }
    }
    __syncwarp();
    for (int x = c.xlo + lane; x < W; x += 32) c.Pc[x] = c.Q[x];
    __syncwarp();
    csz += added;
    // another round pays |P| row reads again: only when this one removed a good part of P (degrees drop by about as
    // much, which is what makes further vertices fall)
    if (removed * 8 < cnt) {
      const int cnt2 = cnt - added - removed;
      const int Lc2 = *c.Lp + c.strict;
      if (csz + cnt2 < Lc2) return 0;
      if (cnt2 == 0) return 1;
      return 2;
    }
  }
  const int cnt = warp_popc(c.Pc, W, lane, c.xlo);
  if (csz + cnt < *c.Lp + c.strict) return 0;
  if (cnt == 0) return 1;
  return 2;
}

// Greedy sequential colouring of Pc (classes in index order); Bs = vertices whose colour >= kmin.  Returns |Bs|.
//
// A class is the greedy maximal independent set of the uncoloured vertices: take the lowest vertex u of the residual R,
// R &= ~N(u), repeat.  One pick per round trip to the L2-resident bitset would make the warp latency-bound, so up to
// kSpecCand lowest vertices of R are resolved per round trip: (1) the k(k-1)/2 adjacency bits among them are fetched
// by as many lanes at once and the sequential greedy rule is replayed on that little matrix in registers — the
// accepted candidates are exactly the picks the one-at-a-time loop would make, because the lowest vertex of R & ~N(u0)
// is the first candidate not adjacent to u0, and so on; (2) the rows of the accepted candidates are read together
// (independent loads), each only from its own word upwards: bits of R below a pick are already decided.
__device__ int node_colour(WarpCtx& c, int csz) {
  const int W = c.W, lane = c.lane, xlo = c.xlo;
  int kmin = *c.Lp + c.strict - csz;  // colour k bounds cliques by k: need csz + k >= L to tie or beat
  if (kmin < 1) kmin = 1;
  for (int x = xlo + lane; x < W; x += 32) {
    c.Q[x] = c.Pc[x];
    c.Bs[x] = 0u;
  }
  __syncwarp();
  if (c.cnt) {
    const int np = warp_popc(c.Pc, W, lane, xlo);
    if (lane == 0) {
      atomicAdd(c.cnt + 5, 1ull);
      atomicAdd(c.cnt + 6, (unsigned long long)np);
    }
  }
  // pair (i, j), i < j < kSpecCand, handled by this lane in step (1): p = j(j-1)/2 + i
  int pi = 0, pj = 1;
  {
    int base = 0;
    while (base + pj <= lane) {
      base += pj;
      ++pj;
    }
    pi = lane - base;
  }
  int nB = 0;
  int qstart = xlo;
  bool singles = false;  // the last class had one member: a clique-like remainder, try the singleton path first
  int k = 1;
  while (true) {
    // anything left uncoloured?
    int xq;
    const int first = warp_first_bit(c.Q, W, lane, qstart, &xq);
    if (first < 0) break;
    qstart = xq;
    if (singles) {
      // ---- singleton path.  When what is left is (nearly) a clique every vertex needs a class of its own, and the
      // general loop would pay two round trips per class.  Here the rows of the lowest <= kSpecCand uncoloured
      // vertices are read in ONE round trip (only the words where Q still has vertices) and each is tested for
      // "no uncoloured non-neighbour above it"; the leading vertices that pass are the next classes, one each —
      // exactly what the greedy rule yields, because a class started at u only looks at uncoloured vertices above u,
      // and those are not changed by the singleton classes of lower vertices.
      const int x = qstart + lane;
      const uint32_t w = x < W ? c.Q[x] : 0u;
      const int pc = __popc(w);
      int incl = pc;
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      const int total = __shfl_sync(0xffffffffu, incl, 31);  // >= 1: the first vertex lies in this window
      {
        int rank = incl - pc;
        uint32_t ww = w;
        while (ww && rank < kSpecCand) {
          c.cand[rank++] = x * 32 + __ffs(ww) - 1;
          ww &= ww - 1;
        }
      }
      __syncwarp();
      const int nc = total < kSpecCand ? total : kSpecCand;
      int u[kSpecCand];
      const uint32_t* r[kSpecCand];
      uint32_t ne[kSpecCand];
#pragma unroll
      for (int q = 0; q < kSpecCand; ++q) {
        u[q] = c.cand[q < nc ? q : 0];
        r[q] = adj_row32(*c.bt, c.b, u[q]);
        ne[q] = 0u;
      }
      for (int y = (u[0] >> 5) + lane; y < W; y += 32) {
        const uint32_t qy = c.Q[y];
        uint32_t rr[kSpecCand];
#pragma unroll
        for (int q = 0; q < kSpecCand; ++q) rr[q] = (qy != 0u && q < nc && y >= (u[q] >> 5)) ? r[q][y] : 0xffffffffu;
#pragma unroll
        for (int q = 0; q < kSpecCand; ++q) {
          uint32_t tq = qy & ~rr[q];
          if (y == (u[q] >> 5)) tq &= ~((2u << (u[q] & 31)) - 1u);  // strictly above u
          ne[q] |= tq;
        }
      }
      int ns = 0;  // leading singleton classes
      bool open = true;
#pragma unroll
      for (int q = 0; q < kSpecCand; ++q) {
        const bool nonempty = __any_sync(0xffffffffu, ne[q] != 0u);
        if (q < nc && open && !nonempty) ++ns;
        else open = false;
      }
      __syncwarp();
      if (lane < ns) {
        const int ul = c.cand[lane];
        const uint32_t bit = 1u << (ul & 31);
        atomicAnd(&c.Q[ul >> 5], ~bit);
        if (k + lane >= kmin) {
          atomicOr(&c.Bs[ul >> 5], bit);
        }
      }
      for (int q = 0; q < ns; ++q)
        if (k + q >= kmin) ++nB;
      k += ns;
      __syncwarp();
      if (ns == nc) continue;       // all of them: look at the next ones the same way
      if (ns == 0) singles = false; // not clique-like (any more)
      const int first2 = warp_first_bit(c.Q, W, lane, qstart, &xq);
      if (first2 < 0) break;
      qstart = xq;
    }
    // ---- general path: one class, the greedy maximal independent set of Q
    for (int x = qstart + lane; x < W; x += 32) c.R[x] = c.Q[x];
    __syncwarp();
    int xr = qstart;
    int members = 0;
    while (xr < W) {
      // ---- the lowest <= kSpecCand vertices of R inside the 32-word window at xr
      const int x = xr + lane;
      const uint32_t w = x < W ? c.R[x] : 0u;
      const int pc = __popc(w);
      int incl = pc;
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      const int total = __shfl_sync(0xffffffffu, incl, 31);
      if (total == 0) {
        xr += 32;
        continue;
      }
      {
        int rank = incl - pc;
        uint32_t ww = w;
        while (ww && rank < kSpecCand) {
          c.cand[rank++] = x * 32 + __ffs(ww) - 1;
          ww &= ww - 1;
        }
      }
      __syncwarp();
      const int nc = total < kSpecCand ? total : kSpecCand;
      const int xlast = c.cand[nc - 1] >> 5;
      int u[kSpecCand];
#pragma unroll
      for (int q = 0; q < kSpecCand; ++q) u[q] = c.cand[q < nc ? q : 0];
      // ---- (1) adjacency among the candidates, greedy rule replayed in registers
      bool e = false;
      if (lane < kSpecCand * (kSpecCand - 1) / 2 && pj < nc) {
        const int ui = c.cand[pi], uj = c.cand[pj];
        e = (adj_row32(*c.bt, c.b, ui)[uj >> 5] >> (uj & 31)) & 1u;
      }
      const unsigned em = __ballot_sync(0xffffffffu, e);
      unsigned acc = 1u;
#pragma unroll
      for (int j = 1; j < kSpecCand; ++j) {
        const unsigned col = (em >> (j * (j - 1) / 2)) & ((1u << j) - 1u);  // bit i: candidate i adjacent to j
        if (j < nc && !(col & acc)) acc |= 1u << j;
      }
      // ---- (2) R &= ~(union of the accepted rows), each row from its own word upwards, only where R has vertices
      const uint32_t* r[kSpecCand];
#pragma unroll
      for (int q = 0; q < kSpecCand; ++q) r[q] = adj_row32(*c.bt, c.b, u[q]);
      int left = 0;
      // groups of kYU words per lane: all row loads of a group are issued before any is used (no branch in between:
      // a data-dependent branch around the loads costs one round trip per word instead of one per group)
      for (int y0 = (u[0] >> 5) + lane; y0 < W; y0 += 32 * kYU) {
        uint32_t rw[kYU], m[kYU];
#pragma unroll
        for (int t = 0; t < kYU; ++t) {
          const int y = y0 + 32 * t;
          rw[t] = y < W ? c.R[y] : 0u;
          m[t] = 0u;
        }
#pragma unroll
        for (int t = 0; t < kYU; ++t) {
          const int y = y0 + 32 * t;
#pragma unroll
          for (int q = 0; q < kSpecCand; ++q)
            if (rw[t] != 0u && ((acc >> q) & 1u) && y >= (u[q] >> 5)) m[t] |= r[q][y];
        }
#pragma unroll
        for (int t = 0; t < kYU; ++t) {
          const int y = y0 + 32 * t;
          if (rw[t] != 0u) {
            const uint32_t nw = rw[t] & ~m[t];
            c.R[y] = nw;
            left += __popc(nw);
          }
        }
      }
      left = __reduce_add_sync(0xffffffffu, left);  // includes the accepted candidates themselves
      __syncwarp();
      if (lane < nc && ((acc >> lane) & 1u)) {
        const int ul = c.cand[lane];
        const uint32_t bit = 1u << (ul & 31);
        atomicAnd(&c.R[ul >> 5], ~bit);
        atomicAnd(&c.Q[ul >> 5], ~bit);
        if (k >= kmin) atomicOr(&c.Bs[ul >> 5], bit);
      }
      const int na = __popc(acc);
      members += na;
      if (k >= kmin) nB += na;
      xr = xlast;  // everything below the last candidate is decided
      __syncwarp();
      if (left == na) break;  // nothing but the picks themselves was left: the class is complete
    }
    singles = members == 1 && !(c.bt->flags_dbg & 8192u);  // 8192: A/B switch
    ++k;
  }
  return nB;
}

// Block colour bound of the node in Pc: true when it proves that the node cannot even tie the incumbent.
//
// The full greedy colouring reads one adjacency row per vertex of P, a few per dependent round trip.  Most roots need
// far less: an outlier's later neighbourhood is a sparse random graph whose clique number is an order of magnitude
// below the incumbent.  Here P is cut (in index order) into blocks of <= blk vertices that lie within 32 consecutive
// bitset words; for a block, ONE word of every member's row covers the whole block, so the induced blk x blk
// adjacency is fetched with independent loads (one round trip), packed to local numbering in shared memory (the Q/R/Bs
// scratch, unused at this point) and coloured greedily without touching global memory again.  Colours of different
// blocks are different colours, so the sum over the blocks is a valid (weaker) colour bound: ~0.085 colours per vertex
// at 15 % density and 128-vertex blocks against ~0.04 for the full greedy colouring — enough whenever
// |P| is below ~12x the incumbent size, at a fraction of the row traffic and without the dependent round trips.
// Measured on B200 (C3, one problem, scripts/gpu_r2_s2_clique_ab.sh): the search is FASTER without this bound (18.7 ms vs
// 20.0 ms with the counters of debug flag 4 on), and inlined into the ~10 k-instruction search kernel the build faults
// with "illegal instruction" at a warp collective (the kernel runs out of convergence-barrier registers; out of line it
// is correct).  So it is compiled only with EXTRA=-DTZR_BLOCK_BOUND, out of line, for A/B runs.
#ifndef TZR_BLOCK_BOUND
__device__ __forceinline__ bool node_block_bound(WarpCtx&, int) { return false; }
#else
__noinline__ __device__ bool node_block_bound(WarpCtx& c, int csz) {
  const int W = c.W, lane = c.lane, S = c.blk;
  const int kmin = *c.Lp + c.strict - csz;
  if (S == 0 || kmin <= 1 || (c.bt->flags_dbg & 4096u)) return false;  // 4096: A/B switch (bench/profiling)
  const int SW = S >> 5;                  // words per local row
  uint32_t* M = c.Q;                      // S x SW local adjacency (Q, R, Bs are contiguous: 3 W words)
  int* list = reinterpret_cast<int*>(M + S * SW);  // S global vertex ids
  int remaining = warp_popc(c.Pc, W, lane, c.xlo);
  // colours per vertex seen so far in this problem say the bound would come out above kmin: do not pay for it
  if (c.bb_vtx >= 4 * S && (long long)remaining * c.bb_col > (long long)(kmin + (kmin >> 3)) * c.bb_vtx) return false;
  int colours = 0;
  int x = c.xlo;
  uint32_t carry = 0xffffffffu;  // bits of word x not yet consumed by an earlier block
  while (x < W && remaining > 0) {
    if (colours + remaining < kmin) return true;
    // ---- the block: the next <= S vertices of P inside words [x, x + 32)
    const int xw = x + lane;
    uint32_t w = xw < W ? c.Pc[xw] : 0u;
    if (lane == 0) w &= carry;
    int pc = __popc(w);
    int incl = pc;
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    if (total == 0) {
      x += 32;
      carry = 0xffffffffu;
      continue;
    }
    int off = incl - pc;  // local number of this lane's first vertex
    int xnext = x + 32;
    uint32_t cnext = 0xffffffffu;
    if (total > S) {
      // cut after the S-th vertex: the lane holding it keeps its lowest (S - off) bits, later lanes nothing
      uint32_t keep = w;
      if (off >= S) keep = 0u;
      else if (incl > S) {
        uint32_t m = w;
        keep = 0u;
        for (int q = 0; q < S - off; ++q) {
          keep |= m & (0u - m);
          m &= m - 1;
        }
      }
      const unsigned cutl = __ballot_sync(0xffffffffu, incl > S && off < S) | __ballot_sync(0xffffffffu, off >= S && pc > 0);
      const int ln = __ffs(cutl) - 1;  // first lane with unconsumed vertices
      const uint32_t wn = __shfl_sync(0xffffffffu, w & ~keep, ln);
      xnext = x + ln;
      cnext = wn;  // word xnext keeps exactly its unconsumed bits (the original word ANDed again next time)
      w = keep;
      pc = __popc(w);
    }
    const int nb = total > S ? S : total;
    remaining -= nb;
    // ---- vertex list and zeroed local matrix
    {
      uint32_t m = w;
      int q = off;
      while (m) {
        list[q++] = xw * 32 + __ffs(m) - 1;
        m &= m - 1;
      }
    }
    for (int q = lane; q < nb * SW; q += 32) M[q] = 0u;
    __syncwarp();
    // ---- rows: word xw of every member's row, packed to local numbering (software bit-gather on the lane's mask w).
    // Two batches of kBlkBatch independent loads are kept in flight (ping-pong) while the previous batch is packed.
    if (pc > 0) {
      const int wo = off >> 5, sh = off & 31;
      const uint32_t* colp = reinterpret_cast<const uint32_t*>(c.bt->adj) + (size_t)c.b * c.n * W + xw;  // word xw of row 0
      auto load = [&](uint32_t (&dst)[kBlkBatch], int i0) {
#pragma unroll
        for (int q = 0; q < kBlkBatch; ++q) {
          const int i = i0 + q < nb ? i0 + q : nb - 1;
          dst[q] = colp[(size_t)list[i] * W];
        }
      };
      auto pack = [&](const uint32_t (&src)[kBlkBatch], int i0) {
#pragma unroll
        for (int q = 0; q < kBlkBatch; ++q) {
          if (i0 + q < nb) {
            const uint32_t a = src[q] & w;
            if (a) {
              uint32_t val = 0u, m = w;
              int kbit = 0;
              while (m) {
                const int bpos = __ffs(m) - 1;
                m &= m - 1;
                val |= ((a >> bpos) & 1u) << kbit;
                ++kbit;
              }
              uint32_t* row = M + (i0 + q) * SW;
              atomicOr(row + wo, val << sh);
              if (sh && (val >> (32 - sh))) atomicOr(row + wo + 1, val >> (32 - sh));
            }
          }
        }
      };
      uint32_t ra[kBlkBatch], rb[kBlkBatch];
      load(ra, 0);
      for (int i0 = 0; i0 < nb; i0 += 2 * kBlkBatch) {
        if (i0 + kBlkBatch < nb) load(rb, i0 + kBlkBatch);
        pack(ra, i0);
        if (i0 + 2 * kBlkBatch < nb) load(ra, i0 + 2 * kBlkBatch);
        if (i0 + kBlkBatch < nb) pack(rb, i0 + kBlkBatch);
      }
    }
    __syncwarp();
    // ---- greedy colouring of the block in shared memory (warp-uniform scalar work on <= 4-word sets)
    {
      uint32_t U[4] = {0u, 0u, 0u, 0u};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int lo = j * 32;
        if (lo < nb) U[j] = nb - lo >= 32 ? 0xffffffffu : ((1u << (nb - lo)) - 1u);
      }
      c.bb_vtx += nb;
      while ((U[0] | U[1] | U[2] | U[3]) != 0u) {
        ++colours;
        ++c.bb_col;
        uint32_t R[4] = {U[0], U[1], U[2], U[3]};
        while (true) {
          int u = -1;
#pragma unroll
          for (int j = 3; j >= 0; --j)
            if (R[j]) u = j * 32 + __ffs(R[j]) - 1;
          if (u < 0) break;
          const uint32_t* row = M + u * SW;
          const uint32_t bit = 1u << (u & 31);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (j < SW) {
              uint32_t rj = row[j];
              if (j == (u >> 5)) {
                rj |= bit;
                U[j] &= ~bit;
              }
              R[j] &= ~rj;
            }
          }
        }
        if (colours >= kmin) return false;  // this bound cannot decide: the caller colours P properly
      }
    }
    __syncwarp();
    x = xnext;
    carry = cnext;
  }
  return colours < kmin;
}
#endif  // TZR_BLOCK_BOUND

// Offer the clique cv[0..csz) as incumbent.  Larger wins; on equal size the lexicographically smaller
// sorted index set wins (== the set that owns the lowest vertex of the symmetric difference), which makes
// the final answer independent of the order in which warps find cliques.
__device__ void record_clique(WarpCtx& c, int csz) {
  const int W = c.W, lane = c.lane;
  for (int x = lane; x < W; x += 32) c.Q[x] = 0u;
  __syncwarp();
  for (int i = lane; i < csz; i += 32) {
    const int v = c.cv[i];
    atomicOr(&c.Q[v >> 5], 1u << (v & 31));
  }
  __syncwarp();
  int32_t* lock = c.bt->lock + c.b;
  if (lane == 0) {
    while (atomicCAS(lock, 0, 1) != 0) {
    }
    __threadfence();
  }
  __syncwarp();
  const int Lc = *c.Lp;
  volatile uint32_t* bb = c.bt->best_bits + (size_t)c.b * W;
  bool take = csz > Lc;
  if (csz == Lc) {
    for (int base = 0; base < W; base += 32) {
      const int x = base + lane;
      const uint32_t mine = x < W ? c.Q[x] : 0u;
      const uint32_t diff = x < W ? (mine ^ bb[x]) : 0u;
      const unsigned nz = __ballot_sync(0xffffffffu, diff != 0u);
      if (nz) {
        const int srcl = __ffs(nz) - 1;
        const uint32_t d0 = __shfl_sync(0xffffffffu, diff, srcl);
        const uint32_t m0 = __shfl_sync(0xffffffffu, mine, srcl);
        take = ((m0 >> (__ffs(d0) - 1)) & 1u) != 0u;
        break;
      }
    }
  }
  if (take) {
    int32_t* dst = c.bt->clq + (size_t)c.b * c.n;
    for (int i = lane; i < csz; i += 32) dst[i] = c.cv[i];
    for (int x = lane; x < W; x += 32) bb[x] = c.Q[x];
    __threadfence();
    __syncwarp();
    if (lane == 0) atomicExch(c.bt->L + c.b, csz);
  }
  __syncwarp();
  if (lane == 0) {
    __threadfence();
    atomicExch(lock, 0);
  }
  __syncwarp();
}

// Branch and bound below one root vertex after another of problem b, until its root counter runs out.
__device__ void exact_search_problem(const Batch& bt, WarpCtx& c, int b) {
  const int n = bt.n, W = c.W, lane = c.lane;
  c.b = b;
  c.bb_col = 0;
  c.bb_vtx = 0;
  c.Lp = bt.L + b;
  c.strict = (bt.flags[b] & 8) ? 1 : 0;
  const int ub_stop = c.strict ? (bt.flags[b] >> 8) : 0x7fffffff;  // LP bound of the NT step: reaching it ends the search
  const uint32_t* alive = bt.alive + (size_t)b * W;
  // Params::max_clique_time_limit (graph.cc:44): budget counted from the first search warp of this problem
  unsigned long long deadline = 0ull;
  if (bt.budget_ns) {
    unsigned long long t0 = 0ull;
    if (lane == 0) {
      const unsigned long long now = globaltimer_ns();
      const unsigned long long old = atomicCAS(bt.t_start + b, 0ull, now);
      t0 = old ? old : now;
    }
    t0 = __shfl_sync(0xffffffffu, t0, 0);
    deadline = t0 + bt.budget_ns;
  }

  while (true) {
    int v = 0;
    if (lane == 0) v = atomicAdd(bt.root_ctr + b, 1);
    v = __shfl_sync(0xffffffffu, v, 0);
    if (v >= n) break;
    if (!((alive[v >> 5] >> (v & 31)) & 1u)) continue;
    if (bt.flags[b] & 2) break;  // deadline hit elsewhere
    if (*c.Lp >= ub_stop) break;
    // root node: P = N(v) ∩ alive ∩ {u > v}
    c.xlo = v >> 5;
    {
      const uint32_t* rv = adj_row32(bt, b, v);
      const int xv = v >> 5;
      for (int x = xv + lane; x < W; x += 32) {
        uint32_t m = rv[x] & alive[x];
        if (x == xv) m &= ~((2u << (v & 31)) - 1u);  // keep bits strictly above v ((2<<31)-1 wraps to all ones)
        c.Pc[x] = m;
      }
      __syncwarp();
    }
    if (lane == 0) c.cv[0] = v;
    __syncwarp();
    int csz = 1;
    int depth = 0;  // number of saved levels
    bool fresh = true;
    bool at_root = true;
    const unsigned long long t_root = c.cnt ? globaltimer_ns() : 0ull;  // debug flag 4: per-root wall time
    long long ck_first = 0, ck_reduce = 0, ck_colour = 0;                // and cycles per phase
    while (true) {
      if (fresh) {
        // ---- process the node in Pc
        if (deadline && (globaltimer_ns() > deadline)) {
          if (lane == 0) atomicOr(bt.flags + b, 3);
          depth = 0;
          break;
        }
        if (*c.Lp >= ub_stop) {
          depth = 0;
          break;
        }
        if (c.cnt && lane == 0) atomicAdd(c.cnt + 2, 1ull);
        int r = 2;
        long long ck0 = c.cnt ? clock64() : 0ll;
        if (at_root) {
          // Most roots fall to the colour bound at once (an outlier's later neighbourhood holds no clique anywhere near
          // the incumbent): try it before paying the same number of row reads for the degree rules.
          const int cnt = warp_popc(c.Pc, W, lane, c.xlo);
          if (csz + cnt < *c.Lp + c.strict) r = 0;
          else if (cnt > 0 && node_block_bound(c, csz)) {
            r = 0;
            if (c.cnt && lane == 0) atomicAdd(c.cnt + 14, 1ull);
          } else if (cnt > 0 && node_colour(c, csz) == 0) r = 0;
          at_root = false;
          if (c.cnt) {
            const long long ck1 = clock64();
            ck_first += ck1 - ck0;
            ck0 = ck1;
          }
        }
        if (r) r = node_reduce(c, csz);
        if (c.cnt) {
          const long long ck1 = clock64();
          ck_reduce += ck1 - ck0;
          ck0 = ck1;
        }
        if (r == 1) {
          if (csz >= *c.Lp + c.strict) record_clique(c, csz);
        } else if (r == 2) {
          const int nB = node_colour(c, csz);
          if (c.cnt) ck_colour += clock64() - ck0;
          if (nB > 0) {
            if (depth >= bt.max_depth) {
              if (lane == 0) atomicOr(bt.flags + b, 1);
            } else {
              uint32_t* Pd = c.stack + (size_t)depth * 2 * W;
              for (int x = c.xlo + lane; x < W; x += 32) {
                Pd[x] = c.Pc[x];
                Pd[W + x] = c.Bs[x];
              }
              if (lane == 0) c.centry[depth] = csz;
              __syncwarp();
              ++depth;
            }
          }
        }
        fresh = false;
      }
      // ---- branch: next candidate of the top saved level
      if (depth == 0) break;
      const int d = depth - 1;
      uint32_t* Pd = c.stack + (size_t)d * 2 * W;
      uint32_t* Bd = Pd + W;
      const int ce = c.centry[d];
      int xf;
      // cheap level bound: every remaining clique of this level has size <= ce + |P_d| (ties still explored)
      const int cntP = warp_popc(Pd, W, lane, c.xlo);
      int u = -1;
      if (ce + cntP >= *c.Lp + c.strict) u = warp_first_bit(Bd, W, lane, c.xlo, &xf);
      if (u < 0) {
        --depth;
        continue;
      }
      __syncwarp();
      if (lane == 0) {
        Bd[u >> 5] &= ~(1u << (u & 31));
        Pd[u >> 5] &= ~(1u << (u & 31));
        c.cv[ce] = u;
      }
      __syncwarp();
      const uint32_t* ru = adj_row32(bt, b, u);
      for (int x = c.xlo + lane; x < W; x += 32) c.Pc[x] = Pd[x] & ru[x];
      __syncwarp();
      csz = ce + 1;
      fresh = true;
    }
    if (c.cnt && lane == 0) {
      const unsigned long long dt = globaltimer_ns() - t_root;
      atomicAdd(c.cnt + 8, (unsigned long long)ck_first);
      atomicAdd(c.cnt + 9, (unsigned long long)ck_reduce);
      atomicAdd(c.cnt + 10, (unsigned long long)ck_colour);
      atomicMax(c.cnt + 11, (dt << 16) | (unsigned long long)(v & 0xffff));  // slowest root: ns << 16 | vertex
      atomicAdd(c.cnt + 12, dt);
      if (dt > 1000000ull) atomicAdd(c.cnt + 13, 1ull);  // roots that took more than 1 ms
    }
  }
}

}  // namespace

// Persistent grid (as many CTAs as fit the GPU), every warp on its own: it sweeps the problems of the batch once,
// starting at one of `exact_conc` evenly spaced problems, and on each problem that still has roots takes root vertices
// from that problem's counter until they run out.  All warps of a start group therefore work on the same problem and
// move on together: at most ~exact_conc adjacency bitsets are live at a time, chosen on the host so that they fit the
// L2 (one 10k-vertex bitset is 12.5 MB; a chunk of eight of them under search at once ran at HBM speed, ~2.7x slower
// per problem than one at a time).  Scratch (stack, clique, entry sizes) belongs to the warp, not to the problem.
__global__ void __launch_bounds__(kExactThreads, TZR_EXACT_MIN_BLOCKS) clique_exact_kernel(Batch bt) {
  const int n = bt.n, W = pitch32(n), B = bt.B;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t* wbase = reinterpret_cast<uint32_t*>(smem_raw) + (size_t)wid * (4 * W + kSpecCand);
  WarpCtx c;
  c.cnt = (bt.flags_dbg & 4u) ? bt.mismatches : nullptr;
  c.bt = &bt;
  c.b = 0;
  c.n = n;
  c.W = W;
  c.lane = lane;
  c.Pc = wbase;
  c.Q = wbase + W;
  c.R = wbase + 2 * W;
  c.Bs = wbase + 3 * W;
  c.cand = reinterpret_cast<int*>(wbase + 4 * W);
  {
    int S = 128;  // block colour bound: S*S/32 matrix words + S list entries must fit the 3 W scratch words
    while (S > 0 && S * (S >> 5) + S > 3 * W) S -= 32;
    c.blk = S;
  }
  const size_t gw = (size_t)blockIdx.x * kExactWarps + wid;  // this warp's scratch slot
  c.stack = bt.stack + gw * (size_t)bt.max_depth * 2 * W;
  c.cv = bt.cv + gw * (size_t)n;
  c.centry = bt.centry + gw * (size_t)bt.max_depth;
  c.Lp = bt.L;
  c.strict = 0;
  c.xlo = 0;
  const int nstart = bt.exact_conc < 1 ? 1 : (bt.exact_conc > B ? B : bt.exact_conc);
  // the warps of a CTA share a start problem; the start groups are interleaved over the grid (and so over the SMs)
  const int bstart = (int)((long long)(blockIdx.x % nstart) * B / nstart);
  const volatile int32_t* rc = bt.root_ctr;
  for (int off = 0; off < B; off += 32) {
    int bb = bstart + off + lane;
    if (bb >= B) bb -= B;
    const bool act = (off + lane < B) && bt.alive_cnt[bb] != 0 && rc[bb] < n && !(bt.flags[bb] & 2);
    unsigned m = __ballot_sync(0xffffffffu, act);
    while (m) {
      const int l = __ffs(m) - 1;
      m &= m - 1;
      int b = bstart + off + l;
      if (b >= B) b -= B;
      exact_search_problem(bt, c, b);
    }
  }
}

// =================================================================================================
// host-side launcher
// =================================================================================================

// =================================================================================================
// K4: Nemhauser–Trotter bound / reduction for problems whose exact search ran out of its first budget.
//
// Dense inlier graphs (noise bound comparable to the object size: the reference's Python example has 99 % density
// among ~800 surviving vertices) defeat colouring bounds, but their COMPLEMENT H inside the alive set A is sparse, and
// max clique of G[A] = |A| - min vertex cover of H[A].  The LP relaxation of vertex cover equals half the maximum
// matching of H's bipartite double cover and is usually tight here (LP 212.5 vs optimum 213 on that example), so:
//   * maximum matching by augmenting paths, one warp per problem, H rows formed on the fly as ~adj[u] & A;
//   * if |A| - ceil(matching / 2) <= L the incumbent is optimal: done (flag 4);
//   * otherwise König's construction gives the half-integral LP optimum; by the Nemhauser–Trotter theorem some maximum
//     clique avoids every vertex with LP value 1, so those leave A (flag 8) and the second search pass runs on the rest.
// Either way the returned clique has maximum SIZE; which maximum clique is no longer the canonical (lexicographically
// smallest) one, reported as clique_proven_optimal = 2.  Problems whose first pass completed are not touched.
// Scratch: the exact-phase cv slots of the problem (free between the passes): mateL | mateR | parent | queue.
// =================================================================================================
__global__ void __launch_bounds__(32) clique_lp_kernel(Batch bt) {
  const int b = blockIdx.x, lane = threadIdx.x;
  if (!(bt.flags[b] & 2)) return;  // only problems that hit the first-pass deadline
  const int n = bt.n, W = pitch32(n);
  __shared__ uint32_t s_vis[1024], s_free[1024], s_lz[1024];  // visited R / free R (then: reached L), W <= 1024
  __shared__ int s_tail;
  uint32_t* A = bt.alive + (size_t)b * W;
  const int L = bt.L[b];
  int cntA = 0;
  for (int x = lane; x < W; x += 32) cntA += __popc(A[x]);
  for (int o = 16; o; o >>= 1) cntA += __shfl_xor_sync(0xffffffffu, cntA, o);
  if (2 * L < cntA) return;  // far from a clique: the LP bound cannot close such a gap
  int32_t* base = bt.cv + (size_t)b * 4 * (size_t)n;  // cv holds max(search warps, 4 B) rows of n: free between the passes
  int32_t *mateL = base, *mateR = base + n, *parent = base + 2 * (size_t)n, *queue = base + 3 * (size_t)n;
  for (int v = lane; v < n; v += 32) {
    mateL[v] = -1;
    mateR[v] = -1;
  }
  for (int x = lane; x < W; x += 32) s_free[x] = A[x];
  __syncwarp();
  auto hword = [&](const uint32_t* row, int u, int x) {  // word x of H's row u inside A
    uint32_t m = ~row[x] & A[x];
    if (x == (u >> 5)) m &= ~(1u << (u & 31));
    return m;
  };
  int matching = 0;
  // ---- greedy start
  for (int x0 = 0; x0 < W; ++x0) {
    uint32_t aw = A[x0];
    while (aw) {
      const int u = x0 * 32 + __ffs(aw) - 1;
      aw &= aw - 1;
      const uint32_t* row = adj_row32(bt, b, u);
      int found = -1;
      for (int base_x = 0; base_x < W && found < 0; base_x += 32) {
        const int x = base_x + lane;
        const uint32_t m = x < W ? (hword(row, u, x) & s_free[x]) : 0u;
        const unsigned nz = __ballot_sync(0xffffffffu, m != 0u);
        if (nz) {
          const int sl = __ffs(nz) - 1;
          const uint32_t mm = __shfl_sync(0xffffffffu, m, sl);
          found = (base_x + sl) * 32 + __ffs(mm) - 1;
        }
      }
      if (found >= 0) {
        if (lane == 0) {
          mateL[u] = found;
          mateR[found] = u;
          s_free[found >> 5] &= ~(1u << (found & 31));
        }
        ++matching;
        __syncwarp();
      }
    }
  }
  // alternating BFS from the left vertices in queue[0..tail); stops at the first free right vertex when `augment`.
  // Marks reached right vertices in s_vis and (when !augment) reached left vertices in s_lz.
  auto bfs = [&](int tail0, bool augment) -> int {
    if (lane == 0) s_tail = tail0;
    __syncwarp();
    int head = 0, found = -1;
    while (found < 0) {
      const int tail = s_tail;
      if (head >= tail) break;
      const int xq = queue[head++];
      const uint32_t* row = adj_row32(bt, b, xq);
      for (int base_x = 0; base_x < W; base_x += 32) {
        const int x = base_x + lane;
        uint32_t m = 0u;
        if (x < W) {
          m = hword(row, xq, x) & ~s_vis[x];
          s_vis[x] |= m;
        }
        while (m) {
          const int v = x * 32 + __ffs(m) - 1;
          m &= m - 1;
          parent[v] = xq;
          const int mv = mateR[v];
          if (mv < 0) {
            if (augment) found = v;  // lane-local; the lowest lane wins below
          } else {
            const int pos = atomicAdd(&s_tail, 1);
            queue[pos] = mv;
            if (!augment) atomicOr(&s_lz[mv >> 5], 1u << (mv & 31));
          }
        }
        const unsigned anyf = __ballot_sync(0xffffffffu, found >= 0);
        if (anyf) {
          found = __shfl_sync(0xffffffffu, found, __ffs(anyf) - 1);
          break;
        }
        __syncwarp();
      }
      __syncwarp();
    }
    return found;
  };
  // ---- augmenting paths from every free left vertex
  for (int x0 = 0; x0 < W; ++x0) {
    uint32_t aw = A[x0];
    while (aw) {
      const int u = x0 * 32 + __ffs(aw) - 1;
      aw &= aw - 1;
      if (mateL[u] >= 0) continue;
      for (int x = lane; x < W; x += 32) s_vis[x] = 0u;
      if (lane == 0) queue[0] = u;
      __syncwarp();
      const int f = bfs(1, true);
      if (f >= 0) {
        if (lane == 0) {
          int v = f;
          while (v >= 0) {
            const int xl = parent[v];
            const int nv = mateL[xl];
            mateL[xl] = v;
            mateR[v] = xl;
            v = nv;
          }
        }
        ++matching;
      }
      __syncwarp();
    }
  }
  const int ub = cntA - (matching + 1) / 2;
  if (ub <= L) {  // LP bound closes the gap: the incumbent is a maximum clique
    if (lane == 0) {
      bt.flags[b] = 4;
      bt.alive_cnt[b] = 0;
    }
    return;
  }
  // ---- König: Z = everything reachable from the free left vertices by alternating paths
  for (int x = lane; x < W; x += 32) {
    s_vis[x] = 0u;
    s_lz[x] = 0u;
  }
  __syncwarp();
  int tail0 = 0;
  if (lane == 0) {
    for (int x0 = 0; x0 < W; ++x0) {
      uint32_t aw = A[x0];
      while (aw) {
        const int u = x0 * 32 + __ffs(aw) - 1;
        aw &= aw - 1;
        if (mateL[u] < 0) {
          queue[tail0++] = u;
          s_lz[u >> 5] |= 1u << (u & 31);
        }
      }
    }
  }
  tail0 = __shfl_sync(0xffffffffu, tail0, 0);
  __syncwarp();
  bfs(tail0, false);
  __syncwarp();
  // cover C = (L \ Z) u (R n Z); LP value 1 <=> u in both halves: u not reached on the left, reached on the right
  int removed = 0;
  for (int x = lane; x < W; x += 32) {
    const uint32_t v1 = A[x] & ~s_lz[x] & s_vis[x];
    removed += __popc(v1);
    A[x] &= ~v1;
  }
  for (int o = 16; o; o >>= 1) removed += __shfl_xor_sync(0xffffffffu, removed, o);
  if (lane == 0) {
    bt.alive_cnt[b] = cntA - removed;
    // flag 8: second pass in "beat the incumbent" mode, stopping as soon as it reaches the LP bound kept in bits 8..
    bt.flags[b] = (bt.flags[b] & 3) | 8 | (ub << 8);
  }
}

// Between the two exact passes: problems still open (deadline hit, not closed by the LP bound) get a fresh work counter
// and clock; everything else is switched off for the second pass.
__global__ void clique_resume_kernel(Batch bt) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= bt.B) return;
  const int f = bt.flags[b];
  if ((f & 2) && !(f & 4)) {
    bt.flags[b] = f & ~3;
    bt.root_ctr[b] = 0;
    bt.t_start[b] = 0ull;
  } else {
    bt.alive_cnt[b] = 0;
  }
}

namespace {
void clique_set_attrs() {
  // per device: a process may hold contexts on several GPUs
  static bool attr_done_dev[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  bool& attr_done = attr_done_dev[dev & 63];
  if (!attr_done) {
    cudaFuncSetAttribute(clique_heur_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(clique_peel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(clique_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute(clique_kcore_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    attr_done = true;
  }
}
}  // namespace

int clique_exact_grid(int n, int num_sms) {
  clique_set_attrs();
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, clique_exact_kernel, kExactThreads, clique_exact_smem(n)) !=
          cudaSuccess ||
      occ < 1)
    occ = 1;
  return occ * num_sms;
}

void launch_clique(const Batch& bt, const tzr_params& p, int mode, cudaStream_t st, int* n_launches) {
  const int n = bt.n;
  clique_set_attrs();
  int launches = 0;
  Batch b2 = bt;
  if (mode == 2) {  // KCORE_HEU (graph.cc:66-81)
    clique_kcore_kernel<<<bt.B, kPeelThreads, clique_kcore_smem(n), st>>>(bt, p.kcore_heuristic_threshold);
    ++launches;
  } else {
    b2.kcore_final = nullptr;
  }
  dim3 g1(kHeurRoots, (unsigned)bt.B);
  clique_heur_kernel<<<g1, kHeurThreads, clique_heur_smem(n), st>>>(b2);
  clique_peel_kernel<<<bt.B, kPeelThreads, clique_peel_smem(n), st>>>(b2, mode == 0 ? 0 : 1);
  launches += 2;
  if (mode == 0) {
    // Two passes: a short first one (every instance the canonical enumeration can finish does so here), then the
    // Nemhauser–Trotter bound / reduction for whatever ran into that deadline, then the rest of the caller's budget.
    constexpr unsigned long long kFirstPassNs = 50ull * 1000 * 1000;
    const unsigned long long total = bt.budget_ns;  // 0 = unlimited
    const unsigned g3 = (unsigned)bt.exact_ctas;
    Batch p1 = b2;
    p1.budget_ns = (total == 0ull || total > kFirstPassNs) ? kFirstPassNs : total;
    clique_exact_kernel<<<g3, kExactThreads, clique_exact_smem(n), st>>>(p1);
    clique_lp_kernel<<<bt.B, 32, 0, st>>>(b2);
    launches += 2;
    if (total == 0ull || total > kFirstPassNs) {
      Batch p2 = b2;
      p2.budget_ns = total ? total - kFirstPassNs : 0ull;
      clique_resume_kernel<<<(bt.B + 127) / 128, 128, 0, st>>>(b2);
      clique_exact_kernel<<<g3, kExactThreads, clique_exact_smem(n), st>>>(p2);
      launches += 2;
    }
  }
  if (n_launches) *n_launches += launches;
}

}  // namespace tzr
