// C-ABI of libteaser_b200.so: context, workspace, stage entry points and the fused batch solve.
// See include/teaser_b200.h for the contract and the reference functions each symbol replaces.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "tzr_internal.cuh"

using namespace tzr;

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
};

struct tzr_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  std::string last_error;
  int64_t launches = 0;
  uint32_t flags = 0;
  int num_sms = 148;
  // device buffers (grow-only)
  DevBuf src, dst, sf, df, pk, opnd, tclist, gc, adj, deg, nedges, hclq, hsize, clq, L, alive, best_bits, alive_cnt, root_ctr, lock, flg, kfinal, tstart, stack, cv,
      centry, ps, pd, wgt, res, skey, sidx, sorted, rmask, tmask, sol, dbg, misc, sc_x, sc_r, sc_key, sc_idx, m_in, m_scratch, m_out, cert;
  // n > kMaxN: scratch of the clique front end, and the clique buffers of the compacted (L-1)-cores
  DevBuf large, compact;
  LargeScratch lscr{};
  // pinned host staging
  void* h_pin = nullptr;
  size_t h_pin_cap = 0;
  // last batch geometry
  Batch last{};
  bool have_last = false;
  cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // start | prep | graph tiles | clique (incl. degrees) | rot+trans
  std::vector<cudaEvent_t> graph_ev;  // pairs around every graph-kernel launch of the last call (roofline timing)
  int graph_ev_used = 0;
  std::vector<cudaEvent_t> stage_ev;  // 5 per chunk; [stage_first, stage_chunks) belong to the last pipelined call
  int stage_chunks = 0, stage_first = 0, graph_first = 0;
  bool stage_log = false;  // keep the events of every call since the last tzr_ctx_stage_log_read (bench.py: no sync per step)
  int stage_log_calls = 0;
  uint64_t generation = 0;   // bumped by every call that rebuilds or invalidates the retained graph (ctx->last)
  bool last_has_graph = false;  // false: the last solve ran with inlier selection NONE (no graph was built)
  // chunked batches run on two lanes: the issue-bound graph kernels queue back to back on the low-priority gstream,
  // the latency-/HBM-bound degree, clique and rotation kernels of the previous chunk run on the high-priority hstream
  // and slot into the SMs as graph CTAs retire
  cudaStream_t gstream = nullptr, hstream = nullptr;
  cudaEvent_t join_ev = nullptr, join_ev2 = nullptr;
  std::vector<cudaEvent_t> gdone_ev;
  void* solver_handle = nullptr;  // cusolverDnHandle_t of the certifier, created on first use (certify.cu)
  cudaStream_t copy_stream = nullptr;  // H2D of chunk k+1 overlaps the kernels of chunk k (host-pointer batches)
  std::vector<cudaEvent_t> chunk_ev;
};

namespace {

#define CK(call)                                                                  \
  do {                                                                            \
    cudaError_t _e = (call);                                                      \
    if (_e != cudaSuccess) {                                                      \
      ctx->last_error = std::string(#call) + ": " + cudaGetErrorString(_e);       \
      return TZR_ERR_CUDA;                                                        \
    }                                                                             \
  } while (0)

int ensure(tzr_ctx* ctx, DevBuf& b, size_t bytes) {
  if (bytes <= b.cap && b.p) return TZR_OK;
  if (b.p) {
    cudaFree(b.p);
    b.p = nullptr;
    b.cap = 0;
  }
  size_t want = bytes + bytes / 8 + 256;
  cudaError_t e = cudaMalloc(&b.p, want);
  if (e != cudaSuccess) {
    ctx->last_error = std::string("cudaMalloc: ") + cudaGetErrorString(e);
    return TZR_ERR_ALLOC;
  }
  b.cap = want;
  return TZR_OK;
}

int ensure_pinned(tzr_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->h_pin_cap) return TZR_OK;
  if (ctx->h_pin) cudaFreeHost(ctx->h_pin);
  ctx->h_pin = nullptr;
  ctx->h_pin_cap = 0;
  cudaError_t e = cudaMallocHost(&ctx->h_pin, bytes + bytes / 8 + 256);
  if (e != cudaSuccess) {
    ctx->last_error = std::string("cudaMallocHost: ") + cudaGetErrorString(e);
    return TZR_ERR_ALLOC;
  }
  ctx->h_pin_cap = bytes + bytes / 8 + 256;
  return TZR_OK;
}

// Copy `count` caller buffers of `per` bytes each into a contiguous pinned area with a few host threads (pageable
// host memory cannot be DMA'd asynchronously; one thread moves ~10 GB/s, which is slower than the GPU consumes it).
void parallel_stage(char* dst_base, const double* const* bufs, int first, int count, size_t per) {
  const size_t total = per * (size_t)count;
  int T = (int)std::min<size_t>(8, total / ((size_t)4 << 20));
  const unsigned hw = std::thread::hardware_concurrency();
  if (hw && (unsigned)T > hw) T = (int)hw;
  if (T <= 1) {
    for (int b = 0; b < count; ++b) memcpy(dst_base + per * b, bufs[first + b], per);
    return;
  }
  std::vector<std::thread> th;
  for (int t = 0; t < T; ++t)
    th.emplace_back([=] {
      for (int b = t; b < count; b += T) memcpy(dst_base + per * b, bufs[first + b], per);
    });
  for (auto& x : th) x.join();
}

int next_pow2_host(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// effective inlier selection mode (registration.cc:574-583)
int effective_mode(const tzr_params& p) {
  int mode = p.inlier_selection_mode;
  if (!p.use_max_clique) mode = 3;
  if (!p.max_clique_exact_solution) mode = 1;
  return mode;
}

// Exact clique phase of a (B, n <= kMaxN) batch: a persistent grid that fills the GPU; its warps own the search scratch
// (any problem).  Sets exact_ctas, max_depth and exact_conc of bt; returns the number of search warps.
size_t exact_geometry(const tzr_ctx* ctx, int B, int n, Batch* bt) {
  int G = clique_exact_grid(n, ctx->num_sms);
  {
    const long long roots = ((long long)B * n + 7) / 8;  // never more warps than root vertices
    if ((long long)G > roots) G = (int)std::max<long long>(1, roots);
  }
  const size_t warps = (size_t)G * 8;
  const size_t level_bytes = (size_t)2 * pitch32(n) * sizeof(uint32_t);
  size_t depth = ((size_t)4 << 30) / (warps * level_bytes);
  if (depth > 512) depth = 512;
  if (depth > (size_t)n) depth = (size_t)n;
  if (depth < 16) depth = 16;
  bt->exact_ctas = G;
  bt->max_depth = (int)depth;
  {
    // problems under search at a time: their bitsets should stay in the L2 together (~48 MB of the 126 MB: the
    // stacks, the other lane's graph kernel and the two L2 partitions take the rest)
    const size_t bits = (size_t)n * pitch32(n) * sizeof(uint32_t);
    const size_t conc = ((size_t)48 << 20) / std::max<size_t>(bits, 1);
    bt->exact_conc = (int)std::min<size_t>(std::max<size_t>(conc, 1), (size_t)B);
  }
  return warps;
}

// Size the workspace for a (B, n) batch and fill the Batch descriptor (src/dst left to the caller).
int setup_batch(tzr_ctx* ctx, int B, int n, bool own_points, Batch* out, bool complete_graph = false) {
  if (B <= 0 || n <= 0) return TZR_ERR_INVALID_ARG;
  if (n > kMaxNGraph) {
    ctx->last_error = "n = " + std::to_string(n) + " correspondences: at most " + std::to_string(kMaxNGraph) +
                      " per problem are supported";
    return TZR_ERR_TOO_LARGE;
  }
  // the workspace is about to be re-used (and possibly re-allocated): the retained graph of the previous call is gone
  ctx->have_last = false;
  ctx->last_has_graph = false;
  ++ctx->generation;
  Batch bt{};
  bt.B = B;
  bt.n = n;
  const size_t Bn = (size_t)B * n;
  const int W32 = pitch32(n);
  int rc;
#define ENS(buf, bytes)                                  \
  if ((rc = ensure(ctx, ctx->buf, (bytes))) != TZR_OK) return rc;
  if (own_points) {
    ENS(src, Bn * 3 * sizeof(double));
    ENS(dst, Bn * 3 * sizeof(double));
  }
  ENS(sf, Bn * sizeof(float4));
  ENS(df, Bn * sizeof(float4));
  ENS(pk, (size_t)B * 6 * npad128(n) * sizeof(float));
  ENS(opnd, tc_operand_bytes(B, n));
  bt.tc_list_cap = (unsigned int)tc_list_entries(B, n);
  ENS(tclist, (size_t)bt.tc_list_cap * sizeof(uint2) + 256);
  ENS(gc, (size_t)B * sizeof(GraphConsts));
  ENS(adj, Bn * pitch64(n) * sizeof(uint64_t));
  ENS(deg, Bn * sizeof(int32_t));
  ENS(nedges, (size_t)B * sizeof(unsigned long long));
  ENS(hclq, Bn * kHeurRoots * sizeof(int32_t));
  ENS(hsize, (size_t)B * kHeurRoots * sizeof(int32_t));
  ENS(clq, Bn * sizeof(int32_t));
  ENS(L, (size_t)B * sizeof(int32_t));
  ENS(alive, (size_t)B * W32 * sizeof(uint32_t));
  ENS(best_bits, (size_t)B * W32 * sizeof(uint32_t));
  ENS(alive_cnt, (size_t)B * sizeof(int32_t));
  ENS(root_ctr, (size_t)B * sizeof(int32_t));
  ENS(lock, (size_t)B * sizeof(int32_t));
  ENS(flg, (size_t)B * sizeof(int32_t));
  ENS(kfinal, (size_t)B * sizeof(int32_t));
  ENS(tstart, (size_t)B * sizeof(unsigned long long));
  if (n <= kMaxN) {
    const size_t warps = exact_geometry(ctx, B, n, &bt);
    const size_t depth = (size_t)bt.max_depth, level_bytes = (size_t)2 * W32 * sizeof(uint32_t);
    ENS(stack, warps * depth * level_bytes);
    ENS(cv, std::max(warps, (size_t)4 * B) * (size_t)n * sizeof(int32_t));
    ENS(centry, warps * depth * sizeof(int32_t));
  } else {  // the exact search runs on the compacted cores (setup_clique_batch)
    ENS(large, large_scratch_bytes(B, n));
    ctx->lscr = large_scratch_carve(ctx->large.p, B, n);
  }
  bt.sort_cap = next_pow2_host(2 * n);
  ENS(ps, Bn * 3 * sizeof(double));
  ENS(pd, Bn * 3 * sizeof(double));
  // rotation TIM capacity: n for CHAIN; for COMPLETE min(n(n-1)/2, what a 4 GiB budget allows)
  bt.rot_cap = n;
  if (complete_graph) {
    const long long full = (long long)n * (n - 1) / 2;
    const long long budget = ((long long)4 << 30) / (9LL * B);
    bt.rot_cap = std::max<long long>(n, std::min(full, budget));
  }
  ENS(wgt, (size_t)B * bt.rot_cap * sizeof(double));
  ENS(res, Bn * sizeof(double));
  ENS(skey, (size_t)B * 3 * bt.sort_cap * sizeof(double));
  ENS(sidx, (size_t)B * 3 * bt.sort_cap * sizeof(int32_t));
  ENS(sorted, Bn * sizeof(int32_t));
  ENS(rmask, (size_t)B * bt.rot_cap);
  ENS(tmask, Bn);
  ENS(sol, (size_t)B * sizeof(tzr_solution));
  ENS(dbg, 16 * sizeof(unsigned long long));
#undef ENS
  bt.src = (const double*)ctx->src.p;
  bt.dst = (const double*)ctx->dst.p;
  bt.sf = (float4*)ctx->sf.p;
  bt.df = (float4*)ctx->df.p;
  bt.pk = (float*)ctx->pk.p;
  bt.opnd = (float*)ctx->opnd.p;
  bt.tc_list_count = (unsigned int*)ctx->tclist.p;
  bt.tc_list = (uint2*)((char*)ctx->tclist.p + 256);
  bt.gc = (GraphConsts*)ctx->gc.p;
  bt.adj = (uint64_t*)ctx->adj.p;
  bt.deg = (int32_t*)ctx->deg.p;
  bt.n_edges2 = (unsigned long long*)ctx->nedges.p;
  bt.hclq = (int32_t*)ctx->hclq.p;
  bt.hsize = (int32_t*)ctx->hsize.p;
  bt.clq = (int32_t*)ctx->clq.p;
  bt.L = (int32_t*)ctx->L.p;
  bt.alive = (uint32_t*)ctx->alive.p;
  bt.best_bits = (uint32_t*)ctx->best_bits.p;
  bt.alive_cnt = (int32_t*)ctx->alive_cnt.p;
  bt.root_ctr = (int32_t*)ctx->root_ctr.p;
  bt.lock = (int32_t*)ctx->lock.p;
  bt.flags = (int32_t*)ctx->flg.p;
  bt.kcore_final = (int32_t*)ctx->kfinal.p;
  bt.t_start = (unsigned long long*)ctx->tstart.p;
  bt.stack = (uint32_t*)ctx->stack.p;
  bt.cv = (int32_t*)ctx->cv.p;
  bt.centry = (int32_t*)ctx->centry.p;
  bt.ps = (double*)ctx->ps.p;
  bt.pd = (double*)ctx->pd.p;
  bt.wgt = (double*)ctx->wgt.p;
  bt.res = (double*)ctx->res.p;
  bt.skey = (double*)ctx->skey.p;
  bt.sidx = (int32_t*)ctx->sidx.p;
  bt.sorted_clq = (int32_t*)ctx->sorted.p;
  bt.rot_mask = (uint8_t*)ctx->rmask.p;
  bt.trans_mask = (uint8_t*)ctx->tmask.p;
  bt.sol = (tzr_solution*)ctx->sol.p;
  bt.mismatches = (unsigned long long*)ctx->dbg.p;
  bt.rechecks = (ctx->flags & 4u) ? (unsigned long long*)ctx->dbg.p + 1 : nullptr;
  bt.flags_dbg = ctx->flags;
  if (n > kMaxNTc) bt.flags_dbg &= ~(1024u | 2048u);  // both re-check queues pack j in 16 bits: default graph kernel
  {
    static const double kappa_env = [] {
      const char* e = std::getenv("TZR_TC_KAPPA");
      return e ? std::atof(e) : 0.0;
    }();
    static const int swap_env = [] {
      const char* e = std::getenv("TZR_TC_SWAP");
      return e ? std::atoi(e) : 0;
    }();
    bt.tc_kappa = kappa_env;
    bt.tc_desc_swap = swap_env;
  }
  bt.budget_ns = 0ull;
  *out = bt;
  return TZR_OK;
}

// Clique buffers of a compacted batch: the B (L-1)-cores of a batch with n > kMaxN, nc <= kMaxN vertices each.  They
// have their own region, so the full batch's bitset and clique stay in place for tzr_last_graph and the rotation stage.
int setup_clique_batch(tzr_ctx* ctx, const Batch& full, int nc, Batch* out) {
  const int B = full.B;
  Batch cb{};
  cb.B = B;
  cb.n = nc;
  const size_t Bn = (size_t)B * nc, W32 = (size_t)pitch32(nc);
  const size_t warps = exact_geometry(ctx, B, nc, &cb);
  const size_t depth = (size_t)cb.max_depth;
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t sizes[] = {Bn * pitch64(nc) * sizeof(uint64_t),     // adj
                          Bn * sizeof(int32_t),                    // deg
                          (size_t)B * sizeof(unsigned long long),  // n_edges2
                          Bn * kHeurRoots * sizeof(int32_t),       // hclq
                          Bn * sizeof(int32_t),                    // clq
                          (size_t)B * W32 * sizeof(uint32_t),      // alive
                          (size_t)B * W32 * sizeof(uint32_t),      // best_bits
                          (size_t)B * (kHeurRoots + 5) * sizeof(int32_t),  // hsize (kHeurRoots) | L | alive_cnt | root_ctr | lock | flags
                          (size_t)B * sizeof(unsigned long long),  // t_start
                          warps * depth * 2 * W32 * sizeof(uint32_t),                      // stack
                          std::max(warps, (size_t)4 * B) * (size_t)nc * sizeof(int32_t),   // cv
                          warps * depth * sizeof(int32_t)};                                // centry
  size_t total = 0;
  for (size_t x : sizes) total += al(x);
  const int rc = ensure(ctx, ctx->compact, total);
  if (rc != TZR_OK) return rc;
  char* p = (char*)ctx->compact.p;
  char* part[12];
  for (int i = 0; i < 12; ++i) {
    part[i] = p;
    p += al(sizes[i]);
  }
  cb.adj = (uint64_t*)part[0];
  cb.deg = (int32_t*)part[1];
  cb.n_edges2 = (unsigned long long*)part[2];
  cb.hclq = (int32_t*)part[3];
  cb.clq = (int32_t*)part[4];
  cb.alive = (uint32_t*)part[5];
  cb.best_bits = (uint32_t*)part[6];
  int32_t* small = (int32_t*)part[7];
  cb.hsize = small;
  cb.L = small + (size_t)B * kHeurRoots;
  cb.alive_cnt = cb.L + B;
  cb.root_ctr = cb.alive_cnt + B;
  cb.lock = cb.root_ctr + B;
  cb.flags = cb.lock + B;
  cb.t_start = (unsigned long long*)part[8];
  cb.stack = (uint32_t*)part[9];
  cb.cv = (int32_t*)part[10];
  cb.centry = (int32_t*)part[11];
  cb.kcore_final = nullptr;
  cb.mismatches = full.mismatches;
  cb.rechecks = full.rechecks;
  cb.flags_dbg = full.flags_dbg;
  cb.budget_ns = full.budget_ns;
  *out = cb;
  return TZR_OK;
}

int check_launch(tzr_ctx* ctx, const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    ctx->last_error = std::string(what) + ": " + cudaGetErrorString(e);
    return TZR_ERR_CUDA;
  }
  return TZR_OK;
}

__global__ void init_solutions_kernel(tzr_solution* sol, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  tzr_solution s;
  memset(&s, 0, sizeof(s));
  s.valid = 1;
  s.scale = 1.0;  // ScaleInliersSelector: *scale = 1  (registration.cc:432)
  sol[b] = s;
}

// View of problems [b0, b0+Bc) of a batch: every per-problem buffer is offset, geometry is unchanged.
Batch sub_batch(const Batch& bt, int b0, int Bc) {
  Batch s = bt;
  const size_t n = (size_t)bt.n, o = (size_t)b0;
  const size_t W32 = (size_t)pitch32(bt.n);
  s.B = Bc;
  s.src = bt.src + o * n * 3;
  s.dst = bt.dst + o * n * 3;
  s.sf = bt.sf + o * n;
  s.df = bt.df + o * n;
  s.pk = bt.pk + o * 6 * (size_t)npad128(bt.n);
  s.opnd = bt.opnd + tc_operand_bytes(b0, bt.n) / sizeof(float);
  s.gc = bt.gc + o;
  s.adj = bt.adj + o * n * pitch64(bt.n);
  s.deg = bt.deg + o * n;
  s.n_edges2 = bt.n_edges2 + o;
  s.hclq = bt.hclq + o * kHeurRoots * n;
  s.hsize = bt.hsize + o * kHeurRoots;
  s.clq = bt.clq + o * n;
  s.L = bt.L + o;
  s.alive = bt.alive + o * W32;
  s.best_bits = bt.best_bits + o * W32;
  s.alive_cnt = bt.alive_cnt + o;
  s.root_ctr = bt.root_ctr + o;
  s.lock = bt.lock + o;
  s.flags = bt.flags + o;
  s.kcore_final = bt.kcore_final + o;
  s.t_start = bt.t_start + o;
  s.ps = bt.ps + o * n * 3;
  s.pd = bt.pd + o * n * 3;
  s.wgt = bt.wgt + o * (size_t)bt.rot_cap;
  s.res = bt.res + o * n;
  s.skey = bt.skey + o * 3 * (size_t)bt.sort_cap;
  s.sidx = bt.sidx + o * 3 * (size_t)bt.sort_cap;
  s.sorted_clq = bt.sorted_clq + o * n;
  s.rot_mask = bt.rot_mask + o * (size_t)bt.rot_cap;
  s.trans_mask = bt.trans_mask + o * n;
  s.sol = bt.sol + o;
  return s;
}

// Problems per pipeline chunk: small enough that a chunk's adjacency bitsets (written by the graph kernel, then
// read by the degree / clique kernels) stay resident in the 126 MB L2 instead of making a round trip through HBM.
int l2_chunk(const tzr_ctx* ctx, int B, int n, const tzr_params& p) {
  (void)ctx;
  // Optional sub-chunking of graph+degree so the degree pass reads the bitsets from L2 (TZR_L2_CHUNK_MB = MB of
  // adjacency per sub-chunk).  Off by default: with the v5 graph kernel the tail of each small launch costs more
  // than the saved HBM read (measured r01: 84.5 K reg/s unchunked vs 78.1 K at 96 MB, profiles/README.md).
  static const long long budget_mb = [] {
    const char* e = std::getenv("TZR_L2_CHUNK_MB");
    return e ? std::atoll(e) : 0LL;
  }();
  if (budget_mb <= 0 || p.estimate_scaling) return B;
  const size_t per = (size_t)n * pitch64(n) * 8;
  long long c = (long long)((size_t)budget_mb << 20) / (long long)std::max<size_t>(per, 1);
  if (c < 1) c = 1;
  if (c >= B) return B;
  return (int)c;
}

// Clique stage of a batch with n > kMaxN (clique_large.cu): greedy heuristic and core peel on the full graph, then
// (PMC_EXACT) the existing search on the compacted (L-1)-cores.  The host waits once, after the peel, for the largest
// core of the batch, which sizes the compacted batch.
int run_clique_large(tzr_ctx* ctx, const Batch& bt, const tzr_params& p, int mode, cudaStream_t st, int* nl) {
  const int B = bt.B;
  const LargeScratch& ls = ctx->lscr;
  const int k = launch_clique_large_front(bt, ls, mode, p.kcore_heuristic_threshold, st, ctx->num_sms);
  if (k < 0) {
    const int rc = check_launch(ctx, "clique front end (n > 32768)");
    if (rc == TZR_OK) ctx->last_error = "clique front end (n > 32768): launch failed";
    return TZR_ERR_CUDA;
  }
  *nl += k;
  std::vector<int32_t> h(2 * (size_t)B);
  CK(cudaMemcpyAsync(h.data(), ls.nsurv, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(h.data() + B, bt.L, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  int nc = 0;
  for (int b = 0; b < B; ++b) {
    const int core = h[b], L = h[B + b];
    if (mode == 0 && core > kMaxN) {
      ctx->last_error = "problem " + std::to_string(b) + ": the (L-1)-core of its inlier graph (L = " + std::to_string(L) +
                        ", the greedy clique) has " + std::to_string(core) + " vertices; the exact search takes at most " +
                        std::to_string(kMaxN) + " when n > " + std::to_string(kMaxN) +
                        " (PMC_HEU and KCORE_HEU work at this size)";
      return TZR_ERR_TOO_LARGE;
    }
    if (mode != 0 && L > kMaxN) {
      ctx->last_error = "problem " + std::to_string(b) + ": the selected inlier set has " + std::to_string(L) +
                        " vertices; the rotation stage takes at most " + std::to_string(kMaxN);
      return TZR_ERR_TOO_LARGE;
    }
    nc = std::max(nc, core);
  }
  if (mode != 0 || nc == 0) return TZR_OK;  // no problem has an edge: the greedy result (L <= 1) stands
  Batch cb;
  int rc = setup_clique_batch(ctx, bt, nc, &cb);
  if (rc) return rc;
  CK(cudaMemsetAsync(cb.n_edges2, 0, (size_t)B * sizeof(unsigned long long), st));
  launch_clique_compact(bt, ls, cb, st);
  launch_degree(cb, st, true);
  launch_clique(cb, p, 0, st, nl);
  launch_clique_map_back(bt, ls, cb, st);
  *nl += 3;
  return check_launch(ctx, "compacted clique search");
}

// The fused device pipeline for one uniform batch.  src/dst must already be set in bt.
// st: stream of the clique / rotation stages; sg: stream of prep + graph (== st for the single-lane form, otherwise
// gdone is recorded on sg after the graph kernel and st waits for it).
int run_pipeline(tzr_ctx* ctx, Batch& bt, const tzr_params& p, cudaEvent_t* ev, cudaStream_t st,
                 cudaStream_t sg = nullptr, cudaEvent_t gdone = nullptr) {
  if (!sg) sg = st;
  if (p.rotation_estimation_algorithm < 0 || p.rotation_estimation_algorithm > 2 || p.rotation_tim_graph < 0 ||
      p.rotation_tim_graph > 1)
    return TZR_ERR_INVALID_ARG;
  const int mode = effective_mode(p);
  if (bt.n > kMaxN && (p.estimate_scaling || mode == 3)) {
    ctx->last_error = p.estimate_scaling
                          ? "estimate_scaling is supported up to n = " + std::to_string(kMaxN) + " correspondences"
                          : "inlier selection NONE hands all n > " + std::to_string(kMaxN) +
                                " correspondences to the rotation stage, which takes at most " + std::to_string(kMaxN);
    return TZR_ERR_TOO_LARGE;
  }
  bt.beta = 2.0 * p.noise_bound * std::sqrt(p.cbar2);  // registration.cc:438
  // Params::max_clique_time_limit (seconds) -> device-side budget of the exact search
  bt.budget_ns = 0ull;
  if (mode == 0 && p.max_clique_time_limit > 0 && p.max_clique_time_limit < 1e7)
    bt.budget_ns = (unsigned long long)(p.max_clique_time_limit * 1e9);
  // unknown scale (Params default): TLS over the K TIM ratios first (registration.cc:603 -> :410-425)
  constexpr int kScaleSmallN = 256;  // single-CTA bitonic sort + sequential one-thread sweep below (bit-exact vs the
                                     // reference's order; ~1 ms at 256), radix-sort + parallel-scan pipeline above
  bt.scale_mode = p.estimate_scaling ? 1 : 0;
  double *scx = nullptr, *scr = nullptr, *sckey = nullptr;
  int32_t* scidx = nullptr;
  long long sc_npad = 0;
  const bool scale_large = bt.scale_mode && bt.n > kScaleSmallN;
  if (bt.scale_mode) {
    const long long K = (long long)bt.n * (bt.n - 1) / 2;
    int rc;
    if (!scale_large) {
      sc_npad = 1;
      while (sc_npad < 2 * K) sc_npad <<= 1;
      if ((rc = ensure(ctx, ctx->sc_x, (size_t)bt.B * K * 8 + 8)) != TZR_OK) return rc;
      if ((rc = ensure(ctx, ctx->sc_r, (size_t)bt.B * K * 8 + 8)) != TZR_OK) return rc;
      if ((rc = ensure(ctx, ctx->sc_key, (size_t)bt.B * sc_npad * 8)) != TZR_OK) return rc;
      if ((rc = ensure(ctx, ctx->sc_idx, (size_t)bt.B * sc_npad * 4)) != TZR_OK) return rc;
    } else {
      if (2 * K >= (1LL << 31)) {
        ctx->last_error = "estimate_scaling: 2K end points exceed 2^31";
        return TZR_ERR_TOO_LARGE;
      }
      if ((rc = ensure(ctx, ctx->sc_x, (size_t)K * 8 + 8)) != TZR_OK) return rc;
      if ((rc = ensure(ctx, ctx->sc_r, (size_t)K * 8 + 8)) != TZR_OK) return rc;
      if ((rc = ensure(ctx, ctx->sc_key, scale_large_scratch_bytes(bt.n, nullptr))) != TZR_OK) return rc;
    }
    scx = (double*)ctx->sc_x.p;
    scr = (double*)ctx->sc_r.p;
    sckey = (double*)ctx->sc_key.p;
    scidx = (int32_t*)ctx->sc_idx.p;
  }
  cudaEventRecord(ev[0], sg);
  init_solutions_kernel<<<(bt.B + 127) / 128, 128, 0, sg>>>(bt.sol, bt.B);
  if (ctx->flags & 6u) cudaMemsetAsync((void*)ctx->dbg.p, 0, 16 * sizeof(unsigned long long), sg);
  ctx->launches += 1;
  if (bt.scale_mode) {  // before prep: the FP32 filter copies are pre-scaled by the estimate
    bt.beta = 2.0 * p.noise_bound * std::sqrt(p.cbar2);
    if (scale_large) {
      const int nl2 = launch_scale_estimation_large(bt, scx, scr, sckey, sg);
      if (nl2 < 0) return TZR_ERR_TOO_LARGE;
      ctx->launches += nl2;
    } else {
      ctx->launches += launch_scale_estimation(bt, scx, scr, sckey, scidx, sc_npad, sg);
    }
  }
  launch_prep(bt, sg);
  ctx->launches += 1;
  cudaEventRecord(ev[1], sg);
  int nl = 0;
  if (mode != 3) {
    // graph + degree, optionally in L2-sized sub-chunks (see l2_chunk); the graph kernel has its own event pair.
    const int gch = l2_chunk(ctx, bt.B, bt.n, p);
    for (int b0 = 0; b0 < bt.B; b0 += gch) {
      Batch sb = (gch < bt.B) ? sub_batch(bt, b0, std::min(gch, bt.B - b0)) : bt;
      while ((int)ctx->graph_ev.size() < ctx->graph_ev_used + 2) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return TZR_ERR_CUDA;
        ctx->graph_ev.push_back(e);
      }
      cudaEventRecord(ctx->graph_ev[ctx->graph_ev_used], sg);
      nl += launch_graph(sb, sg, ctx->num_sms) - 1;
      cudaEventRecord(ctx->graph_ev[ctx->graph_ev_used + 1], sg);
      ctx->graph_ev_used += 2;
      if (sg != st) {  // two lanes (never combined with L2 sub-chunking: gch == B there)
        cudaEventRecord(gdone, sg);
        cudaStreamWaitEvent(st, gdone, 0);
      }
      launch_degree(sb, st);
      nl += 2;
    }
    cudaEventRecord(ev[2], st);
    if (bt.n > kMaxN) {
      const int rc = run_clique_large(ctx, bt, p, mode, st, &nl);
      if (rc) return rc;
    } else {
      launch_clique(bt, p, mode, st, &nl);
    }
  } else {
    if (sg != st) {
      cudaEventRecord(gdone, sg);
      cudaStreamWaitEvent(st, gdone, 0);
    }
    cudaEventRecord(ev[2], st);
  }
  cudaEventRecord(ev[3], st);
  launch_rot_trans(bt, p, mode != 3 ? 1 : 0, st);
  cudaEventRecord(ev[4], st);
  ctx->launches += nl + 1;
  return check_launch(ctx, "pipeline launch");
}

// Run the pipeline chunk by chunk on the compute stream.  ready[c] (optional) is an event the chunk's inputs wait for.
// bounds = n_chunks+1 ascending problem offsets (bounds[0] = 0, bounds[n_chunks] = B).
int run_chunked(tzr_ctx* ctx, Batch& bt, const tzr_params& p, const std::vector<int>& bounds,
                const cudaEvent_t* ready, const std::function<int(int)>& before_chunk = nullptr) {
  const int n_chunks = (int)bounds.size() - 1;
  if (!ctx->stage_log) {
    ctx->graph_ev_used = 0;
    ctx->stage_chunks = 0;
  }
  ctx->stage_first = ctx->stage_chunks;
  ctx->graph_first = ctx->graph_ev_used;
  while ((int)ctx->stage_ev.size() < 5 * (ctx->stage_first + n_chunks)) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return TZR_ERR_CUDA;
    ctx->stage_ev.push_back(e);
  }
  const bool lanes = n_chunks > 1 && ctx->gstream && ctx->hstream && l2_chunk(ctx, bt.B, bt.n, p) >= bt.B;
  if (lanes) {
    while ((int)ctx->gdone_ev.size() < n_chunks) {
      cudaEvent_t e;
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return TZR_ERR_CUDA;
      ctx->gdone_ev.push_back(e);
    }
    if (cudaEventRecord(ctx->join_ev, ctx->stream) != cudaSuccess) return TZR_ERR_CUDA;
    if (cudaStreamWaitEvent(ctx->gstream, ctx->join_ev, 0) != cudaSuccess) return TZR_ERR_CUDA;
    if (cudaStreamWaitEvent(ctx->hstream, ctx->join_ev, 0) != cudaSuccess) return TZR_ERR_CUDA;
  }
  for (int c = 0; c < n_chunks; ++c) {
    const int b0 = bounds[c], Bc = bounds[c + 1] - b0;
    cudaStream_t st = lanes ? ctx->hstream : ctx->stream;
    cudaStream_t sg = lanes ? ctx->gstream : ctx->stream;
    if (before_chunk) {  // host-side work that produces this chunk's inputs (staging + H2D enqueue)
      const int rcb = before_chunk(c);
      if (rcb) return rcb;
    }
    if (ready) {
      if (cudaStreamWaitEvent(sg, ready[c], 0) != cudaSuccess) return TZR_ERR_CUDA;
    }
    Batch sb = (n_chunks > 1) ? sub_batch(bt, b0, Bc) : bt;
    int rc = run_pipeline(ctx, sb, p, ctx->stage_ev.data() + 5 * (ctx->stage_first + c), st, sg, lanes ? ctx->gdone_ev[c] : nullptr);
    if (rc) return rc;
    if (n_chunks == 1) bt = sb;  // keep fields filled in by run_pipeline (beta, scale_mode, ...)
  }
  if (lanes) {  // everything later on ctx->stream (D2H, the caller's work) is ordered after both lanes
    if (cudaEventRecord(ctx->join_ev, ctx->hstream) != cudaSuccess) return TZR_ERR_CUDA;
    if (cudaStreamWaitEvent(ctx->stream, ctx->join_ev, 0) != cudaSuccess) return TZR_ERR_CUDA;
    if (cudaEventRecord(ctx->join_ev2, ctx->gstream) != cudaSuccess) return TZR_ERR_CUDA;
    if (cudaStreamWaitEvent(ctx->stream, ctx->join_ev2, 0) != cudaSuccess) return TZR_ERR_CUDA;
  }
  ctx->stage_chunks = ctx->stage_first + n_chunks;
  if (ctx->stage_log) ++ctx->stage_log_calls;
  ctx->last = bt;
  ctx->have_last = true;
  ctx->last_has_graph = effective_mode(p) != 3;  // NONE: populateVertices is never called (registration.cc:607-650)
  return TZR_OK;
}

}  // namespace

// ================================================================================================
extern "C" {

int tzr_abi_version(void) { return TZR_ABI_VERSION; }

const char* tzr_status_string(int s) {
  switch (s) {
    case TZR_OK: return "ok";
    case TZR_ERR_INVALID_ARG: return "invalid argument";
    case TZR_ERR_NO_DEVICE: return "no usable CUDA device (the B200 path has no CPU fallback)";
    case TZR_ERR_CUDA: return "CUDA error";
    case TZR_ERR_ALLOC: return "allocation failed";
    case TZR_ERR_UNSUPPORTED: return "unsupported parameter combination";
    case TZR_ERR_TOO_LARGE: return "problem too large";
    default: return "unknown";
  }
}

const char* tzr_last_error(const tzr_ctx* ctx) { return ctx ? ctx->last_error.c_str() : ""; }

void tzr_params_default(tzr_params* p) {
  if (!p) return;
  memset(p, 0, sizeof(*p));
  p->noise_bound = 0.01;
  p->cbar2 = 1;
  p->estimate_scaling = 1;
  p->rotation_estimation_algorithm = 0;
  p->rotation_gnc_factor = 1.4;
  p->rotation_max_iterations = 100;
  p->rotation_cost_threshold = 1e-6;
  p->rotation_tim_graph = 0;
  p->inlier_selection_mode = 0;
  p->kcore_heuristic_threshold = 0.5;
  p->use_max_clique = 1;
  p->max_clique_exact_solution = 1;
  p->max_clique_time_limit = 3600;
  p->max_clique_num_threads = 0;
}

int tzr_words_per_row(int n) { return words64(n); }

int tzr_ctx_create(int device, tzr_ctx** out) {
  if (!out) return TZR_ERR_INVALID_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) return TZR_ERR_NO_DEVICE;
  if (device < 0) {
    if (cudaGetDevice(&device) != cudaSuccess) return TZR_ERR_NO_DEVICE;
  }
  if (device >= count) return TZR_ERR_INVALID_ARG;
  if (cudaSetDevice(device) != cudaSuccess) return TZR_ERR_NO_DEVICE;
  tzr_ctx* ctx = new tzr_ctx();
  ctx->device = device;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->num_sms = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete ctx;
    return TZR_ERR_CUDA;
  }
  for (int i = 0; i < 5; ++i) cudaEventCreate(&ctx->ev[i]);
  cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
  {
    int least = 0, greatest = 0;
    cudaDeviceGetStreamPriorityRange(&least, &greatest);
    cudaStreamCreateWithPriority(&ctx->gstream, cudaStreamNonBlocking, least);
    cudaStreamCreateWithPriority(&ctx->hstream, cudaStreamNonBlocking, greatest);
  }
  cudaEventCreateWithFlags(&ctx->join_ev, cudaEventDisableTiming);
  cudaEventCreateWithFlags(&ctx->join_ev2, cudaEventDisableTiming);
  *out = ctx;
  return TZR_OK;
}

int tzr_ctx_destroy(tzr_ctx* ctx) {
  if (!ctx) return TZR_OK;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  DevBuf* bufs[] = {&ctx->src, &ctx->dst, &ctx->sf, &ctx->df, &ctx->pk, &ctx->opnd, &ctx->tclist, &ctx->gc, &ctx->adj, &ctx->deg, &ctx->nedges,
                    &ctx->hclq, &ctx->hsize, &ctx->clq, &ctx->L, &ctx->alive, &ctx->best_bits, &ctx->alive_cnt, &ctx->root_ctr,
                    &ctx->lock, &ctx->flg, &ctx->kfinal, &ctx->tstart, &ctx->stack, &ctx->cv, &ctx->centry, &ctx->ps, &ctx->pd, &ctx->wgt,
                    &ctx->res, &ctx->skey, &ctx->sidx, &ctx->sorted, &ctx->rmask, &ctx->tmask, &ctx->sol, &ctx->dbg,
                    &ctx->misc, &ctx->sc_x, &ctx->sc_r, &ctx->sc_key, &ctx->sc_idx, &ctx->m_in, &ctx->m_scratch, &ctx->m_out, &ctx->cert,
                    &ctx->large, &ctx->compact};
  for (DevBuf* b : bufs)
    if (b->p) cudaFree(b->p);
  if (ctx->h_pin) cudaFreeHost(ctx->h_pin);
  for (int i = 0; i < 5; ++i)
    if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
  for (cudaEvent_t e : ctx->chunk_ev) cudaEventDestroy(e);
  for (cudaEvent_t e : ctx->stage_ev) cudaEventDestroy(e);
  for (cudaEvent_t e : ctx->graph_ev) cudaEventDestroy(e);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  certify_release(ctx->solver_handle);
  if (ctx->gstream) cudaStreamDestroy(ctx->gstream);
  if (ctx->hstream) cudaStreamDestroy(ctx->hstream);
  if (ctx->join_ev) cudaEventDestroy(ctx->join_ev);
  if (ctx->join_ev2) cudaEventDestroy(ctx->join_ev2);
  for (cudaEvent_t e : ctx->gdone_ev) cudaEventDestroy(e);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return TZR_OK;
}

int tzr_ctx_set_stream(tzr_ctx* ctx, void* s) {
  if (!ctx) return TZR_ERR_INVALID_ARG;
  cudaStreamSynchronize(ctx->stream);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  ctx->stream = (cudaStream_t)s;
  ctx->own_stream = false;
  return TZR_OK;
}

int tzr_ctx_synchronize(tzr_ctx* ctx) {
  if (!ctx) return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  CK(cudaStreamSynchronize(ctx->stream));
  return TZR_OK;
}

int64_t tzr_ctx_kernel_launches(const tzr_ctx* ctx) { return ctx ? ctx->launches : 0; }

int tzr_ctx_set_flags(tzr_ctx* ctx, uint32_t flags) {
  if (!ctx) return TZR_ERR_INVALID_ARG;
  ctx->flags = flags;
  return TZR_OK;
}

int64_t tzr_ctx_filter_mismatches(tzr_ctx* ctx) {
  if (!ctx || !ctx->dbg.p) return -1;
  unsigned long long v = 0;
  cudaStreamSynchronize(ctx->stream);
  if (cudaMemcpy(&v, ctx->dbg.p, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return (int64_t)v;
}

int tzr_ctx_debug_counters(tzr_ctx* ctx, int64_t* out16) {
  if (!ctx || !ctx->dbg.p || !out16) return TZR_ERR_INVALID_ARG;
  cudaStreamSynchronize(ctx->stream);
  if (cudaMemcpy(out16, ctx->dbg.p, 16 * sizeof(int64_t), cudaMemcpyDeviceToHost) != cudaSuccess) return TZR_ERR_CUDA;
  return TZR_OK;
}

int64_t tzr_ctx_filter_rechecks(tzr_ctx* ctx) {
  if (!ctx || !ctx->dbg.p) return -1;
  unsigned long long v = 0;
  cudaStreamSynchronize(ctx->stream);
  if (cudaMemcpy(&v, (unsigned long long*)ctx->dbg.p + 1, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return (int64_t)v;
}

// ------------------------------------------------------------------------------------------------
// stage 1
// ------------------------------------------------------------------------------------------------
int tzr_graph_build(tzr_ctx* ctx, const double* src, const double* dst, int n, double beta, uint64_t* adj_bits,
                    int32_t* degree, int64_t* n_edges) {
  if (!ctx || !src || !dst || !adj_bits || n <= 0) return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  Batch bt;
  int rc = setup_batch(ctx, 1, n, true, &bt);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  bt.beta = beta;
  CK(cudaMemcpyAsync((void*)bt.src, src, (size_t)n * 3 * sizeof(double), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync((void*)bt.dst, dst, (size_t)n * 3 * sizeof(double), cudaMemcpyHostToDevice, st));
  if (ctx->flags & 6u) cudaMemsetAsync((void*)ctx->dbg.p, 0, 16 * sizeof(unsigned long long), st);
  launch_prep(bt, st);
  ctx->launches += 2 + launch_graph(bt, st, ctx->num_sms);
  launch_degree(bt, st);
  rc = check_launch(ctx, "graph build");
  if (rc) return rc;
  CK(cudaMemcpy2DAsync(adj_bits, (size_t)words64(n) * 8, bt.adj, (size_t)pitch64(n) * 8, (size_t)words64(n) * 8, n,
                       cudaMemcpyDeviceToHost, st));
  if (degree) CK(cudaMemcpyAsync(degree, bt.deg, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  unsigned long long e2 = 0;
  CK(cudaMemcpyAsync(&e2, bt.n_edges2, sizeof(e2), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (n_edges) *n_edges = (int64_t)(e2 / 2);
  ctx->last = bt;
  ctx->have_last = true;
  ctx->last_has_graph = true;
  return TZR_OK;
}

// ------------------------------------------------------------------------------------------------
// stage 2
// ------------------------------------------------------------------------------------------------
int tzr_max_clique(tzr_ctx* ctx, const uint64_t* adj_bits, int n, int mode, double kcore_thr, double time_limit_s,
                   int32_t* clique, int32_t* clique_size, int32_t* proven_optimal) {
  if (!ctx || !adj_bits || !clique || !clique_size || n <= 0) return TZR_ERR_INVALID_ARG;
  if (mode < 0 || mode > 2) return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  Batch bt;
  int rc = setup_batch(ctx, 1, n, false, &bt);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  CK(cudaMemsetAsync(bt.adj, 0, (size_t)n * pitch64(n) * 8, st));
  CK(cudaMemcpy2DAsync(bt.adj, (size_t)pitch64(n) * 8, adj_bits, (size_t)words64(n) * 8, (size_t)words64(n) * 8, n,
                       cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(bt.n_edges2, 0, sizeof(unsigned long long), st));
  launch_degree(bt, st, true);
  tzr_params p;
  tzr_params_default(&p);
  p.kcore_heuristic_threshold = kcore_thr;
  if (mode == 0 && time_limit_s > 0 && time_limit_s < 1e7) bt.budget_ns = (unsigned long long)(time_limit_s * 1e9);
  int nl = 1;
  if (n > kMaxN) {
    rc = run_clique_large(ctx, bt, p, mode, st, &nl);
    if (rc) return rc;
  } else {
    launch_clique(bt, p, mode, st, &nl);
  }
  ctx->launches += nl;
  rc = check_launch(ctx, "max clique");
  if (rc) return rc;
  int32_t L = 0, fl = 0;
  CK(cudaMemcpyAsync(&L, bt.L, sizeof(L), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&fl, bt.flags, sizeof(fl), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (L > 0) CK(cudaMemcpy(clique, bt.clq, (size_t)L * sizeof(int32_t), cudaMemcpyDeviceToHost));
  std::sort(clique, clique + L);  // registration.cc:636
  *clique_size = L;
  if (proven_optimal) *proven_optimal = (mode == 0 && !(fl & 1)) ? ((fl & 12) ? 2 : 1) : 0;  // as tzr_solution
  return TZR_OK;
}

// ------------------------------------------------------------------------------------------------
// stage 3 / 4 / scalar TLS
// ------------------------------------------------------------------------------------------------
int tzr_gnc_tls_rotation(tzr_ctx* ctx, const double* src, const double* dst, int m, double noise_bound,
                         double gnc_factor, uint64_t max_iterations, double cost_threshold, double* R,
                         uint8_t* inlier_mask, double* cost, int32_t* iterations) {
  return tzr_rotation_solve(ctx, 0, src, dst, m, noise_bound, gnc_factor, max_iterations, cost_threshold, R,
                            inlier_mask, cost, iterations);
}

int tzr_rotation_solve(tzr_ctx* ctx, int algorithm, const double* src, const double* dst, int m, double noise_bound,
                       double gnc_factor, uint64_t max_iterations, double cost_threshold, double* R,
                       uint8_t* inlier_mask, double* cost, int32_t* iterations) {
  if (!ctx || !src || !dst || !R || m <= 0 || algorithm < 0 || algorithm > 2) return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  const size_t pts = (size_t)m * 3 * sizeof(double);
  int rc = ensure(ctx, ctx->misc, 2 * pts + 2 * (size_t)m * sizeof(double) + (size_t)m + 16 * sizeof(double) + 64);
  if (rc) return rc;
  char* base = (char*)ctx->misc.p;
  double* d_src = (double*)base;
  double* d_dst = d_src + (size_t)m * 3;
  double* d_w = d_dst + (size_t)m * 3;
  double* d_r = d_w + m;
  double* d_out = d_r + m;  // 9 R + 1 cost
  int* d_it = (int*)(d_out + 10);
  uint8_t* d_mask = (uint8_t*)(d_out + 12);
  CK(cudaMemcpyAsync(d_src, src, pts, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_dst, dst, pts, cudaMemcpyHostToDevice, st));
  launch_gnc_only(algorithm, d_src, d_dst, m, noise_bound, gnc_factor, max_iterations, cost_threshold, d_w, d_r, d_out, d_mask,
                  d_out + 9, d_it, st);
  ctx->launches += 1;
  rc = check_launch(ctx, "gnc");
  if (rc) return rc;
  double hout[10];
  int it = 0;
  CK(cudaMemcpyAsync(hout, d_out, sizeof(hout), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&it, d_it, sizeof(int), cudaMemcpyDeviceToHost, st));
  if (inlier_mask) CK(cudaMemcpyAsync(inlier_mask, d_mask, m, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  memcpy(R, hout, 9 * sizeof(double));
  if (cost) *cost = hout[9];
  if (iterations) *iterations = it;
  return TZR_OK;
}

int tzr_tls_translation(tzr_ctx* ctx, const double* src, const double* dst, int m, double noise_bound, double cbar2,
                        double* t3, uint8_t* inlier_mask) {
  if (!ctx || !src || !dst || !t3 || m <= 0) return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  const size_t pts = (size_t)m * 3 * sizeof(double);
  const int npad = next_pow2_host(2 * m);
  const size_t key_bytes = ((size_t)3 * npad + (size_t)3 * m) * sizeof(double);
  const size_t idx_bytes = (size_t)3 * npad * sizeof(int32_t);
  int rc = ensure(ctx, ctx->misc, 2 * pts + key_bytes + idx_bytes + (size_t)m + 64);
  if (rc) return rc;
  double* d_src = (double*)ctx->misc.p;
  double* d_dst = d_src + (size_t)m * 3;
  double* d_key = d_dst + (size_t)m * 3;
  int32_t* d_idx = (int32_t*)(d_key + (size_t)3 * npad + (size_t)3 * m);
  double* d_t = (double*)(d_idx + (size_t)3 * npad + ((3 * npad) & 1));
  uint8_t* d_mask = (uint8_t*)(d_t + 4);
  // the tail (d_t, d_mask) needs 4 doubles + m bytes more
  rc = ensure(ctx, ctx->misc, (size_t)((char*)d_mask - (char*)ctx->misc.p) + (size_t)m + 64);
  if (rc) return rc;
  if ((double*)ctx->misc.p != d_src) {  // buffer moved on growth: recompute pointers
    d_src = (double*)ctx->misc.p;
    d_dst = d_src + (size_t)m * 3;
    d_key = d_dst + (size_t)m * 3;
    d_idx = (int32_t*)(d_key + (size_t)3 * npad + (size_t)3 * m);
    d_t = (double*)(d_idx + (size_t)3 * npad + ((3 * npad) & 1));
    d_mask = (uint8_t*)(d_t + 4);
  }
  CK(cudaMemcpyAsync(d_src, src, pts, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_dst, dst, pts, cudaMemcpyHostToDevice, st));
  const double beta = noise_bound * std::sqrt(cbar2);  // registration.cc:459
  launch_translation_only(d_src, d_dst, m, beta, d_key, d_idx, d_t, d_mask, st);
  ctx->launches += 1;
  rc = check_launch(ctx, "translation");
  if (rc) return rc;
  CK(cudaMemcpyAsync(t3, d_t, 3 * sizeof(double), cudaMemcpyDeviceToHost, st));
  if (inlier_mask) CK(cudaMemcpyAsync(inlier_mask, d_mask, m, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return TZR_OK;
}

int tzr_scalar_tls(tzr_ctx* ctx, const double* x, const double* ranges, int64_t m, double* estimate,
                   uint8_t* inliers) {
  if (!ctx || !x || !ranges || !estimate || m <= 1) return TZR_ERR_INVALID_ARG;  // reference asserts m > 1
  if (m > ((int64_t)1 << 22)) return TZR_ERR_TOO_LARGE;
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  int64_t npad = 1;
  while (npad < 2 * m) npad <<= 1;
  const size_t bytes = 2 * (size_t)m * 8 + (size_t)npad * 8 + (size_t)npad * 4 + 16 + (size_t)m + 64;
  int rc = ensure(ctx, ctx->misc, bytes);
  if (rc) return rc;
  double* d_x = (double*)ctx->misc.p;
  double* d_r = d_x + m;
  double* d_key = d_r + m;
  double* d_est = d_key + npad;
  int32_t* d_idx = (int32_t*)(d_est + 2);
  uint8_t* d_inl = (uint8_t*)(d_idx + npad);
  CK(cudaMemcpyAsync(d_x, x, (size_t)m * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_r, ranges, (size_t)m * 8, cudaMemcpyHostToDevice, st));
  launch_scalar_tls(d_x, d_r, m, d_key, d_idx, d_est, d_inl, st);
  ctx->launches += 1;
  rc = check_launch(ctx, "scalar tls");
  if (rc) return rc;
  CK(cudaMemcpyAsync(estimate, d_est, sizeof(double), cudaMemcpyDeviceToHost, st));
  if (inliers) CK(cudaMemcpyAsync(inliers, d_inl, (size_t)m, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return TZR_OK;
}

// ------------------------------------------------------------------------------------------------
// whole path
// ------------------------------------------------------------------------------------------------
int tzr_solve_batch_dev(tzr_ctx* ctx, const tzr_params* params, int B, int n, const double* src_dev,
                        const double* dst_dev, tzr_solution* solutions_dev, int32_t* cliques_dev) {
  if (!ctx || !params || !src_dev || !dst_dev || !solutions_dev) return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  Batch bt;
  int rc = setup_batch(ctx, B, n, false, &bt, params->rotation_tim_graph == 1);
  if (rc) return rc;
  bt.src = src_dev;
  bt.dst = dst_dev;
  // Sub-batches alternate between the two compute streams: the latency-bound clique / rotation kernels of one
  // sub-batch run under the issue-bound graph kernel of the next (TZR_DEV_CHUNKS overrides the count).
  static const int dev_chunks = [] {
    const char* e = std::getenv("TZR_DEV_CHUNKS");
    return e ? std::max(1, atoi(e)) : 1;
  }();
  std::vector<int> bounds{0};
  // n > kMaxN: one chunk (the clique stage waits for the batch's largest core; its scratch covers the whole batch)
  const int nch = (B >= 64 * dev_chunks && !params->estimate_scaling && n <= kMaxN) ? dev_chunks : 1;
  for (int c = 1; c <= nch; ++c) bounds.push_back((int)((long long)B * c / nch));
  rc = run_chunked(ctx, bt, *params, bounds, nullptr);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  CK(cudaMemcpyAsync(solutions_dev, bt.sol, (size_t)B * sizeof(tzr_solution), cudaMemcpyDeviceToDevice, st));
  if (cliques_dev)
    CK(cudaMemcpyAsync(cliques_dev, bt.sorted_clq, (size_t)B * n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
  return TZR_OK;
}

static int solve_uniform_host(tzr_ctx* ctx, const tzr_params* params, int B, int n, const double* const* src,
                              const double* const* dst, tzr_solution* solutions, int32_t* cliques, int max_n,
                              uint8_t* rot_inliers, uint8_t* trans_inliers) {
  cudaSetDevice(ctx->device);
  Batch bt;
  int rc = setup_batch(ctx, B, n, true, &bt, params->rotation_tim_graph == 1);
  if (rc) return rc;
  cudaStream_t st = ctx->stream;
  const size_t per = (size_t)n * 3 * sizeof(double);
  rc = ensure_pinned(ctx, 2 * per * B + (size_t)B * sizeof(tzr_solution) + (size_t)B * n * sizeof(int32_t));
  if (rc) return rc;
  char* hp = (char*)ctx->h_pin;
  double* h_src = (double*)hp;
  double* h_dst = (double*)(hp + per * B);
  tzr_solution* h_sol = (tzr_solution*)(hp + 2 * per * B);
  int32_t* h_clq = (int32_t*)(hp + 2 * per * B + (size_t)B * sizeof(tzr_solution));
  // Fast path: the caller's buffers are one contiguous, page-locked block (e.g. a pinned batch tensor) ->
  // DMA straight from user memory.  Otherwise stage through the context's pinned buffer.
  bool contiguous = true;
  for (int b = 1; b < B; ++b)
    contiguous &= (src[b] == src[0] + (size_t)b * n * 3) && (dst[b] == dst[0] + (size_t)b * n * 3);
  bool pinned = false;
  if (contiguous) {
    cudaPointerAttributes a1, a2;
    if (cudaPointerGetAttributes(&a1, src[0]) == cudaSuccess && cudaPointerGetAttributes(&a2, dst[0]) == cudaSuccess)
      pinned = (a1.type == cudaMemoryTypeHost) && (a2.type == cudaMemoryTypeHost);
    cudaGetLastError();
  }
  const double* hs = src[0];
  const double* hd = dst[0];
  const bool staged = !(contiguous && pinned);  // stage through the context's pinned buffer, chunk by chunk (below)
  if (staged) {
    hs = h_src;
    hd = h_dst;
  }
  // Chunked pipeline: the H2D copy of chunk k+1 (copy stream) overlaps the kernels of chunk k (compute streams).
  // PCIe moves a problem ~3x faster than the kernels consume it, so only the first chunk's copy is exposed: it is
  // kept small (B/32) and the later chunks grow (3B/32, B/8, then B/4 each) to keep launch tails few.
  std::vector<int> bounds{0};
  if (B >= 64 && !params->estimate_scaling && n <= kMaxN) {
    const int unit = std::max(8, B / 32);
    const int sizes[3] = {unit, 3 * unit, 4 * unit};
    for (int k = 0; bounds.back() < B; ++k) {
      const int sz = k < 3 ? sizes[k] : 8 * unit;
      bounds.push_back(std::min(B, bounds.back() + sz));
    }
  } else {
    bounds.push_back(B);
  }
  const int n_chunks = (int)bounds.size() - 1;
  while ((int)ctx->chunk_ev.size() < n_chunks + 1) {
    cudaEvent_t e;
    CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ctx->chunk_ev.push_back(e);
  }
  cudaStream_t cs = n_chunks > 1 ? ctx->copy_stream : st;
  if (n_chunks > 1) {
    // the copy stream must not overwrite inputs that an earlier call's kernels may still read
    CK(cudaEventRecord(ctx->chunk_ev[n_chunks], st));
    CK(cudaStreamWaitEvent(cs, ctx->chunk_ev[n_chunks], 0));
  }
  // Per chunk, on the host: (staged inputs only) copy the chunk into the pinned area with a few threads, then enqueue its
  // H2D copies; run_chunked enqueues the chunk's kernels right after, so the GPU works on chunk k while the host stages
  // chunk k+1.
  auto feed_chunk = [&](int c) -> int {
    const int b0 = bounds[c], Bc = bounds[c + 1] - b0;
    if (staged) {
      parallel_stage((char*)h_src + per * b0, src, b0, Bc, per);
      parallel_stage((char*)h_dst + per * b0, dst, b0, Bc, per);
    }
    if (cudaMemcpyAsync((void*)(bt.src + (size_t)b0 * n * 3), (const char*)hs + per * b0, per * Bc,
                        cudaMemcpyHostToDevice, cs) != cudaSuccess ||
        cudaMemcpyAsync((void*)(bt.dst + (size_t)b0 * n * 3), (const char*)hd + per * b0, per * Bc,
                        cudaMemcpyHostToDevice, cs) != cudaSuccess)
      return TZR_ERR_CUDA;
    if (n_chunks > 1 && cudaEventRecord(ctx->chunk_ev[c], cs) != cudaSuccess) return TZR_ERR_CUDA;
    return TZR_OK;
  };
  rc = run_chunked(ctx, bt, *params, bounds, n_chunks > 1 ? ctx->chunk_ev.data() : nullptr, feed_chunk);
  if (rc) return rc;
  CK(cudaMemcpyAsync(h_sol, bt.sol, (size_t)B * sizeof(tzr_solution), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (cliques) {  // only the used prefix of every clique row crosses PCIe (rows are n int32 wide, cliques ~5 % of n)
    int max_m = 0;
    for (int b = 0; b < B; ++b) max_m = std::max(max_m, std::min(n, std::max(0, h_sol[b].clique_size)));
    if (max_m > 0) {
      CK(cudaMemcpy2DAsync(h_clq, (size_t)n * sizeof(int32_t), bt.sorted_clq, (size_t)n * sizeof(int32_t),
                           (size_t)max_m * sizeof(int32_t), B, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
    }
  }
  memcpy(solutions, h_sol, (size_t)B * sizeof(tzr_solution));
  for (int b = 0; b < B; ++b)
    if (h_sol[b].clique_proven_optimal == -2) {
      ctx->last_error = "COMPLETE TIM graph of this clique does not fit the rotation workspace";
      return TZR_ERR_TOO_LARGE;
    }
  if (B == 1 && h_sol[0].valid) {  // single-problem masks (getRotationInliersMask / getTranslationInliersMask)
    const long long m = h_sol[0].clique_size;
    const long long n_rot = params->rotation_tim_graph == 1 ? m * (m - 1) / 2 : m;
    if (rot_inliers && n_rot > 0) CK(cudaMemcpy(rot_inliers, bt.rot_mask, (size_t)n_rot, cudaMemcpyDeviceToHost));
    if (trans_inliers && m > 0) CK(cudaMemcpy(trans_inliers, bt.trans_mask, (size_t)m, cudaMemcpyDeviceToHost));
  }
  if (cliques)
    for (int b = 0; b < B; ++b) {
      const int m = std::max(0, std::min(n, h_sol[b].clique_size));
      memcpy(cliques + (size_t)b * max_n, h_clq + (size_t)b * n, (size_t)m * sizeof(int32_t));
    }
  return TZR_OK;
}

int tzr_solve(tzr_ctx* ctx, const tzr_params* params, const double* src, const double* dst, int n,
              tzr_solution* solution, int32_t* clique, uint8_t* rot_inliers, uint8_t* trans_inliers) {
  if (!ctx || !params || !src || !dst || !solution || n <= 0) return TZR_ERR_INVALID_ARG;
  const double* s[1] = {src};
  const double* d[1] = {dst};
  int rc = solve_uniform_host(ctx, params, 1, n, s, d, solution, clique, n, rot_inliers, trans_inliers);
  if (rc) return rc;
  double st4[4] = {0, 0, 0, 0};
  if (tzr_last_stage_ms(ctx, &st4[0], &st4[1], &st4[2], &st4[3]) == TZR_OK) {
    for (int i = 0; i < 4; ++i) solution->stage_ms[i] = st4[i];  // prep | graph | clique | rot+trans
    solution->stage_ms[6] = st4[0] + st4[1] + st4[2] + st4[3];
  }
  return TZR_OK;
}

int tzr_solve_batch(tzr_ctx* ctx, const tzr_params* params, int B, const int32_t* n, const double* const* src,
                    const double* const* dst, tzr_solution* solutions, int32_t* cliques, int max_n) {
  if (!ctx || !params || !n || !src || !dst || !solutions || B <= 0) return TZR_ERR_INVALID_ARG;
  bool uniform = true;
  for (int b = 1; b < B; ++b) uniform &= (n[b] == n[0]);
  if (cliques && max_n < *std::max_element(n, n + B)) return TZR_ERR_INVALID_ARG;
  if (uniform) return solve_uniform_host(ctx, params, B, n[0], src, dst, solutions, cliques, max_n, nullptr, nullptr);
  // ragged batch: problems of equal size are solved together (one device batch per distinct n, largest first)
  std::vector<int> order(B);
  for (int b = 0; b < B; ++b) order[b] = b;
  std::stable_sort(order.begin(), order.end(), [&](int a, int c) { return n[a] > n[c]; });
  std::vector<const double*> gs, gd;
  std::vector<tzr_solution> gsol;
  std::vector<int32_t> gclq;
  for (int lo = 0; lo < B;) {
    int hi = lo;
    while (hi < B && n[order[hi]] == n[order[lo]]) ++hi;
    const int G = hi - lo, ng = n[order[lo]];
    if (ng <= 0) return TZR_ERR_INVALID_ARG;
    gs.resize(G);
    gd.resize(G);
    gsol.resize(G);
    for (int g = 0; g < G; ++g) {
      gs[g] = src[order[lo + g]];
      gd[g] = dst[order[lo + g]];
      if (!gs[g] || !gd[g]) return TZR_ERR_INVALID_ARG;
    }
    if (cliques) gclq.resize((size_t)G * ng);
    int rc = solve_uniform_host(ctx, params, G, ng, gs.data(), gd.data(), gsol.data(), cliques ? gclq.data() : nullptr,
                                ng, nullptr, nullptr);
    if (rc) return rc;
    for (int g = 0; g < G; ++g) {
      const int b = order[lo + g];
      solutions[b] = gsol[g];
      if (cliques) {
        const int m = std::max(0, std::min(ng, gsol[g].clique_size));
        memcpy(cliques + (size_t)b * max_n, gclq.data() + (size_t)g * ng, (size_t)m * sizeof(int32_t));
      }
    }
    lo = hi;
  }
  return TZR_OK;
}

int tzr_last_graph(tzr_ctx* ctx, int b, uint64_t* adj_bits, int32_t* degree) {
  if (!ctx || !ctx->have_last || b < 0 || b >= ctx->last.B) return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  const Batch& bt = ctx->last;
  const int n = bt.n;
  if (!ctx->last_has_graph) {  // inlier selection NONE: the reference never populates the graph -> no edges
    if (adj_bits) memset(adj_bits, 0, (size_t)n * words64(n) * 8);
    if (degree) memset(degree, 0, (size_t)n * 4);
    return TZR_OK;
  }
  cudaStream_t st = ctx->stream;
  if (adj_bits)
    CK(cudaMemcpy2DAsync(adj_bits, (size_t)words64(n) * 8, bt.adj + (size_t)b * n * pitch64(n), (size_t)pitch64(n) * 8,
                         (size_t)words64(n) * 8, n, cudaMemcpyDeviceToHost, st));
  if (degree) CK(cudaMemcpyAsync(degree, bt.deg + (size_t)b * n, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return TZR_OK;
}

int tzr_last_graph_info(const tzr_ctx* ctx, int32_t* B, int32_t* n, int32_t* has_graph, uint64_t* generation) {
  if (!ctx) return TZR_ERR_INVALID_ARG;
  if (B) *B = ctx->have_last ? ctx->last.B : 0;
  if (n) *n = ctx->have_last ? ctx->last.n : 0;
  if (has_graph) *has_graph = (ctx->have_last && ctx->last_has_graph) ? 1 : 0;
  if (generation) *generation = ctx->generation;
  return TZR_OK;
}

int tzr_match_correspondences(tzr_ctx* ctx, const float* src_pts, int ns, const float* dst_pts, int nd,
                              const float* src_feat, const float* dst_feat, int dim, int use_absolute_scale,
                              int use_crosscheck, int use_tuple_test, float tuple_scale, uint64_t tuple_seed,
                              int32_t* pairs, int64_t capacity, int64_t* n_pairs, float* global_scale) {
  if (!ctx || !src_pts || !dst_pts || !src_feat || !dst_feat || !pairs || !n_pairs || ns <= 0 || nd <= 0 ||
      dim < 1 || dim > kMatchMaxDim || capacity < 0)
    return TZR_ERR_INVALID_ARG;
  if ((long long)ns + nd > (1ll << 30)) return TZR_ERR_TOO_LARGE;
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  const size_t pb_s = (size_t)ns * 3 * 4, pb_d = (size_t)nd * 3 * 4, fb_s = (size_t)ns * dim * 4,
               fb_d = (size_t)nd * dim * 4;
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  int rc;
  if ((rc = ensure(ctx, ctx->m_in, al(pb_s) + al(pb_d) + al(fb_s) + al(fb_d))) != TZR_OK) return rc;
  if ((rc = ensure(ctx, ctx->m_scratch, match_scratch_bytes(ns, nd))) != TZR_OK) return rc;
  const size_t cap = (size_t)ns + nd;
  if ((rc = ensure(ctx, ctx->m_out, cap * 8 + 256)) != TZR_OK) return rc;
  char* in = (char*)ctx->m_in.p;
  float* d_sp = (float*)in;
  float* d_dp = (float*)(in + al(pb_s));
  float* d_sf = (float*)(in + al(pb_s) + al(pb_d));
  float* d_df = (float*)(in + al(pb_s) + al(pb_d) + al(fb_s));
  int32_t* d_pairs = (int32_t*)ctx->m_out.p;
  int* d_count = (int*)((char*)ctx->m_out.p + cap * 8);
  float* d_g = (float*)(d_count + 1);
  CK(cudaMemcpyAsync(d_sp, src_pts, pb_s, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_dp, dst_pts, pb_d, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_sf, src_feat, fb_s, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_df, dst_feat, fb_d, cudaMemcpyHostToDevice, st));
  const int nl = launch_match(d_sp, ns, d_dp, nd, d_sf, d_df, dim, use_absolute_scale, use_crosscheck,
                              use_tuple_test, tuple_scale, tuple_seed, ctx->m_scratch.p, d_pairs, d_count, d_g,
                              ctx->num_sms, st);
  if (nl < 0) return nl;
  ctx->launches += nl;
  if ((rc = check_launch(ctx, "matcher launch")) != TZR_OK) return rc;
  struct {
    int count;
    float g;
  } tail;
  CK(cudaMemcpyAsync(&tail, d_count, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  *n_pairs = tail.count;
  if (global_scale) *global_scale = tail.g;
  if ((int64_t)tail.count > capacity) {
    ctx->last_error = "pairs capacity too small";
    return TZR_ERR_INVALID_ARG;
  }
  if (tail.count > 0) {
    CK(cudaMemcpyAsync(pairs, d_pairs, (size_t)tail.count * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  return TZR_OK;
}

void tzr_certifier_params_default(tzr_certifier_params* p) {
  if (!p) return;
  p->noise_bound = 0.01;      // certification.h:74
  p->cbar2 = 1;               // :80
  p->sub_optimality = 1e-3;   // :87
  p->max_iterations = 2e2;    // :92
  p->gamma_tau = 1.999999;    // :98
  p->eig_decomposition_solver = 0;
  p->reserved = 0;
}

int tzr_certify(tzr_ctx* ctx, const tzr_certifier_params* params, const double* R_colmajor9, const double* src_3xN,
                const double* dst_3xN, const double* theta, int n, tzr_certification_result* result, double* traj,
                int traj_capacity) {
  if (!ctx || !params || !R_colmajor9 || !src_3xN || !dst_3xN || !theta || !result || n <= 0 || traj_capacity < 0)
    return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  int opt = 0, iters = 0;
  double best = 0;
  const int rc = certify_device(0, params->noise_bound, params->cbar2, params->sub_optimality, params->max_iterations,
                                params->gamma_tau, R_colmajor9, src_3xN, dst_3xN, theta, n, &opt, &best, &iters, traj,
                                traj_capacity, nullptr, nullptr, nullptr, nullptr, &ctx->cert.p, &ctx->cert.cap,
                                &ctx->solver_handle, &ctx->launches, ctx->stream, &ctx->last_error);
  if (rc != TZR_OK) return rc;
  result->is_optimal = opt;
  result->n_iterations = iters;
  result->best_suboptimality = best;
  return TZR_OK;
}

int tzr_certifier_initial_matrix(tzr_ctx* ctx, const tzr_certifier_params* params, const double* R_colmajor9,
                                 const double* src_3xN, const double* dst_3xN, const double* theta, int n,
                                 double* M_init, double* mu) {
  if (!ctx || !params || !R_colmajor9 || !src_3xN || !dst_3xN || !theta || !M_init || !mu || n <= 0)
    return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  return certify_device(1, params->noise_bound, params->cbar2, 0, 0, 0, R_colmajor9, src_3xN, dst_3xN, theta, n,
                        nullptr, nullptr, nullptr, nullptr, 0, M_init, mu, nullptr, nullptr, &ctx->cert.p,
                        &ctx->cert.cap, &ctx->solver_handle, &ctx->launches, ctx->stream, &ctx->last_error);
}

int tzr_certifier_dual_projection(tzr_ctx* ctx, const double* W, const double* theta, int n, double* W_dual) {
  if (!ctx || !W || !theta || !W_dual || n <= 0) return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  return certify_device(2, 0, 0, 0, 0, 0, nullptr, nullptr, nullptr, theta, n, nullptr, nullptr, nullptr, nullptr, 0,
                        nullptr, nullptr, W, W_dual, &ctx->cert.p, &ctx->cert.cap, &ctx->solver_handle, &ctx->launches, ctx->stream,
                        &ctx->last_error);
}

int tzr_compute_fpfh(tzr_ctx* ctx, const float* pts, int n, double normal_search_radius, double fpfh_search_radius,
                     float* fpfh_out, float* normals_out) {
  if (!ctx || !pts || !fpfh_out || n <= 0 || !(normal_search_radius > 0) || !(fpfh_search_radius > 0))
    return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t pb = (size_t)n * 12, nb = (size_t)n * 16, hb = (size_t)n * 33 * 4;
  int rc;
  if ((rc = ensure(ctx, ctx->m_in, al(pb))) != TZR_OK) return rc;
  const size_t gb = fpfh_grid_scratch_bytes(n);
  if ((rc = ensure(ctx, ctx->m_scratch, al(nb) + al(hb) + 256 + gb)) != TZR_OK) return rc;
  if ((rc = ensure(ctx, ctx->m_out, al(hb))) != TZR_OK) return rc;
  float* d_pts = (float*)ctx->m_in.p;
  float4* d_normals = (float4*)ctx->m_scratch.p;
  float* d_spfh = (float*)((char*)ctx->m_scratch.p + al(nb));
  int* d_overflow = (int*)((char*)ctx->m_scratch.p + al(nb) + al(hb));
  float* d_out = (float*)ctx->m_out.p;
  CK(cudaMemcpyAsync(d_pts, pts, pb, cudaMemcpyHostToDevice, st));
  void* d_grid = gb ? (void*)((char*)ctx->m_scratch.p + al(nb) + al(hb) + 256) : nullptr;
  ctx->launches += launch_fpfh(d_pts, n, normal_search_radius, fpfh_search_radius, d_normals, d_spfh, d_out,
                               d_overflow, d_grid, st);
  if ((rc = check_launch(ctx, "fpfh launch")) != TZR_OK) return rc;
  int overflow = 0;
  CK(cudaMemcpyAsync(&overflow, d_overflow, sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(fpfh_out, d_out, hb, cudaMemcpyDeviceToHost, st));
  if (normals_out) CK(cudaMemcpyAsync(normals_out, d_normals, nb, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (overflow) {
    ctx->last_error = "a point has more than 4096 neighbours inside a search radius";
    return TZR_ERR_TOO_LARGE;
  }
  return TZR_OK;
}

int tzr_feature_nn(tzr_ctx* ctx, const float* query, int nq, const float* db, int ndb, int dim, int32_t* nn_index,
                   float* nn_dist) {
  if (!ctx || !query || !db || !nn_index || nq <= 0 || ndb <= 0 || dim < 1 || dim > kMatchMaxDim)
    return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  cudaStream_t st = ctx->stream;
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t qb = (size_t)nq * dim * 4, dbb = (size_t)ndb * dim * 4;
  int rc;
  if ((rc = ensure(ctx, ctx->m_in, al(qb) + al(dbb))) != TZR_OK) return rc;
  if ((rc = ensure(ctx, ctx->m_out, (size_t)nq * 8)) != TZR_OK) return rc;
  float* d_q = (float*)ctx->m_in.p;
  float* d_db = (float*)((char*)ctx->m_in.p + al(qb));
  unsigned long long* d_best = (unsigned long long*)ctx->m_out.p;
  CK(cudaMemcpyAsync(d_q, query, qb, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_db, db, dbb, cudaMemcpyHostToDevice, st));
  ctx->launches += launch_feature_nn(d_q, nq, d_db, ndb, dim, d_best, ctx->num_sms, st);
  if ((rc = check_launch(ctx, "feature nn launch")) != TZR_OK) return rc;
  std::vector<unsigned long long> h((size_t)nq);
  CK(cudaMemcpyAsync(h.data(), d_best, (size_t)nq * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (int q = 0; q < nq; ++q) {
    nn_index[q] = (int32_t)(h[q] & 0xffffffffu);
    if (nn_dist) {
      const uint32_t bits = (uint32_t)(h[q] >> 32);
      memcpy(&nn_dist[q], &bits, 4);
    }
  }
  return TZR_OK;
}

static int sum_stage_events(tzr_ctx* ctx, int c0, int c1, int g0, int g1, double acc[4]) {
  for (int i = 0; i < 4; ++i) acc[i] = 0;
  for (int c = c0; c < c1; ++c)
    for (int i = 0; i < 4; ++i) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, ctx->stage_ev[5 * c + i], ctx->stage_ev[5 * c + i + 1]) != cudaSuccess)
        return TZR_ERR_CUDA;
      acc[i] += ms;
    }
  // graph = the graph kernel launches alone (operand tiles + tensor-core kernel + strip kernel); the interleaved degree
  // launches are booked under "clique"
  double g = 0;
  for (int k = g0; k + 1 < g1; k += 2) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ctx->graph_ev[k], ctx->graph_ev[k + 1]) != cudaSuccess) return TZR_ERR_CUDA;
    g += ms;
  }
  if (g1 > g0) {
    acc[2] += acc[1] - g;
    acc[1] = g;
  }
  return TZR_OK;
}

int tzr_last_stage_ms(tzr_ctx* ctx, double* prep_ms, double* graph_ms, double* clique_ms, double* rot_trans_ms) {
  if (!ctx || !ctx->have_last) return TZR_ERR_INVALID_ARG;
  double acc[4];
  const int rc = sum_stage_events(ctx, ctx->stage_first, ctx->stage_chunks, ctx->graph_first, ctx->graph_ev_used, acc);
  if (rc) return rc;
  double* outs[4] = {prep_ms, graph_ms, clique_ms, rot_trans_ms};
  for (int i = 0; i < 4; ++i)
    if (outs[i]) *outs[i] = acc[i];
  return TZR_OK;
}

int tzr_ctx_stage_log(tzr_ctx* ctx, int enable) {
  if (!ctx) return TZR_ERR_INVALID_ARG;
  ctx->stage_log = enable != 0;
  ctx->stage_chunks = ctx->stage_first = 0;
  ctx->graph_ev_used = ctx->graph_first = 0;
  ctx->stage_log_calls = 0;
  return TZR_OK;
}

int tzr_ctx_stage_log_read(tzr_ctx* ctx, double* sums_ms4, int32_t* n_calls) {
  if (!ctx || !sums_ms4) return TZR_ERR_INVALID_ARG;
  cudaSetDevice(ctx->device);
  CK(cudaStreamSynchronize(ctx->stream));
  const int rc = sum_stage_events(ctx, 0, ctx->stage_chunks, 0, ctx->graph_ev_used, sums_ms4);
  if (rc) return rc;
  if (n_calls) *n_calls = ctx->stage_log_calls;
  ctx->stage_chunks = ctx->stage_first = 0;
  ctx->graph_ev_used = ctx->graph_first = 0;
  ctx->stage_log_calls = 0;
  return TZR_OK;
}

// ------------------------------------------------------------------------------------------------
// multi-GPU fan-out inside the library: one context + one host thread per device, contiguous shards balanced by
// sum n_b^2 (the graph stage dominates), no collective (SURVEY §8e).
// ------------------------------------------------------------------------------------------------
namespace {
struct DevicePool {
  std::mutex mu;
  std::map<int, tzr_ctx*> ctxs;
  ~DevicePool() {
    for (auto& kv : ctxs) tzr_ctx_destroy(kv.second);
  }
};
DevicePool& device_pool() {
  static DevicePool pool;
  return pool;
}
}  // namespace

int tzr_solve_batch_multi(const int32_t* devices, int n_devices, const tzr_params* params, int B, const int32_t* n,
                          const double* const* src, const double* const* dst, tzr_solution* solutions,
                          int32_t* cliques, int max_n) {
  if (!params || !n || !src || !dst || !solutions || B <= 0) return TZR_ERR_INVALID_ARG;
  std::vector<int> devs;
  if (!devices || n_devices <= 0) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) return TZR_ERR_NO_DEVICE;
    for (int d = 0; d < count; ++d) devs.push_back(d);
  } else {
    devs.assign(devices, devices + n_devices);
  }
  DevicePool& pool = device_pool();
  std::lock_guard<std::mutex> lock(pool.mu);
  for (int d : devs)
    if (!pool.ctxs.count(d)) {
      tzr_ctx* c = nullptr;
      const int rc = tzr_ctx_create(d, &c);
      if (rc) return rc;
      pool.ctxs[d] = c;
    }
  const int G = std::min<int>((int)devs.size(), B);
  // contiguous shards with balanced sum n^2
  std::vector<double> cum(B + 1, 0.0);
  for (int b = 0; b < B; ++b) cum[b + 1] = cum[b] + (double)n[b] * (double)n[b];
  std::vector<int> cut(G + 1, 0);
  cut[G] = B;
  for (int g = 1; g < G; ++g) {
    const double target = cum[B] * g / G;
    int b = cut[g - 1] + 1;  // at least one problem per shard
    while (b < B - (G - g) && cum[b] < target) ++b;
    cut[g] = b;
  }
  std::vector<int> rcs(G, TZR_OK);
  std::vector<std::thread> threads;
  for (int g = 0; g < G; ++g) {
    threads.emplace_back([&, g] {
      const int b0 = cut[g], Bg = cut[g + 1] - cut[g];
      if (Bg <= 0) return;
      rcs[g] = tzr_solve_batch(pool.ctxs[devs[g]], params, Bg, n + b0, src + b0, dst + b0, solutions + b0,
                               cliques ? cliques + (size_t)b0 * max_n : nullptr, max_n);
    });
  }
  for (auto& t : threads) t.join();
  for (int g = 0; g < G; ++g)
    if (rcs[g]) return rcs[g];
  return TZR_OK;
}

}  // extern "C"
