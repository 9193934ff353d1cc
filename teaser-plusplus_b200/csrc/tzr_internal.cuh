// Internal declarations shared by the CUDA translation units of libteaser_b200.so.
// Product code: nothing here (or in any file of this directory) includes or links oracle/.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>

#include "../../include/teaser_b200.h"

namespace tzr {

// ---- adjacency layout -------------------------------------------------------------------------
// Device-internal adjacency: n rows, pitch64(n) uint64 words per row.  The pitch is padded to whole
// 128-column tiles (2 words) so that every 128x128 tile of the graph kernel maps to one aligned
// 16-byte segment per row.  The ABI layout (ceil(n/64) words per row) is produced by a pitched copy.
__host__ __device__ inline int pitch64(int n) { return 2 * ((n + 127) / 128); }
__host__ __device__ inline int pitch32(int n) { return 2 * pitch64(n); }
__host__ __device__ inline int words64(int n) { return (n + 63) / 64; }
__host__ __device__ inline int npad128(int n) { return 128 * ((n + 127) / 128); }

constexpr int kTile = 128;          // graph tile edge (pairs per tile = 128*128)
constexpr int kGraphThreads = 128;  // 4 warps, each owns a 32x128 sub-tile (4 pairs per lane per step)
constexpr int kHeurRoots = 4;       // heuristic start vertices per problem (top degrees); a global-peeling
                                    // second chance in the peel kernel covers the cases they all miss
constexpr int kMatchMaxDim = 128;   // feature dimension limit of the matcher's NN kernel (FPFH: 33)
constexpr double kTcKappa = 12.0;   // bound on the tensor-core Gram error |a' - a| in units of 2^-24 * D^2 (D = largest distance
                                    // inside the cloud); measured with csrc/tc_probe (profiles/), x4 safety
constexpr int kMaxN = 32768;        // per-problem size limit of the shared-memory clique kernels
constexpr int kMaxNGraph = 131072;  // per-problem size limit of every entry point: above kMaxN the clique stage runs on
                                    // the compacted (L-1)-core (clique_large.cu); one problem's bitset is then 2 GiB
constexpr int kMaxNTc = 65535;      // the re-check queues of the tensor-core and v7 graph kernels pack i << 16 | j

// Per-problem constants of the FP32 filter (see graph_build.cu).
struct GraphConsts {
  float b1;       // x = ||ds| - |dd|| <= b1  : surely an edge      (beta - delta; -1 = never)
  float b2;       // x > b2                   : surely not an edge  (beta + delta; +inf = never)
  int use_fp64;   // 1: FP32 filter disabled for this problem (range/NaN guard or debug flag)
  int pad;
  double beta;    // 2*noise_bound*sqrt(cbar2)
  double cs[3], cd[3];  // centres subtracted before the float conversion
  float f3_nlo, f3_nhi;  // graph_strip3_kernel: -(beta^2 + K), -(beta^2 - K)   (K: undecided band relative to w)
  float f3_eps;          // bias of the squared norms (keeps w > 0)
  int pad2;
  double s_hat;   // scale applied to the centred source copies (1 unless estimate_scaling)
  // tensor-core filter (graph_tc.cu): d = (a-b)^2 - 2 beta^2 (a+b) + beta^4 from the Gram-form squared norms (no square root)
  int use_tc;     // 1: this problem goes through graph_tc_kernel, 0: through the CUDA-core strip kernel
  float tc_c2;    // 2 beta^2
  float tc_b4;    // beta^4
  float tc_kap, tc_c0;  // |d| <= kap (t^2 + beta^4) + c0 : undecided -> exact FP64 re-check   (t = a - b)
  float tc_pad;
};

// Everything the device kernels need to know about one batch (passed by value).
struct Batch {
  int B;          // problems
  double tc_kappa; // bound on the tensor-core Gram error in units of 2^-24 D^2 (kTcKappa; env TZR_TC_KAPPA for experiments)
  int tc_desc_swap; // debug (env TZR_TC_SWAP): exchange the leading/stride byte offsets of the MMA operand descriptors
  int tc_active;  // 1: problems with gc.use_tc are built by graph_tc_kernel and skipped by the CUDA-core strip kernel
  int scale_mode; // 1: estimate_scaling=true (TLSScaleSolver predicate, scale from sol[b].scale)
  int n;          // correspondences per problem (uniform inside a device batch)
  double beta;    // 2*noise_bound*sqrt(cbar2)  (registration.cc:438)
  const double* src;  // B*n*3
  const double* dst;  // B*n*3
  float4* sf;     // B*n centred float copies (w unused)
  float4* df;
  float* opnd;    // B * ceil(n/128) * 2 roles * 2 clouds * 6 planes * 128 rows * 4: tf32-split MMA operand tiles of the
                  // tensor-core graph kernel (graph_tc.cu), written by tc_prep_kernel
  uint2* tc_list;         // re-check queue of the tensor-core graph kernel: (problem, i << 16 | j)
  unsigned int* tc_list_count;  // 1 (may exceed the capacity: writers past it evaluate in place)
  unsigned int tc_list_cap;
  float* pk;      // B*6*npad128(n): the same centred floats, pair-interleaved per 128-column block for the packed
                  // FP32x2 graph kernel (arrays sx,sy,sz,dx,dy,dz; element of point j at blk*128 + k*64 + lane*2 + half)
  GraphConsts* gc;        // B
  uint64_t* adj;          // B*n*pitch64(n)
  int32_t* deg;           // B*n
  unsigned long long* n_edges2;  // B (sum of degrees = 2*edges)
  // clique state
  int32_t* hclq;          // B*kHeurRoots*n heuristic cliques
  int32_t* hsize;         // B*kHeurRoots
  int32_t* clq;           // B*n incumbent clique (unsorted)
  int32_t* L;             // B incumbent size
  uint32_t* alive;        // B*pitch32(n) bitset of vertices surviving the (L-1)-core peel
  uint32_t* best_bits;    // B*pitch32(n) incumbent clique as a bitset (canonical tie-break)
  int32_t* alive_cnt;     // B
  int32_t* root_ctr;      // B work counter for the exact phase
  int32_t* lock;          // B spin lock for incumbent updates
  int32_t* flags;         // B bit0: search incomplete (depth/time budget)
  int32_t* kcore_final;   // B (KCORE_HEU only, else nullptr): 1 = clq/L already final (max-core shortcut)
  // exact-phase scratch
  uint32_t* stack;        // per warp: max_depth * 2 * pitch32 words
  int32_t* cv;            // per warp: n ints (current clique)
  int32_t* centry;        // per warp: max_depth ints
  int max_depth;
  int exact_ctas;         // CTAs of the (persistent) exact-phase grid; scratch above is per warp of that grid
  int exact_conc;         // problems searched at a time (bitsets that fit the L2 together)
  // rotation / translation scratch (per problem)
  double* ps;             // B*3*n chain TIMs src
  double* pd;             // B*3*n chain TIMs dst (de-scaled)
  double* wgt;            // B*rot_cap GNC weights (one per rotation TIM)
  double* res;            // B*n scratch
  long long rot_cap;      // rotation TIMs per problem the workspace can hold (n for CHAIN)
  double* skey;           // B*3*sort_cap sort keys (per axis)
  int32_t* sidx;          // B*3*sort_cap sort payload
  int sort_cap;           // next_pow2(2n): per-axis capacity of skey/sidx
  int32_t* sorted_clq;    // B*n sorted clique (output order)
  uint8_t* rot_mask;      // B*rot_cap
  uint8_t* trans_mask;    // B*n
  tzr_solution* sol;      // B
  // debug
  unsigned long long* mismatches;  // 1
  unsigned long long* rechecks;    // 1
  uint32_t flags_dbg;
  unsigned long long budget_ns;    // time budget of the exact clique search per problem (0 = none), Params::max_clique_time_limit
  unsigned long long* t_start;     // B: %globaltimer when the first search warp of the problem started (0 = not yet)
};

// ||v_j - v_i|| exactly as the reference computes a TIM norm: IEEE double, no FMA contraction,
// src.array().square().colwise().sum() summed as (x^2 + y^2) + z^2   (registration.cc:415-418, :434-437)
__device__ __forceinline__ double tim_norm_exact(const double* __restrict__ p, int i, int j) {
  const double dx = __dsub_rn(p[3 * j + 0], p[3 * i + 0]);
  const double dy = __dsub_rn(p[3 * j + 1], p[3 * i + 1]);
  const double dz = __dsub_rn(p[3 * j + 2], p[3 * i + 2]);
  const double s = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
  return __dsqrt_rn(s);
}

// exact predicate: the reference's operation sequence in IEEE double, no contraction (registration.cc:427-443).
// Deliberately NOT inlined: it runs for ~1e-4 of the pairs; keeping its two DSQRT expansions out of the unrolled
// sweeps keeps the hot loops small enough for the instruction cache.
static __device__ __noinline__ bool edge_exact(const double* __restrict__ src, const double* __restrict__ dst, int i,
                                               int j, double beta) {
  const double d1 = tim_norm_exact(src, i, j);
  const double d2 = tim_norm_exact(dst, i, j);
  return fabs(__dsub_rn(d1, d2)) <= beta;  // (v1_dist - v2_dist).abs() <= beta   registration.cc:442
}

// Unknown-scale predicate (TLSScaleSolver, registration.cc:410-425 + :86): the pair is an inlier iff
// | d2/d1 - s_hat | <= beta * (1/d1), with s_hat the TLS scale estimate.
static __device__ __noinline__ bool edge_exact_scale(const double* __restrict__ src, const double* __restrict__ dst,
                                                     int i, int j, double beta, double s_hat) {
  const double d1 = tim_norm_exact(src, i, j);
  const double d2 = tim_norm_exact(dst, i, j);
  const double ratio = __ddiv_rn(d2, d1);
  const double alpha = __dmul_rn(beta, __ddiv_rn(1.0, d1));
  return fabs(__dsub_rn(ratio, s_hat)) <= alpha;
}

// Scratch of the clique front end of problems with n > kMaxN (clique_large.cu).  Per-problem arrays are indexed by
// the full n; bt.alive holds the survivors of the last peel.
struct LargeScratch {
  int32_t* hl;       // B*kHeurRoots*2n: member list | in-P degrees of each greedy heuristic
  int32_t* dcur;     // B*n: degree inside the surviving set while peeling
  uint32_t* dying;   // B*pitch32(n): vertices removed in the current peel round
  int32_t* k;        // B: peel threshold (a vertex with fewer than k surviving neighbours is removed); < 0: problem skipped
  int32_t* lo;       // B: core-number bisection (KCORE_HEU): the lo-core is non-empty ...
  int32_t* hi;       // B: ... and the hi-core is empty
  int32_t* surv;     // B*n: survivors of the last peel in ascending order
  int32_t* nsurv;    // B: survivors of the last peel
  unsigned int* total;  // 3: vertices removed so far in the running peel (its convergence test) | grid barrier (2)
};

// kernels (defined in the .cu files) -------------------------------------------------------------
void launch_prep(const Batch& bt, cudaStream_t st);
int launch_graph(const Batch& bt, cudaStream_t st, int num_sms);  // returns the number of kernels launched
// graph_tc.cu: tensor-core path (operand tiles + tcgen05 kernel) for the problems prep_kernel marked use_tc
int launch_graph_tc(const Batch& bt, cudaStream_t st, int num_sms);
size_t tc_operand_bytes(int B, int n);
size_t tc_list_entries(int B, int n);
void launch_graph_patch(const Batch& bt, cudaStream_t st, int num_sms);  // tc_patch_kernel over the re-check queue
// bitset_only: the adjacency did not come from launch_graph (tzr_max_clique on a caller's bitset): always popcount
void launch_degree(const Batch& bt, cudaStream_t st, bool bitset_only = false);
void launch_clique(const Batch& bt, const tzr_params& p, int mode, cudaStream_t st, int* n_launches);
int launch_scale_estimation(const Batch& bt, double* X, double* Rg, double* key, int32_t* idx, long long npad,
                            cudaStream_t st);
size_t scale_large_scratch_bytes(int n, size_t* cub_temp_bytes);
int launch_scale_estimation_large(const Batch& bt, double* X, double* Rg, void* scratch, cudaStream_t st);
void launch_rot_trans(const Batch& bt, const tzr_params& p, int use_clique, cudaStream_t st);
size_t clique_heur_smem(int n);
size_t clique_peel_smem(int n);
size_t clique_exact_smem(int n);
int clique_exact_grid(int n, int num_sms);  // CTAs of the persistent exact-phase grid on the current device
// clique_large.cu: front end of the clique stage for kMaxN < n <= kMaxNGraph
size_t large_scratch_bytes(int B, int n);
LargeScratch large_scratch_carve(void* base, int B, int n);
// Greedy heuristic on the full graph, then per mode: PMC_EXACT peels to the (L-1)-core and lists the survivors
// (ls.surv / ls.nsurv); PMC_HEU leaves the best greedy clique in L / clq; KCORE_HEU finds the max core by bisection and
// leaves the innermost core in L / clq when it exceeds the threshold (kcore_final), the greedy clique otherwise.
// Returns the number of kernels launched, -1 if a launch failed.
int launch_clique_large_front(const Batch& bt, const LargeScratch& ls, int mode, double kcore_thr, cudaStream_t st,
                              int num_sms);
// PMC_EXACT, after launch_clique_large_front: cb.adj = the sub-graph induced by the survivors (cb.n = the largest
// survivor count of the batch, shorter problems padded with isolated vertices) ...
void launch_clique_compact(const Batch& bt, const LargeScratch& ls, const Batch& cb, cudaStream_t st);
// ... and, after launch_clique on cb, its clique in the indices of the full problem (L, clq, flags of bt).
void launch_clique_map_back(const Batch& bt, const LargeScratch& ls, const Batch& cb, cudaStream_t st);

// stand-alone stage helpers used by the per-stage C-ABI entry points
void launch_gnc_only(int alg, const double* src, const double* dst, int m, double noise_bound, double gnc_factor,
                     unsigned long long max_iter, double cost_thr, double* wgt, double* res, double* out_R,
                     uint8_t* mask, double* out_cost, int* out_iters, cudaStream_t st);
void launch_translation_only(const double* src, const double* dst, int m, double beta, double* skey, int32_t* sidx,
                             double* out_t, uint8_t* mask, cudaStream_t st);
void launch_scalar_tls(const double* x, const double* ranges, long long m, double* skey, int32_t* sidx,
                       double* out_est, uint8_t* inliers, cudaStream_t st);

// fpfh.cu (FPFHEstimation::computeFPFHFeatures, fpfh.cc:15-43)
size_t fpfh_grid_scratch_bytes(int n);
int launch_fpfh(const float* pts, int n, double normal_radius, double fpfh_radius, float4* normals, float* spfh,
                float* out, int* overflow, void* grid_scratch, cudaStream_t st);

// certify.cu (DRSCertifier::certify, certification.cc:40-190); mode 0 certify, 1 initial matrix, 2 dual projection
int certify_device(int mode, double noise_bound, double cbar2, double sub_optimality, double max_iterations,
                   double gamma_tau, const double* R_cm, const double* src, const double* dst, const double* theta,
                   int N, int* is_optimal, double* best_subopt, int* n_iters, double* traj, int traj_cap,
                   double* M_init_out, double* mu_out, const double* W_in, double* Wd_out, void** scratch,
                   size_t* scratch_cap, void** solver_handle, int64_t* launches, cudaStream_t st, std::string* err);
void certify_release(void* solver_handle);

// matcher.cu (Matcher::calculateCorrespondences, matcher.cc:21-337)
int launch_feature_nn(const float* query, int nq, const float* db, int ndb, int dim, unsigned long long* best,
                      int num_sms, cudaStream_t st);
size_t match_scratch_bytes(int ns, int nd);
int launch_match(float* src_pts, int ns, float* dst_pts, int nd, const float* src_feat, const float* dst_feat, int dim,
                 int use_absolute_scale, int use_crosscheck, int use_tuple_test, float tuple_scale, uint64_t seed,
                 void* scratch, int32_t* pairs, int* count, float* gscale, int num_sms, cudaStream_t st);


}  // namespace tzr
