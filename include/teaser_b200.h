/*
 * teaser_b200.h — C-ABI of the B200-native TEASER++ registration hot path.
 *
 * This is the drop-in boundary: plain C, caller-owned buffers, no STL / Eigen / torch types.
 * The reference has no FFI layer of its own (SURVEY.md §8b); each entry point below names the
 * reference function(s) it replaces (paths relative to the reference tree).  The C++ facade
 * `teaser::RobustRegistrationSolver` (teaser-plusplus_b200/host/include/teaser/registration.h) and the
 * Python module `teaserpp_python` call exactly these symbols; INTEGRATION.md shows the binding a
 * TEASER++ maintainer would add.
 *
 * Conventions
 *   - Points are 3xN column-major double == N contiguous (x,y,z) triples, i.e. the memory of an
 *     Eigen::Matrix<double,3,Dynamic> (teaser/src/registration.cc:568-570).
 *   - 3x3 rotations are column-major (Eigen::Matrix3d).
 *   - The inlier graph is a packed, symmetric adjacency bitset: n rows of `tzr_words_per_row(n)`
 *     little-endian uint64 words; bit j of row i is set iff TIM (i,j) passed the scale test
 *     (replaces teaser::Graph's vector<vector<int>>, teaser/include/teaser/graph.h:29-207).
 *   - Every function returns 0 on success or a negative tzr_status; no exceptions cross the ABI.
 *   - "_dev" variants take DEVICE pointers and enqueue on the context's stream without
 *     synchronising (tzr_ctx_synchronize does); the plain variants take HOST pointers and are
 *     synchronous, host<->device copies included.
 *   - Problem size: every entry point that takes n accepts n <= 131072 correspondences (one problem's bitset is then
 *     2 GiB) and returns TZR_ERR_TOO_LARGE above.  For n <= 32768 the clique stage runs on the whole graph.  Above,
 *     it first finds a greedy clique of size L on the whole graph and peels the graph to its (L-1)-core, which holds
 *     every maximum clique; PMC_EXACT then searches that core, and TZR_ERR_TOO_LARGE is returned (tzr_last_error
 *     names the problem and the core size) when the core has more than 32768 vertices, as on dense (~15 %) inlier
 *     graphs, where PMC_HEU and KCORE_HEU still work.  The vertex set handed to the rotation stage (the clique or
 *     the innermost core) must have <= 32768 vertices; estimate_scaling and inlier selection NONE need n <= 32768.
 *     In a batch, one problem over a limit fails the whole call.
 *   - A context owns one CUDA device, one stream and a growable workspace; it is not thread-safe,
 *     distinct contexts are independent.  There is NO CPU fallback: without a usable CUDA device
 *     tzr_ctx_create fails with TZR_ERR_NO_DEVICE.
 */
#ifndef TEASER_B200_H_
#define TEASER_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TZR_ABI_VERSION 2

typedef enum tzr_status {
  TZR_OK = 0,
  TZR_ERR_INVALID_ARG = -1,
  TZR_ERR_NO_DEVICE = -2,
  TZR_ERR_CUDA = -3,
  TZR_ERR_ALLOC = -4,
  TZR_ERR_UNSUPPORTED = -5,
  TZR_ERR_TOO_LARGE = -6
} tzr_status;

/* teaser::RobustRegistrationSolver::Params (teaser/include/teaser/registration.h:419-514).
 * Enum values are the reference's (registration.h:382-412). */
typedef struct tzr_params {
  double noise_bound;                    /* default 0.01 */
  double cbar2;                          /* default 1 */
  int32_t estimate_scaling;              /* default 1 (true) */
  int32_t rotation_estimation_algorithm; /* 0 GNC_TLS (default), 1 FGR, 2 QUATRO */
  double rotation_gnc_factor;            /* default 1.4 */
  uint64_t rotation_max_iterations;      /* default 100 */
  double rotation_cost_threshold;        /* default 1e-6 */
  int32_t rotation_tim_graph;            /* 0 CHAIN (default), 1 COMPLETE */
  int32_t inlier_selection_mode;         /* 0 PMC_EXACT (default), 1 PMC_HEU, 2 KCORE_HEU, 3 NONE */
  double kcore_heuristic_threshold;      /* default 0.5 */
  int32_t use_max_clique;                /* deprecated, default 1 */
  int32_t max_clique_exact_solution;     /* deprecated, default 1 */
  double max_clique_time_limit;          /* seconds, default 3600 */
  int32_t max_clique_num_threads;        /* ignored on the GPU */
  int32_t reserved;
} tzr_params;

/* teaser::RegistrationSolution (registration.h:32-39) plus diagnostics the getters expose. */
typedef struct tzr_solution {
  int32_t valid;                  /* solution_.valid (registration.cc:643-647,734) */
  int32_t clique_size;            /* getInlierMaxClique().size() */
  double scale;
  double translation[3];
  double rotation[9];             /* column-major */
  int32_t clique_proven_optimal;  /* 1: maximum clique proven by complete enumeration (canonical = lexicographically
                                   * smallest among ties); 2: maximum SIZE proven through the vertex-cover LP bound /
                                   * Nemhauser-Trotter reduction after the first 50 ms search pass (dense graphs; a
                                   * maximum clique, not necessarily the canonical one); 0: heuristic mode or budget hit */
  int32_t gnc_iterations;         /* loop bodies entered by the GNC rotation solver */
  double gnc_cost;                /* getGNCRotationCostAtTermination() */
  int32_t n_rotation_inliers;
  int32_t n_translation_inliers;
  int64_t n_edges;                /* edges of the inlier graph */
  double stage_ms[8];             /* filled by tzr_solve only: 0 h2d, 1 graph, 2 clique, 3 rot+trans, 4 d2h, 6 total */
} tzr_solution;

typedef struct tzr_ctx tzr_ctx;

/* ---- context ------------------------------------------------------------------------------- */
int tzr_abi_version(void);
const char* tzr_status_string(int status);
/* Last CUDA error text seen by this context (empty string if none). */
const char* tzr_last_error(const tzr_ctx* ctx);
/* Fill `p` with the reference's Params defaults (registration.h:419-514). */
void tzr_params_default(tzr_params* p);
/* device < 0: current device.  Fails (TZR_ERR_NO_DEVICE) when no CUDA device is usable. */
int tzr_ctx_create(int device, tzr_ctx** out);
int tzr_ctx_destroy(tzr_ctx* ctx);
/* Use an existing CUDA stream (cudaStream_t as void*) instead of the context's own. */
int tzr_ctx_set_stream(tzr_ctx* ctx, void* cuda_stream);
int tzr_ctx_synchronize(tzr_ctx* ctx);
/* Number of kernels this context has launched so far (bench.py's gpu_launches). */
int64_t tzr_ctx_kernel_launches(const tzr_ctx* ctx);
/* 64-bit words per adjacency row: ceil(n/64). */
int tzr_words_per_row(int n);

/* ---- stage 1: TIMs + scale consistency + inlier graph ---------------------------------------
 * Replaces computeTIMs (registration.cc:512-551) x2, ScaleInliersSelector::solveForScale
 * (registration.cc:427-443) and the Graph::addEdge loop (registration.cc:614-619) — fused, the
 * N(N-1)/2 TIMs are never materialised.  beta = 2*noise_bound*sqrt(cbar2).
 * adj_bits: n * tzr_words_per_row(n) uint64 (fully overwritten); degree: n int32 (may be NULL). */
int tzr_graph_build(tzr_ctx* ctx, const double* src_3xN, const double* dst_3xN, int n, double beta,
                    uint64_t* adj_bits, int32_t* degree, int64_t* n_edges);

/* ---- stage 2: maximum clique ----------------------------------------------------------------
 * Replaces teaser::MaxCliqueSolver::findMaxClique (teaser/src/graph.cc:12-125) including the PMC
 * library calls it makes.  mode: 0 PMC_EXACT, 1 PMC_HEU, 2 KCORE_HEU.  clique: capacity n, returned
 * sorted ascending (solve() sorts it, registration.cc:636).  *proven_optimal: 1 / 2 / 0 with the meaning of
 * tzr_solution.clique_proven_optimal. */
int tzr_max_clique(tzr_ctx* ctx, const uint64_t* adj_bits, int n, int mode, double kcore_heuristic_threshold,
                   double time_limit_s, int32_t* clique, int32_t* clique_size, int32_t* proven_optimal);

/* ---- stage 3: GNC-TLS rotation --------------------------------------------------------------
 * Replaces GNCTLSRotationSolver::solveForRotation (registration.cc:764-866) + utils::svdRot
 * (teaser/include/teaser/utils.h:121-136).  inlier_mask (m bytes) and the scalar outputs may be NULL. */
int tzr_gnc_tls_rotation(tzr_ctx* ctx, const double* src_3xM, const double* dst_3xM, int m, double noise_bound,
                         double gnc_factor, uint64_t max_iterations, double cost_threshold, double* R_colmajor9,
                         uint8_t* inlier_mask, double* cost_at_termination, int32_t* iterations);

/* Same stage for any of the reference's rotation back-ends on caller-supplied TIMs: algorithm 0 GNC_TLS
 * (registration.cc:764-866), 1 FGR (FastGlobalRegistrationSolver::solveForRotation, registration.cc:206-278),
 * 2 QUATRO (QuatroSolver::solveForRotation, registration.cc:280-408; yaw only). */
int tzr_rotation_solve(tzr_ctx* ctx, int algorithm, const double* src_3xM, const double* dst_3xM, int m,
                       double noise_bound, double gnc_factor, uint64_t max_iterations, double cost_threshold,
                       double* R_colmajor9, uint8_t* inlier_mask, double* cost_at_termination, int32_t* iterations);

/* ---- stage 4: TLS translation ---------------------------------------------------------------
 * Replaces TLSTranslationSolver::solveForTranslation (registration.cc:445-471): per-axis
 * ScalarTLSEstimator::estimate on dst - src with range noise_bound*sqrt(cbar2). */
int tzr_tls_translation(tzr_ctx* ctx, const double* src_3xM, const double* dst_3xM, int m, double noise_bound,
                        double cbar2, double* t3, uint8_t* inlier_mask);

/* ScalarTLSEstimator::estimate (registration.cc:21-88), standalone. */
int tzr_scalar_tls(tzr_ctx* ctx, const double* x, const double* ranges, int64_t m, double* estimate,
                   uint8_t* inliers);

/* ---- upstream of solve(): correspondence generation ------------------------------------------
 * Replaces Matcher::calculateCorrespondences (teaser/src/matcher.cc:21-53 -> normalizePoints :55-113 and
 * advancedMatching :114-297).  Host pointers.  src_pts/dst_pts: ns x 3 / nd x 3 float xyz (PointXYZ AoS,
 * geometry.h:15-24); src_feat/dst_feat: row-major ns x dim / nd x dim float descriptors (FPFH: dim = 33,
 * pcl::FPFHSignature33::histogram), 1 <= dim <= 128.  The nearest-neighbour search is exact under
 * flann::L2<float> (what KDTreeSingleIndex with eps = 0 returns), lowest index among equal distances.
 * use_tuple_test + tuple_scale != 0 runs 100 * ncorr trials (:236); the reference seeds rand() with time(NULL),
 * here the draws are splitmix64(tuple_seed + 3 t + k) >> 33 so a seed reproduces a run.
 * pairs: capacity x 2 int32 rows (source index, target index), sorted and unique like the reference's output;
 * capacity >= ns + nd is always enough.  global_scale (optional) receives Matcher::global_scale_. */
int tzr_match_correspondences(tzr_ctx* ctx, const float* src_pts, int ns, const float* dst_pts, int nd,
                              const float* src_feat, const float* dst_feat, int dim, int use_absolute_scale,
                              int use_crosscheck, int use_tuple_test, float tuple_scale, uint64_t tuple_seed,
                              int32_t* pairs, int64_t capacity, int64_t* n_pairs, float* global_scale);

/* Descriptor estimation: replaces FPFHEstimation::computeFPFHFeatures (teaser/src/fpfh.cc:15-43), i.e. PCL's
 * NormalEstimationOMP (radius normal_search_radius, viewpoint at the origin) followed by FPFHEstimationOMP (radius
 * fpfh_search_radius) on the same cloud.  Host pointers.  pts: n x 3 float xyz.  fpfh_out: n x 33 floats
 * (pcl::FPFHSignature33::histogram rows).  normals_out (optional): n x 4 floats (normal_x, normal_y, normal_z,
 * curvature — FPFHEstimation::getNormals(), fpfh.h:55); NaN where a point has fewer than 3 neighbours.
 * TZR_ERR_TOO_LARGE when some point has more than 4096 neighbours inside a radius (downsample the cloud). */
int tzr_compute_fpfh(tzr_ctx* ctx, const float* pts, int n, double normal_search_radius, double fpfh_search_radius,
                     float* fpfh_out, float* normals_out);

/* The matcher's search primitive on its own (Matcher::searchKDTree with nn = 1, matcher.cc:314-335, for every
 * query row): nn_index[q] = argmin_i L2(query[q], db[i]), nn_dist[q] (optional) the squared distance. */
int tzr_feature_nn(tzr_ctx* ctx, const float* query, int nq, const float* db, int ndb, int dim, int32_t* nn_index,
                   float* nn_dist);

/* ---- downstream of solve(): certification ------------------------------------------------------
 * Replaces DRSCertifier::certify (teaser/src/certification.cc:40-190; Params certification.h:70-108).  Host pointers.
 * R: 3x3 column-major rotation estimate; src/dst: 3 x N column-major (the TIMs the rotation was estimated from);
 * theta: N doubles, +1 inlier / -1 outlier (the bool overload of the reference maps true -> +1, :22-38).
 * traj (optional, capacity traj_capacity): the sub-optimality gap of every iteration
 * (CertificationResult::suboptimality_traj).  eig_decomposition_solver is accepted for source compatibility; both
 * values use the device eigensolver. */
typedef struct tzr_certifier_params {
  double noise_bound;     /* 0.01 */
  double cbar2;           /* 1 */
  double sub_optimality;  /* 1e-3 */
  double max_iterations;  /* 2e2 (a double in the reference too) */
  double gamma_tau;       /* 1.999999 */
  int32_t eig_decomposition_solver; /* 0 EIGEN, 1 SPECTRA */
  int32_t reserved;
} tzr_certifier_params;

typedef struct tzr_certification_result {
  int32_t is_optimal;
  int32_t n_iterations;        /* length of the trajectory */
  double best_suboptimality;
} tzr_certification_result;

void tzr_certifier_params_default(tzr_certifier_params* p);

int tzr_certify(tzr_ctx* ctx, const tzr_certifier_params* params, const double* R_colmajor9, const double* src_3xN,
                const double* dst_3xN, const double* theta, int n, tzr_certification_result* result, double* traj,
                int traj_capacity);

/* Building blocks, exposed so that each can be checked against the reference's fixtures
 * (test/teaser/certification-test.cc:355-497):
 * tzr_certifier_initial_matrix: M_init = D^T Q_cost D - mu J - lambda_guess (certification.cc:60-100), dense
 *   (4n+4)^2 column-major, and mu (:92) — covers getQCost, getBlockDiagOmega/getOmega1, getLambdaGuess.
 * tzr_certifier_dual_projection: getOptimalDualProjection (:316-446) with getLinearProjection's inverse map (:531-655)
 *   applied in closed form; W and W_dual are dense (4n+4)^2 column-major, theta as in tzr_certify. */
int tzr_certifier_initial_matrix(tzr_ctx* ctx, const tzr_certifier_params* params, const double* R_colmajor9,
                                 const double* src_3xN, const double* dst_3xN, const double* theta, int n,
                                 double* M_init, double* mu);
int tzr_certifier_dual_projection(tzr_ctx* ctx, const double* W, const double* theta, int n, double* W_dual);

/* ---- whole path -----------------------------------------------------------------------------
 * Replaces RobustRegistrationSolver::solve(src, dst) (registration.cc:568-737) for one problem
 * (tzr_solve) or B independent problems (tzr_solve_batch).  All intermediates stay on the device.
 * clique: capacity n, sorted.  rot_inliers: one byte per rotation TIM — clique_size bytes for CHAIN (capacity n
 * is always enough), clique_size*(clique_size-1)/2 for COMPLETE (capacity n*(n-1)/2 is always enough).
 * trans_inliers: clique_size bytes (capacity n).  Optional outputs may be NULL. */
int tzr_solve(tzr_ctx* ctx, const tzr_params* params, const double* src_3xN, const double* dst_3xN, int n,
              tzr_solution* solution, int32_t* clique, uint8_t* rot_inliers, uint8_t* trans_inliers);

/* B problems, problem b has n[b] correspondences at src[b] / dst[b] (host pointers).
 * cliques: B*max_n int32, problem b's clique at cliques + b*max_n (may be NULL). */
int tzr_solve_batch(tzr_ctx* ctx, const tzr_params* params, int B, const int32_t* n, const double* const* src,
                    const double* const* dst, tzr_solution* solutions, int32_t* cliques, int max_n);

/* Device-resident batch of equally sized problems: src_dev/dst_dev hold B*n*3 doubles each
 * (problem-major), solutions_dev B tzr_solution, cliques_dev B*n int32 (may be NULL).  Asynchronous on
 * the context's stream; this is what bench.py's kernel-only timing and the multi-GPU shards drive.  Exception: for
 * n > 32768 the call synchronises the context's stream once, after the (L-1)-core peel, because the host needs the
 * largest core of the batch to size the clique search. */
int tzr_solve_batch_dev(tzr_ctx* ctx, const tzr_params* params, int B, int n, const double* src_dev,
                        const double* dst_dev, tzr_solution* solutions_dev, int32_t* cliques_dev);

/* Retrieve the adjacency bitset / degrees of problem b of the most recent solve on this context
 * (lazy materialisation of getInlierGraph(), registration.h:772; SURVEY a16). Host pointers. */
int tzr_last_graph(tzr_ctx* ctx, int b, uint64_t* adj_bits, int32_t* degree);
/* What tzr_last_graph would return: batch size and n of the retained solve (0, 0 if none), whether a graph was
 * built (0 after inlier selection NONE: the reference never populates the graph, registration.cc:607-650, and
 * tzr_last_graph then yields an empty adjacency), and a generation counter that changes with every call that
 * rebuilds or invalidates the retained graph — callers that share a context (the C++ facade's per-thread context)
 * compare it with the value they saw after their own solve before trusting tzr_last_graph. */
int tzr_last_graph_info(const tzr_ctx* ctx, int32_t* B, int32_t* n, int32_t* has_graph, uint64_t* generation);

/* Graph-stage timing of the most recent tzr_solve_batch_dev, in milliseconds, measured with CUDA
 * events on the context's stream (for the roofline line in bench.py). Requires a prior synchronize. */
int tzr_last_stage_ms(tzr_ctx* ctx, double* prep_ms, double* graph_ms, double* clique_ms, double* rot_trans_ms);
/* Stage-timing log: while enabled the context keeps the CUDA events of EVERY pipeline call instead of re-using
 * them, so a benchmark loop can run without a host synchronisation per step; tzr_ctx_stage_log_read synchronises
 * once, returns the sums {prep, graph, clique, rot+trans} in ms over all calls since the last read (or enable) and
 * their count, and clears the log. */
int tzr_ctx_stage_log(tzr_ctx* ctx, int enable);
int tzr_ctx_stage_log_read(tzr_ctx* ctx, double* sums_ms4, int32_t* n_calls);

/* ---- multi-GPU ------------------------------------------------------------------------------
 * tzr_solve_batch over several devices of one node from a single host call (SURVEY §8e: independent problems,
 * no exchange step, no collective): the library keeps one context per device, cuts the batch into contiguous
 * shards balanced by sum n_b^2 and drives each shard from its own host thread.  devices == NULL or n_devices <= 0:
 * every visible device.  Same argument meaning as tzr_solve_batch; thread-safe (calls are serialised). */
int tzr_solve_batch_multi(const int32_t* devices, int n_devices, const tzr_params* params, int B, const int32_t* n,
                          const double* const* src, const double* const* dst, tzr_solution* solutions,
                          int32_t* cliques, int max_n);

/* Debug/verification switches: bit 0 (1) = force the pure-FP64 graph predicate (no FP32 filter),
 * bit 1 (2) = verify the FP32 / tensor-core filter against FP64 for every pair and count mismatches,
 * bit 2 (4) = count exact re-checks and clique search nodes, bit 8 (256) = degrees by a separate pass,
 * bit 10 (1024) = build the graph with the tensor-core kernel (tcgen05 Gram norms; bit-identical, measured slower than
 * the default CUDA-core kernel on B200: DESIGN.md 3.1), bit 9 (512) overrides it, bit 11 (2048) = the one-MUFU
 * CUDA-core variant (graph_strip3_kernel; bit-identical, FMA-pipe bound, 8 % slower), bit 13 (8192) = exact clique
 * search without the singleton-class path of the colouring (A/B), bit 12 (4096) = without the block colour bound (only
 * present in builds with -DTZR_BLOCK_BOUND).  For n > 65535 bits 10 and 11 are ignored (both kernels' re-check queues
 * pack a column index in 16 bits): the default graph kernel runs and counter [7] reports 0. */
int tzr_ctx_set_flags(tzr_ctx* ctx, uint32_t flags);
int64_t tzr_ctx_filter_mismatches(tzr_ctx* ctx);
/* Number of pairs of the most recent graph build that needed the exact FP64 re-check. */
int64_t tzr_ctx_filter_rechecks(tzr_ctx* ctx);
/* Debug counters of the most recent call (flag bit 2 set): [0] filter mismatches, [1] filter re-checks, [2] clique
 * search nodes, [3] reduce rounds, [4] vertices scanned by reduce rounds, [5] colourings, [6] vertices coloured,
 * [7] problems whose graph was built by the tensor-core kernel, [8]-[10] clock cycles of the exact search in the root
 * colour bound / degree rules / colourings, [11] slowest root (ns << 16 | vertex), [12] summed root time (ns),
 * [13] roots above 1 ms, [14] roots closed by the block colour bound, [15] n > 32768, PMC_EXACT: the largest number of
 * vertices handed to the clique search after compaction to the (L-1)-core (0 on the n <= 32768 path). */
int tzr_ctx_debug_counters(tzr_ctx* ctx, int64_t* out16);

#ifdef __cplusplus
}
#endif
#endif /* TEASER_B200_H_ */
