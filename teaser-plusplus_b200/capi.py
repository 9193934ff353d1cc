"""ctypes binding of the C-ABI product library (csrc/libteaser_b200.so, include/teaser_b200.h).

There is no CPU fallback: every entry point raises if the library is missing or no CUDA device is
usable.  Points are (N,3) float64 C-contiguous numpy arrays (== the reference's column-major 3xN).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC_DIR = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(CSRC_DIR, "libteaser_b200.so")


class TzrError(RuntimeError):
    pass


class Params(C.Structure):
    """tzr_params == teaser::RobustRegistrationSolver::Params (registration.h:419-514)."""
    _fields_ = [
        ("noise_bound", C.c_double),
        ("cbar2", C.c_double),
        ("estimate_scaling", C.c_int32),
        ("rotation_estimation_algorithm", C.c_int32),
        ("rotation_gnc_factor", C.c_double),
        ("rotation_max_iterations", C.c_uint64),
        ("rotation_cost_threshold", C.c_double),
        ("rotation_tim_graph", C.c_int32),
        ("inlier_selection_mode", C.c_int32),
        ("kcore_heuristic_threshold", C.c_double),
        ("use_max_clique", C.c_int32),
        ("max_clique_exact_solution", C.c_int32),
        ("max_clique_time_limit", C.c_double),
        ("max_clique_num_threads", C.c_int32),
        ("reserved", C.c_int32),
    ]


class Solution(C.Structure):
    """tzr_solution == teaser::RegistrationSolution (registration.h:32-39) + diagnostics."""
    _fields_ = [
        ("valid", C.c_int32),
        ("clique_size", C.c_int32),
        ("scale", C.c_double),
        ("translation", C.c_double * 3),
        ("rotation", C.c_double * 9),
        ("clique_proven_optimal", C.c_int32),
        ("gnc_iterations", C.c_int32),
        ("gnc_cost", C.c_double),
        ("n_rotation_inliers", C.c_int32),
        ("n_translation_inliers", C.c_int32),
        ("n_edges", C.c_int64),
        ("stage_ms", C.c_double * 8),
    ]

    @property
    def R(self):
        return np.array(self.rotation[:]).reshape(3, 3).T.copy()

    @property
    def t(self):
        return np.array(self.translation[:])


SOLUTION_DTYPE = np.dtype([
    ("valid", np.int32), ("clique_size", np.int32), ("scale", np.float64), ("translation", np.float64, (3,)),
    ("rotation", np.float64, (9,)), ("clique_proven_optimal", np.int32), ("gnc_iterations", np.int32),
    ("gnc_cost", np.float64), ("n_rotation_inliers", np.int32), ("n_translation_inliers", np.int32),
    ("n_edges", np.int64), ("stage_ms", np.float64, (8,))], align=True)
assert SOLUTION_DTYPE.itemsize == C.sizeof(Solution), (SOLUTION_DTYPE.itemsize, C.sizeof(Solution))

_lib = None

class CertifierParams(C.Structure):
    """tzr_certifier_params == DRSCertifier::Params (certification.h:70-108)."""
    _fields_ = [("noise_bound", C.c_double), ("cbar2", C.c_double), ("sub_optimality", C.c_double),
                ("max_iterations", C.c_double), ("gamma_tau", C.c_double), ("eig_decomposition_solver", C.c_int32),
                ("reserved", C.c_int32)]


class CertificationResult(C.Structure):
    _fields_ = [("is_optimal", C.c_int32), ("n_iterations", C.c_int32), ("best_suboptimality", C.c_double)]


_SYMBOLS = [
    "tzr_abi_version", "tzr_status_string", "tzr_last_error", "tzr_params_default", "tzr_ctx_create",
    "tzr_ctx_destroy", "tzr_ctx_set_stream", "tzr_ctx_synchronize", "tzr_ctx_kernel_launches", "tzr_words_per_row",
    "tzr_graph_build", "tzr_max_clique", "tzr_gnc_tls_rotation", "tzr_rotation_solve", "tzr_tls_translation", "tzr_scalar_tls",
    "tzr_solve", "tzr_solve_batch", "tzr_solve_batch_dev", "tzr_last_graph", "tzr_last_stage_ms",
    "tzr_ctx_set_flags", "tzr_ctx_filter_mismatches", "tzr_ctx_filter_rechecks", "tzr_ctx_debug_counters",
    "tzr_match_correspondences", "tzr_feature_nn", "tzr_compute_fpfh", "tzr_certifier_params_default", "tzr_certify",
    "tzr_certifier_initial_matrix", "tzr_certifier_dual_projection", "tzr_last_graph_info", "tzr_ctx_stage_log",
    "tzr_ctx_stage_log_read", "tzr_solve_batch_multi",
]


def build(verbose: bool = False):
    """Compile csrc/*.cu for sm_100a with nvcc (cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC_DIR] + ([] if verbose else ["-s"])
    subprocess.check_call(cmd)


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TzrError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    dp, u8p, i32p, i64p, u64p = (C.POINTER(C.c_double), C.POINTER(C.c_uint8), C.POINTER(C.c_int32),
                                 C.POINTER(C.c_int64), C.POINTER(C.c_uint64))
    vp = C.c_void_p
    L.tzr_abi_version.restype = C.c_int
    L.tzr_status_string.restype = C.c_char_p
    L.tzr_status_string.argtypes = [C.c_int]
    L.tzr_last_error.restype = C.c_char_p
    L.tzr_last_error.argtypes = [vp]
    L.tzr_params_default.argtypes = [C.POINTER(Params)]
    L.tzr_params_default.restype = None
    L.tzr_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.tzr_ctx_destroy.argtypes = [vp]
    L.tzr_ctx_set_stream.argtypes = [vp, vp]
    L.tzr_ctx_synchronize.argtypes = [vp]
    L.tzr_ctx_kernel_launches.argtypes = [vp]
    L.tzr_ctx_kernel_launches.restype = C.c_int64
    L.tzr_words_per_row.argtypes = [C.c_int]
    L.tzr_graph_build.argtypes = [vp, dp, dp, C.c_int, C.c_double, u64p, i32p, i64p]
    L.tzr_max_clique.argtypes = [vp, u64p, C.c_int, C.c_int, C.c_double, C.c_double, i32p, i32p, i32p]
    L.tzr_gnc_tls_rotation.argtypes = [vp, dp, dp, C.c_int, C.c_double, C.c_double, C.c_uint64, C.c_double, dp, u8p,
                                       dp, i32p]
    L.tzr_rotation_solve.argtypes = [vp, C.c_int, dp, dp, C.c_int, C.c_double, C.c_double, C.c_uint64, C.c_double, dp,
                                     u8p, dp, i32p]
    L.tzr_tls_translation.argtypes = [vp, dp, dp, C.c_int, C.c_double, C.c_double, dp, u8p]
    L.tzr_scalar_tls.argtypes = [vp, dp, dp, C.c_int64, dp, u8p]
    L.tzr_solve.argtypes = [vp, C.POINTER(Params), dp, dp, C.c_int, C.POINTER(Solution), i32p, u8p, u8p]
    L.tzr_solve_batch.argtypes = [vp, C.POINTER(Params), C.c_int, i32p, C.POINTER(dp), C.POINTER(dp),
                                  C.POINTER(Solution), i32p, C.c_int]
    L.tzr_solve_batch_dev.argtypes = [vp, C.POINTER(Params), C.c_int, C.c_int, vp, vp, vp, vp]
    L.tzr_last_graph.argtypes = [vp, C.c_int, u64p, i32p]
    L.tzr_last_stage_ms.argtypes = [vp, dp, dp, dp, dp]
    L.tzr_last_graph_info.argtypes = [vp, i32p, i32p, i32p, u64p]
    L.tzr_ctx_stage_log.argtypes = [vp, C.c_int]
    L.tzr_ctx_stage_log_read.argtypes = [vp, dp, i32p]
    L.tzr_solve_batch_multi.argtypes = [i32p, C.c_int, C.POINTER(Params), C.c_int, i32p, C.POINTER(dp), C.POINTER(dp),
                                        C.POINTER(Solution), i32p, C.c_int]
    L.tzr_ctx_set_flags.argtypes = [vp, C.c_uint32]
    L.tzr_ctx_filter_mismatches.argtypes = [vp]
    L.tzr_ctx_filter_mismatches.restype = C.c_int64
    L.tzr_ctx_filter_rechecks.argtypes = [vp]
    L.tzr_ctx_filter_rechecks.restype = C.c_int64
    L.tzr_ctx_debug_counters.argtypes = [vp, i64p]
    fp = C.POINTER(C.c_float)
    L.tzr_match_correspondences.argtypes = [vp, fp, C.c_int, fp, C.c_int, fp, fp, C.c_int, C.c_int, C.c_int, C.c_int,
                                            C.c_float, C.c_uint64, i32p, C.c_int64, i64p, fp]
    L.tzr_feature_nn.argtypes = [vp, fp, C.c_int, fp, C.c_int, C.c_int, i32p, fp]
    L.tzr_compute_fpfh.argtypes = [vp, fp, C.c_int, C.c_double, C.c_double, fp, fp]
    L.tzr_certifier_params_default.argtypes = [C.POINTER(CertifierParams)]
    L.tzr_certifier_params_default.restype = None
    L.tzr_certify.argtypes = [vp, C.POINTER(CertifierParams), dp, dp, dp, dp, C.c_int, C.POINTER(CertificationResult),
                              dp, C.c_int]
    L.tzr_certifier_initial_matrix.argtypes = [vp, C.POINTER(CertifierParams), dp, dp, dp, dp, C.c_int, dp, dp]
    L.tzr_certifier_dual_projection.argtypes = [vp, dp, dp, C.c_int, dp]
    for s in _SYMBOLS:
        getattr(L, s)  # raises AttributeError if the header and the library disagree
    _lib = L
    return L


def default_params(**kw) -> Params:
    p = Params()
    lib().tzr_params_default(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def _pts(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if a.ndim != 2 or a.shape[1] != 3:
        raise ValueError("points must be (N,3)")
    return a


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


class Context:
    """One CUDA device + stream + workspace (tzr_ctx)."""

    def __init__(self, device: int = -1):
        self._h = C.c_void_p()
        rc = lib().tzr_ctx_create(device, C.byref(self._h))
        if rc != 0:
            raise TzrError(f"tzr_ctx_create failed: {lib().tzr_status_string(rc).decode()}")

    def close(self):
        if self._h:
            lib().tzr_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise TzrError(f"{lib().tzr_status_string(rc).decode()}: {lib().tzr_last_error(self._h).decode()}")

    # -- utilities
    def set_flags(self, flags: int):
        self._ck(lib().tzr_ctx_set_flags(self._h, flags))

    def filter_mismatches(self) -> int:
        return int(lib().tzr_ctx_filter_mismatches(self._h))

    def filter_rechecks(self) -> int:
        return int(lib().tzr_ctx_filter_rechecks(self._h))

    def debug_counters(self):
        out = np.zeros(16, dtype=np.int64)
        self._ck(lib().tzr_ctx_debug_counters(self._h, _p(out, C.c_int64)))
        return dict(filter_mismatches=int(out[0]), filter_rechecks=int(out[1]), clique_nodes=int(out[2]),
                    reduce_rounds=int(out[3]), reduce_vertices=int(out[4]), colourings=int(out[5]),
                    coloured_vertices=int(out[6]), tc_problems=int(out[7]),
                    # exact clique search, per-root timing (flag 4): cycles in the root colour bound / degree rules /
                    # colourings, slowest root (ns, vertex), summed root time, roots above 1 ms
                    root_colour_cycles=int(out[8]), reduce_cycles=int(out[9]), colour_cycles=int(out[10]),
                    slowest_root_ns=int(out[11]) >> 16, slowest_root_vertex=int(out[11]) & 0xffff,
                    root_ns_total=int(out[12]), roots_over_1ms=int(out[13]), block_bound_prunes=int(out[14]),
                    # n > 32768 (flag 4): largest compacted (L-1)-core handed to the exact clique search in the batch
                    clique_stage_vertices=int(out[15]))

    def kernel_launches(self) -> int:
        return int(lib().tzr_ctx_kernel_launches(self._h))

    def synchronize(self):
        self._ck(lib().tzr_ctx_synchronize(self._h))

    def set_stream(self, cuda_stream_ptr: int):
        self._ck(lib().tzr_ctx_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def last_stage_ms(self):
        v = [C.c_double() for _ in range(4)]
        self._ck(lib().tzr_last_stage_ms(self._h, C.byref(v[0]), C.byref(v[1]), C.byref(v[2]), C.byref(v[3])))
        return dict(prep=v[0].value, graph=v[1].value, clique=v[2].value, rot_trans=v[3].value)

    def stage_log(self, enable: bool):
        """Keep the stage events of every call (no host sync per step); read them with stage_log_read()."""
        self._ck(lib().tzr_ctx_stage_log(self._h, 1 if enable else 0))

    def stage_log_read(self):
        v = (C.c_double * 4)()
        calls = C.c_int32()
        self._ck(lib().tzr_ctx_stage_log_read(self._h, v, C.byref(calls)))
        return dict(prep=v[0], graph=v[1], clique=v[2], rot_trans=v[3]), int(calls.value)

    def last_graph_info(self):
        B, n, has, gen = C.c_int32(), C.c_int32(), C.c_int32(), C.c_uint64()
        self._ck(lib().tzr_last_graph_info(self._h, C.byref(B), C.byref(n), C.byref(has), C.byref(gen)))
        return dict(B=B.value, n=n.value, has_graph=bool(has.value), generation=int(gen.value))

    # -- stages
    def graph_build(self, src, dst, beta):
        s, d = _pts(src), _pts(dst)
        n = s.shape[0]
        W = lib().tzr_words_per_row(n)
        bits = np.zeros((n, W), dtype=np.uint64)
        deg = np.zeros(n, dtype=np.int32)
        ne = C.c_int64()
        self._ck(lib().tzr_graph_build(self._h, _p(s, C.c_double), _p(d, C.c_double), n, beta, _p(bits, C.c_uint64),
                                       _p(deg, C.c_int32), C.byref(ne)))
        return bits, deg, int(ne.value)

    def max_clique(self, bits, n, mode=0, kcore_thr=0.5, time_limit=3600.0):
        bits = np.ascontiguousarray(bits, dtype=np.uint64)
        out = np.zeros(n, dtype=np.int32)
        m = C.c_int32()
        proven = C.c_int32()
        self._ck(lib().tzr_max_clique(self._h, _p(bits, C.c_uint64), n, mode, kcore_thr, time_limit,
                                      _p(out, C.c_int32), C.byref(m), C.byref(proven)))
        return out[:m.value].copy(), bool(proven.value)

    def gnc_tls_rotation(self, src, dst, noise_bound, gnc_factor=1.4, max_iterations=100, cost_threshold=1e-6):
        return self.rotation_solve(0, src, dst, noise_bound, gnc_factor, max_iterations, cost_threshold)

    def rotation_solve(self, algorithm, src, dst, noise_bound, gnc_factor=1.4, max_iterations=100,
                       cost_threshold=1e-6):
        """algorithm: 0 GNC_TLS, 1 FGR, 2 QUATRO (ROTATION_ESTIMATION_ALGORITHM, registration.h:382-386)."""
        s, d = _pts(src), _pts(dst)
        m = s.shape[0]
        R = np.zeros(9)
        mask = np.zeros(m, dtype=np.uint8)
        cost = C.c_double()
        it = C.c_int32()
        self._ck(lib().tzr_rotation_solve(self._h, int(algorithm), _p(s, C.c_double), _p(d, C.c_double), m, noise_bound,
                                          gnc_factor, int(max_iterations), cost_threshold, _p(R, C.c_double),
                                          _p(mask, C.c_uint8), C.byref(cost), C.byref(it)))
        return dict(R=R.reshape(3, 3).T.copy(), inliers=mask.astype(bool), cost=cost.value, iterations=it.value)

    def tls_translation(self, src, dst, noise_bound, cbar2=1.0):
        s, d = _pts(src), _pts(dst)
        m = s.shape[0]
        t = np.zeros(3)
        mask = np.zeros(m, dtype=np.uint8)
        self._ck(lib().tzr_tls_translation(self._h, _p(s, C.c_double), _p(d, C.c_double), m, noise_bound, cbar2,
                                           _p(t, C.c_double), _p(mask, C.c_uint8)))
        return t, mask.astype(bool)

    def scalar_tls(self, x, ranges):
        x = np.ascontiguousarray(x, dtype=np.float64)
        r = np.ascontiguousarray(ranges, dtype=np.float64)
        est = C.c_double()
        inl = np.zeros(x.size, dtype=np.uint8)
        self._ck(lib().tzr_scalar_tls(self._h, _p(x, C.c_double), _p(r, C.c_double), x.size, C.byref(est),
                                      _p(inl, C.c_uint8)))
        return est.value, inl.astype(bool)

    # -- downstream of solve(): DRSCertifier (certification.cc)
    @staticmethod
    def _cert_inputs(R, src, dst, theta):
        Rc = np.ascontiguousarray(np.asarray(R, dtype=np.float64).T)      # column-major 3x3
        s = np.ascontiguousarray(np.asarray(src, dtype=np.float64).T)     # (3,N) -> N xyz triples == column-major 3xN
        d = np.ascontiguousarray(np.asarray(dst, dtype=np.float64).T)
        th = np.asarray(theta)
        th = np.where(th, 1.0, -1.0) if th.dtype == np.bool_ else th.astype(np.float64)
        th = np.ascontiguousarray(th.ravel())
        if s.shape[1] != 3 or d.shape != s.shape or th.size != s.shape[0]:
            raise TzrError("certify: src/dst must be (3,N) and theta (N,)")
        return Rc, s, d, th

    @staticmethod
    def certifier_params(**kw) -> "CertifierParams":
        p = CertifierParams()
        lib().tzr_certifier_params_default(C.byref(p))
        for k, v in kw.items():
            if not hasattr(p, k):
                raise AttributeError(k)
            setattr(p, k, v)
        return p

    def certify(self, R, src, dst, theta, **params):
        """DRSCertifier(params).certify(R, src, dst, theta) (certification.cc:22-190); src/dst are (3,N)."""
        p = self.certifier_params(**params)
        Rc, s, d, th = self._cert_inputs(R, src, dst, theta)
        cap = int(max(1, np.ceil(p.max_iterations)))
        traj = np.zeros(cap)
        res = CertificationResult()
        self._ck(lib().tzr_certify(self._h, C.byref(p), _p(Rc, C.c_double), _p(s, C.c_double), _p(d, C.c_double),
                                   _p(th, C.c_double), th.size, C.byref(res), _p(traj, C.c_double), cap))
        return dict(is_optimal=bool(res.is_optimal), best_suboptimality=res.best_suboptimality,
                    suboptimality_traj=traj[:res.n_iterations].copy())

    def certifier_initial_matrix(self, R, src, dst, theta, **params):
        p = self.certifier_params(**params)
        Rc, s, d, th = self._cert_inputs(R, src, dst, theta)
        n = 4 * th.size + 4
        M = np.zeros((n, n))
        mu = C.c_double()
        self._ck(lib().tzr_certifier_initial_matrix(self._h, C.byref(p), _p(Rc, C.c_double), _p(s, C.c_double),
                                                    _p(d, C.c_double), _p(th, C.c_double), th.size,
                                                    _p(M, C.c_double), C.byref(mu)))
        return M.T.copy(), mu.value      # column-major buffer -> numpy row-major view of the same matrix

    def certifier_dual_projection(self, W, theta):
        th = np.ascontiguousarray(np.asarray(theta, dtype=np.float64).ravel())
        Wc = np.ascontiguousarray(np.asarray(W, dtype=np.float64).T)
        n = 4 * th.size + 4
        if Wc.shape != (n, n):
            raise TzrError("certifier_dual_projection: W must be (4N+4, 4N+4)")
        out = np.zeros((n, n))
        self._ck(lib().tzr_certifier_dual_projection(self._h, _p(Wc, C.c_double), _p(th, C.c_double), th.size,
                                                     _p(out, C.c_double)))
        return out.T.copy()

    # -- upstream of solve(): Matcher::calculateCorrespondences (matcher.cc:21-337)
    def match_correspondences(self, src_pts, dst_pts, src_feat, dst_feat, use_absolute_scale=True,
                              use_crosscheck=True, use_tuple_test=True, tuple_scale=0.0, tuple_seed=0,
                              return_scale=False):
        """Same argument order and defaults as the reference method (matcher.h:39-43); points are (n,3) float32,
        features (n,dim) float32.  Returns an (m,2) int32 array of sorted unique (source, target) index pairs."""
        sp = np.ascontiguousarray(src_pts, dtype=np.float32)
        tp = np.ascontiguousarray(dst_pts, dtype=np.float32)
        sf = np.ascontiguousarray(src_feat, dtype=np.float32)
        tf = np.ascontiguousarray(dst_feat, dtype=np.float32)
        ns, nd = sp.shape[0], tp.shape[0]
        if sp.shape != (ns, 3) or tp.shape != (nd, 3) or sf.ndim != 2 or tf.ndim != 2 or sf.shape[0] != ns or \
                tf.shape[0] != nd or sf.shape[1] != tf.shape[1]:
            raise TzrError("match_correspondences: points must be (n,3) and features (n,dim) with one row per point")
        cap = ns + nd
        pairs = np.zeros((cap, 2), dtype=np.int32)
        cnt = C.c_int64()
        g = C.c_float()
        self._ck(lib().tzr_match_correspondences(
            self._h, _p(sp, C.c_float), ns, _p(tp, C.c_float), nd, _p(sf, C.c_float), _p(tf, C.c_float), sf.shape[1],
            int(bool(use_absolute_scale)), int(bool(use_crosscheck)), int(bool(use_tuple_test)), float(tuple_scale),
            int(tuple_seed), _p(pairs, C.c_int32), cap, C.byref(cnt), C.byref(g)))
        out = pairs[:cnt.value].copy()
        return (out, g.value) if return_scale else out

    def compute_fpfh(self, pts, normal_search_radius=0.03, fpfh_search_radius=0.05, return_normals=False):
        """FPFHEstimation::computeFPFHFeatures (fpfh.h:39-41, same defaults): (n,3) float32 -> (n,33) float32."""
        p = np.ascontiguousarray(pts, dtype=np.float32)
        if p.ndim != 2 or p.shape[1] != 3:
            raise TzrError("compute_fpfh: points must be (n,3)")
        out = np.zeros((p.shape[0], 33), dtype=np.float32)
        nor = np.zeros((p.shape[0], 4), dtype=np.float32)
        self._ck(lib().tzr_compute_fpfh(self._h, _p(p, C.c_float), p.shape[0], float(normal_search_radius),
                                        float(fpfh_search_radius), _p(out, C.c_float), _p(nor, C.c_float)))
        return (out, nor) if return_normals else out

    def feature_nn(self, query, db):
        """Exact 1-NN (flann::L2<float> accumulation order, lowest index among ties) of every query row in db."""
        q = np.ascontiguousarray(query, dtype=np.float32)
        d = np.ascontiguousarray(db, dtype=np.float32)
        if q.ndim != 2 or d.ndim != 2 or q.shape[1] != d.shape[1]:
            raise TzrError("feature_nn: query and db must be (n,dim) with equal dim")
        idx = np.zeros(q.shape[0], dtype=np.int32)
        dist = np.zeros(q.shape[0], dtype=np.float32)
        self._ck(lib().tzr_feature_nn(self._h, _p(q, C.c_float), q.shape[0], _p(d, C.c_float), d.shape[0], q.shape[1],
                                      _p(idx, C.c_int32), _p(dist, C.c_float)))
        return idx, dist

    # -- whole path
    def solve(self, src, dst, params: Params):
        s, d = _pts(src), _pts(dst)
        n = s.shape[0]
        sol = Solution()
        clique = np.zeros(n, dtype=np.int32)
        complete = params.rotation_tim_graph == 1
        rm = np.zeros(n * (n - 1) // 2 if complete else n, dtype=np.uint8)
        tm = np.zeros(n, dtype=np.uint8)
        self._ck(lib().tzr_solve(self._h, C.byref(params), _p(s, C.c_double), _p(d, C.c_double), n, C.byref(sol),
                                 _p(clique, C.c_int32), _p(rm, C.c_uint8), _p(tm, C.c_uint8)))
        m = sol.clique_size
        nrot = m * (m - 1) // 2 if complete else m
        return dict(sol=sol, valid=bool(sol.valid), scale=sol.scale, R=sol.R, t=sol.t, clique=clique[:m].copy(),
                    rot_inliers=rm[:nrot].astype(bool), trans_inliers=tm[:m].astype(bool),
                    gnc_iterations=sol.gnc_iterations, proven=bool(sol.clique_proven_optimal),
                    n_edges=int(sol.n_edges), stage_ms=list(sol.stage_ms))

    def solve_batch(self, srcs, dsts, params: Params):
        """srcs/dsts: lists of (N_b,3) arrays (host). Returns (solutions structured array, list of cliques)."""
        B = len(srcs)
        S = [_pts(a) for a in srcs]
        D = [_pts(a) for a in dsts]
        ns = np.array([a.shape[0] for a in S], dtype=np.int32)
        max_n = int(ns.max())
        dp = C.POINTER(C.c_double)
        sp = (dp * B)(*[_p(a, C.c_double) for a in S])
        dpp = (dp * B)(*[_p(a, C.c_double) for a in D])
        sols = np.zeros(B, dtype=SOLUTION_DTYPE)
        cl = np.zeros((B, max_n), dtype=np.int32)
        self._ck(lib().tzr_solve_batch(self._h, C.byref(params), B, _p(ns, C.c_int32), sp, dpp,
                                       sols.ctypes.data_as(C.POINTER(Solution)), _p(cl, C.c_int32), max_n))
        cliques = [cl[b, :max(0, int(sols[b]["clique_size"]))].copy() for b in range(B)]
        return sols, cliques

    def solve_batch_array(self, src, dst, params: Params, cliques_out=None, sols_out=None):
        """Batch of equally sized problems held in two (B, N, 3) float64 C-contiguous arrays (ideally page-locked,
        e.g. numpy views of torch pinned tensors: the library then DMAs straight from them and overlaps the copy
        of chunk k+1 with the kernels of chunk k).  No per-problem Python work.
        Returns (solutions structured array (B,), cliques (B, N) int32 padded, valid prefix = clique_size)."""
        src = np.asarray(src)
        dst = np.asarray(dst)
        if src.dtype != np.float64 or dst.dtype != np.float64 or src.ndim != 3 or src.shape != dst.shape or \
                src.shape[2] != 3 or not src.flags.c_contiguous or not dst.flags.c_contiguous:
            raise ValueError("src/dst must be C-contiguous float64 arrays of shape (B, N, 3)")
        B, n = src.shape[0], src.shape[1]
        stride = n * 3 * 8
        sp = (src.ctypes.data + np.arange(B, dtype=np.uint64) * np.uint64(stride)).astype(np.uint64)
        dp_ = (dst.ctypes.data + np.arange(B, dtype=np.uint64) * np.uint64(stride)).astype(np.uint64)
        ns = np.full(B, n, dtype=np.int32)
        sols = sols_out if sols_out is not None else np.zeros(B, dtype=SOLUTION_DTYPE)
        cl = cliques_out if cliques_out is not None else np.empty((B, n), dtype=np.int32)
        pp = C.POINTER(C.POINTER(C.c_double))
        self._ck(lib().tzr_solve_batch(self._h, C.byref(params), B, _p(ns, C.c_int32),
                                       C.cast(sp.ctypes.data, pp), C.cast(dp_.ctypes.data, pp),
                                       sols.ctypes.data_as(C.POINTER(Solution)), _p(cl, C.c_int32), n))
        return sols, cl

    def solve_batch_dev(self, params: Params, B: int, n: int, src_ptr: int, dst_ptr: int, sol_ptr: int,
                        clique_ptr: int = 0):
        """Device pointers (e.g. torch tensors' data_ptr()); asynchronous on the context's stream."""
        self._ck(lib().tzr_solve_batch_dev(self._h, C.byref(params), B, n, C.c_void_p(src_ptr), C.c_void_p(dst_ptr),
                                           C.c_void_p(sol_ptr), C.c_void_p(clique_ptr) if clique_ptr else None))

    def last_graph(self, b: int, n: int):
        W = lib().tzr_words_per_row(n)
        bits = np.zeros((n, W), dtype=np.uint64)
        deg = np.zeros(n, dtype=np.int32)
        self._ck(lib().tzr_last_graph(self._h, b, _p(bits, C.c_uint64), _p(deg, C.c_int32)))
        return bits, deg


def rotation_from_solution_record(rec) -> np.ndarray:
    return np.asarray(rec["rotation"]).reshape(3, 3).T.copy()


def solve_batch_multi(src_list, dst_list, params: Params, devices=None):
    """tzr_solve_batch_multi: one host call, the batch sharded over several GPUs inside the library (no torchrun).
    src_list/dst_list: sequences of (N_b,3) float64 arrays.  Returns (solutions structured array, list of cliques)."""
    B = len(src_list)
    srcs = [_pts(a) for a in src_list]
    dsts = [_pts(a) for a in dst_list]
    n = np.array([a.shape[0] for a in srcs], dtype=np.int32)
    max_n = int(n.max())
    sp = (C.POINTER(C.c_double) * B)(*[_p(a, C.c_double) for a in srcs])
    dp_ = (C.POINTER(C.c_double) * B)(*[_p(a, C.c_double) for a in dsts])
    sols = (Solution * B)()
    clq = np.zeros((B, max_n), dtype=np.int32)
    if devices is None:
        dev_p, n_dev = None, 0
    else:
        dev = np.ascontiguousarray(devices, dtype=np.int32)
        dev_p, n_dev = _p(dev, C.c_int32), int(dev.size)
    rc = lib().tzr_solve_batch_multi(dev_p, n_dev, C.byref(params), B, _p(n, C.c_int32), sp, dp_, sols,
                                     _p(clq, C.c_int32), max_n)
    if rc != 0:
        raise TzrError(f"tzr_solve_batch_multi: {lib().tzr_status_string(rc).decode()}")
    out = np.frombuffer(bytes(sols), dtype=SOLUTION_DTYPE).copy()
    return out, [clq[b, :out[b]["clique_size"]].copy() for b in range(B)]
