"""ctypes binding of oracle/_ref/libplstvo_ref.so — the reference's OWN pose code (function bodies cut verbatim out of
/root/reference by oracle/make_ref.py and compiled against the stand-in headers of oracle/ref_shim/).

TEST INFRASTRUCTURE: it pins the oracle (tests/test_oracle_ref.py); the product never loads it.  Method names and
argument meaning mirror oracle.oracle.Oracle so a test can run the same inputs through both.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from stvo_pl_b200 import types as T

from . import make_ref


class Ref:
    def __init__(self):
        self.lib = L = C.CDLL(make_ref.build())
        dp, u8p = T.c_double_p, T.c_uint8_p
        L.ref_describe.restype = C.c_char_p
        for name in ("ref_inverse_se3", "ref_expmap_se3", "ref_logmap_se3", "ref_adjoint_se3", "ref_inv6", "ref_eig6_sym"):
            getattr(L, name).restype = None
            getattr(L, name).argtypes = [dp, dp]
        L.ref_unccomp_se3.restype = None
        L.ref_unccomp_se3.argtypes = [dp, dp, dp, dp]
        L.ref_is_finite.restype = C.c_int
        L.ref_is_finite.argtypes = [dp, C.c_int]
        L.ref_vector_mean_stdv_mad.restype = None
        L.ref_vector_mean_stdv_mad.argtypes = [dp, C.c_int, dp, dp]
        L.ref_vector_stdv_mad.restype = C.c_double
        L.ref_vector_stdv_mad.argtypes = [dp, C.c_int]
        L.ref_robust_weight_cauchy.restype = C.c_double
        L.ref_robust_weight_cauchy.argtypes = [C.c_double]
        L.ref_line_segment_overlap.restype = C.c_double
        L.ref_line_segment_overlap.argtypes = [dp, dp, dp, dp]
        L.ref_projection.restype = None
        L.ref_projection.argtypes = [C.POINTER(T.PlCamera), dp, dp]
        L.ref_back_projection.restype = None
        L.ref_back_projection.argtypes = [C.POINTER(T.PlCamera), C.c_double, C.c_double, C.c_double, dp]
        L.ref_qr6_solve.restype = C.c_int
        L.ref_qr6_solve.argtypes = [dp, dp, dp, dp]
        L.ref_optimize_functions.restype = None
        L.ref_optimize_functions.argtypes = [C.POINTER(T.PlCamera), C.POINTER(T.PlConfig), C.POINTER(T.PlMatchedBatch),
                                             C.c_int, dp, C.c_int, dp, dp, dp]
        L.ref_gauss_newton.restype = None
        L.ref_gauss_newton.argtypes = [C.POINTER(T.PlCamera), C.POINTER(T.PlConfig), C.POINTER(T.PlMatchedBatch), C.c_int,
                                       dp, C.c_int, C.c_int, dp, dp, dp]
        L.ref_remove_outliers.restype = C.c_int
        L.ref_remove_outliers.argtypes = [C.POINTER(T.PlCamera), C.POINTER(T.PlConfig), C.POINTER(T.PlMatchedBatch), C.c_int,
                                          dp, u8p, u8p, T.c_int32_p]
        L.ref_optimize_pose.restype = C.c_int
        L.ref_optimize_pose.argtypes = [C.POINTER(T.PlCamera), C.POINTER(T.PlConfig), C.POINTER(T.PlMatchedBatch),
                                        C.c_void_p, C.c_void_p, u8p, u8p]

    @staticmethod
    def _d(a):
        return np.ascontiguousarray(a, dtype=np.float64)

    @staticmethod
    def _dp(a):
        return a.ctypes.data_as(T.c_double_p)

    def describe(self) -> str:
        return self.lib.ref_describe().decode()

    def _unary(self, name, x, n_out):
        x = self._d(x).ravel()
        out = np.zeros(n_out)
        getattr(self.lib, name)(self._dp(x), self._dp(out))
        return out

    def inverse_se3(self, Tm):
        return self._unary("ref_inverse_se3", Tm, 16).reshape(4, 4)

    def expmap_se3(self, x):
        return self._unary("ref_expmap_se3", x, 16).reshape(4, 4)

    def logmap_se3(self, Tm):
        return self._unary("ref_logmap_se3", Tm, 6)

    def adjoint_se3(self, Tm):
        return self._unary("ref_adjoint_se3", Tm, 36).reshape(6, 6)

    def inv6(self, A):
        return self._unary("ref_inv6", A, 36).reshape(6, 6)

    def eig6_sym(self, A):
        return self._unary("ref_eig6_sym", A, 6)

    def unccomp_se3(self, T1, c1, cinc):
        T1, c1, cinc = self._d(T1).ravel(), self._d(c1).ravel(), self._d(cinc).ravel()
        out = np.zeros(36)
        self.lib.ref_unccomp_se3(self._dp(T1), self._dp(c1), self._dp(cinc), self._dp(out))
        return out.reshape(6, 6)

    def qr6_solve(self, H, g):
        H, g = self._d(H).ravel(), self._d(g).ravel()
        x, lad = np.zeros(6), np.zeros(1)
        rank = self.lib.ref_qr6_solve(self._dp(H), self._dp(g), self._dp(x), self._dp(lad))
        return x, float(lad[0]), rank

    def is_finite(self, x) -> bool:
        x = self._d(x).ravel()
        return bool(self.lib.ref_is_finite(self._dp(x), len(x)))

    def vector_mean_stdv_mad(self, res):
        res = self._d(res).ravel()
        m, s = np.zeros(1), np.zeros(1)
        self.lib.ref_vector_mean_stdv_mad(self._dp(res), len(res), self._dp(m), self._dp(s))
        return float(m[0]), float(s[0])

    def vector_stdv_mad(self, res) -> float:
        res = self._d(res).ravel()
        return float(self.lib.ref_vector_stdv_mad(self._dp(res), len(res)))

    def robust_weight_cauchy(self, r) -> float:
        return float(self.lib.ref_robust_weight_cauchy(float(r)))

    def line_segment_overlap(self, spl_obs, epl_obs, spl_proj, epl_proj) -> float:
        a, b, c, d = (self._d(v).ravel() for v in (spl_obs, epl_obs, spl_proj, epl_proj))
        return float(self.lib.ref_line_segment_overlap(self._dp(a), self._dp(b), self._dp(c), self._dp(d)))

    def projection(self, cam, P):
        P = self._d(P).ravel()
        uv = np.zeros(2)
        self.lib.ref_projection(C.byref(cam), self._dp(P), self._dp(uv))
        return uv

    def back_projection(self, cam, u, v, disp):
        P = np.zeros(3)
        self.lib.ref_back_projection(C.byref(cam), float(u), float(v), float(disp), self._dp(P))
        return P

    def optimize_functions(self, cam, cfg, matched: T.MatchedBatch, p, DT, robust=False):
        DT = self._d(DT).ravel()
        H, g, e = np.zeros(36), np.zeros(6), np.zeros(1)
        mc = matched.as_c()
        self.lib.ref_optimize_functions(C.byref(cam), C.byref(cfg), C.byref(mc), int(p), self._dp(DT), int(robust),
                                        self._dp(H), self._dp(g), self._dp(e))
        return H.reshape(6, 6), g, float(e[0])

    def gauss_newton(self, cam, cfg, matched: T.MatchedBatch, p, DT0, robust, max_iters):
        DT0 = self._d(DT0).ravel()
        DT, cov, e = np.zeros(16), np.zeros(36), np.zeros(1)
        mc = matched.as_c()
        self.lib.ref_gauss_newton(C.byref(cam), C.byref(cfg), C.byref(mc), int(p), self._dp(DT0), int(robust), int(max_iters),
                                  self._dp(DT), self._dp(cov), self._dp(e))
        return DT.reshape(4, 4), cov.reshape(6, 6), float(e[0])

    def remove_outliers(self, cam, cfg, matched: T.MatchedBatch, p, DT):
        DT = self._d(DT).ravel()
        n_pt = int(matched.pt_off[p + 1] - matched.pt_off[p])
        n_ls = int(matched.ls_off[p + 1] - matched.ls_off[p])
        ip, il, cnt = np.zeros(n_pt + 1, np.uint8), np.zeros(n_ls + 1, np.uint8), np.zeros(3, np.int32)
        mc = matched.as_c()
        rc = self.lib.ref_remove_outliers(C.byref(cam), C.byref(cfg), C.byref(mc), int(p), self._dp(DT),
                                          ip.ctypes.data_as(T.c_uint8_p), il.ctypes.data_as(T.c_uint8_p),
                                          cnt.ctypes.data_as(T.c_int32_p))
        return rc, ip[:n_pt], il[:n_ls], cnt

    def optimize_pose(self, cam, cfg, matched: T.MatchedBatch, priors=None):
        B = matched.B
        res = np.zeros(B, dtype=T.POSE_RESULT_DTYPE)
        inl_pt = np.zeros(int(matched.pt_off[-1]) + 1, np.uint8)
        inl_ls = np.zeros(int(matched.ls_off[-1]) + 1, np.uint8)
        mc = matched.as_c()
        rc = self.lib.ref_optimize_pose(C.byref(cam), C.byref(cfg), C.byref(mc),
                                        priors.ctypes.data if priors is not None else None, res.ctypes.data,
                                        inl_pt.ctypes.data_as(T.c_uint8_p), inl_ls.ctypes.data_as(T.c_uint8_p))
        return rc, res, inl_pt[:-1], inl_ls[:-1]
