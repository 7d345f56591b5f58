"""ctypes binding of the CPU oracle (oracle/plstvo_oracle.c).

TEST INFRASTRUCTURE: only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs import this module.  The product package (stvo_pl_b200) never does.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from stvo_pl_b200 import types as T

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = [os.path.join(_HERE, "plstvo_oracle.c"), os.path.join(_HERE, "plstvo_oracle.h"),
        os.path.join(_HERE, "..", "include", "plstvo.h")]


def _build(out: str, march: str) -> None:
    """Same flags as oracle/Makefile (= the reference's CMakeLists.txt:18 flags)."""
    os.makedirs(os.path.dirname(out), exist_ok=True)
    tmp = f"{out}.{os.getpid()}.tmp"      # renamed into place: a concurrent loader never sees a half-written library
    cmd = ["gcc", "-O3", f"-march={march}", f"-mtune={'native' if march == 'native' else 'generic'}",
           "-std=gnu11", "-fPIC", "-ffp-contract=off", "-shared", "-o", tmp, _SRC[0], "-lm", "-lpthread"]
    subprocess.run(cmd, check=True, capture_output=True)
    os.replace(tmp, out)


def _stale(lib: str) -> bool:
    return (not os.path.exists(lib)) or any(os.path.getmtime(s) > os.path.getmtime(lib) for s in _SRC)


def lib_path(native: bool = False) -> str:
    """Portable build (x86-64-v3: AVX2 + POPCNT) travels with the repo; the native build used for the CPU
    baseline is compiled on the machine that times it (-march=native, the reference's own flag).  That one goes to the
    system's temporary directory, keyed by the sources and the CPU's flags, so that the benchmark runs from a read-only
    tree."""
    override = os.environ.get("PLSTVO_ORACLE_LIB")   # e.g. an -fsanitize=address,undefined build (tools/oracle_asan.sh)
    if override:
        return override
    if not native:
        lib = os.path.join(_HERE, "libplstvo_oracle.so")
        if _stale(lib):
            _build(lib, "x86-64-v3")
        return lib
    try:
        with open("/proc/cpuinfo") as f:
            flags = next((l for l in f if l.startswith("flags")), "")
    except OSError:
        flags = ""
    key = hashlib.sha1(flags.encode())
    for s in _SRC:
        with open(s, "rb") as f:
            key.update(f.read())
    lib = os.path.join(tempfile.gettempdir(), f"plstvo_oracle_native_{os.getuid()}", key.hexdigest()[:16], "libplstvo_oracle.so")
    if not os.path.exists(lib):
        _build(lib, "native")
    return lib


class OrcHandlerConfig(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("adaptative_fast", "fast_min_th", "fast_max_th", "fast_inc_th", "fast_feat_th",
                                         "orb_fast_th")] + [("fast_err_th", C.c_float), ("min_entropy_ratio", C.c_double),
                                                            ("max_kf_t_dist", C.c_double), ("max_kf_r_dist", C.c_double)]


class OrcKfState(C.Structure):
    _fields_ = [("prev_f_iskf", C.c_int32), ("N_prevKF_currF", C.c_int32), ("entropy_first_prevKF", C.c_double),
                ("T_prevKF", C.c_double * 16), ("cov_prevKF_currF", C.c_double * 36), ("entropy_curr", C.c_double),
                ("entropy_ratio", C.c_double), ("t", C.c_double), ("r", C.c_double)]


class Oracle:
    def __init__(self, native: bool = False):
        self.lib = L = C.CDLL(lib_path(native))
        u8p, i32p, dp = T.c_uint8_p, T.c_int32_p, T.c_double_p
        L.orc_distance.restype = C.c_int
        L.orc_distance.argtypes = [u8p, u8p]
        L.orc_match_nnr.restype = C.c_int
        L.orc_match_nnr.argtypes = [u8p, C.c_int, u8p, C.c_int, C.c_float, i32p]
        L.orc_match.restype = C.c_int
        L.orc_match.argtypes = [u8p, C.c_int, u8p, C.c_int, C.c_float, C.c_int, C.c_int, i32p]
        L.orc_knn2.restype = None
        L.orc_knn2.argtypes = [u8p, C.c_int, u8p, C.c_int, i32p, i32p]
        L.orc_match_grid_points.restype = C.c_int
        L.orc_match_grid_points.argtypes = [C.c_int, C.c_int, T.PlGridWindow, C.c_int, C.c_double, i32p, u8p, C.c_int,
                                            i32p, u8p, C.c_int, i32p]
        L.orc_match_grid_lines.restype = C.c_int
        L.orc_match_grid_lines.argtypes = [C.c_int, C.c_int, T.PlGridWindow, C.c_int, C.c_double, C.c_double, i32p, u8p,
                                           C.c_int, dp, dp, u8p, C.c_int, i32p]
        fp, scp = T.c_float_p, C.POINTER(T.PlStereoConfig)
        L.orc_stereo_lift_points.restype = C.c_int
        L.orc_stereo_lift_points.argtypes = [C.POINTER(T.PlCamera), scp, C.c_int, fp, i32p, u8p, fp, i32p, dp, dp, dp, dp, i32p,
                                             u8p, i32p]
        L.orc_stereo_lift_lines.restype = C.c_int
        L.orc_stereo_lift_lines.argtypes = [C.POINTER(T.PlCamera), scp, C.c_int, fp, fp, i32p, u8p, fp, i32p, dp, dp, dp, dp,
                                            dp, dp, dp, dp, dp, i32p, u8p, i32p]
        mcp = C.POINTER(T.PlStereoMatchConfig)
        L.orc_match_stereo_points.restype = C.c_int
        L.orc_match_stereo_points.argtypes = [C.POINTER(T.PlCamera), mcp, scp, C.c_int, fp, i32p, u8p, C.c_int, fp, u8p, i32p, dp, dp,
                                              dp, dp, i32p, u8p, i32p]
        L.orc_match_stereo_lines.restype = C.c_int
        L.orc_match_stereo_lines.argtypes = [C.POINTER(T.PlCamera), mcp, scp, C.c_int, fp, fp, i32p, u8p, C.c_int, fp, u8p, i32p, dp,
                                             dp, dp, dp, dp, dp, dp, dp, dp, i32p, u8p, i32p]
        L.orc_stereo_batch.restype = C.c_int
        L.orc_stereo_batch.argtypes = [C.POINTER(T.PlCamera), mcp, scp, C.c_int, i32p, fp, i32p, u8p, i32p, fp, u8p, i32p, fp, fp, i32p,
                                       u8p, i32p, fp, u8p, C.c_int, i32p]
        L.orc_line_segment_overlap_stereo.restype = C.c_double
        L.orc_line_segment_overlap_stereo.argtypes = [scp, C.c_double, C.c_double, C.c_double, C.c_double]
        L.orc_handler_default_config.restype = None
        L.orc_handler_default_config.argtypes = [C.POINTER(OrcHandlerConfig)]
        L.orc_update_fast_threshold.restype = C.c_int
        L.orc_update_fast_threshold.argtypes = [C.POINTER(OrcHandlerConfig), C.c_int, dp, C.c_double, C.c_int]
        L.orc_kf_reset.restype = None
        L.orc_kf_reset.argtypes = [C.POINTER(OrcKfState)]
        L.orc_det6.restype = C.c_double
        L.orc_det6.argtypes = [dp]
        L.orc_unctinv_se3.restype = None
        L.orc_unctinv_se3.argtypes = [dp, dp, dp]
        L.orc_need_new_kf.restype = C.c_int
        L.orc_need_new_kf.argtypes = [C.POINTER(OrcHandlerConfig), C.POINTER(OrcKfState), dp, dp, dp]
        L.orc_line_cells.restype = C.c_int
        L.orc_line_cells.argtypes = [C.c_double, C.c_double, C.c_double, C.c_double, i32p, C.c_int]
        for name, n_in, n_out in [("orc_inverse_se3", 16, 16), ("orc_expmap_se3", 6, 16),
                                  ("orc_logmap_se3", 16, 6), ("orc_adjoint_se3", 16, 36),
                                  ("orc_inv6", 36, 36), ("orc_eig6_sym", 36, 6)]:
            getattr(L, name).restype = None
            getattr(L, name).argtypes = [dp, dp]
        L.orc_unccomp_se3.restype = None
        L.orc_unccomp_se3.argtypes = [dp, dp, dp, dp]
        L.orc_is_finite.restype = C.c_int
        L.orc_is_finite.argtypes = [dp, C.c_int]
        L.orc_vector_mean_stdv_mad.restype = None
        L.orc_vector_mean_stdv_mad.argtypes = [dp, C.c_int, dp, dp]
        L.orc_vector_stdv_mad.restype = C.c_double
        L.orc_vector_stdv_mad.argtypes = [dp, C.c_int]
        L.orc_robust_weight_cauchy.restype = C.c_double
        L.orc_robust_weight_cauchy.argtypes = [C.c_double]
        L.orc_line_segment_overlap.restype = C.c_double
        L.orc_line_segment_overlap.argtypes = [dp, dp, dp, dp]
        L.orc_projection.restype = None
        L.orc_projection.argtypes = [C.POINTER(T.PlCamera), dp, dp]
        L.orc_back_projection.restype = None
        L.orc_back_projection.argtypes = [C.POINTER(T.PlCamera), C.c_double, C.c_double, C.c_double, dp]
        L.orc_qr6_solve.restype = C.c_int
        L.orc_qr6_solve.argtypes = [dp, dp, dp, dp]
        L.orc_optimize_functions.restype = None
        L.orc_optimize_functions.argtypes = [C.POINTER(T.PlCamera), C.POINTER(T.PlConfig),
                                             C.POINTER(T.PlMatchedBatch), C.c_int, dp, C.c_int, dp, dp, dp]
        L.orc_optimize_pose.restype = C.c_int
        L.orc_optimize_pose.argtypes = [C.POINTER(T.PlCamera), C.POINTER(T.PlConfig),
                                        C.POINTER(T.PlMatchedBatch), C.c_void_p, C.c_void_p, u8p, u8p]
        L.orc_f2f_tracking.restype = C.c_int
        L.orc_f2f_tracking.argtypes = [C.POINTER(T.PlConfig), C.POINTER(T.PlFrameBatch),
                                       C.POINTER(T.PlFrameBatch), i32p, i32p, i32p]
        L.orc_track_batch.restype = C.c_int
        L.orc_track_batch.argtypes = [C.POINTER(T.PlCamera), C.POINTER(T.PlConfig), C.POINTER(T.PlFrameBatch),
                                      C.POINTER(T.PlFrameBatch), C.c_void_p, C.c_void_p, i32p, i32p, u8p, u8p,
                                      C.c_int, C.c_int, dp]

    # ---- helpers ----
    @staticmethod
    def _d(a):
        return np.ascontiguousarray(a, dtype=np.float64)

    @staticmethod
    def _dp(a):
        return a.ctypes.data_as(T.c_double_p)

    def _unary(self, name, x, n_out):
        x = self._d(x).ravel()
        out = np.zeros(n_out)
        getattr(self.lib, name)(self._dp(x), self._dp(out))
        return out

    # ---- matching ----
    def distance(self, a, b) -> int:
        a, b = np.ascontiguousarray(a, np.uint8), np.ascontiguousarray(b, np.uint8)
        return self.lib.orc_distance(a.ctypes.data_as(T.c_uint8_p), b.ctypes.data_as(T.c_uint8_p))

    def knn2(self, d1, d2):
        d1, d2 = np.ascontiguousarray(d1, np.uint8), np.ascontiguousarray(d2, np.uint8)
        idx = np.full((len(d1), 2), -1, np.int32)
        dist = np.full((len(d1), 2), -1, np.int32)
        self.lib.orc_knn2(d1.ctypes.data_as(T.c_uint8_p), len(d1), d2.ctypes.data_as(T.c_uint8_p), len(d2),
                          idx.ctypes.data_as(T.c_int32_p), dist.ctypes.data_as(T.c_int32_p))
        return idx, dist

    def match_nnr(self, d1, d2, nnr):
        d1, d2 = np.ascontiguousarray(d1, np.uint8), np.ascontiguousarray(d2, np.uint8)
        m12 = np.full(len(d1), -1, np.int32)
        n = self.lib.orc_match_nnr(d1.ctypes.data_as(T.c_uint8_p), len(d1), d2.ctypes.data_as(T.c_uint8_p),
                                   len(d2), C.c_float(nnr), m12.ctypes.data_as(T.c_int32_p))
        return n, m12

    def match(self, d1, d2, nnr, best_lr=True, threads=False):
        d1, d2 = np.ascontiguousarray(d1, np.uint8), np.ascontiguousarray(d2, np.uint8)
        m12 = np.full(len(d1), -1, np.int32)
        n = self.lib.orc_match(d1.ctypes.data_as(T.c_uint8_p), len(d1), d2.ctypes.data_as(T.c_uint8_p), len(d2),
                               C.c_float(nnr), int(best_lr), int(threads), m12.ctypes.data_as(T.c_int32_p))
        return n, m12

    def match_grid_points(self, q_cell, d1, t_cell, d2, window, ratio, best_lr=True, rows=T.GRID_ROWS, cols=T.GRID_COLS):
        q_cell, t_cell = np.ascontiguousarray(q_cell, np.int32), np.ascontiguousarray(t_cell, np.int32)
        d1, d2 = np.ascontiguousarray(d1, np.uint8), np.ascontiguousarray(d2, np.uint8)
        m12 = np.full(len(d1), -1, np.int32)
        n = self.lib.orc_match_grid_points(rows, cols, window, int(best_lr), float(ratio), q_cell.ctypes.data_as(T.c_int32_p),
                                           d1.ctypes.data_as(T.c_uint8_p), len(d1), t_cell.ctypes.data_as(T.c_int32_p),
                                           d2.ctypes.data_as(T.c_uint8_p), len(d2), m12.ctypes.data_as(T.c_int32_p))
        return n, m12

    def match_grid_lines(self, q_line, d1, t_line, t_dir, d2, window, ratio, line_sim_th, best_lr=True,
                         rows=T.GRID_ROWS, cols=T.GRID_COLS):
        q_line = np.ascontiguousarray(q_line, np.int32)
        t_line, t_dir = np.ascontiguousarray(t_line, np.float64), np.ascontiguousarray(t_dir, np.float64)
        d1, d2 = np.ascontiguousarray(d1, np.uint8), np.ascontiguousarray(d2, np.uint8)
        m12 = np.full(len(d1), -1, np.int32)
        n = self.lib.orc_match_grid_lines(rows, cols, window, int(best_lr), float(ratio), float(line_sim_th),
                                          q_line.ctypes.data_as(T.c_int32_p), d1.ctypes.data_as(T.c_uint8_p), len(d1),
                                          self._dp(t_line), self._dp(t_dir), d2.ctypes.data_as(T.c_uint8_p), len(d2),
                                          m12.ctypes.data_as(T.c_int32_p))
        return n, m12

    # ---- host-side state machine (adaptive FAST threshold, key-frame test) ----
    def handler_default_config(self):
        c = OrcHandlerConfig()
        self.lib.orc_handler_default_config(C.byref(c))
        return c

    def update_fast_threshold(self, c, th, DT, err_norm, n_inliers_pt):
        DT = np.ascontiguousarray(DT, np.float64)
        return self.lib.orc_update_fast_threshold(C.byref(c), int(th), self._dp(DT), float(err_norm), int(n_inliers_pt))

    def kf_state(self):
        s = OrcKfState()
        self.lib.orc_kf_reset(C.byref(s))
        return s

    def need_new_kf(self, c, state, Tfw, DT, DT_cov):
        Tfw, DT, DT_cov = (np.ascontiguousarray(a, np.float64) for a in (Tfw, DT, DT_cov))
        return bool(self.lib.orc_need_new_kf(C.byref(c), C.byref(state), self._dp(Tfw), self._dp(DT), self._dp(DT_cov)))

    def det6(self, A):
        return self.lib.orc_det6(self._dp(np.ascontiguousarray(A, np.float64)))

    def unctinv_se3(self, T, cov):
        out = np.zeros((6, 6))
        self.lib.orc_unctinv_se3(self._dp(np.ascontiguousarray(T, np.float64)), self._dp(np.ascontiguousarray(cov, np.float64)),
                                 self._dp(out))
        return out

    # ---- 3-D lifting of the stereo matches (one frame) ----
    def stereo_lift_points(self, cam, scfg, kp_l, octave_l, desc_l, kp_r, m12):
        kp_l, kp_r = np.ascontiguousarray(kp_l, np.float32).reshape(-1, 2), np.ascontiguousarray(kp_r, np.float32).reshape(-1, 2)
        octave_l, m12 = np.ascontiguousarray(octave_l, np.int32), np.ascontiguousarray(m12, np.int32)
        desc_l = np.ascontiguousarray(desc_l, np.uint8).reshape(-1, 32)
        n = len(kp_l)
        out = dict(pl=np.zeros((n, 2)), disp=np.zeros(n), P=np.zeros((n, 3)), sigma2=np.zeros(n), level=np.zeros(n, np.int32),
                   desc=np.zeros((n, 32), np.uint8), src_idx=np.full(n, -1, np.int32))
        i32, u8, f32 = T.c_int32_p, T.c_uint8_p, T.c_float_p
        k = self.lib.orc_stereo_lift_points(
            C.byref(cam), C.byref(scfg), n, kp_l.ctypes.data_as(f32), octave_l.ctypes.data_as(i32), desc_l.ctypes.data_as(u8),
            kp_r.ctypes.data_as(f32), m12.ctypes.data_as(i32), self._dp(out["pl"]), self._dp(out["disp"]), self._dp(out["P"]),
            self._dp(out["sigma2"]), out["level"].ctypes.data_as(i32), out["desc"].ctypes.data_as(u8),
            out["src_idx"].ctypes.data_as(i32))
        return k, {key: v[:k] for key, v in out.items()}

    def stereo_lift_lines(self, cam, scfg, seg_l, angle_l, octave_l, desc_l, seg_r, m12):
        seg_l, seg_r = np.ascontiguousarray(seg_l, np.float32).reshape(-1, 4), np.ascontiguousarray(seg_r, np.float32).reshape(-1, 4)
        angle_l = np.ascontiguousarray(angle_l, np.float32)
        octave_l, m12 = np.ascontiguousarray(octave_l, np.int32), np.ascontiguousarray(m12, np.int32)
        desc_l = np.ascontiguousarray(desc_l, np.uint8).reshape(-1, 32)
        n = len(seg_l)
        out = dict(spl=np.zeros((n, 2)), epl=np.zeros((n, 2)), sdisp=np.zeros(n), edisp=np.zeros(n), sP=np.zeros((n, 3)),
                   eP=np.zeros((n, 3)), le=np.zeros((n, 3)), angle=np.zeros(n), sigma2=np.zeros(n),
                   level=np.zeros(n, np.int32), desc=np.zeros((n, 32), np.uint8), src_idx=np.full(n, -1, np.int32))
        i32, u8, f32 = T.c_int32_p, T.c_uint8_p, T.c_float_p
        k = self.lib.orc_stereo_lift_lines(
            C.byref(cam), C.byref(scfg), n, seg_l.ctypes.data_as(f32), angle_l.ctypes.data_as(f32),
            octave_l.ctypes.data_as(i32), desc_l.ctypes.data_as(u8), seg_r.ctypes.data_as(f32), m12.ctypes.data_as(i32),
            self._dp(out["spl"]), self._dp(out["epl"]), self._dp(out["sdisp"]), self._dp(out["edisp"]), self._dp(out["sP"]),
            self._dp(out["eP"]), self._dp(out["le"]), self._dp(out["angle"]), self._dp(out["sigma2"]),
            out["level"].ctypes.data_as(i32), out["desc"].ctypes.data_as(u8), out["src_idx"].ctypes.data_as(i32))
        return k, {key: v[:k] for key, v in out.items()}

    def match_stereo_points(self, cam, mcfg, scfg, kp_l, octave_l, desc_l, kp_r, desc_r):
        """matchStereoPoints for one frame: returns m12, k, records (first k rows)."""
        kp_l, kp_r = np.ascontiguousarray(kp_l, np.float32).reshape(-1, 2), np.ascontiguousarray(kp_r, np.float32).reshape(-1, 2)
        octave_l = np.ascontiguousarray(octave_l, np.int32)
        desc_l, desc_r = np.ascontiguousarray(desc_l, np.uint8).reshape(-1, 32), np.ascontiguousarray(desc_r, np.uint8).reshape(-1, 32)
        n = len(kp_l)
        m12 = np.full(n, -1, np.int32)
        out = dict(pl=np.zeros((n, 2)), disp=np.zeros(n), P=np.zeros((n, 3)), sigma2=np.zeros(n), level=np.zeros(n, np.int32),
                   desc=np.zeros((n, 32), np.uint8), src_idx=np.full(n, -1, np.int32))
        i32, u8, f32 = T.c_int32_p, T.c_uint8_p, T.c_float_p
        k = self.lib.orc_match_stereo_points(
            C.byref(cam), C.byref(mcfg), C.byref(scfg), n, kp_l.ctypes.data_as(f32), octave_l.ctypes.data_as(i32),
            desc_l.ctypes.data_as(u8), len(kp_r), kp_r.ctypes.data_as(f32), desc_r.ctypes.data_as(u8), m12.ctypes.data_as(i32),
            self._dp(out["pl"]), self._dp(out["disp"]), self._dp(out["P"]), self._dp(out["sigma2"]),
            out["level"].ctypes.data_as(i32), out["desc"].ctypes.data_as(u8), out["src_idx"].ctypes.data_as(i32))
        return m12, k, {key: v[:k] for key, v in out.items()}

    def match_stereo_lines(self, cam, mcfg, scfg, seg_l, angle_l, octave_l, desc_l, seg_r, desc_r):
        seg_l, seg_r = np.ascontiguousarray(seg_l, np.float32).reshape(-1, 4), np.ascontiguousarray(seg_r, np.float32).reshape(-1, 4)
        angle_l, octave_l = np.ascontiguousarray(angle_l, np.float32), np.ascontiguousarray(octave_l, np.int32)
        desc_l, desc_r = np.ascontiguousarray(desc_l, np.uint8).reshape(-1, 32), np.ascontiguousarray(desc_r, np.uint8).reshape(-1, 32)
        n = len(seg_l)
        m12 = np.full(n, -1, np.int32)
        out = dict(spl=np.zeros((n, 2)), epl=np.zeros((n, 2)), sdisp=np.zeros(n), edisp=np.zeros(n), sP=np.zeros((n, 3)),
                   eP=np.zeros((n, 3)), le=np.zeros((n, 3)), angle=np.zeros(n), sigma2=np.zeros(n),
                   level=np.zeros(n, np.int32), desc=np.zeros((n, 32), np.uint8), src_idx=np.full(n, -1, np.int32))
        i32, u8, f32 = T.c_int32_p, T.c_uint8_p, T.c_float_p
        k = self.lib.orc_match_stereo_lines(
            C.byref(cam), C.byref(mcfg), C.byref(scfg), n, seg_l.ctypes.data_as(f32), angle_l.ctypes.data_as(f32),
            octave_l.ctypes.data_as(i32), desc_l.ctypes.data_as(u8), len(seg_r), seg_r.ctypes.data_as(f32),
            desc_r.ctypes.data_as(u8), m12.ctypes.data_as(i32), self._dp(out["spl"]), self._dp(out["epl"]), self._dp(out["sdisp"]),
            self._dp(out["edisp"]), self._dp(out["sP"]), self._dp(out["eP"]), self._dp(out["le"]), self._dp(out["angle"]),
            self._dp(out["sigma2"]), out["level"].ctypes.data_as(i32), out["desc"].ctypes.data_as(u8),
            out["src_idx"].ctypes.data_as(i32))
        return m12, k, {key: v[:k] for key, v in out.items()}

    def stereo_batch(self, cam, mcfg, scfg, pl_off, kp_l, poct, pd1, pr_off, kp_r, pd2, ll_off, seg_l, angle, loct, ld1, lr_off,
                     seg_r, ld2, threads=1):
        """matchStereoPoints + matchStereoLines for B frames on `threads` host threads; returns counts[B, 2]."""
        i32, u8, f32 = T.c_int32_p, T.c_uint8_p, T.c_float_p
        cv = lambda a, dt: np.ascontiguousarray(a, dt)
        arrs = [cv(pl_off, np.int32), cv(kp_l, np.float32), cv(poct, np.int32), cv(pd1, np.uint8), cv(pr_off, np.int32),
                cv(kp_r, np.float32), cv(pd2, np.uint8), cv(ll_off, np.int32), cv(seg_l, np.float32), cv(angle, np.float32),
                cv(loct, np.int32), cv(ld1, np.uint8), cv(lr_off, np.int32), cv(seg_r, np.float32), cv(ld2, np.uint8)]
        typ = [i32, f32, i32, u8, i32, f32, u8, i32, f32, f32, i32, u8, i32, f32, u8]
        B = len(arrs[0]) - 1
        counts = np.zeros((B, 2), np.int32)
        self.lib.orc_stereo_batch(C.byref(cam), C.byref(mcfg), C.byref(scfg), B, *[a.ctypes.data_as(t) for a, t in zip(arrs, typ)],
                                  int(threads), counts.ctypes.data_as(i32))
        return counts

    def line_segment_overlap_stereo(self, scfg, spl_obs, epl_obs, spl_proj, epl_proj):
        return self.lib.orc_line_segment_overlap_stereo(C.byref(scfg), float(spl_obs), float(epl_obs), float(spl_proj), float(epl_proj))

    def line_cells(self, x1, y1, x2, y2, cap=512):
        cells = np.zeros((cap, 2), np.int32)
        n = self.lib.orc_line_cells(float(x1), float(y1), float(x2), float(y2), cells.ctypes.data_as(T.c_int32_p), cap)
        return cells[:min(n, cap)]

    # ---- SE(3) / statistics ----
    def inverse_se3(self, Tm):
        return self._unary("orc_inverse_se3", Tm, 16).reshape(4, 4)

    def expmap_se3(self, x):
        return self._unary("orc_expmap_se3", x, 16).reshape(4, 4)

    def logmap_se3(self, Tm):
        return self._unary("orc_logmap_se3", Tm, 6)

    def adjoint_se3(self, Tm):
        return self._unary("orc_adjoint_se3", Tm, 36).reshape(6, 6)

    def inv6(self, A):
        return self._unary("orc_inv6", A, 36).reshape(6, 6)

    def eig6_sym(self, A):
        return self._unary("orc_eig6_sym", A, 6)

    def unccomp_se3(self, T1, c1, cinc):
        T1, c1, cinc = self._d(T1).ravel(), self._d(c1).ravel(), self._d(cinc).ravel()
        out = np.zeros(36)
        self.lib.orc_unccomp_se3(self._dp(T1), self._dp(c1), self._dp(cinc), self._dp(out))
        return out.reshape(6, 6)

    def qr6_solve(self, H, g):
        H, g = self._d(H).ravel(), self._d(g).ravel()
        x, lad = np.zeros(6), np.zeros(1)
        rank = self.lib.orc_qr6_solve(self._dp(H), self._dp(g), self._dp(x), self._dp(lad))
        return x, float(lad[0]), rank

    def is_finite(self, x) -> bool:
        x = self._d(x).ravel()
        return bool(self.lib.orc_is_finite(self._dp(x), len(x)))

    def vector_mean_stdv_mad(self, res):
        res = self._d(res).ravel()
        m, s = np.zeros(1), np.zeros(1)
        self.lib.orc_vector_mean_stdv_mad(self._dp(res), len(res), self._dp(m), self._dp(s))
        return float(m[0]), float(s[0])

    def vector_stdv_mad(self, res) -> float:
        res = self._d(res).ravel()
        return float(self.lib.orc_vector_stdv_mad(self._dp(res), len(res)))

    def robust_weight_cauchy(self, r) -> float:
        return float(self.lib.orc_robust_weight_cauchy(float(r)))

    def line_segment_overlap(self, spl_obs, epl_obs, spl_proj, epl_proj) -> float:
        a, b, c, d = (self._d(v).ravel() for v in (spl_obs, epl_obs, spl_proj, epl_proj))
        return float(self.lib.orc_line_segment_overlap(self._dp(a), self._dp(b), self._dp(c), self._dp(d)))

    def projection(self, cam, P):
        P = self._d(P).ravel()
        uv = np.zeros(2)
        self.lib.orc_projection(C.byref(cam), self._dp(P), self._dp(uv))
        return uv

    def back_projection(self, cam, u, v, disp):
        P = np.zeros(3)
        self.lib.orc_back_projection(C.byref(cam), float(u), float(v), float(disp), self._dp(P))
        return P

    # ---- solver ----
    def optimize_functions(self, cam, cfg, matched: T.MatchedBatch, p, DT, robust=False):
        DT = self._d(DT).ravel()
        H, g, e = np.zeros(36), np.zeros(6), np.zeros(1)
        mc = matched.as_c()
        self.lib.orc_optimize_functions(C.byref(cam), C.byref(cfg), C.byref(mc), int(p), self._dp(DT), int(robust),
                                        self._dp(H), self._dp(g), self._dp(e))
        return H.reshape(6, 6), g, float(e[0])

    def optimize_pose(self, cam, cfg, matched: T.MatchedBatch, priors=None):
        B = matched.B
        res = np.zeros(B, dtype=T.POSE_RESULT_DTYPE)
        inl_pt = np.zeros(int(matched.pt_off[-1]), np.uint8)
        inl_ls = np.zeros(int(matched.ls_off[-1]), np.uint8)
        mc = matched.as_c()
        rc = self.lib.orc_optimize_pose(C.byref(cam), C.byref(cfg), C.byref(mc),
                                        priors.ctypes.data if priors is not None else None, res.ctypes.data,
                                        inl_pt.ctypes.data_as(T.c_uint8_p), inl_ls.ctypes.data_as(T.c_uint8_p))
        return rc, res, inl_pt, inl_ls

    def f2f_tracking(self, cfg, prev: T.FrameBatch, curr: T.FrameBatch):
        m12_pt = np.full(prev.n_pt, -1, np.int32)
        m12_ls = np.full(prev.n_ls, -1, np.int32)
        n = np.zeros((prev.B, 2), np.int32)
        pc, cc = prev.as_c(), curr.as_c()
        rc = self.lib.orc_f2f_tracking(C.byref(cfg), C.byref(pc), C.byref(cc), m12_pt.ctypes.data_as(T.c_int32_p),
                                       m12_ls.ctypes.data_as(T.c_int32_p), n.ctypes.data_as(T.c_int32_p))
        return rc, m12_pt, m12_ls, n

    def track_batch(self, cam, cfg, prev: T.FrameBatch, curr: T.FrameBatch, priors=None, threads=1,
                    faithful=False):
        B = prev.B
        res = np.zeros(B, dtype=T.POSE_RESULT_DTYPE)
        m12_pt = np.full(prev.n_pt, -1, np.int32)
        m12_ls = np.full(prev.n_ls, -1, np.int32)
        inl_pt = np.zeros(prev.n_pt, np.uint8)
        inl_ls = np.zeros(prev.n_ls, np.uint8)
        stage = np.zeros(2)
        pc, cc = prev.as_c(), curr.as_c()
        rc = self.lib.orc_track_batch(C.byref(cam), C.byref(cfg), C.byref(pc), C.byref(cc),
                                      priors.ctypes.data if priors is not None else None, res.ctypes.data,
                                      m12_pt.ctypes.data_as(T.c_int32_p), m12_ls.ctypes.data_as(T.c_int32_p),
                                      inl_pt.ctypes.data_as(T.c_uint8_p), inl_ls.ctypes.data_as(T.c_uint8_p),
                                      int(threads), int(faithful), self._dp(stage))
        return dict(rc=rc, results=res, m12_pt=m12_pt, m12_ls=m12_ls, inlier_pt=inl_pt, inlier_ls=inl_ls,
                    stage_ms=stage)
