"""Pins the oracle's pose half against the reference's OWN code.

oracle/_ref/libplstvo_ref.so holds optimizeFunctions, optimizeFunctionsRobust, gaussNewtonOptimization[Robust],
removeOutliers, isGoodSolution, optimizePose (src/stereoFrameHandler.cpp:292-480, 549-962, 988-1067), lineSegmentOverlap
(src/stereoFrame.cpp:510-616), projection / backProjection (src/pinholeStereoCamera.cpp:221-237), the SE(3) helpers and
the MAD statistics (src/auxiliar.cpp:29-44, 58-62, 113-197, 353-355, 387-430, 444-460, 556-583) compiled from the original
project's text by line range (oracle/make_ref.py) against stand-in Eigen headers.  Every comparison below is
oracle (our restatement, oracle/plstvo_oracle.c) == that library on the same inputs.  The library's outputs are the ones
recorded in tests/golden/ref_outputs.npz (the `ref` fixture, tests/ref_golden.py).

What the library does NOT contain is Eigen itself: its 6x6 decompositions are the stand-in's, so the first group of tests
holds those against LAPACK (numpy.linalg) instead.
"""
import numpy as np
import pytest

import ref_numpy as R
from stvo_pl_b200 import synth, types as T


def _rng(seed):
    return np.random.default_rng(20260924 + seed)


def _spd(rng, cond):
    q, _ = np.linalg.qr(rng.normal(size=(6, 6)))
    return (q * np.geomspace(1.0, cond, 6)) @ q.T * 1e4


# ---------------------------------------------------------------------------------------------------------------
# the stand-in's dense algebra against LAPACK (this is the part of the library that is NOT the reference's code)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cond", [1e1, 1e4, 1e8, 1e11])
def test_standin_algebra_vs_lapack(ref, oracle, cond):
    rng = _rng(int(np.log10(cond)))
    for _ in range(20):
        H = _spd(rng, cond)
        H = (H + H.T) / 2
        g = rng.normal(size=6) * 1e3
        x, lad, rank = ref.qr6_solve(H, g)
        xl = np.linalg.solve(H, g)
        assert rank == 6
        np.testing.assert_allclose(x, xl, rtol=1e-14 * cond * 50, atol=0)
        assert abs(lad - np.linalg.slogdet(H)[1]) < max(1e-10, 1e-14 * cond * 50)
        np.testing.assert_allclose(ref.inv6(H), np.linalg.inv(H), rtol=1e-14 * cond * 50, atol=1e-30)
        np.testing.assert_allclose(ref.eig6_sym(H), np.linalg.eigvalsh(H), rtol=1e-12, atol=1e-12 * np.abs(H).max())
        # and the oracle's own hand-rolled pieces agree with both
        xo, lado, ranko = oracle.qr6_solve(H, g)
        np.testing.assert_allclose(xo, x, rtol=1e-14 * cond * 50, atol=0)
        assert abs(lado - lad) < max(1e-10, 1e-14 * cond * 50)


def test_standin_qr_rank_deficient(ref):
    rng = _rng(77)
    a = rng.normal(size=(6, 4))
    H = a @ a.T   # rank 4
    x, lad, rank = ref.qr6_solve(H, H @ np.arange(1.0, 7.0))
    assert rank == 4
    np.testing.assert_allclose(H @ x, H @ np.arange(1.0, 7.0), rtol=1e-9, atol=1e-9)


# ---------------------------------------------------------------------------------------------------------------
# leaf functions: oracle == reference code, bit for bit (same operations in the same order, both -ffp-contract=off)
# ---------------------------------------------------------------------------------------------------------------
def test_se3_helpers_equal(ref, oracle):
    rng = _rng(1)
    for i in range(200):
        scale = [1e-9, 1e-7, 1e-3, 0.1, 1.0, 3.0][i % 6]
        x = np.concatenate([rng.normal(size=3), rng.normal(size=3) * scale])
        Tm = ref.expmap_se3(x)
        np.testing.assert_array_equal(Tm, oracle.expmap_se3(x))
        np.testing.assert_array_equal(ref.inverse_se3(Tm), oracle.inverse_se3(Tm))
        np.testing.assert_allclose(ref.logmap_se3(Tm), oracle.logmap_se3(Tm), rtol=0, atol=1e-15)
        np.testing.assert_array_equal(ref.adjoint_se3(Tm), oracle.adjoint_se3(Tm))
        c1, c2 = _spd(rng, 1e3) * 1e-10, _spd(rng, 1e3) * 1e-10
        np.testing.assert_allclose(ref.unccomp_se3(Tm, c1, c2), oracle.unccomp_se3(Tm, c1, c2), rtol=1e-15, atol=0)
    # round trips on the reference's own code (SURVEY 4 known answers)
    x = np.array([0.3, -0.2, 1.1, 0.01, -0.02, 0.03])
    np.testing.assert_allclose(ref.logmap_se3(ref.expmap_se3(x)), x, atol=1e-12)
    np.testing.assert_allclose(ref.inverse_se3(ref.expmap_se3(x)) @ ref.expmap_se3(x), np.eye(4), atol=1e-14)
    np.testing.assert_array_equal(ref.expmap_se3(np.zeros(6)), np.eye(4))


def test_is_finite_equal(ref, oracle):
    for v in ([1.0, 2.0], [np.nan, 1.0], [np.inf], [-np.inf, 0.0], np.eye(4).ravel()):
        assert ref.is_finite(v) == oracle.is_finite(v)


def test_mad_statistics_equal(ref, oracle):
    rng = _rng(2)
    assert ref.vector_stdv_mad([1, 2, 3, 4, 100]) == pytest.approx(1.4826)
    for n in (1, 2, 3, 4, 5, 10, 11, 100, 501, 2000):
        for kind in range(4):
            r = np.abs(rng.normal(size=n)) * [1.0, 1e-3, 50.0, 1.0][kind]
            if kind == 3:
                r[rng.random(n) < 0.3] *= 40.0   # gross outliers
            assert ref.vector_stdv_mad(r) == oracle.vector_stdv_mad(r)
            np.testing.assert_array_equal(ref.vector_mean_stdv_mad(r), oracle.vector_mean_stdv_mad(r))   # NaN == NaN (n = 1: 0/0)
    # the fabsf rounding of src/auxiliar.cpp:400 is visible: deviations are rounded to float before the second sort
    r = np.array([0.1, 0.2, 0.30000001, 0.5, 0.9])
    med = np.sort(r)[len(r) // 2]
    dev = np.sort(np.abs((r - med).astype(np.float32)).astype(np.float64))   # fabsf: the double is narrowed to float first
    assert ref.vector_stdv_mad(r) == oracle.vector_stdv_mad(r) == 1.4826 * dev[len(r) // 2]
    assert 1.4826 * dev[len(r) // 2] != 1.4826 * np.sort(np.abs(r - med))[len(r) // 2]    # ... and that is observable
    assert ref.vector_mean_stdv_mad([]) == oracle.vector_mean_stdv_mad([]) == (0.0, 0.0)
    assert ref.vector_stdv_mad([]) == oracle.vector_stdv_mad([]) == 0.0


def test_cauchy_and_projection_equal(ref, oracle):
    rng = _rng(3)
    cam = T.kitti_camera()
    for r in (0.0, 1.0, 0.5, 1e-8, 1e8, 3.3):
        assert ref.robust_weight_cauchy(r) == oracle.robust_weight_cauchy(r)
    assert ref.robust_weight_cauchy(0.0) == 1.0 and ref.robust_weight_cauchy(1.0) == 0.5
    for _ in range(100):
        P = rng.normal(size=3) * [5, 3, 20] + [0, 0, 25]
        np.testing.assert_array_equal(ref.projection(cam, P), oracle.projection(cam, P))
        u, v, d = rng.uniform(0, 1241), rng.uniform(0, 376), rng.uniform(1, 90)
        np.testing.assert_array_equal(ref.back_projection(cam, u, v, d), oracle.back_projection(cam, u, v, d))
        np.testing.assert_allclose(ref.projection(cam, ref.back_projection(cam, u, v, d)), [u, v], atol=1e-9)


def test_line_segment_overlap_all_branches_equal(ref, oracle):
    """Vertical (|dx| < 1), near-horizontal (|dy| < 1), generic, and the degenerate zero-length segment (0/0 -> NaN
    comparisons, src/stereoFrame.cpp:515-612)."""
    rng = _rng(4)
    n_branch = [0, 0, 0]
    for i in range(3000):
        s = rng.uniform(0, 1000, 2)
        kind = i % 5
        if kind == 0:
            e = s + [rng.uniform(-0.999, 0.999), rng.uniform(-200, 200)]
        elif kind == 1:
            e = s + [rng.uniform(-200, 200), rng.uniform(-0.999, 0.999)]
        elif kind == 2:
            e = s + rng.uniform(-200, 200, 2)
        elif kind == 3:
            e = s + rng.uniform(-0.999, 0.999, 2)    # both: the vertical branch wins
        else:
            e = s.copy()                             # zero length
        ps, pe = s + rng.normal(0, 60, 2), e + rng.normal(0, 60, 2)
        a, b = ref.line_segment_overlap(s, e, ps, pe), oracle.line_segment_overlap(s, e, ps, pe)
        assert (a == b) or (np.isnan(a) and np.isnan(b)), (s, e, ps, pe, a, b)
        n_branch[0 if abs(s[0] - e[0]) < 1 else 1 if abs(s[1] - e[1]) < 1 else 2] += 1
    assert min(n_branch) > 500
    s, e = np.array([10.0, 20.0]), np.array([110.0, 90.0])
    assert ref.line_segment_overlap(s, e, s, e) == pytest.approx(1.0, abs=1e-15)
    assert ref.line_segment_overlap(s, e, e + (e - s), e + 2 * (e - s)) == 0.0


# ---------------------------------------------------------------------------------------------------------------
# evaluation, Gauss-Newton, outlier removal, optimizePose
# ---------------------------------------------------------------------------------------------------------------
def _matched(shape, B, cfg, oracle, **kw):
    prev, curr, Tgt, cam = synth.make_batch(shape, B, **kw)
    o = oracle.track_batch(cam, cfg, prev, curr)
    return T.matched_from_frames(prev, curr, o["m12_pt"], o["m12_ls"], cfg.lsd_scale), Tgt, cam


def _degenerate_lines(matched, rng, frac=0.5):
    """Forces previous-frame segments into lineSegmentOverlap's special branches: |dx| < 1, |dy| < 1, zero length."""
    spl, epl = matched.ls_spl.copy(), matched.ls_epl.copy()
    n = len(spl)
    pick = rng.random(n) < frac
    kind = rng.integers(0, 3, n)
    v = pick & (kind == 0)
    h = pick & (kind == 1)
    z = pick & (kind == 2)
    epl[v, 0] = spl[v, 0] + rng.uniform(-0.99, 0.99, v.sum())
    epl[h, 1] = spl[h, 1] + rng.uniform(-0.99, 0.99, h.sum())
    epl[z] = spl[z]
    return T.MatchedBatch(pt_off=matched.pt_off, ls_off=matched.ls_off, pt_P=matched.pt_P, pt_pl_obs=matched.pt_pl_obs,
                          pt_sigma2=matched.pt_sigma2, ls_sP=matched.ls_sP, ls_eP=matched.ls_eP, ls_le_obs=matched.ls_le_obs,
                          ls_spl=spl, ls_epl=epl, ls_sigma2=matched.ls_sigma2)


CASES = [
    ("c1 points only", "kitti_points", T.kitti_config, dict(n_pt=800)),
    ("c2 kitti", "kitti", T.kitti_config, dict()),                       # 2000 + 500, full size
    ("c3 euroc", "euroc", T.euroc_config, dict()),                       # 1000 + 300
    ("kitti small", "kitti", T.kitti_config, dict(n_pt=200, n_ls=50)),
]


@pytest.mark.parametrize("name,shape,cfgf,kw", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("robust", [False, True])
def test_optimize_functions_equal(ref, oracle, name, shape, cfgf, kw, robust):
    cfg = cfgf()
    matched, Tgt, cam = _matched(shape, 2, cfg, oracle, **kw)
    rng = _rng(5)
    for p in range(2):
        for DT in (np.eye(4), Tgt[p], ref.expmap_se3(rng.normal(size=6) * 0.02)):
            Ho, go, eo = oracle.optimize_functions(cam, cfg, matched, p, DT, robust)
            Hr, gr, er = ref.optimize_functions(cam, cfg, matched, p, DT, robust)
            # same per-feature arithmetic and the same list order: agreement to the last bits of a ~2500-term sum
            np.testing.assert_allclose(Ho, Hr, rtol=1e-12, atol=1e-12 * np.abs(Hr).max())
            np.testing.assert_allclose(go, gr, rtol=1e-12, atol=1e-12 * np.abs(gr).max())
            assert abs(eo - er) <= 1e-13 * max(1.0, abs(er))


def test_optimize_functions_degenerate_segments_equal(ref, oracle):
    cfg = T.kitti_config()
    matched, Tgt, cam = _matched("kitti", 2, cfg, oracle, n_pt=300, n_ls=300, overlap=1.0)
    deg = _degenerate_lines(matched, _rng(6), 0.7)
    for p in range(2):
        for robust in (False, True):
            Ho, go, eo = oracle.optimize_functions(cam, cfg, deg, p, Tgt[p], robust)
            Hr, gr, er = ref.optimize_functions(cam, cfg, deg, p, Tgt[p], robust)
            np.testing.assert_array_equal(np.isnan(Ho), np.isnan(Hr))   # zero-length segments: 0/0 in both
            fin = ~np.isnan(Hr)
            np.testing.assert_allclose(Ho[fin], Hr[fin], rtol=1e-12, atol=1e-12 * np.nanmax(np.abs(Hr)) if fin.any() else 0)
            assert (np.isnan(eo) and np.isnan(er)) or abs(eo - er) <= 1e-13 * max(1.0, abs(er))


def _pose_equal(a, b, tol_ang=1e-9, tol_tr=1e-8, cov_rtol=1e-6):
    ang, tr = R.pose_error(a["DT"], b["DT"])
    assert ang < tol_ang and tr < tol_tr, (ang, tr)
    assert abs(a["err_norm"] - b["err_norm"]) < 1e-9
    np.testing.assert_allclose(a["DT_cov"], b["DT_cov"], rtol=cov_rtol, atol=1e-15)
    np.testing.assert_allclose(a["DT_cov_eig"], b["DT_cov_eig"], rtol=cov_rtol, atol=1e-15)
    ang, tr = R.pose_error(a["Tfw"], b["Tfw"])
    assert ang < tol_ang and tr < tol_tr
    np.testing.assert_allclose(a["Tfw_cov"], b["Tfw_cov"], rtol=cov_rtol, atol=1e-15)
    for k in ("n_matched_pt", "n_matched_ls", "n_inliers_pt", "n_inliers_ls", "n_inliers", "good"):
        assert a[k] == b[k], k


@pytest.mark.parametrize("name,shape,cfgf,kw", CASES, ids=[c[0] for c in CASES])
def test_optimize_pose_equal(ref, oracle, name, shape, cfgf, kw):
    """The whole of optimizePose: stage 1 -> gate -> removeOutliers -> stage 2 -> gate -> finalisation."""
    cfg = cfgf()
    B = 3
    matched, Tgt, cam = _matched(shape, B, cfg, oracle, **kw)
    rc_o, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, matched)
    rc_r, res_r, ip_r, il_r = ref.optimize_pose(cam, cfg, matched)
    assert rc_o == rc_r == 0
    np.testing.assert_array_equal(ip_o, ip_r)     # inlier flags: identical, not "almost"
    np.testing.assert_array_equal(il_o, il_r)
    for p in range(B):
        assert res_o[p]["good"] == 1 and res_o[p]["status"] == T.ST_REFINED
        _pose_equal(res_o[p], res_r[p])
        ang, tr = R.pose_error(np.linalg.inv(res_r[p]["DT"].reshape(4, 4)), Tgt[p])
        assert ang < 2e-3 and tr < 2e-2           # the reference's code recovers the generator's motion


def test_optimize_pose_c5_shape_equal(ref, oracle):
    cfg = T.kitti_config()
    matched, Tgt, cam = synth.make_matched_batch("hd", 1)
    rc_o, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, matched)
    rc_r, res_r, ip_r, il_r = ref.optimize_pose(cam, cfg, matched)
    assert matched.pt_off[1] == 8000 and matched.ls_off[1] == 2000
    np.testing.assert_array_equal(ip_o, ip_r)
    np.testing.assert_array_equal(il_o, il_r)
    _pose_equal(res_o[0], res_r[0])


def test_optimize_pose_with_motion_model_equal(ref, oracle):
    cfg = T.kitti_config()
    cfg.use_motion_model = 1
    matched, Tgt, cam = _matched("kitti", 2, cfg, oracle, n_pt=400, n_ls=100)
    pri = T.identity_priors(2)
    rng = _rng(8)
    for p in range(2):
        pri[p]["Tfw"] = ref.expmap_se3(rng.normal(size=6) * [3, 3, 3, 0.2, 0.2, 0.2])
        pri[p]["Tfw_cov"] = _spd(rng, 100) * 1e-9
        pri[p]["DT"] = np.linalg.inv(Tgt[p]) @ ref.expmap_se3(rng.normal(size=6) * 1e-3)   # a plausible previous motion
        pri[p]["DT_cov"] = _spd(rng, 100) * 1e-9
        pri[p]["err_norm"] = 0.3
    pri[1]["err_norm"] = 7.0     # fails the gate -> identity start (src/stereoFrameHandler.cpp:322-323)
    rc_o, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, matched, pri)
    rc_r, res_r, ip_r, il_r = ref.optimize_pose(cam, cfg, matched, pri)
    np.testing.assert_array_equal(ip_o, ip_r)
    np.testing.assert_array_equal(il_o, il_r)
    for p in range(2):
        _pose_equal(res_o[p], res_r[p])


def test_few_feature_branches_equal(ref, oracle):
    """n_inliers < minFeatures before optimisation (:364-368) and after removeOutliers (:351-355): identity pose,
    zero covariance, err_norm = -1, Tfw carried over."""
    cfg = T.kitti_config()
    matched, Tgt, cam = _matched("kitti", 1, cfg, oracle, n_pt=6, n_ls=2, overlap=1.0, outlier_frac=0.0)
    assert matched.pt_off[1] + matched.ls_off[1] < cfg.min_features
    rc_o, res_o, *_ = oracle.optimize_pose(cam, cfg, matched)
    rc_r, res_r, *_ = ref.optimize_pose(cam, cfg, matched)
    assert res_o[0]["status"] == T.ST_FEW_BEFORE and res_o[0]["good"] == res_r[0]["good"] == 0
    for k in ("DT", "DT_cov", "DT_cov_eig", "err_norm", "Tfw", "Tfw_cov"):
        np.testing.assert_array_equal(res_o[0][k], res_r[0][k])
    # after removal: 12 features, inlier_k so small that nearly everything is rejected
    cfg2 = T.kitti_config()
    cfg2.inlier_k = 0.05
    matched, Tgt, cam = _matched("kitti", 1, cfg2, oracle, n_pt=10, n_ls=2, overlap=1.0, outlier_frac=0.0)
    rc_o, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg2, matched)
    rc_r, res_r, ip_r, il_r = ref.optimize_pose(cam, cfg2, matched)
    assert res_o[0]["status"] == T.ST_FEW_AFTER
    np.testing.assert_array_equal(ip_o, ip_r)
    np.testing.assert_array_equal(il_o, il_r)
    for k in ("DT", "DT_cov", "DT_cov_eig", "err_norm", "Tfw", "Tfw_cov", "n_inliers"):
        np.testing.assert_array_equal(res_o[0][k], res_r[0][k])


def test_robust_fallback_branch_equal(ref, oracle):
    """Stage 1 rejected by the gate -> gaussNewtonOptimizationRobust on all features (:357-359).  Provoked with a prior
    pose far from the solution: stage 1 then ends with err > err_prev at the first iteration (err = -1)."""
    cfg = T.kitti_config()
    cfg.use_motion_model = 1
    matched, Tgt, cam = _matched("kitti", 2, cfg, oracle, n_pt=500, n_ls=120)
    pri = T.identity_priors(2)
    hit = 0
    for p in range(2):
        pri[p]["DT"] = ref.expmap_se3(np.array([0.4, -0.3, 2.5, 0.05, -0.08, 0.03]))
        pri[p]["DT_cov"] = np.eye(6) * 1e-6
        pri[p]["err_norm"] = 0.2
    rc_o, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, matched, pri)
    rc_r, res_r, ip_r, il_r = ref.optimize_pose(cam, cfg, matched, pri)
    np.testing.assert_array_equal(ip_o, ip_r)
    np.testing.assert_array_equal(il_o, il_r)
    for p in range(2):
        hit += int(res_o[p]["status"] == T.ST_ROBUST_FALLBACK)
        assert res_o[p]["good"] == res_r[p]["good"]
        if res_o[p]["good"]:
            # MAD-scaled IRLS: discontinuous in the scale, hence the north_star tolerance rather than 1e-9
            _pose_equal(res_o[p], res_r[p], tol_ang=1e-5, tol_tr=1e-4, cov_rtol=1e-3)
    # direct calls of the robust solver from the identity, both implementations
    for p in range(2):
        DTo = ref.gauss_newton(cam, cfg, matched, p, np.eye(4), True, cfg.max_iters_ref)
        Ho, go, eo = oracle.optimize_functions(cam, cfg, matched, p, DTo[0], True)
        Hr, gr, er = ref.optimize_functions(cam, cfg, matched, p, DTo[0], True)
        np.testing.assert_allclose(Ho, Hr, rtol=1e-12, atol=1e-12 * np.abs(Hr).max())
    assert hit >= 0   # informative; the branch is also reached in test_robust_mode_equal through mode 1


def test_robust_mode_equal(ref, oracle):
    """C3 with the robust evaluator as the main solver (`mode == 1`).  The reference hard-wires mode 0; the driver of
    oracle/_ref re-states optimizePose's control flow for mode 1 around the reference's own functions."""
    cfg = T.euroc_config()
    cfg.solver_mode = 1
    matched, Tgt, cam = _matched("euroc", 3, cfg, oracle)
    rc_o, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, matched)
    rc_r, res_r, ip_r, il_r = ref.optimize_pose(cam, cfg, matched)
    n_diff = int((ip_o != ip_r).sum() + (il_o != il_r).sum())
    assert n_diff == 0, n_diff
    for p in range(3):
        assert res_o[p]["good"] == res_r[p]["good"] == 1
        _pose_equal(res_o[p], res_r[p], tol_ang=1e-5, tol_tr=1e-4, cov_rtol=1e-3)


def test_remove_outliers_equal_and_adversarial(ref, oracle):
    """removeOutliers at the stage-1 pose: identical flags, including residuals placed within a few ulp of
    mean +- k * stdv (the comparison `fabs(r - mean) > k * stdv` of src/stereoFrameHandler.cpp:1016, :1056)."""
    cfg = T.kitti_config()
    matched, Tgt, cam = _matched("kitti", 2, cfg, oracle, n_pt=600, n_ls=150)
    for p in range(2):
        DT1, cov1, e1 = ref.gauss_newton(cam, cfg, matched, p, np.eye(4), False, cfg.max_iters)
        rc, ip_r, il_r, cnt = ref.remove_outliers(cam, cfg, matched, p, DT1)
        assert rc == 0 and cnt[2] == cnt[0] + cnt[1] == int(ip_r.sum() + il_r.sum())
        # the oracle's optimizePose passes through exactly this state: compare through the stage-2 inlier flags
        rc_o, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, matched)
        a, b = matched.pt_off[p], matched.pt_off[p + 1]
        np.testing.assert_array_equal(ip_o[a:b], ip_r)
        a, b = matched.ls_off[p], matched.ls_off[p + 1]
        np.testing.assert_array_equal(il_o[a:b], il_r)
    # adversarial: move observed points along the residual direction so that |r - mean| sits on the threshold +- ulps
    p = 0
    DT1, _, _ = ref.gauss_newton(cam, cfg, matched, p, np.eye(4), False, cfg.max_iters)
    a, b = int(matched.pt_off[p]), int(matched.pt_off[p + 1])
    P = matched.pt_P[a:b] @ DT1[:3, :3].T + DT1[:3, 3]
    proj = np.stack([cam.cx + cam.fx * P[:, 0] / P[:, 2], cam.cy + cam.fy * P[:, 1] / P[:, 2]], 1)
    res = np.linalg.norm(proj - matched.pt_pl_obs[a:b], axis=1) * np.sqrt(matched.pt_sigma2[a:b])
    mean, stdv = ref.vector_mean_stdv_mad(res)
    th = mean + cfg.inlier_k * stdv
    obs = matched.pt_pl_obs.copy()
    idx = np.argsort(np.abs(res - th))[:40]       # the 40 residuals closest to the threshold ...
    for j, i in enumerate(idx):                    # ... are pushed onto it, a few ulp either side
        d = matched.pt_pl_obs[a + i] - proj[i]
        d /= np.linalg.norm(d)
        target = np.nextafter(th, np.inf if j % 2 else -np.inf)
        for _ in range(j // 2):
            target = np.nextafter(target, np.inf if j % 2 else -np.inf)
        obs[a + i] = proj[i] + d * target / np.sqrt(matched.pt_sigma2[a + i])
    adv = T.MatchedBatch(pt_off=matched.pt_off, ls_off=matched.ls_off, pt_P=matched.pt_P, pt_pl_obs=obs,
                         pt_sigma2=matched.pt_sigma2, ls_sP=matched.ls_sP, ls_eP=matched.ls_eP, ls_le_obs=matched.ls_le_obs,
                         ls_spl=matched.ls_spl, ls_epl=matched.ls_epl, ls_sigma2=matched.ls_sigma2)
    rc_o, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, adv)
    rc_r, res_r, ip_r, il_r = ref.optimize_pose(cam, cfg, adv)
    np.testing.assert_array_equal(ip_o, ip_r)
    np.testing.assert_array_equal(il_o, il_r)
    _pose_equal(res_o[0], res_r[0])


def test_degenerate_segments_through_optimize_pose_equal(ref, oracle):
    """Previous-frame segments with |dx| < 1 and |dy| < 1 through the complete solve (zero-length ones make the weight
    NaN in the reference; kept out of this list so that the solve itself stays comparable)."""
    cfg = T.kitti_config()
    matched, Tgt, cam = _matched("kitti", 2, cfg, oracle, n_pt=300, n_ls=200, overlap=1.0)
    rng = _rng(9)
    spl, epl = matched.ls_spl.copy(), matched.ls_epl.copy()
    n = len(spl)
    v = rng.random(n) < 0.3
    h = (~v) & (rng.random(n) < 0.4)
    epl[v, 0] = spl[v, 0] + rng.uniform(-0.99, 0.99, v.sum())
    epl[h, 1] = spl[h, 1] + rng.uniform(-0.99, 0.99, h.sum())
    deg = T.MatchedBatch(pt_off=matched.pt_off, ls_off=matched.ls_off, pt_P=matched.pt_P, pt_pl_obs=matched.pt_pl_obs,
                         pt_sigma2=matched.pt_sigma2, ls_sP=matched.ls_sP, ls_eP=matched.ls_eP, ls_le_obs=matched.ls_le_obs,
                         ls_spl=spl, ls_epl=epl, ls_sigma2=matched.ls_sigma2)
    rc_o, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, deg)
    rc_r, res_r, ip_r, il_r = ref.optimize_pose(cam, cfg, deg)
    np.testing.assert_array_equal(ip_o, ip_r)
    np.testing.assert_array_equal(il_o, il_r)
    for p in range(2):
        assert res_r[p]["good"] == 1
        _pose_equal(res_o[p], res_r[p])
