"""GPU parity on the thin spots VERDICT r1 named: lineSegmentOverlap's vertical / near-horizontal / zero-length branches
(src/stereoFrame.cpp:515, :545), residuals within a few ulp of removeOutliers' threshold (src/stereoFrameHandler.cpp:1016,
:1056 with src/auxiliar.cpp:399-427), and the robust (MAD-scaled) mode with the number of differing inlier flags reported.
Everything runs through the C-ABI (plstvo_optimize_pose / plstvo_track_batch / plstvo_gn_eval_stream) and is compared
with the oracle; the reference's own compiled code (as recorded in tests/golden/ref_outputs.npz) is the third party."""
import numpy as np
import pytest

import ref_numpy as R
from stvo_pl_b200 import synth, types as T

pytestmark = pytest.mark.gpu


def _matched(oracle, shape, B, cfg, **kw):
    prev, curr, Tgt, cam = synth.make_batch(shape, B, **kw)
    o = oracle.track_batch(cam, cfg, prev, curr)
    return T.matched_from_frames(prev, curr, o["m12_pt"], o["m12_ls"], cfg.lsd_scale), Tgt, cam, prev, curr


def _with_lines(m, spl, epl):
    return T.MatchedBatch(pt_off=m.pt_off, ls_off=m.ls_off, pt_P=m.pt_P, pt_pl_obs=m.pt_pl_obs, pt_sigma2=m.pt_sigma2,
                          ls_sP=m.ls_sP, ls_eP=m.ls_eP, ls_le_obs=m.ls_le_obs, ls_spl=spl, ls_epl=epl, ls_sigma2=m.ls_sigma2)


def _with_obs(m, obs):
    return T.MatchedBatch(pt_off=m.pt_off, ls_off=m.ls_off, pt_P=m.pt_P, pt_pl_obs=obs, pt_sigma2=m.pt_sigma2,
                          ls_sP=m.ls_sP, ls_eP=m.ls_eP, ls_le_obs=m.ls_le_obs, ls_spl=m.ls_spl, ls_epl=m.ls_epl,
                          ls_sigma2=m.ls_sigma2)


def _same_pose(a, b, ang_tol=1e-9, tr_tol=1e-8):
    ang, tr = R.pose_error(a["DT"], b["DT"])
    assert ang < ang_tol and tr < tr_tol, (ang, tr)
    assert a["good"] == b["good"] and a["n_inliers_pt"] == b["n_inliers_pt"] and a["n_inliers_ls"] == b["n_inliers_ls"]


def _degenerate(m, rng, frac_v=0.3, frac_h=0.3, frac_z=0.0):
    spl, epl = m.ls_spl.copy(), m.ls_epl.copy()
    n = len(spl)
    u = rng.random(n)
    v, h, z = u < frac_v, (u >= frac_v) & (u < frac_v + frac_h), (u >= frac_v + frac_h) & (u < frac_v + frac_h + frac_z)
    epl[v, 0] = spl[v, 0] + rng.uniform(-0.99, 0.99, v.sum())      # |dx| < 1: the "vertical" branch
    epl[h, 1] = spl[h, 1] + rng.uniform(-0.99, 0.99, h.sum())      # |dy| < 1: the "horizontal" branch
    epl[z] = spl[z]                                                # zero length: 0/0 in the vertical branch
    return _with_lines(m, spl, epl), int(v.sum()), int(h.sum()), int(z.sum())


def test_degenerate_previous_segments_through_the_solver(engine, oracle, ref):
    """|dx| < 1 and |dy| < 1 previous-frame segments through plstvo_optimize_pose (K2's pre-computed overlap coefficients
    must reproduce all three branches of lineSegmentOverlap)."""
    cfg = T.kitti_config()
    m, Tgt, cam, *_ = _matched(oracle, "kitti", 4, cfg, n_pt=300, n_ls=250, overlap=1.0)
    deg, nv, nh, _ = _degenerate(m, np.random.default_rng(11))
    assert nv > 150 and nh > 150
    res, ip, il = engine.optimize_pose(cam, cfg, deg)
    rc, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, deg)
    np.testing.assert_array_equal(ip, ip_o)
    np.testing.assert_array_equal(il, il_o)
    res_r = ref.optimize_pose(cam, cfg, deg)[1]
    for p in range(4):
        assert res[p]["good"] == 1
        _same_pose(res[p], res_o[p])
        _same_pose(res[p], res_r[p])


def test_degenerate_segments_through_the_streamed_evaluator(engine, oracle):
    """The same segments through plstvo_gn_eval_stream (fp32 records: H, g, e at fp32 level)."""
    cfg = T.kitti_config()
    m, Tgt, cam, *_ = _matched(oracle, "kitti", 3, cfg, n_pt=600, n_ls=600, overlap=1.0)
    deg, nv, nh, _ = _degenerate(m, np.random.default_rng(12), 0.35, 0.35)
    H, g, e, _ = engine.gn_eval_stream(cam, cfg, deg, Tgt, iters=1)
    for p in range(3):
        Ho, go, eo = oracle.optimize_functions(cam, cfg, deg, p, Tgt[p])
        np.testing.assert_allclose(H[p], Ho, rtol=5e-4, atol=5e-4 * np.abs(Ho).max())
        np.testing.assert_allclose(g[p], go, rtol=5e-3, atol=5e-4 * np.abs(go).max())
        assert abs(e[p] - eo) < 5e-4 * max(1.0, abs(eo))


def test_zero_length_previous_segments(engine, oracle, ref):
    """A zero-length previous segment divides by l(1) = 0 in the vertical branch (src/stereoFrame.cpp:515-544): the lambdas
    are +-inf (NaN only when the projected end point has exactly the same v), the overlap comes out as 0 or 1.  The GPU
    must take the same route: identical flags and pose, also against the reference's compiled code."""
    cfg = T.kitti_config()
    m, Tgt, cam, *_ = _matched(oracle, "kitti", 3, cfg, n_pt=200, n_ls=120, overlap=1.0)
    deg, _, _, nz = _degenerate(m, np.random.default_rng(13), 0.1, 0.1, 0.4)
    assert nz > 60
    res, ip, il = engine.optimize_pose(cam, cfg, deg)
    rc, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, deg)
    np.testing.assert_array_equal(ip, ip_o)
    np.testing.assert_array_equal(il, il_o)
    res_r = ref.optimize_pose(cam, cfg, deg)[1]
    for p in range(3):
        _same_pose(res[p], res_o[p])
        _same_pose(res[p], res_r[p])


def test_outlier_threshold_adversarial(engine, oracle, ref):
    """Observations moved along their residual direction so that |r - mean| lands within a few ulp of k * stdv on either
    side: the inlier flags must still be identical (the trimmed mean is a block-parallel sum in K2, a sequential one in the
    reference)."""
    cfg = T.kitti_config()
    m, Tgt, cam, *_ = _matched(oracle, "kitti", 2, cfg, n_pt=700, n_ls=150)
    obs = m.pt_pl_obs.copy()
    for p in range(2):
        a, b = int(m.pt_off[p]), int(m.pt_off[p + 1])
        one = T.MatchedBatch(pt_off=[0, b - a], ls_off=[0, 0], pt_P=m.pt_P[a:b], pt_pl_obs=m.pt_pl_obs[a:b],
                             pt_sigma2=m.pt_sigma2[a:b], ls_sP=np.zeros((0, 3)), ls_eP=np.zeros((0, 3)),
                             ls_le_obs=np.zeros((0, 3)), ls_spl=np.zeros((0, 2)), ls_epl=np.zeros((0, 2)), ls_sigma2=np.zeros(0))
        # stage-1 pose of the full problem from the oracle's diagnostic field is not exposed: re-derive the residuals at the
        # final pose instead (close to the stage-1 pose; the construction only needs residuals NEAR the threshold)
        rc, r0, _, _ = oracle.optimize_pose(cam, cfg, m)
        DT = r0[p]["DT_opt"].reshape(4, 4)
        P = m.pt_P[a:b] @ DT[:3, :3].T + DT[:3, 3]
        proj = np.stack([cam.cx + cam.fx * P[:, 0] / P[:, 2], cam.cy + cam.fy * P[:, 1] / P[:, 2]], 1)
        res = np.linalg.norm(proj - m.pt_pl_obs[a:b], axis=1) * np.sqrt(m.pt_sigma2[a:b])
        mean, stdv = oracle.vector_mean_stdv_mad(res)
        th = mean + cfg.inlier_k * stdv
        idx = np.argsort(np.abs(res - th))[:60]
        for j, i in enumerate(idx):
            d = m.pt_pl_obs[a + i] - proj[i]
            d /= np.linalg.norm(d)
            target = th
            for _ in range(1 + j // 2):
                target = np.nextafter(target, np.inf if j % 2 else -np.inf)
            obs[a + i] = proj[i] + d * target / np.sqrt(m.pt_sigma2[a + i])
    adv = _with_obs(m, obs)
    res, ip, il = engine.optimize_pose(cam, cfg, adv)
    rc, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, adv)
    assert int((ip != ip_o).sum()) == 0 and int((il != il_o).sum()) == 0
    for p in range(2):
        _same_pose(res[p], res_o[p])
    rc, res_r, ip_r, il_r = ref.optimize_pose(cam, cfg, adv)
    assert int((ip != ip_r).sum()) == 0 and int((il != il_r).sum()) == 0


def test_robust_mode_flag_differences_are_counted(engine, oracle):
    """C3 robust mode (MAD-scaled Cauchy weights, a discontinuous fixed-point iteration): pose within north_star's
    1e-5 rad / 1e-4 m; the number of differing inlier flags is REPORTED and must stay at the few-borderline level
    (SURVEY 8(c)-(3))."""
    cfg = T.euroc_config()
    cfg.solver_mode = 1
    m, Tgt, cam, prev, curr = _matched(oracle, "euroc", 8, cfg)
    res, ip, il = engine.optimize_pose(cam, cfg, m)
    rc, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, m)
    n_diff = int((ip != ip_o).sum() + (il != il_o).sum())
    n_all = len(ip) + len(il)
    print(f"robust mode: {n_diff} of {n_all} inlier flags differ between the GPU and the oracle")
    assert n_diff <= max(2, n_all // 2000)
    for p in range(8):
        ang, tr = R.pose_error(res[p]["DT"], res_o[p]["DT"])
        assert res[p]["good"] == res_o[p]["good"] == 1 and ang < 1e-5 and tr < 1e-4, (p, ang, tr)


def test_near_singular_normal_equations_take_the_qr_path(engine, oracle):
    """Ill-conditioned H (all points at nearly the same depth and direction: rotation and translation barely separable):
    K2's Cholesky fast path must hand over to the column-pivoted QR where the two would differ; the result follows the
    oracle (ColPivHouseholderQR semantics, src/stereoFrameHandler.cpp:417-418)."""
    cfg = T.kitti_config()
    cfg.has_lines = 0
    rng = np.random.default_rng(3)
    n = 60
    cam = T.kitti_camera()
    u, v = rng.uniform(600, 615, n), rng.uniform(180, 190, n)      # a tiny patch of the image, one depth
    d = np.full(n, cam.b * cam.fx / 40.0)
    P = synth.back_projection(cam, u, v, d)
    Tgt = synth.expmap_se3(np.array([0.01, 0.0, -0.3, 0.001, -0.002, 0.0005]))
    obs = synth.projection(cam, P @ Tgt[:3, :3].T + Tgt[:3, 3]) + rng.normal(0, 0.05, (n, 2))
    m = T.MatchedBatch(pt_off=[0, n], ls_off=[0, 0], pt_P=P, pt_pl_obs=obs, pt_sigma2=np.ones(n), ls_sP=np.zeros((0, 3)),
                       ls_eP=np.zeros((0, 3)), ls_le_obs=np.zeros((0, 3)), ls_spl=np.zeros((0, 2)), ls_epl=np.zeros((0, 2)),
                       ls_sigma2=np.zeros(0))
    res, ip, il = engine.optimize_pose(cam, cfg, m)
    rc, res_o, ip_o, il_o = oracle.optimize_pose(cam, cfg, m)
    assert res[0]["good"] == res_o[0]["good"] and res[0]["status"] == res_o[0]["status"]
    np.testing.assert_array_equal(ip, ip_o)
    if res_o[0]["good"]:
        ang, tr = R.pose_error(res[0]["DT"], res_o[0]["DT"])
        assert ang < 1e-5 and tr < 1e-4, (ang, tr)
