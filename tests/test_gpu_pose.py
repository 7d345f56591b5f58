"""Parity of the fused CUDA path (K1 -> K2: match, gather, optimizePose) with the oracle, through the C-ABI.
Bars: match indices and inlier flags bit-exact; pose within 1e-5 rad / 1e-4 m (north_star)."""
import os

import numpy as np
import pytest

import ref_numpy as R
from conftest import GOLDEN
from stvo_pl_b200 import synth, types as T

pytestmark = pytest.mark.gpu
TOL_ANG, TOL_TR = 1e-5, 1e-4      # north_star tolerance
TIGHT_ANG, TIGHT_TR = 1e-9, 1e-8  # what an all-fp64 implementation actually achieves on the GN path


def compare(gpu, ref, prev, tight=True, flags_exact=True):
    np.testing.assert_array_equal(gpu["m12_pt"], ref["m12_pt"])
    np.testing.assert_array_equal(gpu["m12_ls"], ref["m12_ls"])
    worst = (0.0, 0.0)
    for p in range(prev.B):
        g, r = gpu["results"][p], ref["results"][p]
        assert g["status"] == r["status"] and g["good"] == r["good"], (p, g["status"], r["status"])
        assert g["n_matched_pt"] == r["n_matched_pt"] and g["n_matched_ls"] == r["n_matched_ls"]
        ang, tr = R.pose_error(g["DT"], r["DT"])
        worst = (max(worst[0], ang), max(worst[1], tr))
        assert ang < (TIGHT_ANG if tight else TOL_ANG) and tr < (TIGHT_TR if tight else TOL_TR), (p, ang, tr)
        if tight:
            assert g["iters_stage1"] == r["iters_stage1"] and g["iters_stage2"] == r["iters_stage2"]
            assert g["n_inliers_pt"] == r["n_inliers_pt"] and g["n_inliers_ls"] == r["n_inliers_ls"]
            assert abs(g["err_norm"] - r["err_norm"]) < 1e-9
            np.testing.assert_allclose(g["DT_cov"], r["DT_cov"], rtol=1e-6, atol=1e-15)
            np.testing.assert_allclose(g["DT_cov_eig"], r["DT_cov_eig"], rtol=1e-6, atol=1e-16)
            np.testing.assert_allclose(g["Tfw"], r["Tfw"], atol=1e-8)
            np.testing.assert_allclose(g["Tfw_cov"], r["Tfw_cov"], rtol=1e-6, atol=1e-12)
    if flags_exact:
        np.testing.assert_array_equal(gpu["inlier_pt"], ref["inlier_pt"])
        np.testing.assert_array_equal(gpu["inlier_ls"], ref["inlier_ls"])
    return worst


@pytest.mark.parametrize("shape,cfgf,B,kw", [
    ("kitti", T.kitti_config, 3, dict(n_pt=400, n_ls=100)),
    ("kitti", T.kitti_config, 2, dict()),                       # C2 full size: 2000 + 500
    ("kitti", T.kitti_config, 2, dict(overlap=1.0)),            # bench workload: every feature re-observed
    ("euroc", T.euroc_config, 3, dict()),                       # 1000 + 300, 4 pyramid levels (sigma2 != 1)
    ("kitti_points", T.kitti_config, 2, dict()),                # C1: points only
    ("kitti", T.kitti_config, 2, dict(n_pt=700, n_ls=300, tie_stress=True)),
])
def test_track_vs_oracle(engine, oracle, shape, cfgf, B, kw):
    cfg = cfgf()
    prev, curr, Tgt, cam = synth.make_batch(shape, B, **kw)
    ref = oracle.track_batch(cam, cfg, prev, curr, threads=4)
    gpu = engine.track_batch(cam, cfg, prev, curr)
    compare(gpu, ref, prev)
    for p in range(B):
        if gpu["results"][p]["good"]:
            ang, tr = R.pose_error(gpu["results"]["DT_opt"][p], Tgt[p])
            assert ang < 3e-3 and tr < 3e-2


def test_points_only_config_flags(engine, oracle):
    cfg = T.kitti_config()
    cfg.has_lines = 0
    prev, curr, _, cam = synth.make_batch("kitti", 2, n_pt=500, n_ls=100)
    compare(engine.track_batch(cam, cfg, prev, curr), oracle.track_batch(cam, cfg, prev, curr), prev)
    cfg.has_lines, cfg.has_points = 1, 0
    compare(engine.track_batch(cam, cfg, prev, curr), oracle.track_batch(cam, cfg, prev, curr), prev)
    cfg.has_points, cfg.best_lr_matches = 1, 0
    compare(engine.track_batch(cam, cfg, prev, curr), oracle.track_batch(cam, cfg, prev, curr), prev)


def test_robust_mode(engine, oracle):
    """C3 'robust weights on': the `mode == 1` evaluator (MAD-scaled Cauchy weights).  The MAD-scaled IRLS is a
    discontinuous iteration (see tests/test_oracle_pose.py), so the bar is north_star's tolerance."""
    cfg = T.euroc_config()
    cfg.solver_mode = 1
    prev, curr, _, cam = synth.make_batch("euroc", 4)
    compare(engine.track_batch(cam, cfg, prev, curr), oracle.track_batch(cam, cfg, prev, curr, threads=4), prev,
            tight=False, flags_exact=False)


def test_explicit_list_api(engine, oracle):
    cfg = T.kitti_config()
    prev, curr, _, cam = synth.make_batch("kitti", 3, n_pt=600, n_ls=150)
    o = oracle.track_batch(cam, cfg, prev, curr)
    matched = T.matched_from_frames(prev, curr, o["m12_pt"], o["m12_ls"], cfg.lsd_scale)
    rc, ref, rp, rl = oracle.optimize_pose(cam, cfg, matched)
    res, ip, il = engine.optimize_pose(cam, cfg, matched)
    for p in range(3):
        ang, tr = R.pose_error(res["DT"][p], ref["DT"][p])
        assert ang < TIGHT_ANG and tr < TIGHT_TR
        assert res["status"][p] == ref["status"][p]
    np.testing.assert_array_equal(ip, rp)
    np.testing.assert_array_equal(il, rl)


def test_failure_encodings(engine, oracle):
    cfg = T.kitti_config()
    for kw in (dict(n_pt=6, n_ls=2, overlap=1.0), dict(n_pt=0, n_ls=0), dict(n_pt=30, n_ls=0, overlap=0.2)):
        prev, curr, _, cam = synth.make_batch("kitti", 2, **kw)
        ref = oracle.track_batch(cam, cfg, prev, curr)
        gpu = engine.track_batch(cam, cfg, prev, curr)
        compare(gpu, ref, prev)
        for p in range(2):
            if not gpu["results"][p]["good"]:
                np.testing.assert_array_equal(gpu["results"][p]["DT"], np.eye(4))
                np.testing.assert_array_equal(gpu["results"][p]["DT_cov"], np.zeros((6, 6)))
                assert gpu["results"][p]["err_norm"] == -1.0


def test_robust_fallback_branch(engine, oracle):
    cfg = T.kitti_config()
    cam = T.kitti_camera()
    rng = np.random.default_rng(2)
    n = 40
    P = np.stack([rng.normal(0, 1e-4, n), rng.normal(0, 1e-4, n), 400 + rng.normal(0, 1e-3, n)], 1)
    obs = np.stack([cam.cx + rng.normal(0, 0.3, n), cam.cy + rng.normal(0, 0.3, n)], 1)
    m = T.MatchedBatch(pt_off=[0, n], ls_off=[0, 0], pt_P=P, pt_pl_obs=obs, pt_sigma2=np.ones(n),
                       ls_sP=np.zeros((0, 3)), ls_eP=np.zeros((0, 3)), ls_le_obs=np.zeros((0, 3)),
                       ls_spl=np.zeros((0, 2)), ls_epl=np.zeros((0, 2)), ls_sigma2=np.zeros(0))
    rc, ref, _, _ = oracle.optimize_pose(cam, cfg, m)
    res, _, _ = engine.optimize_pose(cam, cfg, m)
    assert res[0]["status"] == ref[0]["status"] == T.ST_ROBUST_FALLBACK
    assert res[0]["good"] == ref[0]["good"]


def test_priors_motion_model_and_chaining(engine, oracle):
    cfg = T.kitti_config()
    cfg.use_motion_model = 1
    prev, curr, Tgt, cam = synth.make_batch("kitti", 2, n_pt=500, n_ls=120)
    pri = T.identity_priors(2)
    for p in range(2):
        pri["Tfw"][p] = R.expmap_se3([1.0, 2.0, 3.0, 0.1, -0.2, 0.05 * p])
        pri["Tfw_cov"][p] = np.eye(6) * 0.01
        pri["DT"][p] = Tgt[p]
        pri["DT_cov"][p] = np.eye(6) * 1e-6
        pri["err_norm"][p] = 0.2
    compare(engine.track_batch(cam, cfg, prev, curr, priors=pri),
            oracle.track_batch(cam, cfg, prev, curr, priors=pri), prev)


def test_line_level_sigma_rule(engine, oracle):
    cfg = T.kitti_config()
    prev, curr, _, cam = synth.make_batch("kitti", 2, n_pt=300, n_ls=100, overlap=1.0)
    prev.ls_level[:] = np.arange(prev.n_ls) % 3
    prev.ls_sigma2[:] = 1.0 / (1.2 ** prev.ls_level) ** 2
    compare(engine.track_batch(cam, cfg, prev, curr), oracle.track_batch(cam, cfg, prev, curr), prev)


def test_resident_batch_equals_host_call_and_is_deterministic(engine):
    cfg = T.kitti_config()
    prev, curr, _, cam = synth.make_batch("kitti", 6, n_pt=600, n_ls=150)
    a = engine.track_batch(cam, cfg, prev, curr)
    db = engine.upload(cam, cfg, prev, curr)
    db.run()
    b = db.download()
    db.run()
    c = db.download()
    db.free()
    for k in ("m12_pt", "m12_ls", "inlier_pt", "inlier_ls"):
        np.testing.assert_array_equal(a[k], b[k])
        np.testing.assert_array_equal(b[k], c[k])
    assert a["results"].tobytes() == b["results"].tobytes() == c["results"].tobytes()   # bit-identical reruns


def test_pose_golden_vectors(engine):
    for shape, cfgf in (("kitti", T.kitti_config), ("euroc", T.euroc_config)):
        g = np.load(os.path.join(GOLDEN, f"pose_{shape}.npz"))
        prev, curr, _, cam = synth.make_batch(shape, int(g["B"]), n_pt=int(g["n_pt"]), n_ls=int(g["n_ls"]))
        gpu = engine.track_batch(cam, cfgf(), prev, curr)
        np.testing.assert_array_equal(gpu["m12_pt"], g["m12_pt"])
        np.testing.assert_array_equal(gpu["m12_ls"], g["m12_ls"])
        np.testing.assert_array_equal(gpu["inlier_pt"], g["oracle_inlier_pt"])
        np.testing.assert_array_equal(gpu["inlier_ls"], g["oracle_inlier_ls"])
        for p in range(prev.B):
            for key in ("oracle_DT", "numpy_DT"):
                ang, tr = R.pose_error(gpu["results"]["DT"][p], g[key][p])
                assert ang < TIGHT_ANG and tr < TIGHT_TR


def _flag_diffs(a, b):
    return int((np.asarray(a) != np.asarray(b)).sum())


def test_large_frames_take_the_streamed_solver(engine, oracle):
    """C5 shape (8000 + 2000) does not fit K2's shared-memory feature store: optimizePose runs as HBM-bound evaluation sweeps
    (fp32 per-feature arithmetic, fp64 sums / 6x6 algebra / outlier residuals) with a per-problem step kernel in between.
    Match indices stay bit-exact; the pose is held to north_star's tolerance (1e-5 rad / 1e-4 m); inlier flags may differ
    only for residuals within fp32 reach of the threshold (count reported)."""
    cfg = T.kitti_config()
    prev, curr, _, cam = synth.make_batch("hd", 2)
    gpu, ref = engine.track_batch(cam, cfg, prev, curr), oracle.track_batch(cam, cfg, prev, curr)
    worst = compare(gpu, ref, prev, tight=False, flags_exact=False)
    n_diff = _flag_diffs(gpu["inlier_pt"], ref["inlier_pt"]) + _flag_diffs(gpu["inlier_ls"], ref["inlier_ls"])
    print(f"streamed solver, C5 shape: worst pose deviation {worst}, {n_diff} of {prev.n_pt + prev.n_ls} inlier flags differ")
    assert n_diff <= 4
    assert worst[0] < 1e-7 and worst[1] < 1e-6      # measured 2.3e-10 / 6e-9 (delta-form residuals): far inside the 1e-5 / 1e-4 bar


def test_batch_of_64_pairs_sharded_invariance(engine, oracle):
    """A batch processed in one call equals the same pairs processed as two half batches (what two ranks do)."""
    cfg = T.kitti_config()
    prev, curr, _, cam = synth.make_batch("kitti", 8, n_pt=500, n_ls=120)
    full = engine.track_batch(cam, cfg, prev, curr)
    lo = engine.track_batch(cam, cfg, prev.select(range(0, 4)), curr.select(range(0, 4)))
    hi = engine.track_batch(cam, cfg, prev.select(range(4, 8)), curr.select(range(4, 8)))
    assert full["results"].tobytes() == lo["results"].tobytes() + hi["results"].tobytes()
    np.testing.assert_array_equal(full["m12_pt"], np.concatenate([lo["m12_pt"], hi["m12_pt"]]))


def test_gn_eval_stream_vs_oracle(engine, oracle):
    """optimizeFunctions streamed from HBM (the C5 roofline kernel: fp32-packed records, fp32 per-feature math, fp64
    reduction) against the oracle's double evaluation: agreement at the fp32 level (1e-4 relative on H, g, e), and the
    Gauss-Newton step computed from it within the 1e-5 rad / 1e-4 m bar."""
    cfg = T.kitti_config()
    prev, curr, Tgt, cam = synth.make_batch("kitti", 3, n_pt=900, n_ls=250)
    o = oracle.track_batch(cam, cfg, prev, curr)
    matched = T.matched_from_frames(prev, curr, o["m12_pt"], o["m12_ls"], cfg.lsd_scale)
    DT = np.stack([np.eye(4), Tgt[1], o["results"]["DT_opt"][2]])
    H, g, e, ms = engine.gn_eval_stream(cam, cfg, matched, DT, iters=2)
    for p in range(3):
        Hr, gr, er = oracle.optimize_functions(cam, cfg, matched, p, DT[p])
        np.testing.assert_allclose(H[p], Hr, rtol=2e-4, atol=2e-5 * np.abs(Hr).max())
        # g = sum J r w cancels almost completely near the optimum: bound the error by the Cauchy-Schwarz scale
        # |g_i| <= sqrt(H_ii * sum r^2 w) instead of by |g_i| itself
        n_feat = (matched.pt_off[p + 1] - matched.pt_off[p]) + (matched.ls_off[p + 1] - matched.ls_off[p])
        scale = np.sqrt(np.diag(Hr) * er * n_feat)
        assert (np.abs(g[p] - gr) < 2e-4 * scale).all(), (g[p], gr, scale)
        assert abs(e[p] - er) < 1e-5
        inc, inc_r = np.linalg.solve(H[p], g[p]), np.linalg.solve(Hr, gr)
        assert np.linalg.norm(inc[:3] - inc_r[:3]) < 1e-4 and np.linalg.norm(inc[3:] - inc_r[3:]) < 1e-5
    assert ms > 0
    # ragged / tiny problems and explicit outlier flags
    mb, Ts, cam2 = synth.make_matched_batch("kitti", 2)
    mb.pt_inlier = (np.arange(len(mb.pt_sigma2)) % 7 != 0).astype(np.uint8)
    mb.ls_inlier = (np.arange(len(mb.ls_sigma2)) % 5 != 0).astype(np.uint8)
    H, g, e, _ = engine.gn_eval_stream(cam2, cfg, mb, Ts, iters=1)
    for p in range(2):
        Hr, gr, er = oracle.optimize_functions(cam2, cfg, mb, p, Ts[p])
        np.testing.assert_allclose(H[p], Hr, rtol=2e-4, atol=2e-5 * np.abs(Hr).max())
        assert abs(e[p] - er) < 1e-5


def _ragged(mb, keep_pt, keep_ls):
    """First keep_pt[p] points / keep_ls[p] lines of every problem of an equal-sized MatchedBatch."""
    ip = np.concatenate([np.arange(mb.pt_off[p], mb.pt_off[p] + k) for p, k in enumerate(keep_pt)]).astype(np.int64)
    il = np.concatenate([np.arange(mb.ls_off[p], mb.ls_off[p] + k) for p, k in enumerate(keep_ls)]).astype(np.int64)
    return T.MatchedBatch(pt_off=np.concatenate([[0], np.cumsum(keep_pt)]), ls_off=np.concatenate([[0], np.cumsum(keep_ls)]),
                          pt_P=mb.pt_P[ip], pt_pl_obs=mb.pt_pl_obs[ip], pt_sigma2=mb.pt_sigma2[ip], ls_sP=mb.ls_sP[il],
                          ls_eP=mb.ls_eP[il], ls_le_obs=mb.ls_le_obs[il], ls_spl=mb.ls_spl[il], ls_epl=mb.ls_epl[il],
                          ls_sigma2=mb.ls_sigma2[il])


def _check_stream(engine, oracle, cam, cfg, mb, Ts, probs):
    H, g, e, _ = engine.gn_eval_stream(cam, cfg, mb, Ts, iters=1)
    for p in probs:
        Hr, gr, er = oracle.optimize_functions(cam, cfg, mb, p, Ts[p])
        n_feat = (mb.pt_off[p + 1] - mb.pt_off[p]) + (mb.ls_off[p + 1] - mb.ls_off[p])
        # fp32 level: a residual of ~0.5 px is the difference of two ~1000 px values (ulp 6e-5 px), i.e. 1e-4 .. 1e-3 relative
        # per feature; it averages out over a list, so short lists get the per-feature bound
        tol = 2e-4 if n_feat >= 1000 else 5e-3
        np.testing.assert_allclose(H[p], Hr, rtol=tol, atol=0.1 * tol * np.abs(Hr).max(), err_msg=f"problem {p}")
        scale = np.sqrt(np.diag(Hr) * er * n_feat)
        assert (np.abs(g[p] - gr) < tol * scale + 1e-12).all(), (p, g[p], gr)
        assert abs(e[p] - er) < (1e-5 if n_feat >= 1000 else 1e-4) * max(1.0, er), (p, e[p], er)


def test_gn_eval_stream_tiles_and_slices(engine, oracle):
    """The streamed evaluator's tiling: partial 16 KB tiles (512 points / 256 lines), problems without lines, a single point,
    large problems cut into several slices, sigma2 != 1, and more work items than persistent CTAs (the ring of stages runs
    on across item boundaries)."""
    cfg = T.kitti_config()
    mb, Ts, cam = synth.make_matched_batch("hd", 8)                       # 8000 + 2000 per problem
    rng = np.random.default_rng(3)
    mb.pt_sigma2 = 1.0 / 1.2 ** (2 * rng.integers(0, 8, len(mb.pt_sigma2)))   # pyramid levels 0..7
    mb.ls_sigma2 = 1.0 / 1.2 ** (2 * rng.integers(0, 2, len(mb.ls_sigma2)))
    rg = _ragged(mb, [8000, 512, 513, 1, 7999, 1024, 300, 4097], [2000, 0, 256, 1, 257, 1999, 5, 511])
    _check_stream(engine, oracle, cam, cfg, rg, Ts, range(8))
    many, Tm, cam2 = synth.make_matched_batch("kitti", 700)               # 700 items on 2 x 148 CTAs
    many.pt_inlier = (np.arange(len(many.pt_sigma2)) % 11 != 0).astype(np.uint8)
    _check_stream(engine, oracle, cam2, cfg, many, Tm, [0, 1, 295, 296, 297, 591, 592, 698, 699])


def test_onchip_6x6_algebra(engine, oracle):
    """The warp-level 6x6 routines of K2 (lanes-as-columns Householder QR, LU inverse, parallel-order Jacobi)
    against numpy and the oracle's restatements."""
    rng = np.random.default_rng(42)
    Hs, gs = [], []
    for k in range(64):
        J = rng.normal(0, 1, (40, 6)) * np.array([1, 1, 1, 30, 30, 30]) ** (k % 3)
        Hs.append(J.T @ J)
        gs.append(rng.normal(0, 1, 6))
    Hs.append(np.diag([1.0, 2.0, 3.0, 0.0, 0.0, 0.0]))     # rank deficient: truncated solve, like Eigen
    gs.append(np.ones(6))
    Hs.append(np.eye(6))
    gs.append(np.arange(6.0))
    H, g = np.stack(Hs), np.stack(gs)
    x, lad, inv, eig = engine.debug_algebra(H, g)
    for k in range(64):
        np.testing.assert_allclose(x[k], np.linalg.solve(H[k], g[k]), rtol=1e-9, atol=1e-12)
        assert abs(lad[k] - np.linalg.slogdet(H[k])[1]) < 1e-9
        np.testing.assert_allclose(inv[k], np.linalg.inv(H[k]), rtol=1e-8, atol=1e-14)
        np.testing.assert_allclose(eig[k], np.linalg.eigvalsh(H[k], UPLO="L"), rtol=1e-9, atol=1e-12 * eig[k].max())
    xo, lado, rank = oracle.qr6_solve(H[64], g[64])
    np.testing.assert_allclose(x[64], xo, atol=1e-12)
    np.testing.assert_allclose(x[65], g[65], atol=1e-14)
    np.testing.assert_allclose(eig[65], np.ones(6), atol=1e-14)


def test_block_radix_selection(engine):
    """The radix selection behind the streamed solver's median / MAD (solve.cu: block_select_wide) against numpy's sort, bit for
    bit, on lists that stress it: every length from 1 up, heavy ties, all-equal lists, values straddling zero, sub-normals,
    infinities, huge dynamic range (many digits under the common prefix), clustered values (many candidates in one bin), and
    residual-like positive data at KITTI and C5 list lengths; every rank k for the short lists, median-type ranks for the long."""
    rng = np.random.default_rng(7)
    lists, ks = [], []

    def add(x, k):
        lists.append(np.asarray(x, np.float64))
        ks.append(int(k))

    for n in list(range(1, 40)) + [63, 64, 65, 255, 256, 257, 511, 513]:
        x = rng.normal(0, 3, n)
        for k in sorted({0, n // 2, n - 1, int(rng.integers(0, n))}):
            add(x, k)
    for n in (300, 2000, 8000, 9000):
        res = np.abs(rng.standard_cauchy(n)) * rng.choice([0.3, 1.0, 40.0], n)           # residual-like, heavy tail
        add(res, n // 2)
        add(res, n // 2 - 1)
        add(np.round(res, 1), n // 2)                                                    # heavy ties
        add(np.full(n, 3.25), n // 2)                                                    # all equal
        add(np.concatenate([np.full(n // 2, 1.0), np.full(n - n // 2, 1.0 + 2.0 ** -52)]), n // 2)   # two values one ulp apart
        add(1.0 + rng.integers(0, 300, n) * 2.0 ** -50, n // 3)                          # > 256 candidates under one 11-bit digit
        add(rng.normal(0, 1, n) * 10.0 ** rng.integers(-300, 300, n), n // 2)            # full exponent range, both signs
        add(np.concatenate([rng.normal(0, 1, n - 7), [np.inf] * 4, [-np.inf] * 3]), n // 2)
        add(np.concatenate([rng.normal(0, 1e-310, n // 2), rng.normal(0, 1, n - n // 2)]), n // 4)   # sub-normals
    got = engine.debug_select(lists, ks)
    for x, k, g in zip(lists, ks, got):
        want = np.sort(x)[k]
        assert g == want or (np.isnan(g) and np.isnan(want)), (len(x), k, g, want)
    # the MAD form: k-th smallest of |x - median| rounded to float (src/auxiliar.cpp:399-402)
    ml, mk, mp = [], [], []
    for n in (5, 33, 500, 2000, 8000):
        for scale in (1.0, 1e-3, 250.0):
            x = np.abs(rng.standard_cauchy(n)) * scale
            med = np.sort(x)[n // 2]
            ml.append(x); mk.append(n // 2); mp.append(med)
    got = engine.debug_select(ml, mk, pivots=mp)
    for x, k, piv, g in zip(ml, mk, mp, got):
        dev = np.abs((x - piv).astype(np.float32)).astype(np.float64)
        assert g == np.sort(dev)[k], (len(x), k, g)


def test_handler_mirror_sequence(engine, oracle):
    """app/imagesStVO.cpp:88-124 call sequence through the Python mirror of StereoFrameHandler: a 4-frame sequence,
    poses chained through Tfw, against the oracle run pair by pair with the same priors."""
    from stvo_pl_b200.handler import StereoFrameHandler
    from stvo_pl_b200 import matching
    cfg = T.kitti_config()
    cam = T.kitti_camera()
    frames = []
    for k in range(3):
        prev, curr, _, _ = synth.make_batch("kitti", 1, first_pair=50 + k, n_pt=500, n_ls=120)
        frames.append((prev, curr))
    h = StereoFrameHandler(cam, cfg, engine)
    h.initialize(frames[0][0])
    pri = T.identity_priors(1)
    for k, (prev, curr) in enumerate(frames):
        h.prev_frame.features = prev          # synthetic pairs are independent: swap in the pair's prev features
        h.insertStereoPair(curr, k + 1)
        h.optimizePose()
        ref = oracle.track_batch(cam, cfg, prev, curr, priors=pri)
        r = ref["results"][0]
        ang, tr = R.pose_error(h.curr_frame.DT, r["DT"])
        assert ang < TIGHT_ANG and tr < TIGHT_TR
        np.testing.assert_allclose(h.curr_frame.Tfw, r["Tfw"], atol=1e-8)
        assert h.n_inliers_pt == r["n_inliers_pt"] and len(h.matched_pt) == r["n_matched_pt"]
        pri["Tfw"][0], pri["Tfw_cov"][0] = r["Tfw"], r["Tfw_cov"]
        pri["DT"][0], pri["DT_cov"][0], pri["err_norm"][0] = r["DT"], r["DT_cov"], r["err_norm"]
        h.updateFrame()
    n, m = matching.match(frames[0][0].pdesc, frames[0][1].pdesc, 0.75, True, engine)
    np.testing.assert_array_equal(m, oracle.match(frames[0][0].pdesc, frames[0][1].pdesc, 0.75)[1])
    with pytest.raises(RuntimeError):
        matching.matchNNR(np.zeros((3, 16), np.uint8), np.zeros((3, 32), np.uint8), 0.9, engine)


def test_async_streaming_equals_blocking_call(engine):
    """plstvo_track_batch_async / plstvo_wait with two batches in flight give the blocking call's bytes."""
    cfg = T.kitti_config()
    batches = [synth.make_batch("kitti", 5, first_pair=10 * k, n_pt=400 + 50 * k, n_ls=100)[:2] for k in range(4)]
    cam = T.kitti_camera()
    ref = [engine.track_batch(cam, cfg, p, c) for p, c in batches]
    pinned = [(engine.pinned.pin_frames(p), engine.pinned.pin_frames(c), engine.pinned_outputs(p)) for p, c in batches]
    pending = None
    for k, (p, c, o) in enumerate(pinned):
        t = engine.track_batch_async(cam, cfg, p, c, o)
        if pending is not None:
            engine.wait(pending)
        pending = t
    engine.wait(pending)
    for k in range(4):
        for key in ("m12_pt", "m12_ls", "inlier_pt", "inlier_ls"):
            np.testing.assert_array_equal(pinned[k][2][key], ref[k][key])
        assert pinned[k][2]["results"].tobytes() == ref[k]["results"].tobytes()


def test_explicit_lists_c5_size(engine, oracle, ref):
    """C5-size explicit lists (8000 + 2000 per problem) through plstvo_optimize_pose: the streamed solver against the oracle
    and against the reference's compiled code."""
    cfg = T.kitti_config()
    mb, Ts, cam = synth.make_matched_batch("hd", 3)
    rc, res_o, rp, rl = oracle.optimize_pose(cam, cfg, mb)
    res, ip, il = engine.optimize_pose(cam, cfg, mb)
    for p in range(3):
        assert res["status"][p] == res_o["status"][p] and res["good"][p] == res_o["good"][p] == 1
        ang, tr = R.pose_error(res["DT"][p], res_o["DT"][p])
        assert ang < TOL_ANG and tr < TOL_TR
        a, b, c, d = mb.pt_off[p], mb.pt_off[p + 1], mb.ls_off[p], mb.ls_off[p + 1]
        flips = _flag_diffs(ip[a:b], rp[a:b]) + _flag_diffs(il[c:d], rl[c:d])
        # same inlier set: the error agrees to the fp32 evaluation's noise; a flag that flipped (a residual within fp32 reach of the
        # removeOutliers threshold) moves it by about one feature's share
        assert abs(res["err_norm"][p] - res_o["err_norm"][p]) < (1e-6 if flips == 0 else 2e-4 * flips)
        np.testing.assert_allclose(res["DT_cov"][p], res_o["DT_cov"][p], rtol=2e-3, atol=1e-12)
        ang, tr = R.pose_error(res["DT_opt"][p], Ts[p])
        assert ang < 1e-3 and tr < 1e-2
    n_diff = _flag_diffs(ip, rp) + _flag_diffs(il, rl)
    print(f"streamed solver, explicit C5 lists: {n_diff} of {len(ip) + len(il)} inlier flags differ")
    assert n_diff <= 6
    rr = ref.optimize_pose(cam, cfg, mb)[1]
    for p in range(3):
        ang, tr = R.pose_error(res["DT"][p], rr["DT"][p])
        assert ang < TOL_ANG and tr < TOL_TR


def test_streamed_solver_is_bit_reproducible(engine):
    """The streamed solver on lists longer than its TMA ring (24 record tiles per problem through 6 stages: every stage is reused
    four times per iteration) gives identical bytes run after run: fixed summation order, and no stage is overwritten before its
    readers are done (a race there would show up as run-to-run differences)."""
    cfg = T.kitti_config()
    mb, Ts, cam = synth.make_matched_batch("hd", 6)
    first = None
    for _ in range(4):
        res, ip, il = engine.optimize_pose(cam, cfg, mb)
        blob = res.tobytes() + ip.tobytes() + il.tobytes()
        if first is None:
            first = blob
        assert blob == first


def test_two_contexts_on_two_devices_in_one_process(oracle):
    """One context per GPU inside a single process (device arenas and kernel attributes are per context / per device):
    the same batch through both devices, interleaved, gives identical bytes.  Skipped on single-GPU boxes."""
    import torch
    from stvo_pl_b200.engine import Engine
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cfg = T.kitti_config()
    prev, curr, _, cam = synth.make_batch("kitti", 6, n_pt=900, n_ls=220)
    e0, e1 = Engine(0), Engine(1)
    try:
        a = e0.track_batch(cam, cfg, prev, curr)
        b = e1.track_batch(cam, cfg, prev, curr)
        a2 = e0.track_batch(cam, cfg, prev, curr)
        assert a["results"].tobytes() == b["results"].tobytes() == a2["results"].tobytes()
        mb, Ts, cam2 = synth.make_matched_batch("kitti", 40)
        H0, g0, _, _ = e0.gn_eval_stream(cam2, cfg, mb, Ts, iters=1)
        H1, g1, _, _ = e1.gn_eval_stream(cam2, cfg, mb, Ts, iters=1)
        assert H0.tobytes() == H1.tobytes() and g0.tobytes() == g1.tobytes()
        q_cell, d1, t_cell, d2 = __import__("stvo_pl_b200.stereo_synth", fromlist=["x"]).make_stereo_points(500, 480, seed=1)
        w = T.PlGridWindow(10, 0, 0, 0)
        m0 = e0.match_grid_points([0, 500], q_cell, d1, [0, 480], t_cell, d2, w, 0.75)[1]
        m1 = e1.match_grid_points([0, 500], q_cell, d1, [0, 480], t_cell, d2, w, 0.75)[1]
        np.testing.assert_array_equal(m0, m1)
    finally:
        e0.close()
        e1.close()
