"""The oracle restatement against THE REFERENCE'S OWN CODE.

oracle/_ref/libellc_ref.so is the reference's unmodified src/Frame.cpp, PixelWisePyramid.cpp, Pyramid.cpp, UserDefinedFunc.cpp
and ImageFunc.cpp, compiled where they lie under /root/reference against the stand-in OpenCV / Eigen / Boost headers of
oracle/shim/ (oracle/ref_driver.cpp, `make -C oracle ref`).  tests/golden/reference_track_480x270.npz holds what that library
produced on seeded inputs at the reference's compiled-in configuration (generator: tests/golden/make_reference_golden.py).

  * fixture tests run everywhere (the fixture is committed);
  * the tests that take `R` call the reference through it: where the library exists or can be built, R is the library and every
    call is also checked against tests/golden/reference_live_calls.npz; elsewhere R returns what that file recorded for the
    call (generator: tests/golden/make_reference_live_golden.py), so the oracle is compared with the reference's outputs
    everywhere.
"""
import os
import sys

import numpy as np
import pytest

from oracle import refbinding as ref

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLD)
from make_reference_live_golden import Replay, same  # noqa: E402


@pytest.fixture
def R(request):
    """The reference's binding for this test: live where the library is available, its recorded results elsewhere."""
    variant = "640x480" if "640x480" in request.node.name else "default"
    return Replay(request.node.name, live=ref if ref.available(variant) else None)


@pytest.fixture(scope="module")
def fx():
    return np.load(os.path.join(GOLD, "reference_track_480x270.npz"))


def _ocfg(oracle_mod, g, **over):
    fxv, fyv, cx, cy = (float(v) for v in g["intr"])
    return oracle_mod.default_config(int(g["width"][0]), int(g["height"][0]), fx=fxv, fy=fyv, cx=cx, cy=cy, **over)


def _depth(g):
    return [g[f"depth{l}"] for l in range(4)], [g[f"var{l}"] for l in range(4)]


def test_oracle_is_bit_identical_to_the_reference_trace(oracle_mod, fx):
    """Every iteration of every level: hessian, sd_param, weightedPose and the updated pose of the reference's
    PixelWisePyramid object (src/PixelWisePyramid.h:38-107) are BIT-IDENTICAL to the oracle's; so are the selected-pixel
    counts, the iteration counts (early-out, src/ImageFunc.cpp:251-252) and the final pose.  480x270 is not divisible by 8,
    so the reference's `height/2^L` vs pyrDown `(h+1)/2` quirk (src/Frame.cpp:110-112, :321-322) is exercised."""
    g = fx
    ocfg = _ocfg(oracle_mod, g)
    depth, var = _depth(g)
    n_pairs = len(g["frames"])
    total_iters = 0
    for i in range(n_pairs):
        pose, tr = oracle_mod.track(ocfg, g["kf_image"], g["frames"][i], depth, var, g["init"][i])
        assert tr["n_selected"] == list(g[f"p{i}_n_selected"])
        assert tr["n_iters"] == list(g[f"p{i}_n_iters"])
        assert np.array_equal(pose, g[f"p{i}_pose"])
        for l in range(4):
            its = tr["levels"][l]
            assert np.array_equal(np.stack([it["H"] for it in its]).reshape(-1, 6, 6), g[f"p{i}_H_{l}"]), (i, l)
            assert np.array_equal(np.stack([it["b"] for it in its]), g[f"p{i}_b_{l}"]), (i, l)
            assert np.array_equal(np.array([it["weighted_pose"] for it in its], np.float32), g[f"p{i}_wp_{l}"]), (i, l)
            assert np.array_equal(np.stack([it["pose_after"] for it in its]), g[f"p{i}_pose_{l}"]), (i, l)
            total_iters += len(its)
    assert total_iters >= 40                                      # the large-rotation pair runs many iterations
    assert np.abs(g["p0_pose"] - g["gt"][0]).max() < 2e-3         # and the reference does track the synthetic scene


def test_oracle_weight_image_is_bit_identical_to_the_reference(oracle_mod, fx):
    """display_weightimg of the last executed level-0 iteration (src/PixelWisePyramid.cpp:334-361): per-pixel Huber x
    variance weights, 0 for unselected and out-of-bounds pixels."""
    g = fx
    ocfg = _ocfg(oracle_mod, g)
    depth, var = _depth(g)
    kpyr = oracle_mod.image_pyramid(g["kf_image"])
    for i in range(len(g["frames"])):
        poses0 = g[f"p{i}_pose_0"]
        before = poses0[-2] if len(poses0) > 1 else g[f"p{i}_pose_1"][-1]          # pose the last level-0 iteration started from
        cpyr = oracle_mod.image_pyramid(g["frames"][i])
        o = oracle_mod.gn_evaluate(ocfg, 0, kpyr[0], cpyr[0], depth[0], var[0], before, want_weights=True)
        assert np.array_equal(o["weights"], g[f"p{i}_weights_l0"]), i
        assert np.array_equal(np.asarray(o["H"], np.float32).reshape(6, 6), g[f"p{i}_H_0"][-1]), i


def test_oracle_matches_the_reference_driver(oracle_mod, fx):
    """GetImagePoseEstimate itself (src/ImageFunc.cpp:49-315): initial pose = log(exp(t-1 world pose) exp(keyframe world
    pose)^-1) (:97-108), result, and the poseWrtOrigin / poseWrtWorld post-conditions (:305-307)."""
    g = fx
    ocfg = _ocfg(oracle_mod, g)
    depth, var = _depth(g)
    zero = np.zeros(6, np.float32)
    for i in range(len(g["frames"])):
        init = oracle_mod.concat_origin(g["init"][i], zero)
        pose, _ = oracle_mod.track(ocfg, g["kf_image"], g["frames"][i], depth, var, init, want_trace=False)
        assert np.array_equal(pose, g[f"p{i}_driver_pose"]), i
        assert np.array_equal(oracle_mod.concat_relative(pose, zero), g[f"p{i}_driver_pose_wrt_origin"]), i
        assert np.array_equal(oracle_mod.concat_relative(pose, zero), g[f"p{i}_driver_pose_wrt_world"]), i


def _oracle_lc_weights(oracle_mod, g, ocfg):
    depth, var = _depth(g)
    h, w = int(g["height"][0]), int(g["width"][0])
    wp = [np.zeros((h >> l, w >> l), np.float32) for l in range(4)]
    cnt = [0] * 4
    zero = np.zeros(6, np.float32)
    poses = []
    for i in range(len(g["frames"])):
        pose, _, wl = oracle_mod.track_with_weights(ocfg, g["kf_image"], g["frames"][i], depth, var, oracle_mod.concat_origin(g["init"][i], zero))
        oracle_mod.accumulate_weights(wp, cnt, wl)
        poses.append(pose)
    return oracle_mod.finalise_weights(wp, cnt), cnt, np.stack(poses)


def test_oracle_loop_closure_flow_is_bit_identical_to_the_reference(oracle_mod, fx):
    """SURVEY 8a row M with the reference's own driver: saveWeights(true) during the sequential tracks
    (src/ImageFunc.cpp:280-288), frame::finaliseWeights (src/Frame.cpp:678-695), then the constant-weight inverse-compositional
    tracker (src/PixelWisePyramid.cpp:561-974): precomputed hessian, sd_param, weightedPose and pose of every iteration."""
    g = fx
    ocfg = _ocfg(oracle_mod, g, lc_parallel=1)
    depth, _ = _depth(g)
    wf, cnt, seq_poses = _oracle_lc_weights(oracle_mod, g, ocfg)
    assert cnt == list(g["lc_counts"]) and np.array_equal(seq_poses, g["lc_seq_poses"])
    assert np.array_equal(np.array([float(w.astype(np.float64).sum()) for w in wf]), g["lc_weight_sums"])
    init = oracle_mod.concat_origin(g["lc_tminus1"], np.zeros(6, np.float32))
    pose, tr = oracle_mod.track_lc(ocfg, g["kf_image"], g["frames"][2], depth, wf, init)
    assert tr["n_iters"] == list(g["lc_n_iters"]) and np.array_equal(pose, g["lc_pose"])
    for l in range(4):
        its = tr["levels"][l]
        assert np.array_equal(np.stack([it["H"] for it in its]).reshape(-1, 6, 6), g[f"lc_H_{l}"]), l
        assert np.array_equal(np.stack([it["b"] for it in its]), g[f"lc_b_{l}"]), l
        assert np.array_equal(np.array([it["weighted_pose"] for it in its], np.float32), g[f"lc_wp_{l}"]), l
        assert np.array_equal(np.stack([it["pose_after"] for it in its]), g[f"lc_pose_{l}"]), l


def test_oracle_depth_pyramids_and_gating_are_bit_identical_to_the_reference(oracle_mod, fx):
    """SURVEY 8f rows 2 and 3 against the reference's own src/DepthPropagation.cpp (updateDepthImage :1254-1315, buildInvVarDepth
    :1637-1719, mapDepthArr2Mat, calculate_no_of_Seeds :1804-1830) and src/GlobalOptimize.cpp (calculateImageHistogram :40-100,
    compareImageHistogram :116-122, calculateRotationStats :419-452).  The reference's depth / variance pyramids are stored as
    SHA-256 digests: equal digests = bit-identical arrays (incl. inf depths from zero inverse depths and the NaN view angle of
    identical poses)."""
    import sys
    sys.path.insert(0, GOLD)
    from make_reference_golden import digest, hypotheses_case
    g = fx
    valid, idep, var = hypotheses_case(int(g["height"][0]), int(g["width"][0]))
    o = oracle_mod.update_depth_image(valid, idep, var)
    assert np.float32(o["occupancy"]) == g["hyp_occupancy"][0]
    assert digest(o["valid_out"]) == str(g["hyp_valid_sha"])
    assert [digest(a) for a in o["depth"]] == list(g["hyp_depth_sha"])
    assert [digest(a) for a in o["var"]] == list(g["hyp_var_sha"])
    n = len(g["frames"])
    hists = [oracle_mod.image_histogram(g["frames"][i]) for i in range(n)]
    assert np.array_equal(np.stack(hists), g["gate_hist"])
    for i in range(n):
        for j in range(n):
            assert oracle_mod.hist_kl_div(hists[i], hists[j]) == g["gate_kl"][i, j]
            rms, ang = oracle_mod.rotation_stats(g["gt"][i], g["gt"][j])
            assert np.float32(rms) == g["gate_rms"][i, j]
            assert np.array_equal(np.float32(ang), g["gate_angle"][i, j], equal_nan=True)


def test_oracle_pyramid_cpp_variant_is_bit_identical_to_the_reference(oracle_mod, fx):
    """SURVEY 8a row L: the oracle's `jacobian_at_warped` variant against the reference's matrix-form src/Pyramid.cpp
    (calculateSteepestDescent :43-148 at the warped pixel and Z', calResidualAndWeights :558-694 with the weight of an
    out-of-bounds pixel not zeroed, calculateHessianInv :153-207, updatePose :528-553): per-pixel weights, hessianInv and the
    updated pose bit-identical; sum w r^2 / n within the float rounding of the reference's own division."""
    import sys
    sys.path.insert(0, GOLD)
    from make_reference_golden import digest
    g = fx
    ocfg = _ocfg(oracle_mod, g, jacobian_at_warped=1)
    depth, var = _depth(g)
    kpyr = oracle_mod.image_pyramid(g["kf_image"])
    for c, (fi, level) in enumerate(g["pyr_frame_level"]):
        pose = g["pyr_pose_in"][c]
        cpyr = oracle_mod.image_pyramid(g["frames"][fi])
        o = oracle_mod.gn_evaluate(ocfg, int(level), kpyr[level], cpyr[level], depth[level], var[level], pose, want_weights=True)
        sel = depth[level] > 0
        assert int(sel.sum()) == int(g["pyr_n"][c])
        assert digest(o["weights"][sel]) == str(g["pyr_weights_sha"][c]), c
        assert abs(o["res_sum_f32"] / g["pyr_n"][c] - g["pyr_last_err"][c]) <= 2e-6 * g["pyr_last_err"][c], c
        Hinv, ok = oracle_mod.invert6(o["H"])
        assert ok and np.array_equal(Hinv, g["pyr_hessian_inv"][c]), c
        pose_after, _, _ = oracle_mod.update_pose(ocfg, Hinv, o["b"], pose)
        assert np.array_equal(pose_after, g["pyr_poses_after"][c][0]), c


# ---- the library itself, or what it returned (R) ---------------------------------------------------------------------------
def test_fixture_is_what_the_reference_produces(fx, R):
    g = fx
    depth, var = _depth(g)
    k = R.dims()
    assert (k["width"], k["height"]) == (int(g["width"][0]), int(g["height"][0]))
    assert np.array_equal(np.array([k["fx"], k["fy"], k["cx"], k["cy"]], np.float32), g["intr"])
    tr = R.track_trace(g["kf_image"], g["frames"][1], depth, var, g["init"][1], want_weights=True)
    assert tr["n_iters"] == list(g["p1_n_iters"]) and np.array_equal(tr["final_pose"], g["p1_pose"])
    assert same(tr["weights_l0"], g["p1_weights_l0"])
    pose, po, pw = R.get_image_pose_estimate(g["kf_image"], g["frames"][1], depth, var, g["init"][1])
    assert np.array_equal(pose, g["p1_driver_pose"]) and np.array_equal(po, g["p1_driver_pose_wrt_origin"])


def test_reference_stages_vs_oracle(oracle_mod, fx, R):
    """constructImagePyramids / calculateGradient / calculateNonZeroDepthPts (src/Frame.cpp:170-327) on every level, incl. NaN,
    negative and -0 depths."""
    g = fx
    depth, _ = _depth(g)
    opyr = oracle_mod.image_pyramid(g["frames"][0])
    rng = np.random.default_rng(3)
    for l in range(4):
        d = depth[l].copy()
        idx = rng.integers(0, d.size, 40)
        d.reshape(-1)[idx[:10]] = np.nan; d.reshape(-1)[idx[10:20]] = -1.0; d.reshape(-1)[idx[20:30]] = -0.0; d.reshape(-1)[idx[30:]] = np.inf
        r = R.frame_level(g["frames"][0], l, d)
        assert same(r["image"], opyr[l]), l
        rows, cols = d.shape
        ogx, ogy = oracle_mod.gradient(opyr[l], rows, cols)
        assert same(r["gradx"], ogx) and same(r["grady"], ogy), l
        omask, ocount = oracle_mod.mask_count(d)
        assert same(r["mask"], omask) and r["count"] == ocount, l


def test_reference_samplers_vs_oracle(oracle_mod, fx, R):
    """frame::getInterpolatedElement (src/Frame.h:181-394) at random, integer, border and out-of-bounds coordinates."""
    g = fx
    img = g["frames"][0]
    rng = np.random.default_rng(9)
    for l in (0, 2, 3):
        rows, cols = img.shape[0] >> l, img.shape[1] >> l
        xs = np.concatenate([rng.uniform(-3, cols + 3, 400), rng.integers(-2, cols + 2, 100).astype(np.float64),
                             [0, cols - 1, cols - 1 + 1e-4, cols - 0.5, -1e-6, -0.5, cols, 0.5]]).astype(np.float32)
        ys = np.concatenate([rng.uniform(-3, rows + 3, 400), rng.integers(-2, rows + 2, 100).astype(np.float64),
                             [0, rows - 1, rows - 1 + 1e-4, rows - 0.5, -1e-6, 2.0, 3.0, rows]]).astype(np.float32)
        ri, rgx, rgy = R.interpolate(img, l, xs, ys)
        lvl = oracle_mod.image_pyramid(img)[l]
        ogx, ogy = oracle_mod.gradient(lvl, rows, cols)
        oi = np.array([oracle_mod.interp_u8(lvl, x, y, 1, rows, cols) for x, y in zip(xs, ys)], np.float32)
        ox = np.array([oracle_mod.interp_f32(ogx, x, y) for x, y in zip(xs, ys)], np.float32)
        oy = np.array([oracle_mod.interp_f32(ogy, x, y) for x, y in zip(xs, ys)], np.float32)
        assert np.array_equal(ri, oi) and np.array_equal(rgx, ox) and np.array_equal(rgy, oy), l
        assert (ri == -1).sum() > 5 and (ri > 0).sum() > 200


def test_reference_pose_algebra_vs_oracle(oracle_mod, R):
    """frame::concatenateRelativePose / concatenateOriginPose (src/Frame.cpp:503-562)."""
    rng = np.random.default_rng(4)
    for n in range(60):
        s = 10.0 ** rng.uniform(-3, 0.3)
        a = (rng.standard_normal(6) * s).astype(np.float32); b = (rng.standard_normal(6) * s).astype(np.float32)
        assert np.array_equal(R.concat_relative(a, b), oracle_mod.concat_relative(a, b)), n
        assert np.array_equal(R.concat_origin(a, b), oracle_mod.concat_origin(a, b)), n


def test_reference_live_random_pairs(oracle_mod, R):
    """Fresh seeds (not the fixture's): the oracle stays bit-identical to the reference, including an all-out-of-bounds start
    (zero step: H = 0, cv::Mat::inv() returns zeros) and a keyframe without depth."""
    import sys
    sys.path.insert(0, os.path.join(GOLD))
    from make_reference_golden import reference_case
    case = reference_case(n_frames=2, seed=77, k=R.dims())
    k, kf = case["k"], case["kf"]
    ocfg = oracle_mod.default_config(k["width"], k["height"], fx=float(k["fx"]), fy=float(k["fy"]), cx=float(k["cx"]), cy=float(k["cy"]))
    far = np.array([0, 0, 0, 50.0, 0, 0], np.float32)                                        # every warp lands outside the image
    nodepth = [np.zeros_like(d) for d in kf["depth"]]
    runs = [(case["frames"][0], kf["depth"], np.zeros(6, np.float32)), (case["frames"][1], kf["depth"], (case["gt"][1] * 0.5).astype(np.float32)),
            (case["frames"][0], kf["depth"], far), (case["frames"][0], nodepth, np.zeros(6, np.float32))]
    for n, (fr, depth, init) in enumerate(runs):
        pose, tr = oracle_mod.track(ocfg, kf["image"], fr, depth, kf["var"], init)
        r = R.track_trace(kf["image"], fr, depth, kf["var"], init)
        assert tr["n_selected"] == r["n_selected"] and tr["n_iters"] == r["n_iters"], n
        assert np.array_equal(pose, r["final_pose"]), n
        for l in range(4):
            for o, q in zip(tr["levels"][l], r["levels"][l]):
                assert np.array_equal(np.asarray(o["H"], np.float32).reshape(6, 6), q["H"]) and np.array_equal(o["b"], q["b"]), (n, l)
                assert np.float32(o["weighted_pose"]) == q["weighted_pose"], (n, l)
    assert tr["n_iters"] == [1, 1, 1, 1]                          # no depth: one zero step per level


@pytest.mark.parametrize("parallel", [True, False])
def test_reference_live_loop_closure_flow(oracle_mod, fx, parallel, R):
    """Both settings of FLAG_DO_PARALLEL_CONST_WEIGHT_POSE_EST (3 + 2 row bands on threads / one band), a keyframe with three
    saved weight images (1/3 is not a power of two: cv::Mat / scalar multiplies by the float reciprocal)."""
    g = fx
    depth, var = _depth(g)
    ocfg = _ocfg(oracle_mod, g, lc_parallel=int(parallel))
    r = R.lc_flow(g["kf_image"], list(g["frames"]), g["init"], depth, var, g["frames"][1], g["gt"][1] * 0.4, parallel=parallel)
    wf, cnt, seq_poses = _oracle_lc_weights(oracle_mod, g, ocfg)
    assert cnt == r["counts"] and np.array_equal(seq_poses, r["seq_poses"])
    for l in range(4):
        assert same(r["weights"][l], wf[l]), l
    init = oracle_mod.concat_origin((g["gt"][1] * 0.4).astype(np.float32), np.zeros(6, np.float32))
    pose, tr = oracle_mod.track_lc(ocfg, g["kf_image"], g["frames"][1], depth, wf, init)
    assert np.array_equal(pose, r["lc_pose"]) and np.array_equal(pose, r["lc_trace"]["final_pose"])
    assert tr["n_iters"] == r["lc_trace"]["n_iters"]
    for l in range(4):
        for o, q in zip(tr["levels"][l], r["lc_trace"]["levels"][l]):
            assert np.array_equal(np.asarray(o["H"], np.float32).reshape(6, 6), q["H"]) and np.array_equal(o["b"], q["b"]), l


def test_reference_live_randomised_sweep(oracle_mod, R):
    """Eight more seeded pairs with random ground-truth motions (0.3 - 4 degrees, up to 0.06 units) and random initial poses,
    forward tracker: counts, iteration counts, every hessian / sd_param / weightedPose / pose bit-identical to the reference."""
    import sys
    sys.path.insert(0, GOLD)
    from egomotion_with_local_loop_closures_b200 import synth
    k = R.dims()
    kk = dict(fx=k["fx"], fy=k["fy"], cx=k["cx"], cy=k["cy"])
    ocfg = oracle_mod.default_config(k["width"], k["height"], fx=float(k["fx"]), fy=float(k["fy"]), cx=float(k["cx"]), cy=float(k["cy"]))
    rng = np.random.default_rng(2026)
    total = 0
    for scene_seed in (7, 19):
        scene = synth.SynthScene(k["width"], k["height"], seed_tex=1000 + scene_seed, k=kk)
        kf = scene.keyframe(noise_seed=scene_seed)
        for _ in range(4):
            gt = synth.random_pose(rng, rot=np.deg2rad(rng.uniform(0.3, 4.0)), trans=rng.uniform(0.005, 0.06))
            cur = scene.render(synth.se3_exp(gt), noise_seed=int(rng.integers(1, 10**6)))
            init = (gt * rng.uniform(0.0, 1.2) + rng.normal(0, 1e-3, 6)).astype(np.float32)
            pose, tr = oracle_mod.track(ocfg, kf["image"], cur, kf["depth"], kf["var"], init)
            r = R.track_trace(kf["image"], cur, kf["depth"], kf["var"], init)
            assert tr["n_selected"] == r["n_selected"] and tr["n_iters"] == r["n_iters"]
            assert np.array_equal(pose, r["final_pose"])
            for l in range(4):
                for o, q in zip(tr["levels"][l], r["levels"][l]):
                    assert np.array_equal(np.asarray(o["H"], np.float32).reshape(6, 6), q["H"]) and np.array_equal(o["b"], q["b"])
                    assert np.float32(o["weighted_pose"]) == q["weighted_pose"] and np.array_equal(o["pose_after"], q["pose_after"])
                    total += 1
    assert total > 100


# ---- the reference's own code at the METRIC resolution (640x480) ----------------------------------------------------------
@pytest.fixture(scope="module")
def fx640():
    return np.load(os.path.join(GOLD, "reference_track_640x480.npz"))


def _pyramids640(g):
    import sys
    sys.path.insert(0, GOLD)
    from make_reference_golden import digest
    from make_reference_golden_640x480 import rebuild_pyramids
    depth, var = rebuild_pyramids(g["depth0"])
    assert [digest(a) for a in depth] == list(g["depth_sha"]) and [digest(a) for a in var] == list(g["var_sha"])
    return depth, var


def test_oracle_is_bit_identical_to_the_reference_at_640x480(oracle_mod, fx640):
    """The committed fixture of the reference's own outputs at 640x480 (BASELINE.json's metric resolution; the reference's camera
    is a compile-time constant, so this is a second build of the same unmodified sources -- tests/golden/
    make_reference_golden_640x480.py): the oracle reproduces counts, iteration counts and every iteration's hessian / sd_param /
    weightedPose / pose BIT FOR BIT, and the driver's result."""
    g = fx640
    depth, var = _pyramids640(g)
    fxv, fyv, cx, cy = (float(v) for v in g["intr"])
    ocfg = oracle_mod.default_config(640, 480, fx=fxv, fy=fyv, cx=cx, cy=cy)
    n_it = 0
    for i in range(len(g["frames"])):
        pose, tr = oracle_mod.track(ocfg, g["kf_image"], g["frames"][i], depth, var, g["init"][i])
        assert tr["n_selected"] == list(g[f"p{i}_n_selected"]) and tr["n_iters"] == list(g[f"p{i}_n_iters"]), i
        assert np.array_equal(pose, g[f"p{i}_pose"]), i
        for l in range(4):
            for k, o in enumerate(tr["levels"][l]):
                assert np.array_equal(np.asarray(o["H"], np.float32).reshape(6, 6), g[f"p{i}_H_{l}"][k]), (i, l, k)
                assert np.array_equal(o["b"], g[f"p{i}_b_{l}"][k]) and np.float32(o["weighted_pose"]) == g[f"p{i}_wp_{l}"][k], (i, l, k)
                assert np.array_equal(o["pose_after"], g[f"p{i}_pose_{l}"][k]), (i, l, k)
                n_it += 1
        # GetImagePoseEstimate with the t-1 frame at world pose init and the keyframe at the origin (src/ImageFunc.cpp:97-108, :305-306)
        init = oracle_mod.concat_origin(g["init"][i], np.zeros(6, np.float32))
        dpose, _ = oracle_mod.track(ocfg, g["kf_image"], g["frames"][i], depth, var, init)
        assert np.array_equal(dpose, g[f"p{i}_driver_pose"]), i
        assert np.array_equal(oracle_mod.concat_relative(dpose, np.zeros(6, np.float32)), g[f"p{i}_driver_pose_wrt_world"]), i
    assert n_it > 20


def test_fixture_640x480_is_what_the_reference_produces(fx640, R):
    prev = R.select("640x480")
    try:
        k = R.dims()
        assert (k["width"], k["height"], float(k["fx"]), float(k["cx"]), float(k["cy"])) == (640, 480, 512.0, 320.0, 240.0)
        g = fx640
        depth, var = _pyramids640(g)
        tr = R.track_trace(g["kf_image"], g["frames"][1], depth, var, g["init"][1])
        assert tr["n_iters"] == list(g["p1_n_iters"]) and np.array_equal(tr["final_pose"], g["p1_pose"])
    finally:
        R.select(prev)


def test_reference_live_random_pairs_at_640x480(oracle_mod, scene_vga, R):
    """Fresh pairs at 640x480 (the parity tests' own scene_vga case and two perturbed starts): oracle vs the reference's own code,
    bit-identical at every iteration."""
    prev = R.select("640x480")
    try:
        case = scene_vga
        ocfg = oracle_mod.default_config(640, 480, fx=512.0, fy=512.0, cx=320.0, cy=240.0)
        kf = case["kf"]
        runs = [(case["frames"][0], np.zeros(6, np.float32)), (case["frames"][1], (case["gt"][1] * 0.5).astype(np.float32)),
                (case["frames"][0], (case["gt"][0] * 1.4).astype(np.float32))]
        total = 0
        for n, (fr, init) in enumerate(runs):
            pose, tr = oracle_mod.track(ocfg, kf["image"], fr, kf["depth"], kf["var"], init)
            r = R.track_trace(kf["image"], fr, kf["depth"], kf["var"], init)
            assert tr["n_selected"] == r["n_selected"] and tr["n_iters"] == r["n_iters"], n
            assert np.array_equal(pose, r["final_pose"]), n
            for l in range(4):
                for o, q in zip(tr["levels"][l], r["levels"][l]):
                    assert np.array_equal(np.asarray(o["H"], np.float32).reshape(6, 6), q["H"]) and np.array_equal(o["b"], q["b"]), (n, l)
                    assert np.float32(o["weighted_pose"]) == q["weighted_pose"] and np.array_equal(o["pose_after"], q["pose_after"]), (n, l)
                    total += 1
        assert total > 30
    finally:
        R.select(prev)
