"""Generates tests/golden/reference_track_480x270.npz from THE REFERENCE'S OWN CODE (run in the build container, where
/root/reference is mounted): oracle/_ref/libellc_ref.so = the reference's unmodified src/Frame.cpp, PixelWisePyramid.cpp,
UserDefinedFunc.cpp, ImageFunc.cpp ... compiled against the stand-in headers under oracle/shim/ (oracle/ref_driver.cpp).

The fixture holds seeded inputs at the reference's compiled-in configuration (480x270, its intrinsics) and, for every pair,
what the reference produced: per-level selected-pixel counts and iteration counts, hessian / sd_param / weightedPose / pose
of every iteration, display_weightimg of the last level-0 iteration, the result of GetImagePoseEstimate() and its
poseWrtOrigin / poseWrtWorld post-conditions.  tests/test_reference_pin.py checks the oracle against it (CPU) and
tests/test_gpu_parity.py the CUDA path (GPU box, where /root/reference does not exist).

    python tests/golden/make_reference_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))


def reference_case(n_frames=3, seed=31, k=None):
    """Keyframe + frames at the reference's compiled-in size and intrinsics (`k`: refbinding.dims(), asked of the library when not
    given); the last frame is a large rotation (out-of-bounds warps, more iterations)."""
    from egomotion_with_local_loop_closures_b200 import synth
    from oracle import refbinding as ref
    k = k or ref.dims()
    kk = dict(fx=k["fx"], fy=k["fy"], cx=k["cx"], cy=k["cy"])
    scene = synth.SynthScene(k["width"], k["height"], k=kk)
    kf = scene.keyframe(noise_seed=seed)
    rng = np.random.default_rng(seed)
    frames, gt = [], []
    for i in range(n_frames):
        big = (i == n_frames - 1)
        p = synth.random_pose(rng, rot=np.deg2rad(3.5 if big else 1.2), trans=0.04 if big else 0.015)
        frames.append(scene.render(synth.se3_exp(p), noise_seed=seed * 100 + i))
        gt.append(p.astype(np.float32))
    return dict(k=k, kf=kf, frames=frames, gt=gt)


def hypotheses_case(h, w, seed=8):
    """Seeded depth hypotheses (isValid / invDepthSmoothed / varianceSmoothed) with the awkward values: inverse depths below the
    -0.05 gate, slightly negative, zero (depth = inf) and denormal-small."""
    rng = np.random.default_rng(seed)
    valid = (rng.random((h, w)) < 0.35).astype(np.uint8)
    idep = rng.uniform(0.3, 2.0, (h, w)).astype(np.float32)
    for value, count in ((-0.2, 200), (-0.01, 200), (0.0, 50), (1e-30, 50)):
        idep.reshape(-1)[rng.integers(0, h * w, count)] = value
    var = rng.uniform(1e-4, 0.05, (h, w)).astype(np.float32)
    return valid, idep, var


def digest(a):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main():
    from oracle import refbinding as ref
    case = reference_case()
    k, kf = case["k"], case["kf"]
    out = dict(width=np.array([k["width"]]), height=np.array([k["height"]]),
               intr=np.array([k["fx"], k["fy"], k["cx"], k["cy"]], np.float32), kf_image=kf["image"],
               frames=np.stack(case["frames"]), gt=np.stack(case["gt"]))
    for l in range(4):
        out[f"depth{l}"] = kf["depth"][l]
        out[f"var{l}"] = kf["var"][l]
    inits = [np.zeros(6, np.float32), (case["gt"][1] * 0.6).astype(np.float32), np.zeros(6, np.float32)]
    out["init"] = np.stack(inits)
    for i, (fr, init) in enumerate(zip(case["frames"], inits)):
        tr = ref.track_trace(kf["image"], fr, kf["depth"], kf["var"], init, want_weights=True)
        out[f"p{i}_n_selected"] = np.array(tr["n_selected"], np.int32)
        out[f"p{i}_n_iters"] = np.array(tr["n_iters"], np.int32)
        out[f"p{i}_pose"] = tr["final_pose"]
        out[f"p{i}_weights_l0"] = tr["weights_l0"]
        for l in range(4):
            its = tr["levels"][l]
            out[f"p{i}_H_{l}"] = np.stack([it["H"] for it in its])
            out[f"p{i}_b_{l}"] = np.stack([it["b"] for it in its])
            out[f"p{i}_wp_{l}"] = np.array([it["weighted_pose"] for it in its], np.float32)
            out[f"p{i}_pose_{l}"] = np.stack([it["pose_after"] for it in its])
        # the reference's own driver: the t-1 frame's world pose is its initialisation (src/ImageFunc.cpp:97-108)
        pose, po, pw = ref.get_image_pose_estimate(kf["image"], fr, kf["depth"], kf["var"], init)
        out[f"p{i}_driver_pose"] = pose
        out[f"p{i}_driver_pose_wrt_origin"] = po
        out[f"p{i}_driver_pose_wrt_world"] = pw
    # the constant-weight loop-closure flow with the reference's own driver (weights saved by the three sequential tracks,
    # frame::finaliseWeights, GetImagePoseEstimate(fromLoopClosure=true) on the last frame); the weight pyramid itself is not
    # stored (0.7 MB): whoever replays the flow rebuilds it
    lc_tm1 = (case["gt"][2] * 0.7).astype(np.float32)
    r = ref.lc_flow(kf["image"], case["frames"], inits, kf["depth"], kf["var"], case["frames"][2], lc_tm1, parallel=True)
    out["lc_tminus1"] = lc_tm1
    out["lc_counts"] = np.array(r["counts"], np.int32)
    out["lc_seq_poses"] = r["seq_poses"]
    out["lc_pose"] = r["lc_pose"]
    out["lc_weight_sums"] = np.array([float(w.astype(np.float64).sum()) for w in r["weights"]])
    out["lc_n_iters"] = np.array(r["lc_trace"]["n_iters"], np.int32)
    for l in range(4):
        its = r["lc_trace"]["levels"][l]
        out[f"lc_H_{l}"] = np.stack([it["H"] for it in its])
        out[f"lc_b_{l}"] = np.stack([it["b"] for it in its])
        out[f"lc_wp_{l}"] = np.array([it["weighted_pose"] for it in its], np.float32)
        out[f"lc_pose_{l}"] = np.stack([it["pose_after"] for it in its])
    # SURVEY 8f row 2: depthMap::updateDepthImage / buildInvVarDepth / mapDepthArr2Mat / calculate_no_of_Seeds on seeded
    # hypotheses (inputs are regenerated from the seed by the tests; the reference's outputs are stored as SHA-256 digests)
    valid, idep, var = hypotheses_case(k["height"], k["width"])
    r = ref.update_depth_image(kf["image"], valid, idep, var)
    out["hyp_occupancy"] = np.array([r["occupancy"]], np.float32)
    out["hyp_valid_sha"] = np.array(digest(r["valid_out"]))
    out["hyp_depth_sha"] = np.array([digest(a) for a in r["depth"]])
    out["hyp_var_sha"] = np.array([digest(a) for a in r["var"]])
    out["hyp_selected"] = np.array([int((a > 0).sum()) for a in r["depth"]], np.int32)
    # SURVEY 8f row 3: calculateImageHistogram / compareImageHistogram / calculateRotationStats on the fixture's frames
    n = len(case["frames"])
    out["gate_hist"] = np.stack([ref.gating(case["frames"][i], case["frames"][i], case["gt"][i], case["gt"][i])["hist_a"] for i in range(n)])
    kl = np.zeros((n, n)); rms = np.zeros((n, n), np.float32); ang = np.zeros((n, n), np.float32)
    for i in range(n):
        for j in range(n):
            gt = ref.gating(case["frames"][i], case["frames"][j], case["gt"][i], case["gt"][j])
            kl[i, j], rms[i, j], ang[i, j] = gt["kl"], gt["rms_error"], gt["relative_view_angle"]
    out["gate_kl"], out["gate_rms"], out["gate_angle"] = kl, rms, ang
    # SURVEY 8a row L: the matrix-form src/Pyramid.cpp driven as its comments describe (performPrecomputation at a pose, then
    # performIterationSteps): per-pixel weights digest, sum w r^2 / n (:682), hessianInv and the pose after the first update
    pyr_cases = [(0, 2, np.zeros(6, np.float32)), (1, 1, (case["gt"][1] * 0.5).astype(np.float32)), (2, 3, np.zeros(6, np.float32))]
    out["pyr_frame_level"] = np.array([(f, l) for f, l, _ in pyr_cases], np.int32)
    out["pyr_pose_in"] = np.stack([p for _, _, p in pyr_cases])
    rr = [ref.pyramid_run(kf["image"], case["frames"][f], kf["depth"], kf["var"], l, p, iters=2) for f, l, p in pyr_cases]
    out["pyr_n"] = np.array([r["n"] for r in rr], np.int32)
    out["pyr_last_err"] = np.array([r["last_err"] for r in rr], np.float32)
    out["pyr_weights_sha"] = np.array([digest(r["weights"]) for r in rr])
    out["pyr_hessian_inv"] = np.stack([r["hessian_inv"] for r in rr])
    out["pyr_poses_after"] = np.stack([r["poses_after"] for r in rr])
    path = os.path.join(HERE, "reference_track_480x270.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
