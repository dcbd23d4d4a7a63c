"""ELLC_ARITH_REFERENCE on the GPU: the tracker reproduces the reference's own arithmetic bit for bit.

Every comparison here is exact (the float bits; two NaNs count as equal, their payloads are not part of IEEE results):
  a. teacher-forced along the reference's own trajectories (ELLC's fixtures at 480x270 and 640x480): hessian, sd_param,
     weightedPose, pose after updatePose(), the level-0 weight image;
  b. free-running on the same fixtures: counts, iterations, every traced iteration, final poses;
  c. against the live oracle (3 row bands) on seeded scenes and corner cases: empty bands, an empty level, an all-out-of-bounds
     pose (inf depths: reproducible records, see the test);
  d. K5 alone on random systems (rotations 1e-7 .. 0.3 rad: both small-angle branches of the logarithm, every Pade branch);
  e. the loop-closure flow fixture (lc_bands = 2) and the live oracle's constant-weight tracker with 1 and 2 bands;
  f. a mixed 64-pair batch equals its pairs tracked one at a time, and two runs are identical.
"""
import os

import numpy as np
import pytest

from tests.helpers import gpu_config, make_case, oracle_config

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def capi():
    from egomotion_with_local_loop_closures_b200 import capi as m
    m.lib()
    return m


def same(a, b):
    """Bit-identical float32 arrays (NaN == NaN)."""
    a = np.ascontiguousarray(np.asarray(a, np.float32)).reshape(-1)
    b = np.ascontiguousarray(np.asarray(b, np.float32)).reshape(-1)
    if a.shape != b.shape:
        return False
    nan = np.isnan(a) & np.isnan(b)
    return bool(np.all(nan | (a.view(np.uint32) == b.view(np.uint32))))


def _fixture_pyramids(g):
    if "depth1" in g:
        return [g[f"depth{l}"] for l in range(4)], [g[f"var{l}"] for l in range(4)]
    import sys
    sys.path.insert(0, GOLD)
    from make_reference_golden import digest
    from make_reference_golden_640x480 import rebuild_pyramids
    depth, var = rebuild_pyramids(g["depth0"])                 # the 640x480 fixture stores level 0 and the digests
    assert [digest(a) for a in depth] == list(g["depth_sha"]) and [digest(a) for a in var] == list(g["var_sha"])
    return depth, var


def _fixture_tracker(capi, g, **over):
    w, h = int(g["width"][0]), int(g["height"][0])
    fxv, fyv, cx, cy = (float(v) for v in g["intr"])
    n = len(g["frames"])
    t = capi.Tracker(capi.default_config(w, h, fx=fxv, fy=fyv, cx=cx, cy=cy, max_keyframes=1, max_frames=n,
                                         arithmetic=capi.ARITH_REFERENCE, **over))
    depth, var = _fixture_pyramids(g)
    t.upload_keyframe(0, g["kf_image"], depth, var)
    for i in range(n):
        t.upload_frame(i, g["frames"][i])
    return t, n


@pytest.mark.parametrize("name", ["reference_track_480x270.npz", "reference_track_640x480.npz"])
def test_teacher_forced_on_reference_fixtures(capi, name):
    g = np.load(os.path.join(GOLD, name))
    t, n = _fixture_tracker(capi, g)
    has_w = "p0_weights_l0" in g
    for i in range(n):
        pose_before = g["init"][i]
        for l in (3, 2, 1, 0):
            m = len(g[f"p{i}_H_{l}"])
            for k in range(m):
                want_w = has_w and l == 0 and k == m - 1
                f = t.gn_evaluate(0, i, l, pose_before, want_weights=want_w)
                if want_w:
                    f, gw = f
                    assert same(gw, g[f"p{i}_weights_l0"]), i
                assert same(f["H"], g[f"p{i}_H_{l}"][k]), (i, l, k)
                assert same(f["b"], g[f"p{i}_b_{l}"][k]), (i, l, k)
                gp, gd, gwp = t.solve_update(g[f"p{i}_H_{l}"][k], g[f"p{i}_b_{l}"][k], pose_before)
                assert same(gwp, g[f"p{i}_wp_{l}"][k]), (i, l, k)
                assert same(gp, g[f"p{i}_pose_{l}"][k]), (i, l, k, gp, g[f"p{i}_pose_{l}"][k])
                pose_before = g[f"p{i}_pose_{l}"][k]
    t.close()


@pytest.mark.parametrize("name", ["reference_track_480x270.npz", "reference_track_640x480.npz"])
def test_free_running_on_reference_fixtures(capi, name):
    g = np.load(os.path.join(GOLD, name))
    t, n = _fixture_tracker(capi, g)
    res, tr = t.track_batch(t.make_pairs([0] * n, list(range(n)), g["init"]), want_trace=True)
    for i in range(n):
        assert list(res[i]["n_selected"]) == list(g[f"p{i}_n_selected"]), i
        assert list(res[i]["n_iters"]) == list(g[f"p{i}_n_iters"]), (i, list(res[i]["n_iters"]), list(g[f"p{i}_n_iters"]))
        for l in range(4):
            for k in range(int(g[f"p{i}_n_iters"][l])):
                it = tr[i, l, k]
                assert it["executed"] == 1
                assert same(it["H"], g[f"p{i}_H_{l}"][k]), (i, l, k)
                assert same(it["b"], g[f"p{i}_b_{l}"][k]), (i, l, k)
                assert same(it["weighted_pose"], g[f"p{i}_wp_{l}"][k]), (i, l, k)
                assert same(it["pose_after"], g[f"p{i}_pose_{l}"][k]), (i, l, k)
        assert same(res[i]["pose"], g[f"p{i}_pose"]), (i, res[i]["pose"], g[f"p{i}_pose"])
    t.close()


def _compare_with_oracle_trace(res, tr, opose, otr, where):
    assert list(res["n_selected"]) == otr["n_selected"], where
    assert list(res["n_iters"]) == otr["n_iters"], (where, list(res["n_iters"]), otr["n_iters"])
    for l in range(4):
        for k, o in enumerate(otr["levels"][l]):
            it = tr[l, k]
            w = (where, l, k)
            assert same(it["H"], o["H"]), w
            assert same(it["b"], o["b"]), w
            assert same(it["delta"], o["delta"]), w
            assert same(it["weighted_pose"], o["weighted_pose"]), w
            assert same(it["pose_after"], o["pose_after"]), w
            assert same(it["res_sum"], o["res_sum_f32"]), w
            assert int(it["n_oob"]) == o["n_oob"], w
        if otr["levels"][l]:
            assert same(res["res_first"][l], otr["levels"][l][0]["res_sum_f32"]), (where, l)
            assert same(res["res_last"][l], otr["levels"][l][-1]["res_sum_f32"]), (where, l)
    assert same(res["pose"], opose), (where, res["pose"], opose)


def _track_live(capi, oracle_mod, case, inits, depth=None):
    depth = depth if depth is not None else case["kf"]["depth"]
    n = len(case["frames"])
    t = capi.Tracker(gpu_config(capi, case, max_keyframes=1, max_frames=n, arithmetic=capi.ARITH_REFERENCE))
    t.upload_keyframe(0, case["kf"]["image"], depth, case["kf"]["var"])
    for i, f in enumerate(case["frames"]):
        t.upload_frame(i, f)
    res, tr = t.track_batch(t.make_pairs([0] * n, list(range(n)), inits), want_trace=True)
    ocfg = oracle_config(oracle_mod, case)
    assert ocfg.num_bands == 3
    for i in range(n):
        opose, otr = oracle_mod.track(ocfg, case["kf"]["image"], case["frames"][i], depth, case["kf"]["var"], inits[i])
        _compare_with_oracle_trace(res[i], tr[i], opose, otr, i)
    t.close()


@pytest.mark.parametrize("size", [(480, 270), (122, 94)])
def test_live_oracle_seeded_scenes(capi, oracle_mod, size):
    """rows % 3 != 0 at some level: 480x270 has 67 and 33 rows at levels 2 and 3, 122x94 has 94, 47, 23 and 11."""
    case = make_case(size[0], size[1], n_frames=3, seed=size[0] + size[1])
    rng = np.random.default_rng(7)
    inits = [rng.normal(0, 0.002, 6).astype(np.float32) for _ in case["frames"]]
    _track_live(capi, oracle_mod, case, inits)


def test_live_oracle_band_corner_cases(capi, oracle_mod):
    case = make_case(160, 120, n_frames=1, seed=5)
    zero = [np.zeros(6, np.float32)]
    # every selected pixel in the middle band of every level (bands 1 and 3 empty)
    d = []
    for l, dl in enumerate(case["kf"]["depth"]):
        rows = dl.shape[0]
        m = np.zeros_like(dl)
        m[rows // 3:2 * (rows // 3)] = dl[rows // 3:2 * (rows // 3)]
        d.append(m)
    _track_live(capi, oracle_mod, case, zero, depth=d)
    # an empty level: nothing selected at level 2 (N_L = 0)
    d = [x.copy() for x in case["kf"]["depth"]]
    d[2][:] = 0.0
    _track_live(capi, oracle_mod, case, zero, depth=d)
    # inf depths at a few pixels of every level.  Their back-projection gives NaN image coordinates, which the CPU oracle's sampler
    # turns into array indices (undefined behaviour: it crashes), so there is no oracle trace to compare with; the device selects
    # them as the reference does and its records are reproducible.
    d = [x.copy() for x in case["kf"]["depth"]]
    for x in d:
        x[x.shape[0] // 2, 3:x.shape[1]:17] = np.inf
    t = capi.Tracker(gpu_config(capi, case, max_keyframes=1, max_frames=1, arithmetic=capi.ARITH_REFERENCE))
    t.upload_keyframe(0, case["kf"]["image"], d, case["kf"]["var"])
    t.upload_frame(0, case["frames"][0])
    a = t.track_batch(t.make_pairs([0], [0], zero))
    assert a.tobytes() == t.track_batch(t.make_pairs([0], [0], zero)).tobytes()
    assert list(a[0]["n_selected"]) == [oracle_mod.mask_count(x)[1] for x in d]
    t.close()
    # a pose that warps every pixel out of bounds
    _track_live(capi, oracle_mod, case, [np.array([0, 0, 0, 50.0, 0, 0], np.float32)])


def test_k5_against_oracle_randomised(capi, oracle_mod, scene_small):
    case = scene_small
    t = capi.Tracker(gpu_config(capi, case, max_keyframes=1, max_frames=1, arithmetic=capi.ARITH_REFERENCE))
    ocfg = oracle_config(oracle_mod, case)
    rng = np.random.default_rng(20261020)
    branches, angles, misses = set(), [], []
    for n in range(300):
        J = (rng.standard_normal((300, 6)) * np.array([800, 800, 800, 90, 90, 90])).astype(np.float32)
        H = (J.T @ J).astype(np.float32) if n % 2 == 0 else rng.standard_normal((6, 6)).astype(np.float32)
        Hinv, ok = oracle_mod.invert6(H)
        assert ok
        rot = 10.0 ** rng.uniform(-7, np.log10(0.3))                           # rotation of the step, rad
        want = np.concatenate([rng.standard_normal(3), rng.standard_normal(3) * 10.0 ** rng.uniform(-4, 0.6) / rot])
        want[:3] *= rot / np.linalg.norm(want[:3])
        want[3:] *= rot
        if n % 3 == 0:
            want[3:] = rng.standard_normal(3) * 10.0 ** rng.uniform(-3, 0.6)   # large translations: Pade-7 with squarings
        b = (-(H.astype(np.float64) @ want)).astype(np.float32)
        pose0 = np.concatenate([rng.standard_normal(3) * 10.0 ** rng.uniform(-7, -0.6), rng.standard_normal(3) * 10.0 ** rng.uniform(-3, 0.3)]).astype(np.float32)
        op, od, owp = oracle_mod.update_pose(ocfg, Hinv, b, pose0)
        gp, gd, gwp = t.solve_update(H, b, pose0)
        assert same(gd, od) and same(gwp, owp), n
        if not same(gp, op):
            misses.append((n, gp.tolist(), op.tolist()))
        angles.append(float(np.linalg.norm(op[:3].astype(np.float64))))
        for v in (od, op):
            l1 = max(abs(v[2]) + abs(v[1]), abs(v[2]) + abs(v[0]), abs(v[1]) + abs(v[0]), abs(v[3]) + abs(v[4]) + abs(v[5]))
            branches.add(0 if l1 < 0.42587 else 1 if l1 < 1.88015 else 2 if l1 < 3.92572 else 3)
    assert branches == {0, 1, 2, 3}
    assert min(angles) < 1e-6 and max(angles) > 0.1                             # both small-angle branches of the log and the closed form
    assert not misses, misses[:5]
    t.close()


def _lc_flow(capi, g, n, t):
    zero = np.zeros(6, np.float32)
    inits = np.stack([capi.concat_origin(g["init"][i], zero) for i in range(n)])        # src/ImageFunc.cpp:106
    seq = t.track_batch(t.make_pairs([0] * n, list(range(n)), inits, flags=capi.PAIR_SAVE_WEIGHTS))
    t.reset_keyframe_weights(0)
    t.accumulate_weights(0, list(range(n)))
    t.finalise_weights(0)
    t.prepare_keyframes_lc([0])
    return seq


def test_loop_closure_flow_fixture(capi):
    g = np.load(os.path.join(GOLD, "reference_track_480x270.npz"))
    t, n = _fixture_tracker(capi, g)
    seq = _lc_flow(capi, g, n, t)
    assert same(seq["pose"], g["lc_seq_poses"])
    for l in range(4):
        gw, c = t.read_keyframe_weights(0, l)
        assert c == int(g["lc_counts"][l])
        assert float(gw.astype(np.float64).sum()) == float(g["lc_weight_sums"][l]), l
    lc_init = capi.concat_origin(g["lc_tminus1"], np.zeros(6, np.float32))
    res, tr = t.track_batch(t.make_pairs([0], [2], [lc_init], flags=capi.PAIR_CONST_WEIGHT), want_trace=True)
    assert list(res[0]["n_iters"]) == list(g["lc_n_iters"])
    for l in range(4):
        for k in range(int(g["lc_n_iters"][l])):
            it = tr[0, l, k]
            assert same(it["H"], g[f"lc_H_{l}"][k]), (l, k)
            assert same(it["b"], g[f"lc_b_{l}"][k]), (l, k)
            assert same(it["weighted_pose"], g[f"lc_wp_{l}"][k]), (l, k)
            assert same(it["pose_after"], g[f"lc_pose_{l}"][k]), (l, k)
    assert same(res[0]["pose"], g["lc_pose"])
    t.close()


def _oracle_lc_weights(oracle_mod, case):
    ocfg = oracle_config(oracle_mod, case)
    h, w = case["height"], case["width"]
    wp = [np.zeros((h >> l, w >> l), np.float32) for l in range(4)]
    cnt = [0] * 4
    for f in case["frames"]:
        _, _, wl = oracle_mod.track_with_weights(ocfg, case["kf"]["image"], f, case["kf"]["depth"], case["kf"]["var"], np.zeros(6, np.float32))
        oracle_mod.accumulate_weights(wp, cnt, wl)
    return oracle_mod.finalise_weights(wp, cnt), cnt


@pytest.mark.parametrize("bands", [1, 2])
def test_loop_closure_live_oracle(capi, oracle_mod, scene_small, bands):
    case = scene_small
    wf, cnt = _oracle_lc_weights(oracle_mod, case)
    n = len(case["frames"])
    t = capi.Tracker(gpu_config(capi, case, max_keyframes=1, max_frames=n, arithmetic=capi.ARITH_REFERENCE, lc_bands=bands))
    t.upload_keyframe(0, case["kf"]["image"], case["kf"]["depth"], case["kf"]["var"])
    for i, f in enumerate(case["frames"]):
        t.upload_frame(i, f)
    t.upload_keyframe_weights(0, wf, cnt)
    t.prepare_keyframes_lc([0])
    rng = np.random.default_rng(3)
    inits = [rng.normal(0, 0.003, 6).astype(np.float32) for _ in range(n)]
    res, tr = t.track_batch(t.make_pairs([0] * n, list(range(n)), inits, flags=capi.PAIR_CONST_WEIGHT), want_trace=True)
    ocfg = oracle_config(oracle_mod, case, lc_parallel=1 if bands == 2 else 0)
    for i in range(n):
        opose, otr = oracle_mod.track_lc(ocfg, case["kf"]["image"], case["frames"][i], case["kf"]["depth"], wf, inits[i])
        _compare_with_oracle_trace(res[i], tr[i], opose, otr, i)
    t.close()


def test_mixed_batch_equals_single_pairs(capi, oracle_mod):
    case = make_case(160, 120, n_frames=4, seed=19)
    wf, cnt = _oracle_lc_weights(oracle_mod, case)
    n = len(case["frames"])
    t = capi.Tracker(gpu_config(capi, case, max_keyframes=1, max_frames=n, arithmetic=capi.ARITH_REFERENCE))
    t.upload_keyframe(0, case["kf"]["image"], case["kf"]["depth"], case["kf"]["var"])
    for i, f in enumerate(case["frames"]):
        t.upload_frame(i, f)
    t.upload_keyframe_weights(0, wf, cnt)
    t.prepare_keyframes_lc([0])
    rng = np.random.default_rng(64)
    frames = [int(v) for v in rng.integers(0, n, 64)]
    inits = [rng.normal(0, 0.003, 6).astype(np.float32) for _ in range(64)]
    flags = [capi.PAIR_CONST_WEIGHT if k % 3 == 0 else capi.PAIR_DEFAULT for k in range(64)]
    pairs = np.concatenate([t.make_pairs([0], [frames[k]], [inits[k]], flags=flags[k]) for k in range(64)])
    a = t.track_batch(pairs)
    b = t.track_batch(pairs)
    assert a.tobytes() == b.tobytes()
    for k in range(64):
        one = t.track_batch(pairs[k:k + 1])[0]
        assert one.tobytes() == a[k].tobytes(), k
    t.close()
