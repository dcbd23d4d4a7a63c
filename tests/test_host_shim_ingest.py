"""The C++ host shim's camera constructor frame(camera_image, cols, rows, channels) + util::configure_camera: builds on CPU; on GPU
its frames carry the oracle's level-0 images and track to the same poses as the gray constructor fed those images."""
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

from tests import ingest_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "egomotion_with_local_loop_closures_b200")
EXE = os.path.join(ROOT, "tests", "cpp", "test_shim_ingest")
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))


def build_shim_ingest():
    import __graft_entry__ as g
    g.build()
    src = [os.path.join(ROOT, "tests", "cpp", "test_shim_ingest.cpp"), os.path.join(PKG, "host", "HostShim.cpp"),
           os.path.join(PKG, "host", "PoseFiles.cpp")]
    deps = src + [os.path.join(PKG, "libellc_gn.so"), os.path.join(PKG, "host", "ExternVariable.h"), os.path.join(PKG, "host", "Frame.h")]
    if not os.path.exists(EXE) or any(os.path.getmtime(s) > os.path.getmtime(EXE) for s in deps):
        subprocess.check_call(["g++", "-std=c++11", "-O2", "-pthread", "-I", os.path.join(PKG, "host"), "-o", EXE] + src +
                              ["-L", PKG, "-lellc_gn", "-Wl,-rpath," + PKG])
    return EXE


def test_shim_ingest_builds():
    assert os.access(build_shim_ingest(), os.X_OK)


@pytest.mark.gpu
def test_camera_frames_track_like_gray_frames(tmp_path):
    import make_ingest_golden as mk
    from egomotion_with_local_loop_closures_b200 import synth
    exe = build_shim_ingest()
    w, h, n, F = 320, 240, 3, 4
    W, H = w * F, h * F
    scene = synth.SynthScene(w, h)
    kf = scene.keyframe(noise_seed=5)
    T = synth.smooth_trajectory(n + 1, seed_pose=3)
    frames = [scene.render(T[i + 1], noise_seed=50 + i) for i in range(n)]
    rng = np.random.default_rng(9)

    def cam(gray):
        big = np.kron(gray.astype(np.int16), np.ones((F, F), np.int16))
        return np.clip(np.stack([big + rng.integers(-3, 4, big.shape) for _ in range(3)], -1), 0, 255).astype(np.uint8)
    kf_cam, cams = cam(kf["image"]), [cam(f) for f in frames]
    K = mk.camera_matrix(W, H)
    alpha = 1.0
    newK = ingest_oracle.optimal_new_camera_matrix(K, mk.DIST, W, H, alpha)
    grays = [ingest_oracle.ingest(c, w, h, True, K, mk.DIST, newK) for c in [kf_cam] + cams]
    k = synth.intrinsics(w, h)
    blob = tmp_path / "case.bin"
    with open(blob, "wb") as f:
        f.write(struct.pack("<5i4f", w, h, W, H, n, float(k["fx"]), float(k["fy"]), float(k["cx"]), float(k["cy"])))
        f.write(np.ascontiguousarray(K, np.float64).tobytes() + np.ascontiguousarray(mk.DIST, np.float64).tobytes() + struct.pack("<d", alpha))
        f.write(kf_cam.tobytes())
        for l in range(4):
            f.write(np.ascontiguousarray(kf["depth"][l], np.float32).tobytes())
        for l in range(4):
            f.write(np.ascontiguousarray(kf["var"][l], np.float32).tobytes())
        for c in cams:
            f.write(c.tobytes())
        for g in grays:
            f.write(g.tobytes())
    out = subprocess.check_output([exe, str(blob)], text=True)
    lines = [l.split() for l in out.strip().splitlines()]
    assert lines[0] == ["size", str(w), str(h)]
    assert [l[1] for l in lines if l[0] == "img"] == ["1"] * (n + 1)
    poses = {(int(l[1]), int(l[2])): l[3:] for l in lines if l[0] == "pose"}
    assert len(poses) == 2 * n
    for i in range(n):
        assert poses[(0, i)] == poses[(1, i)], i
        assert np.all(np.isfinite(np.array(poses[(0, i)], np.float64)))
