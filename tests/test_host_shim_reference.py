"""The C++ host shim with util::GPU_ARITHMETIC = ELLC_ARITH_REFERENCE: builds on CPU; on GPU one GetImagePoseEstimate returns what
the reference's own driver returned for tests/golden/reference_track_480x270.npz, bit for bit (pose, poseWrtOrigin, poseWrtWorld)."""
import os
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "egomotion_with_local_loop_closures_b200")
EXE = os.path.join(ROOT, "tests", "cpp", "test_shim_reference")


def build_shim_reference():
    import __graft_entry__ as g
    g.build()
    src = [os.path.join(ROOT, "tests", "cpp", "test_shim_reference.cpp"), os.path.join(PKG, "host", "HostShim.cpp"),
           os.path.join(PKG, "host", "PoseFiles.cpp")]
    deps = src + [os.path.join(PKG, "libellc_gn.so"), os.path.join(PKG, "host", "ExternVariable.h")]
    if not os.path.exists(EXE) or any(os.path.getmtime(s) > os.path.getmtime(EXE) for s in deps):
        subprocess.check_call(["g++", "-std=c++11", "-O2", "-pthread", "-I", os.path.join(PKG, "host"), "-o", EXE] + src +
                              ["-L", PKG, "-lellc_gn", "-Wl,-rpath," + PKG])
    return EXE


def test_shim_reference_builds():
    assert os.access(build_shim_reference(), os.X_OK)


@pytest.mark.gpu
def test_shim_reference_mode_reproduces_the_reference_driver(tmp_path):
    g = np.load(os.path.join(ROOT, "tests", "golden", "reference_track_480x270.npz"))
    exe = build_shim_reference()
    w, h = int(g["width"][0]), int(g["height"][0])
    blob = tmp_path / "ref_case.bin"
    with open(blob, "wb") as f:
        f.write(struct.pack("<iii4f", w, h, 1, *(float(v) for v in g["intr"])))
        f.write(g["kf_image"].tobytes())
        for l in range(4):
            f.write(np.ascontiguousarray(g[f"depth{l}"], np.float32).tobytes())
        for l in range(4):
            f.write(np.ascontiguousarray(g[f"var{l}"], np.float32).tobytes())
        f.write(g["frames"][0].tobytes())
    out = subprocess.check_output([exe, str(blob)], text=True)
    got = {l.split()[0]: np.array(l.split()[1:7], np.float32) for l in out.strip().splitlines() if l.split()}
    # %.9g round-trips a float exactly
    for key, ref in (("pose", "p0_driver_pose"), ("origin", "p0_driver_pose_wrt_origin"), ("world", "p0_driver_pose_wrt_world")):
        want = np.asarray(g[ref], np.float32).reshape(6)
        assert np.array_equal(got[key].view(np.uint32), want.view(np.uint32)), (key, got[key], want)
