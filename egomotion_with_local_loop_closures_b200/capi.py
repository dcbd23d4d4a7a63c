"""ctypes binding of the C-ABI in include/ellc_gn.h (libellc_gn.so).

This is plumbing for tests and bench.py; the product is the CUDA library.  There is no fallback: if the shared
library is missing the import of the symbols fails loudly, and every compute call fails with ELLC_ERR_CUDA when no
sm_100 device is usable.
"""
import ctypes as C
import os

import numpy as np

LEVELS = 4
MAX_TRACE_ITERS = 16
ARITH_FAST, ARITH_STRICT = 0, 1
PAIR_DEFAULT, PAIR_CONST_WEIGHT, PAIR_SAVE_WEIGHTS = 0, 1, 2
_LIB_PATH = os.environ.get("ELLC_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libellc_gn.so")


class EllcError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32),
                ("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float),
                ("max_iter", C.c_int32 * LEVELS), ("huber_d", C.c_float), ("camera_pixel_noise_2", C.c_float),
                ("weight", C.c_float * 6), ("stop_threshold", C.c_float), ("arithmetic", C.c_int32),
                ("jacobian_at_warped", C.c_int32), ("max_keyframes", C.c_int32), ("max_frames", C.c_int32),
                ("ctas_per_pair", C.c_int32), ("device", C.c_int32), ("pairs_per_cta", C.c_int32),
                ("lm_lambda", C.c_float), ("lm_up", C.c_float), ("lm_down", C.c_float)]


class Pair(C.Structure):
    _fields_ = [("kf_slot", C.c_int32), ("frame_slot", C.c_int32), ("init_pose", C.c_float * 6), ("flags", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("pose", C.c_float * 6), ("H", C.c_float * 21), ("b", C.c_float * 6),
                ("n_selected", C.c_int32 * LEVELS), ("n_iters", C.c_int32 * LEVELS),
                ("res_first", C.c_float * LEVELS), ("res_last", C.c_float * LEVELS),
                ("weighted_pose", C.c_float * LEVELS), ("n_oob", C.c_int32 * LEVELS),
                ("status", C.c_int32), ("reserved", C.c_int32 * 6)]


class IterTrace(C.Structure):
    _fields_ = [("H", C.c_float * 36), ("b", C.c_float * 6), ("delta", C.c_float * 6), ("weighted_pose", C.c_float),
                ("pose_after", C.c_float * 6), ("res_sum", C.c_float), ("weight_sum", C.c_float),
                ("n_oob", C.c_int32), ("executed", C.c_int32), ("lm_lambda", C.c_float), ("lm_rejected", C.c_int32),
                ("pad", C.c_int32 * 3)]


class Camera(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("channels", C.c_int32), ("pitch", C.c_int32),
                ("undistort", C.c_int32), ("reserved", C.c_int32), ("K", C.c_double * 9), ("dist", C.c_double * 5),
                ("new_K", C.c_double * 9)]


assert C.sizeof(Camera) == 208
assert C.sizeof(Result) == 256 and C.sizeof(IterTrace) == 256 and C.sizeof(Pair) == 36

PAIR_DTYPE = np.dtype([("kf_slot", "<i4"), ("frame_slot", "<i4"), ("init_pose", "<f4", 6), ("flags", "<i4")])
RESULT_DTYPE = np.dtype([("pose", "<f4", 6), ("H", "<f4", 21), ("b", "<f4", 6), ("n_selected", "<i4", 4),
                         ("n_iters", "<i4", 4), ("res_first", "<f4", 4), ("res_last", "<f4", 4),
                         ("weighted_pose", "<f4", 4), ("n_oob", "<i4", 4), ("status", "<i4"), ("reserved", "<i4", 6)])
TRACE_DTYPE = np.dtype([("H", "<f4", 36), ("b", "<f4", 6), ("delta", "<f4", 6), ("weighted_pose", "<f4"),
                        ("pose_after", "<f4", 6), ("res_sum", "<f4"), ("weight_sum", "<f4"), ("n_oob", "<i4"),
                        ("executed", "<i4"), ("lm_lambda", "<f4"), ("lm_rejected", "<i4"), ("pad", "<i4", 3)])
LC_CAND_DTYPE = np.dtype([("loop_frame_slot", "<i4"), ("test_frame_slot", "<i4"), ("loop_pose_world", "<f4", 6), ("test_pose_world", "<f4", 6)])
LC_STATS_DTYPE = np.dtype([("match_value", "<f8"), ("rms_error", "<f4"), ("relative_view_angle", "<f4"), ("pass", "<i4"), ("reserved", "<i4")])
LC_RING_DTYPE = np.dtype([("frame_id", "<i4"), ("is_valid", "<i4"), ("frame_slot", "<i4"), ("kf_slot", "<i4"), ("pose_world", "<f4", 6)])
LC_QUERY_DTYPE = np.dtype([("current_array_id", "<i4"), ("match_window_beg", "<i4"), ("match_window_end", "<i4"), ("frame_id", "<i4"),
                           ("frame_slot", "<i4"), ("stray", "<i4"), ("pose_world", "<f4", 6)])
assert LC_CAND_DTYPE.itemsize == 56 and LC_STATS_DTYPE.itemsize == 24 and LC_RING_DTYPE.itemsize == 40 and LC_QUERY_DTYPE.itemsize == 48
assert PAIR_DTYPE.itemsize == 36 and RESULT_DTYPE.itemsize == 256 and TRACE_DTYPE.itemsize == 256

# every symbol include/ellc_gn.h declares
SYMBOLS = ["ellc_default_config", "ellc_create", "ellc_destroy", "ellc_last_error_string", "ellc_version",
           "ellc_upload_frame", "ellc_upload_keyframe", "ellc_frame_image_devptr", "ellc_keyframe_devptrs",
           "ellc_prepare_frames", "ellc_prepare_keyframes", "ellc_track_batch", "ellc_track_batch_async",
           "ellc_results_download",
           "ellc_synchronize", "ellc_gn_evaluate", "ellc_solve_update", "ellc_solve_update_rt", "ellc_read_frame_level",
           "ellc_read_keyframe_level", "ellc_level_dims", "ellc_concat_relative", "ellc_concat_origin",
           "ellc_se3_exp", "ellc_launch_count", "ellc_reset_launch_count", "ellc_stream", "ellc_stream_of", "ellc_selftest_division", "ellc_selftest_unzero", "ellc_reset_keyframe_weights", "ellc_accumulate_weights",
           "ellc_finalise_weights", "ellc_upload_keyframe_weights", "ellc_read_keyframe_weights", "ellc_read_frame_weights",
           "ellc_prepare_keyframes_lc", "ellc_prepare_keyframes_lc_async", "ellc_frame_histograms", "ellc_lc_gate", "ellc_upload_keyframe_hypotheses", "ellc_read_keyframe_occupancy", "ellc_read_keyframe_depth", "ellc_last_track_kernel_ms",
           "ellc_prepare_async", "ellc_batch_kernel_ms", "ellc_batch_interval_ms", "ellc_fence",
           "ellc_exchange_create", "ellc_exchange_attach_ipc", "ellc_exchange_attach_local", "ellc_track_batch_exchange",
           "ellc_exchange_wait", "ellc_exchange_destroy", "ellc_se3_exp_closed", "ellc_se3_log_closed",
           "ellc_gn_iterate", "ellc_hessian_inverse", "ellc_lc_generate_pairs", "ellc_track_generated_pairs",
           "ellc_optimal_new_camera_matrix", "ellc_set_camera", "ellc_ingest_frames", "ellc_ingest_keyframe", "ellc_read_camera_tables"]
VARIANT_FORWARD, VARIANT_CONST_WEIGHT, VARIANT_PYRAMID = 0, 1, 2


class DisplayPlanes(C.Structure):
    _fields_ = [("warped_image", C.c_void_p), ("iteration_residual", C.c_void_p), ("warped_x", C.c_void_p), ("warped_y", C.c_void_p)]
MAX_RANKS = 8
IPC_HANDLE_BYTES = 64

_lib = None


def lib():
    """Load libellc_gn.so (built in-tree by _build.build()).  Raises if it is missing -- no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise EllcError(f"{_LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(the CUDA extension is mandatory, there is no CPU fallback)")
        L = C.CDLL(_LIB_PATH)
        L.ellc_last_error_string.restype = C.c_char_p
        L.ellc_last_error_string.argtypes = [C.c_void_p]
        L.ellc_version.restype = C.c_char_p
        L.ellc_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_void_p)]
        L.ellc_destroy.argtypes = [C.c_void_p]
        L.ellc_upload_frame.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.ellc_upload_keyframe.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ellc_frame_image_devptr.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]
        L.ellc_keyframe_devptrs.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                            C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]
        L.ellc_prepare_frames.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.ellc_prepare_keyframes.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.ellc_track_batch.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ellc_track_batch_async.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.POINTER(C.c_void_p)]
        L.ellc_synchronize.argtypes = [C.c_void_p]
        L.ellc_results_download.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
        L.ellc_gn_evaluate.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ellc_solve_update.argtypes = [C.c_void_p] + [C.c_void_p] * 5 + [C.POINTER(C.c_float)]
        L.ellc_solve_update_rt.argtypes = [C.c_void_p] + [C.c_void_p] * 5 + [C.POINTER(C.c_float), C.c_void_p]
        L.ellc_read_frame_level.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ellc_read_keyframe_level.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32)]
        L.ellc_level_dims.argtypes = [C.c_void_p, C.c_int32] + [C.POINTER(C.c_int32)] * 4
        L.ellc_concat_relative.argtypes = [C.c_void_p] * 3
        L.ellc_concat_origin.argtypes = [C.c_void_p] * 3
        L.ellc_se3_exp.argtypes = [C.c_void_p] * 2
        L.ellc_launch_count.restype = C.c_int64
        L.ellc_launch_count.argtypes = [C.c_void_p]
        L.ellc_reset_launch_count.argtypes = [C.c_void_p]
        L.ellc_stream.restype = C.c_void_p
        L.ellc_stream.argtypes = [C.c_void_p]
        L.ellc_reset_keyframe_weights.argtypes = [C.c_void_p, C.c_int32]
        L.ellc_accumulate_weights.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
        L.ellc_finalise_weights.argtypes = [C.c_void_p, C.c_int32]
        L.ellc_upload_keyframe_weights.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        L.ellc_read_keyframe_weights.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.POINTER(C.c_int32)]
        L.ellc_read_frame_weights.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
        L.ellc_prepare_keyframes_lc.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.ellc_prepare_keyframes_lc_async.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.ellc_upload_keyframe_hypotheses.argtypes = [C.c_void_p, C.c_int32] + [C.c_void_p] * 5
        L.ellc_read_keyframe_occupancy.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_float)]
        L.ellc_read_keyframe_depth.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
        L.ellc_frame_histograms.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        L.ellc_lc_gate.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_float, C.c_float, C.c_void_p]
        L.ellc_selftest_division.argtypes = [C.c_void_p, C.c_int64, C.c_uint64, C.POINTER(C.c_int64)]
        L.ellc_selftest_unzero.argtypes = [C.c_void_p, C.c_int64, C.c_uint64, C.POINTER(C.c_int64)]
        L.ellc_stream_of.restype = C.c_void_p
        L.ellc_stream_of.argtypes = [C.c_void_p, C.c_int32]
        L.ellc_last_track_kernel_ms.restype = C.c_float
        L.ellc_last_track_kernel_ms.argtypes = [C.c_void_p]
        L.ellc_batch_kernel_ms.restype = C.c_float
        L.ellc_batch_kernel_ms.argtypes = [C.c_void_p, C.c_int32]
        L.ellc_prepare_async.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]
        L.ellc_batch_interval_ms.restype = C.c_float
        L.ellc_batch_interval_ms.argtypes = [C.c_void_p, C.c_int32]
        L.ellc_fence.argtypes = [C.c_void_p]
        L.ellc_exchange_create.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
        L.ellc_exchange_attach_ipc.argtypes = [C.c_void_p, C.c_void_p]
        L.ellc_exchange_attach_local.argtypes = [C.c_void_p, C.c_void_p]
        L.ellc_track_batch_exchange.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int64)]
        L.ellc_exchange_wait.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
        L.ellc_exchange_destroy.argtypes = [C.c_void_p]
        L.ellc_se3_exp_closed.argtypes = [C.c_void_p] * 2
        L.ellc_gn_iterate.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.POINTER(DisplayPlanes)]
        L.ellc_hessian_inverse.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32)]
        L.ellc_lc_generate_pairs.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_float, C.c_float, C.c_int32,
                                             C.POINTER(C.c_int32), C.c_void_p, C.c_void_p, C.c_void_p]
        L.ellc_track_generated_pairs.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.ellc_se3_log_closed.restype = C.c_int
        L.ellc_optimal_new_camera_matrix.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_double, C.c_void_p]
        L.ellc_set_camera.argtypes = [C.c_void_p, C.POINTER(Camera)]
        L.ellc_ingest_frames.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32]
        L.ellc_ingest_keyframe.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        L.ellc_read_camera_tables.argtypes = [C.c_void_p] + [C.c_void_p] * 4
        L.ellc_se3_log_closed.argtypes = [C.c_void_p] * 2
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def default_config(width, height, **over):
    cfg = Config()
    lib().ellc_default_config(C.byref(cfg), int(width), int(height))
    for k, v in over.items():
        if k in ("max_iter", "weight"):
            arr = getattr(cfg, k)
            for i, x in enumerate(v):
                arr[i] = x
        else:
            setattr(cfg, k, v)
    return cfg


def optimal_new_camera_matrix(K, dist, width, height, alpha):
    """cv::getOptimalNewCameraMatrix(K, dist, (width, height), alpha) of OpenCV 3.0.0 (host code)."""
    K = np.ascontiguousarray(np.asarray(K, np.float64).reshape(9)); d = np.ascontiguousarray(np.asarray(dist, np.float64).reshape(5))
    out = np.empty(9, np.float64)
    rc = lib().ellc_optimal_new_camera_matrix(_p(K), _p(d), int(width), int(height), float(alpha), _p(out))
    if rc != 0:
        raise EllcError(f"ellc_optimal_new_camera_matrix failed ({rc})")
    return out.reshape(3, 3)


def make_camera(width, height, channels=3, undistort=False, K=None, dist=None, new_K=None, pitch=None):
    """An ellc_camera record; K / dist / new_K only matter with undistort."""
    cam = Camera()
    cam.width, cam.height, cam.channels = int(width), int(height), int(channels)
    cam.pitch = int(pitch) if pitch is not None else int(width) * int(channels)
    cam.undistort = 1 if undistort else 0
    for name, v, n in (("K", K, 9), ("dist", dist, 5), ("new_K", new_K, 9)):
        if v is not None:
            arr = getattr(cam, name)
            for i, x in enumerate(np.asarray(v, np.float64).reshape(n)):
                arr[i] = float(x)
    return cam


def concat_relative(a, b):
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    out = np.empty(6, np.float32)
    lib().ellc_concat_relative(_p(a), _p(b), _p(out))
    return out


def concat_origin(a, b):
    a = np.ascontiguousarray(a, np.float32); b = np.ascontiguousarray(b, np.float32)
    out = np.empty(6, np.float32)
    lib().ellc_concat_origin(_p(a), _p(b), _p(out))
    return out


def se3_exp(pose):
    pose = np.ascontiguousarray(pose, np.float32)
    out = np.empty(16, np.float32)
    lib().ellc_se3_exp(_p(pose), _p(out))
    return out.reshape(4, 4)


def se3_exp_closed(pose):
    """The FAST flavour's closed-form exp(hat(pose)) (rows 0..2 + [0 0 0 1]); small rotations only."""
    pose = np.ascontiguousarray(pose, np.float32)
    out = np.empty(16, np.float32)
    lib().ellc_se3_exp_closed(_p(pose), _p(out))
    return out.reshape(4, 4)


def se3_log_closed(T):
    """The FAST flavour's closed-form logarithm of a rigid 4x4; None when the rotation is outside its small-angle range."""
    T = np.ascontiguousarray(np.asarray(T, np.float32).reshape(16))
    out = np.empty(6, np.float32)
    ok = lib().ellc_se3_log_closed(_p(T), _p(out))
    return out if ok == 1 else None


class Tracker:
    """Thin owner of one ellc_handle (CUDA streams + device pools)."""

    def __init__(self, cfg):
        self.cfg = cfg
        self._h = C.c_void_p()
        rc = lib().ellc_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            raise EllcError(f"ellc_create failed ({rc}): {lib().ellc_last_error_string(None).decode()}")

    def close(self):
        if self._h:
            lib().ellc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != 0:
            raise EllcError(f"ellc call failed ({rc}): {lib().ellc_last_error_string(self._h).decode()}")

    # -- uploads from host memory
    def upload_frame(self, slot, image):
        image = np.ascontiguousarray(image, np.uint8)
        assert image.shape == (self.cfg.height, self.cfg.width)
        self._keep = getattr(self, "_keep", [])
        self._keep.append(image)
        self._chk(lib().ellc_upload_frame(self._h, slot, _p(image)))

    def upload_keyframe(self, slot, image, depth, var):
        image = np.ascontiguousarray(image, np.uint8)
        d = [np.ascontiguousarray(a, np.float32) for a in depth]
        v = [np.ascontiguousarray(a, np.float32) for a in var]
        dp = (C.c_void_p * LEVELS)(*[_p(a) for a in d])
        vp = (C.c_void_p * LEVELS)(*[_p(a) for a in v])
        self._keep = getattr(self, "_keep", [])
        self._keep += [image] + d + v
        self._chk(lib().ellc_upload_keyframe(self._h, slot, _p(image), dp, vp))

    # -- camera images (gray + undistortion + resize on the device)
    def set_camera(self, cam):
        self._cam = cam
        self._chk(lib().ellc_set_camera(self._h, C.byref(cam)))

    def _camera_image(self, img):
        """(pointer, on_device, object to keep alive) of one camera image: a numpy array (host) or a CUDA torch tensor (device),
        (height, width, channels) or (height, width) uint8, rows contiguous (the camera's pitch = width * channels)."""
        cam = self._cam
        shape = (cam.height, cam.width) if cam.channels == 1 else (cam.height, cam.width, cam.channels)
        if cam.pitch != cam.width * cam.channels:
            raise EllcError("the Python binding takes unpadded images (pitch = width * channels); the C-ABI takes any pitch")
        if type(img).__module__.startswith("torch"):
            import torch
            if not img.is_cuda or img.dtype != torch.uint8 or not img.is_contiguous() or tuple(img.shape) != shape:
                raise EllcError(f"camera tensor must be a contiguous uint8 CUDA tensor of shape {shape}")
            return img.data_ptr(), 1, img
        a = np.ascontiguousarray(img, np.uint8)
        if a.shape != shape:
            raise EllcError(f"camera image shape {a.shape} != {shape}")
        return a.ctypes.data, 0, a

    def ingest_frames(self, slots, images):
        """Camera images (all numpy, or all CUDA torch tensors) -> level-0 images of these frame slots."""
        s = np.ascontiguousarray(slots, np.int32)
        got = [self._camera_image(im) for im in images]
        if len({g[1] for g in got}) > 1:
            raise EllcError("mixed host and device camera images in one call")
        if got and got[0][1] == 1:
            import torch
            torch.cuda.current_stream().synchronize()           # the images must be complete: the library reads them on its own streams
        ptrs = (C.c_void_p * max(1, len(got)))(*[g[0] for g in got])
        self._keep = getattr(self, "_keep", []) + [g[2] for g in got]
        self._chk(lib().ellc_ingest_frames(self._h, len(s), _p(s), ptrs, got[0][1] if got else 0))

    def ingest_keyframe(self, slot, image, depth, var):
        ptr, dev, keep = self._camera_image(image)
        if dev:
            import torch
            torch.cuda.current_stream().synchronize()
        d = [np.ascontiguousarray(a, np.float32) for a in depth]
        v = [np.ascontiguousarray(a, np.float32) for a in var]
        dp = (C.c_void_p * LEVELS)(*[_p(a) for a in d])
        vp = (C.c_void_p * LEVELS)(*[_p(a) for a in v])
        self._keep = getattr(self, "_keep", []) + [keep] + d + v
        self._chk(lib().ellc_ingest_keyframe(self._h, int(slot), C.c_void_p(ptr), dev, dp, vp))

    def read_camera_tables(self):
        """(tap_x [width, 2], tap_y [height, 2], map_xy [2h, 2w, 2], map_frac [2h, 2w]) as the ingestion kernel reads them."""
        w, h = self.cfg.width, self.cfg.height
        tx = np.zeros((w, 2), np.int32); ty = np.zeros((h, 2), np.int32)
        xy = np.zeros((2 * h, 2 * w, 2), np.int16); fr = np.zeros((2 * h, 2 * w), np.uint16)
        self._chk(lib().ellc_read_camera_tables(self._h, _p(tx), _p(ty), _p(xy), _p(fr)))
        return tx, ty, xy, fr

    def synchronize(self):
        self._chk(lib().ellc_synchronize(self._h))
        self._keep = []

    # -- device-resident inputs
    def frame_image_devptr(self, slot):
        p = C.c_void_p()
        self._chk(lib().ellc_frame_image_devptr(self._h, slot, C.byref(p)))
        return p.value

    def keyframe_devptrs(self, slot):
        pi, pd, pv = C.c_void_p(), C.c_void_p(), C.c_void_p()
        off = (C.c_int64 * (LEVELS + 1))()
        self._chk(lib().ellc_keyframe_devptrs(self._h, slot, C.byref(pi), C.byref(pd), C.byref(pv), off))
        return pi.value, pd.value, pv.value, list(off)

    def prepare_frames(self, slots):
        s = np.ascontiguousarray(slots, np.int32)
        self._chk(lib().ellc_prepare_frames(self._h, len(s), _p(s)))

    def prepare_keyframes(self, slots):
        s = np.ascontiguousarray(slots, np.int32)
        self._chk(lib().ellc_prepare_keyframes(self._h, len(s), _p(s)))

    # -- hot path
    @staticmethod
    def make_pairs(kf_slots, frame_slots, init_poses=None, flags=0):
        n = len(kf_slots)
        pairs = np.zeros(n, PAIR_DTYPE)
        pairs["kf_slot"] = kf_slots
        pairs["frame_slot"] = frame_slots
        if init_poses is not None:
            pairs["init_pose"] = np.asarray(init_poses, np.float32).reshape(n, 6)
        pairs["flags"] = flags
        return pairs

    def track_batch(self, pairs, want_trace=False):
        pairs = np.ascontiguousarray(pairs, PAIR_DTYPE)
        n = len(pairs)
        res = np.zeros(n, RESULT_DTYPE)
        tr = np.zeros((n, LEVELS, MAX_TRACE_ITERS), TRACE_DTYPE) if want_trace else None
        self._chk(lib().ellc_track_batch(self._h, n, _p(pairs), _p(res), _p(tr)))
        self._keep = []
        return (res, tr) if want_trace else res

    def track_batch_async(self, pairs):
        pairs = np.ascontiguousarray(pairs, PAIR_DTYPE)
        dres = C.c_void_p()
        self._chk(lib().ellc_track_batch_async(self._h, len(pairs), _p(pairs), C.byref(dres)))
        # host arrays of the uploads issued so far must outlive their copies: they are released when the records of this batch
        # (which was enqueued behind those copies) have been fetched
        self._keep_inflight = getattr(self, "_keep_inflight", [])
        self._keep_inflight.append(getattr(self, "_keep", []))
        self._keep = []
        return dres.value

    def results_download(self, device_ptr, n):
        res = np.zeros(n, RESULT_DTYPE)
        self._chk(lib().ellc_results_download(self._h, device_ptr, n, _p(res)))
        if getattr(self, "_keep_inflight", None):
            self._keep_inflight.pop(0)
        return res

    def gn_evaluate(self, kf_slot, frame_slot, level, pose, want_weights=False):
        pose = np.ascontiguousarray(pose, np.float32)
        out = np.zeros(1, TRACE_DTYPE)
        w = None
        if want_weights:
            cols, rows = self.level_dims(level)[2:]
            w = np.zeros((rows, cols), np.float32)
        self._chk(lib().ellc_gn_evaluate(self._h, kf_slot, frame_slot, level, _p(pose), _p(out), _p(w)))
        return (out[0], w) if want_weights else out[0]

    def gn_iterate(self, kf_slot, frame_slot, level, pose, variant=VARIANT_FORWARD, update=True, want_weights=False, want_display=False):
        """One iteration of a reference per-level driver (ellc_gn_iterate).  Returns the trace record, plus the weight image and /
        or a dict of the display planes when asked for."""
        pose = np.ascontiguousarray(pose, np.float32)
        out = np.zeros(1, TRACE_DTYPE)
        cols, rows = self.level_dims(level)[2:]
        w = np.zeros((rows, cols), np.float32) if want_weights else None
        planes, dp = None, None
        if want_display:
            planes = {k: np.zeros((rows, cols), np.float32) for k in ("warped_image", "iteration_residual", "warped_x", "warped_y")}
            dp = DisplayPlanes(*[planes[k].ctypes.data for k in ("warped_image", "iteration_residual", "warped_x", "warped_y")])
        self._chk(lib().ellc_gn_iterate(self._h, kf_slot, frame_slot, level, int(variant), 1 if update else 0, _p(pose), _p(out), _p(w),
                                        C.byref(dp) if dp is not None else None))
        ret = [out[0]]
        if want_weights:
            ret.append(w)
        if want_display:
            ret.append(planes)
        return ret[0] if len(ret) == 1 else tuple(ret)

    def hessian_inverse(self, H):
        H = np.ascontiguousarray(np.asarray(H, np.float32).reshape(36))
        out = np.zeros(36, np.float32)
        ok = C.c_int32()
        self._chk(lib().ellc_hessian_inverse(self._h, _p(H), _p(out), C.byref(ok)))
        return out.reshape(6, 6), bool(ok.value)

    def solve_update(self, H, b, pose):
        H = np.ascontiguousarray(np.asarray(H, np.float32).reshape(36))
        b = np.ascontiguousarray(b, np.float32); pose = np.ascontiguousarray(pose, np.float32)
        po = np.empty(6, np.float32); de = np.empty(6, np.float32); wp = C.c_float()
        self._chk(lib().ellc_solve_update(self._h, _p(H), _p(b), _p(pose), _p(po), _p(de), C.byref(wp)))
        return po, de, wp.value

    def solve_update_rt(self, H, b, pose):
        """solve_update + rows 0..2 of exp(hat(new pose)) exactly as K5 hands them to the next iteration."""
        H = np.ascontiguousarray(np.asarray(H, np.float32).reshape(36))
        b = np.ascontiguousarray(b, np.float32); pose = np.ascontiguousarray(pose, np.float32)
        po = np.empty(6, np.float32); de = np.empty(6, np.float32); wp = C.c_float(); rt = np.empty(12, np.float32)
        self._chk(lib().ellc_solve_update_rt(self._h, _p(H), _p(b), _p(pose), _p(po), _p(de), C.byref(wp), _p(rt)))
        return po, de, wp.value, rt

    # -- read-back
    def level_dims(self, level):
        a, b, c, d = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        self._chk(lib().ellc_level_dims(self._h, level, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return a.value, b.value, c.value, d.value

    def read_frame_level(self, slot, level):
        pw, ph, cols, rows = self.level_dims(level)
        img = np.empty((ph, pw), np.uint8); gx = np.empty((rows, cols), np.float32); gy = np.empty((rows, cols), np.float32)
        self._chk(lib().ellc_read_frame_level(self._h, slot, level, _p(img), _p(gx), _p(gy)))
        return img, gx, gy

    def read_keyframe_level(self, slot, level):
        pw, ph, cols, rows = self.level_dims(level)
        img = np.empty((ph, pw), np.uint8); mask = np.empty((rows, cols), np.uint8); cnt = C.c_int32()
        self._chk(lib().ellc_read_keyframe_level(self._h, slot, level, _p(img), _p(mask), C.byref(cnt)))
        return img, mask, cnt.value

    # -- introspection
    def launch_count(self):
        return lib().ellc_launch_count(self._h)

    def reset_launch_count(self):
        lib().ellc_reset_launch_count(self._h)

    def stream(self):
        return lib().ellc_stream(self._h)

    # -- keyframe from depth hypotheses (depth / variance pyramids built on the device)
    def upload_keyframe_hypotheses(self, slot, image, valid, inv_depth_smoothed, variance_smoothed, want_valid_out=False):
        image = np.ascontiguousarray(image, np.uint8)
        valid = np.ascontiguousarray(valid, np.uint8)
        idep = np.ascontiguousarray(inv_depth_smoothed, np.float32)
        vs = np.ascontiguousarray(variance_smoothed, np.float32)
        assert image.shape == valid.shape == idep.shape == vs.shape == (self.cfg.height, self.cfg.width)
        vout = np.zeros_like(valid) if want_valid_out else None
        self._keep = getattr(self, "_keep", []) + [image, valid, idep, vs]
        self._chk(lib().ellc_upload_keyframe_hypotheses(self._h, slot, _p(image), _p(valid), _p(idep), _p(vs), _p(vout) if want_valid_out else None))
        return vout

    def read_keyframe_occupancy(self, slot):
        n, occ = C.c_int32(), C.c_float()
        self._chk(lib().ellc_read_keyframe_occupancy(self._h, slot, C.byref(n), C.byref(occ)))
        return n.value, occ.value

    def read_keyframe_depth(self, slot, level):
        shape = (self.cfg.height >> level, self.cfg.width >> level)
        d, v = np.zeros(shape, np.float32), np.zeros(shape, np.float32)
        self._chk(lib().ellc_read_keyframe_depth(self._h, slot, level, _p(d), _p(v)))
        return d, v

    # -- loop-closure candidate gating
    def frame_histograms(self, frame_slots):
        fs = np.ascontiguousarray(frame_slots, np.int32)
        out = np.zeros((len(fs), 256), np.float32)
        self._chk(lib().ellc_frame_histograms(self._h, len(fs), _p(fs), _p(out)))
        return out

    def lc_gate(self, loop_slots, test_slots, loop_poses, test_poses, match_threshold=0.1, max_rel_view_angle=10.0):
        n = len(loop_slots)
        cand = np.zeros(n, LC_CAND_DTYPE)
        cand["loop_frame_slot"] = loop_slots; cand["test_frame_slot"] = test_slots
        cand["loop_pose_world"] = np.asarray(loop_poses, np.float32).reshape(n, 6)
        cand["test_pose_world"] = np.asarray(test_poses, np.float32).reshape(n, 6)
        out = np.zeros(n, LC_STATS_DTYPE)
        self._chk(lib().ellc_lc_gate(self._h, n, _p(cand), float(match_threshold), float(max_rel_view_angle), _p(out)))
        return out

    def lc_generate_pairs(self, ring, queries, min_match_difference=8, match_threshold=0.1, max_rel_view_angle=10.0, pair_flags=0):
        """findMatch's ring walk + gating for all queries on the device.  Returns (pairs, stats, query_of_pair); the list also
        stays on the device for track_generated_pairs()."""
        ring = np.ascontiguousarray(ring, LC_RING_DTYPE); queries = np.ascontiguousarray(queries, LC_QUERY_DTYPE)
        cap = max(1, len(ring) * len(queries))
        pairs = np.zeros(cap, PAIR_DTYPE); stats = np.zeros(cap, LC_STATS_DTYPE); qi = np.zeros(cap, np.int32)
        n = C.c_int32()
        self._chk(lib().ellc_lc_generate_pairs(self._h, len(ring), _p(ring), len(queries), _p(queries), int(min_match_difference),
                                               float(match_threshold), float(max_rel_view_angle), int(pair_flags), C.byref(n), _p(pairs), _p(stats), _p(qi)))
        return pairs[:n.value], stats[:n.value], qi[:n.value]

    def track_generated_pairs(self, n_pairs):
        res = np.zeros(n_pairs, RESULT_DTYPE)
        self._chk(lib().ellc_track_generated_pairs(self._h, int(n_pairs), _p(res)))
        return res

    # -- constant-weight loop-closure variant
    def reset_keyframe_weights(self, kf_slot):
        self._chk(lib().ellc_reset_keyframe_weights(self._h, kf_slot))

    def accumulate_weights(self, kf_slot, frame_slots):
        fs = np.ascontiguousarray(frame_slots, np.int32)
        self._chk(lib().ellc_accumulate_weights(self._h, kf_slot, len(fs), _p(fs)))

    def finalise_weights(self, kf_slot):
        self._chk(lib().ellc_finalise_weights(self._h, kf_slot))

    def upload_keyframe_weights(self, kf_slot, weights, counts=None):
        keep = [np.ascontiguousarray(w, np.float32) for w in weights]
        ptrs = (C.c_void_p * 4)(*[_p(w) for w in keep])
        cnt = np.ascontiguousarray(counts, np.int32) if counts is not None else None
        self._chk(lib().ellc_upload_keyframe_weights(self._h, kf_slot, ptrs, _p(cnt) if cnt is not None else None))

    def read_keyframe_weights(self, kf_slot, level):
        out = np.zeros((self.cfg.height >> level, self.cfg.width >> level), np.float32)
        cnt = C.c_int32()
        self._chk(lib().ellc_read_keyframe_weights(self._h, kf_slot, level, _p(out), C.byref(cnt)))
        return out, cnt.value

    def read_frame_weights(self, frame_slot, level):
        out = np.zeros((self.cfg.height >> level, self.cfg.width >> level), np.float32)
        self._chk(lib().ellc_read_frame_weights(self._h, frame_slot, level, _p(out)))
        return out

    def prepare_keyframes_lc(self, kf_slots):
        ks = np.ascontiguousarray(kf_slots, np.int32)
        self._chk(lib().ellc_prepare_keyframes_lc(self._h, len(ks), _p(ks)))

    def prepare_keyframes_lc_async(self, kf_slots):
        ks = np.ascontiguousarray(kf_slots, np.int32)
        self._chk(lib().ellc_prepare_keyframes_lc_async(self._h, len(ks), _p(ks)))

    def selftest_division(self, n, seed=1):
        out = (C.c_int64 * 2)()
        self._chk(lib().ellc_selftest_division(self._h, int(n), int(seed), out))
        return int(out[0]), int(out[1])

    def selftest_unzero(self, n, seed=1):
        out = C.c_int64(0)
        self._chk(lib().ellc_selftest_unzero(self._h, int(n), int(seed), C.byref(out)))
        return int(out.value)

    def stream_of(self, which):
        return lib().ellc_stream_of(self._h, which)

    def last_track_kernel_ms(self):
        return lib().ellc_last_track_kernel_ms(self._h)

    def batch_kernel_ms(self, batches_ago=0):
        return lib().ellc_batch_kernel_ms(self._h, int(batches_ago))

    def batch_interval_ms(self, batches_ago=0):
        return lib().ellc_batch_interval_ms(self._h, int(batches_ago))

    def fence(self):
        self._chk(lib().ellc_fence(self._h))

    # -- multi-GPU result exchange (NVLink peer memory)
    def exchange_create(self, rank, world, capacity):
        buf = np.zeros(IPC_HANDLE_BYTES, np.uint8)
        self._chk(lib().ellc_exchange_create(self._h, int(rank), int(world), int(capacity), _p(buf)))
        return buf

    def exchange_attach_ipc(self, handles):
        hs = np.ascontiguousarray(np.asarray(handles, np.uint8).reshape(-1))
        self._chk(lib().ellc_exchange_attach_ipc(self._h, _p(hs)))

    def exchange_attach_local(self, trackers):
        arr = (C.c_void_p * len(trackers))(*[t._h for t in trackers])
        self._chk(lib().ellc_exchange_attach_local(self._h, arr))

    def track_batch_exchange(self, pairs, global_index, n_total, root=-1):
        pairs = np.ascontiguousarray(pairs, PAIR_DTYPE)
        gi = np.ascontiguousarray(global_index, np.int32)
        assert len(gi) == len(pairs)
        tok = C.c_int64()
        self._chk(lib().ellc_track_batch_exchange(self._h, len(pairs), _p(pairs), _p(gi), int(n_total), int(root), C.byref(tok)))
        self._keep_inflight = getattr(self, "_keep_inflight", [])
        self._keep_inflight.append(getattr(self, "_keep", []))
        self._keep = []
        return tok.value

    def exchange_wait(self, token, n_total=None, out=None):
        """Wait for the batch `token`; on a receiving rank returns the n_total gathered records (global pair order)."""
        res = out if out is not None else (np.zeros(n_total, RESULT_DTYPE) if n_total else None)
        self._chk(lib().ellc_exchange_wait(self._h, int(token), _p(res) if res is not None else None))
        if getattr(self, "_keep_inflight", None):
            self._keep_inflight.pop(0)
        return res

    def exchange_destroy(self):
        self._chk(lib().ellc_exchange_destroy(self._h))

    def prepare_async(self, frame_slots, kf_slots):
        """Preparation of these slots on the low-priority preparation stream (overlaps the batch that is tracking now)."""
        f = np.ascontiguousarray(frame_slots, np.int32); k = np.ascontiguousarray(kf_slots, np.int32)
        self._chk(lib().ellc_prepare_async(self._h, len(f), _p(f), len(k), _p(k)))
