"""Generates tests/golden/reference_live_calls.npz: what the reference's own code returned to every call that the comparison tests
of tests/test_reference_pin.py make on it (the tests that take the `R` fixture: samplers, pyramid / gradient / mask stages with
NaN / -1 / -0 / inf depths, pose algebra, the all-out-of-bounds start and the keyframe without depth, both loop-closure modes,
the randomised sweep, the 640x480 pairs).

With the library (oracle/_ref/libellc_ref*.so, see oracle/refbinding.py) those tests call it live and also check every call
against this file; without it they compare the oracle with this file.  Each call is stored under "<test id>/<n>" as a JSON
description of the returned structure; its arrays sit in one flat pool per dtype ("pool_<dtype>"), and arrays above DIGEST_BYTES
are stored as SHA-256 digests of their bytes.

    python tests/golden/make_reference_live_golden.py                # from the reference's library
    python tests/golden/make_reference_live_golden.py --from-oracle  # from the oracle, where the library cannot be built

--from-oracle records what the oracle returns in the reference's place.  It is only a record of the reference where the oracle is
bit-identical to the reference on exactly these inputs, which is what these tests assert when the library is present; the file
names its source in its "source" entry.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
PATH = os.path.join(HERE, "reference_live_calls.npz")
DIGEST_BYTES = 16384


def digest(a):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


class Digest(str):
    """An array the file holds as the SHA-256 of its bytes."""


def same(want, got):
    """`want` from the file (an array, or a Digest of one) against an array computed now."""
    if isinstance(want, Digest):
        return want == digest(got)
    return np.array_equal(want, got)


def _pack(x, pools):
    if isinstance(x, dict):
        return {"d": {k: _pack(v, pools) for k, v in x.items()}}
    if isinstance(x, (list, tuple)):
        return {"l": [_pack(v, pools) for v in x], "t": isinstance(x, tuple)}
    if isinstance(x, (np.ndarray, np.generic)):
        a = np.asarray(x)
        if a.nbytes > DIGEST_BYTES:
            return {"sha": digest(a)}
        pool = pools.setdefault(a.dtype.str, [])
        off = sum(p.size for p in pool)
        pool.append(a.reshape(-1))
        return {"a": [a.dtype.str, off, list(a.shape)], "s": isinstance(x, np.generic)}
    return {"v": x}


def _unpack(s, pools):
    if "d" in s:
        return {k: _unpack(v, pools) for k, v in s["d"].items()}
    if "l" in s:
        v = [_unpack(x, pools) for x in s["l"]]
        return tuple(v) if s["t"] else v
    if "sha" in s:
        return Digest(s["sha"])
    if "a" in s:
        dt, off, shape = s["a"]
        a = pools["pool_" + dt][off:off + int(np.prod(shape, dtype=np.int64))].reshape(shape)
        return a[()] if s["s"] else a
    return s["v"]


def _agree(want, got):
    if isinstance(want, dict):
        return set(want) == set(got) and all(_agree(want[k], got[k]) for k in want)
    if isinstance(want, (list, tuple)):
        return len(want) == len(got) and all(_agree(w, g) for w, g in zip(want, got))
    if isinstance(want, (np.ndarray, np.generic, Digest)):
        return same(want, got) or (np.asarray(want).dtype.kind == "f" and np.array_equal(want, got, equal_nan=True))
    return want == got


class Recorder:
    """Calls `impl` (refbinding or OracleAsReference) and keeps what every call returned, in call order."""

    def __init__(self, impl, test_id, meta, pools):
        self.impl, self.test_id, self.meta, self.pools, self.n = impl, test_id, meta, pools, 0

    def __getattr__(self, name):
        def call(*args, **kw):
            out = getattr(self.impl, name)(*args, **kw)
            key = f"{self.test_id}/{self.n}"
            self.meta[key] = {"f": name, "r": _pack(out, self.pools)}
            self.n += 1
            return out
        return call


class Replay:
    """Returns the recorded results of test `test_id`, call by call.  With `live` (the reference's library) it calls the library
    instead, checks that it returns what the file holds, and returns the library's result."""

    def __init__(self, test_id, live=None, path=PATH):
        z = np.load(path)
        self.meta = json.loads(str(z["meta"]))
        self.pools = {k: z[k] for k in z.files if k.startswith("pool_")}
        self.test_id, self.live, self.n = test_id, live, 0

    def __getattr__(self, name):
        def call(*args, **kw):
            key = f"{self.test_id}/{self.n}"
            self.n += 1
            assert key in self.meta and self.meta[key]["f"] == name, f"{key}: no recorded call of {name}"
            want = _unpack(self.meta[key]["r"], self.pools)
            if self.live is None:
                return want
            got = getattr(self.live, name)(*args, **kw)
            assert _agree(want, got), f"{key}: the reference's {name} no longer returns what {os.path.basename(PATH)} holds"
            return got
        return call


class OracleAsReference:
    """The calls of oracle/refbinding.py that the tests make, answered by the oracle (same return structures and dtypes)."""

    def __init__(self):
        import oracle
        self.o = oracle
        g = np.load(os.path.join(HERE, "reference_track_480x270.npz"))
        g640 = np.load(os.path.join(HERE, "reference_track_640x480.npz"))
        self.variants = {"default": (int(g["width"][0]), int(g["height"][0]), g["intr"]), "640x480": (640, 480, g640["intr"])}
        self.variant = "default"

    def select(self, variant="default"):
        prev, self.variant = self.variant, variant
        return prev

    def dims(self):
        w, h, k = self.variants[self.variant]
        return dict(width=w, height=h, fx=np.float32(k[0]), fy=np.float32(k[1]), cx=np.float32(k[2]), cy=np.float32(k[3]))

    def _cfg(self, **over):
        k = self.dims()
        return self.o.default_config(k["width"], k["height"], fx=float(k["fx"]), fy=float(k["fy"]), cx=float(k["cx"]), cy=float(k["cy"]), **over)

    def frame_level(self, image, level, depth_level=None):
        k = self.dims()
        rows, cols = k["height"] >> level, k["width"] >> level
        img = self.o.image_pyramid(image)[level]
        gx, gy = self.o.gradient(img, rows, cols)
        out = dict(image=img, gradx=gx, grady=gy)
        if depth_level is not None:
            mask, count = self.o.mask_count(depth_level)
            out.update(mask=mask, count=count)
        return out

    def interpolate(self, image, level, xs, ys):
        lvl = self.o.image_pyramid(image)[level]
        rows, cols = image.shape[0] >> level, image.shape[1] >> level
        gx, gy = self.o.gradient(lvl, rows, cols)
        i = np.array([self.o.interp_u8(lvl, x, y, 1, rows, cols) for x, y in zip(xs, ys)], np.float32)
        return (i, np.array([self.o.interp_f32(gx, x, y) for x, y in zip(xs, ys)], np.float32),
                np.array([self.o.interp_f32(gy, x, y) for x, y in zip(xs, ys)], np.float32))

    def concat_relative(self, a, b):
        return self.o.concat_relative(a, b)

    def concat_origin(self, a, b):
        return self.o.concat_origin(a, b)

    @staticmethod
    def _trace(pose, tr):
        levels = [[dict(H=np.asarray(it["H"], np.float32).reshape(6, 6), b=np.asarray(it["b"], np.float32),
                        weighted_pose=np.float32(it["weighted_pose"]), pose_after=np.asarray(it["pose_after"], np.float32))
                   for it in tr["levels"][l]] for l in range(4)]
        return dict(n_selected=list(tr["n_selected"]), n_iters=list(tr["n_iters"]), levels=levels, final_pose=np.asarray(pose, np.float32))

    def track_trace(self, kf_image, cur_image, depth_pyr, var_pyr, init_pose, want_weights=False):
        if want_weights:
            pose, tr, wl = self.o.track_with_weights(self._cfg(), kf_image, cur_image, depth_pyr, var_pyr, init_pose)
            return dict(self._trace(pose, tr), weights_l0=wl[0])
        pose, tr = self.o.track(self._cfg(), kf_image, cur_image, depth_pyr, var_pyr, init_pose)
        return self._trace(pose, tr)

    def get_image_pose_estimate(self, kf_image, cur_image, depth_pyr, var_pyr, tminus1_pose_wrt_world):
        zero = np.zeros(6, np.float32)                 # the keyframe at the world origin, as in ref_driver.cpp
        pose, _ = self.o.track(self._cfg(), kf_image, cur_image, depth_pyr, var_pyr, self.o.concat_origin(tminus1_pose_wrt_world, zero),
                               want_trace=False)
        return pose, self.o.concat_relative(pose, zero), self.o.concat_relative(pose, zero)

    def lc_flow(self,kf_image, seq_images, seq_tminus1, depth_pyr, var_pyr, lc_image, lc_tminus1, parallel=True):
        cfg = self._cfg(lc_parallel=int(bool(parallel)))
        k = self.dims()
        zero = np.zeros(6, np.float32)
        wp = [np.zeros((k["height"] >> l, k["width"] >> l), np.float32) for l in range(4)]
        cnt, poses = [0] * 4, []
        for img, tm1 in zip(seq_images, seq_tminus1):
            pose, _, wl = self.o.track_with_weights(cfg, kf_image, img, depth_pyr, var_pyr, self.o.concat_origin(tm1, zero))
            self.o.accumulate_weights(wp, cnt, wl)
            poses.append(pose)
        wf = self.o.finalise_weights(wp, cnt)
        pose, tr = self.o.track_lc(cfg, kf_image, lc_image, depth_pyr, wf, self.o.concat_origin(lc_tminus1, zero))
        return dict(weights=wf, counts=list(cnt), seq_poses=np.stack(poses).astype(np.float32), lc_pose=np.asarray(pose, np.float32),
                    lc_trace=self._trace(pose, tr))


def main():
    sys.path.insert(0, ROOT)
    import oracle
    from oracle import refbinding
    from tests import test_reference_pin as T
    from tests.helpers import make_case
    from_oracle = "--from-oracle" in sys.argv[1:]
    if from_oracle:
        impl = OracleAsReference()
        source = "the oracle (oracle/ellc_oracle.cpp) in the reference's place, on inputs where it is bit-identical to the reference"
    else:
        refbinding.build(); refbinding.build(variant="640x480")
        impl, source = refbinding, "the reference's own sources (oracle/_ref/libellc_ref*.so)"
    oracle.lib()
    fx = np.load(os.path.join(HERE, "reference_track_480x270.npz"))
    fx640 = np.load(os.path.join(HERE, "reference_track_640x480.npz"))
    vga = make_case(640, 480, n_frames=2, seed=23)
    meta, pools = {}, {}
    rec = lambda tid: Recorder(impl, tid, meta, pools)
    T.test_fixture_is_what_the_reference_produces(fx, rec("test_fixture_is_what_the_reference_produces"))
    T.test_reference_stages_vs_oracle(oracle, fx, rec("test_reference_stages_vs_oracle"))
    T.test_reference_samplers_vs_oracle(oracle, fx, rec("test_reference_samplers_vs_oracle"))
    T.test_reference_pose_algebra_vs_oracle(oracle, rec("test_reference_pose_algebra_vs_oracle"))
    T.test_reference_live_random_pairs(oracle, rec("test_reference_live_random_pairs"))
    for parallel in (True, False):
        T.test_reference_live_loop_closure_flow(oracle, fx, parallel, rec(f"test_reference_live_loop_closure_flow[{parallel}]"))
    T.test_reference_live_randomised_sweep(oracle, rec("test_reference_live_randomised_sweep"))
    T.test_fixture_640x480_is_what_the_reference_produces(fx640, rec("test_fixture_640x480_is_what_the_reference_produces"))
    T.test_reference_live_random_pairs_at_640x480(oracle, vga, rec("test_reference_live_random_pairs_at_640x480"))
    np.savez_compressed(PATH, meta=np.array(json.dumps(meta)), source=np.array(source),
                        **{"pool_" + dt: np.concatenate(p) for dt, p in pools.items()})
    print("wrote", PATH, os.path.getsize(PATH), "bytes,", len(meta), "calls")


if __name__ == "__main__":
    main()
