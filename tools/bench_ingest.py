"""Camera-frame ingestion on the GPU (ellc_ingest_frames: gray + undistortion + resize) at batch 512, and its cost next to the tracking
step it feeds.

Part 1, per camera (1920x1080 -> 480x270, 2560x1920 -> 640x480), undistortion off / on, host (pinned) / device sources: ms per batch
of 512 frames (host clock around the call and a device synchronise, median of --reps after a warm-up), the algorithmic bytes (the
32-byte source sectors the taps touch, counted from the tables the library built, + the map entries used, once per batch, + the
output) and their share of the 7.7 TB/s HBM bound.  16 distinct camera images are cycled through the 512 slots (a 512-image host pool
at 2560x1920 would need 7.5 GB of host memory); device pools exceed the 126 MB L2.
Part 2, the flagship workload of bench.py (512 frames against 32 keyframes, 4,608 pairs, 640x480): one step from 2560x1920 device
camera images (ingest + prepare + track) against the plain step (level-0 upload + prepare + track) fed the images the ingestion
produced; the records of both must be identical.

    python tools/bench_ingest.py --out bench_ingest.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
HBM_BPS = 7.7e12
N = 512


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.returncode == 0 else "n/a")


def algorithmic_bytes(t, cam):
    """Per batch: N x (source sectors the taps touch x 32 + output) + the map entries used (once)."""
    tx, ty, mxy, _ = t.read_camera_tables()
    ch, pitch, W, H = cam.channels, cam.pitch, cam.width, cam.height
    if cam.undistort:
        xs, ys = [], []
        for dy in (0, 1):
            for dx in (0, 1):
                x = mxy[..., 0].astype(np.int64) + dx
                y = mxy[..., 1].astype(np.int64) + dy
                ok = (x >= 0) & (x < W) & (y >= 0) & (y < H)
                xs.append(x[ok]); ys.append(y[ok])
        x, y = np.concatenate(xs), np.concatenate(ys)
    else:
        y, x = np.meshgrid(np.unique(ty), np.unique(tx), indexing="ij")
        x, y = x.reshape(-1).astype(np.int64), y.reshape(-1).astype(np.int64)
    first = y * pitch + x * ch
    sectors = np.unique(np.concatenate([(first + c) // 32 for c in range(ch)]))
    w, h = t.cfg.width, t.cfg.height
    map_bytes = 4 * w * h * 8 if cam.undistort else 0
    src = int(sectors.size) * 32
    return dict(source_bytes_per_frame=src, output_bytes_per_frame=w * h, map_bytes=map_bytes,
                bytes_per_batch=N * (src + w * h) + map_bytes, h2d_bytes_per_frame=pitch * H)


def time_calls(fn, sync, reps):
    fn(); sync()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn(); sync()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(np.min(ts))


def part1(capi, mk, reps):
    import torch
    rows = []
    for W, H, w, h in ((1920, 1080, 480, 270), (2560, 1920, 640, 480)):
        rng = np.random.default_rng(W)
        pool = [torch.from_numpy(rng.integers(0, 256, (H, W, 3), dtype=np.uint8)) for _ in range(16)]
        host = [p.pin_memory().numpy() for p in pool]
        dev = [p.cuda() for p in pool]
        K = mk.camera_matrix(W, H)
        t = capi.Tracker(capi.default_config(w, h, max_frames=N, max_keyframes=1))
        slots = list(range(N))
        for ud in (0, 1):
            cam = capi.make_camera(W, H, 3, ud, K, mk.DIST, capi.optimal_new_camera_matrix(K, mk.DIST, W, H, 0.0))
            t.set_camera(cam)
            b = algorithmic_bytes(t, cam)
            for src, imgs in (("host", host), ("device", dev)):
                batch = [imgs[i % 16] for i in range(N)]
                med, best = time_calls(lambda: t.ingest_frames(slots, batch), t.synchronize, reps)
                row = dict(camera=f"{W}x{H}", working=f"{w}x{h}", undistort=ud, source=src, batch=N, ms_per_batch_median=med,
                           ms_per_batch_min=best, **b, hbm_bound_ms=b["bytes_per_batch"] / HBM_BPS * 1e3,
                           share_of_hbm_bound=b["bytes_per_batch"] / HBM_BPS * 1e3 / med)
                if src == "host":
                    row["h2d_gb_per_s"] = N * b["h2d_bytes_per_frame"] / (med * 1e-3) / 1e9
                rows.append(row)
                print(json.dumps(row), flush=True)
        t.close()
        del dev
        torch.cuda.empty_cache()
    return rows


def part2(capi, mk, reps, wl):
    import torch
    from egomotion_with_local_loop_closures_b200 import synth
    w, h, F = 640, 480, 4
    W, H = w * F, h * F
    k = synth.intrinsics(w, h)
    cfg = capi.default_config(w, h, fx=float(k["fx"]), fy=float(k["fy"]), cx=float(k["cx"]), cy=float(k["cy"]), max_frames=N, max_keyframes=32)
    K = mk.camera_matrix(W, H)
    cam = capi.make_camera(W, H, 3, 1, K, mk.DIST, capi.optimal_new_camera_matrix(K, mk.DIST, W, H, 0.0))
    cams = torch.empty((N, H, W, 3), dtype=torch.uint8, device="cuda")                  # F x F-upsampled frames, channels +-3 apart
    gen = torch.Generator("cuda").manual_seed(1)
    for c0 in range(0, N, 32):
        g = torch.from_numpy(np.stack(wl["frames"][c0:c0 + 32])).cuda().to(torch.int16)
        big = g.repeat_interleave(F, 1).repeat_interleave(F, 2)[..., None]
        noise = torch.randint(-3, 4, big.shape[:3] + (3,), device="cuda", dtype=torch.int16, generator=gen)
        cams[c0:c0 + 32] = (big + noise).clamp(0, 255).to(torch.uint8)
    del g, big, noise
    cam_list = [cams[i] for i in range(N)]
    pairs = capi.Tracker.make_pairs(wl["kf_idx"], wl["fr_idx"], wl["init"])
    slots = list(range(N))

    a = capi.Tracker(cfg)
    a.set_camera(cam)
    for i in range(32):
        a.upload_keyframe(i, wl["kf_images"][i], wl["kf_depth"][i], wl["kf_var"][i])
    rec_a = {}

    def step_a():
        a.ingest_frames(slots, cam_list)
        rec_a["r"] = a.track_batch(pairs)
    med_a, min_a = time_calls(step_a, a.synchronize, reps)
    ing_med, ing_min = time_calls(lambda: a.ingest_frames(slots, cam_list), a.synchronize, reps)
    level0 = [a.read_frame_level(i, 0)[0] for i in range(N)]
    from tests import ingest_oracle
    sample_ok = all(np.array_equal(level0[i], ingest_oracle.ingest(cams[i].cpu().numpy(), w, h, True, K, mk.DIST, np.array(cam.new_K).reshape(3, 3)))
                    for i in (0, 1, N - 1))

    b = capi.Tracker(cfg)
    for i in range(32):
        b.upload_keyframe(i, wl["kf_images"][i], wl["kf_depth"][i], wl["kf_var"][i])
    pinned = [torch.from_numpy(im).pin_memory().numpy() for im in level0]
    rec_b = {}

    def step_b():
        for i in range(N):
            b.upload_frame(i, pinned[i])
        rec_b["r"] = b.track_batch(pairs)
    med_b, min_b = time_calls(step_b, b.synchronize, reps)
    track_ms = b.batch_kernel_ms(0)
    out = dict(workload="pair_sweep_640x480 frames from 2560x1920 BGR device camera images, undistortion on", pairs=len(pairs), frames=N,
               step_ingest_ms_median=med_a, step_ingest_ms_min=min_a, step_upload_ms_median=med_b, step_upload_ms_min=min_b,
               ingest_only_ms_median=ing_med, ingest_only_ms_min=ing_min, track_kernel_ms=track_ms,
               ingest_share_of_track_kernel=ing_med / track_ms, records_identical=rec_a["r"].tobytes() == rec_b["r"].tobytes(),
               level0_equals_oracle_on_sample=bool(sample_ok))
    print(json.dumps(out), flush=True)
    a.close(); b.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import bench
    wl = bench.build_workload(32, N, 9, seed=0, conf=bench.CONFIGS["pair_sweep"])      # fork-based rendering: before CUDA starts
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_ingest: no CUDA device (this measurement has no CPU form)")
    import __graft_entry__ as g
    g.build()
    import make_ingest_golden as mk
    from egomotion_with_local_loop_closures_b200 import capi
    res = dict(card=card(), part1=part1(capi, mk, args.reps), part2=part2(capi, mk, args.reps, wl))
    print(json.dumps(res["card"]))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    if not res["part2"]["records_identical"] or not res["part2"]["level0_equals_oracle_on_sample"]:
        sys.exit("bench_ingest: records / level-0 images differ")


if __name__ == "__main__":
    main()
