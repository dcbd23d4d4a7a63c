"""Frame sequences with fixed keyframe depth (BASELINE config 1 and batches of it): the host loop against ellc_track_sequence_steps.

Workloads at 640x480, FAST, keyframe every 8 frames: S = 1, 8, 64 sequences of 100 frames (99 tracks each) and S = 512 sequences of
9 frames (8 tracks each).  The frames come from R rendered trajectories (default 8: 100 frames and 13 keyframes each, ground-truth
keyframe depth, distinct scene textures); sequence s runs trajectory s % R from its own root pose, and the 9-frame sequences start
at keyframe (s // R) % 12 of it.  Sequences that share a trajectory track the same frame-keyframe pairs, so for S > R some pairs
repeat (their images are read from L2 more often than in a workload of S distinct sequences); both arms run the same steps.

Arms, alternated call by call in one process after --warmup calls each:
  host_loop     what a caller does today: per wave (the frame index of every sequence) one ellc_track_batch of the S pairs, then
                ellc_concat_relative / ellc_concat_origin on the host for every sequence (here through ctypes).  `host_loop_track_ms`
                times only the foreign ellc_track_batch calls (pair and result arrays are built before the clock starts): what
                the same loop costs at least, whatever language drives it
  device_chain  one ellc_track_sequence_steps call
Reported per arm: ms per call (host clock around work that ends in a device synchronise), ms per frame (call / tracked frames
per sequence, i.e. per wave),
tracks/s, kernel launches per call, and whether the records and world poses of the two arms are byte-identical.  The card name
and power limit are read in the same run.

    python tools/bench_sequences.py --out profiles/r05_bench_sequences.json
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
KF_INTERVAL = 8
WORKLOADS = ((1, 100), (8, 100), (64, 100), (512, 9))       # (sequences, frames per sequence incl. the first keyframe)


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.returncode == 0 else "n/a")


def render(n_traj, n_frames, workers):
    """n_traj trajectories: frames 1 .. n_frames - 1 and a keyframe at every KF_INTERVAL-th frame (from frame 0)."""
    import bench
    from egomotion_with_local_loop_closures_b200 import synth
    jobs, index = [], []
    for r in range(n_traj):
        T = synth.smooth_trajectory(n_frames, seed_pose=91011 + r)
        for i in range(0, n_frames - 1, KF_INTERVAL):
            jobs.append(("kf", 1234 + r, T[i], 5678 + 100 * r + i)); index.append(("kf", r, i))
        for i in range(1, n_frames):
            jobs.append(("fr", 1234 + r, T[i], 7000 + 100 * r + i)); index.append(("fr", r, i))
    import multiprocessing as mp
    with mp.get_context("fork").Pool(workers) as pool:
        out = pool.map(bench._render_job, jobs, chunksize=max(1, len(jobs) // (4 * workers)))
    return dict(zip(index, out))


def sequence_steps(capi, n_seq, n_frames, n_traj, kf_slot, fr_slot):
    """Steps of S sequences, sequence-major (one sequence's steps in frame order)."""
    rng = np.random.default_rng(5)
    n_starts = (100 - n_frames) // KF_INTERVAL + 1
    per = []
    for s in range(n_seq):
        r, o = s % n_traj, KF_INTERVAL * ((s // n_traj) % n_starts)
        root = (rng.standard_normal(6) * [0.05, 0.05, 0.05, 0.2, 0.2, 0.2]).astype(np.float32)
        L = n_frames - 1
        kf_rel = [KF_INTERVAL * ((j - 1) // KF_INTERVAL) for j in range(1, L + 1)]
        per.append(capi.Tracker.make_steps([kf_slot[(r, o + k)] for k in kf_rel], [fr_slot[(r, o + j)] for j in range(1, L + 1)],
                                           [j - 2 for j in range(1, L + 1)], [k - 1 for k in kf_rel],
                                           prev_world=[root] * L, kf_world=[root] * L))
    base = np.cumsum([0] + [len(p) for p in per])
    steps = np.concatenate(per)
    for s, p in enumerate(per):
        for f in ("prev_step", "kf_step"):
            steps[f][base[s]:base[s + 1]] = np.where(p[f] >= 0, p[f] + base[s], -1)
    return steps


def host_loop(capi, t, steps, n_seq):
    """One ellc_track_batch per wave (sequence-major steps of equal length: wave j = step j of every sequence), pose chain on the host.
    Returns (results, world, ms inside the ellc_track_batch calls: the foreign calls alone, pair and result arrays built outside)."""
    n = len(steps)
    L = n // n_seq
    res = np.zeros(n, capi.RESULT_DTYPE)
    world = np.zeros((n, 6), np.float32)
    track_ms = 0.0
    for j in range(L):
        idx = np.arange(n_seq) * L + j
        inits = np.empty((n_seq, 6), np.float32)
        kfw = []
        for k, i in enumerate(idx):
            s = steps[i]
            pw = world[s["prev_step"]] if s["prev_step"] >= 0 else s["prev_world"]
            kw = world[s["kf_step"]] if s["kf_step"] >= 0 else s["kf_world"]
            kfw.append(kw)
            inits[k] = capi.concat_origin(pw, kw)
        pairs = t.make_pairs(steps["kf_slot"][idx], steps["frame_slot"][idx], inits)
        r = np.zeros(n_seq, capi.RESULT_DTYPE)
        p_pairs, p_res = capi._p(pairs), capi._p(r)
        t0 = time.perf_counter()                            # the foreign call alone: no Python array work inside the window
        rc = capi.lib().ellc_track_batch(t._h, n_seq, p_pairs, p_res, None)
        track_ms += (time.perf_counter() - t0) * 1e3
        if rc != 0:
            raise capi.EllcError(f"ellc_track_batch failed ({rc})")
        res[idx] = r
        for k, i in enumerate(idx):
            world[i] = capi.concat_relative(r[k]["pose"], kfw[k])
    return res, world, track_ms


def run_workload(capi, imgs, n_traj, n_seq, n_frames, calls, warmup):
    kf_keys = sorted(k[1:] for k in imgs if k[0] == "kf")
    fr_keys = sorted(k[1:] for k in imgs if k[0] == "fr")
    kf_slot = {k: i for i, k in enumerate(kf_keys)}
    fr_slot = {k: i for i, k in enumerate(fr_keys)}
    from egomotion_with_local_loop_closures_b200 import synth
    intr = {n: float(v) for n, v in synth.intrinsics(640, 480).items()}
    t = capi.Tracker(capi.default_config(640, 480, max_keyframes=len(kf_keys), max_frames=len(fr_keys), **intr))
    for k in kf_keys:
        im, d, v = imgs[("kf",) + k]
        t.upload_keyframe(kf_slot[k], im, d, v)
    for k in fr_keys:
        t.upload_frame(fr_slot[k], imgs[("fr",) + k])
    steps = sequence_steps(capi, n_seq, n_frames, n_traj, kf_slot, fr_slot)
    L = n_frames - 1

    def arm_host():
        t.reset_launch_count()
        t0 = time.perf_counter()
        res, world, track_ms = host_loop(capi, t, steps, n_seq)
        return (time.perf_counter() - t0) * 1e3, track_ms, t.launch_count(), res, world

    def arm_dev():
        t.reset_launch_count()
        t0 = time.perf_counter()
        res, world = t.track_sequence_steps(steps)
        ms = (time.perf_counter() - t0) * 1e3
        return ms, t.last_track_kernel_ms(), t.launch_count(), res, world

    for _ in range(warmup):
        arm_host(); arm_dev()
    rows = dict(host_loop=[], device_chain=[])
    identical = True
    for _ in range(calls):
        h = arm_host(); d = arm_dev()
        rows["host_loop"].append(h[:3]); rows["device_chain"].append(d[:3])
        identical &= h[3].tobytes() == d[3].tobytes() and h[4].tobytes() == d[4].tobytes()
    t.close()
    out = dict(sequences=n_seq, frames_per_sequence=n_frames, tracks_per_call=len(steps), waves=L, calls=calls, warmup=warmup,
               records_and_world_poses_identical=bool(identical))
    for arm, r in rows.items():
        ms = np.array([x[0] for x in r]); aux = np.array([x[1] for x in r]); launches = sorted({int(x[2]) for x in r})
        med = float(np.median(ms))
        out[arm] = dict(ms_per_call_median=med, ms_per_call_min=float(ms.min()), ms_per_frame=med / L,
                        tracks_per_s=len(steps) / (med / 1e3), launches_per_call=launches[0] if len(launches) == 1 else launches)
        if arm == "host_loop":
            out[arm]["host_loop_track_ms_median"] = float(np.median(aux))
        else:
            out[arm]["device_ms_median"] = float(np.median(aux))       # first chain kernel to last chain kernel (CUDA events)
    out["speedup_ms_per_call"] = out["host_loop"]["ms_per_call_median"] / out["device_chain"]["ms_per_call_median"]
    out["speedup_vs_track_calls_only"] = out["host_loop"]["host_loop_track_ms_median"] / out["device_chain"]["ms_per_call_median"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10, help="timed calls per arm and workload (alternated)")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--trajectories", type=int, default=8)
    ap.add_argument("--workers", type=int, default=min(os.cpu_count() or 1, 32))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_bench_sequences.json"))
    args = ap.parse_args()
    t0 = time.time()
    imgs = render(args.trajectories, 100, args.workers)                    # fork-based rendering: before CUDA starts
    print("rendered %d images in %.0f s" % (len(imgs), time.time() - t0), flush=True)
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_sequences: no CUDA device (this measurement has no CPU form)")
    import __graft_entry__ as g
    g.build()
    from egomotion_with_local_loop_closures_b200 import capi
    res = dict(card=card(), arithmetic="FAST", size="640x480", keyframe_interval=KF_INTERVAL, trajectories=args.trajectories,
               workloads=[])
    for n_seq, n_frames in WORKLOADS:
        w = run_workload(capi, imgs, args.trajectories, n_seq, n_frames, args.calls, args.warmup)
        res["workloads"].append(w)
        print(json.dumps(dict(S=n_seq, F=n_frames, identical=w["records_and_world_poses_identical"],
                              **{a: dict(ms_per_frame=round(w[a]["ms_per_frame"], 4), tracks_per_s=round(w[a]["tracks_per_s"]),
                                         launches=w[a]["launches_per_call"]) for a in ("host_loop", "device_chain")})), flush=True)
    print(json.dumps(res["card"]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    if not all(w["records_and_world_poses_identical"] for w in res["workloads"]):
        sys.exit("bench_sequences: the two arms produced different records")


if __name__ == "__main__":
    main()
