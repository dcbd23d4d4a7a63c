"""Sequences in ELLC's constant-weight loop-closure mode: the composition of existing entry points against ellc_track_sequence_lc.

Workloads at 640x480, FAST, a keyframe every 8 frames: S = 1, 8, 64 sequences of 100 frames (99 tracks each, every track saving its
weight image), 12 keyframes retired per sequence into the sequence's own ring of 43 (pushed at positions 0..11; every query walks down
to the first empty position).  The frames come from R rendered trajectories (default 8, ground-truth keyframe depth, distinct scene
textures); sequence s runs trajectory s % R from its own root pose.  Every sequence has its own frame and keyframe slots, because the
weight images of its tracks are written into its frame slots and summed into its keyframe slots.

Arms, alternated call by call in one process after --warmup calls each (the keyframe weights are reset before every call, outside
the timed window):
  composition  ellc_track_sequence_steps; per keyframe ellc_accumulate_weights (its frames in tracking order), per retired keyframe
               ellc_finalise_weights + ellc_prepare_keyframes_lc; one ellc_frame_histograms; per query ellc_lc_generate_pairs on its
               sequence's ring as of the push (built on the host from the downloaded world poses) + ellc_track_generated_pairs
  one_call     ellc_track_sequence_lc
Reported per arm: ms per call (host clock around work that ends in a device synchronise), ms per frame (call / 99 tracked frames per
sequence), sequential and loop-closure tracks/s, kernel launches per call, and whether every output of the two arms (records, world
poses, pair lists, statistics, loop-closure records, keyframe weight pyramids and counts) is byte-identical; the script exits non-zero
if not.  The card name, power limit and maximum SM clock are read in the same run.

    python tools/bench_sequence_lc.py --out profiles/r06_bench_sequence_lc.json
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
KF_INTERVAL, N_FRAMES, RING_LEN = 8, 100, 43
MMD, THR, ANG = 8, 0.1, 10.0
WORKLOADS = (1, 8, 64)


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.returncode == 0 else "n/a")


def render(n_traj, workers):
    import bench
    from egomotion_with_local_loop_closures_b200 import synth
    jobs, index = [], []
    for r in range(n_traj):
        T = synth.smooth_trajectory(N_FRAMES, seed_pose=91011 + r)
        for i in range(0, N_FRAMES - 1, KF_INTERVAL):
            jobs.append(("kf", 1234 + r, T[i], 5678 + 100 * r + i)); index.append(("kf", r, i))
        for i in range(1, N_FRAMES):
            jobs.append(("fr", 1234 + r, T[i], 7000 + 100 * r + i)); index.append(("fr", r, i))
    import multiprocessing as mp
    with mp.get_context("fork").Pool(workers) as pool:
        out = pool.map(bench._render_job, jobs, chunksize=max(1, len(jobs) // (4 * workers)))
    return dict(zip(index, out))


def build_inputs(capi, n_seq):
    """Steps (sequence-major), keyframe entries (sequence-major, push order per ring), slot maps.  Sequence s: frame slots
    s * 113 + 1 .. + 99 for frames 1..99, s * 113 + 100 + j for the image of keyframe j; keyframe slots s * 13 + j."""
    rng = np.random.default_rng(5)
    kff = list(range(0, N_FRAMES - 1, KF_INTERVAL))
    L, per_steps, per_kfs = N_FRAMES - 1, [], []
    for s in range(n_seq):
        root = (rng.standard_normal(6) * [0.05, 0.05, 0.05, 0.2, 0.2, 0.2]).astype(np.float32)
        kf_rel = [KF_INTERVAL * ((j - 1) // KF_INTERVAL) for j in range(1, L + 1)]
        per_steps.append(capi.Tracker.make_steps([s * 13 + k // KF_INTERVAL for k in kf_rel], [s * 113 + j for j in range(1, L + 1)],
                                                 [j - 2 for j in range(1, L + 1)], [k - 1 for k in kf_rel], prev_world=[root] * L,
                                                 kf_world=[root] * L, flags=capi.PAIR_SAVE_WEIGHTS))
        kfs = capi.Tracker.make_lc_keyframes([s * 13 + j for j in range(len(kff))], [s * 113 + 100 + j for j in range(len(kff))], kff,
                                             [f - 1 for f in kff], world=[root] * len(kff))
        for j, f in enumerate(kff[:-1]):
            kfs[j]["retire_before"] = f + KF_INTERVAL
            kfs[j]["ring"], kfs[j]["ring_pos"], kfs[j]["current_array_id"] = s, j, j + 1
        per_kfs.append(kfs)
    base = np.cumsum([0] + [len(p) for p in per_steps])
    steps = np.concatenate(per_steps)
    for s, p in enumerate(per_steps):
        for f in ("prev_step", "kf_step"):
            steps[f][base[s]:base[s + 1]] = np.where(p[f] >= 0, p[f] + base[s], -1)
    kfs = np.concatenate(per_kfs)
    for s in range(n_seq):
        sl = slice(13 * s, 13 * (s + 1))
        kfs["world_step"][sl] = np.where(kfs["world_step"][sl] >= 0, kfs["world_step"][sl] + base[s], -1)
        kfs["retire_before"][sl] = np.where(kfs["retire_before"][sl] >= 0, kfs["retire_before"][sl] + base[s], -1)
    return steps, kfs


def composition(capi, t, steps, kfs, ring_in):
    """The flow ellc_track_sequence_lc replaces, from existing entry points (sequence-major steps: step order = tracking order)."""
    res, world = t.track_sequence_steps(steps)
    save = (steps["flags"] & capi.PAIR_SAVE_WEIGHTS) != 0
    for kf in kfs:
        frames = steps["frame_slot"][save & (steps["kf_slot"] == kf["kf_slot"])]
        if len(frames):
            t.accumulate_weights(int(kf["kf_slot"]), frames)
    retired = np.nonzero(kfs["retire_before"] >= 0)[0]
    for k in retired:
        t.finalise_weights(int(kfs[k]["kf_slot"]))
        t.prepare_keyframes_lc([int(kfs[k]["kf_slot"])])
    t.frame_histograms(kfs["frame_slot"][retired])
    rings = ring_in.copy()
    out = dict(pairs=[], stats=[], qi=[], lres=[])
    q = np.zeros(1, capi.LC_QUERY_DTYPE)
    for k in retired:
        kf = kfs[k]
        w = world[int(kf["world_step"])] if kf["world_step"] >= 0 else kf["world"]
        ring = rings[int(kf["ring"])]
        ring[int(kf["ring_pos"])] = (kf["frame_id"], 1, kf["frame_slot"], kf["kf_slot"], w)
        q[0] = (kf["current_array_id"], kf["match_window_beg"], kf["match_window_end"], kf["frame_id"], kf["frame_slot"], kf["stray"], w)
        p, s, _ = t.lc_generate_pairs(ring, q, min_match_difference=MMD, match_threshold=THR, max_rel_view_angle=ANG,
                                      pair_flags=capi.PAIR_CONST_WEIGHT)
        out["pairs"].append(p); out["stats"].append(s); out["qi"].append(np.full(len(p), k, np.int32))
        out["lres"].append(t.track_generated_pairs(len(p)))
    return dict(results=res, world=world, lc_pairs=np.concatenate(out["pairs"]), lc_stats=np.concatenate(out["stats"]),
                lc_query_of_pair=np.concatenate(out["qi"]), lc_results=np.concatenate(out["lres"]), ring_out=rings)


def run_workload(capi, imgs, n_traj, n_seq, calls, warmup):
    from egomotion_with_local_loop_closures_b200 import synth
    intr = {n: float(v) for n, v in synth.intrinsics(640, 480).items()}
    t = capi.Tracker(capi.default_config(640, 480, max_keyframes=13 * n_seq, max_frames=113 * n_seq, **intr))
    for s in range(n_seq):
        r = s % n_traj
        for j, f in enumerate(range(0, N_FRAMES - 1, KF_INTERVAL)):
            im, d, v = imgs[("kf", r, f)]
            t.upload_keyframe(s * 13 + j, im, d, v)
            t.upload_frame(s * 113 + 100 + j, im)
        for i in range(1, N_FRAMES):
            t.upload_frame(s * 113 + i, imgs[("fr", r, i)])
    t.synchronize()
    steps, kfs = build_inputs(capi, n_seq)
    ring0 = np.zeros((n_seq, RING_LEN), capi.LC_RING_DTYPE)
    slots = [int(x) for x in kfs["kf_slot"]]
    L = N_FRAMES - 1

    def weights():
        out = []
        for s in slots:
            for l in range(4):
                w, c = t.read_keyframe_weights(s, l)
                out.append(w.tobytes() + np.int32(c).tobytes())
        return b"".join(out)

    def arm(fn):
        for s in slots:
            t.reset_keyframe_weights(s)
        t.synchronize()
        t.reset_launch_count()
        t0 = time.perf_counter()
        out = fn()
        ms = (time.perf_counter() - t0) * 1e3
        return ms, t.launch_count(), out

    comp = lambda: composition(capi, t, steps, kfs, ring0)
    one = lambda: t.track_sequence_lc(steps, kfs, ring0, min_match_difference=MMD, match_threshold=THR, max_rel_view_angle=ANG)
    for _ in range(warmup):
        arm(comp); arm(one)
    rows = dict(composition=[], one_call=[])
    identical = True
    keys = ("results", "world", "lc_pairs", "lc_stats", "lc_query_of_pair", "lc_results", "ring_out")
    for c in range(calls):
        a = arm(comp)
        wa = weights() if c == 0 else None
        b = arm(one)
        wb = weights() if c == 0 else None
        rows["composition"].append(a[:2] + (len(a[2]["lc_pairs"]),)); rows["one_call"].append(b[:2] + (len(b[2]["lc_pairs"]),))
        identical &= all(np.ascontiguousarray(a[2][k]).tobytes() == np.ascontiguousarray(b[2][k]).tobytes() for k in keys)
        if c == 0:
            identical &= wa == wb
    t.close()
    out = dict(sequences=n_seq, frames_per_sequence=N_FRAMES, tracks_per_call=len(steps), retired_keyframes=int((kfs["retire_before"] >= 0).sum()),
               calls=calls, warmup=warmup, outputs_identical=bool(identical))
    for name, r in rows.items():
        ms = np.array([x[0] for x in r]); launches = sorted({int(x[1]) for x in r}); n_lc = r[0][2]
        med = float(np.median(ms))
        out[name] = dict(ms_per_call_median=med, ms_per_call_min=float(ms.min()), ms_per_frame=med / L,
                         sequential_tracks_per_s=len(steps) / (med / 1e3), lc_pairs=n_lc, lc_tracks_per_s=n_lc / (med / 1e3),
                         launches_per_call=launches[0] if len(launches) == 1 else launches)
    out["speedup_ms_per_call"] = out["composition"]["ms_per_call_median"] / out["one_call"]["ms_per_call_median"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10, help="timed calls per arm and workload (alternated)")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--trajectories", type=int, default=8)
    ap.add_argument("--workloads", default=",".join(map(str, WORKLOADS)), help="sequences per workload, comma-separated")
    ap.add_argument("--workers", type=int, default=min(os.cpu_count() or 1, 32))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_bench_sequence_lc.json"))
    args = ap.parse_args()
    t0 = time.time()
    imgs = render(args.trajectories, args.workers)                         # fork-based rendering: before CUDA starts
    print("rendered %d images in %.0f s" % (len(imgs), time.time() - t0), flush=True)
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_sequence_lc: no CUDA device (this measurement has no CPU form)")
    import __graft_entry__ as g
    g.build()
    from egomotion_with_local_loop_closures_b200 import capi
    res = dict(card=card(), arithmetic="FAST", size="640x480", keyframe_interval=KF_INTERVAL, ring_len=RING_LEN,
               trajectories=args.trajectories, workloads=[])
    print(json.dumps(res["card"]), flush=True)
    for n_seq in [int(x) for x in args.workloads.split(",")]:
        w = run_workload(capi, imgs, args.trajectories, n_seq, args.calls, args.warmup)
        res["workloads"].append(w)
        print(json.dumps(dict(S=n_seq, identical=w["outputs_identical"],
                              **{a: dict(ms_per_frame=round(w[a]["ms_per_frame"], 4), seq_tracks_per_s=round(w[a]["sequential_tracks_per_s"]),
                                         lc_pairs=w[a]["lc_pairs"], lc_tracks_per_s=round(w[a]["lc_tracks_per_s"]),
                                         launches=w[a]["launches_per_call"]) for a in ("composition", "one_call")})), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    if not all(w["outputs_identical"] for w in res["workloads"]):
        sys.exit("bench_sequence_lc: the two arms produced different outputs")


if __name__ == "__main__":
    main()
