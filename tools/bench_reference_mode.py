"""Throughput of the three arithmetic flavours (FAST, STRICT, REFERENCE) on the flagship workload of bench.py: 640x480, 32 keyframes,
512 frames, 4,608 pairs per step, inputs resident on the device.

Forward mode tracks the pair list as it is; const_weight mode tracks the loop-closure candidates with the constant-weight variant
(the sequential pair of every frame saves its weights; keyframe weights finalised and loop-closure records built untimed, as
bench.py --lc-mode const_weight does).  One process holds one tracker per flavour; after --warmup steps each, the flavours are
alternated step by step for --steps steps each.  A step is one ellc_track_batch call (host clock around it: the call returns after
the records are copied back) and its tracking kernel time (CUDA events).  A sample of the REFERENCE records is compared bit for bit
with the CPU oracle.  The card name and power limit are read in the same run.

    python tools/bench_reference_mode.py --out profiles/r04_bench_reference_mode.json
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
FLAVOURS = (("fast", 0), ("strict", 1), ("reference", 2))


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.returncode == 0 else "n/a")


def make_tracker(capi, cfg_kw, arith, wl, n_kf, n_fr):
    t = capi.Tracker(capi.default_config(640, 480, max_keyframes=n_kf, max_frames=n_fr, arithmetic=arith, **cfg_kw))
    for i in range(n_kf):
        t.upload_keyframe(i, wl["kf_images"][i], wl["kf_depth"][i], wl["kf_var"][i])
    for i in range(n_fr):
        t.upload_frame(i, wl["frames"][i])
    t.synchronize()
    return t


def lc_setup(capi, t, wl, n_kf, primary):
    seq = t.make_pairs(wl["kf_idx"][primary], wl["fr_idx"][primary], wl["init"][primary], flags=capi.PAIR_SAVE_WEIGHTS)
    t.track_batch(seq)
    for k in range(n_kf):
        t.reset_keyframe_weights(k)
        fr = np.sort(wl["fr_idx"][primary][wl["kf_idx"][primary] == k])
        for lo in range(0, len(fr), 64):
            t.accumulate_weights(k, fr[lo:lo + 64])
        t.finalise_weights(k)
    t.prepare_keyframes_lc(np.arange(n_kf, dtype=np.int32))
    t.synchronize()


def oracle_check(capi, oracle, t, wl, pairs, rec, idx, lc):
    """REFERENCE records of the sampled pairs against the CPU oracle: pose bits and iteration counts."""
    from egomotion_with_local_loop_closures_b200 import synth
    k = synth.intrinsics(640, 480)
    ocfg = oracle.default_config(640, 480, fx=float(k["fx"]), fy=float(k["fy"]), cx=float(k["cx"]), cy=float(k["cy"]))
    out = []
    for i in idx:
        kf, fr = int(pairs[i]["kf_slot"]), int(pairs[i]["frame_slot"])
        init = np.array(pairs[i]["init_pose"], np.float32)
        if lc and (pairs[i]["flags"] & capi.PAIR_CONST_WEIGHT):
            wts = [t.read_keyframe_weights(kf, l)[0] for l in range(4)]
            opose, otr = oracle.track_lc(ocfg, wl["kf_images"][kf], wl["frames"][fr], wl["kf_depth"][kf], wts, init)
        else:
            opose, otr = oracle.track(ocfg, wl["kf_images"][kf], wl["frames"][fr], wl["kf_depth"][kf], wl["kf_var"][kf], init)
        out.append(dict(pair=int(i), const_weight=bool(pairs[i]["flags"] & capi.PAIR_CONST_WEIGHT),
                        pose_bits_equal=bool(np.array_equal(np.asarray(rec[i]["pose"], np.float32).view(np.uint32), opose.view(np.uint32))),
                        iters_equal=[int(v) for v in rec[i]["n_iters"]] == otr["n_iters"]))
    return out


def run_mode(capi, oracle, wl, lc, steps, warmup, n_kf, n_fr, n_check):
    primary = wl["kf_idx"] == (wl["fr_idx"] % n_kf)
    flags = np.where(primary, capi.PAIR_SAVE_WEIGHTS, capi.PAIR_CONST_WEIGHT).astype(np.int32) if lc else 0
    trk = {}
    for name, arith in FLAVOURS:
        trk[name] = make_tracker(capi, {}, arith, wl, n_kf, n_fr)
        if lc:
            lc_setup(capi, trk[name], wl, n_kf, primary)
    pairs = trk["fast"].make_pairs(wl["kf_idx"], wl["fr_idx"], wl["init"], flags=flags)
    n_cw = int((pairs["flags"] & capi.PAIR_CONST_WEIGHT != 0).sum())
    last = {}
    for name, _ in FLAVOURS:
        for _ in range(warmup):
            last[name] = trk[name].track_batch(pairs)
    wall = {name: [] for name, _ in FLAVOURS}
    kern = {name: [] for name, _ in FLAVOURS}
    for _ in range(steps):
        for name, _ in FLAVOURS:
            t0 = time.perf_counter()
            last[name] = trk[name].track_batch(pairs)
            wall[name].append((time.perf_counter() - t0) * 1e3)
            kern[name].append(trk[name].last_track_kernel_ms())
    rows = {}
    for name, _ in FLAVOURS:
        w, k = np.array(wall[name]), np.array(kern[name])
        rows[name] = dict(step_ms_median=float(np.median(w)), step_ms_min=float(w.min()), kernel_ms_median=float(np.median(k)),
                          kernel_ms_min=float(k.min()), tracks_per_s=len(pairs) / (float(np.median(w)) / 1e3),
                          tracks_per_s_kernel=len(pairs) / (float(np.median(k)) / 1e3),
                          deterministic=bool(last[name].tobytes() == trk[name].track_batch(pairs).tobytes()))
    rng = np.random.default_rng(4)
    pick = (np.flatnonzero(pairs["flags"] & capi.PAIR_CONST_WEIGHT) if lc else np.arange(len(pairs)))
    idx = rng.choice(pick, size=min(n_check, len(pick)), replace=False)
    check = oracle_check(capi, oracle, trk["reference"], wl, pairs, last["reference"], idx, lc)
    for t in trk.values():
        t.close()
    return dict(mode="const_weight" if lc else "forward", pairs=len(pairs), const_weight_pairs=n_cw, steps=steps, warmup=warmup,
                flavours=rows, reference_vs_oracle=check)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--check", type=int, default=4, help="REFERENCE records compared with the CPU oracle per mode")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_bench_reference_mode.json"))
    args = ap.parse_args()
    import bench
    n_kf, n_fr = 32, 512
    wl = bench.build_workload(n_kf, n_fr, 9, seed=0, conf=bench.CONFIGS["pair_sweep"])      # fork-based rendering: before CUDA starts
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_reference_mode: no CUDA device (this measurement has no CPU form)")
    import __graft_entry__ as g
    g.build()
    import oracle
    from egomotion_with_local_loop_closures_b200 import capi
    res = dict(card=card(), workload="pair_sweep 640x480: 32 keyframes, 512 frames, 9 pairs per frame, resident inputs",
               modes=[run_mode(capi, oracle, wl, lc, args.steps, args.warmup, n_kf, n_fr, args.check) for lc in (False, True)])
    for m in res["modes"]:
        print(json.dumps(dict(mode=m["mode"], **{k: round(v["tracks_per_s"]) for k, v in m["flavours"].items()})), flush=True)
    print(json.dumps(res["card"]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    bad = [c for m in res["modes"] for c in m["reference_vs_oracle"] if not (c["pose_bits_equal"] and c["iters_equal"])]
    if bad:
        sys.exit("bench_reference_mode: REFERENCE records differ from the oracle: %s" % bad)


if __name__ == "__main__":
    main()
