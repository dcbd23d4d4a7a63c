#!/usr/bin/env python
"""bench.py -- frame-keyframe GN tracks/sec at 640x480 (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N --steps K --warmup W]            # our arm (CUDA path through the C-ABI)
    python bench.py --impl reference [...]                       # reference arm: the CPU tracker on the host cores
    python bench.py --config {pair_sweep,720p_single,1080p_stress} [--lc-mode const_weight]   # the other BASELINE configs
    python bench.py [...] --dump-outputs DIR                    # also write the last timed step's result records as DIR/<field>.npy
                                                                 # (our arm only: the reference arm times a sample of the pairs)

A "step" is one batch of the hot path on one GPU: `frames` new frames (pyramid + gradient texels), `keyframes`
keyframes (pyramid + mask/count/selection) and `pairs` frame-keyframe tracks (each frame against its own keyframe and
K-1 local-loop-closure candidates), i.e. BASELINE config 5 / config 3 at 640x480.  Weak scaling: every rank gets the same
amount of work; ranks shard a global pair list by keyframe affinity; the 256-byte result records are gathered on rank 0 by the
tracking kernel itself (stores into rank 0's result table over NVLink peer memory, ellc_track_batch_exchange); NCCL carries the
IPC handles, the barriers and the max-over-ranks reduction of the timing (and the gather itself with --exchange nccl).

Timed regions
  value : inputs resident in HBM (level-0 u8 images, keyframe depth/variance pyramids, pair list on the host);
          prepare_frames + prepare_keyframes + track_batch + result D2H (for N>1: + the gather of all ranks' records).
  e2e   : the same through the reference-facing C-ABI with HOST (pinned) buffers: H2D of every image and depth/variance
          pyramid, the gather (N>1) and D2H of the results inside the timed region.
Inputs (hundreds of MB per step) are larger than the 126 MB L2, so no explicit L2 flush is needed between steps.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# Keep stdout for the ONE JSON line: libraries (NCCL's version banner, ...) write to fd 1 behind Python's back, so fd 1 is
# pointed at stderr for the whole run and the result line goes to a private duplicate of the original stdout.
_RESULT_FD = os.dup(1)
os.dup2(2, 1)


def emit(line):
    os.write(_RESULT_FD, (json.dumps(line) + "\n").encode())


from egomotion_with_local_loop_closures_b200 import synth  # noqa: E402

W, H = 640, 480
METRIC = "frame-keyframe GN tracks/sec at 640x480"
UNIT = "tracks/s"

# BASELINE.json configs.  pair_sweep (configs 3/5: every frame against its own keyframe + K = 8 loop-closure candidates) is the
# one the metric is quoted on; the other two are reported with the same line format under their own workload names.
CONFIGS = {
    "pair_sweep": dict(size=(640, 480), keyframes=32, frames=512, pairs_per_frame=9, kf_rot=2.0, fr_rot=1.0, fr_trans=0.015,
                       init="previous_frame", workload="pair_sweep_640x480"),
    # config 2: ONE keyframe, ONE frame: single-pair latency (a cluster of 8 CTAs tracks the pair)
    "720p_single": dict(size=(1280, 720), keyframes=1, frames=1, pairs_per_frame=1, kf_rot=0.0, fr_rot=1.0, fr_trans=0.015,
                        init="previous_frame", workload="single_keyframe_1280x720"),
    # config 4: fast head rotation (2-5 degrees between frame and keyframe), zero initial pose: convergence stress
    "1080p_stress": dict(size=(1920, 1080), keyframes=4, frames=64, pairs_per_frame=1, kf_rot=0.0, fr_rot=(2.0, 5.0), fr_trans=0.03,
                         init="zero", workload="fast_rotation_1920x1080"),
}


# ----------------------------------------------------------------------------------------------------------------
# workload
# ----------------------------------------------------------------------------------------------------------------
def _render_job(args):
    kind, seed_scene, T, seed = args
    scene = _render_job.scenes.get((seed_scene, W, H))
    if scene is None:
        scene = _render_job.scenes[(seed_scene, W, H)] = synth.SynthScene(W, H, seed_tex=seed_scene)
    if kind == "kf":
        kf = scene.keyframe(T, seed_depth=seed, noise_seed=seed + 1)
        return kf["image"], kf["depth"], kf["var"]
    return scene.render(T, noise_seed=seed)


_render_job.scenes = {}


def build_workload(n_kf, n_frames, pairs_per_frame, seed, workers=None, conf=None):
    """Seeded pool of keyframes / frames / pairs for one rank.  Rendering is numpy (untimed setup)."""
    conf = conf or CONFIGS["pair_sweep"]
    rng = np.random.default_rng(seed)
    T_kf = [synth.se3_exp(synth.random_pose(rng, rot=np.deg2rad(conf["kf_rot"]), trans=0.04 if conf["kf_rot"] else 0.0)) for _ in range(n_kf)]
    primary = np.arange(n_frames) % n_kf

    def frame_motion():
        if isinstance(conf["fr_rot"], tuple):                 # rotation of a given magnitude range (config 4)
            deg = rng.uniform(*conf["fr_rot"])
            p = synth.random_pose(rng, rot=np.deg2rad(deg), trans=conf["fr_trans"])
            p[:3] *= np.deg2rad(deg) / max(np.linalg.norm(p[:3]), 1e-12)
            return p
        return synth.random_pose(rng, rot=np.deg2rad(conf["fr_rot"]), trans=conf["fr_trans"])
    T_fr = [synth.se3_exp(frame_motion()) @ T_kf[primary[i]] for i in range(n_frames)]
    jobs = [("kf", 1234 + seed, T_kf[k], 5678 + 17 * k + seed) for k in range(n_kf)]
    jobs += [("fr", 1234 + seed, T_fr[i], 91011 + i + 1000 * seed) for i in range(n_frames)]
    workers = workers or min(os.cpu_count() or 1, 32)
    if workers > 1:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(workers) as pool:
            out = pool.map(_render_job, jobs, chunksize=max(1, len(jobs) // (4 * workers)))
    else:
        out = [_render_job(j) for j in jobs]
    kfs, frames = out[:n_kf], out[n_kf:]
    kf_idx, fr_idx, init = [], [], []
    for i in range(n_frames):
        others = [k for k in range(n_kf) if k != primary[i]]
        cand = [int(primary[i])] + list(rng.choice(others, size=min(pairs_per_frame - 1, len(others)), replace=False))
        for k in cand:
            rel = synth.relative_pose(T_fr[i], T_kf[k])
            # init = pose of the "previous frame" (src/ImageFunc.cpp:106): ground truth perturbed by a small motion
            jitter = synth.random_pose(rng, rot=np.deg2rad(0.3), trans=0.004)
            init.append(rel + jitter if conf["init"] == "previous_frame" else np.zeros(6))
            kf_idx.append(k)
            fr_idx.append(i)
    perm = rng.permutation(len(kf_idx))
    return dict(kf_images=[k[0] for k in kfs], kf_depth=[k[1] for k in kfs], kf_var=[k[2] for k in kfs], frames=frames,
                kf_idx=np.array(kf_idx, np.int32)[perm], fr_idx=np.array(fr_idx, np.int32)[perm],
                init=np.array(init, np.float32)[perm])


def algorithmic_bytes(res):
    """SURVEY 8d: per GN iteration at level L, B_iter(L) = 2 P_L + 9 N_L; summed over executed iterations of all tracks."""
    P = np.array([(W >> l) * (H >> l) for l in range(4)], np.float64)
    it = res["n_iters"].astype(np.float64)
    n = res["n_selected"].astype(np.float64)
    return float((it * (2.0 * P[None, :] + 9.0 * n)).sum())


def pixel_iterations(res):
    """Selected-pixel evaluations of a batch: sum over tracks, levels and executed iterations of N_L."""
    return float((res["n_iters"].astype(np.float64) * res["n_selected"].astype(np.float64)).sum())


def setup_bytes(n_frames, n_kf):
    """B_setup: keyframe depth read + mask write (5 P_L) and pyramid build (P_{L-1} + P_L) per frame / keyframe."""
    P = np.array([(W >> l) * (H >> l) for l in range(4)], np.float64)
    pyr = float(sum(P[l - 1] + P[l] for l in range(1, 4)))
    return n_frames * pyr + n_kf * (pyr + 5.0 * P.sum())


def input_bytes_per_step(n_frames, n_kf, n_pairs):
    """Host inputs of one step on one GPU: u8 level-0 images of the frames and keyframes, f32 depth and variance pyramids of the
    keyframes (cv::pyrDown level sizes), the pair list."""
    dims = [(W >> l, H >> l) for l in range(4)]                # depth / variance arrays: ORIG_COLS >> L x ORIG_ROWS >> L
    return n_frames * W * H + n_kf * (W * H + 2 * 4 * sum(w * h for w, h in dims)) + n_pairs * 36


def workload_config(conf, n_kf, n_frames, pairs_per_frame, n_pairs, lc=False):
    """`config` of the bench line: the WORKLOAD and nothing else -- identical in our arm and in the reference arm (which tracks a
    bounded sample of the same pair list; how each arm runs it is under `implementation`)."""
    inb = input_bytes_per_step(n_frames, n_kf, n_pairs)
    return {"workload": conf["workload"] + ("_lc_const_weight" if lc else ""), "width": W, "height": H, "keyframes_per_gpu": n_kf,
            "frames_per_gpu": n_frames, "pairs_per_gpu_per_step": n_pairs, "pairs_per_frame": pairs_per_frame,
            "l2": ("inputs (%.0f MB per step per GPU) exceed the 126 MB L2; no flush" % (inb / 1e6)) if inb > 126e6 else
                  ("inputs (%.1f MB) fit the L2: this configuration measures latency of a resident working set, not bandwidth" % (inb / 1e6))}


# ----------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML in a thread (5 ms period, no start-up latency);
    falls back to `nvidia-smi -lms 50` when pynvml is unavailable.  mark() brackets the timed region; samples outside are dropped."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc, self.stop_flag, self.t0, self.t1, self.nvml = gpu_index, [], None, False, None, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.idx]) if vis and vis.split(",")[self.idx].isdigit() else self.idx
            self.nvml = (pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.nvml[1], pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    PERIOD_S = float(os.environ.get("ELLC_CLOCK_PERIOD_MS", "50")) * 1e-3

    def _sample(self):
        nv, hd = self.nvml
        try:
            mhz = float(nv.nvmlDeviceGetClockInfo(hd, nv.NVML_CLOCK_SM))
            try:
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(hd))
            except Exception:
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(hd))
            self.rows.append((time.perf_counter(), mhz, mask))
        except Exception:
            pass

    def _poll(self):
        # NVML queries go through the same driver as the CUDA calls of the benchmark loop: polled every 5 ms they coincided with
        # sporadic 10-190 ms stalls of the loop's launches (host_ms_per_step.enqueue.max); 50 ms keeps >= 2 samples in any timed
        # region of the default workload, and mark_begin / mark_end add one sample each while the device is under load.
        while not self.stop_flag:
            self._sample()
            time.sleep(self.PERIOD_S)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def sample_now(self):
        """One sample from the calling thread (bench: right after the last timed step has been enqueued, i.e. under load)."""
        if self.nvml:
            self._sample()

    def stop(self):
        self.stop_flag = True
        inside = lambda t: (self.t0 is None or t >= self.t0) and (self.t1 is None or t <= self.t1)
        if self.nvml:
            self.thread.join(timeout=1)
            rows = [r for r in self.rows if inside(r[0])] or self.rows[-3:]
            reasons = sorted({name for _, _, m in rows for bit, name in self.REASONS.items() if m & bit})
            sm = [r[1] for r in rows]
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz, "samples": len(sm), "reasons": reasons,
                    "source": "nvml, %.0f ms period + one sample with the last timed steps in flight, timed region only" % (1e3 * self.PERIOD_S)}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for _, r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 50 (warm-up + timed region)"}


# ----------------------------------------------------------------------------------------------------------------
def run_reference(args, rank, world, conf):
    """Reference arm: the reference's CPU tracker (the oracle restatement -- the real one cannot be compiled as it is, DESIGN.md)
    on the host cores, on a bounded sample of the SAME workload as our arm: the first pairs of rank 0's pair list
    (same keyframes, frames, initial poses).  Two modes (SURVEY 8d): `all-host-core` (one pair per hardware thread: the
    headline baseline, `value`) and `reference-faithful` (what the reference does: NUM_POSE_THREADS = 3 row-band threads per
    pair, pairs one after the other, src/PixelWisePyramid.cpp:426-436), reported beside it."""
    if rank != 0:
        return
    import oracle
    cores = os.cpu_count() or 1
    wl = build_workload(args.keyframes, args.frames, args.pairs_per_frame, seed=0, conf=conf)
    n_pairs = min(len(wl["kf_idx"]), max(cores * 64, 256) if conf is CONFIGS["pair_sweep"] else max(cores * 2, 8))   # ~3 s of CPU work per step
    k = synth.intrinsics(W, H)
    cfg = oracle.default_config(W, H, fx=float(k["fx"]), fy=float(k["fy"]), cx=float(k["cx"]), cy=float(k["cy"]))
    times = []
    for step in range(args.warmup + args.steps):
        _, secs = oracle.track_many(cfg, wl["kf_idx"][:n_pairs], wl["fr_idx"][:n_pairs], wl["kf_images"], wl["frames"],
                                    wl["kf_depth"], wl["kf_var"], wl["init"][:n_pairs], n_workers=cores)
        if step >= args.warmup:
            times.append(secs)
    total = float(sum(times))
    value = n_pairs * len(times) / total
    # reference-faithful mode: three band threads per pair, pairs sequential; a smaller sample (it is ~cores/3 x slower)
    n_f = max(8, min(n_pairs, 3 * 16))
    fcfg = oracle.default_config(W, H, fx=float(k["fx"]), fy=float(k["fy"]), cx=float(k["cx"]), cy=float(k["cy"]), num_bands=3, use_threads=1)
    _, fsecs = oracle.track_many(fcfg, wl["kf_idx"][:n_f], wl["fr_idx"][:n_f], wl["kf_images"], wl["frames"], wl["kf_depth"], wl["kf_var"],
                                 wl["init"][:n_f], n_workers=1)
    faithful = {"value": n_f / fsecs, "unit": UNIT, "cores": 3, "kind": "port",
                "sample": f"first {n_f} pairs, one pair at a time, 3 row-band threads per pair (NUM_POSE_THREADS, src/PixelWisePyramid.cpp:426-436)"}
    sample = (f"first {n_pairs} pairs/step of rank 0's pair list of this workload ({args.keyframes} keyframes, {args.frames} frames), "
              f"{cores} worker threads (1 pair per thread, bands sequential)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(conf, args.keyframes, args.frames, args.pairs_per_frame, len(wl["kf_idx"])),
            "implementation": {"sample_pairs_per_step": n_pairs,
                               "note": "CPU oracle restatement of the reference tracker (g++ -std=c++11 -O3), bit-identical to the reference's own code where "
                                       "that could be compiled (DESIGN.md section 2); it omits the reference's per-pixel cv::Mat/cv::String overhead, so it is "
                                       "FASTER than the real binary; each step tracks a bounded sample -- the first pairs -- of the workload's pair list (a rate: tracks/s)"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "reference_faithful": faithful},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


DUMP_MAX_BYTES = 64 * 10**6


def dump_outputs(out_dir, rec):
    """The result records a caller of the timed path receives, one DIR/<field>.npy per field of ellc_result (float32; the integer
    fields as float64, which holds them exactly), so that two builds can be compared output for output.  The workload is seeded,
    so the same arguments give the same records.  Above DUMP_MAX_BYTES a fixed, seeded sample of the records is written;
    pair_index.npy holds their positions in the result table."""
    fields = [n for n in rec.dtype.names if n != "reserved"]
    row_bytes = 8 + sum(rec.dtype[n].itemsize * (2 if rec.dtype[n].base.kind == "i" else 1) for n in fields)
    cap = (DUMP_MAX_BYTES - 4096 * (len(fields) + 1)) // row_bytes          # 4 KB per file covers the .npy header
    idx = np.arange(len(rec))
    if len(idx) > cap:
        idx = np.sort(np.random.default_rng(0).choice(len(idx), cap, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pair_index.npy"), idx.astype(np.float64))
    for n in fields:
        a = rec[n][idx]
        np.save(os.path.join(out_dir, n + ".npy"), a.astype(np.float64 if a.dtype.kind == "i" else np.float32))


def sass_inst_per_pixel():
    """Static instruction count of the level-0 pixel loop (usual path) from profiles/r02_sass_histogram.json (tools/sass_histogram.py)."""
    try:
        j = json.load(open(os.path.join(ROOT, "profiles", "r02_sass_histogram.json")))
        return j
    except Exception:
        return None


def main():
    global W, H, METRIC
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="pair_sweep", choices=sorted(CONFIGS), help="BASELINE.json config (default: the one the metric is quoted on)")
    ap.add_argument("--keyframes", type=int, default=None, help="keyframes per GPU per step")
    ap.add_argument("--frames", type=int, default=None, help="frames per GPU per step")
    ap.add_argument("--pairs-per-frame", type=int, default=None, help="1 sequential + K=8 loop-closure candidates")
    ap.add_argument("--arith", default="fast", choices=["fast", "strict"])
    ap.add_argument("--cluster", type=int, default=0, help="CTAs per pair (thread-block cluster): 0 = the library chooses from the batch size")
    ap.add_argument("--pairs-per-cta", type=int, default=0, help="pairs one CTA tracks in lockstep: 0 = the library chooses")
    ap.add_argument("--lc-mode", default="forward", choices=["forward", "const_weight"],
                    help="const_weight: the K-1 loop-closure pairs of every frame run the reference's constant-weight "
                         "inverse-compositional tracker (FLAG_DO_CONST_WEIGHT_POSE_ESTIMATION); not the headline workload")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: gather of the result records by in-kernel stores over NVLink peer memory (default) or by NCCL")
    ap.add_argument("--exchange-root", type=int, default=0, help="rank that receives all records; -1 = every rank (all-gather)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the result records of the last one as DIR/<field>.npy (at most 64 MB); N>1: "
                         "the table gathered on the --exchange-root rank (rank 0 for -1).  Not with --impl reference, which tracks only "
                         "a sample of the pair list")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the records of the CUDA path (--impl ours)")
    conf = CONFIGS[args.config]
    W, H = conf["size"]
    if args.config != "pair_sweep":
        METRIC = "frame-keyframe GN tracks/sec at %dx%d" % (W, H)
    args.keyframes = args.keyframes or conf["keyframes"]
    args.frames = args.frames or conf["frames"]
    args.pairs_per_frame = args.pairs_per_frame or conf["pairs_per_frame"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world, conf)
        return

    # ---- data first (fork-based rendering must precede CUDA initialisation)
    t_setup = time.time()
    # every rank renders its own segment: share the host cores between the ranks of the node
    wl = build_workload(args.keyframes, args.frames, args.pairs_per_frame, seed=rank,
                        workers=max(1, min(32, (os.cpu_count() or 1) // max(1, world))), conf=conf)
    n_pairs = len(wl["kf_idx"])

    import torch
    import torch.distributed as dist
    from egomotion_with_local_loop_closures_b200 import capi
    from egomotion_with_local_loop_closures_b200.sharding import shard_pairs

    torch.cuda.set_device(local_rank)
    if world > 1:
        # NCCL carries the IPC handles, barriers and the timing reduction (and, with --exchange nccl, the gather of the records:
        # 1.2 MB per rank and step, latency-bound, WHILE the next step's tracking kernel owns the SMs -- one channel + the
        # low-latency protocol keep its footprint on the SMs small, measured in round 1)
        os.environ.setdefault("NCCL_MAX_NCHANNELS", "1")
        os.environ.setdefault("NCCL_MIN_NCHANNELS", "1")
        os.environ.setdefault("NCCL_PROTO", "LL")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    k = synth.intrinsics(W, H)
    cfg = capi.default_config(W, H, fx=float(k["fx"]), fy=float(k["fy"]), cx=float(k["cx"]), cy=float(k["cy"]),
                              max_keyframes=2 * args.keyframes, max_frames=2 * args.frames, device=local_rank,
                              arithmetic=capi.ARITH_STRICT if args.arith == "strict" else capi.ARITH_FAST,
                              ctas_per_pair=args.cluster, pairs_per_cta=args.pairs_per_cta)
    trk = capi.Tracker(cfg)
    stream = torch.cuda.ExternalStream(trk.stream(), device=torch.device("cuda", local_rank))

    # Global pair list = the sequence segments of all ranks (keyframe / frame ids offset per segment).  shard_pairs deals whole
    # connected components (segments) to ranks, so every rank gets one segment back -- the production path for a mixed list.
    if world > 1:
        g_kf = np.concatenate([wl["kf_idx"].astype(np.int64) + r * args.keyframes for r in range(world)])
        g_fr = np.concatenate([wl["fr_idx"].astype(np.int64) + r * args.frames for r in range(world)])
        shards = shard_pairs(g_kf, g_fr, world)
        seg = [int(g_kf[s][0] // args.keyframes) for s in shards]
        assert sorted(seg) == list(range(world)) and all(len(s) == n_pairs for s in shards)
        my_idx = shards[seg.index(rank)]                       # this rank rendered segment `rank`
        shard_of_rank = [shards[seg.index(r)] for r in range(world)]
    else:
        my_idx = np.arange(n_pairs)
        shard_of_rank = [my_idx]
    n_total = n_pairs * world
    root = args.exchange_root if world > 1 else 0
    receives = (root < 0) or (root == rank)

    # ---- the gather of the result records (N > 1) ------------------------------------------------------------------------
    xmode = "none"
    if world > 1:
        xmode = args.exchange
        if xmode == "p2p":
            ok = 1
            try:
                hnd = trk.exchange_create(rank, world, n_total)
                allh = torch.empty(world * capi.IPC_HANDLE_BYTES, dtype=torch.uint8, device="cuda")
                dist.all_gather_into_tensor(allh, torch.from_numpy(hnd).cuda())
                trk.exchange_attach_ipc(allh.cpu().numpy())
            except capi.EllcError as exc:                      # e.g. CUDA IPC not permitted in this container
                print(f"[rank {rank}] peer-memory exchange unavailable ({exc}); falling back to NCCL", file=sys.stderr)
                ok = 0
            flag = torch.tensor([ok], dtype=torch.int32, device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 0:
                xmode = "nccl"
    nccl_state = {}
    if xmode == "nccl":
        # fixed sharding: the position of every gathered record is known up front -> one all-gather + one index_select per batch,
        # no boolean masks, no host synchronisation; the table is fetched one step later through a pinned buffer
        order = np.concatenate(shard_of_rank)
        inv = np.empty(n_total, np.int64)
        inv[order] = np.arange(n_total)
        nccl_state["inv"] = torch.as_tensor(inv, device="cuda")
        nccl_state["rec"] = torch.empty((n_pairs, 256), dtype=torch.uint8, device="cuda")
        nccl_state["all"] = torch.empty((n_total, 256), dtype=torch.uint8, device="cuda")
        nccl_state["host"] = torch.empty((n_total, 256), dtype=torch.uint8).pin_memory()
        prio = torch.cuda.Stream(priority=-1)                  # NCCL kernels must not queue behind the tracking CTAs
        nccl_state["stream"] = prio

    # pinned host copies (e2e uploads) -----------------------------------------------------------------------------
    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t, t.numpy()
    keep = []
    h_frames, h_kf_img, h_kf_depth, h_kf_var = [], [], [], []
    for f in wl["frames"]:
        t, a = pin(f); keep.append(t); h_frames.append(a)
    for i in range(args.keyframes):
        t, a = pin(wl["kf_images"][i]); keep.append(t); h_kf_img.append(a)
        d, v = [], []
        for l in range(4):
            t, a = pin(wl["kf_depth"][i][l]); keep.append(t); d.append(a)
            t, a = pin(wl["kf_var"][i][l]); keep.append(t); v.append(a)
        h_kf_depth.append(d); h_kf_var.append(v)
    h2d_bytes = sum(a.nbytes for a in h_frames) + sum(a.nbytes for a in h_kf_img) + sum(a.nbytes for d in h_kf_depth for a in d) + \
        sum(a.nbytes for d in h_kf_var for a in d) + n_pairs * capi.PAIR_DTYPE.itemsize
    # records read back by the host per step, whole job: every rank its own (N = 1) / the receiving rank(s) the whole table
    d2h_bytes_job = n_pairs * 256 if world == 1 else n_total * 256 * (world if root < 0 else 1)

    def upload_all(half=0):
        ko, fo = half * args.keyframes, half * args.frames
        for i in range(args.keyframes):
            trk.upload_keyframe(ko + i, h_kf_img[i], h_kf_depth[i], h_kf_var[i])
        for i in range(args.frames):
            trk.upload_frame(fo + i, h_frames[i])

    lc = args.lc_mode == "const_weight"
    primary = (wl["kf_idx"] == (wl["fr_idx"] % args.keyframes))
    flags = np.where(primary, capi.PAIR_SAVE_WEIGHTS, capi.PAIR_CONST_WEIGHT).astype(np.int32) if lc else 0
    pairs = trk.make_pairs(wl["kf_idx"], wl["fr_idx"], wl["init"], flags=flags)
    pairs_half = [pairs, trk.make_pairs(wl["kf_idx"] + args.keyframes, wl["fr_idx"] + args.frames, wl["init"], flags=flags)]
    if lc:
        args.no_e2e = True                                     # an upload invalidates the loop-closure records: resident mode only
        args.no_cpu_baseline = True                            # (the forward CPU baseline is not this workload)
    fr_slots = np.arange(args.frames, dtype=np.int32)
    kf_slots = np.arange(args.keyframes, dtype=np.int32)

    upload_all()
    upload_all(1)                                              # the workload is resident twice: steps alternate between the halves
    trk.synchronize()
    if lc:
        # untimed setup, as in the reference's flow: every keyframe's weight pyramid = average of the last-iteration weights of
        # the sequential tracks of its frames (saveWeights / finaliseWeights), then the loop-closure records -- for both halves
        for half in (0, 1):
            ko, fo = half * args.keyframes, half * args.frames
            seq = trk.make_pairs(wl["kf_idx"][primary] + ko, wl["fr_idx"][primary] + fo, wl["init"][primary], flags=capi.PAIR_SAVE_WEIGHTS)
            trk.track_batch(seq)
            for kslot in range(args.keyframes):
                trk.reset_keyframe_weights(ko + kslot)
                fr = np.sort(wl["fr_idx"][primary][wl["kf_idx"][primary] == kslot])
                for lo in range(0, len(fr), 64):
                    trk.accumulate_weights(ko + kslot, fo + fr[lo:lo + 64])
                trk.finalise_weights(ko + kslot)
            trk.prepare_keyframes_lc(np.arange(args.keyframes, dtype=np.int32) + ko)
        trk.synchronize()
    setup_s = time.time() - t_setup

    kernel_ms = []
    my_idx32 = my_idx.astype(np.int32)

    # ---- one batch: launch, and (one step later) fetch ----------------------------------------------------------------------
    # launch(p) -> ticket; fetch(ticket) -> (records of THIS rank's pairs or None, table of all pairs or None).  The fetch of batch
    # k is issued after the launch of batch k+1, so the gather / download of batch k overlaps the kernels of batch k+1.
    def launch(p):
        if xmode == "p2p":
            return ("x", trk.track_batch_exchange(p, my_idx32, n_total, root=root))
        dptr = trk.track_batch_async(p)
        if xmode == "nccl":
            ev = torch.cuda.Event()
            trk.fence()
            ev.record(stream)
            return ("n", dptr, ev)
        return ("l", dptr)

    def fetch(ticket):
        if ticket[0] == "l":
            own = trk.results_download(ticket[1], n_pairs)
            return own, own
        if ticket[0] == "x":
            table = trk.exchange_wait(ticket[1], n_total if receives else None)
            return (table[my_idx] if table is not None else None), table
        _, dptr, ev = ticket
        from cuda import cudart  # cuda-python is in the image
        ns = nccl_state["stream"]
        with torch.cuda.stream(ns):
            ns.wait_event(ev)                                   # batch k is complete before its records are read
            err, = cudart.cudaMemcpyAsync(nccl_state["rec"].data_ptr(), dptr, n_pairs * 256, cudart.cudaMemcpyKind.cudaMemcpyDeviceToDevice, ns.cuda_stream)
            assert int(err) == 0
            dist.all_gather_into_tensor(nccl_state["all"], nccl_state["rec"])
            if receives:
                nccl_state["host"].copy_(nccl_state["all"].index_select(0, nccl_state["inv"]), non_blocking=True)
        ns.synchronize()
        trk.results_download(dptr, 0)
        if not receives:
            return None, None
        table = nccl_state["host"].numpy().view(capi.RESULT_DTYPE).reshape(-1).copy()
        return table[my_idx], table

    # Forward workload: steps alternate between two resident copies of the inputs (slot halves), so that the preparation of step
    # k+1 (pyramids, texels, selection lists: ellc_prepare_async, low-priority stream) overlaps the tracking kernel of step k, and
    # the records of step k are fetched while step k+1 runs.  Every step still does all of its own work.
    # The host runs PIPE_DEPTH steps ahead of the records it fetches: while it waits for step k, steps k+1 .. k+PIPE_DEPTH are queued on
    # the device.  (Depth 1 idles the GPU whenever the host loses more than one step's time between two launches -- measured: sporadic
    # 10-50 ms gaps in the enqueue half of a step on the shared benchmark boxes, which cost up to 15 % of a 10-step run.)
    PIPE_DEPTH = int(os.environ.get("ELLC_PIPE_DEPTH", "2"))
    pipe = {"k": 0, "pending": [], "last": None, "launched": 0}

    # Consecutive forward batches run on the library's two tracking streams and overlap at their tails (the head of batch k+1 and its
    # preparation fill the last wave of batch k): 345.9k against 342.7k tracks/s serialised (ELLC_OVERLAP=0; tools, profiles/r02_variants.md).
    # Loop-closure batches share the keyframes' weight images and are serialised by the library.
    overlap = os.environ.get("ELLC_OVERLAP", "1") == "1" and not lc

    def note_kernel_time():
        # CUDA events around the tracking kernel of the batch just fetched, on its own stream.  (With ELLC_OVERLAP=1 the kernels of
        # consecutive batches run concurrently: then the completion-to-completion interval is the time a launch occupies the GPU.)
        ms = trk.batch_interval_ms(PIPE_DEPTH) if overlap else trk.batch_kernel_ms(PIPE_DEPTH)
        if ms > 0:
            kernel_ms.append(ms)

    def step_pipelined(e2e=False):
        half = pipe["k"] & 1
        t0 = time.perf_counter()
        if e2e:
            upload_all(half)
        else:
            trk.prepare_async(fr_slots + half * args.frames, kf_slots + half * args.keyframes)
            if lc:
                trk.prepare_keyframes_lc_async(kf_slots + half * args.keyframes)   # the per-keyframe Jacobians / hessians are part of the step
        t1 = time.perf_counter()
        ticket = launch(pairs_half[half])
        pipe["launched"] += 1
        t3 = time.perf_counter()
        host_ms["enqueue"].append(1e3 * (t3 - t0))
        host_ms["prepare"].append(1e3 * (t1 - t0))
        host_ms["launch"].append(1e3 * (t3 - t1))
        if e2e:
            pipe["host_upload_ms"] = pipe.get("host_upload_ms", 0.0) + 1e3 * (t1 - t0)
            pipe["host_launch_ms"] = pipe.get("host_launch_ms", 0.0) + 1e3 * (time.perf_counter() - t1)
        pipe["pending"].append(ticket)
        if len(pipe["pending"]) > PIPE_DEPTH:
            t2 = time.perf_counter()
            pipe["last"] = fetch(pipe["pending"].pop(0))
            host_ms["fetch"].append(1e3 * (time.perf_counter() - t2))
            if not e2e and pipe["launched"] >= PIPE_DEPTH + (2 if overlap else 1):
                note_kernel_time()
        pipe["k"] += 1
        return pipe["last"]

    def drain_pipelined():
        while pipe["pending"]:
            pipe["last"] = fetch(pipe["pending"].pop(0))
        return pipe["last"]

    def step_resident():                                       # loop-closure mode / single-pair latency: one set of slots, no pipelining
        trk.prepare_frames(fr_slots)
        trk.prepare_keyframes(kf_slots)
        if lc:
            trk.prepare_keyframes_lc(kf_slots)                 # the per-keyframe Jacobians / hessians are part of the step
        out = fetch(launch(pairs))
        kernel_ms.append(trk.last_track_kernel_ms())
        return out

    per_rank_ms = []                                           # per timed region: every rank's own ms per step (diagnostic)
    host_ms = {"enqueue": [], "fetch": [], "prepare": [], "launch": []}                     # host time of the two halves of a pipelined step (diagnostic)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, sample_clocks=False, drain=None):
        res = None
        clk = ClockSampler(local_rank) if (sample_clocks and os.environ.get("ELLC_NO_CLOCKS") != "1") else None   # (diagnostic switch)
        if clk:
            clk.start()                                   # sampled over warm-up + timed steps (the same load)
        # The Python collector stays off from here to the end of the timed region (its allocations are a few result arrays per
        # step), and is run NOW, before the warm-up: anything slow between the synchronisation that opens the timed region and its
        # first launch lets the device fall idle, and the first launch after an idle period was measured to block for 1 - 185 ms on
        # the benchmark boxes (host_ms_per_step.launch: always step 0; profiles/r02_host_stalls.md).
        gc.collect()
        gc.disable()
        for _ in range(warmup):
            res = fn()
        if drain:
            r2 = drain()
            res = r2 if r2 is not None else res
        barrier()
        kernel_ms.clear()
        for v in host_ms.values():
            v.clear()
        pipe["launched"] = 0
        trk.reset_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if clk:
            clk.mark_begin()
        e0.record(stream)
        for _ in range(steps):
            res = fn()
        if clk:
            clk.sample_now()                              # the last steps are still running on the device
        if drain:
            r2 = drain()
            res = r2 if r2 is not None else res
        trk.fence()                                       # the event below covers the batches on the tracking streams ...
        stream.wait_stream(torch.cuda.current_stream())   # ... and anything issued on torch's stream
        e1.record(stream)
        barrier()
        gc.enable()
        if clk:
            clk.mark_end()
        ms = e0.elapsed_time(e1)
        launches = trk.launch_count()
        clocks = clk.stop() if clk else None
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            allt = torch.zeros(world, dtype=torch.float64, device="cuda")
            dist.all_gather_into_tensor(allt, t)
            per_rank_ms.append([float(v) / steps for v in allt.cpu().tolist()])
            ms = float(allt.max().item())
        return ms, res, launches, clocks

    pipelined = n_pairs >= 148
    if pipelined:
        ms, res2, launches, clocks = timed(step_pipelined, args.steps, args.warmup, sample_clocks=True, drain=drain_pipelined)
    else:
        ms, res2, launches, clocks = timed(step_resident, args.steps, args.warmup, sample_clocks=True)
    host_diag = {k: {"median": float(np.median(v)), "max": float(np.max(v)), "argmax_step": int(np.argmax(v))} for k, v in host_ms.items() if v}
    own, table = res2 if res2 is not None else (None, None)
    if own is None:                                            # a rank that receives nothing still needs its own counters for the roofline
        own = trk.track_batch(pairs)
    res = own
    k_ms = float(np.mean(kernel_ms)) if kernel_ms else ms / args.steps
    per_rank_kernel_ms = None
    if world > 1:
        kt = torch.zeros(world, dtype=torch.float64, device="cuda")
        dist.all_gather_into_tensor(kt, torch.tensor([k_ms], dtype=torch.float64, device="cuda"))
        per_rank_kernel_ms = [float(v) for v in kt.cpu().tolist()]
    value = n_total * args.steps / (ms * 1e-3)
    alg = algorithmic_bytes(res)
    pix_it = pixel_iterations(res)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg / (k_ms * 1e-3) / 1e9
    # DRAM traffic / executed instructions of the dominant kernel: one `ncu --set full` capture of this command
    # (profiles/r02_traffic.json, made by tools/profile_summary.py), per launch like the algorithmic figure; scaled by pair count if
    # the workload differs.  The file records the library version (a hash of the kernel sources) it was captured with: a capture
    # of another build is refused.
    traffic, traffic_src, inst_launch = None, None, None
    lib_version = capi.lib().ellc_version().decode()
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        if tj.get("library_version") != lib_version:
            traffic_src = "profiles/r02_traffic.json REFUSED: captured with %r, running %r" % (tj.get("library_version"), lib_version)
        elif tj.get("workload", "pair_sweep_640x480") != conf["workload"] or lc:
            traffic_src = "profiles/r02_traffic.json is a capture of another workload"
        else:
            traffic = (tj["dram_bytes_read"] + tj["dram_bytes_write"]) * n_pairs / tj["pairs_per_launch"]
            inst_launch = tj.get("inst_executed", 0) * n_pairs / tj["pairs_per_launch"] or None
            traffic_src = "profiles/r02_traffic.json (%s; dram__bytes_read + write of one launch of %d pairs%s)" % (
                tj["report"], tj["pairs_per_launch"], "" if n_pairs == tj["pairs_per_launch"] else ", scaled by pair count")
    except Exception:
        pass
    sm_mhz = (clocks or {}).get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
    issue_peak = 148 * 4 * sm_mhz * 1e6                        # warp instructions per second: 148 SMs x 4 schedulers x 1 per clock
    sass = sass_inst_per_pixel()
    inst_static = None
    if sass and sass.get("library_version") == lib_version:
        inst_static = sass.get("inst_per_pixel_level0")
    if inst_launch:
        inst_src, inst_used = "ncu smsp__inst_executed.sum of the same capture", inst_launch
    elif inst_static:
        inst_src = "static: SASS instructions per pixel of the level-0 loop's usual path x pixel-iterations / 32 (excludes K5, reductions, prologues)"
        inst_used = inst_static * pix_it / 32.0
    else:
        inst_src, inst_used = None, None
    secondary = None
    if inst_used:
        secondary = {"bound": "issue", "achieved": inst_used / (k_ms * 1e-3), "peak": issue_peak, "unit": "warp-inst/s",
                     "frac": inst_used / (k_ms * 1e-3) / issue_peak, "inst_per_launch": inst_used, "source": inst_src,
                     "inst_per_pixel_iter": inst_used * 32.0 / pix_it,
                     "inst_per_pixel_iter_sass_level0": inst_static,
                     "peak_source": "148 SMs x 4 warp schedulers x %.0f MHz (median SM clock of the timed region)" % sm_mhz}
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_unit": "bytes per launch (compare with algorithmic_bytes_per_launch)", "traffic_source": traffic_src,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                "kernel": "gn_track_lc_kernel + gn_track_kernel" if lc else "gn_track_kernel", "kernel_ms_per_launch": k_ms,
                "kernel_ms_definition": ("completion-to-completion interval of consecutive tracking kernels (ELLC_OVERLAP=1: batches run concurrently)"
                                         if (pipelined and overlap) else "CUDA events around the tracking kernel(s) of a batch on the stream they are launched on, "
                                         "inside the timed loop (the next step's preparation kernels share the GPU with its last wave)"),
                "algorithmic_bytes_per_launch": alg, "pixel_iterations_per_launch": pix_it,
                "kernel_share_of_step": k_ms / (ms / args.steps),
                "mean_iters_per_level": [float(x) for x in res["n_iters"].mean(axis=0)],
                "mean_selected_per_level": [float(x) for x in res["n_selected"].mean(axis=0)],
                "secondary": secondary}

    e2e = None
    if not args.no_e2e and pipelined:
        pipe.update({"k": 0, "pending": [], "last": None})
        ems, eres2, _, _ = timed(lambda: step_pipelined(e2e=True), args.steps, max(1, args.warmup), drain=drain_pipelined)
        e2e = {"value": n_total * args.steps / (ems * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes) * world,
               "d2h_bytes_per_step": int(d2h_bytes_job), "ms_per_step": ems / args.steps,
               "host_enqueue_ms_per_step": {"uploads": pipe.get("host_upload_ms", 0.0) / max(1, pipe["k"]),
                                            "track_launch": pipe.get("host_launch_ms", 0.0) / max(1, pipe["k"])},
               "includes_gather": world > 1,
               "pipelining": "2 slot halves alternate; uploads of step k+1 on the copy stream overlap the kernels of step k; the records of step k "
                             "(N>1: of ALL ranks, gathered on the receiving rank) are fetched during step k+2 (the host runs two steps ahead)"}
        if eres2 is not None and eres2[0] is not None:
            assert np.array_equal(eres2[0]["pose"], res["pose"]), "e2e and resident paths disagree"
    elif not args.no_e2e:
        # small batches (single-pair latency): synchronous through host buffers, every step uploads, tracks and reads back
        def step_e2e_sync():
            upload_all(0)
            return fetch(launch(pairs))
        ems, eres2, _, _ = timed(step_e2e_sync, args.steps, max(1, args.warmup))
        e2e = {"value": n_total * args.steps / (ems * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d_bytes) * world,
               "d2h_bytes_per_step": int(d2h_bytes_job), "ms_per_step": ems / args.steps, "includes_gather": world > 1,
               "pipelining": "none: upload, track, read back, one step after the other"}

    if world > 1 and table is not None:
        # the gathered table is the concatenation of every rank's records at their global indices
        assert np.array_equal(table[my_idx]["pose"], res["pose"])
        assert int((table["n_selected"][:, 0] > 0).sum()) == n_total, "records of some rank are missing from the gathered table"

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import oracle
        cores = os.cpu_count() or 1
        per_pair = (W * H) / (640.0 * 480.0)
        ns = max(1, min(n_pairs, int(max(cores * 256, 1024) / per_pair)))           # ~10-15 s of CPU work on the box's cores
        ocfg = oracle.default_config(W, H, fx=float(k["fx"]), fy=float(k["fy"]), cx=float(k["cx"]), cy=float(k["cy"]))
        oposes, secs = oracle.track_many(ocfg, wl["kf_idx"][:ns], wl["fr_idx"][:ns], wl["kf_images"], wl["frames"], wl["kf_depth"],
                                         wl["kf_var"], wl["init"][:ns], n_workers=cores)
        perr = float(np.abs(oposes - res["pose"][:ns]).max())
        cpu_baseline = {"value": ns / secs, "unit": UNIT, "cores": min(cores, ns), "kind": "port",
                        "sample": f"first {ns} pairs of this step's pair list, {min(cores, ns)} worker threads (1 pair per thread); "
                                  f"max |pose_gpu - pose_cpu| on the sample = {perr:.2e}"}

    if rank == 0:
        gather_desc = {"none": "single GPU", "p2p": "in-kernel stores of the 256 B result records into the result table of %s over NVLink peer memory "
                       "(CUDA IPC; ellc_track_batch_exchange / ellc_exchange_wait), no data-path collective" % ("every rank" if root < 0 else "rank %d" % root),
                       "nccl": "NCCL all-gather of the 256 B result records (1 channel, LL), index_select to the global order"}[xmode]
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": workload_config(conf, args.keyframes, args.frames, args.pairs_per_frame, n_pairs, lc),
                "implementation": {
                    "arithmetic": args.arith, "ctas_per_pair": args.cluster or "auto", "pairs_per_cta": args.pairs_per_cta or "auto", "library": lib_version,
                    "pipelining": ("resident inputs held twice; steps alternate between the two sets of slots: preparation of step k+1 on a "
                                   "low-priority stream overlaps the tracking kernel of step k, records of step k fetched during step k+2 (the host runs two steps ahead of the records it reads)" if pipelined else
                                   "none (one set of slots; every step prepares, tracks and reads back before the next one starts)"),
                    "parallelism": f"pair list sharded by connected components (sequence segments) x{world}; gather: {gather_desc}",
                    "setup_bytes_per_step": setup_bytes(args.frames, args.keyframes) * world, "setup_seconds": setup_s},
                "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks}
        if n_pairs == 1:
            line["latency_ms_per_track"] = ms / args.steps
        if host_diag:
            line["host_ms_per_step"] = dict(host_diag, note="host time of the two halves of a pipelined step on rank 0: enqueue (prepare + launch) and "
                                                                "fetch (blocks until the previous step's records are on the host); a max far above the median "
                                                                "is a host stall that can idle the GPU (the collector is off inside the timed region)")
        if world > 1:
            line["per_rank"] = {"ms_per_step": per_rank_ms[0] if per_rank_ms else None, "kernel_ms_per_launch": per_rank_kernel_ms,
                                "e2e_ms_per_step": per_rank_ms[1] if len(per_rank_ms) > 1 else None,
                                "note": "every rank tracks its own seeded segment: iteration counts, hence kernel times, differ a little between ranks"}
        emit(line)
    if args.dump_outputs and rank == max(root, 0):
        dump_outputs(args.dump_outputs, table)     # the rank that receives the gathered table (--exchange-root; N = 1: its own records)
    trk.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
