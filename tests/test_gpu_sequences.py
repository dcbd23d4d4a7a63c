"""ellc_track_sequence_steps: frame sequences tracked with the pose chain (initial pose from the previous frame, world pose through the
keyframe) on the device.  Every record and world pose must equal, bit for bit, the host loop the call replaces: one ellc_track_batch
per frame (or per wave) and ellc_concat_origin / ellc_concat_relative on the host (src/ImageFunc.cpp:97-108, :305-306)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from tests.helpers import gpu_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def capi():
    import __graft_entry__ as g
    g.build()
    from egomotion_with_local_loop_closures_b200 import capi as m
    return m


# ---- CPU: ABI layout -------------------------------------------------------------------------------------------------------------
def test_seq_step_layout_matches_header(capi):
    hdr = open(os.path.join(ROOT, "include", "ellc_gn.h")).read()
    body = re.search(r"typedef struct ellc_seq_step \{(.*?)\} ellc_seq_step;\s*/\* (\d+) B \*/", hdr, re.S)
    assert body, "ellc_seq_step not found in include/ellc_gn.h"
    fields = re.findall(r"\b(\w+)(?:\[(\d+)\])?\s*[,;]", re.sub(r"/\*.*?\*/", "", body.group(1), flags=re.S))
    names = [f for f, _ in fields if f not in ("int32_t", "float")]
    assert names == [f[0] for f in capi.SeqStep._fields_]
    assert C.sizeof(capi.SeqStep) == capi.SEQ_STEP_DTYPE.itemsize == int(body.group(2)) == 72
    offsets = dict(kf_slot=0, frame_slot=4, prev_step=8, kf_step=12, prev_world=16, kf_world=40, flags=64, reserved=68)
    for name, off in offsets.items():
        assert getattr(capi.SeqStep, name).offset == off, name
        assert capi.SEQ_STEP_DTYPE.fields[name][1] == off, name


def test_sequence_symbol_exported(capi):
    assert "ellc_track_sequence_steps" in capi.SYMBOLS
    assert capi.lib().ellc_track_sequence_steps is not None


# ---- GPU -------------------------------------------------------------------------------------------------------------------------
def _host_loop(t, capi, steps):
    """The loop ellc_track_sequence_steps replaces: the steps' waves in order, one ellc_track_batch per wave, the pose chain on the
    host.  Returns (results, world) in input order."""
    n = len(steps)
    wave = np.zeros(n, np.int64)
    for i in range(n):
        wave[i] = 1 + max(wave[d] if d >= 0 else -1 for d in (int(steps[i]["prev_step"]), int(steps[i]["kf_step"])))
    res = np.zeros(n, capi.RESULT_DTYPE)
    world = np.zeros((n, 6), np.float32)

    def w_of(dep, value):
        return world[dep] if dep >= 0 else value

    for w in range(int(wave.max()) + 1 if n else 0):
        idx = [i for i in range(n) if wave[i] == w]
        inits = [capi.concat_origin(w_of(int(steps[i]["prev_step"]), steps[i]["prev_world"]),
                                    w_of(int(steps[i]["kf_step"]), steps[i]["kf_world"])) for i in idx]
        r = t.track_batch(t.make_pairs([int(steps[i]["kf_slot"]) for i in idx], [int(steps[i]["frame_slot"]) for i in idx], inits,
                                       flags=[int(steps[i]["flags"]) for i in idx]))
        for k, i in enumerate(idx):
            res[i] = r[k]
            world[i] = capi.concat_relative(r[k]["pose"], w_of(int(steps[i]["kf_step"]), steps[i]["kf_world"]))
    return res, world


def _chain_steps(capi, frame_slots, kf_slot_of, interval, root_world, flags=0):
    """Steps of one sequence as src/ImageFunc.cpp drives it: frame r = 1..L (frame 0 is the first keyframe, world pose root_world
    given by value), tracked against keyframe frame interval * ((r - 1) // interval); every interval-th tracked frame becomes the
    next keyframe.  kf_slot_of(r) is the keyframe slot holding frame r."""
    L = len(frame_slots)
    steps = capi.Tracker.make_steps([kf_slot_of(interval * ((r - 1) // interval)) for r in range(1, L + 1)], frame_slots,
                                    [r - 2 for r in range(1, L + 1)],
                                    [interval * ((r - 1) // interval) - 1 for r in range(1, L + 1)],
                                    prev_world=[root_world] * L, kf_world=[root_world] * L, flags=flags)
    return steps


def _same(a, b):
    return a.tobytes() == b.tobytes()


@pytest.fixture(scope="module")
def config1():
    """BASELINE config 1: 640x480, 100 frames of a smooth trajectory, a keyframe (ground-truth depth) every 8 frames."""
    from egomotion_with_local_loop_closures_b200 import synth
    w, h, n = 640, 480, 100
    scene = synth.SynthScene(w, h)
    T = synth.smooth_trajectory(n, seed_pose=91011)
    imgs = [None] + [scene.render(T[i], noise_seed=7000 + i) for i in range(1, n)]
    kfs = {i: scene.keyframe(T[i], seed_depth=5678 + i, noise_seed=7000 + i) for i in range(0, n - 1, 8)}
    return dict(width=w, height=h, n=n, T=T, imgs=imgs, kfs=kfs)


def _config1_tracker(capi, case, arith):
    cfg = gpu_config(capi, case, max_keyframes=len(case["kfs"]), max_frames=case["n"], arithmetic=arith)
    t = capi.Tracker(cfg)
    for i, kf in case["kfs"].items():
        t.upload_keyframe(i // 8, kf["image"], kf["depth"], kf["var"])
    for i in range(1, case["n"]):
        t.upload_frame(i, case["imgs"][i])
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("arith", ["FAST", "STRICT", "REFERENCE"])
def test_config1_one_call_equals_host_loop(capi, config1, arith):
    """All 99 tracks of config 1 (13 keyframes resident) in one call: every record and world pose equals the existing host loop's
    (test_gpu_parity.test_config1_sequence_100_frames_640x480) on the same handle, bit for bit."""
    from egomotion_with_local_loop_closures_b200 import synth
    t = _config1_tracker(capi, config1, getattr(capi, "ARITH_" + arith))
    n = config1["n"]
    zero = np.zeros(6, np.float32)
    # the host loop exactly as the existing config-1 test writes it
    g_world = [zero]
    loop_res = []
    kf_id = 0
    for i in range(1, n):
        g_init = capi.concat_origin(g_world[i - 1], g_world[kf_id])
        r = t.track_batch(t.make_pairs([kf_id // 8], [i], [g_init]))[0]
        loop_res.append(r)
        g_world.append(capi.concat_relative(r["pose"], g_world[kf_id]))
        if i % 8 == 0 and i + 1 < n:
            kf_id = i
    steps = _chain_steps(capi, list(range(1, n)), lambda r: r // 8, 8, zero)
    t.reset_launch_count()
    res, world = t.track_sequence_steps(steps)
    launches = t.launch_count()
    assert _same(res, np.array(loop_res, capi.RESULT_DTYPE))
    assert _same(world, np.array(g_world[1:], np.float32))
    assert launches <= 3 * (n - 1) + 4, launches                # per frame: the tracking kernel and two chain kernels
    assert np.abs(world[-1] - synth.relative_pose(config1["T"][n - 1], config1["T"][0])).max() < 5e-3
    t.close()


@pytest.fixture(scope="module")
def ragged():
    """Two 320x240 scenes, 41 frames each; keyframes at every frame index some sequence uses as a keyframe."""
    from egomotion_with_local_loop_closures_b200 import synth
    w, h, nf = 320, 240, 41
    scenes = []
    for sc in range(2):
        scene = synth.SynthScene(w, h, seed_tex=1234 + 17 * sc)
        T = synth.smooth_trajectory(nf, seed_pose=500 + sc)
        scenes.append(dict(scene=scene, T=T, imgs=[scene.render(T[i], noise_seed=900 * sc + i) for i in range(nf)]))
    rng = np.random.default_rng(7)
    seqs = []
    for s in range(24):
        L = 1 + (s * 17) % 40                                   # lengths 1 .. 40
        seqs.append(dict(scene=s % 2, L=L, interval=(3, 5, 8)[s % 3], start=int(rng.integers(0, nf - L)),
                         root=(rng.standard_normal(6) * [0.05, 0.05, 0.05, 0.2, 0.2, 0.2]).astype(np.float32)))
    kf_frames = sorted({(q["scene"], q["start"] + k) for q in seqs for k in range(0, q["L"], q["interval"])})
    kf_slot = {key: i for i, key in enumerate(kf_frames)}
    kfs = {key: scenes[key[0]]["scene"].keyframe(scenes[key[0]]["T"][key[1]], seed_depth=31 * key[1] + key[0], noise_seed=900 * key[0] + key[1])
           for key in kf_frames}
    return dict(width=w, height=h, nf=nf, scenes=scenes, seqs=seqs, kf_slot=kf_slot, kfs=kfs)


def _ragged_tracker(capi, case, **over):
    t = capi.Tracker(gpu_config(capi, case, max_keyframes=len(case["kf_slot"]) + 1, max_frames=2 * case["nf"] + 2, **over))
    for key, slot in case["kf_slot"].items():
        kf = case["kfs"][key]
        t.upload_keyframe(slot, kf["image"], kf["depth"], kf["var"])
    for sc in range(2):
        for i in range(case["nf"]):
            t.upload_frame(sc * case["nf"] + i, case["scenes"][sc]["imgs"][i])
    return t


def _ragged_seq_steps(capi, case, q, flags=0):
    sc, o = q["scene"], q["start"]
    return _chain_steps(capi, [sc * case["nf"] + o + r for r in range(1, q["L"] + 1)], lambda r: case["kf_slot"][(sc, o + r)],
                        q["interval"], q["root"], flags=flags)


def _topological_shuffle(steps, rng):
    """A random order of the steps in which every step still follows its dependencies; the dependencies renumbered."""
    n = len(steps)
    placed, order = np.zeros(n, bool), []
    while len(order) < n:
        ready = [i for i in range(n) if not placed[i] and all(d < 0 or placed[d] for d in (steps[i]["prev_step"], steps[i]["kf_step"]))]
        i = ready[int(rng.integers(0, len(ready)))]
        placed[i] = True
        order.append(i)
    pos = np.empty(n, np.int64)
    pos[order] = np.arange(n)
    out = steps[order].copy()
    for f in ("prev_step", "kf_step"):
        out[f] = np.where(out[f] >= 0, pos[np.maximum(out[f], 0)], -1)
    return out, np.array(order)


@pytest.mark.gpu
@pytest.mark.parametrize("const_weight", [False, True])
def test_ragged_sequences_shuffled_equal_their_own_host_loops(capi, ragged, const_weight):
    """24 sequences of lengths 1..40, keyframe intervals 3 / 5 / 8, two scenes, roots given by value, all in one call with the steps
    shuffled (dependency order kept): every sequence equals its own host loop (one ellc_track_batch per frame).  With const_weight,
    every third sequence is tracked with the constant-weight variant, so waves mix the two tracking kernels."""
    t = _ragged_tracker(capi, ragged)
    flags_of = [capi.PAIR_CONST_WEIGHT if const_weight and s % 3 == 1 else 0 for s in range(len(ragged["seqs"]))]
    if const_weight:
        slots = sorted(ragged["kf_slot"].values())
        for slot in slots:
            rng = np.random.default_rng(slot)
            t.upload_keyframe_weights(slot, [rng.uniform(0.2, 1.0, (ragged["height"] >> l, ragged["width"] >> l)).astype(np.float32)
                                             for l in range(4)], [1, 1, 1, 1])
        t.prepare_keyframes_lc(slots)
    per_seq = [_ragged_seq_steps(capi, ragged, q, flags_of[s]) for s, q in enumerate(ragged["seqs"])]
    want = [_host_loop(t, capi, st) for st in per_seq]
    base = np.cumsum([0] + [len(st) for st in per_seq])
    allsteps = np.concatenate(per_seq)
    for s, st in enumerate(per_seq):                             # renumber into the concatenation
        for f in ("prev_step", "kf_step"):
            allsteps[f][base[s]:base[s + 1]] = np.where(st[f] >= 0, st[f] + base[s], -1)
    shuffled, order = _topological_shuffle(allsteps, np.random.default_rng(11))
    res, world = t.track_sequence_steps(shuffled)
    back = np.empty(len(order), np.int64)
    back[order] = np.arange(len(order))
    for s in range(len(per_seq)):
        idx = back[base[s]:base[s + 1]]
        assert _same(res[idx], want[s][0]), s
        assert _same(world[idx], want[s][1]), s
    t.close()


def _concat_steps(per_seq):
    """The steps of several sequences in one array, dependencies renumbered into it; also the offset of every sequence."""
    base = np.cumsum([0] + [len(st) for st in per_seq])
    allsteps = np.concatenate(per_seq)
    for s, st in enumerate(per_seq):
        for f in ("prev_step", "kf_step"):
            allsteps[f][base[s]:base[s + 1]] = np.where(st[f] >= 0, st[f] + base[s], -1)
    return allsteps, base


@pytest.mark.gpu
def test_save_weights_steps_write_the_host_loops_weight_images(capi, ragged):
    """ELLC_PAIR_SAVE_WEIGHTS steps (src/ImageFunc.cpp:280-288) inside a sequence call: on a fresh handle the call leaves the same
    weight images in the frame slots as the host loop leaves on another fresh handle, and the same records and world poses.  The
    longest sequence of each scene saves weights (no other flagged step tracks its frames); four more sequences run unflagged in the
    same waves."""
    seqs = ragged["seqs"]
    flagged = [max((s for s in range(len(seqs)) if seqs[s]["scene"] == sc), key=lambda s: seqs[s]["L"]) for sc in range(2)]
    chosen = flagged + [s for s in range(1, 7) if s not in flagged][:4]
    per_seq = [_ragged_seq_steps(capi, ragged, seqs[s], capi.PAIR_SAVE_WEIGHTS if s in flagged else 0) for s in chosen]
    frames = sorted({int(f) for k, s in enumerate(chosen) if s in flagged for f in per_seq[k]["frame_slot"]})

    def weights(t):
        return [t.read_frame_weights(f, l) for f in frames for l in range(4)]

    t_loop = _ragged_tracker(capi, ragged)
    want = [_host_loop(t_loop, capi, st) for st in per_seq]
    w_loop = weights(t_loop)
    t_loop.close()
    t_seq = _ragged_tracker(capi, ragged)
    allsteps, base = _concat_steps(per_seq)
    shuffled, order = _topological_shuffle(allsteps, np.random.default_rng(13))
    res, world = t_seq.track_sequence_steps(shuffled)
    w_seq = weights(t_seq)
    t_seq.close()
    back = np.empty(len(order), np.int64)
    back[order] = np.arange(len(order))
    for k in range(len(per_seq)):
        idx = back[base[k]:base[k + 1]]
        assert _same(res[idx], want[k][0]) and _same(world[idx], want[k][1]), chosen[k]
    assert all(np.count_nonzero(w) > 0 for w in w_loop[::4])          # level 0 of every flagged frame was written
    for a, b in zip(w_seq, w_loop):
        assert _same(a, b)


@pytest.mark.gpu
def test_roots_by_value_and_split_calls(capi, ragged):
    """A sequence split into two calls, the second seeded by value from the first call's world poses, equals the unsplit call; and
    the unsplit call equals the host loop (root pose given by value, not zero)."""
    t = _ragged_tracker(capi, ragged)
    q = max(ragged["seqs"], key=lambda q: q["L"])
    steps = _ragged_seq_steps(capi, ragged, q)
    res, world = t.track_sequence_steps(steps)
    want_res, want_world = _host_loop(t, capi, steps)
    assert _same(res, want_res) and _same(world, want_world)
    for k in (1, q["interval"], q["interval"] + 1, len(steps) - 1):
        r1, w1 = t.track_sequence_steps(steps[:k])
        tail = steps[k:].copy()
        for f, v in (("prev_step", "prev_world"), ("kf_step", "kf_world")):
            early = tail[f] >= 0
            early &= tail[f] < k
            tail[v][early] = w1[tail[f][early]]
            tail[f] = np.where(early, -1, np.where(tail[f] >= k, tail[f] - k, tail[f]))
        r2, w2 = t.track_sequence_steps(tail)
        assert _same(np.concatenate([r1, r2]), res), k
        assert _same(np.concatenate([w1, w2]), world), k
    t.close()


@pytest.mark.gpu
def test_invalid_steps_launch_nothing(capi, ragged):
    t = _ragged_tracker(capi, ragged)
    q = ragged["seqs"][5]
    good = _ragged_seq_steps(capi, ragged, q)
    assert len(good) >= 3
    L = capi.lib()

    def call(steps):
        steps = np.ascontiguousarray(steps, capi.SEQ_STEP_DTYPE)
        res = np.zeros(max(1, len(steps)), capi.RESULT_DTYPE)
        world = np.zeros((max(1, len(steps)), 6), np.float32)
        return L.ellc_track_sequence_steps(t._h, len(steps), capi._p(steps), capi._p(res), capi._p(world))

    assert call(good[:0]) == 0
    t.reset_launch_count()
    for field, value, rc in (("prev_step", 2, -1),            # itself: not an earlier step
                             ("prev_step", 5, -1),            # a later step
                             ("kf_step", -2, -1),             # out of range
                             ("kf_slot", 10 ** 6, -1),        # slot out of range
                             ("frame_slot", 2 * ragged["nf"] + 1, -3),   # never uploaded
                             ("kf_slot", len(ragged["kf_slot"]), -3),
                             ("flags", capi.PAIR_CONST_WEIGHT | capi.PAIR_SAVE_WEIGHTS, -1)):
        bad = good.copy()
        bad[2][field] = value
        assert call(bad) == rc, (field, value)
    assert L.ellc_track_sequence_steps(t._h, -1, None, None, None) == -1
    assert t.launch_count() == 0
    t.close()


@pytest.mark.gpu
def test_async_batch_in_flight_is_left_alone(capi, ragged):
    """An ellc_track_batch_async batch on other slots is in flight while the sequence call runs: its downloaded records equal those of
    the same batch tracked alone, and the sequence equals its host loop."""
    t = _ragged_tracker(capi, ragged)
    nf = ragged["nf"]
    q = max((q for q in ragged["seqs"] if q["scene"] == 0), key=lambda q: q["L"])
    steps = _ragged_seq_steps(capi, ragged, q)
    other = [slot for (sc, _), slot in ragged["kf_slot"].items() if sc == 1][:4]       # scene 1: no slot of the sequence
    pairs = t.make_pairs([other[i % len(other)] for i in range(40)], [nf + i for i in range(40)],
                         np.random.default_rng(3).standard_normal((40, 6)).astype(np.float32) * 0.01)
    alone = t.track_batch(pairs)
    want = _host_loop(t, capi, steps)
    dres = t.track_batch_async(pairs)
    res, world = t.track_sequence_steps(steps)
    got = t.results_download(dres, len(pairs))
    assert _same(got, alone)
    assert _same(res, want[0]) and _same(world, want[1])
    t.close()


@pytest.mark.gpu
def test_launch_count_per_wave(capi, ragged):
    """Launches of one call: per wave the tracking kernel(s) and two chain kernels (world poses of the wave, initial poses of the
    next), within (tracking launches per wave + 2) x waves + a constant."""
    t = _ragged_tracker(capi, ragged)
    per_seq = [_ragged_seq_steps(capi, ragged, q) for q in ragged["seqs"][:6]]
    base = np.cumsum([0] + [len(st) for st in per_seq])
    allsteps = np.concatenate(per_seq)
    for s, st in enumerate(per_seq):
        for f in ("prev_step", "kf_step"):
            allsteps[f][base[s]:base[s + 1]] = np.where(st[f] >= 0, st[f] + base[s], -1)
    waves = max(len(st) for st in per_seq)
    t.prepare_frames(list(range(2 * ragged["nf"])))                      # every uploaded slot: preparation kernels are not the call's
    t.prepare_keyframes(sorted(ragged["kf_slot"].values()))
    t.reset_launch_count()
    t.track_sequence_steps(allsteps)
    got = t.launch_count()
    assert got <= (1 + 2) * waves + 4, (got, waves)
    assert got == 3 * waves + 1, (got, waves)               # staged steps + initial poses of wave 0; per wave track, world, init (not after the last)
    t.close()
