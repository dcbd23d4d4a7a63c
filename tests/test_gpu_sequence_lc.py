"""ellc_track_sequence_lc: sequences in ELLC's constant-weight loop-closure mode in one call.  Every output must equal, bit for bit,
the composition of existing entry points the call replaces: ellc_track_sequence_steps with ELLC_PAIR_SAVE_WEIGHTS steps; per keyframe
ellc_accumulate_weights (its frames in tracking order), ellc_finalise_weights, ellc_prepare_keyframes_lc; ellc_frame_histograms; per
query ellc_lc_generate_pairs on the ring as it stood after that keyframe's push (built on the host from the downloaded world poses)
and ellc_track_generated_pairs (src/ImageFunc.cpp:280-288, src/main.cpp:431-434, src/GlobalOptimize.cpp:151, :274-420, :560-568)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from tests.helpers import gpu_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MMD, THR, ANG = 8, 0.1, 10.0                                     # util::MIN_MATCH_DIFFERENCE, match threshold, max view angle


@pytest.fixture(scope="module")
def capi():
    import __graft_entry__ as g
    g.build()
    from egomotion_with_local_loop_closures_b200 import capi as m
    return m


# ---- CPU: ABI layout -------------------------------------------------------------------------------------------------------------
def _header_struct(name):
    hdr = open(os.path.join(ROOT, "include", "ellc_gn.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;\s*/\* (\d+) B \*/" % (name, name), hdr, re.S)
    assert body, name + " not found in include/ellc_gn.h"
    fields = re.findall(r"\b(\w+)(?:\[(\d+)\])?\s*[,;]", re.sub(r"/\*.*?\*/", "", body.group(1), flags=re.S))
    return [f for f, _ in fields if f not in ("int32_t", "float")], int(body.group(2))


def test_lc_keyframe_layout_matches_header(capi):
    names, size = _header_struct("ellc_lc_keyframe")
    assert names == [f[0] for f in capi.LcKeyframe._fields_] == list(capi.LC_KEYFRAME_DTYPE.names)
    assert C.sizeof(capi.LcKeyframe) == capi.LC_KEYFRAME_DTYPE.itemsize == size == 72
    offsets = dict(kf_slot=0, frame_slot=4, frame_id=8, world_step=12, world=16, retire_before=40, ring=44, ring_pos=48,
                   current_array_id=52, match_window_beg=56, match_window_end=60, stray=64, reserved=68)
    for name, off in offsets.items():
        assert getattr(capi.LcKeyframe, name).offset == off, name
        assert capi.LC_KEYFRAME_DTYPE.fields[name][1] == off, name


def test_lc_ring_params_layout_matches_header(capi):
    names, size = _header_struct("ellc_lc_ring_params")
    assert names == [f[0] for f in capi.LcRingParams._fields_]
    assert C.sizeof(capi.LcRingParams) == size == 24
    offsets = dict(n_rings=0, ring_len=4, min_match_difference=8, match_threshold=12, max_rel_view_angle=16, reserved=20)
    for name, off in offsets.items():
        assert getattr(capi.LcRingParams, name).offset == off, name


def test_sequence_lc_symbol_exported(capi):
    assert "ellc_track_sequence_lc" in capi.SYMBOLS
    assert capi.lib().ellc_track_sequence_lc is not None


# ---- the reference composition ---------------------------------------------------------------------------------------------------
def _waves(steps):
    n = len(steps)
    wave = np.zeros(n, np.int64)
    for i in range(n):
        wave[i] = 1 + max(wave[d] if d >= 0 else -1 for d in (int(steps[i]["prev_step"]), int(steps[i]["kf_step"])))
    return wave


def _composition(t, capi, steps, kfs, ring_in):
    """What ellc_track_sequence_lc replaces, from existing entry points only.  Returns the same dict as Tracker.track_sequence_lc."""
    res, world = t.track_sequence_steps(steps)
    wave = _waves(steps)
    track_order = sorted(range(len(steps)), key=lambda i: (wave[i], i))
    for kf in kfs:
        frames = [int(steps[i]["frame_slot"]) for i in track_order
                  if int(steps[i]["kf_slot"]) == int(kf["kf_slot"]) and int(steps[i]["flags"]) & capi.PAIR_SAVE_WEIGHTS]
        if frames:
            t.accumulate_weights(int(kf["kf_slot"]), frames)
    retired = [k for k in range(len(kfs)) if kfs[k]["retire_before"] >= 0]
    for k in retired:
        t.finalise_weights(int(kfs[k]["kf_slot"]))
        t.prepare_keyframes_lc([int(kfs[k]["kf_slot"])])
    if retired:
        t.frame_histograms([int(kfs[k]["frame_slot"]) for k in retired])
    rings = np.array(ring_in, capi.LC_RING_DTYPE, copy=True)
    out = dict(pairs=[], stats=[], qi=[], lres=[])
    for k in retired:
        kf = kfs[k]
        w = world[int(kf["world_step"])] if kf["world_step"] >= 0 else kf["world"]
        ring = rings[int(kf["ring"])]
        ring[int(kf["ring_pos"])] = (kf["frame_id"], 1, kf["frame_slot"], kf["kf_slot"], w)      # pushToArray
        q = np.zeros(1, capi.LC_QUERY_DTYPE)
        q[0] = (kf["current_array_id"], kf["match_window_beg"], kf["match_window_end"], kf["frame_id"], kf["frame_slot"], kf["stray"], w)
        p, s, qi = t.lc_generate_pairs(ring.copy(), q, min_match_difference=MMD, match_threshold=THR, max_rel_view_angle=ANG,
                                       pair_flags=capi.PAIR_CONST_WEIGHT)
        out["pairs"].append(p); out["stats"].append(s); out["qi"].append(np.full(len(p), k, np.int32))
        out["lres"].append(t.track_generated_pairs(len(p)))
    cat = lambda xs, dt: np.concatenate(xs) if xs else np.zeros(0, dt)
    return dict(results=res, world=world, lc_pairs=cat(out["pairs"], capi.PAIR_DTYPE), lc_stats=cat(out["stats"], capi.LC_STATS_DTYPE),
                lc_query_of_pair=cat(out["qi"], np.int32), lc_results=cat(out["lres"], capi.RESULT_DTYPE), ring_out=rings)


def _weights(t, kf_slots):
    return [t.read_keyframe_weights(int(s), l) for s in kf_slots for l in range(4)]


def _reset(t, kf_slots):
    for s in kf_slots:
        t.reset_keyframe_weights(int(s))


def _same(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def _same_weights(wa, wb):
    return all(_same(a[0], b[0]) and a[1] == b[1] for a, b in zip(wa, wb)) and len(wa) == len(wb)


def _assert_equal(got, want):
    for key in ("results", "world", "lc_pairs", "lc_stats", "lc_query_of_pair", "lc_results", "ring_out"):
        assert _same(got[key], want[key]), key


def _chain(capi, frame_slots, kf_slot_of, interval, root, flags):
    """Steps of one sequence: frame r = 1..L against keyframe frame interval * ((r - 1) // interval); frame 0 (world pose root)
    is the first keyframe."""
    L = len(frame_slots)
    kff = [interval * ((r - 1) // interval) for r in range(1, L + 1)]
    return capi.Tracker.make_steps([kf_slot_of(f) for f in kff], frame_slots, [r - 2 for r in range(1, L + 1)], [f - 1 for f in kff],
                                   prev_world=[root] * L, kf_world=[root] * L, flags=flags)


def _keyframes(capi, L, interval, kf_slot_of, kf_frame_slot_of, root, ring_len, query_of, ring=0, id_base=0):
    """One ellc_lc_keyframe per keyframe frame 0, interval, ... <= L - 1 of a sequence of L tracked frames: keyframe frame f is made
    by the step that tracked it (f - 1) and retired when the next keyframe is made (before step f + interval), the last one stays
    active.  query_of(j) -> (ring_pos, current_array_id, beg, end, stray) of the j-th keyframe."""
    kff = list(range(0, L, interval))
    kfs = capi.Tracker.make_lc_keyframes([kf_slot_of(f) for f in kff], [kf_frame_slot_of(f) for f in kff], [id_base + f for f in kff],
                                         [f - 1 for f in kff], world=[root] * len(kff))
    for j, f in enumerate(kff):
        if j + 1 < len(kff):
            pos, cur, beg, end, stray = query_of(j)
            kfs[j]["retire_before"] = f + interval
            kfs[j]["ring"], kfs[j]["ring_pos"], kfs[j]["current_array_id"] = ring, pos, cur
            kfs[j]["match_window_beg"], kfs[j]["match_window_end"], kfs[j]["stray"] = beg, end, stray
    return kfs


def _empty_ring(capi, n_rings, ring_len):
    return np.zeros((n_rings, ring_len), capi.LC_RING_DTYPE)


# ---- 1. BASELINE config 1 in LC mode ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def config1():
    """640x480, 100 frames of a smooth trajectory, a keyframe (ground-truth depth) every 8 frames: 13 keyframes, 12 retired."""
    from egomotion_with_local_loop_closures_b200 import synth
    w, h, n = 640, 480, 100
    scene = synth.SynthScene(w, h)
    T = synth.smooth_trajectory(n, seed_pose=91011)
    imgs = [None] + [scene.render(T[i], noise_seed=7000 + i) for i in range(1, n)]
    kfs = {i: scene.keyframe(T[i], seed_depth=5678 + i, noise_seed=7000 + i) for i in range(0, n - 1, 8)}
    return dict(width=w, height=h, n=n, imgs=imgs, kfs=kfs)


@pytest.mark.gpu
@pytest.mark.parametrize("arith", ["FAST", "STRICT", "REFERENCE"])
def test_config1_lc_mode_equals_composition(capi, config1, arith):
    """All 99 tracks saving weights, 12 keyframes retired into a ring of 43 (pushed at 0..11, each query walking down to the first
    empty position): records, world poses, every keyframe's weight pyramid and counts, the pair list, its statistics and records
    equal the composition's byte for byte, and loop-closure pairs do pass the gate."""
    n, K = config1["n"], len(config1["kfs"])
    t = capi.Tracker(gpu_config(capi, config1, max_keyframes=K, max_frames=n + K, arithmetic=getattr(capi, "ARITH_" + arith)))
    for i, kf in config1["kfs"].items():
        t.upload_keyframe(i // 8, kf["image"], kf["depth"], kf["var"])
        t.upload_frame(n + i // 8, kf["image"])                  # the keyframe's image as a frame: histogram, test frame of its query
    for i in range(1, n):
        t.upload_frame(i, config1["imgs"][i])
    zero = np.zeros(6, np.float32)
    steps = _chain(capi, list(range(1, n)), lambda f: f // 8, 8, zero, capi.PAIR_SAVE_WEIGHTS)
    kfs = _keyframes(capi, n, 8, lambda f: f // 8, lambda f: n + f // 8, zero, 43, lambda j: (j, j + 1, 0, 0, 0))
    assert int((kfs["retire_before"] >= 0).sum()) == 12
    ring0 = _empty_ring(capi, 1, 43)
    slots = list(range(K))
    _reset(t, slots)
    want = _composition(t, capi, steps, kfs, ring0)
    w_want = _weights(t, slots)
    _reset(t, slots)
    got = t.track_sequence_lc(steps, kfs, ring0, min_match_difference=MMD, match_threshold=THR, max_rel_view_angle=ANG)
    w_got = _weights(t, slots)
    _assert_equal(got, want)
    assert _same_weights(w_got, w_want)
    assert [c for _, c in w_got[::4]] == [8] * 12 + [3]          # frames per keyframe (the last one's 3 frames: 97, 98, 99)
    assert len(got["lc_pairs"]) >= 5, len(got["lc_pairs"])
    assert np.all(got["lc_stats"]["pass"] == 1) and np.all(got["lc_pairs"]["flags"] == capi.PAIR_CONST_WEIGHT)
    t.close()


# ---- a small scene for the ring, split, multi-sequence, validation and launch-count tests -----------------------------------------
@pytest.fixture(scope="module")
def small():
    """320x240: four sequences of their own frames in one scene (lengths 48, 29, 37, 21; keyframe intervals 4, 3, 5, 4)."""
    from egomotion_with_local_loop_closures_b200 import synth
    w, h = 320, 240
    scene = synth.SynthScene(w, h, seed_tex=4321)
    seqs, fbase, kbase = [], 0, 0
    for s, (L, interval) in enumerate(((48, 4), (29, 3), (37, 5), (21, 4))):
        T = synth.smooth_trajectory(L + 1, seed_pose=300 + s)
        kff = list(range(0, L, interval))
        seqs.append(dict(L=L, interval=interval, fbase=fbase, kbase=kbase, kff=kff,
                         imgs=[scene.render(T[i], noise_seed=100 * s + i) for i in range(L + 1)],
                         kfs={f: scene.keyframe(T[f], seed_depth=40 * s + f, noise_seed=100 * s + f) for f in kff},
                         root=np.array([0.01 * s, -0.02, 0.005 * s, 0.03, 0.0, -0.01 * s], np.float32)))
        fbase += (L + 1) + len(kff)                               # frames 1..L at fbase + r, keyframe images behind them
        kbase += len(kff)
    return dict(width=w, height=h, seqs=seqs, n_frames=fbase, n_kf=kbase)


def _small_tracker(capi, case, **over):
    t = capi.Tracker(gpu_config(capi, case, max_keyframes=case["n_kf"] + 2, max_frames=case["n_frames"] + 2, **over))
    for q in case["seqs"]:
        for j, f in enumerate(q["kff"]):
            kf = q["kfs"][f]
            t.upload_keyframe(q["kbase"] + j, kf["image"], kf["depth"], kf["var"])
            t.upload_frame(q["fbase"] + q["L"] + 1 + j, kf["image"])
        for r in range(1, q["L"] + 1):
            t.upload_frame(q["fbase"] + r, q["imgs"][r])
    return t


def _seq_steps(capi, q):
    return _chain(capi, [q["fbase"] + r for r in range(1, q["L"] + 1)], lambda f: q["kbase"] + f // q["interval"], q["interval"], q["root"],
                  capi.PAIR_SAVE_WEIGHTS)


def _seq_kfs(capi, q, ring_len, query_of, ring=0):
    return _keyframes(capi, q["L"], q["interval"], lambda f: q["kbase"] + f // q["interval"],
                      lambda f: q["fbase"] + q["L"] + 1 + f // q["interval"], q["root"], ring_len, query_of, ring=ring)


def _mixed_queries(ring_len, start=2):
    """Pushes at (start + j) % ring_len; queries by j % 4: walk to the first empty position, a window of 3 below the push (wraps at
    small positions), a stray query, a window holding only the keyframe itself (no candidate)."""
    def query_of(j):
        pos = (start + j) % ring_len
        kind = j % 4
        if kind == 0:
            return pos, pos + 1, 0, 0, 0
        if kind == 1:
            return pos, pos + 1, (pos - 3) % ring_len, pos, 0
        if kind == 2:
            return pos, pos + 1, 0, 0, 1
        return pos, pos + 1, pos, (pos + 1) % ring_len, 0
    return query_of


# ---- 2. ring wrap and overwrite ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_small_ring_wraps_and_later_pushes_stay_invisible(capi, small):
    """11 keyframes retired into a ring of 5 (every position overwritten, some twice): each query sees the ring as of its own push.
    The call equals the composition with the ring as of each push, which differs from walking the final ring.  Covered: empty
    (invalid) positions that end a walk, stray queries, windows that wrap, queries with no candidate."""
    q = small["seqs"][0]
    t = _small_tracker(capi, small)
    steps = _seq_steps(capi, q)
    kfs = _seq_kfs(capi, q, 5, _mixed_queries(5))
    ret = [k for k in range(len(kfs)) if kfs[k]["retire_before"] >= 0]
    assert len(ret) == 11
    slots = [int(s) for s in kfs["kf_slot"]]
    ring0 = _empty_ring(capi, 1, 5)
    _reset(t, slots)
    want = _composition(t, capi, steps, kfs, ring0)
    w_want = _weights(t, slots)
    _reset(t, slots)
    got = t.track_sequence_lc(steps, kfs, ring0, min_match_difference=MMD, match_threshold=THR, max_rel_view_angle=ANG)
    _assert_equal(got, want)
    assert _same_weights(_weights(t, slots), w_want)
    qi, pos = got["lc_query_of_pair"], got["lc_stats"]["reserved"]
    n_of = {k: int((qi == k).sum()) for k in ret}
    assert any(n_of[k] > 0 for k in ret if kfs[k]["stray"]), n_of                       # stray queries match
    assert all(n_of[k] == 0 for k in ret if k % 4 == 3), n_of                           # only the keyframe itself in the window
    assert any(kfs[k]["match_window_beg"] > kfs[k]["match_window_end"] and n_of[k] > 0 for k in ret), n_of     # a wrapped window used
    overwritten = [(int(k), int(p)) for k, p in zip(qi, pos) if any(kfs[j]["ring_pos"] == p for j in ret if j > k)]
    assert overwritten, "no matched position is overwritten by a later push"
    assert int(got["ring_out"][0]["is_valid"].sum()) == 5
    assert n_of[ret[0]] == 0                                                           # the ring is empty below the first push
    t.close()


# ---- 3. split calls ------------------------------------------------------------------------------------------------------------------
def _split_call(t, capi, steps, kfs, ring0, cuts):
    """The steps in calls [cuts[c], cuts[c + 1]): world poses of earlier calls passed by value, every keyframe listed in the calls
    whose steps track against it and retired in the call that contains its retirement, the ring of call c passed to call c + 1."""
    n = len(steps)
    bounds = [0] + list(cuts) + [n]
    world = np.zeros((n, 6), np.float32)
    res = np.zeros(n, capi.RESULT_DTYPE)
    ring = ring0
    parts = dict(lc_pairs=[], lc_stats=[], lc_query_of_pair=[], lc_results=[])
    for c in range(len(bounds) - 1):
        a, b = bounds[c], bounds[c + 1]
        part = steps[a:b].copy()
        for f, v in (("prev_step", "prev_world"), ("kf_step", "kf_world")):
            early = (part[f] >= 0) & (part[f] < a)
            part[v][early] = world[part[f][early]]
            part[f] = np.where(early, -1, np.where(part[f] >= a, part[f] - a, part[f]))
        keep = []
        for k in range(len(kfs)):
            kf = kfs[k]
            used = any(a <= i < b for i in range(n) if steps[i]["kf_slot"] == kf["kf_slot"])
            retired_here = a < kf["retire_before"] <= b
            if used or retired_here:
                keep.append(k)
        sub = kfs[keep].copy()
        for j, k in enumerate(keep):
            ws = int(kfs[k]["world_step"])
            if 0 <= ws < a:
                sub[j]["world_step"] = -1
                sub[j]["world"] = world[ws]
            elif ws >= a:
                sub[j]["world_step"] = ws - a
            sub[j]["retire_before"] = kfs[k]["retire_before"] - a if a < kfs[k]["retire_before"] <= b else -1
        out = t.track_sequence_lc(part, sub, ring, min_match_difference=MMD, match_threshold=THR, max_rel_view_angle=ANG)
        res[a:b], world[a:b] = out["results"], out["world"]
        out["lc_query_of_pair"] = np.array([keep[j] for j in out["lc_query_of_pair"]], np.int32)
        for key in parts:
            parts[key].append(out[key])
        ring = out["ring_out"]
    got = {key: np.concatenate(v) for key, v in parts.items()}
    got.update(results=res, world=world, ring_out=ring)
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("cuts", [(10,), (10, 30)])
def test_split_calls_equal_one_call_and_continue_the_ring(capi, small, cuts):
    """The sequence of 48 frames in two or three calls (keyframe frame 8 spans the first cut: steps 8..11; the second cut lies in
    keyframe 28's span), the ring of each call handed to the next, world poses seeded by value: byte for byte the one call."""
    q = small["seqs"][0]
    t = _small_tracker(capi, small)
    steps = _seq_steps(capi, q)
    kfs = _seq_kfs(capi, q, 5, _mixed_queries(5))
    slots = [int(s) for s in kfs["kf_slot"]]
    ring0 = _empty_ring(capi, 1, 5)
    _reset(t, slots)
    one = t.track_sequence_lc(steps, kfs, ring0, min_match_difference=MMD, match_threshold=THR, max_rel_view_angle=ANG)
    w_one = _weights(t, slots)
    _reset(t, slots)
    split = _split_call(t, capi, steps, kfs, ring0, cuts)
    _assert_equal(split, one)
    assert _same_weights(_weights(t, slots), w_one)
    assert len(one["lc_pairs"]) > 0
    t.close()


# ---- 4. several sequences in one call ------------------------------------------------------------------------------------------------
def _topological_shuffle(steps, rng):
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
    return out, pos


@pytest.mark.gpu
def test_several_sequences_with_their_own_rings(capi, small):
    """Four ragged sequences, each with its own ring of 6 (different push offsets), steps shuffled across sequences (dependencies
    kept), keyframe entries interleaved round-robin (push order kept per ring): every sequence equals its own composition."""
    t = _small_tracker(capi, small)
    seqs = small["seqs"]
    per = []
    for s, q in enumerate(seqs):
        per.append((_seq_steps(capi, q), _seq_kfs(capi, q, 6, _mixed_queries(6, start=s), ring=s)))
    all_slots = [int(x) for _, kfs in per for x in kfs["kf_slot"]]
    want = []
    for s, (steps, kfs) in enumerate(per):
        k1 = kfs.copy()
        k1["ring"] = np.where(k1["retire_before"] >= 0, 0, k1["ring"])
        _reset(t, k1["kf_slot"])
        want.append((_composition(t, capi, steps, k1, _empty_ring(capi, 1, 6)), _weights(t, k1["kf_slot"])))
    # one call
    base = np.cumsum([0] + [len(st) for st, _ in per])
    allsteps = np.concatenate([st for st, _ in per])
    for s, (st, _) in enumerate(per):
        for f in ("prev_step", "kf_step"):
            allsteps[f][base[s]:base[s + 1]] = np.where(st[f] >= 0, st[f] + base[s], -1)
    shuffled, pos = _topological_shuffle(allsteps, np.random.default_rng(5))
    n = len(shuffled)
    entries, owner = [], []
    for j in range(max(len(k) for _, k in per)):
        for s, (_, kfs) in enumerate(per):
            if j < len(kfs):
                e = kfs[j].copy()
                e["world_step"] = pos[e["world_step"] + base[s]] if e["world_step"] >= 0 else -1
                e["retire_before"] = n if e["retire_before"] >= 0 else -1
                entries.append(e)
                owner.append((s, j))
    allkfs = np.array(entries, capi.LC_KEYFRAME_DTYPE)
    _reset(t, all_slots)
    got = t.track_sequence_lc(shuffled, allkfs, _empty_ring(capi, len(seqs), 6), min_match_difference=MMD, match_threshold=THR,
                              max_rel_view_angle=ANG)
    for s, (steps, kfs) in enumerate(per):
        w, w_weights = want[s]
        idx = pos[base[s]:base[s + 1]]
        assert _same(got["results"][idx], w["results"]) and _same(got["world"][idx], w["world"]), s
        assert _same(got["ring_out"][s], w["ring_out"][0]), s
        assert _same_weights(_weights(t, kfs["kf_slot"]), w_weights), s
        mine = [g for g, (o, _) in enumerate(owner) if o == s]
        sel = np.isin(got["lc_query_of_pair"], mine)
        for key in ("lc_pairs", "lc_stats", "lc_results"):
            assert _same(got[key][sel], w[key]), (s, key)
        assert [owner[g][1] for g in got["lc_query_of_pair"][sel]] == list(w["lc_query_of_pair"]), s
    assert len(got["lc_pairs"]) > 0
    t.close()


# ---- 5. validation -----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_invalid_inputs_launch_nothing_and_leave_the_weights(capi, small):
    q, other = small["seqs"][1], small["seqs"][0]
    t = _small_tracker(capi, small)
    steps = _seq_steps(capi, q)
    kfs = _seq_kfs(capi, q, 5, _mixed_queries(5))
    slots = [int(s) for s in kfs["kf_slot"]]
    ring0 = _empty_ring(capi, 1, 5)
    # a keyframe of another sequence: uploaded and with a histogram, but no finalised weights / loop-closure records
    stranger_kf, stranger_fr = other["kbase"], other["fbase"] + other["L"] + 1
    t.frame_histograms([stranger_fr])
    t.upload_keyframe_weights(slots[0], [np.full((small["height"] >> l, small["width"] >> l), 0.5, np.float32) for l in range(4)], [2, 2, 2, 2])
    before = _weights(t, slots)
    pairs = t.make_pairs([other["kbase"]] * 8, [other["fbase"] + 1 + i for i in range(8)],
                         np.random.default_rng(3).standard_normal((8, 6)).astype(np.float32) * 0.01)
    alone = t.track_batch(pairs)
    cases = []
    bad = steps.copy(); bad[2]["prev_step"] = 5
    cases.append(("forward dependency", bad, kfs, ring0, -1))
    k2 = kfs.copy(); k2[0]["retire_before"] = 2                                  # steps 2 .. 2 still track against keyframe 0
    cases.append(("step after its keyframe's retirement", steps, k2, ring0, -1))
    k3 = kfs.copy(); k3[1]["ring_pos"] = 5
    cases.append(("ring position", steps, k3, ring0, -1))
    k4 = kfs.copy(); k4[1]["match_window_end"] = -1
    cases.append(("window", steps, k4, ring0, -1))
    cases.append(("ring_len > 64", steps, kfs, _empty_ring(capi, 1, 65), -1))
    r5 = ring0.copy(); r5[0][4] = (500, 1, stranger_fr, stranger_kf, np.zeros(6, np.float32))
    cases.append(("loop keyframe without finalised weights", steps, kfs, r5, -3))
    t.reset_launch_count()
    dres = t.track_batch_async(pairs)
    launched = t.launch_count()
    for what, st, kf, ring, rc in cases:
        with pytest.raises(capi.EllcError, match=r"\(%d\)" % rc):
            t.track_sequence_lc(st, kf, ring)
        assert t.launch_count() == launched, what
    assert _same(t.results_download(dres, len(pairs)), alone)
    assert _same_weights(_weights(t, slots), before)
    t.close()


# ---- 6. launch count -----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_launch_count_per_call(capi, small):
    """3 x waves + 1 (the sequence call's) + 2 (frame lists, weights) + 5 per call with retired keyframes (loop-closure records,
    histograms, pushes, walk, pack) + 1 for the tracking of the pairs."""
    q = small["seqs"][0]
    t = _small_tracker(capi, small)
    t.prepare_frames([p["fbase"] + r for p in small["seqs"] for r in range(1, p["L"] + 1 + len(p["kff"]))])   # every uploaded slot: the
    t.prepare_keyframes(list(range(small["n_kf"])))                                                             # preparation is not the call's
    steps = _seq_steps(capi, q)
    kfs = _seq_kfs(capi, q, 5, _mixed_queries(5))
    waves = len(steps)
    _reset(t, kfs["kf_slot"])
    t.reset_launch_count()
    got = t.track_sequence_lc(steps, kfs, _empty_ring(capi, 1, 5))
    assert len(got["lc_pairs"]) > 0
    assert t.launch_count() == 3 * waves + 1 + 2 + 5 + 1, (t.launch_count(), waves)
    # no retired keyframe: only the weights of the listed ones
    _reset(t, kfs["kf_slot"])
    k0 = kfs.copy(); k0["retire_before"] = -1
    t.reset_launch_count()
    got = t.track_sequence_lc(steps, k0, _empty_ring(capi, 1, 5))
    assert len(got["lc_pairs"]) == 0 and t.launch_count() == 3 * waves + 1 + 2
    t.close()
