"""Sequence calls: consecutive frames of one stream in one batch (vnect_submit_sequence, vnect_estimate_device_sequence,
vnect_postprocess_sequence).  Frame i of a sequence call must give bit for bit what the untracked entry points give
when the frames go in one at a time in call order: joints, raw argmax, packed results, and afterwards every stream's
exported state.

* Chosen maps, no CNN: postprocess_sequence against oracle.prepost.OracleEstimator stepped per frame with injected
  clocks, and against a second engine fed one frame per postprocess call.  The peaks jump (cutoff moves), sit in the
  first and last heat-map cells (filtered points below 3.5 extrapolate, points at or above 8(hs-1)+3.5 give exactly 0),
  the root joint moves, clocks are epoch-like or small, a few readings are 0, a stream is fresh or just reset.
* On the CNN (W1): submit_sequence in BGR / NV12 / I420 on both lanes and estimate_device_sequence, against a second
  engine fed one time step per estimate_frames call and against the oracle on the sequence call's own maps.
* Refusals leave every stream exactly as if the refused call had not been made.
"""
import cv2
import numpy as np
import pytest

from oracle import prepost


class _Clock:
    def __init__(self):
        self.q = []

    def __call__(self):
        return self.q.pop(0)


def seq_maps(scales, box, sid, k):
    """(hm, xm, ym, zm) of frame k of stream sid, each [NS, hs, hs, 21] float32: one peak per joint in the identity
    scale over a weak background.  Joints 0-3 sit in corner cells (first / last row and column), joint 14 (the root)
    moves one cell per frame, the others jump to a new random cell every third frame."""
    hs, ns = box // 8, len(scales)
    rng = np.random.default_rng([sid, k, box, ns])
    base = np.random.default_rng([sid, k // 3, box]).integers(0, hs, (21, 2))
    base[0] = (0, 0)
    base[1] = (hs - 1, hs - 1)
    base[2] = (0, hs - 1)
    base[3] = (hs - 1, (k * 7) % hs)
    base[14] = ((5 + k) % hs, (11 + 2 * k) % hs)
    hm = (0.2 * rng.random((ns, hs, hs, 21))).astype(np.float32)
    ident = [i for i, s in enumerate(scales) if s == 1.0][0]
    hm[ident, base[:, 0], base[:, 1], np.arange(21)] = np.float32(2.0) + rng.uniform(0, 0.5, 21).astype(np.float32)
    loc = []
    nc = -(-hs // 8)
    for _ in range(3):
        coarse = rng.uniform(-5, 5, size=(ns, nc, nc, 21))
        fine = np.kron(coarse, np.ones((1, 8, 8, 1)))[:, :hs, :hs, :]
        loc.append((fine + 0.05 * rng.standard_normal(fine.shape)).astype(np.float32))
    return (hm, *loc)


def stream_clock(sid, k):
    """(t2d, t3d) of frame k of stream sid: epoch-like 1/30 s steps for even ids, irregular small ones for odd ids,
    and a 0 reading at frame 5 of streams 1 and 4."""
    if sid in (1, 4) and k == 5:
        return 0.0, 0.0
    if sid % 2 == 0:
        t = 1.7e9 + sid + k / 30.0
    else:
        t = 500.0 + sid + float(np.cumsum(np.random.default_rng(sid).uniform(0.015, 0.09, k + 1))[-1])
    return t, t + 0.002


CONFIGS = [("368_1_0.7", [1.0, 0.7], 368), ("448_0.7_1", [0.7, 1.0], 448), ("368_1", [1.0], 368),
           ("368_ref", [1.0, 0.85, 0.7], 368)]


def compositions(name, call):
    """Stream id of every frame of call `call` (frames of one stream in time order)."""
    rng = np.random.default_rng([sum(map(ord, name)), call])
    if name == "one":
        return [3] * 64
    if name == "interleaved":
        ids = np.repeat(np.arange(8), 8)
        return [int(i) for i in rng.permutation(ids)]
    if name == "ragged":
        counts = {0: 20, 1: 1, 4: 13, 5: 7, 6: 3, 9 + call: 20}  # stream 9 + call: fresh in every call
        ids = np.concatenate([[s] * c for s, c in counts.items()])
        return [int(i) for i in rng.permutation(ids)]
    return [int(i) for i in rng.permutation(64)]  # "distinct"


class _Streams:
    """Per-stream frame counters, oracles and clocks of the reference side."""

    def __init__(self, scales, box):
        self.scales, self.box = scales, box
        self.k, self.refs, self.clocks = {}, {}, {}

    def reset(self, sid):
        self.k[sid] = 0
        self.clocks[sid] = _Clock()
        self.refs[sid] = prepost.OracleEstimator(None, self.scales, clock=self.clocks[sid], promotion="legacy",
                                                 box_size=self.box)

    def next(self, sid):
        if sid not in self.k:
            self.reset(sid)
        k = self.k[sid]
        self.k[sid] += 1
        return k

    def step(self, sid, maps, t2, t3, scaler, offsets):
        ref = self.refs[sid]
        ref.forward = lambda b, m=maps: m
        self.clocks[sid].q = [t2, t3]
        _, r3 = ref(np.zeros((self.box, self.box, 3), np.uint8))
        r2 = ref.last["joints_2d_box"].copy()
        r2[:, 0] = (r2[:, 0] - offsets[1]) / scaler
        r2[:, 1] = (r2[:, 1] - offsets[0]) / scaler
        return r2, r3, ref.last["joints_2d_raw"].astype(np.int32)


def _batch(per_frame):
    return tuple(np.concatenate([m[c] for m in per_frame]) for c in range(4))


# ------------------------------------------------------------------------------------------------ chosen maps
@pytest.mark.gpu
@pytest.mark.parametrize("comp", ["one", "interleaved", "ragged", "distinct"])
@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_postprocess_sequence_bit_exact(cfg, comp):
    from vnect_b200 import VNectEngine
    _, scales, box = cfg
    scaler, offsets = 0.6133, (7, 41)
    seq = VNectEngine(False, scales, box_size=box, max_frames=64, max_streams=80)
    one = VNectEngine(False, scales, box_size=box, max_frames=64, max_streams=80)
    streams = _Streams(scales, box)
    try:
        for call in range(3):
            if call == 2:  # a stream after reset, on both engines and the reference
                for e in (seq, one):
                    e.reset(4)
                streams.reset(4)
            ids = compositions(comp, call)
            frames = [(sid, streams.next(sid)) for sid in ids]
            per = [seq_maps(scales, box, sid, k) for sid, k in frames]
            t = np.array([stream_clock(sid, k) for sid, k in frames])
            j2, j3, raw = seq.postprocess_sequence(_batch(per), scaler, offsets, ids, t[:, 0], t[:, 1])
            if comp == "distinct":  # one ordinary call on the same input
                o2, o3, oraw = one.postprocess(_batch(per), scaler, offsets, ids, t[:, 0], t[:, 1])
                assert np.array_equal(j2, o2) and np.array_equal(j3, o3) and np.array_equal(raw, oraw), call
            for i, (sid, k) in enumerate(frames):
                if comp != "distinct":
                    o2, o3, oraw = one.postprocess(per[i], scaler, offsets, [sid], t[i, 0], t[i, 1])
                    assert np.array_equal(j2[i], o2[0]) and np.array_equal(j3[i], o3[0]), (call, i)
                    assert np.array_equal(raw[i], oraw[0]), (call, i)
                r2, r3, rraw = streams.step(sid, per[i], float(t[i, 0]), float(t[i, 1]), scaler, offsets)
                assert np.array_equal(raw[i], rraw), (call, i, sid, k)
                assert np.array_equal(j2[i], r2), (call, i, sid, k)
                assert np.array_equal(j3[i], r3), (call, i, sid, k)
            for sid in set(ids):
                assert np.array_equal(seq.export_stream_state(sid), one.export_stream_state(sid), equal_nan=True), sid
    finally:
        seq.close()
        one.close()


@pytest.mark.gpu
def test_stream_alternates_between_ordinary_and_sequence_calls():
    from vnect_b200 import VNectEngine
    scales, box = [1.0, 0.7], 368
    eng = VNectEngine(False, scales, box_size=box, max_frames=16, max_streams=8)
    streams = _Streams(scales, box)
    try:
        for call in range(6):
            n = 1 if call % 2 else 5
            frames = [(2, streams.next(2)) for _ in range(n)]
            per = [seq_maps(scales, box, s, k) for s, k in frames]
            t = np.array([stream_clock(s, k) for s, k in frames])
            fn = eng.postprocess if n == 1 else eng.postprocess_sequence
            j2, j3, raw = fn(_batch(per), 1.0, (0, 0), [2] * n, t[:, 0], t[:, 1])
            for i, (s, k) in enumerate(frames):
                r2, r3, rraw = streams.step(s, per[i], float(t[i, 0]), float(t[i, 1]), 1.0, (0, 0))
                assert np.array_equal(j2[i], r2) and np.array_equal(j3[i], r3) and np.array_equal(raw[i], rraw)
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------------ refusals
@pytest.mark.gpu
@pytest.mark.parametrize("bad", ["repeat_in_call", "repeat_vs_previous", "earlier", "id_range", "too_many"])
def test_refused_sequence_call_changes_nothing(bad):
    from vnect_b200 import VNectEngine
    scales, box = [1.0, 0.7], 368
    engs = [VNectEngine(False, scales, box_size=box, max_frames=8, max_streams=4) for _ in range(2)]
    maps = lambda sid, ks: _batch([seq_maps(scales, box, sid, k) for k in ks])
    try:
        for e in engs:
            e.postprocess_sequence(maps(1, [0, 1, 2]), 1.0, (0, 0), [1, 1, 1], [10.0, 10.1, 10.2], [10.0, 10.1, 10.2])
        ids, t2 = [1, 1], [10.3, 10.4]
        err = ZeroDivisionError if bad.startswith("repeat") else ValueError
        if bad == "repeat_in_call":
            t2 = [10.3, 10.3]
        elif bad == "repeat_vs_previous":
            t2 = [10.2, 10.4]
        elif bad == "earlier":
            t2 = [10.3, 10.25]
        elif bad == "id_range":
            ids = [1, 4]
        n = 9 if bad == "too_many" else 2
        with pytest.raises(err):
            engs[0].postprocess_sequence(maps(1, range(3, 3 + n)), 1.0, (0, 0), (ids * 5)[:n], (t2 * 5)[:n],
                                         (t2 * 5)[:n])
        for sid in range(4):
            assert np.array_equal(engs[0].export_stream_state(sid), engs[1].export_stream_state(sid), equal_nan=True)
        got = [e.postprocess_sequence(maps(1, [3, 4]), 1.0, (0, 0), [1, 1], [10.5, 10.6], [10.5, 10.6]) for e in engs]
        for a, b in zip(*got):
            assert np.array_equal(a, b)
    finally:
        for e in engs:
            e.close()


@pytest.mark.gpu
def test_sequence_call_reports_non_finite_maps(w0):
    from oracle import synth
    from vnect_b200 import VNectEngine
    huge = dict(w0)
    huge["conv1/weights"] = w0["conv1/weights"] * np.float32(1e6)
    eng = VNectEngine(huge, [1.0], max_frames=4, max_streams=1)
    try:
        frames = [synth.frame_c2(3)] * 3
        eng.submit_sequence(0, frames, [0, 0, 0], [1.0, 1.1, 1.2], [1.0, 1.1, 1.2])
        with pytest.raises(FloatingPointError, match="non-finite"):
            eng.wait(0)
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------------ on the CNN
def moving_frames(n_steps, sizes, seed):
    """C4-style frames: seeded noise shifted k px per step, per stream its own size."""
    out = []
    for i, (h, w) in enumerate(sizes):
        rng = np.random.default_rng([seed, i])
        big = cv2.GaussianBlur(rng.integers(0, 256, (h + 64, w + 2 * n_steps + 8, 3), dtype=np.uint8), (7, 7), 0)
        out.append([np.ascontiguousarray(big[(3 * k) % 64:(3 * k) % 64 + h, 2 * k:2 * k + w]) for k in range(n_steps)])
    return out


def _to_yuv(f, fmt):
    f = f[:f.shape[0] & ~1, :f.shape[1] & ~1]
    yuv = cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420)
    if fmt == "i420":
        return yuv, cv2.cvtColor(yuv, cv2.COLOR_YUV2BGR_I420)
    h, w = f.shape[:2]
    q = (h // 2) * (w // 2)
    nv12 = yuv.copy()
    nv12[h:] = np.stack([yuv[h:].reshape(-1)[:q], yuv[h:].reshape(-1)[q:]], axis=1).reshape(h // 2, w)
    return nv12, cv2.cvtColor(nv12, cv2.COLOR_YUV2BGR_NV12)


CNN_INPUTS = ["moving_540x960", "moving_mixed", "golden_video"]
CNN_ENTRIES = ["submit_bgr", "submit_nv12", "submit_i420", "device"]


def interleave(n_streams, k0, k1, seed):
    """(stream, step) of steps k0..k1-1 of every stream in a random interleaving, each stream in time order."""
    order = np.random.default_rng(seed).permutation(np.repeat(np.arange(n_streams), k1 - k0))
    nxt = {s: k0 for s in range(n_streams)}
    out = []
    for s in order:
        out.append((int(s), nxt[int(s)]))
        nxt[int(s)] += 1
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("entry", CNN_ENTRIES)
@pytest.mark.parametrize("inputs", CNN_INPUTS)
def test_sequence_calls_on_cnn_maps(inputs, entry, w1, golden):
    import torch
    from vnect_b200 import VNectEngine
    scales, S, steps, n_streams = [1.0, 0.7], 368, 28, 4
    if inputs == "golden_video":
        video = golden("video.npz")["frames"]
        clips = [[np.ascontiguousarray(video[(k + 3 * i) % len(video)]) for k in range(steps)] for i in range(n_streams)]
    else:
        sizes = [(540, 960)] * 4 if inputs == "moving_540x960" else [(540, 960), (301, 517), (480, 640), (256, 256)]
        clips = moving_frames(steps, sizes, 11)
    fmt = {"submit_nv12": "nv12", "submit_i420": "i420"}.get(entry, "bgr")
    given = clips
    if fmt != "bgr":  # the engines take the YUV frames, the oracle the frames cv2 decodes from them
        pairs = [[_to_yuv(f, fmt) for f in clip] for clip in clips]
        given = [[p[0] for p in clip] for clip in pairs]
        clips = [[p[1] for p in clip] for clip in pairs]
    sids = [7, 2, 11, 5]
    rng = np.random.default_rng(5)
    t2 = 1.76e9 + np.cumsum(rng.uniform(0.02, 0.05, (steps, n_streams)), axis=0)
    t3 = t2 + rng.uniform(0.001, 0.004, t2.shape)
    seq = VNectEngine(w1, scales, max_frames=64, max_streams=16, max_input=(540, 960))
    ref = VNectEngine(w1, scales, max_frames=64, max_streams=16, max_input=(540, 960))
    packed = torch.zeros((64, 21, 5), dtype=torch.float64, device="cuda")
    dev_j2 = torch.empty((64, 21, 2), dtype=torch.float64, device="cuda")
    dev_j3 = torch.empty((64, 21, 3), dtype=torch.float32, device="cuda")
    oracle = _Streams(scales, S)
    try:
        # reference 1: one time step per estimate_frames call, distinct ids; its maps, raw argmax and states kept
        want = {}
        states = {}
        for k in range(steps):
            o2, o3 = ref.estimate_frames([given[s][k] for s in range(n_streams)], sids, t2[k], t3[k], pixel_format=fmt)
            maps, raw = ref.maps(n_streams), ref.raw_argmax(n_streams)
            for s in range(n_streams):
                want[s, k] = (o2[s].copy(), o3[s].copy(), raw[s].copy(), tuple(m[2 * s:2 * s + 2] for m in maps))
            if k in (7, 15, 23, 27):
                states[k] = [ref.export_stream_state(sid) for sid in sids]
        seq.set_packed_results(packed.data_ptr())
        # three calls of 32 frames with different compositions (time-major, stream-major, random), then one call split
        # over the two lanes with lane 1 submitted first
        calls = [[(s, k) for k in range(0, 8) for s in range(n_streams)],
                 [(s, k) for s in range(n_streams) for k in range(8, 16)],
                 interleave(n_streams, 16, 24, 3),
                 interleave(n_streams, 24, 28, 4)]
        launches, keys = [], set()
        for c, call in enumerate(calls):
            n = len(call)
            ids = [sids[s] for s, _ in call]
            ct2 = np.array([t2[k, s] for s, k in call])
            ct3 = np.array([t3[k, s] for s, k in call])
            frames = [given[s][k] for s, k in call]
            before = seq.launch_count()
            own = np.ones(n, bool)  # frames whose maps / raw argmax the engine still holds afterwards
            if entry == "device":
                dev = [torch.from_numpy(f).cuda() for f in frames]
                torch.cuda.synchronize()
                seq.estimate_device_sequence([dict(ptr=d.data_ptr(), h=d.shape[0], w=d.shape[1]) for d in dev],
                                             dev_j2.data_ptr(), dev_j3.data_ptr(), ids, ct2, ct3)
                seq.synchronize()
                j2, j3 = dev_j2[:n].cpu().numpy(), dev_j3[:n].cpu().numpy()
                keys.add((c & 1, n))
            elif c < 3:
                j2, j3 = seq.estimate_sequence(frames, ids, ct2, ct3, pixel_format=fmt)
                keys.add((0, n))
            else:
                early = np.array([k < 26 for _, k in call])
                a, b = np.nonzero(early)[0], np.nonzero(~early)[0]
                seq.submit_sequence(1, [frames[i] for i in a], [ids[i] for i in a], ct2[a], ct3[a], pixel_format=fmt)
                seq.submit_sequence(0, [frames[i] for i in b], [ids[i] for i in b], ct2[b], ct3[b], pixel_format=fmt)
                b2, b3 = seq.wait(0)
                a2, a3 = seq.wait(1)
                j2, j3 = np.empty((n, 21, 2)), np.empty((n, 21, 3), np.float32)
                j2[a], j3[a], j2[b], j3[b] = a2, a3, b2, b3
                keys.update({(1, len(a)), (0, len(b))})
                own = ~early
                call = [call[i] for i in np.concatenate([a, b])]  # the lane-0 frames are the engine's last call
                j2, j3 = np.concatenate([j2[a], j2[b]]), np.concatenate([j3[a], j3[b]])
                own = np.concatenate([own[a], own[b]])
            launches.append(seq.launch_count() - before)
            m_own = own.sum()
            maps = seq.maps(int(m_own)) if c < 3 or entry == "device" else seq.maps(len(b))
            raw = seq.raw_argmax(int(maps[0].shape[0] // 2))
            if c < 3 or entry == "device":
                pk = packed[:n].cpu().numpy()
                assert np.array_equal(pk[..., :2], j2) and np.array_equal(pk[..., 2:], j3.astype(np.float64)), c
            base = n - int(m_own)
            for i, (s, k) in enumerate(call):
                w2, w3, wraw, wmaps = want[s, k]
                tag = (c, i, s, k)
                assert np.array_equal(j2[i], w2) and np.array_equal(j3[i], w3), tag
                m_i = wmaps
                if own[i]:
                    r = i - base
                    assert np.array_equal(raw[r], wraw), tag
                    m_i = tuple(m[2 * r:2 * r + 2] for m in maps)
                # reference 2: the oracle stepped per stream on the sequence call's own maps
                oracle.next(sids[s])
                est = oracle.refs[sids[s]]
                est.forward = lambda b_, m=m_i: m
                oracle.clocks[sids[s]].q = [float(t2[k, s]), float(t3[k, s])]
                r2, r3 = est(clips[s][k])
                assert np.array_equal(est.last["joints_2d_raw"].astype(np.int32), wraw), tag
                assert np.array_equal(j2[i], r2) and np.array_equal(j3[i], r3), tag
            last_k = max(k for _, k in call)
            for sid, st in zip(sids, states[last_k]):
                assert np.array_equal(seq.export_stream_state(sid), st, equal_nan=True), (c, sid)
        # the third call replays the graph the second captured; one cached entry per (lane, n_frames, format)
        assert launches[1] == launches[2], launches
        assert seq.info("cached_graphs") == len(keys), (seq.info("cached_graphs"), keys)
    finally:
        seq.close()
        ref.close()


@pytest.mark.gpu
def test_sequence_without_filters_equals_per_frame_calls(w1):
    from vnect_b200 import VNectEngine
    scales = [1.0, 0.7]
    clips = moving_frames(6, [(540, 960), (480, 640)], 3)
    engs = [VNectEngine(w1, scales, max_frames=16, max_streams=4, max_input=(540, 960), filters=False)
            for _ in range(2)]
    try:
        frames = [clips[s][k] for k in range(6) for s in range(2)]
        ids = [0, 1] * 6
        j2, j3 = engs[0].estimate_sequence(frames, ids)
        for i, f in enumerate(frames):
            o2, o3 = engs[1].estimate_frames([f], [ids[i]])
            assert np.array_equal(j2[i], o2[0]) and np.array_equal(j3[i], o3[0]), i
    finally:
        for e in engs:
            e.close()
