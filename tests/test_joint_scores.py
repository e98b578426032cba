"""Joint confidence scores (vnect_request_scores) and lost-person recovery of tracked streams (vnect_set_track_recovery).

The score of joint j of a frame is the float64 value utils.extract_2d_joints takes its argmax of (src/utils.py:153-175):
the x8 INTER_LINEAR upsample of the multi-scale float64 average hm_avg at its first maximum.  The reference below is
`extract_2d_scores` on oracle.prepost.average_scales; every GPU comparison is np.array_equal.

Chosen maps reach the branches of postprocess_kernel's step D that produce `best`:
* "blobs" (oracle.synth.synthetic_maps): a few surviving quads, evaluated on warp 0 (nq <= 32);
* "flat" (every cell equal) and "saturated" (a large constant plus a tiny ramp): more than 192 surviving quads, the
  full in-place scan; the flat map also ties every sample, so the first index wins;
* "plateau": a 2 x 2 block of equal maxima (tied candidates in four quads);
* "border": the peak on a corner and an edge cell (the border candidates d = 0 and d = 8(hs-1)+4);
* "near_flat": a quad whose corners agree to ~1e-12 relative, where an interior sample can beat the candidates.
Frames cycle through the kinds; the frame counts 5, 20 and 50 give the three block shapes (8, 4 and 2 rows per pass),
the configurations NS = 1..4, the compile-time identity mask (scale 1.0 first) and the run-time one (MASK = -1), and
box sizes 368, 448 and 512; postprocess_sequence reaches the RAW_ONLY instantiations.
"""
import cv2
import numpy as np
import pytest

from oracle import prepost, synth
from tests.golden.make_golden import POST_CASES, post_frame_maps
from vnect_b200 import _capi

HUGE = 1 << 30


# ------------------------------------------------------------------------------------------------ reference
def extract_2d_scores(hm_avg, hm_factor=8):
    """Each joint's score: the value of the float64 x8 upsample at the argmax extract_2d_joints reports."""
    out = np.zeros(hm_avg.shape[2])
    for j in range(hm_avg.shape[2]):
        up = cv2.resize(hm_avg[:, :, j], (0, 0), fx=hm_factor, fy=hm_factor, interpolation=cv2.INTER_LINEAR)
        out[j] = up.flat[np.argmax(up)]
    return out


def mean_score(scores):
    """What recovery compares with the threshold: Python's sum from joint 0 on (not np.mean, which sums pairwise)."""
    return sum(float(s) for s in scores) / len(scores)


class RecoveringTracker(prepost.OracleTracker):
    """OracleTracker with lost-person recovery: below a positive mean score the next box is the whole frame."""

    def __init__(self, estimator, rect, min_mean_score=0.0):
        super().__init__(estimator, rect)
        self.min_mean_score = float(min_mean_score)

    def __call__(self, frame):
        j2, j3, used = super().__call__(frame)
        self.scores = extract_2d_scores(self.estimator.last["hm_avg"], self.estimator.hm_factor)
        if self.min_mean_score > 0 and mean_score(self.scores) < self.min_mean_score:
            self.rect = (0, 0, HUGE, HUGE)
        return j2, j3, used


def oracle_scores(maps, scales, S):
    """(hm, xm, ym, zm) NHWC [n*ns, hs, hs, 21] -> float64 [n, 21] scores and the raw argmax [n, 21, 2]."""
    ns = len(scales)
    n = maps[0].shape[0] // ns
    sc, raw = [], []
    for f in range(n):
        hm = prepost.average_scales(tuple(m[f * ns:(f + 1) * ns] for m in maps), scales, S)[0]
        sc.append(extract_2d_scores(hm))
        raw.append(prepost.extract_2d_joints(hm, S))
    return np.array(sc), np.array(raw, np.int32)


# ------------------------------------------------------------------------------------------------ chosen maps
KINDS = ["blobs", "flat", "saturated", "plateau", "border", "near_flat"]


def chosen_frame(kind, seed, ns, hs):
    rng = np.random.default_rng(seed)
    hm, xm, ym, zm = synth.synthetic_maps(seed, ns, hs=hs)
    hm = hm.copy()
    if kind == "flat":
        hm[:] = np.float32(0.25)
    elif kind == "saturated":
        hm[:] = np.float32(3e4) + np.arange(hs, dtype=np.float32)[None, :, None, None] * np.float32(1e-3)
    elif kind == "plateau":
        hm *= np.float32(0.1)
        r, c = rng.integers(2, hs - 3, 2)
        hm[:, r:r + 2, c:c + 2, :] = np.float32(1.5)
    elif kind == "border":
        hm *= np.float32(0.1)
        hm[:, 0, 0, ::2] = np.float32(2.0)
        hm[:, hs - 1, rng.integers(0, hs), 1::2] = np.float32(2.0)
    elif kind == "near_flat":
        hm *= np.float32(0.1)
        r, c = rng.integers(2, hs - 3, 2)
        hm[:, r:r + 2, c:c + 2, :] = np.float32(1.0)
        hm[:, r + 1, c + 1, :] = np.nextafter(np.float32(1.0), np.float32(2.0))
    return hm, xm, ym, zm


def chosen_maps(n, ns, hs, seed):
    frames = [chosen_frame(KINDS[(seed + f) % len(KINDS)], seed * 1000 + f, ns, hs) for f in range(n)]
    return tuple(np.ascontiguousarray(np.concatenate([fr[m] for fr in frames]), np.float32) for m in range(4))


# (name, scales, box): NS 1..4, MASK 1 (scale 1.0 first) and -1 (run-time mask), boxes 368 / 448 / 512
CONFIGS = [("s1_368", [1.0], 368), ("s1_rt_448", [0.8], 448), ("s2_368", [1.0, 0.7], 368),
           ("s2_rt_448", [0.7, 1.0], 448), ("s3_512", [1.0, 0.85, 0.7], 512), ("s4_rt_368", [0.6, 0.7, 0.85, 1.0], 368)]


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("case", POST_CASES, ids=[c[0] for c in POST_CASES])
def test_score_is_the_upsample_maximum_on_post_fixture(case):
    name, seed, scales, nf, _ = case
    for k in range(nf):
        hm = prepost.average_scales(post_frame_maps(seed, k, scales), scales)[0]
        s = extract_2d_scores(hm)
        raw = prepost.extract_2d_joints(hm)
        for j in range(21):
            up = cv2.resize(hm[:, :, j], (0, 0), fx=8, fy=8, interpolation=cv2.INTER_LINEAR)
            assert s[j] == up.max() and s[j] == up[int(raw[j, 0]), int(raw[j, 1])]


def test_score_is_the_upsample_maximum_on_e2e_fixture():
    from oracle.forward import OracleNet
    from oracle.weights import make_weights
    net = OracleNet(make_weights("W0"))
    for scales, img in (([1.0, 0.7], synth.frame_c2(0)), ([1.0, 0.7], synth.stream_frame(0, 1))):
        batch, _, _ = prepost.gen_input_batch(img, 368, scales)
        hm = prepost.average_scales(net(batch), scales)[0]
        s = extract_2d_scores(hm)
        for j in range(21):
            up = cv2.resize(hm[:, :, j], (0, 0), fx=8, fy=8, interpolation=cv2.INTER_LINEAR)
            assert s[j] == up.max()


def test_mean_score_sums_left_to_right():
    """A row where Python's left-to-right sum and np.mean's pairwise sum fall on opposite sides of a threshold."""
    row = np.array([1e16, 1.0, -1e16] + [1.0] * 18)
    left = mean_score(row)
    pairwise = float(np.mean(row))
    assert left != pairwise
    tau = (left + pairwise) / 2
    assert (left < tau) != (pairwise < tau)


def test_capi_declares_the_new_entry_points():
    for name in ("vnect_request_scores", "vnect_set_track_recovery", "vnect_get_track_recovery"):
        assert name in _capi.SIGNATURES


def test_python_refuses_malformed_score_buffers():
    from vnect_b200.estimator import VNectEngine
    assert VNectEngine._scores_out(False, 3) is None
    assert VNectEngine._scores_out(True, 3).shape == (3, 21)
    for bad in (np.zeros((3, 21), np.float32), np.zeros((2, 21)), np.zeros((21, 3)).T, [[0.0] * 21] * 3):
        with pytest.raises(ValueError):
            VNectEngine._scores_out(bad, 3)


# ------------------------------------------------------------------------------------------------ GPU: chosen maps
def _engine(scales, S, n, streams=None, weights=False, **kw):
    from vnect_b200 import VNectEngine
    return VNectEngine(weights, scales, S, max_frames=n, max_streams=streams or n, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_scores_on_chosen_maps(cfg):
    name, scales, S = cfg
    ns, hs = len(scales), S // 8
    eng = _engine(scales, S, 50, max_input=(1080, 1920))
    t = 100.0
    try:
        for n in (5, 20, 50):  # the three block shapes
            maps = chosen_maps(n, ns, hs, n)
            want, want_raw = oracle_scores(maps, scales, S)
            t += 1
            j2, j3, raw, sc = eng.postprocess(maps, 1.0, (0, 0), np.arange(n), t, t + 0.004, scores=True)
            assert np.array_equal(sc, want), (name, n, np.argwhere(sc != want)[:5])
            assert np.array_equal(raw, want_raw)
            # the same call without a request: identical results, nothing else written
            eng.reset()
            j2b, j3b, rawb = eng.postprocess(maps, 1.0, (0, 0), np.arange(n), t, t + 0.004)
            assert np.array_equal(j2, j2b) and np.array_equal(j3, j3b) and np.array_equal(raw, rawb)
            eng.reset()
        # RAW_ONLY: a sequence call, one stream's 20 frames
        n = 20
        maps = chosen_maps(n, ns, hs, 7)
        want, _ = oracle_scores(maps, scales, S)
        ts = 200.0 + np.arange(n) / 30
        *_, sc = eng.postprocess_sequence(maps, 1.0, (0, 0), np.zeros(n, np.int32), ts, ts + 0.004, scores=True)
        assert np.array_equal(sc, want)
        # the tracked tail
        n = 12
        maps = chosen_maps(n, ns, hs, 11)
        want, _ = oracle_scores(maps, scales, S)
        hw = np.array([(540, 960)] * n, np.int32)
        *_, sc = eng.track_postprocess(maps, hw, np.arange(n), 300.0, 300.004, scores=True)
        assert np.array_equal(sc, want)
    finally:
        eng.close()


@pytest.mark.gpu
def test_asking_changes_nothing_else():
    """Twin engines on the same tracked maps, one asking for scores every step: everything else is identical."""
    scales, S, n = [1.0, 0.7], 368, 24
    a, b = _engine(scales, S, n), _engine(scales, S, n)
    try:
        hw = np.array([(540, 960), (720, 1280), (480, 640)] * 8, np.int32)
        for k in range(6):
            maps = chosen_maps(n, 2, 46, 40 + k)
            t = 500.0 + k / 30
            ra = a.track_postprocess(maps, hw, np.arange(n), t, t + 0.004, scores=True)
            rb = b.track_postprocess(maps, hw, np.arange(n), t, t + 0.004)
            for x, y in zip(ra[:3], rb):
                assert np.array_equal(x, y)
            assert np.array_equal(a.raw_argmax(n), b.raw_argmax(n))
            for sid in range(n):
                assert np.array_equal(a.export_stream_state(sid), b.export_stream_state(sid), equal_nan=True)
    finally:
        a.close()
        b.close()


# ------------------------------------------------------------------------------------------------ GPU: entry points
def _nv12(bgr):
    h, w = bgr.shape[:2]
    i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
    nv = i420.copy()
    u = i420[h:h + h // 4].reshape(-1)
    v = i420[h + h // 4:].reshape(-1)
    uv = nv[h:].reshape(-1)
    uv[0::2], uv[1::2] = u, v
    return nv


ENTRIES = ["estimate", "estimate_nv12", "submit", "estimate_frames", "submit_frames", "estimate_sequence",
           "submit_sequence", "track", "track_nv12", "track_frames", "submit_track", "submit_track_frames",
           "estimate_device", "estimate_device_nv12", "estimate_device_frames", "estimate_device_sequence",
           "track_device_frames"]


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ENTRIES)
def test_every_entry_point_reports_the_oracle_score(entry, w1):
    import torch
    scales, S, n = [1.0, 0.7], 368, 3
    eng = _engine(scales, S, n, weights=w1, max_input=(480, 640))
    frames = [synth.stream_frame(i, 0, 368) for i in range(n)]
    frames = [np.ascontiguousarray(cv2.resize(f, (480 - 40 * i, 360 + 20 * i))) for i, f in enumerate(frames)]
    uniform = np.stack([cv2.resize(f, (400, 320)) for f in frames])
    nv = "nv12" in entry
    dev = "device" in entry
    ids = np.arange(n, dtype=np.int32)
    graphs = []
    try:
        bufs = [np.full((n, 21), np.nan) for _ in range(4)] if not dev else \
            [torch.full((n, 21), float("nan"), dtype=torch.float64, device="cuda") for _ in range(4)]
        d_j2 = torch.empty((n, 21, 2), dtype=torch.float64, device="cuda")
        d_j3 = torch.empty((n, 21, 3), dtype=torch.float32, device="cuda")
        d_uni = torch.from_numpy(np.stack([_nv12(f) for f in uniform]) if nv else uniform).cuda()
        d_fr = [torch.from_numpy(f).cuda() for f in frames]
        for step in range(4):
            t2 = np.full(n, 1000.0 + step / 30)
            t3 = t2 + 0.004
            lane = step % 2
            buf = bufs[step]
            arg = buf if not dev else buf.data_ptr()
            if entry in ("estimate", "estimate_nv12"):
                eng.estimate(np.stack([_nv12(f) for f in uniform]) if nv else uniform, ids, t2, t3,
                             pixel_format="nv12" if nv else "bgr", scores=arg)
            elif entry == "submit":
                eng.submit(lane, uniform, ids, t2, t3, scores=arg)
                assert eng.wait(lane)[-1] is buf
            elif entry == "estimate_frames":
                eng.estimate_frames(frames, ids, t2, t3, scores=arg)
            elif entry == "submit_frames":
                eng.submit_frames(lane, frames, ids, t2, t3, scores=arg)
                eng.wait(lane)
            elif entry == "estimate_sequence":
                eng.estimate_sequence(frames, ids, t2, t3, scores=arg)
            elif entry == "submit_sequence":
                eng.submit_sequence(lane, frames, ids, t2, t3, scores=arg)
                eng.wait(lane)
            elif entry in ("track", "track_nv12"):
                eng.track(np.stack([_nv12(f) for f in uniform]) if nv else uniform, ids, t2, t3,
                          pixel_format="nv12" if nv else "bgr", scores=arg)
            elif entry == "track_frames":
                eng.track_frames(frames, ids, t2, t3, scores=arg)
            elif entry == "submit_track":
                eng.submit_track(lane, uniform, ids, t2, t3, scores=arg)
                eng.wait(lane)
            elif entry == "submit_track_frames":
                eng.submit_track_frames(lane, frames, ids, t2, t3, scores=arg)
                eng.wait(lane)
            elif entry in ("estimate_device", "estimate_device_nv12"):
                h, w = uniform.shape[1:3]
                eng.estimate_device(d_uni.data_ptr(), n, h, w, d_j2.data_ptr(), d_j3.data_ptr(), ids, t2, t3,
                                    pixel_format="nv12" if nv else "bgr", dev_scores_ptr=arg)
            else:
                descs = [dict(ptr=d.data_ptr(), h=f.shape[0], w=f.shape[1]) for d, f in zip(d_fr, frames)]
                fn = getattr(eng, entry)
                if entry == "track_device_frames":
                    fn(descs, d_j2.data_ptr(), d_j3.data_ptr(), None, ids, t2, t3, dev_scores_ptr=arg)
                else:
                    fn(descs, d_j2.data_ptr(), d_j3.data_ptr(), ids, t2, t3, dev_scores_ptr=arg)
            eng.synchronize()
            got = buf if not dev else buf.cpu().numpy()
            want, _ = oracle_scores(eng.maps(n), scales, S)
            assert np.array_equal(got, want), (entry, step)
            graphs.append(eng.info("cached_graphs"))
            if step > 0:  # the call after a request did not write to the previous call's buffer
                prev = bufs[step - 1] if not dev else bufs[step - 1].cpu().numpy()
                assert np.isnan(prev).all(), (entry, step)
            if not dev:
                buf[:] = np.nan
            else:
                buf.fill_(float("nan"))
        assert graphs[3] == graphs[2], graphs  # rotating buffers replay the same graphs
        # a refused call consumes the request and writes nothing; neither does the call after it
        bad = np.full(n, 10 ** 6, np.int32)
        buf = bufs[0]
        with pytest.raises(ValueError):
            if dev:
                eng.estimate_device_frames([dict(ptr=d.data_ptr(), h=f.shape[0], w=f.shape[1])
                                            for d, f in zip(d_fr, frames)], d_j2.data_ptr(), d_j3.data_ptr(), bad,
                                           dev_scores_ptr=buf.data_ptr())
            else:
                eng.estimate_frames(frames, bad, scores=buf)
        eng.estimate_frames(frames, ids, 2000.0, 2000.004)
        eng.synchronize()
        assert np.isnan(buf if not dev else buf.cpu().numpy()).all()
    finally:
        eng.close()


@pytest.mark.gpu
def test_untouched_path_launches_and_graphs(w1):
    """No request and no recovery: a call makes the launches it made before asking, and asking adds one graph key."""
    eng = _engine([1.0, 0.7], 368, 2, weights=w1)
    frames = np.stack([synth.frame_c2(i) for i in range(2)])
    try:
        counts, t = [], 100.0

        def call(**kw):
            nonlocal t
            t += 1
            before = eng.launch_count()
            eng.estimate(frames, [0, 1], t, t + 0.004, **kw)
            counts.append(eng.launch_count() - before)

        for _ in range(3):
            call()
        g0 = eng.info("cached_graphs")
        for _ in range(3):
            call(scores=True)
        g1 = eng.info("cached_graphs")
        for _ in range(3):
            call()
        assert g1 == g0 + 1 and eng.info("cached_graphs") == g1
        assert len(set(counts[1:])) == 1, counts  # the first call also lays the shrunken scales' constant surround
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------------ GPU: recovery
STEPS = 24


def recovery_streams():
    """(frame (h, w), seeded box, threshold, lost steps): frames whose maps are weak (mean score below the threshold)
    at the listed own steps."""
    return [
        ((540, 960), (300, 100, 360, 380), 0.5, {3, 4, 11}),
        ((720, 1280), (500, 200, 300, 500), 0.5, {0, 7}),
        ((481, 641), (100, 50, 400, 300), 1.2, {5, 6, 7, 15}),
        ((333, 517), (30, 18, 217, 153), 0.5, set()),
        ((540, 960), (200, 100, 300, 300), 0.0, {2, 9}),     # no threshold: weak maps change nothing
        ((360, 640), None, 0.7, {1, 13}),
        ((700, 500), (480, 0, 20, 400), 0.5, {4}),
        ((480, 640), (200, 100, 300, 300), 0.0, set()),
    ]


def recovery_maps(sid, k, lost, S):
    hs = S // 8
    rng = np.random.default_rng([77, sid, k])
    hm = (0.2 * rng.random((2, hs, hs, 21))).astype(np.float32)
    cells = np.stack([rng.integers(hs // 8, 7 * hs // 8, 21), rng.integers(hs // 4, 3 * hs // 4, 21)], axis=1)
    hm[0, cells[:, 0], cells[:, 1], np.arange(21)] = np.float32(2.0) + rng.uniform(0, 0.5, 21).astype(np.float32)
    if k in lost:
        hm *= np.float32(0.1)
    loc = [rng.uniform(-5, 5, (2, hs, hs, 21)).astype(np.float32) for _ in range(3)]
    return (hm, *loc)


class _Clock:
    def __init__(self):
        self.q = []

    def __call__(self):
        return self.q.pop(0)


@pytest.mark.gpu
def test_recovery_matches_the_reference_step_for_step():
    scales, S = [1.0, 0.7], 368
    streams = recovery_streams()
    n = len(streams)
    eng = _engine(scales, S, n)
    plain = _engine(scales, S, n)  # no stream has a threshold
    try:
        ids = np.arange(n, dtype=np.int32)
        eng.set_track_recovery(ids, [s[2] for s in streams])
        assert [eng.track_recovery(i) for i in range(n)] == [s[2] for s in streams]
        refs = []
        for sid, (hw, seed, tau, lost) in enumerate(streams):
            clock = _Clock()
            est = prepost.OracleEstimator(None, scales, clock=clock, promotion="legacy", box_size=S)
            refs.append((RecoveringTracker(est, seed or (0, 0, HUGE, HUGE), tau), clock))
            for e in (eng, plain):
                if seed:
                    e.set_box(sid, seed)
        hw = np.array([s[0] for s in streams], np.int32)
        recovered = 0
        for k in range(STEPS):
            maps_f = [recovery_maps(sid, k, s[3], S) for sid, s in enumerate(streams)]
            maps = tuple(np.concatenate([m[i] for m in maps_f]) for i in range(4))
            t2 = 800.0 + k / 30 + np.arange(n) * 1e-3
            t3 = t2 + 0.004
            j2, j3, used, sc = eng.track_postprocess(maps, hw, ids, t2, t3, scores=True)
            pj2, pj3, pused = plain.track_postprocess(maps, hw, ids, t2, t3)
            for sid, (tr, clock) in enumerate(refs):
                tr.estimator.forward = lambda batch, m=maps_f[sid]: m
                clock.q = [float(t2[sid]), float(t3[sid])]
                rj2, rj3, rused = tr(np.zeros((*streams[sid][0], 3), np.uint8))
                assert np.array_equal(j2[sid], rj2) and np.array_equal(j3[sid], rj3), (k, sid)
                assert tuple(used[sid]) == tuple(rused), (k, sid)
                assert np.array_equal(sc[sid], tr.scores)
                assert eng.get_box(sid) == tuple(tr.rect), (k, sid)
                recovered += tr.rect == (0, 0, HUGE, HUGE) and streams[sid][2] > 0
                if streams[sid][2] == 0:  # streams without a threshold: as on an engine where none has one
                    assert np.array_equal(j2[sid], pj2[sid]) and np.array_equal(used[sid], pused[sid])
                    assert np.array_equal(eng.export_stream_state(sid), plain.export_stream_state(sid),
                                          equal_nan=True)
            if k == 10:  # set_boxes after a recovery wins
                eng.set_boxes([0], [(10, 20, 300, 200)])
                refs[0][0].rect = (10, 20, 300, 200)
        assert recovered >= 8
        # refusals leave the configuration unchanged
        before = [eng.track_recovery(i) for i in range(n)]
        for sids, taus in (([0, 0], [1.0, 1.0]), ([n], [1.0]), ([-1], [1.0]), ([1], [-0.5]), ([1], [np.nan]),
                           ([1], [np.inf])):
            with pytest.raises(ValueError):
                eng.set_track_recovery(sids, taus)
        lib = _capi.load_library()
        assert lib.vnect_set_track_recovery(eng._h, -1, None, None) == _capi.E_INVALID
        assert lib.vnect_set_track_recovery(eng._h, 1, None, None) == _capi.E_INVALID
        assert [eng.track_recovery(i) for i in range(n)] == before
        eng.reset()  # reset keeps the thresholds
        assert [eng.track_recovery(i) for i in range(n)] == before
    finally:
        eng.close()
        plain.close()


@pytest.mark.gpu
def test_recovery_on_cnn_entry_points(w1):
    """Oriented and mixed-size tracked streams with recovery on the CNN: submit_track_frames on alternating lanes and
    track_device_frames give what the synchronous track_frames gives; a threshold changed while calls are in flight
    applies only to later submissions; an oriented stream gives what an identity stream gives on the materialised
    frame; uniform track() builds its table and matches track_frames."""
    import torch
    scales, S = [1.0, 0.7], 368
    sizes = [(480, 640), (360, 480), (480, 360), (400, 400)]
    n = len(sizes)
    base = [cv2.resize(synth.stream_frame(i, 0, 368), (w, h)) for i, (h, w) in enumerate(sizes)]
    orient = [0, 1, 0, 2]  # rot90_cw on stream 1 (sides swap), rot180 on stream 3
    stored = [np.ascontiguousarray(np.rot90(f, 1)) if o == 1 else np.ascontiguousarray(f[::-1, ::-1])
              if o == 2 else f for f, o in zip(base, orient)]
    engs = [_engine(scales, S, n, weights=w1, max_input=(640, 640)) for _ in range(4)]
    try:
        ids = np.arange(n, dtype=np.int32)
        for e in engs[:3]:
            e.set_orientations(ids, orient)
        steps = 6
        taus = [[1e9 if (k % 3 == 1 and s % 2 == 0) else 0.0 for s in range(n)] for k in range(steps)]
        res = {i: [] for i in range(4)}
        d_fr = [torch.from_numpy(f).cuda() for f in stored]
        descs = [dict(ptr=d.data_ptr(), h=f.shape[0], w=f.shape[1]) for d, f in zip(d_fr, stored)]
        d_j2 = torch.empty((n, 21, 2), dtype=torch.float64, device="cuda")
        d_j3 = torch.empty((n, 21, 3), dtype=torch.float32, device="cuda")
        d_b = torch.empty((n, 4), dtype=torch.int32, device="cuda")
        pending = {}
        for k in range(steps):
            t2 = np.full(n, 50.0 + k / 30)
            t3 = t2 + 0.004
            for e in engs:
                e.set_track_recovery(ids, taus[k])
            res[0].append(engs[0].track_frames(stored, ids, t2, t3, scores=True))
            lane = k % 2
            if lane in pending:
                res[1].append(engs[1].wait(lane))
            pending[lane] = engs[1].submit_track_frames(lane, stored, ids, t2, t3, scores=True)
            engs[1].set_track_recovery(ids, np.full(n, 1e9))  # in flight: must not reach the call above
            engs[2].track_device_frames(descs, d_j2.data_ptr(), d_j3.data_ptr(), d_b.data_ptr(), ids, t2, t3)
            engs[2].synchronize()  # the results are written on the engine's own stream
            res[2].append((d_j2.cpu().numpy(), d_j3.cpu().numpy(), d_b.cpu().numpy()))
            res[3].append(engs[3].track_frames(base, ids, t2, t3))  # identity streams on the oriented frames
        for lane in ((steps - 2) % 2, (steps - 1) % 2):
            res[1].append(engs[1].wait(lane))
        for k in range(steps):
            for i in (1, 2, 3):
                for a, b in zip(res[0][k][:3], res[i][k][:3]):
                    assert np.array_equal(a, b), (k, i)
        lost_steps = [k for k in range(steps) if any(taus[k])]
        assert lost_steps
        for k in lost_steps:  # the step after a lost frame crops the whole (oriented) frame
            if k + 1 < steps:
                for s in range(n):
                    if taus[k][s] > 0:
                        h, w = base[s].shape[:2]
                        assert tuple(res[0][k + 1][2][s]) == (0, 0, w, h), (k, s)
        # uniform track() with recovery runs the table path and matches track_frames on the same frames
        u = [_engine(scales, S, 2, weights=w1, max_input=(640, 640)) for _ in range(2)]
        try:
            fr = np.stack([base[0], cv2.resize(base[1], (640, 480))])
            for e in u:
                e.set_track_recovery([0, 1], [1e9, 0.0])
            for k in range(3):
                a = u[0].track(fr, [0, 1], 90.0 + k, 90.004 + k, scores=True)
                b = u[1].track_frames(list(fr), [0, 1], 90.0 + k, 90.004 + k, scores=True)
                for x, y in zip(a, b):
                    assert np.array_equal(x, y)
        finally:
            for e in u:
                e.close()
    finally:
        for e in engs:
            e.close()
