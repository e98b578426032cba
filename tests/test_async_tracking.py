"""Pipelined and device-resident tracking (vnect_submit_track_frames, vnect_track_device_frames,
vnect_track_set_boxes).  Frame i of an asynchronous tracked call must give bit for bit what the synchronous
vnect_track_frames / vnect_track gives for the same submission order: joints, boxes_used, raw argmax, the box left
behind and the filter state.

CPU: the tables submit_track / track_device build, and the ctypes prototypes.  GPU: every asynchronous path against
the synchronous one on the same engine, on disjoint stream ids (+ REF) with identical timestamps, compared with
np.array_equal.  The frames are the real video of tests/golden/video.npz, shifted, padded or cropped per stream, so
the tracked boxes actually move.  The ordering tests park the engine's stream behind a spin kernel (hold()) and use
pinned frames and results, so the calls under test are enqueued while the GPU is still busy and are all in flight
together; each asserts that the stream had not drained when the last of them returned.
"""
import ctypes as C

import cv2
import numpy as np
import pytest

from tests.test_yuv_input import _device_surface, _padded
from vnect_b200 import _capi
from vnect_b200.estimator import frame_table, strided_device_frames, uniform_frame_table, yuv_layout

SCALES2 = [1.0, 0.7]
REF = 32  # reference stream ids are the asynchronous call's ids + REF


# ------------------------------------------------------------------------------------------------ CPU
def test_uniform_table_bgr_is_views():
    a = np.zeros((3, 5, 7, 3), np.uint8)
    table, keep = uniform_frame_table(a)
    assert keep is a and len(table) == 3
    for i in range(3):
        assert (table[i].data, table[i].height, table[i].width, table[i].pitch) == (a[i].ctypes.data, 5, 7, 21)
        assert (table[i].uv_pitch, table[i].u_offset, table[i].v_offset) == (0, 0, 0)
    wide = np.zeros((6, 5, 20, 3), np.uint8)
    view = wide[::2, :, 3:10]  # the array's own row pitch (60) and frame stride (2 * 300): no copy
    table, keep = uniform_frame_table(view)
    assert keep is view
    assert [t.data for t in table] == [view[i].ctypes.data for i in range(3)]
    assert table[0].pitch == 60 and table[1].data - table[0].data == 600
    table, keep = uniform_frame_table(a[0])  # one [H,W,3] frame
    assert len(table) == 1 and table[0].data == a.ctypes.data


def test_uniform_table_yuv():
    h, w = 6, 10
    nv12 = np.zeros((2, 9, 16), np.uint8)[:, :, :w]  # rows padded to 16 bytes
    table, keep = uniform_frame_table(nv12, "nv12")
    assert keep is nv12
    for i in range(2):
        t = table[i]
        assert (t.data, t.height, t.width) == (nv12[i].ctypes.data, h, w)
        assert (t.pitch, t.uv_pitch, t.u_offset, t.v_offset) == (16, 16, 16 * h, 16 * h + 1)
    i420 = np.zeros((2, 9, w), np.uint8)
    table, keep = uniform_frame_table(i420, "i420")
    lay = yuv_layout("i420", h, w)
    assert keep is i420 and table[1].data == i420[1].ctypes.data
    assert (table[0].pitch, table[0].uv_pitch, table[0].u_offset, table[0].v_offset) == (
        w, w // 2, h * w, lay.v_offset)
    padded = np.zeros((2, 9, 16), np.uint8)[:, :, :w]  # I420 chroma has no single pitch in padded rows: copied
    table, keep = uniform_frame_table(padded, "i420")
    assert keep.flags.c_contiguous and table[0].data == keep.ctypes.data and table[0].pitch == w


def test_uniform_table_refuses_malformed_frames():
    for frames, fmt in [
        (np.zeros((2, 4, 4, 3), np.uint16), "bgr"),
        (np.zeros((2, 4, 4, 4), np.uint8), "bgr"),
        (np.zeros((2, 10, 4), np.uint8), "nv12"),  # rows not 3H/2
        (np.zeros((2, 9, 5), np.uint8), "i420"),   # odd width
        (np.zeros((0, 9, 4), np.uint8), "nv12"),   # no frames
        (np.zeros((2, 9, 4), np.int8), "nv12"),
        (np.zeros((2, 4, 4, 3), np.uint8), "yuyv"),
    ]:
        with pytest.raises(ValueError):
            uniform_frame_table(frames, fmt)


def test_strided_device_frames():
    f = strided_device_frames(4096, 3, 5, 7)
    assert f == [dict(ptr=4096 + i * 105, h=5, w=7, pitch=21) for i in range(3)]
    f = strided_device_frames(4096, 2, 5, 7, pitch=32, frame_stride=1000)
    assert [d["ptr"] for d in f] == [4096, 5096] and f[1]["pitch"] == 32
    lay = _padded("nv12", 6, 10)
    f = strided_device_frames(8192, 2, 6, 10, pixel_format="nv12", layout=lay)
    assert f[1]["ptr"] == 8192 + lay["frame_stride"]
    assert (f[0]["y_pitch"], f[0]["uv_pitch"], f[0]["u_offset"], f[0]["v_offset"]) == (
        lay["y_pitch"], lay["uv_pitch"], lay["u_offset"], lay["v_offset"])
    f = strided_device_frames(8192, 2, 6, 10, pixel_format="i420")
    assert f[1]["ptr"] == 8192 + 90 and f[0]["uv_pitch"] == 5
    for kw in (dict(pixel_format="nv12", pitch=64), dict(layout={}), dict(pixel_format="rgb")):
        with pytest.raises(ValueError):
            strided_device_frames(4096, 2, 6, 10, **kw)
    with pytest.raises(ValueError):
        strided_device_frames(4096, 0, 6, 10)


def test_capi_prototypes():
    sig = _capi.SIGNATURES
    P, FR, I32 = C.c_void_p, C.POINTER(_capi.Frame), C.c_int32
    assert sig["vnect_submit_track_frames"] == (C.c_int, [P, I32, FR, I32, I32, P, P, P, P, P, P])
    assert sig["vnect_track_device_frames"] == (C.c_int, [P, FR, I32, I32, P, P, P, P, P, P])
    assert sig["vnect_track_set_boxes"] == (C.c_int, [P, I32, P, P])


# ------------------------------------------------------------------------------------------------ GPU
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine(w0):
    import torch
    from vnect_b200 import VNectEngine
    eng = VNectEngine(w0, SCALES2, max_frames=8, max_streams=64, max_input=(1080, 1920))
    stream = torch.cuda.Stream()  # the engine runs on a torch stream, so that hold() can park it
    eng.set_cuda_stream(stream.cuda_stream)
    eng.stream = stream
    yield eng
    eng.close()


def hold(engine, ms=50):
    """Keeps the engine's stream busy for about `ms` (a spin kernel of ms * 2e6 cycles, the B200 clocks below 2 GHz):
    the calls enqueued next are all in flight together, and a call that waited for its own results would only return
    after the stream had drained."""
    import torch
    with torch.cuda.stream(engine.stream):
        torch.cuda._sleep(int(ms * 2e6))


def in_flight(engine):
    return not engine.stream.query()


def pin(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()


def pinned_out(n):
    """(joints_2d, joints_3d, boxes_used) result arrays in pinned memory: the copies into them do not block the host."""
    import torch
    return tuple(torch.empty(shape, dtype=dt).pin_memory().numpy()
                 for shape, dt in (((n, 21, 2), torch.float64), ((n, 21, 3), torch.float32), ((n, 4), torch.int32)))


@pytest.fixture(scope="module")
def video(golden):
    g = golden("video.npz")
    return g["frames"], g["t"]


def variant(frame, kind):
    """One stream's full frame derived from a 540x960 video frame."""
    if kind == "video":
        return frame
    if kind == "shift":
        return np.roll(frame, (17, -40), (0, 1))
    if kind == "pad":  # 720x1280, the video in the middle
        out = np.zeros((720, 1280, 3), np.uint8)
        out[90:630, 160:1120] = frame
        return out
    if kind == "crop":  # 480x640
        return np.ascontiguousarray(frame[30:510, 160:800])
    if kind == "odd":  # 367x491
        return np.ascontiguousarray(frame[50:417, 200:691])
    raise ValueError(kind)


def to_yuv(bgr, fmt):
    """cv2's [3H/2, W] YUV 4:2:0 frame of a BGR frame with even sides."""
    i420 = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
    if fmt == "i420":
        return i420
    h, w = bgr.shape[:2]
    q = (h // 2) * (w // 2)
    chroma = i420[h:].reshape(-1)
    return np.vstack([i420[:h], np.stack([chroma[:q], chroma[q:]], -1).reshape(h // 2, w)])


def frames_for(video, k, kinds, fmt):
    out = [variant(video[k], kind) for kind in kinds]
    return out if fmt == "bgr" else [to_yuv(f, fmt) for f in out]


def seed(engine, ids, rects):
    """set_boxes on the asynchronous ids, set_box on the reference ids; None leaves a stream unseeded."""
    pairs = [(s, r) for s, r in zip(ids, rects) if r is not None]
    engine.set_boxes([s for s, _ in pairs], [r for _, r in pairs])
    for s, r in pairs:
        engine.set_box(s + REF, r)


def same_state(engine, ids):
    return all(engine.get_box(s) == engine.get_box(s + REF) and
               np.array_equal(engine.export_stream_state(s), engine.export_stream_state(s + REF), equal_nan=True)
               for s in ids)


KINDS = ["video", "shift", "pad", "crop"]
RECTS = [(100, 0, 800, 540), None, (250, 60, 820, 560), (40, 10, 560, 470)]


@gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12", "i420"])
def test_two_lanes_match_synchronous_tracking(engine, video, fmt):
    """Every step of every stream goes to the other lane than the step before, each wait lags one submission (lane 1
    is submitted before lane 0 is waited on), and one call mixes 540x960, 720x1280 and 480x640 frames.  Pinned frames
    and results; the first two steps are enqueued behind hold()."""
    frames, t = video
    engine.reset()
    ids = list(range(len(KINDS)))
    seed(engine, ids, RECTS)
    steps = len(frames)
    got = []
    hold(engine)
    for k in range(steps):
        tk = float(t[k])
        host = [pin(f) for f in frames_for(frames, k, KINDS, fmt)]
        got.append(engine.submit_track_frames(k % 2, host, ids, tk, tk, out=pinned_out(len(ids)), pixel_format=fmt))
        if k == 1:
            assert in_flight(engine)  # neither submission waited for the GPU
        if k:
            engine.wait((k - 1) % 2)
    engine.wait((steps - 1) % 2)
    raw = engine.raw_argmax(len(ids))
    moved = set()  # (stream, box used)
    for k in range(steps):
        tk = float(t[k])
        r2, r3, rused = engine.track_frames(frames_for(frames, k, KINDS, fmt), [s + REF for s in ids], tk, tk,
                                            pixel_format=fmt)
        j2, j3, used = got[k]
        assert np.array_equal(used, rused), (fmt, k, used, rused)
        assert np.array_equal(j2, r2) and np.array_equal(j3, r3), (fmt, k)
        moved |= {(s, tuple(b)) for s, b in zip(ids, used)}
    assert np.array_equal(raw, engine.raw_argmax(len(ids)))
    assert len(moved) > len(ids) + 2  # the crops really move
    assert same_state(engine, ids)


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _outputs(torch, n):
    return (torch.empty((n, 21, 2), dtype=torch.float64, device="cuda"),
            torch.empty((n, 21, 3), dtype=torch.float32, device="cuda"),
            torch.empty((n, 4), dtype=torch.int32, device="cuda"))


@gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12"])
def test_device_frames_match_host_tracking(engine, video, fmt):
    """One allocation per stream: 480x640, 720x1280 and the unchanged video frame (unseeded: the C3 loop of
    tests/golden/video.npz), plus 367x491 in BGR or, in NV12, a decoder-like padded surface."""
    import torch
    frames, t = video
    engine.reset()
    kinds = ["crop", "pad", "video"] + (["odd"] if fmt == "bgr" else ["shift"])
    ids = list(range(len(kinds)))
    seed(engine, ids, [(40, 10, 560, 470), (250, 60, 820, 560), None, (30, 20, 400, 300)])
    j2, j3, used = _outputs(torch, len(ids))
    for k in range(len(frames)):
        tk = float(t[k])
        host = frames_for(frames, k, kinds, fmt)
        bufs, descs = [], []
        for i, f in enumerate(host):
            h, w = (f.shape[0] * 2 // 3, f.shape[1]) if fmt != "bgr" else f.shape[:2]
            if fmt == "nv12" and i == len(host) - 1:  # padded rows, chroma after padding rows
                layout = _padded(fmt, h, w)
                bufs.append(_dev(torch, _device_surface(f[None], fmt, yuv_layout(fmt, h, w, **layout))))
                descs.append(dict(ptr=bufs[-1].data_ptr(), h=h, w=w, **layout))
            else:
                bufs.append(_dev(torch, f))
                descs.append(dict(ptr=bufs[-1].data_ptr(), h=h, w=w))
        torch.cuda.synchronize()  # the engine runs on its own non-blocking stream
        engine.track_device_frames(descs, j2.data_ptr(), j3.data_ptr(), used.data_ptr(), ids, tk, tk,
                                   pixel_format=fmt)
        engine.synchronize()
        raw = engine.raw_argmax(len(ids))
        r2, r3, rused = engine.track_frames(host, [s + REF for s in ids], tk, tk, pixel_format=fmt)
        assert np.array_equal(used.cpu().numpy(), rused), (fmt, k)
        assert np.array_equal(j2.cpu().numpy(), r2) and np.array_equal(j3.cpu().numpy(), r3), (fmt, k)
        assert np.array_equal(raw, engine.raw_argmax(len(ids))), (fmt, k)
    assert same_state(engine, ids)


@gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12"])
def test_device_steps_in_flight_with_seeding(engine, video, fmt):
    """Six track_device_frames steps with set_boxes after steps 0 and 3 and a single synchronise at the end, each step
    into its own output buffers.  Step 0, the seed and step 1 are enqueued behind hold(); later steps queue behind the
    lane their predecessor-but-one used.  Against track_frames with set_box at the same points."""
    import torch
    frames, t = video
    engine.reset()
    kinds = ["video", "pad", "crop"]
    ids = [0, 1, 2]
    seed(engine, ids, [None, (250, 60, 820, 560), (40, 10, 560, 470)])
    seeds = {0: [(300, 20, 400, 500), (10, 5, 1260, 700), (200, 100, 300, 250)],
             3: [(120, 0, 700, 540), (200, 50, 900, 600), (20, 20, 600, 440)]}
    steps = 6
    host = [frames_for(frames, k, kinds, fmt) for k in range(steps)]
    dev = [[_dev(torch, f) for f in fs] for fs in host]
    outs = [_outputs(torch, len(ids)) for _ in range(steps)]
    torch.cuda.synchronize()
    hold(engine)
    for k in range(steps):
        descs = [dict(ptr=d.data_ptr(), h=(f.shape[0] * 2 // 3 if fmt != "bgr" else f.shape[0]), w=f.shape[1])
                 for d, f in zip(dev[k], host[k])]
        j2, j3, used = outs[k]
        engine.track_device_frames(descs, j2.data_ptr(), j3.data_ptr(), used.data_ptr(), ids, 1.0 + k, 1.0 + k,
                                   pixel_format=fmt)
        if k in seeds:
            engine.set_boxes(ids, seeds[k])
        if k == 1:
            assert in_flight(engine)  # step 0, the seed and step 1 are all queued behind hold()
    engine.synchronize()
    for k in range(steps):
        r2, r3, rused = engine.track_frames(host[k], [s + REF for s in ids], 1.0 + k, 1.0 + k, pixel_format=fmt)
        if k in seeds:
            for s, r in zip(ids, seeds[k]):
                engine.set_box(s + REF, r)
        j2, j3, used = (o.cpu().numpy() for o in outs[k])
        assert np.array_equal(used, rused), (fmt, k, used, rused)
        assert np.array_equal(j2, r2) and np.array_equal(j3, r3), (fmt, k)
        if k - 1 in seeds:
            assert [tuple(u) for u in used] == seeds[k - 1], (fmt, k)  # the seed landed between steps k-1 and k
    assert same_state(engine, ids)


@gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12"])
def test_track_device_matches_track(engine, video, fmt):
    """track_device on one strided device buffer (padded rows and frames) against track() on the host frames: the
    unchanged, unseeded video stream is the golden C3 loop."""
    import torch
    frames, t = video
    engine.reset()
    n, h, w = 2, 540, 960
    ids = [0, 1]
    j2, j3, used = _outputs(torch, n)
    pitch, stride = w * 3 + 64, (w * 3 + 64) * h + 4096
    layout = _padded(fmt, h, w) if fmt != "bgr" else None
    for k in range(len(frames)):
        tk = float(t[k])
        bgr = np.stack([variant(frames[k], "video"), variant(frames[k], "shift")])
        if fmt == "bgr":
            buf = np.zeros((n, stride), np.uint8)
            for i in range(n):
                buf[i, :pitch * h].reshape(h, pitch)[:, :w * 3] = bgr[i].reshape(h, w * 3)
            host, kw = bgr, dict(pitch=pitch, frame_stride=stride)
        else:
            host = np.stack([to_yuv(f, fmt) for f in bgr])
            buf = _device_surface(host, fmt, yuv_layout(fmt, h, w, **layout))
            kw = dict(layout=layout)
        dev = _dev(torch, buf)
        torch.cuda.synchronize()
        engine.track_device(dev.data_ptr(), n, h, w, j2.data_ptr(), j3.data_ptr(), used.data_ptr(), ids, tk, tk,
                            pixel_format=fmt, **kw)
        engine.synchronize()
        r2, r3, rused = engine.track(host, [s + REF for s in ids], tk, tk, pixel_format=fmt)
        assert np.array_equal(used.cpu().numpy(), rused), (fmt, k)
        assert np.array_equal(j2.cpu().numpy(), r2) and np.array_equal(j3.cpu().numpy(), r3), (fmt, k)
    assert same_state(engine, ids)


@gpu
def test_set_boxes_is_stream_ordered(engine, video):
    """Submit A on lane 0, set_boxes, submit B on lane 1, no wait in between, all three in flight behind hold(): A
    crops with the old boxes, B with the new ones, exactly as track_frames, set_box, track_frames do."""
    frames, t = video
    engine.reset()
    ids = [0, 1, 2]
    kinds = ["video", "pad", "crop"]
    old = [None, (250, 60, 820, 560), (40, 10, 560, 470)]
    new = [(300, 20, 400, 500), (10, 5, 1260, 700), (200, 100, 300, 250)]
    seed(engine, ids, old)
    fa = [pin(f) for f in frames_for(frames, 0, kinds, "bgr")]
    fb = [pin(f) for f in frames_for(frames, 1, kinds, "bgr")]
    hold(engine)
    a = engine.submit_track_frames(0, fa, ids, 1.0, 1.0, out=pinned_out(3))
    engine.set_boxes(ids, new)
    b = engine.submit_track_frames(1, fb, ids, 2.0, 2.0, out=pinned_out(3))
    assert in_flight(engine)
    engine.wait(0)
    engine.wait(1)
    assert [tuple(u) for u in a[2]] == [(0, 0, 960, 540), old[1], old[2]]
    assert [tuple(u) for u in b[2]] == new
    ra = engine.track_frames(fa, [s + REF for s in ids], 1.0, 1.0)
    for s, r in zip(ids, new):
        engine.set_box(s + REF, r)
    rb = engine.track_frames(fb, [s + REF for s in ids], 2.0, 2.0)
    for got, ref in ((a, ra), (b, rb)):
        assert all(np.array_equal(x, y) for x, y in zip(got, ref))
    assert same_state(engine, ids)


@gpu
def test_set_boxes_refusals_touch_nothing(engine, video):
    frames, t = video
    engine.reset()
    ids = [0, 1, 2]
    seed(engine, ids, [(10, 20, 300, 200), None, (5, 6, 7, 8)])
    engine.track_frames(frames_for(frames, 0, ["video"] * 3, "bgr"), ids, 1.0, 1.0)
    boxes = [engine.get_box(s) for s in range(64)]
    states = [engine.export_stream_state(s) for s in ids]
    launches = engine.launch_count()
    good = (1, 2, 30, 40)
    for sid, rects in [
        ([0, 64], [good, good]),            # id past max_streams
        ([0, -1], [good, good]),            # negative id
        ([0, 1, 0], [good, good, good]),    # duplicate id
        ([0, 1], [good, (-1, 0, 30, 40)]),  # negative x
        ([0, 1], [good, (0, -3, 30, 40)]),  # negative y
        ([0, 1], [good, (0, 0, 1, 40)]),    # w below 2
        ([0, 1], [good, (0, 0, 30, 1)]),    # h below 2
    ]:
        with pytest.raises(ValueError):
            engine.set_boxes(sid, rects)
        assert engine.launch_count() == launches, sid
    with pytest.raises(ValueError):
        engine.set_boxes([0, 1], [good])  # one rect short
    engine.set_boxes([], np.zeros((0, 4)))  # nothing to seed: nothing happens
    assert engine.launch_count() == launches
    assert [engine.get_box(s) for s in range(64)] == boxes
    assert all(np.array_equal(engine.export_stream_state(s), st, equal_nan=True) for s, st in zip(ids, states))


@gpu
def test_set_boxes_beyond_one_launch():
    """More boxes than one seeding launch carries (64)."""
    from vnect_b200 import VNectEngine
    eng = VNectEngine(False, [1.0], max_frames=1, max_streams=200)
    try:
        rng = np.random.default_rng(3)
        ids = rng.permutation(200)[:150].astype(np.int32)
        rects = np.stack([rng.integers(0, 500, 150), rng.integers(0, 500, 150), rng.integers(2, 900, 150),
                          rng.integers(2, 900, 150)], -1)
        eng.set_boxes(ids, rects)
        for s, r in zip(ids, rects):
            assert eng.get_box(int(s)) == tuple(int(v) for v in r), s
        assert eng.get_box(int(rng.permutation(np.setdiff1d(np.arange(200), ids))[0]))[2] == 1 << 30  # untouched
    finally:
        eng.close()


@gpu
def test_graphs_bounded_by_lanes_and_formats(engine, video):
    """40 tracked device steps: the crop moves every step, the frames come from a pool of 20 device allocations per
    format (more than the 16 cached graphs), the sizes change, and the format changes every other call.  The graph
    cache grows by lanes x formats, not with pointers, sizes or boxes, and every step still equals the host reference."""
    import torch
    frames, t = video
    engine.reset()
    engine.set_packed_results(0)  # also empties the graph cache, so that no LRU eviction hides an entry
    kinds = ["video", "pad", "crop"]
    pool = {fmt: [] for fmt in ("bgr", "nv12")}
    for j in range(20):
        f = variant(frames[j % len(frames)], kinds[j % 3])
        for fmt in pool:
            host = f if fmt == "bgr" else to_yuv(f, fmt)
            pool[fmt].append((host, _dev(torch, host), f.shape[:2]))
    torch.cuda.synchronize()
    ids = [0, 1]
    seed(engine, ids, [(100, 0, 800, 540), None])
    j2, j3, used = _outputs(torch, 2)
    before = engine.info("cached_graphs")
    runs, boxes = [], set()
    for k in range(40):
        fmt = ("bgr", "nv12")[(k // 2) % 2]
        picks = [pool[fmt][k % 20], pool[fmt][(k + 7) % 20]]
        descs = [dict(ptr=d.data_ptr(), h=h, w=w) for _, d, (h, w) in picks]
        tk = 1000.0 + k / 25
        engine.track_device_frames(descs, j2.data_ptr(), j3.data_ptr(), used.data_ptr(), ids, tk, tk, pixel_format=fmt)
        engine.synchronize()
        runs.append((fmt, [p[0] for p in picks], tk, j2.cpu().numpy(), j3.cpu().numpy(), used.cpu().numpy()))
        boxes.add(tuple(runs[-1][5][0]))
    growth = engine.info("cached_graphs") - before
    assert growth == 4, growth  # two lanes x two formats
    assert len(boxes) > 4
    for k, (fmt, host, tk, a, b, u) in enumerate(runs):
        r2, r3, ru = engine.track_frames(host, [s + REF for s in ids], tk, tk, pixel_format=fmt)
        assert np.array_equal(u, ru) and np.array_equal(a, r2) and np.array_equal(b, r3), k
    assert same_state(engine, ids)


@gpu
def test_refused_calls_touch_nothing(engine, video):
    import torch
    frames, t = video
    engine.reset()
    ids = [0, 1, 2]
    host = frames_for(frames, 0, ["video", "crop", "pad"], "bgr")
    seed(engine, ids, [(100, 0, 800, 540), (40, 10, 560, 470), None])
    engine.track_frames(host, ids, 5.0, 5.0)  # the streams now hold filter state, moved boxes and the clock 5.0
    boxes = [engine.get_box(s) for s in range(64)]
    states = [engine.export_stream_state(s) for s in ids]
    launches = engine.launch_count()
    bufs = [_dev(torch, f) for f in host]
    torch.cuda.synchronize()
    descs = [dict(ptr=d.data_ptr(), h=f.shape[0], w=f.shape[1]) for d, f in zip(bufs, host)]
    j2, j3, used = _outputs(torch, 8)
    out2, out3, outb = np.empty((8, 21, 2)), np.empty((8, 21, 3), np.float32), np.empty((8, 4), np.int32)
    t6 = np.full(8, 6.0)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731

    def host_call(table, lane=0, n=3, sid=ids, tt=t6, o2=out2, o3=out3):
        sid = np.asarray(sid, np.int32)
        rc = engine._lib.vnect_submit_track_frames(engine._h, lane, table, n, 0, p(sid), p(tt), p(tt),
                                                   None if o2 is None else p(o2), None if o3 is None else p(o3),
                                                   p(outb))
        _capi.raise_for(engine._lib, engine._h, rc)

    def dev_call(table, n=3, sid=ids, tt=t6, o2=True):
        sid = np.asarray(sid, np.int32)
        rc = engine._lib.vnect_track_device_frames(engine._h, table, n, 0, p(sid), p(tt), p(tt),
                                                   C.c_void_p(j2.data_ptr()) if o2 else None,
                                                   C.c_void_p(j3.data_ptr()), C.c_void_p(used.data_ptr()))
        _capi.raise_for(engine._lib, engine._h, rc)

    def table(**bad):
        tab, keep = frame_table(host)
        for k_, v in bad.items():
            setattr(tab[1], k_, v)  # the entries point into `host`, which outlives the call
        return tab

    from vnect_b200.estimator import device_frame_table

    def dtable(**bad):
        tab = device_frame_table(descs)
        for k_, v in bad.items():
            setattr(tab[1], k_, v)
        return tab

    big = np.zeros((1080, 1922, 3), np.uint8)
    bad = [
        (ValueError, lambda: host_call(table(), lane=2)),                      # bad lane
        (ValueError, lambda: host_call(table(), lane=-1)),
        (ValueError, lambda: host_call(table(), o2=None)),                     # null outputs
        (ValueError, lambda: host_call(table(), o3=None)),
        (ValueError, lambda: host_call(table(pitch=100))),                     # malformed table
        (ValueError, lambda: host_call(table(data=None))),
        (ValueError, lambda: host_call(None)),
        (ValueError, lambda: host_call(table(), n=0)),
        (ValueError, lambda: engine.submit_track_frames(1, [host[0], big, host[2]], ids, 6.0, 6.0)),  # over max_input
        (ValueError, lambda: engine.submit_track_frames(1, host, [0, 1, 0], 6.0, 6.0)),  # duplicate id
        (ZeroDivisionError, lambda: engine.submit_track_frames(0, host, ids, 5.0, 5.0)),  # repeated timestamp
        (ValueError, lambda: engine.submit_track_frames(1, host, ids, 4.0, 4.0)),        # earlier timestamp
        (ValueError, lambda: dev_call(dtable(), o2=False)),                    # device: null outputs
        (ValueError, lambda: dev_call(dtable(pitch=100))),                     # device: malformed table
        (ValueError, lambda: dev_call(dtable(height=1))),
        (ValueError, lambda: dev_call(dtable(), sid=[0, 1, 1])),               # device: duplicate id
        (ZeroDivisionError, lambda: dev_call(dtable(), tt=np.full(8, 5.0))),   # device: repeated timestamp
        (ValueError, lambda: dev_call(dtable(), tt=np.full(8, 4.0))),          # device: earlier timestamp
    ]
    for i, (exc, call) in enumerate(bad):
        with pytest.raises(exc):
            call()
        assert engine.launch_count() == launches, i
    assert [engine.get_box(s) for s in range(64)] == boxes
    for s in ids:
        assert np.array_equal(engine.export_stream_state(s), states[s], equal_nan=True), s
    # the streams continue from 5.0 as if nothing had been attempted
    got = engine.submit_track_frames(1, host, ids, 6.0, 6.0)
    engine.wait(1)
    for s in ids:
        engine.import_stream_state(states[s], s + REF)
    ref = engine.track_frames(host, [s + REF for s in ids], 6.0, 6.0)
    assert all(np.array_equal(x, y) for x, y in zip(got, ref))


@gpu
def test_fp16_guard_reported_by_wait(w0):
    """The overflow weights of test_fp16_range_guard: an asynchronous tracked call's wait raises FloatingPointError."""
    from oracle import synth
    from vnect_b200 import VNectEngine
    huge = dict(w0)
    huge["conv1/weights"] = w0["conv1/weights"] * np.float32(1e6)
    eng = VNectEngine(huge, [1.0], max_frames=1, max_streams=1)
    try:
        eng.submit_track(0, synth.frame_c2(3), [0], [1.0], [1.1])
        with pytest.raises(FloatingPointError, match="non-finite"):
            eng.wait(0)
        eng.submit_track(1, synth.frame_c2(3), [0], [2.0], [2.1])  # every batch reports, not only the first
        eng.export_stream_state(0)  # waits for the GPU, but leaves the report to the lane's wait
        eng.raw_argmax(1)
        with pytest.raises(FloatingPointError):
            eng.wait(1)
    finally:
        eng.close()


@gpu
def test_packed_results(engine, video):
    """With set_packed_results on, both asynchronous tracked paths write the same [n][21][5] buffer as
    track_frames."""
    import torch
    frames, t = video
    engine.reset()
    ids = [0, 1, 2]
    kinds = ["video", "pad", "crop"]
    seed(engine, ids, [None, (250, 60, 820, 560), (40, 10, 560, 470)])
    packed = torch.full((engine.max_frames, 21, 5), float("nan"), dtype=torch.float64, device="cuda")
    j2, j3, used = _outputs(torch, 3)
    torch.cuda.synchronize()
    engine.set_packed_results(packed.data_ptr())
    try:
        for k in range(4):
            tk = float(t[k])
            host = frames_for(frames, k, kinds, "bgr")
            if k % 2 == 0:
                engine.submit_track_frames(k % 4 // 2, host, ids, tk, tk)
                engine.wait(k % 4 // 2)
            else:
                bufs = [_dev(torch, f) for f in host]
                torch.cuda.synchronize()
                engine.track_device_frames([dict(ptr=d.data_ptr(), h=f.shape[0], w=f.shape[1])
                                            for d, f in zip(bufs, host)], j2.data_ptr(), j3.data_ptr(), None,
                                           ids, tk, tk)
                engine.synchronize()
            got = packed.cpu().numpy()[:3].copy()
            r2, r3, _ = engine.track_frames(host, [s + REF for s in ids], tk, tk)
            ref = packed.cpu().numpy()[:3]
            assert np.array_equal(got, ref), k
            assert np.array_equal(ref[:, :, :2], r2) and np.array_equal(ref[:, :, 2:], r3.astype(np.float64)), k
    finally:
        engine.set_packed_results(0)
    assert same_state(engine, ids)
