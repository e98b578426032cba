"""Mixed-size batches: frames of different sizes, pitches and addresses in one call (vnect_submit_frames,
vnect_estimate_device_frames, vnect_track_frames).  Frame i of a mixed call must give bit-for-bit what the uniform
entry point gives for that frame alone: joints_2d, joints_3d, the raw argmax, the tracked box and the filter state.

CPU: the ctypes structure and the frame-table helpers.  GPU: every mixed entry point against the same engine's uniform
call per frame, on disjoint stream ids with identical timestamps (the CNN is batch-invariant, so everything is
compared with np.array_equal); YUV frames against the BGR call on cv2.cvtColor of them.
"""
import ctypes as C

import numpy as np
import pytest

from tests.test_yuv_input import _device_surface, _padded, random_yuv, to_bgr
from vnect_b200 import _capi
from vnect_b200.estimator import device_frame_table, frame_table, yuv_layout

SCALES2 = [1.0, 0.7]
REF = 32  # reference stream ids are the mixed call's ids + REF


# ------------------------------------------------------------------------------------------------ CPU
def test_frame_struct_layout():
    assert C.sizeof(_capi.Frame) == 48
    assert (_capi.Frame.data.offset, _capi.Frame.height.offset, _capi.Frame.width.offset) == (0, 8, 12)
    assert (_capi.Frame.pitch.offset, _capi.Frame.uv_pitch.offset) == (16, 24)
    assert (_capi.Frame.u_offset.offset, _capi.Frame.v_offset.offset) == (32, 40)


def test_frame_table_bgr_contiguous_and_strided_rows():
    a = np.zeros((5, 7, 3), np.uint8)
    wide = np.zeros((4, 20, 3), np.uint8)
    view = wide[:, 3:12]  # rows keep the wide array's pitch
    table, keep = frame_table([a, view])
    assert len(table) == 2
    assert (table[0].height, table[0].width, table[0].pitch) == (5, 7, 21)
    assert (table[1].height, table[1].width, table[1].pitch) == (4, 9, 60)
    assert table[0].data == a.ctypes.data and table[1].data == view.ctypes.data  # no copy
    assert (table[1].uv_pitch, table[1].u_offset, table[1].v_offset) == (0, 0, 0)
    flipped = a[::-1]  # negative row pitch: staged from a contiguous copy
    table, keep = frame_table([flipped])
    assert table[0].pitch == 21 and table[0].data == keep[0].ctypes.data and keep[0].flags.c_contiguous


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_frame_table_yuv(fmt):
    frames = [np.zeros((9, 10), np.uint8), np.zeros((12, 4), np.uint8)]  # 6x10 and 8x4
    table, keep = frame_table(frames, fmt)
    for i, (h, w) in enumerate([(6, 10), (8, 4)]):
        lay = yuv_layout(fmt, h, w)
        t = table[i]
        assert (t.height, t.width, t.pitch, t.uv_pitch) == (h, w, w, lay.uv_pitch)
        assert (t.u_offset, t.v_offset) == (h * w, lay.v_offset)
        assert t.data == keep[i].ctypes.data
    assert table[0].v_offset == (6 * 10 + 1 if fmt == "nv12" else 6 * 10 + 3 * 5)


def test_frame_table_refuses_malformed_frames():
    ok = np.zeros((4, 4, 3), np.uint8)
    for frames, fmt in [
        ([ok, ok.astype(np.uint16)], "bgr"),             # dtype
        ([ok, np.zeros((4, 4), np.uint8)], "bgr"),       # not [H,W,3]
        ([ok, np.zeros((4, 4, 4), np.uint8)], "bgr"),    # four channels
        ([np.zeros((10, 4), np.uint8)], "nv12"),         # rows not 3H/2
        ([np.zeros((9, 5), np.uint8)], "i420"),          # odd width
        ([np.zeros((0, 4), np.uint8)], "nv12"),          # empty
        ([np.zeros((9, 4, 1), np.uint8)], "nv12"),       # not 2-D
        ([np.zeros((9, 4), np.int8)], "nv12"),           # dtype
        ([], "bgr"),                                     # no frames
        ([ok], "yuyv"),                                  # format
    ]:
        with pytest.raises(ValueError):
            frame_table(frames, fmt)


def test_device_frame_table():
    table = device_frame_table([dict(ptr=4096, h=5, w=7), dict(ptr=8192, h=6, w=8, pitch=32)])
    assert (table[0].data, table[0].pitch, table[1].data, table[1].pitch) == (4096, 21, 8192, 32)
    table = device_frame_table([dict(ptr=4096, h=6, w=10, y_pitch=64, u_offset=64 * 8)], "nv12")
    assert (table[0].pitch, table[0].uv_pitch, table[0].u_offset, table[0].v_offset) == (64, 64, 512, 513)
    with pytest.raises(ValueError):
        device_frame_table([dict(ptr=4096, h=6, w=10, y_pitch=64)], "bgr")
    with pytest.raises(ValueError):
        device_frame_table([dict(ptr=4096, h=6, w=10, pitch=64)], "i420")


# ------------------------------------------------------------------------------------------------ GPU
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine(w0):
    from vnect_b200 import VNectEngine
    eng = VNectEngine(w0, SCALES2, max_frames=8, max_streams=64, max_input=(1080, 1920))
    yield eng
    eng.close()


# 368x368 was the BGR alias size, 736x736 the exact-2x area mode, 960x540 a portrait frame
MIXED = [(368, 368), (736, 736), (540, 960), (1080, 1920), (960, 540), (2, 2), (367, 491)]


def make_frames(rng, sizes, fmt):
    """(frames as the mixed call takes them, their BGR equivalents).  BGR: the 540x960 frame has strided rows."""
    if fmt == "bgr":
        out = []
        for h, w in sizes:
            f = rng.integers(0, 256, (h, w + 5 if (h, w) == (540, 960) else w, 3), dtype=np.uint8)
            out.append(f[:, :w])
        return out, out
    yuv = [random_yuv(rng, 1, h, w)[0] for h, w in sizes]
    return yuv, [to_bgr(f[None], fmt)[0] for f in yuv]


def reference(engine, bgr, ids, t):
    """The uniform BGR entry point, one frame per call, on stream ids + REF: (joints_2d, joints_3d, raw argmax)."""
    j2, j3, raw = [], [], []
    for f, sid in zip(bgr, ids):
        a, b = engine.estimate(f[None], [sid + REF], [t], [t])
        j2.append(a[0])
        j3.append(b[0])
        raw.append(engine.raw_argmax(1)[0])
    return np.stack(j2), np.stack(j3), np.stack(raw)


def same_state(engine, ids):
    return all(np.array_equal(engine.export_stream_state(s), engine.export_stream_state(s + REF), equal_nan=True)
               for s in ids)


def sizes_for(fmt):
    return MIXED if fmt == "bgr" else [hw for hw in MIXED if hw[0] % 2 == 0 and hw[1] % 2 == 0]


@gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12", "i420"])
def test_estimate_frames_matches_uniform_calls(engine, fmt):
    engine.reset()
    rng = np.random.default_rng(1)
    sizes = sizes_for(fmt)
    ids = list(range(len(sizes)))
    for k in range(2):  # the second step runs the filters on state the first one left
        t = 1.0 + k
        frames, bgr = make_frames(rng, sizes, fmt)
        j2, j3 = engine.estimate_frames(frames, ids, t, t, pixel_format=fmt)
        raw = engine.raw_argmax(len(ids))
        r2, r3, rraw = reference(engine, bgr, ids, t)
        assert np.array_equal(j2, r2) and np.array_equal(j3, r3) and np.array_equal(raw, rraw), (fmt, k)
        assert same_state(engine, ids), (fmt, k)


@gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12"])
def test_submit_frames_on_both_lanes(engine, fmt):
    """Lane 1's table and frames are staged while lane 0's batch still runs."""
    engine.reset()
    rng = np.random.default_rng(2)
    sizes = sizes_for(fmt)
    ids0, ids1 = list(range(4)), list(range(4, len(sizes) + 4))
    for k in range(2):
        t = 10.0 + k
        f0, b0 = make_frames(rng, sizes[::-1][:4], fmt)
        f1, b1 = make_frames(rng, sizes, fmt)
        got0 = engine.submit_frames(0, f0, ids0, t, t, pixel_format=fmt)
        got1 = engine.submit_frames(1, f1, ids1, t, t, pixel_format=fmt)
        engine.wait(0)
        engine.wait(1)
        for got, bgr, ids in ((got0, b0, ids0), (got1, b1, ids1)):
            r2, r3, _ = reference(engine, bgr, ids, t)
            assert np.array_equal(got[0], r2) and np.array_equal(got[1], r3), (fmt, k)
        assert same_state(engine, ids0 + ids1)


def _torch_bgr(torch, f, pitch):
    h, w = f.shape[:2]
    buf = np.random.default_rng(h * w).integers(0, 256, (h, pitch), dtype=np.uint8)
    buf[:, : w * 3] = f.reshape(h, w * 3)
    return torch.from_numpy(buf).cuda()


@gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12", "i420"])
def test_estimate_device_frames_matches_estimate_device(engine, fmt):
    """Each frame in its own allocation; padded BGR pitches and decoder-like YUV surfaces (pitch > W, chroma after
    padding rows) beside contiguous ones."""
    import torch
    engine.reset()
    rng = np.random.default_rng(3)
    sizes = [(540, 960), (1080, 1920), (368, 368), (720, 1280), (2, 2)]
    n = len(sizes)
    j2 = torch.empty((n, 21, 2), dtype=torch.float64, device="cuda")
    j3 = torch.empty((n, 21, 3), dtype=torch.float32, device="cuda")
    r2 = torch.empty((1, 21, 2), dtype=torch.float64, device="cuda")
    r3 = torch.empty((1, 21, 3), dtype=torch.float32, device="cuda")
    ids = list(range(n))
    for k in range(2):
        t = 20.0 + k
        bufs, descs, uniform = [], [], []
        for i, (h, w) in enumerate(sizes):
            padded = i % 2 == 0
            if fmt == "bgr":
                f = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
                pitch = w * 3 + (64 if padded else 0)
                bufs.append(_torch_bgr(torch, f, pitch))
                descs.append(dict(ptr=bufs[-1].data_ptr(), h=h, w=w, pitch=pitch))
                uniform.append(dict(pitch=pitch))
            else:
                layout = _padded(fmt, h, w) if padded else {}
                lay = yuv_layout(fmt, h, w, **layout)
                bufs.append(torch.from_numpy(_device_surface(random_yuv(rng, 1, h, w), fmt, lay)).cuda())
                descs.append(dict(ptr=bufs[-1].data_ptr(), h=h, w=w, **layout))
                uniform.append(dict(pixel_format=fmt, layout=layout or None))
        torch.cuda.synchronize()  # the engine runs on its own non-blocking stream
        engine.estimate_device_frames(descs, j2.data_ptr(), j3.data_ptr(), ids, t, t, pixel_format=fmt)
        engine.synchronize()
        got2, got3, raw = j2.cpu().numpy(), j3.cpu().numpy(), engine.raw_argmax(n)
        for i, (h, w) in enumerate(sizes):
            engine.estimate_device(descs[i]["ptr"], 1, h, w, r2.data_ptr(), r3.data_ptr(), [i + REF], t, t,
                                   **uniform[i])
            engine.synchronize()
            assert np.array_equal(got2[i], r2.cpu().numpy()[0]), (fmt, k, i)
            assert np.array_equal(got3[i], r3.cpu().numpy()[0]), (fmt, k, i)
            assert np.array_equal(raw[i], engine.raw_argmax(1)[0]), (fmt, k, i)
        assert same_state(engine, ids)


@gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12"])
def test_track_frames_matches_uniform_track(engine, fmt):
    """Streams with different full-frame sizes: odd boxes, an exact-2x box (longer side 736), a box partly outside
    its (smaller) frame, and one unseeded stream that starts from its whole frame."""
    engine.reset()
    sizes = [(540, 960), (1080, 1920), (480, 640), (720, 1280), (368, 368)]
    rects = [(201, 33, 501, 459), (23, 41, 736, 453), (401, 301, 500, 400), None, (7, 9, 301, 211)]
    ids = list(range(len(sizes)))
    for s, r in zip(ids, rects):
        if r is not None:
            engine.set_box(s, r)
            engine.set_box(s + REF, r)
    rng = np.random.default_rng(4)
    for k in range(3):
        t = 100 + k / 25
        frames, bgr = make_frames(rng, sizes, fmt)
        j2, j3, used = engine.track_frames(frames, ids, t, t, pixel_format=fmt)
        raw = engine.raw_argmax(len(ids))
        if k == 0:
            assert tuple(used[3]) == (0, 0, 1280, 720)
        for i, f in enumerate(bgr):
            r2, r3, rused = engine.track(f[None], [i + REF], [t], [t])
            assert np.array_equal(used[i], rused[0]), (fmt, k, i, used[i], rused[0])
            assert np.array_equal(j2[i], r2[0]) and np.array_equal(j3[i], r3[0]), (fmt, k, i)
            assert np.array_equal(raw[i], engine.raw_argmax(1)[0]), (fmt, k, i)
            assert engine.get_box(i) == engine.get_box(i + REF), (fmt, k, i)
        assert same_state(engine, ids)


@gpu
def test_one_graph_serves_every_composition(engine):
    """Six host calls and six device calls with three frames each; sizes, pointers and the format change between
    calls.  Each (lane, kind, format) key is warmed up, captured and replayed, and every result still equals the
    per-frame reference; the graph cache grows by one entry per key, not per composition."""
    import torch
    engine.reset()
    engine.set_packed_results(0)  # also empties the graph cache, so that no LRU eviction hides an entry
    rng = np.random.default_rng(5)
    pool = [(368, 368), (540, 960), (720, 1280), (480, 640), (2, 2), (1080, 1920), (736, 736), (960, 540)]
    ids = [0, 1, 2]
    j2 = torch.empty((3, 21, 2), dtype=torch.float64, device="cuda")
    j3 = torch.empty((3, 21, 3), dtype=torch.float32, device="cuda")
    runs = []  # (bgr frames, t, joints_2d, joints_3d, raw argmax) in call order
    before = engine.info("cached_graphs")
    for k in range(6):  # host: lane 0, BGR and NV12 alternating
        fmt = ("bgr", "nv12")[k % 2]
        sizes = [pool[(k + 3 * j) % len(pool)] for j in range(3)]
        frames, bgr = make_frames(rng, sizes, fmt)
        t = 1.0 + k
        a, b = engine.estimate_frames(frames, ids, t, t, pixel_format=fmt)
        runs.append((bgr, t, a, b, engine.raw_argmax(3)))
    host_growth = engine.info("cached_graphs") - before
    before = engine.info("cached_graphs")
    for k in range(6):  # device: the lanes alternate, so do BGR and I420 to give each key three uses
        fmt = ("bgr", "i420")[k % 2]
        sizes = [pool[(2 * k + j) % len(pool)] for j in range(3)]
        frames, bgr = make_frames(rng, sizes, fmt)
        bufs = [torch.from_numpy(np.ascontiguousarray(f)).cuda() for f in frames]  # fresh allocations every call
        torch.cuda.synchronize()
        descs = [dict(ptr=d.data_ptr(), h=h, w=w) for d, (h, w) in zip(bufs, sizes)]
        t = 10.0 + k
        engine.estimate_device_frames(descs, j2.data_ptr(), j3.data_ptr(), ids, t, t, pixel_format=fmt)
        engine.synchronize()
        runs.append((bgr, t, j2.cpu().numpy(), j3.cpu().numpy(), engine.raw_argmax(3)))
    device_growth = engine.info("cached_graphs") - before
    assert host_growth == 2 and device_growth == 2, (host_growth, device_growth)
    for k, (bgr, t, a, b, raw) in enumerate(runs):
        r2, r3, rraw = reference(engine, bgr, ids, t)
        assert np.array_equal(a, r2) and np.array_equal(b, r3) and np.array_equal(raw, rraw), k


@gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12"])
def test_capacity_and_packed_results(engine, fmt):
    """max_frames frames of max_input size each fill the lane's frame buffer exactly; the packed multi-GPU layout
    receives the mixed call's joints."""
    import torch
    engine.reset()
    n = engine.max_frames
    frames, bgr = make_frames(np.random.default_rng(6), [engine.max_input] * n, fmt)
    packed = torch.full((n, 21, 5), float("nan"), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    engine.set_packed_results(packed.data_ptr())
    try:
        j2, j3 = engine.estimate_frames(frames, list(range(n)), 1.0, 1.0, pixel_format=fmt)
        p = packed.cpu().numpy()
    finally:
        engine.set_packed_results(0)
    assert np.array_equal(p[:, :, :2], j2) and np.array_equal(p[:, :, 2:], j3.astype(np.float64))
    r2, r3, _ = reference(engine, bgr, list(range(n)), 1.0)
    assert np.array_equal(j2, r2) and np.array_equal(j3, r3)


@gpu
def test_malformed_calls_are_refused_before_anything_runs(engine):
    import torch
    engine.reset()
    rng = np.random.default_rng(7)
    ids = [0, 1, 2]
    bgr = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in [(480, 640), (540, 960), (368, 368)]]
    yuv = [random_yuv(rng, 1, h, w)[0] for h, w in [(480, 640), (540, 960), (368, 368)]]
    engine.estimate_frames(bgr, ids, 5.0, 5.0)  # the streams now hold filter state and the clock reading 5.0
    states = [engine.export_stream_state(s) for s in ids]
    launches = engine.launch_count()
    dev = torch.from_numpy(bgr[1]).cuda()
    j2 = torch.empty((3, 21, 2), dtype=torch.float64, device="cuda")
    j3 = torch.empty((3, 21, 3), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    out2, out3 = np.empty((8, 21, 2)), np.empty((8, 21, 3), np.float32)
    t6 = np.full(8, 6.0)

    def raw(table, fmt=0, n=None, sid=ids, t=t6, device=False):
        sid = np.asarray(sid, np.int32)
        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        n = len(table) if n is None else n
        if device:
            rc = engine._lib.vnect_estimate_device_frames(engine._h, table, n, fmt, p(sid), p(t), p(t),
                                                          C.c_void_p(j2.data_ptr()), C.c_void_p(j3.data_ptr()))
        else:
            rc = engine._lib.vnect_submit_frames(engine._h, 0, table, n, fmt, p(sid), p(t), p(t), p(out2), p(out3))
        _capi.raise_for(engine._lib, engine._h, rc)

    def bgr_table(**bad):
        table, keep = frame_table(bgr)
        for k, v in bad.items():
            setattr(table[1], k, v)  # a bad entry in the middle of the table
        return table

    def yuv_table(fmt="nv12", **bad):
        table, keep = frame_table(yuv, fmt)
        for k, v in bad.items():
            setattr(table[1], k, v)
        return table

    def dev_table(**bad):
        table = device_frame_table([dict(ptr=dev.data_ptr(), h=540, w=960)] * 3)
        for k, v in bad.items():
            setattr(table[1], k, v)
        return table

    big = rng.integers(0, 256, (1080, 1922, 3), dtype=np.uint8)
    bad = [
        (ValueError, lambda: raw(bgr_table(pitch=959 * 3))),                  # BGR pitch below 3W
        (ValueError, lambda: raw(bgr_table(data=None))),                      # null data
        (ValueError, lambda: raw(bgr_table(height=1))),                       # side below 2
        (ValueError, lambda: raw(bgr_table(width=0))),
        (ValueError, lambda: raw(bgr_table(), fmt=7)),                        # unknown format
        (ValueError, lambda: raw(bgr_table(), n=0)),                          # n below 1
        (ValueError, lambda: raw(bgr_table(), n=9, sid=list(range(9)), t=np.full(9, 6.0))),  # n above max_frames
        (ValueError, lambda: raw(None, n=3)),                                 # null table
        (ValueError, lambda: raw(yuv_table(v_offset=540 * 960 + 2))),         # NV12 with V not right after U
        (ValueError, lambda: raw(yuv_table(u_offset=100, v_offset=101))),     # chroma inside the luma plane
        (ValueError, lambda: raw(yuv_table("i420", uv_pitch=100))),           # I420 chroma pitch below W/2
        (ValueError, lambda: raw(yuv_table(width=961))),                      # odd width
        (ValueError, lambda: raw(dev_table(data=None), device=True)),         # device: null data
        (ValueError, lambda: raw(dev_table(pitch=100), device=True)),         # device: pitch below a row
        (ValueError, lambda: engine.estimate_frames([bgr[0], big, bgr[2]], ids, 6.0, 6.0)),  # wider than max_input
        (ValueError, lambda: engine.track_frames([bgr[0], big, bgr[2]], ids, 6.0, 6.0)),
        (ValueError, lambda: engine.estimate_frames(bgr, [0, 1, 0], 6.0, 6.0)),       # duplicate stream id
        (ZeroDivisionError, lambda: engine.estimate_frames(bgr, ids, 5.0, 5.0)),      # repeated timestamp
        (ValueError, lambda: engine.estimate_frames(bgr, ids, 4.0, 4.0)),             # earlier timestamp
        (ZeroDivisionError, lambda: engine.track_frames(yuv, ids, 5.0, 5.0, pixel_format="nv12")),
    ]
    for i, (exc, call) in enumerate(bad):
        with pytest.raises(exc):
            call()
        assert engine.launch_count() == launches, i
    for s in ids:
        assert np.array_equal(engine.export_stream_state(s), states[s], equal_nan=True), s
    # the streams continue from 5.0 as if nothing had been attempted
    j2h, j3h = engine.estimate_frames(bgr, ids, 6.0, 6.0)
    engine.estimate_frames(bgr, [s + REF for s in ids], 5.0, 5.0)
    r2, r3 = engine.estimate_frames(bgr, [s + REF for s in ids], 6.0, 6.0)
    assert np.array_equal(j2h, r2) and np.array_equal(j3h, r3)
