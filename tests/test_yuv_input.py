"""YUV 4:2:0 input (NV12 / I420): a YUV frame must give exactly the results of the BGR frame
cv2.cvtColor(frame, COLOR_YUV2BGR_NV12 / _I420) fed through the BGR path.

CPU: the integer restatement of OpenCV's conversion (what squarify_kernel's Yuv420Src computes) against cv2, over every
(Y, U, V) triple.  GPU: every YUV entry point against the same engine's BGR entry point on the converted frames, on
disjoint stream ids with identical timestamps; the CNN is batch-invariant, so joints_2d, joints_3d and the raw argmax
must be bit-identical.
"""
import cv2
import numpy as np
import pytest

from vnect_b200.estimator import yuv_layout

CV_CODE = {"nv12": cv2.COLOR_YUV2BGR_NV12, "i420": cv2.COLOR_YUV2BGR_I420}
SCALES2 = [1.0, 0.7]


def yuv420_to_bgr(frame, fmt):
    """cv2.cvtColor(frame, COLOR_YUV2BGR_NV12 / _I420) restated in integers: BT.601 limited range in OpenCV's 20-bit
    fixed point, one (U, V) pair per 2x2 luma block, no interpolation.  frame: uint8 [3H/2, W] in cv2's layout."""
    h, w = frame.shape[0] * 2 // 3, frame.shape[1]
    y = frame[:h].astype(np.int64)
    chroma = frame[h:].reshape(-1)
    q = (h // 2) * (w // 2)
    u, v = (chroma[0::2], chroma[1::2]) if fmt == "nv12" else (chroma[:q], chroma[q:])
    up = lambda c: np.repeat(np.repeat(c.reshape(h // 2, w // 2).astype(np.int64) - 128, 2, 0), 2, 1)  # noqa: E731
    uu, vv = up(u), up(v)
    half = 1 << 19
    yy = np.maximum(y - 16, 0) * 1220542
    bgr = [yy + half + 2116026 * uu, yy + half - 852492 * vv - 409993 * uu, yy + half + 1673527 * vv]
    return np.clip(np.stack(bgr, -1) >> 20, 0, 255).astype(np.uint8)


def random_yuv(rng, n, h, w):
    return rng.integers(0, 256, (n, h * 3 // 2, w), dtype=np.uint8)


def to_bgr(frames, fmt):
    return np.stack([cv2.cvtColor(f, CV_CODE[fmt]) for f in frames])


# ------------------------------------------------------------------------------------------------ CPU: the rule
def test_restatement_matches_cv2_on_every_yuv_triple():
    """NV12 over all 2^24 (Y, U, V) triples: one frame per U value, every (V, Y) pair in it (64 blocks of four luma
    samples per V)."""
    yb = np.arange(256, dtype=np.uint8).reshape(64, 4)  # the four luma samples of block j
    k = np.arange(128 * 128)
    blocks = yb[k % 64].reshape(128, 128, 2, 2)
    luma = blocks.transpose(0, 2, 1, 3).reshape(256, 256)
    v = (k // 64).astype(np.uint8).reshape(128, 128)
    for u in range(256):
        uv = np.stack([np.full_like(v, u), v], -1).reshape(128, 256)
        frame = np.vstack([luma, uv])
        assert np.array_equal(yuv420_to_bgr(frame, "nv12"), cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12)), u


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
@pytest.mark.parametrize("hw", [(2, 2), (6, 10), (14, 6), (8, 12), (540, 960), (1080, 1920)])
def test_restatement_matches_cv2_on_random_frames(fmt, hw):
    h, w = hw  # H a multiple of 4 and not: the I420 chroma planes then split cv2's [3H/2, W] rows differently
    frame = random_yuv(np.random.default_rng(h * 31 + w), 1, h, w)[0]
    assert np.array_equal(yuv420_to_bgr(frame, fmt), cv2.cvtColor(frame, CV_CODE[fmt]))


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_default_layout_is_cv2_contiguous(fmt):
    h, w = 6, 10
    lay = yuv_layout(fmt, h, w)
    assert (lay.y_pitch, lay.u_offset, lay.frame_stride) == (w, h * w, h * w * 3 // 2)
    if fmt == "nv12":
        assert (lay.uv_pitch, lay.v_offset) == (w, h * w + 1)
    else:  # U plane [H/2][W/2] then V plane, packed
        assert (lay.uv_pitch, lay.v_offset) == (w // 2, h * w + (h // 2) * (w // 2))
    with pytest.raises(ValueError):
        yuv_layout("nv21", h, w)


# ------------------------------------------------------------------------------------------------ GPU
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine(w0):
    from vnect_b200 import VNectEngine
    eng = VNectEngine(w0, SCALES2, max_frames=4, max_streams=16, max_input=(1080, 1920))
    yield eng
    eng.close()


def same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


SIZES = [(368, 368), (540, 960), (736, 736), (1080, 1920), (2, 2), (16, 16)]


@gpu
@pytest.mark.parametrize("fmt", ["nv12", "i420"])
@pytest.mark.parametrize("hw", SIZES)
def test_estimate_matches_bgr(engine, fmt, hw):
    """368x368 was the alias case of BGR (no squarify), 736x736 is the exact 2x area mode, 2x2 / 16x16 upscale."""
    h, w = hw
    engine.reset()
    rng = np.random.default_rng(h + w)
    for k in range(2):
        yuv = random_yuv(rng, 2, h, w)
        t = [1.0 + k, 1.0 + k]
        got = engine.estimate(yuv, [0, 1], t, t, pixel_format=fmt)
        raw_got = engine.raw_argmax(2)
        ref = engine.estimate(to_bgr(yuv, fmt), [2, 3], t, t)
        raw_ref = engine.raw_argmax(2)
        assert same(got, ref) and np.array_equal(raw_got, raw_ref), (k, fmt, hw)


@gpu
@pytest.mark.parametrize("fmt", ["nv12", "i420"])
@pytest.mark.parametrize("hw", SIZES)
def test_pipelined_submit_matches_bgr(engine, fmt, hw):
    h, w = hw
    engine.reset()
    rng = np.random.default_rng(7 * h + w)
    for k in range(3):
        yuv = random_yuv(rng, 2, h, w)
        bgr = to_bgr(yuv, fmt)
        t = [1.0 + k, 1.0 + k]
        got = engine.submit(0, yuv, [0, 1], t, t, pixel_format=fmt)
        ref = engine.submit(1, bgr, [2, 3], t, t)
        engine.wait(0)
        engine.wait(1)
        assert same(got, ref), (k, fmt, hw)


def _device_surface(yuv, fmt, lay):
    """Contiguous cv2-layout frames [n, 3H/2, W] -> bytes laid out as `lay` describes (padding filled with noise)."""
    n, rows, w = yuv.shape
    h = rows * 2 // 3
    buf = np.random.default_rng(99).integers(0, 256, (n, lay.frame_stride), dtype=np.uint8)
    cw = w if fmt == "nv12" else w // 2
    for i in range(n):
        planes = [(0, lay.y_pitch, yuv[i, :h])]
        chroma = yuv[i, h:].reshape(-1)
        if fmt == "nv12":
            planes.append((lay.u_offset, lay.uv_pitch, chroma.reshape(h // 2, w)))
        else:
            q = (h // 2) * cw
            planes += [(lay.u_offset, lay.uv_pitch, chroma[:q].reshape(h // 2, cw)),
                       (lay.v_offset, lay.uv_pitch, chroma[q:].reshape(h // 2, cw))]
        for off, pitch, plane in planes:
            for r in range(plane.shape[0]):
                buf[i, off + r * pitch: off + r * pitch + plane.shape[1]] = plane[r]
    return buf


def _padded(fmt, h, w):
    """A decoder-like surface: rows padded to y_pitch > W, the chroma plane after H + 16 luma rows."""
    yp = w + 64
    up = yp if fmt == "nv12" else yp // 2
    u = yp * (h + 16)
    v = u + 1 if fmt == "nv12" else u + up * (h // 2 + 8)
    return dict(y_pitch=yp, uv_pitch=up, u_offset=u, v_offset=v, frame_stride=v + up * (h // 2) + 4096)


@gpu
@pytest.mark.parametrize("fmt", ["nv12", "i420"])
@pytest.mark.parametrize("padded", [False, True])
def test_estimate_device_matches_bgr(engine, fmt, padded):
    import torch
    h, w, n = 540, 960, 3
    engine.reset()
    layout = _padded(fmt, h, w) if padded else None
    lay = yuv_layout(fmt, h, w, **(layout or {}))
    yuv = random_yuv(np.random.default_rng(5), n, h, w)
    dev = torch.from_numpy(_device_surface(yuv, fmt, lay)).cuda()
    torch.cuda.synchronize()  # the engine runs on its own non-blocking stream
    j2 = torch.empty((n, 21, 2), dtype=torch.float64, device="cuda")
    j3 = torch.empty((n, 21, 3), dtype=torch.float32, device="cuda")
    t = [1.0] * n
    engine.estimate_device(dev.data_ptr(), n, h, w, j2.data_ptr(), j3.data_ptr(), [0, 1, 2], t, t, pixel_format=fmt,
                           layout=layout)
    engine.synchronize()
    raw = engine.raw_argmax(n)
    ref = engine.estimate(to_bgr(yuv, fmt), [3, 4, 5], t, t)
    assert same((j2.cpu().numpy(), j3.cpu().numpy()), ref)
    assert np.array_equal(raw, engine.raw_argmax(n))


@gpu
@pytest.mark.parametrize("fmt", ["nv12", "i420"])
def test_track_matches_bgr(w0, fmt):
    """Odd crop boxes: the chroma row / column come from full-frame coordinates.  Stream 1's box is exact 2x
    (longer side 736) with an odd other side, i.e. the area mode with a partial last row of blocks."""
    from vnect_b200 import VNectEngine
    fh, fw = 540, 960
    eng = VNectEngine(w0, SCALES2, max_frames=2, max_streams=4, max_input=(fh, fw))
    try:
        rects = [(201, 33, 501, 459), (23, 41, 736, 453)]
        for s in range(2):
            eng.set_box(s, rects[s])
            eng.set_box(s + 2, rects[s])
        rng = np.random.default_rng(11)
        for k in range(3):
            yuv = random_yuv(rng, 2, fh, fw)
            t = [100 + k / 25] * 2
            j2, j3, used = eng.track(yuv, [0, 1], t, t, pixel_format=fmt)
            raw = eng.raw_argmax(2)
            r2, r3, rused = eng.track(to_bgr(yuv, fmt), [2, 3], t, t)
            assert np.array_equal(used, rused) and same((j2, j3), (r2, r3)), (k, fmt)
            assert np.array_equal(raw, eng.raw_argmax(2)), (k, fmt)
            assert [eng.get_box(s) for s in (0, 1)] == [eng.get_box(s) for s in (2, 3)], (k, fmt)
    finally:
        eng.close()


@gpu
def test_graphs_never_replay_another_format(engine):
    """Four rounds (warm-up, capture, replays) with new frame contents.  On the device path NV12, I420 and BGR calls
    share the pointers and geometry; the NV12 and I420 layouts even share every pitch and offset (I420 read with
    uv_pitch W, U and V rows side by side), so only the format tells their graphs apart."""
    import torch
    h, w, n = 368, 368, 2
    fs = h * w * 3 // 2
    engine.reset()
    common = dict(y_pitch=w, uv_pitch=w, u_offset=h * w, v_offset=h * w + 1, frame_stride=fs)
    dev = torch.empty(n * h * w * 3, dtype=torch.uint8, device="cuda")  # BGR frames, or YUV frames in its first half
    j2 = torch.empty((n, 21, 2), dtype=torch.float64, device="cuda")
    j3 = torch.empty((n, 21, 3), dtype=torch.float32, device="cuda")
    rng = np.random.default_rng(3)
    ids = {"nv12": [0, 1], "i420": [2, 3], "bgr": [4, 5]}
    # the I420 reading of `common`: U row r = chroma bytes [r*W, r*W + W/2), V row r = the same shifted by one byte
    vi = 1 + np.arange(h // 2)[:, None] * w + np.arange(w // 2)[None, :]
    for k in range(4):
        t = [1.0 + k] * n
        for fmt in ("nv12", "i420", "bgr"):
            if fmt == "bgr":
                bgr = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
                dev.copy_(torch.from_numpy(bgr.reshape(-1)))
                torch.cuda.synchronize()
                engine.estimate_device(dev.data_ptr(), n, h, w, j2.data_ptr(), j3.data_ptr(), ids[fmt], t, t)
            else:
                buf = rng.integers(0, 256, (n, fs), dtype=np.uint8)
                dev[: n * fs].copy_(torch.from_numpy(buf.reshape(-1)))
                torch.cuda.synchronize()
                engine.estimate_device(dev.data_ptr(), n, h, w, j2.data_ptr(), j3.data_ptr(), ids[fmt], t, t,
                                       pixel_format=fmt, layout=common)
                chroma = buf[:, h * w:]
                if fmt == "i420":
                    u = chroma.reshape(n, h // 2, w)[:, :, : w // 2].reshape(n, -1)
                    chroma = np.concatenate([u, chroma[:, vi].reshape(n, -1)], 1)
                bgr = to_bgr(np.concatenate([buf[:, : h * w], chroma], 1).reshape(n, h * 3 // 2, w), fmt)
            engine.synchronize()
            got = (j2.cpu().numpy(), j3.cpu().numpy())
            ref = engine.estimate(bgr, [ids[fmt][0] + 6, ids[fmt][1] + 6], t, t)
            assert same(got, ref), (k, fmt)


@gpu
def test_malformed_yuv_input_is_refused_before_anything_runs(engine):
    import ctypes as C
    import torch
    from vnect_b200 import _capi
    h, w = 540, 960
    engine.reset()
    yuv = random_yuv(np.random.default_rng(8), 1, h, w)
    dev = torch.from_numpy(yuv.reshape(1, -1)).cuda()
    torch.cuda.synchronize()
    j2 = torch.empty((1, 21, 2), dtype=torch.float64, device="cuda")
    j3 = torch.empty((1, 21, 3), dtype=torch.float32, device="cuda")
    t = [5.0]

    def device_call(hh=h, ww=w, ptr=None, fmt="nv12", **layout):
        engine.estimate_device(dev.data_ptr() if ptr is None else ptr, 1, hh, ww, j2.data_ptr(), j3.data_ptr(), [0],
                               t, t, pixel_format=fmt, layout=layout)

    def raw_call(fmt_code, reserved):
        lay = yuv_layout("nv12", h, w)
        lay.format, lay.reserved = fmt_code, reserved
        ids, tt = np.zeros(1, np.int32), np.array(t)
        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        rc = engine._lib.vnect_estimate_device_yuv(engine._h, C.c_void_p(dev.data_ptr()), 1, h, w, C.byref(lay), p(ids),
                                                   p(tt), p(tt), C.c_void_p(j2.data_ptr()), C.c_void_p(j3.data_ptr()))
        _capi.raise_for(engine._lib, engine._h, rc)

    bad = [
        lambda: raw_call(3, 0),                                        # unknown format
        lambda: raw_call(_capi.FMT_NV12, 1),                           # reserved != 0
        lambda: device_call(hh=0),                                     # H below 2
        lambda: device_call(hh=h - 1),                                 # odd H
        lambda: device_call(ww=w - 1),                                 # odd W
        lambda: device_call(y_pitch=w - 2),                            # luma pitch smaller than a row
        lambda: device_call(uv_pitch=w - 2),                           # NV12 chroma pitch smaller than a row
        lambda: device_call(fmt="i420", uv_pitch=w // 2 - 2),          # I420 chroma pitch smaller than a row
        lambda: device_call(u_offset=h * w - w, v_offset=h * w - w + 1),  # chroma plane inside the luma plane
        lambda: device_call(fmt="i420", v_offset=h * w - 1),           # I420 V plane inside the luma plane
        lambda: device_call(v_offset=h * w + 2),                       # NV12 with V not right after U
        lambda: device_call(ptr=0),                                    # null frames
        lambda: engine.estimate(random_yuv(np.random.default_rng(1), 1, 1080, 1922), [0], t, t,
                                pixel_format="nv12"),                  # wider than max_input
        lambda: engine.estimate(np.zeros((h * 3 // 2, w - 1), np.uint8), [0], t, t, pixel_format="nv12"),  # odd W
        lambda: engine.estimate(np.zeros((h * 3 // 2 + 1, w), np.uint8), [0], t, t, pixel_format="i420"),  # 3H/2 rows
        lambda: engine.estimate(yuv.astype(np.uint16), [0], t, t, pixel_format="i420"),                    # dtype
        lambda: engine.estimate(yuv, [0], t, t, pixel_format="yuyv"),                                      # format
    ]
    for i, call in enumerate(bad):
        with pytest.raises(ValueError):
            call()
    # stream 0 at t = 5.0 is still untouched: a repeated timestamp would raise ZeroDivisionError here
    got = engine.estimate(yuv, [0], t, t, pixel_format="nv12")
    ref = engine.estimate(to_bgr(yuv, "nv12"), [1], t, t)
    assert same(got, ref)
