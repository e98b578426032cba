"""Host side of the B200-native VNect hot path.

* ``VNectEstimator`` -- drop-in for the reference class (src/estimator.py:16-142): same constructor call, attributes,
  methods and return types, so ``run_pic.py`` / ``run_estimator.py`` / ``run_estimator_ps.py`` work unchanged once
  ``src/estimator.py`` re-exports it (INTEGRATION.md).
* ``VNectEngine`` -- the batched, multi-stream form of the same path (independent frames or video streams per call),
  which is what throughput on a B200 needs; it is what ``bench.py`` drives.

Both are thin ctypes callers of ``libvnect_b200.so`` (include/vnect_b200.h).  There is no CPU path.
"""
import ctypes as C
import time

import numpy as np

from . import _capi, weights as _weights

JOINTS = 21


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


_YUV_FORMATS = {"nv12": _capi.FMT_NV12, "i420": _capi.FMT_I420}


def yuv_layout(pixel_format, h, w, y_pitch=None, uv_pitch=None, u_offset=None, v_offset=None, frame_stride=None):
    """``vnect_yuv_layout`` of h x w YUV 4:2:0 frames ("nv12" or "i420"); byte offsets relative to each frame's start.
    Fields left out follow the planes from ``y_pitch`` (default w) on without gaps, i.e. cv2's contiguous
    [3h/2, w] layout.  A decoder surface whose chroma plane starts after padding rows gives ``u_offset``
    (``y_pitch * aligned_height``) and, for several frames, ``frame_stride``."""
    if pixel_format not in _YUV_FORMATS:
        raise ValueError(f"pixel_format must be 'bgr', 'nv12' or 'i420', got {pixel_format!r}")
    nv12 = pixel_format == "nv12"
    lay = _capi.YuvLayout()
    lay.format = _YUV_FORMATS[pixel_format]
    lay.y_pitch = w if y_pitch is None else y_pitch
    lay.uv_pitch = (lay.y_pitch if nv12 else lay.y_pitch // 2) if uv_pitch is None else uv_pitch
    lay.u_offset = lay.y_pitch * h if u_offset is None else u_offset
    chroma_rows = (h // 2) * lay.uv_pitch
    lay.v_offset = (lay.u_offset + 1 if nv12 else lay.u_offset + chroma_rows) if v_offset is None else v_offset
    lay.frame_stride = ((lay.u_offset if nv12 else lay.v_offset) + chroma_rows) if frame_stride is None else frame_stride
    return lay


_FORMATS = {"bgr": _capi.FMT_BGR, **_YUV_FORMATS}

# VNECT_ORIENT_* (include/vnect_b200.h): how a stream's camera is mounted.  The name gives the numpy form of the
# oriented frame the engine sees for a stored frame f: rot90_cw = np.rot90(f, 3) (cv2.ROTATE_90_CLOCKWISE),
# rot180 = np.rot90(f, 2), rot90_ccw = np.rot90(f, 1), flip_h = f[:, ::-1] (a mirror), flip_v = f[::-1],
# transpose = f.transpose(1, 0, 2), transverse = np.rot90(f, 2).transpose(1, 0, 2).
ORIENTATIONS = {"identity": 0, "rot90_cw": 1, "rot180": 2, "rot90_ccw": 3, "flip_h": 4, "flip_v": 5, "transpose": 6,
                "transverse": 7}


def _format_code(pixel_format):
    if pixel_format not in _FORMATS:
        raise ValueError(f"pixel_format must be 'bgr', 'nv12' or 'i420', got {pixel_format!r}")
    return _FORMATS[pixel_format]


def frame_table(frames, pixel_format="bgr"):
    """Host frames of any sizes -> (``vnect_frame`` table as a ctypes array, the arrays it points into, which must
    stay alive while the call uses them).  "bgr": uint8 [H_i, W_i, 3] arrays with any row pitch; "nv12" / "i420":
    uint8 [3H_i/2, W_i] arrays in cv2's layout with even sides.  Raises ValueError on anything else."""
    _format_code(pixel_format)
    frames = list(frames)
    if not frames:
        raise ValueError("no frames")
    table, keep = (_capi.Frame * len(frames))(), []
    for i, f in enumerate(frames):
        f = np.asarray(f)
        if pixel_format == "bgr":
            if f.dtype != np.uint8 or f.ndim != 3 or f.shape[2] != 3:
                raise ValueError(f"frame {i}: BGR frames must be uint8 [H,W,3], got {f.dtype} {f.shape}")
            st = f.strides
            if not (st[2] == 1 and st[1] == 3 and st[0] >= f.shape[1] * 3):
                f = np.ascontiguousarray(f)
            h, w = f.shape[:2]
            table[i] = _capi.Frame(f.ctypes.data, h, w, f.strides[0], 0, 0, 0)
        else:
            if f.dtype != np.uint8 or f.ndim != 2 or f.shape[0] % 3 or f.shape[0] == 0:
                raise ValueError(f"frame {i}: {pixel_format} frames must be uint8 [3H/2,W], got {f.dtype} {f.shape}")
            h, w = f.shape[0] // 3 * 2, f.shape[1]
            if h % 2 or w % 2:
                raise ValueError(f"frame {i}: {pixel_format} frames need an even height and width, got {h}x{w}")
            f = np.ascontiguousarray(f)
            lay = yuv_layout(pixel_format, h, w)
            table[i] = _capi.Frame(f.ctypes.data, h, w, lay.y_pitch, lay.uv_pitch, lay.u_offset, lay.v_offset)
        keep.append(f)
    return table, keep


def device_frame_table(frames, pixel_format="bgr"):
    """Device frames -> ``vnect_frame`` table.  Each frame is a dict {ptr, h, w} plus, for BGR, an optional ``pitch``
    (default 3w) or, for "nv12" / "i420", optional yuv_layout() fields (y_pitch, uv_pitch, u_offset, v_offset;
    default cv2's contiguous layout)."""
    _format_code(pixel_format)
    frames = list(frames)
    if not frames:
        raise ValueError("no frames")
    table = (_capi.Frame * len(frames))()
    for i, d in enumerate(frames):
        d = dict(d)
        ptr, h, w = int(d.pop("ptr")), int(d.pop("h")), int(d.pop("w"))
        if pixel_format == "bgr":
            pitch = d.pop("pitch", None)
            if d:
                raise ValueError(f"frame {i}: unknown BGR frame fields {sorted(d)}")
            table[i] = _capi.Frame(ptr, h, w, w * 3 if pitch is None else pitch, 0, 0, 0)
        else:
            if set(d) - {"y_pitch", "uv_pitch", "u_offset", "v_offset", "frame_stride"}:
                raise ValueError(f"frame {i}: unknown YUV frame fields {sorted(d)}")
            lay = yuv_layout(pixel_format, h, w, **d)
            table[i] = _capi.Frame(ptr, h, w, lay.y_pitch, lay.uv_pitch, lay.u_offset, lay.v_offset)
    return table


def uniform_frame_table(frames, pixel_format="bgr"):
    """A batch of equal-size host frames as track() takes it -> (``vnect_frame`` table, the array it points into).
    Entry i is a view of frame i: its address, the array's row pitch and, between entries, the array's frame stride.
    Nothing is copied unless the rows are not byte-packed, or for I420 not contiguous (its chroma planes then have no
    single pitch).  "bgr": uint8 [n,H,W,3] or [H,W,3]; "nv12" / "i420": uint8 [n,3H/2,W] or [3H/2,W].  Raises
    ValueError on anything else."""
    _format_code(pixel_format)
    if pixel_format == "bgr":
        frames, st = VNectEngine._frames(frames)
        n, h, w = frames.shape[:3]
        table = (_capi.Frame * n)()
        for i in range(n):
            table[i] = _capi.Frame(frames.ctypes.data + i * st[0], h, w, st[1], 0, 0, 0)
        return table, frames
    frames = np.asarray(frames)
    if frames.ndim == 2:
        frames = frames[None]
    if frames.dtype != np.uint8 or frames.ndim != 3 or frames.shape[1] % 3 or 0 in frames.shape:
        raise ValueError(f"{pixel_format} frames must be uint8 [n,3H/2,W] or [3H/2,W], got {frames.dtype} "
                         f"{frames.shape}")
    n, h, w = frames.shape[0], frames.shape[1] // 3 * 2, frames.shape[2]
    if h % 2 or w % 2:
        raise ValueError(f"{pixel_format} frames need an even height and width, got {h}x{w}")
    st = frames.strides
    if not (st[2] == 1 and st[1] >= w and st[0] >= 0 and (pixel_format == "nv12" or st[1] == w)):
        frames = np.ascontiguousarray(frames)
        st = frames.strides
    lay = yuv_layout(pixel_format, h, w, y_pitch=st[1])
    table = (_capi.Frame * n)()
    for i in range(n):
        table[i] = _capi.Frame(frames.ctypes.data + i * st[0], h, w, lay.y_pitch, lay.uv_pitch, lay.u_offset,
                               lay.v_offset)
    return table, frames


def strided_device_frames(dev_frames_ptr, n, h, w, pitch=None, frame_stride=None, pixel_format="bgr", layout=None):
    """The n frames estimate_device() describes (frame i at ``dev_frames_ptr + i * frame_stride``) as the list of
    frames device_frame_table() takes.  BGR: ``pitch`` (default 3w) and ``frame_stride`` (default pitch * h); YUV:
    ``layout``, a dict of yuv_layout() fields (default cv2's contiguous layout)."""
    _format_code(pixel_format)
    if n < 1:
        raise ValueError(f"n must be at least 1, got {n}")
    if pixel_format == "bgr":
        if layout is not None:
            raise ValueError("BGR frames are described by pitch / frame_stride, not by `layout`")
        pitch = w * 3 if pitch is None else int(pitch)
        stride = pitch * h if frame_stride is None else int(frame_stride)
        return [dict(ptr=int(dev_frames_ptr) + i * stride, h=h, w=w, pitch=pitch) for i in range(n)]
    if pitch is not None or frame_stride is not None:
        raise ValueError("YUV frames are described by `layout`, not by pitch / frame_stride")
    lay = yuv_layout(pixel_format, h, w, **(layout or {}))
    planes = dict(y_pitch=lay.y_pitch, uv_pitch=lay.uv_pitch, u_offset=lay.u_offset, v_offset=lay.v_offset)
    return [dict(ptr=int(dev_frames_ptr) + i * lay.frame_stride, h=h, w=w, **planes) for i in range(n)]


def planar_to_nhwc(planar):
    """Planar maps float32 [n][84][hs][hs] (what the CNN writes and vnect_get_maps returns: channel 21 * m + j is joint
    j of map m = hm, xm, ym, zm) -> the 4-tuple (hm, xm, ym, zm) of NHWC [n][hs][hs][21] arrays that postprocess(),
    track_postprocess() and the reference's sess.run (src/estimator.py:100-104) use."""
    planar = np.asarray(planar, dtype=np.float32)
    n, c, hs = planar.shape[:3]
    if c != 4 * JOINTS or planar.shape != (n, c, hs, hs):
        raise ValueError(f"expected planar maps [n,{4 * JOINTS},hs,hs], got {planar.shape}")
    nhwc = planar.reshape(n, 4, JOINTS, hs, hs).transpose(1, 0, 3, 4, 2)
    return tuple(np.ascontiguousarray(m) for m in nhwc)


def nhwc_to_planar(maps):
    """Inverse of planar_to_nhwc: the transposition vnect_postprocess / vnect_track_postprocess apply to their maps."""
    maps = np.stack([np.asarray(m, dtype=np.float32) for m in maps])  # [4][n][hs][hs][21]
    if maps.ndim != 5 or maps.shape[4] != JOINTS or maps.shape[2] != maps.shape[3]:
        raise ValueError(f"expected 4 maps [n,hs,hs,{JOINTS}], got {maps.shape[1:]}")
    return np.ascontiguousarray(maps.transpose(1, 0, 4, 2, 3).reshape(maps.shape[1], 4 * JOINTS, *maps.shape[2:4]))


def check_maps(maps, n_scales, hs):
    """(hm, xm, ym, zm), each [n*n_scales, hs, hs, 21] -> (contiguous float32 maps, n).  vnect_postprocess and
    vnect_track_postprocess read exactly that many floats from each, so any other shape is refused here."""
    maps = [np.ascontiguousarray(m, dtype=np.float32) for m in maps]
    n = maps[0].shape[0] // n_scales if maps and maps[0].ndim == 4 else 0
    want = (n * n_scales, hs, hs, JOINTS)
    if len(maps) != 4 or n < 1 or any(m.shape != want for m in maps):
        raise ValueError(f"expected 4 maps [n*{n_scales}, {hs}, {hs}, {JOINTS}] with n >= 1, got "
                         f"{[m.shape for m in maps]}")
    return maps, n


class VNectEngine:
    """Batched estimator: ``estimate(frames[n,H,W,3] uint8 BGR) -> (joints_2d [n,21,2] f64, joints_3d [n,21,3] f32)``.

    One engine = one GPU + one CUDA stream.  Frames of one call are independent (distinct ``stream_ids``); successive
    calls with the same stream id continue that stream's OneEuroFilter state (src/estimator.py:83-95).
    """

    def __init__(self, weights=None, scales=(1, 0.85, 0.7), box_size=368, max_frames=1, max_streams=None,
                 max_input=None, device=0, filters=True):
        self._lib = _capi.load_library()
        self._h = C.c_void_p()
        self.scales = [float(s) for s in scales]
        self.box_size = int(box_size)
        self.hm_size = self.box_size // 8
        self.max_frames = int(max_frames)
        self.max_streams = int(max_streams if max_streams is not None else max_frames)
        self.max_input = tuple(max_input) if max_input else (self.box_size, self.box_size)
        self.device = int(device)
        self.filters = bool(filters)
        cfg = _capi.Config()
        cfg.device = self.device
        cfg.box_size = self.box_size
        cfg.n_scales = len(self.scales)
        if not 1 <= len(self.scales) <= _capi.MAX_SCALES:
            raise ValueError("1..4 scales supported")
        for i, s in enumerate(self.scales):
            cfg.scales[i] = s
        cfg.max_frames = self.max_frames
        cfg.max_streams = self.max_streams
        cfg.max_input_h, cfg.max_input_w = int(self.max_input[0]), int(self.max_input[1])
        cfg.filters = 1 if filters else 0
        rc = self._lib.vnect_create(C.byref(self._h), C.byref(cfg))
        try:
            self._check(rc)
            if weights is not False:  # False: pre/post-processing only, no CNN
                self._load(_weights.resolve(weights))
        except Exception:
            self.close()
            raise

    # ------------------------------------------------------------------------------------------------ plumbing
    def _check(self, rc):
        _capi.raise_for(self._lib, self._h, rc)

    def _load(self, wdict):
        """VNect.load_weights (src/vnect_model.py:219-236): every variable of the graph, by TF name."""
        for name in _weights.variable_shapes():
            if name not in wdict:
                raise KeyError(f"weights lack variable '{name}'")
            arr = np.ascontiguousarray(wdict[name], dtype=np.float32)
            shape = (C.c_int64 * arr.ndim)(*arr.shape)
            self._check(self._lib.vnect_set_weight(self._h, name.encode(), _ptr(arr), shape, arr.ndim))
        self._check(self._lib.vnect_finalize(self._h))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.vnect_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------------------------------------ operators
    def forward(self, batch):
        """sess.run([split_2:0..3], {Placeholder:0: batch}) (src/estimator.py:100-104)."""
        batch = np.ascontiguousarray(batch, dtype=np.float32)
        n, s = batch.shape[0], self.box_size
        if batch.shape != (n, s, s, 3):
            raise ValueError(f"expected [n,{s},{s},3], got {batch.shape}")
        outs = [np.empty((n, self.hm_size, self.hm_size, JOINTS), np.float32) for _ in range(4)]
        self._check(self._lib.vnect_forward(self._h, _ptr(batch), n, *[_ptr(o) for o in outs]))
        return tuple(outs)

    @staticmethod
    def _frames(frames):
        frames = np.asarray(frames)
        if frames.ndim == 3:
            frames = frames[None]
        if frames.dtype != np.uint8 or frames.ndim != 4 or frames.shape[3] != 3:
            raise ValueError("frames must be uint8 [n,H,W,3] (BGR)")
        st = frames.strides
        if not (st[3] == 1 and st[2] == 3 and st[1] >= frames.shape[2] * 3 and st[0] >= 0):
            frames = np.ascontiguousarray(frames)
            st = frames.strides
        return frames, st

    def _source(self, frames, pixel_format):
        """Frames of any accepted pixel format -> (host array, n, H, W, the C entry point's frame-description
        arguments).  BGR: uint8 [n,H,W,3]; "nv12" / "i420": uint8 [n,3H/2,W] or [3H/2,W] in cv2's layout."""
        if pixel_format == "bgr":
            frames, st = self._frames(frames)
            n, h, w = frames.shape[:3]
            return frames, n, h, w, (st[1], st[0] if n > 1 else st[1] * h)
        yuv_layout(pixel_format, 2, 2)  # rejects an unknown format before the frames are looked at
        frames = np.asarray(frames)
        if frames.ndim == 2:
            frames = frames[None]
        if frames.dtype != np.uint8 or frames.ndim != 3 or frames.shape[1] % 3 or frames.shape[1] == 0:
            raise ValueError(f"{pixel_format} frames must be uint8 [n,3H/2,W] or [3H/2,W], got {frames.dtype} "
                             f"{frames.shape}")
        n, h, w = frames.shape[0], frames.shape[1] // 3 * 2, frames.shape[2]
        if h % 2 or w % 2:
            raise ValueError(f"{pixel_format} frames need an even height and width, got {h}x{w}")
        frames = np.ascontiguousarray(frames)
        return frames, n, h, w, (C.byref(yuv_layout(pixel_format, h, w)),)

    def _meta(self, n, stream_ids, t2d, t3d):
        ids = np.arange(n, dtype=np.int32) if stream_ids is None else np.ascontiguousarray(stream_ids, dtype=np.int32)
        if t2d is None:
            t2d = np.full(n, time.time())
        if t3d is None:
            t3d = np.full(n, time.time())
        t2d = np.ascontiguousarray(np.broadcast_to(np.asarray(t2d, dtype=np.float64), (n,)))
        t3d = np.ascontiguousarray(np.broadcast_to(np.asarray(t3d, dtype=np.float64), (n,)))
        if ids.shape != (n,):
            raise ValueError("stream_ids must have one entry per frame")
        return ids, t2d, t3d

    @staticmethod
    def _scores_out(scores, n):
        """The ``scores`` argument of a host-result method -> None (False) or the float64 [n, 21] array the call writes
        every joint's score to (True: a new one; an array: that array, which must be C-contiguous and writable)."""
        if scores is False or scores is None:
            return None
        if scores is True:
            return np.empty((n, JOINTS), np.float64)
        if not (isinstance(scores, np.ndarray) and scores.dtype == np.float64 and scores.shape == (n, JOINTS)
                and scores.flags.c_contiguous and scores.flags.writeable):
            raise ValueError(f"scores must be True, False or a writable C-contiguous float64 [{n}, {JOINTS}] array")
        return scores

    def _request_scores(self, ptr):
        """vnect_request_scores: the C call made right after this one also writes its scores to ``ptr`` (a host
        array's or a device address); nothing that can raise may run in between."""
        if ptr is not None:
            self._check(self._lib.vnect_request_scores(self._h, ptr))

    def estimate(self, frames, stream_ids=None, t2d=None, t3d=None, out=None, pixel_format="bgr", scores=False):
        """VNectEstimator.__call__ for n independent frames (host arrays in, host arrays out).  ``pixel_format``
        "nv12" / "i420" takes YUV 4:2:0 frames (uint8 [n,3H/2,W]) and gives exactly the results of the BGR frames
        cv2.cvtColor(frame, COLOR_YUV2BGR_NV12 / _I420); the conversion runs inside the pre-processing.
        ``scores``: True, or a float64 [n, 21] array, adds every joint's confidence (vnect_request_scores: the
        reference's float64 upsampled heat-map value at its argmax) as a last result.  The same holds for every
        host-result method below."""
        if pixel_format != "bgr":
            res = self.submit(0, frames, stream_ids, t2d, t3d, out, pixel_format=pixel_format, scores=scores)
            self.wait(0)
            return res
        frames, st = self._frames(frames)
        n, h, w = frames.shape[:3]
        ids, t2d, t3d = self._meta(n, stream_ids, t2d, t3d)
        j2, j3 = out if out is not None else (np.empty((n, JOINTS, 2), np.float64), np.empty((n, JOINTS, 3), np.float32))
        sc = self._scores_out(scores, n)
        self._request_scores(None if sc is None else _ptr(sc))
        self._check(self._lib.vnect_estimate(self._h, _ptr(frames), n, h, w, st[1], st[0] if n > 1 else st[1] * h,
                                             _ptr(ids), _ptr(t2d), _ptr(t3d), _ptr(j2), _ptr(j3)))
        return (j2, j3) if sc is None else (j2, j3, sc)

    def _enqueued(self, lane, keep, results, sc):
        """Records a submitted call's buffers until wait(lane) and returns its results (+ scores when asked)."""
        results = tuple(results) + ((sc,) if sc is not None else ())
        self._inflight = getattr(self, "_inflight", {})
        self._inflight[int(lane)] = (keep, *results)  # keep the buffers alive
        return results

    def submit(self, lane, frames, stream_ids=None, t2d=None, t3d=None, out=None, pixel_format="bgr", scores=False):
        """Pipelined estimate(): enqueue a batch on lane 0/1 and return (joints_2d, joints_3d) arrays that are filled
        once wait(lane) returns.  `frames` and the result arrays must stay alive until then (pinned memory makes the
        copies truly asynchronous).  ``pixel_format`` and ``scores`` as in estimate()."""
        frames, n, h, w, layout = self._source(frames, pixel_format)
        ids, t2d, t3d = self._meta(n, stream_ids, t2d, t3d)
        j2, j3 = out if out is not None else (np.empty((n, JOINTS, 2), np.float64), np.empty((n, JOINTS, 3), np.float32))
        sc = self._scores_out(scores, n)
        fn = self._lib.vnect_submit if pixel_format == "bgr" else self._lib.vnect_submit_yuv
        self._request_scores(None if sc is None else _ptr(sc))
        self._check(fn(self._h, int(lane), _ptr(frames), n, h, w, *layout, _ptr(ids), _ptr(t2d), _ptr(t3d), _ptr(j2),
                       _ptr(j3)))
        return self._enqueued(lane, frames, (j2, j3), sc)

    def estimate_frames(self, frames, stream_ids=None, t2d=None, t3d=None, out=None, pixel_format="bgr", scores=False):
        """estimate() for frames of different sizes in one batch: ``frames`` is a sequence of host arrays as
        frame_table() takes them.  Frame i gives exactly what estimate() gives for that frame alone."""
        res = self.submit_frames(0, frames, stream_ids, t2d, t3d, out, pixel_format=pixel_format, scores=scores)
        self.wait(0)
        return res

    def submit_frames(self, lane, frames, stream_ids=None, t2d=None, t3d=None, out=None, pixel_format="bgr",
                      scores=False):
        """submit() for frames of different sizes (see estimate_frames); completes with wait(lane)."""
        table, keep = frame_table(frames, pixel_format)
        n = len(table)
        ids, t2d, t3d = self._meta(n, stream_ids, t2d, t3d)
        j2, j3 = out if out is not None else (np.empty((n, JOINTS, 2), np.float64), np.empty((n, JOINTS, 3), np.float32))
        sc = self._scores_out(scores, n)
        self._request_scores(None if sc is None else _ptr(sc))
        self._check(self._lib.vnect_submit_frames(self._h, int(lane), table, n, _format_code(pixel_format), _ptr(ids),
                                                  _ptr(t2d), _ptr(t3d), _ptr(j2), _ptr(j3)))
        return self._enqueued(lane, keep, (j2, j3), sc)

    def _sequence_meta(self, n, stream_ids, t2d, t3d):
        """_meta for a sequence call: ids are required and, with filters on, one 2D and one 3D reading per frame (a
        default clock reading would repeat within the call)."""
        if stream_ids is None:
            raise ValueError("a sequence call needs stream_ids")
        if self.filters and (t2d is None or t3d is None):
            raise ValueError("a sequence call with filters on needs t2d and t3d for every frame")
        return self._meta(n, stream_ids, 0.0 if t2d is None else t2d, 0.0 if t3d is None else t3d)

    def estimate_sequence(self, frames, stream_ids, t2d=None, t3d=None, out=None, pixel_format="bgr", scores=False):
        """estimate_frames() where a stream id may appear several times: the frames of one stream are consecutive in
        time in call order (they may be interleaved with other streams' frames).  Frame i gets bit for bit what
        estimate_frames() gives when the frames go in one per call in call order; the CNN runs over the whole call at
        batch size.  A call refused for its ids or timestamps processes none of its frames."""
        res = self.submit_sequence(0, frames, stream_ids, t2d, t3d, out, pixel_format=pixel_format, scores=scores)
        self.wait(0)
        return res

    def submit_sequence(self, lane, frames, stream_ids, t2d=None, t3d=None, out=None, pixel_format="bgr",
                        scores=False):
        """submit_frames() for a sequence call (see estimate_sequence); completes with wait(lane)."""
        table, keep = frame_table(frames, pixel_format)
        n = len(table)
        ids, t2d, t3d = self._sequence_meta(n, stream_ids, t2d, t3d)
        j2, j3 = out if out is not None else (np.empty((n, JOINTS, 2), np.float64), np.empty((n, JOINTS, 3), np.float32))
        sc = self._scores_out(scores, n)
        self._request_scores(None if sc is None else _ptr(sc))
        self._check(self._lib.vnect_submit_sequence(self._h, int(lane), table, n, _format_code(pixel_format),
                                                    _ptr(ids), _ptr(t2d), _ptr(t3d), _ptr(j2), _ptr(j3)))
        return self._enqueued(lane, keep, (j2, j3), sc)

    def estimate_device_sequence(self, frames, dev_j2_ptr, dev_j3_ptr, stream_ids, t2d=None, t3d=None,
                                 pixel_format="bgr", dev_scores_ptr=None):
        """estimate_device_frames() for a sequence call (see estimate_sequence).  Asynchronous."""
        table = device_frame_table(frames, pixel_format)
        n = len(table)
        ids, t2d, t3d = self._sequence_meta(n, stream_ids, t2d, t3d)
        self._request_scores(C.c_void_p(dev_scores_ptr) if dev_scores_ptr else None)
        self._check(self._lib.vnect_estimate_device_sequence(self._h, table, n, _format_code(pixel_format), _ptr(ids),
                                                             _ptr(t2d), _ptr(t3d), C.c_void_p(dev_j2_ptr),
                                                             C.c_void_p(dev_j3_ptr)))

    def wait(self, lane):
        """Completes the lane's submission: (joints_2d, joints_3d), or (joints_2d, joints_3d, boxes_used) after
        submit_track / submit_track_frames, followed by the scores when the submission asked for them."""
        self._check(self._lib.vnect_wait(self._h, int(lane)))
        return self.__dict__.get("_inflight", {}).pop(int(lane), (None, None, None))[1:]

    def set_box(self, stream_id, rect):
        """Seed the tracked crop box (x, y, w, h) of a stream (what HOGBox provides in run_estimator.py:66-83)."""
        x, y, w, h = (int(v) for v in rect)
        self._check(self._lib.vnect_track_set_box(self._h, int(stream_id), x, y, w, h))

    def get_box(self, stream_id):
        out = (C.c_int32 * 4)()
        self._check(self._lib.vnect_track_get_box(self._h, int(stream_id), out))
        return tuple(out)

    def track(self, frames, stream_ids=None, t2d=None, t3d=None, pixel_format="bgr", scores=False):
        """One step of the reference's video loop (run_estimator.py:98-119) for n streams: crop each full frame by
        its stream's box, estimate, shift joints_2d to full-frame coordinates, update the box on the device.
        Returns (joints_2d [n,21,2], joints_3d [n,21,3], boxes_used [n,4]).  ``pixel_format`` as in estimate()."""
        frames, n, h, w, layout = self._source(frames, pixel_format)
        ids, t2d, t3d = self._meta(n, stream_ids, t2d, t3d)
        j2, j3 = np.empty((n, JOINTS, 2), np.float64), np.empty((n, JOINTS, 3), np.float32)
        boxes = np.empty((n, 4), np.int32)
        sc = self._scores_out(scores, n)
        fn = self._lib.vnect_track if pixel_format == "bgr" else self._lib.vnect_track_yuv
        self._request_scores(None if sc is None else _ptr(sc))
        self._check(fn(self._h, _ptr(frames), n, h, w, *layout, _ptr(ids), _ptr(t2d), _ptr(t3d), _ptr(j2), _ptr(j3),
                       _ptr(boxes)))
        return (j2, j3, boxes) if sc is None else (j2, j3, boxes, sc)

    def track_frames(self, frames, stream_ids=None, t2d=None, t3d=None, pixel_format="bgr", scores=False):
        """track() for streams whose full frames differ in size: each frame is cropped by its stream's box clipped to
        that frame.  Returns (joints_2d [n,21,2], joints_3d [n,21,3], boxes_used [n,4])."""
        table, keep = frame_table(frames, pixel_format)
        n = len(table)
        ids, t2d, t3d = self._meta(n, stream_ids, t2d, t3d)
        j2, j3 = np.empty((n, JOINTS, 2), np.float64), np.empty((n, JOINTS, 3), np.float32)
        boxes = np.empty((n, 4), np.int32)
        sc = self._scores_out(scores, n)
        self._request_scores(None if sc is None else _ptr(sc))
        self._check(self._lib.vnect_track_frames(self._h, table, n, _format_code(pixel_format), _ptr(ids), _ptr(t2d),
                                                 _ptr(t3d), _ptr(j2), _ptr(j3), _ptr(boxes)))
        return (j2, j3, boxes) if sc is None else (j2, j3, boxes, sc)

    def submit_track(self, lane, frames, stream_ids=None, t2d=None, t3d=None, out=None, pixel_format="bgr",
                     scores=False):
        """Pipelined track(): enqueue one tracked step on lane 0/1 and return (joints_2d, joints_3d, boxes_used)
        arrays that are filled once wait(lane) returns.  Same frames as track(); the call reads them in place
        (uniform_frame_table), so they, and ``out`` if given, must stay alive until the wait (pinned memory makes the
        copies truly asynchronous).  Steps of one stream may alternate between the lanes."""
        table, keep = uniform_frame_table(frames, pixel_format)
        return self._submit_track(lane, table, keep, stream_ids, t2d, t3d, out, pixel_format, scores)

    def submit_track_frames(self, lane, frames, stream_ids=None, t2d=None, t3d=None, out=None, pixel_format="bgr",
                            scores=False):
        """submit_track() for streams whose full frames differ in size, as track_frames() takes them."""
        table, keep = frame_table(frames, pixel_format)
        return self._submit_track(lane, table, keep, stream_ids, t2d, t3d, out, pixel_format, scores)

    def _submit_track(self, lane, table, keep, stream_ids, t2d, t3d, out, pixel_format, scores):
        n = len(table)
        ids, t2d, t3d = self._meta(n, stream_ids, t2d, t3d)
        j2, j3, boxes = out if out is not None else (np.empty((n, JOINTS, 2), np.float64),
                                                     np.empty((n, JOINTS, 3), np.float32), np.empty((n, 4), np.int32))
        sc = self._scores_out(scores, n)
        self._request_scores(None if sc is None else _ptr(sc))
        self._check(self._lib.vnect_submit_track_frames(self._h, int(lane), table, n, _format_code(pixel_format),
                                                        _ptr(ids), _ptr(t2d), _ptr(t3d), _ptr(j2), _ptr(j3),
                                                        _ptr(boxes)))
        return self._enqueued(lane, keep, (j2, j3, boxes), sc)

    def track_device_frames(self, frames, dev_j2_ptr, dev_j3_ptr, dev_boxes_ptr=None, stream_ids=None, t2d=None,
                            t3d=None, pixel_format="bgr", dev_scores_ptr=None):
        """track_frames() on device full frames (``frames`` as device_frame_table() takes them) with device results:
        joints_2d float64 [n,21,2], joints_3d float32 [n,21,3] and, when ``dev_boxes_ptr`` is given, boxes_used int32
        [n,4]; when ``dev_scores_ptr`` is given, every joint's score float64 [n,21] (as for every *_device* method).
        Asynchronous on the engine's stream."""
        table = device_frame_table(frames, pixel_format)
        n = len(table)
        ids, t2d, t3d = self._meta(n, stream_ids, t2d, t3d)
        self._request_scores(C.c_void_p(dev_scores_ptr) if dev_scores_ptr else None)
        self._check(self._lib.vnect_track_device_frames(self._h, table, n, _format_code(pixel_format), _ptr(ids),
                                                        _ptr(t2d), _ptr(t3d), C.c_void_p(dev_j2_ptr),
                                                        C.c_void_p(dev_j3_ptr),
                                                        C.c_void_p(dev_boxes_ptr) if dev_boxes_ptr else None))

    def track_device(self, dev_frames_ptr, n, h, w, dev_j2_ptr, dev_j3_ptr, dev_boxes_ptr=None, stream_ids=None,
                     t2d=None, t3d=None, pitch=None, frame_stride=None, pixel_format="bgr", layout=None,
                     dev_scores_ptr=None):
        """track_device_frames() on n equal-size device frames described as estimate_device() takes them."""
        frames = strided_device_frames(dev_frames_ptr, n, h, w, pitch, frame_stride, pixel_format, layout)
        self.track_device_frames(frames, dev_j2_ptr, dev_j3_ptr, dev_boxes_ptr, stream_ids, t2d, t3d, pixel_format,
                                 dev_scores_ptr)

    def set_boxes(self, stream_ids, rects):
        """set_box() for several streams, in submission order: after every call already submitted and before every
        later one, without waiting for the GPU."""
        ids = np.ascontiguousarray(stream_ids, dtype=np.int32).reshape(-1)
        rects = np.ascontiguousarray(rects, dtype=np.int32)
        if rects.shape != (len(ids), 4):
            raise ValueError(f"expected one (x, y, w, h) per stream id: {len(ids)} ids, rects {rects.shape}")
        self._check(self._lib.vnect_track_set_boxes(self._h, len(ids), _ptr(ids), _ptr(rects)))

    def set_orientations(self, stream_ids, orientations):
        """Set how each stream's camera is mounted: a code or a name of ``ORIENTATIONS`` per stream id.  Every later
        call, on either lane, reads that stream's frames as stored and sees them oriented; joints, boxes and
        ``boxes_used`` are in the oriented frame.  Calls already submitted keep their orientation; reset() keeps it
        and export_stream_state() does not carry it."""
        ids = np.ascontiguousarray(stream_ids, dtype=np.int32).reshape(-1)
        codes = [ORIENTATIONS[o] if isinstance(o, str) and o in ORIENTATIONS else o
                 for o in np.asarray(orientations, dtype=object).reshape(-1)]
        if any(isinstance(o, str) for o in codes):
            raise ValueError(f"unknown orientation name in {orientations!r}: expected one of {list(ORIENTATIONS)}")
        codes = np.ascontiguousarray(codes, dtype=np.int32)
        if codes.shape != ids.shape:
            raise ValueError(f"expected one orientation per stream id: {len(ids)} ids, {len(codes)} orientations")
        self._check(self._lib.vnect_set_orientations(self._h, len(ids), _ptr(ids), _ptr(codes)))

    def orientation(self, stream_id):
        """The orientation code of a stream (see ``ORIENTATIONS``)."""
        out = C.c_int32()
        self._check(self._lib.vnect_get_orientation(self._h, int(stream_id), C.byref(out)))
        return out.value

    def set_track_recovery(self, stream_ids, min_mean_scores):
        """Recover lost people in tracked streams: when the mean score (sum(scores[f]) / 21, summed in joint order)
        of a stream's tracked frame falls below its threshold, its next frame is cropped to the whole frame instead of
        the box built from the current joints.  One threshold per stream id; 0 turns recovery off (the default).
        Calls already submitted keep the thresholds they were submitted with; reset() keeps them and
        export_stream_state() does not carry them."""
        ids = np.ascontiguousarray(stream_ids, dtype=np.int32).reshape(-1)
        tau = np.ascontiguousarray(min_mean_scores, dtype=np.float64).reshape(-1)
        if tau.shape != ids.shape:
            raise ValueError(f"expected one threshold per stream id: {len(ids)} ids, {len(tau)} thresholds")
        self._check(self._lib.vnect_set_track_recovery(self._h, len(ids), _ptr(ids), _ptr(tau)))

    def track_recovery(self, stream_id):
        """The recovery threshold of a stream (0 = off)."""
        out = C.c_double()
        self._check(self._lib.vnect_get_track_recovery(self._h, int(stream_id), C.byref(out)))
        return out.value

    def estimate_device_frames(self, frames, dev_j2_ptr, dev_j3_ptr, stream_ids=None, t2d=None, t3d=None,
                               pixel_format="bgr", dev_scores_ptr=None):
        """estimate_device() for device frames of different sizes, each at its own address (e.g. one tensor or
        decoder surface per camera): ``frames`` as device_frame_table() takes them.  Asynchronous."""
        table = device_frame_table(frames, pixel_format)
        n = len(table)
        ids, t2d, t3d = self._meta(n, stream_ids, t2d, t3d)
        self._request_scores(C.c_void_p(dev_scores_ptr) if dev_scores_ptr else None)
        self._check(self._lib.vnect_estimate_device_frames(self._h, table, n, _format_code(pixel_format), _ptr(ids),
                                                           _ptr(t2d), _ptr(t3d), C.c_void_p(dev_j2_ptr),
                                                           C.c_void_p(dev_j3_ptr)))

    def estimate_device(self, dev_frames_ptr, n, h, w, dev_j2_ptr, dev_j3_ptr, stream_ids=None, t2d=None, t3d=None,
                        pitch=None, frame_stride=None, pixel_format="bgr", layout=None, dev_scores_ptr=None):
        """Same path with frames / results resident in device memory (raw device pointers, e.g. tensor.data_ptr()).
        For "nv12" / "i420" frames of h x w pixels, ``layout`` is a dict of yuv_layout() fields (y_pitch, uv_pitch,
        u_offset, v_offset, frame_stride) describing e.g. a padded decoder surface; by default cv2's contiguous
        layout.  ``pitch`` and ``frame_stride`` describe BGR frames only.  ``dev_scores_ptr``: device float64 [n,21]
        that also receives every joint's score, in stream order."""
        ids, t2d, t3d = self._meta(n, stream_ids, t2d, t3d)
        sc = C.c_void_p(dev_scores_ptr) if dev_scores_ptr else None
        if pixel_format != "bgr":
            if pitch is not None or frame_stride is not None:
                raise ValueError("YUV frames are described by `layout`, not by pitch / frame_stride")
            lay = yuv_layout(pixel_format, h, w, **(layout or {}))
            self._request_scores(sc)
            self._check(self._lib.vnect_estimate_device_yuv(self._h, C.c_void_p(dev_frames_ptr), n, h, w, C.byref(lay),
                                                            _ptr(ids), _ptr(t2d), _ptr(t3d), C.c_void_p(dev_j2_ptr),
                                                            C.c_void_p(dev_j3_ptr)))
            return
        pitch = pitch or w * 3
        frame_stride = frame_stride or pitch * h
        self._request_scores(sc)
        self._check(self._lib.vnect_estimate_device(self._h, C.c_void_p(dev_frames_ptr), n, h, w, pitch, frame_stride,
                                                    _ptr(ids), _ptr(t2d), _ptr(t3d), C.c_void_p(dev_j2_ptr),
                                                    C.c_void_p(dev_j3_ptr)))

    def preprocess(self, frames):
        """gen_input_batch (src/estimator.py:70-81) -> (batch f32 [n*n_scales,S,S,3], scaler, [offset_x, offset_y])."""
        frames, st = self._frames(frames)
        n, h, w = frames.shape[:3]
        s = self.box_size
        out = np.empty((n * len(self.scales), s, s, 3), np.float32)
        meta = np.zeros(3, np.float64)
        self._check(self._lib.vnect_preprocess(self._h, _ptr(frames), n, h, w, st[1], st[0] if n > 1 else st[1] * h,
                                               _ptr(out), _ptr(meta)))
        return out, float(meta[0]), [int(meta[1]), int(meta[2])]

    def postprocess(self, maps, scaler=1.0, offsets=(0, 0), stream_ids=None, t2d=None, t3d=None, scores=False):
        """src/estimator.py:105-142 on given (hm, xm, ym, zm) maps, each [n*n_scales, S/8, S/8, 21] float32.
        Returns (joints_2d, joints_3d, raw_argmax) (+ scores, as in estimate())."""
        maps, n = check_maps(maps, len(self.scales), self.hm_size)
        ids, t2d, t3d = self._meta(n, stream_ids, t2d, t3d)
        j2, j3 = np.empty((n, JOINTS, 2), np.float64), np.empty((n, JOINTS, 3), np.float32)
        raw = np.empty((n, JOINTS, 2), np.int32)
        sc = self._scores_out(scores, n)
        self._request_scores(None if sc is None else _ptr(sc))
        self._check(self._lib.vnect_postprocess(self._h, *[_ptr(m) for m in maps], n, _ptr(ids), _ptr(t2d), _ptr(t3d),
                                                float(scaler), int(offsets[0]), int(offsets[1]), _ptr(j2), _ptr(j3),
                                                _ptr(raw)))
        return (j2, j3, raw) if sc is None else (j2, j3, raw, sc)

    def postprocess_sequence(self, maps, scaler=1.0, offsets=(0, 0), stream_ids=None, t2d=None, t3d=None,
                             scores=False):
        """postprocess() for a sequence call (see estimate_sequence) on given maps.  Returns (joints_2d, joints_3d,
        raw_argmax) (+ scores, as in estimate())."""
        maps, n = check_maps(maps, len(self.scales), self.hm_size)
        ids, t2d, t3d = self._sequence_meta(n, stream_ids, t2d, t3d)
        j2, j3 = np.empty((n, JOINTS, 2), np.float64), np.empty((n, JOINTS, 3), np.float32)
        raw = np.empty((n, JOINTS, 2), np.int32)
        sc = self._scores_out(scores, n)
        self._request_scores(None if sc is None else _ptr(sc))
        self._check(self._lib.vnect_postprocess_sequence(self._h, *[_ptr(m) for m in maps], n, _ptr(ids), _ptr(t2d),
                                                         _ptr(t3d), float(scaler), int(offsets[0]), int(offsets[1]),
                                                         _ptr(j2), _ptr(j3), _ptr(raw)))
        return (j2, j3, raw) if sc is None else (j2, j3, raw, sc)

    def track_postprocess(self, maps, frame_hw, stream_ids=None, t2d=None, t3d=None, scores=False):
        """The tracked tail of track_frames() on given (hm, xm, ym, zm) maps, each [n*n_scales, S/8, S/8, 21] float32:
        frame f of stream stream_ids[f] is a full frame of frame_hw[f] = (height, width), cropped by the stream's box.
        Returns (joints_2d [n,21,2] in full-frame pixels, joints_3d [n,21,3], boxes_used [n,4]); the box update runs on
        the device as in track_frames().  The raw argmax comes from raw_argmax()."""
        maps, n = check_maps(maps, len(self.scales), self.hm_size)
        hw = np.ascontiguousarray(frame_hw, dtype=np.int32).reshape(-1)
        if hw.shape != (2 * n,):
            raise ValueError(f"frame_hw must give (height, width) for each of the {n} frames")
        ids, t2d, t3d = self._meta(n, stream_ids, t2d, t3d)
        j2, j3 = np.empty((n, JOINTS, 2), np.float64), np.empty((n, JOINTS, 3), np.float32)
        boxes = np.empty((n, 4), np.int32)
        sc = self._scores_out(scores, n)
        self._request_scores(None if sc is None else _ptr(sc))
        self._check(self._lib.vnect_track_postprocess(self._h, *[_ptr(m) for m in maps], n, _ptr(hw), _ptr(ids),
                                                      _ptr(t2d), _ptr(t3d), _ptr(j2), _ptr(j3), _ptr(boxes)))
        return (j2, j3, boxes) if sc is None else (j2, j3, boxes, sc)

    def maps(self, n_frames=1):
        """The CNN output maps of the first n_frames frames of the last call (all their scales) as the 4-tuple
        (hm, xm, ym, zm) of NHWC [n_frames*n_scales, S/8, S/8, 21] float32 arrays that postprocess() takes."""
        dims = (C.c_int32 * 4)()
        self._check(self._lib.vnect_get_maps(self._h, int(n_frames), None, 0, dims))
        out = np.empty(tuple(dims), np.float32)
        self._check(self._lib.vnect_get_maps(self._h, int(n_frames), _ptr(out), out.size, dims))
        return planar_to_nhwc(out)

    def filter(self, values, dim, t, stream_id=0, is_f32=None):
        """One joint_filter step (src/estimator.py:83-95) on explicit values [21, dim].  ``is_f32`` says whether the
        caller's array is float32 like the reference's joints_3d (default: dim == 3); the result is float64-typed
        either way and float32-valued when it is."""
        is_f32 = (dim == 3) if is_f32 is None else bool(is_f32)
        v = np.ascontiguousarray(values, dtype=np.float64).reshape(-1).copy()
        if v.size != JOINTS * dim:
            raise ValueError(f"expected [21, {dim}] values")
        self._check(self._lib.vnect_filter(self._h, int(stream_id), int(dim), 1 if is_f32 else 0, float(t), _ptr(v)))
        return v.reshape(JOINTS, dim)

    def joints2angles(self, joints_3d, stream_ids=None, t=None):
        """src/joints2angles.py:60-110 for n frames: [n,21,3] float32 -> [n,8] float64 radians, one-euro filtered per
        stream when clock readings ``t`` are given."""
        j = np.ascontiguousarray(joints_3d, dtype=np.float32)
        if j.ndim == 2:
            j = j[None]
        n = j.shape[0]
        ids = np.arange(n, dtype=np.int32) if stream_ids is None else np.ascontiguousarray(stream_ids, dtype=np.int32)
        tt = None if t is None else np.ascontiguousarray(np.broadcast_to(np.asarray(t, dtype=np.float64), (n,)))
        out = np.empty((n, 8), np.float64)
        self._check(self._lib.vnect_joints2angles(self._h, _ptr(j), n, _ptr(ids), _ptr(tt) if tt is not None else None,
                                                  _ptr(out)))
        return out

    def raw_argmax(self, n=1):
        """Unfiltered (row, col) argmax in box pixels of the last estimate / submit / track call, int32 [n,21,2]."""
        out = np.empty((n, JOINTS, 2), np.int32)
        self._check(self._lib.vnect_get_raw_argmax(self._h, int(n), _ptr(out)))
        return out

    def export_stream_state(self, stream_id=0):
        """Temporal state of a stream (filters, last clock readings, tracked box) as a float64 vector."""
        out = np.empty(_capi.STREAM_STATE_DOUBLES, np.float64)
        self._check(self._lib.vnect_export_stream_state(self._h, int(stream_id), _ptr(out)))
        return out

    def import_stream_state(self, state, stream_id=0):
        state = np.ascontiguousarray(state, dtype=np.float64)
        if state.shape != (_capi.STREAM_STATE_DOUBLES,):
            raise ValueError("stream state has the wrong size")
        self._check(self._lib.vnect_import_stream_state(self._h, int(stream_id), _ptr(state)))

    def tap(self, name, n=1):
        """Intermediate activation `name` of the last forward as float32 NHWC (fp16 on the device)."""
        dims = (C.c_int32 * 4)()
        self._check(self._lib.vnect_get_tap(self._h, name.encode(), n, None, 0, dims))
        out = np.empty(tuple(dims), np.float32)
        self._check(self._lib.vnect_get_tap(self._h, name.encode(), n, _ptr(out), out.size, dims))
        return out

    def stem_input(self, n=1):
        """The network input of the first n forwards of the last call as the stem reads it: the raw fp16 bits, uint16
        [n, 2 parities, S/2 + 3, (S + 6) * 4], zero border and 4th channel included."""
        dims = (C.c_int32 * 4)()
        self._check(self._lib.vnect_get_input(self._h, int(n), None, 0, dims))
        out = np.empty(tuple(dims), np.uint16)
        self._check(self._lib.vnect_get_input(self._h, int(n), _ptr(out), out.size, dims))
        return out

    def check_finite(self, n=1):
        """{launch name: count of NaN / Inf / saturated fp16 values in its output} for the first n forwards of the last
        batch -- names the layer where un-normalised weights overflow fp16 (65504)."""
        names = self.step_names()
        counts = np.zeros(len(names), np.int64)
        self._check(self._lib.vnect_check_finite(self._h, int(n), _ptr(counts)))
        return dict(zip(names, counts.tolist()))

    def reset(self, stream_id=-1):
        self._check(self._lib.vnect_reset_stream(self._h, int(stream_id)))

    def set_cuda_stream(self, stream_ptr):
        self._check(self._lib.vnect_set_stream(self._h, C.c_void_p(stream_ptr)))

    def set_packed_results(self, dev_ptr):
        """Device pointer to float64 [max_frames,21,5]: later calls also write (row, col, x, y, z) there (0 = off)."""
        self._check(self._lib.vnect_set_packed_results(self._h, C.c_void_p(dev_ptr) if dev_ptr else None))

    def synchronize(self):
        self._check(self._lib.vnect_synchronize(self._h))

    def launch_count(self):
        return int(self._lib.vnect_launch_count(self._h))

    def info(self, key):
        return float(self._lib.vnect_info(self._h, key.encode()))

    def step_names(self):
        out, i = [], 0
        while True:
            s = self._lib.vnect_step_name(self._h, i)
            if s is None:
                return out
            out.append(s.decode())
            i += 1

    _CONV_PATH_FIELDS = ("block_n", "epi", "cg", "b_resident", "halo", "im2col", "mode", "n2", "tw", "th", "H", "W")

    def step_paths(self):
        """How each launch of one forward runs (vnect_step_path), in step_names() order: {"kind": "stem", "cg", "n_xt"}
        for conv1+pool1, {"kind": "conv", block_n, epi, cg, b_resident, halo, im2col, mode, n2, tw, th, H, W} for the
        implicit-GEMM convs."""
        out = []
        for i, name in enumerate(self.step_names()):
            v = (C.c_int32 * 12)()
            self._check(self._lib.vnect_step_path(self._h, i, v))
            if name == "conv1+pool1":
                out.append({"kind": "stem", "cg": v[0], "n_xt": v[1]})
            else:
                out.append({"kind": "conv", **dict(zip(self._CONV_PATH_FIELDS, v))})
        return out

    def time_forward(self, n, reps=5, per_layer=False):
        """Device time (ms) of one forward of n images already resident; optionally per launch."""
        total = C.c_float()
        names = self.step_names()
        per = np.zeros(len(names), np.float32) if per_layer else None
        self._check(self._lib.vnect_time_forward(self._h, n, reps, C.byref(total), _ptr(per) if per_layer else None))
        return (total.value, dict(zip(names, per.tolist()))) if per_layer else total.value


    def time_prepost(self, n_frames, reps=10):
        """Device time (ms) of the pre-processing kernels and of the post-process kernel for n_frames box-size frames."""
        pre, post = C.c_float(), C.c_float()
        self._check(self._lib.vnect_time_prepost(self._h, int(n_frames), int(reps), C.byref(pre), C.byref(post)))
        return pre.value, post.value


class VNectEstimator:
    """Drop-in for the reference ``VNectEstimator`` (src/estimator.py:16-142).

    ``VNectEstimator()`` then ``joints_2d, joints_3d = estimator(img_bgr)``: ``joints_2d`` float64 [21,2] (row, col) in
    input-image pixels, ``joints_3d`` float32 [21,3] in mm relative to joint 14; fresh writable host arrays each call.
    Optional keyword arguments (all absent in the reference) choose weights, scales, clock and device.
    """

    box_size = 368  # src/estimator.py:19
    hm_factor = 8  # :21
    joints_sum = 21  # :23
    joint_parents = [16, 15, 1, 2, 3, 1, 5, 6, 14, 8, 9, 14, 11, 12, 14, 14, 1, 4, 7, 10, 13]  # :25

    # Largest frame the device context is sized for up front.  The reference's video loop hands in a crop whose size
    # changes every frame (run_estimator.py:100, 110-119), so sizing by the first frame would rebuild mid-video.
    default_max_input = (1080, 1920)

    def __init__(self, weights=None, scales=None, box_size=None, device=0, clock=None, verbose=True, max_input=None):
        self._verbose = verbose
        if verbose:
            print('Initializing VNect Estimator...')
        self.scales = [1, 0.85, 0.7] if scales is None else list(scales)  # src/estimator.py:32
        if box_size is not None:
            self.box_size = int(box_size)
        self._weights = _weights.resolve(weights)
        self._device = device
        self._clock = clock or time.time
        self._engine = None
        self._engine_key = None
        self._max_input = tuple(max_input) if max_input else self.default_max_input
        self._ensure_engine((self.box_size, self.box_size))
        if verbose:
            print('VNect Estimator initialized.')

    def _ensure_engine(self, hw):
        """(Re)build the device context when `scales` was changed by the caller (the reference reads self.scales on
        every call, src/estimator.py:99) or a frame larger than `max_input` arrives.  The OneEuroFilter state belongs
        to the estimator object in the reference (src/estimator.py:46-53) and survives both: it is carried over."""
        need_h = max(hw[0], self.box_size, self._max_input[0])
        need_w = max(hw[1], self.box_size, self._max_input[1])
        key = (tuple(float(s) for s in self.scales), self.box_size)
        if self._engine is not None and key == self._engine_key and need_h <= self._engine.max_input[0] \
                and need_w <= self._engine.max_input[1]:
            return
        state = None
        if self._engine is not None:
            need_h = max(need_h, self._engine.max_input[0])
            need_w = max(need_w, self._engine.max_input[1])
            state = self._engine.export_stream_state(0)
            self._engine.close()
        self._max_input = (need_h, need_w)
        self._engine = VNectEngine(self._weights, self.scales, self.box_size, max_frames=1, max_streams=1,
                                   max_input=(need_h, need_w), device=self._device, filters=True)
        if state is not None:
            self._engine.import_stream_state(state, 0)
        self._engine_key = key

    @staticmethod
    def gen_input_batch(img_input, box_size, scales):
        """src/estimator.py:70-81; computed by the CUDA preprocessing kernels (values are the fp16 network input)."""
        img = np.asarray(img_input)
        eng = VNectEngine(False, scales, box_size, max_frames=1, max_input=(max(img.shape[0], box_size),
                                                                           max(img.shape[1], box_size)))
        try:
            return eng.preprocess(img)
        finally:
            eng.close()

    def joint_filter(self, joints, dim=2):
        """src/estimator.py:83-95: in-place one-euro filtering of [21, dim] joints at the current clock reading.  A
        float32 array (the reference's joints_3d) is filtered with float32 raw differences and float32 results, a
        float64 one (joints_2d) in float64."""
        is_f32 = getattr(joints, "dtype", None) == np.float32
        joints[...] = self._engine.filter(joints, dim, self._clock(), is_f32=is_f32)
        return joints

    def __call__(self, img_input):
        t0 = time.time()
        img = np.asarray(img_input)
        self._ensure_engine(img.shape[:2])
        # The reference reads the clock once per filter group, AFTER its sess.run (src/estimator.py:84, 132-135).  Here
        # pre-processing, CNN and post-processing are one device submission, so both readings are taken just before
        # it: every reading is earlier by about the CNN latency, the differences between frames -- all the filters
        # use -- are unchanged.
        t2d = self._clock()
        t3d = self._clock()
        j2, j3 = self._engine.estimate(img, stream_ids=[0], t2d=[t2d], t3d=[t3d])
        joints_2d, joints_3d = j2[0].copy(), j3[0].copy()
        if self._verbose:
            print('FPS: {:>2.2f}'.format(1 / (time.time() - t0)))
        return joints_2d, joints_3d


class Joints2Angles:
    """Drop-in for the reference class (src/joints2angles.py:23-57): ``angles = Joints2Angles()(joints_3d)`` returns the
    list [s0_l, s1_l, e0_l, e1_l, s0_r, s1_r, e0_r, e1_r] in radians and prints them, computed (and one-euro filtered) on
    the device.  ``engine`` may be shared with an estimator; otherwise a small CNN-less context is created."""

    def __init__(self, filter=True, engine=None, clock=None, verbose=True):
        if verbose:
            print('Initializing Joints2Angles...')
        self.filter = filter
        self._engine = engine or VNectEngine(False, [1.0], max_frames=1, max_streams=1)
        self._clock = clock or time.time
        self._verbose = verbose
        if verbose:
            print('Joints2Angles initialized.')

    def __call__(self, joints_3d):
        t = [self._clock()] if self.filter else None
        angles = [float(a) for a in self._engine.joints2angles(np.asarray(joints_3d)[None], [0], t)[0]]
        if self._verbose:
            print('%5.2f | %5.2f | %5.2f | %5.2f | %5.2f | %5.2f | %5.2f | %5.2f' % tuple(angles))
        return angles

    @staticmethod
    def joints2angles(joints_3d, engine=None):
        eng = engine or VNectEngine(False, [1.0], max_frames=1, max_streams=1)
        try:
            return tuple(float(a) for a in eng.joints2angles(np.asarray(joints_3d)[None])[0])
        finally:
            if engine is None:
                eng.close()
