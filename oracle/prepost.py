"""CPU restatement of the estimator's pre- and post-processing (reference: src/estimator.py:70-142,
src/utils.py:13-21,58-219, src/OneEuroFilter.py:13-75).

TEST INFRASTRUCTURE (see oracle/__init__.py).

The reference does its image arithmetic with OpenCV (``cv2.resize``) and numpy; both exist in this image, so the
oracle calls them exactly where the reference does.  Beside that it carries *restatements* of the OpenCV arithmetic
(SURVEY.md App. C) that the CUDA kernels follow, pinned against cv2 by tests/test_oracle_prepost.py:

* ``resize_u8_int``      -- 8-bit INTER_LINEAR: 11-bit fixed-point coefficients, x indices clamped with f reset,
  y indices clamped without reset, vertical pass ``(((b0*(T0>>4))>>16) + ((b1*(T1>>4))>>16) + 2) >> 2``.
* ``resize_f32_np``      -- float32 INTER_LINEAR: ``S0*(1-f) + S1*f`` per axis, separate multiplies and add (no FMA).
* ``upsample8_f64_point``-- float64 x8 upsample as OpenCV+IPP computes it here: ``fma(S1-S0, f, S0)`` per axis
  (found by exhaustive comparison against cv2 4.13.0; evaluated exactly with rationals, point-wise, for tests).
"""
import math
import time
from fractions import Fraction

import cv2
import numpy as np

BOX_SIZE = 368
HM_FACTOR = 8
JOINTS = 21
ROOT_JOINT = 14
FILTER_2D = dict(freq=30, mincutoff=1.7, beta=0.3, dcutoff=0.4)  # estimator.py:34-39
FILTER_3D = dict(freq=30, mincutoff=0.8, beta=0.4, dcutoff=0.4)  # estimator.py:40-45


# ----------------------------------------------------------------------------------------------------------------
# OpenCV arithmetic, restated
def cv_round(x):
    """cvRound: round half to even."""
    return int(np.rint(x))


def linear_coords(dst, src, inv_scale, reset_f):
    """Source index / fraction of every destination index (SURVEY.md App. C.1): f is computed in double, stored as
    float32; the x axis clamps the index AND zeroes f, the y axis leaves f alone (rows are clamped when read)."""
    d = np.arange(dst, dtype=np.float64)
    f = ((d + 0.5) * inv_scale - 0.5).astype(np.float32)
    i = np.floor(f).astype(np.int64)
    f = (f - i.astype(np.float32)).astype(np.float32)
    if reset_f:
        lo = i < 0
        f[lo] = 0
        i[lo] = 0
        hi = i >= src - 1
        f[hi] = 0
        i[hi] = src - 1
    return i, f


def resize_u8_int(img, fx, fy):
    """Integer restatement of cv2.resize(u8, (0,0), fx, fy, INTER_LINEAR); bit-exact (utils.py:13-21 call site)."""
    h, w = img.shape[:2]
    dw, dh = cv_round(w * fx), cv_round(h * fy)
    if (dh, dw) == (h, w):  # cv::resize copies when dsize == ssize, whatever fx and fy are
        return img.copy()
    ix, ffx = linear_coords(dw, w, 1.0 / fx, True)
    iy, ffy = linear_coords(dh, h, 1.0 / fy, False)
    one, sc = np.float32(1), np.float32(2048)
    a0 = np.rint((one - ffx) * sc).astype(np.int32)
    a1 = np.rint(ffx * sc).astype(np.int32)
    b0 = np.rint((one - ffy) * sc).astype(np.int32)
    b1 = np.rint(ffy * sc).astype(np.int32)
    ix1 = np.minimum(ix + 1, w - 1)
    s = img.astype(np.int32)
    t = s[:, ix] * a0[None, :, None] + s[:, ix1] * a1[None, :, None]
    y0 = np.clip(iy, 0, h - 1)
    y1 = np.clip(iy + 1, 0, h - 1)
    out = (((b0[:, None, None] * (t[y0] >> 4)) >> 16) + ((b1[:, None, None] * (t[y1] >> 4)) >> 16) + 2) >> 2
    return out.astype(np.uint8)


def resize_f32_np(img, fx, fy):
    """float32 INTER_LINEAR restatement (bit-exact vs cv2 4.13.0 on [h,w,21] maps; estimator.py:111-116 call site)."""
    assert img.dtype == np.float32
    h, w = img.shape[:2]
    dw, dh = cv_round(w * fx), cv_round(h * fy)
    if (dh, dw) == (h, w):  # cv::resize copies when dsize == ssize (a scale s > hs / (hs + 0.5) of a heat-map)
        return img.copy()
    ix, ffx = linear_coords(dw, w, 1.0 / fx, True)
    iy, ffy = linear_coords(dh, h, 1.0 / fy, False)
    ix1 = np.minimum(ix + 1, w - 1)
    a0 = (np.float32(1) - ffx)[None, :, None]
    a1 = ffx[None, :, None]
    t = img[:, ix] * a0 + img[:, ix1] * a1
    y0 = np.clip(iy, 0, h - 1)
    y1 = np.clip(iy + 1, 0, h - 1)
    b0 = (np.float32(1) - ffy)[:, None, None]
    b1 = ffy[:, None, None]
    return t[y0] * b0 + t[y1] * b1


def area2x_u8(img):
    """cv2.resize(u8, fx=fy=0.5, INTER_LINEAR) == INTER_AREA with scale 2 (resizeAreaFast): full 2x2 blocks are
    (sum + 2) >> 2; a partial last block (odd source side, dsize = cvRound(side / 2)) averages its in-range pixels as
    saturate_cast<uchar>(float(sum) / count).  Restated for squarify_kernel mode 1; pinned against cv2 by
    tests/test_oracle_prepost.py."""
    h, w = img.shape[:2]
    dw, dh = cv_round(w * 0.5), cv_round(h * 0.5)
    s = img.astype(np.int32)
    out = np.zeros((dh, dw, img.shape[2]), np.uint8)
    for dy in range(dh):
        ys = [y for y in (2 * dy, 2 * dy + 1) if y < h]
        for dx in range(dw):
            xs = [x for x in (2 * dx, 2 * dx + 1) if x < w]
            tot = sum(s[y, x] for y in ys for x in xs)
            if len(ys) == 2 and len(xs) == 2:
                out[dy, dx] = (tot + 2) >> 2
            else:
                out[dy, dx] = np.rint(tot.astype(np.float32) / np.float32(len(ys) * len(xs))).astype(np.uint8)
    return out


def _fma(a, b, c):
    return float(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def upsample8_f64_point(hm, dy, dx, factor=HM_FACTOR):
    """Value of cv2.resize(hm_f64, fx=fy=8, INTER_LINEAR)[dy, dx] as computed by OpenCV 4.13 + IPP: horizontal
    ``fma(S1 - S0, fx, S0)`` on the two source rows, then vertical ``fma(H1 - H0, fy, H0)`` (utils.py:169-171)."""
    h, w = hm.shape
    ix, ffx = linear_coords(w * factor, w, 1.0 / factor, True)
    iy, ffy = linear_coords(h * factor, h, 1.0 / factor, False)
    x0, x1 = ix[dx], min(ix[dx] + 1, w - 1)
    y0, y1 = int(np.clip(iy[dy], 0, h - 1)), int(np.clip(iy[dy] + 1, 0, h - 1))
    h0 = _fma(np.float64(hm[y0, x1]) - np.float64(hm[y0, x0]), ffx[dx], hm[y0, x0])
    h1 = _fma(np.float64(hm[y1, x1]) - np.float64(hm[y1, x0]), ffx[dx], hm[y1, x0])
    return _fma(np.float64(h1) - np.float64(h0), ffy[dy], h0)


# ----------------------------------------------------------------------------------------------------------------
# utils.py / estimator.py, restated (cv2 + numpy called exactly where the reference calls them)
def img_scale(img, scale):
    """utils.py:13-21"""
    return cv2.resize(img, (0, 0), fx=scale, fy=scale, interpolation=cv2.INTER_LINEAR)


def img_scale_squarify(img, box_size):
    """utils.py:82-120: scale the longer side to box_size, centre on black."""
    h, w = img.shape[:2]
    scaler = box_size / max(h, w)
    scaled = img_scale(img, scaler)
    sh, sw = scaled.shape[:2]
    out = np.zeros((box_size, box_size, 3), np.uint8)
    ox = oy = 0
    if sh > sw:
        ox = box_size // 2 - sw // 2
        out[:, ox:box_size // 2 + int(np.ceil(sw / 2)), :] = scaled
    else:
        oy = box_size // 2 - sh // 2
        out[oy:box_size // 2 + int(np.ceil(sh / 2)), :, :] = scaled
    return out, scaler, [ox, oy]


def img_scale_padding(img, scale, box_size):
    """utils.py:123-150: shrink the square box image, zero-pad back (floor(pad/2) before, the rest after)."""
    scaled = img_scale(img, scale)
    ph = (box_size - scaled.shape[0]) // 2
    pw = (box_size - scaled.shape[1]) // 2
    pho = (box_size - scaled.shape[0]) % 2
    pwo = (box_size - scaled.shape[1]) % 2
    return np.pad(scaled, ((pw, pw + pwo), (ph, ph + pho), (0, 0)), mode="constant", constant_values=0)


def gen_input_batch(img, box_size, scales):
    """estimator.py:70-81"""
    sq, scaler, offs = img_scale_squarify(img, box_size)
    batch = [img_scale_padding(sq, s, box_size) if s < 1 else sq for s in scales]
    return np.asarray(batch, dtype=np.float32) / 255 - 0.4, scaler, offs


def average_scales(maps, scales, box_size=BOX_SIZE, hm_factor=HM_FACTOR):
    """estimator.py:105-129: per-scale resize by 1/s, centre crop, float64 mean.  maps = (hm, xm, ym, zm)."""
    hs = box_size // hm_factor
    avgs = [np.zeros((hs, hs, JOINTS)) for _ in range(4)]
    for i, s in enumerate(scales):
        rescale = 1.0 / s
        for a, m in zip(avgs, maps):
            sm = img_scale(m[i], rescale)
            mid = [sm.shape[0] // 2, sm.shape[1] // 2]
            a += sm[mid[0] - hs // 2:mid[0] + hs // 2, mid[1] - hs // 2:mid[1] + hs // 2, :]
    for a in avgs:
        a /= len(scales)
    return avgs


def extract_2d_joints(hm_avg, box_size=BOX_SIZE, hm_factor=HM_FACTOR):
    """utils.py:153-175: x8 upsample of each float64 heat-map, first-maximum argmax -> (row, col)."""
    out = np.zeros((hm_avg.shape[2], 2))
    for j in range(hm_avg.shape[2]):
        up = cv2.resize(hm_avg[:, :, j], (0, 0), fx=hm_factor, fy=hm_factor, interpolation=cv2.INTER_LINEAR)
        out[j, :] = np.unravel_index(np.argmax(up), (box_size, box_size))
    return out


def hm_pt_interp_bilinear(src, scale, point):
    """utils.py:58-79 (weights are not clamped: extrapolates below 3.5 px, returns exactly 0 at the far border)."""
    sh, sw = src.shape
    dy, dx = point
    sx = (dx + 0.5) / scale - 0.5
    sy = (dy + 0.5) / scale - 0.5
    x0, y0 = int(sx), int(sy)
    x1, y1 = min(x0 + 1, sw - 1), min(y0 + 1, sh - 1)
    v0 = (x1 - sx) * src[y0, x0] + (sx - x0) * src[y0, x1]
    v1 = (x1 - sx) * src[y1, x0] + (sx - x0) * src[y1, x1]
    return (y1 - sy) * v0 + (sy - y0) * v1


def extract_3d_joints(joints_2d, xm, ym, zm, hm_factor=HM_FACTOR):
    """utils.py:178-219: sample the location maps at the (filtered) 2D joints, x100 -> mm, root-relative (joint 14)."""
    out = np.zeros((xm.shape[2], 3), dtype=np.float32)
    for j in range(xm.shape[2]):
        y2, x2 = joints_2d[j][:]
        out[j, :] = [hm_pt_interp_bilinear(m[:, :, j], hm_factor, (y2, x2)) * 100 for m in (xm, ym, zm)]
    out -= out[ROOT_JOINT, :].copy()
    return out


# ----------------------------------------------------------------------------------------------------------------
# OneEuroFilter.py:13-75, restated
class _LowPass:
    def __init__(self):
        self.y = None  # last raw value
        self.s = None  # last smoothed value

    def __call__(self, value, alpha):
        alpha = float(alpha)
        if alpha <= 0 or alpha > 1.0:
            raise ValueError("alpha (%s) should be in (0.0, 1.0]" % alpha)  # OneEuroFilter.py:21-22
        s = value if self.y is None else alpha * value + (1.0 - alpha) * self.s
        self.y = value
        self.s = s
        return s


class OneEuroFilter:
    """Scalar 1-euro filter with the reference's exact control flow (timestamp truthiness test included)."""

    def __init__(self, freq, mincutoff=1.0, beta=0.0, dcutoff=1.0):
        if freq <= 0:
            raise ValueError("freq should be >0")
        if mincutoff <= 0:
            raise ValueError("mincutoff should be >0")
        if dcutoff <= 0:
            raise ValueError("dcutoff should be >0")
        self.freq, self.mincutoff, self.beta, self.dcutoff = float(freq), float(mincutoff), float(beta), float(dcutoff)
        self.x, self.dx = _LowPass(), _LowPass()
        self.lasttime = None

    def alpha(self, cutoff):
        te = 1.0 / self.freq
        tau = 1.0 / (2 * math.pi * cutoff)
        return 1.0 / (1.0 + tau / te)

    def __call__(self, x, timestamp=None):
        if self.lasttime and timestamp:
            self.freq = 1.0 / (timestamp - self.lasttime)  # ZeroDivisionError on a repeated timestamp
        self.lasttime = timestamp
        prev = self.x.y
        dx = 0.0 if prev is None else (x - prev) * self.freq
        edx = self.dx(dx, self.alpha(self.dcutoff))
        cutoff = self.mincutoff + self.beta * math.fabs(edx)
        return self.x(x, self.alpha(cutoff))


class OracleEstimator:
    """Restatement of VNectEstimator (estimator.py:16-142) around an injected forward function and clock.

    ``forward(batch_nhwc_f32) -> (hm, xm, ym, zm)``.  ``promotion``: 'numpy' lets the 3D filter run on numpy float32
    scalars exactly like the reference does under the installed numpy (NEP 50 keeps them float32 on numpy >= 2);
    'legacy' restates numpy 1.x value-based casting, the behaviour the TF1-era reference ran with: the raw
    difference ``x - x_prev`` is float32, everything after it float64.  The CUDA path implements 'legacy'.
    """

    box_size = BOX_SIZE
    hm_factor = HM_FACTOR
    joints_sum = JOINTS

    def __init__(self, forward, scales=(1, 0.85, 0.7), clock=time.time, promotion="legacy", box_size=BOX_SIZE):
        self.forward = forward
        self.scales = list(scales)
        self.clock = clock
        self.promotion = promotion
        self.box_size = box_size
        self.filter_2d = [(OneEuroFilter(**FILTER_2D), OneEuroFilter(**FILTER_2D)) for _ in range(JOINTS)]
        self.filter_3d = [tuple(OneEuroFilter(**FILTER_3D) for _ in range(3)) for _ in range(JOINTS)]
        self.last = {}

    def joint_filter(self, joints, dim=2):
        t = self.clock()
        filt = self.filter_2d if dim == 2 else self.filter_3d
        for i in range(JOINTS):
            for c in range(dim):
                if dim == 3 and self.promotion == "legacy":
                    joints[i, c] = _legacy_f32_filter(filt[i][c], joints[i, c], t)
                else:
                    joints[i, c] = filt[i][c](joints[i, c], t)
        return joints

    def __call__(self, img):
        batch, scaler, (ox, oy) = gen_input_batch(img, self.box_size, self.scales)
        maps = self.forward(batch)
        hm, xm, ym, zm = average_scales(maps, self.scales, self.box_size, self.hm_factor)
        j2 = extract_2d_joints(hm, self.box_size, self.hm_factor)
        raw2 = j2.copy()
        j2 = self.joint_filter(j2, 2)
        j3 = extract_3d_joints(j2, xm, ym, zm, self.hm_factor)
        raw3 = j3.copy()
        j3 = self.joint_filter(j3, 3)
        self.last = dict(batch=batch, maps=maps, hm_avg=hm, xm_avg=xm, ym_avg=ym, zm_avg=zm, joints_2d_raw=raw2,
                         joints_2d_box=j2.copy(), joints_3d_raw=raw3, scaler=scaler, offsets=(ox, oy))
        j2[:, 0] = (j2[:, 0] - oy) / scaler
        j2[:, 1] = (j2[:, 1] - ox) / scaler
        return j2, j3


def _legacy_f32_filter(f, x32, t):
    """One OneEuroFilter step on a float32 sample with numpy-1.x promotion: (x - prev) in float32, rest float64."""
    x32 = np.float32(x32)
    if f.lasttime and t:
        f.freq = 1.0 / (t - f.lasttime)
    f.lasttime = t
    prev = f.x.y
    dx = 0.0 if prev is None else float(np.float32(x32 - np.float32(prev))) * f.freq
    edx = f.dx(dx, f.alpha(f.dcutoff))
    cutoff = f.mincutoff + f.beta * math.fabs(edx)
    alpha = f.alpha(cutoff)
    s = float(x32) if f.x.y is None else alpha * float(x32) + (1.0 - alpha) * f.x.s
    f.x.y = x32
    f.x.s = s
    return s


# ----------------------------------------------------------------------------------------------------------------
# run_estimator.py:98-119, restated: crop by the tracked box, estimate, shift to frame coordinates, update the box
def tracker_update(joints_2d, w_img, h_img):
    """run_estimator.py:110-119: next crop box (x, y, w, h) from this frame's full-frame 2D joints."""
    y_min = np.min(joints_2d[:, 0])
    y_max = np.max(joints_2d[:, 0])
    x_min = np.min(joints_2d[:, 1])
    x_max = np.max(joints_2d[:, 1])
    buffer_x = 0.8 * (x_max - x_min + 1)
    buffer_y = 0.2 * (y_max - y_min + 1)
    x, y = (max(int(x_min - buffer_x / 2), 0), max(int(y_min - buffer_y / 2), 0))
    w, h = (int(min(x_max - x_min + buffer_x, w_img - x)), int(min(y_max - y_min + buffer_y, h_img - y)))
    return x, y, w, h


class OracleTracker:
    """The reference's video loop body (run_estimator.py:98-119) around an OracleEstimator."""

    def __init__(self, estimator, rect):
        self.estimator = estimator
        self.rect = tuple(int(v) for v in rect)

    def __call__(self, frame):
        h_img, w_img = frame.shape[:2]
        x, y, w, h = self.rect
        # numpy slicing clips to the frame; the CUDA path additionally keeps at least 2 x 2 pixels
        x = min(max(x, 0), w_img - 2)
        y = min(max(y, 0), h_img - 2)
        w = max(min(w, w_img - x), 2)
        h = max(min(h, h_img - y), 2)
        used = (x, y, w, h)
        j2, j3 = self.estimator(np.ascontiguousarray(frame[y:y + h, x:x + w, :]))
        j2[:, 0] += y
        j2[:, 1] += x
        self.rect = tracker_update(j2, w_img, h_img)
        return j2, j3, used


# ----------------------------------------------------------------------------------------------------------------
# joints2angles.py:60-110, restated (numpy called exactly where the reference calls it, so the float32 / float64 mix of
# the intermediate results is the reference's own)
def _cal_angle(v1, v2):
    return np.arccos(np.dot(v1, v2) / (np.linalg.norm(v1) * np.linalg.norm(v2)))


def joints2angles(joints_3d):
    """Eight arm angles (radians): s0_l, s1_l, e0_l, e1_l, s0_r, s1_r, e0_r, e1_r."""
    s2e_l, e2w_l = joints_3d[6] - joints_3d[5], joints_3d[7] - joints_3d[6]
    s2e_r, e2w_r = joints_3d[3] - joints_3d[2], joints_3d[4] - joints_3d[3]
    v1_l = joints_3d[2] - joints_3d[5]
    v1_r = -v1_l
    v2 = [0, 1, 0]
    v3_l, v3_r = np.cross(s2e_l, v2), np.cross(s2e_r, v2)
    v4_l, v4_r = np.cross(s2e_l, e2w_l), np.cross(s2e_r, e2w_r)
    s0_l = np.pi * 3 / 4 - _cal_angle(v1_l, v3_l)
    s1_l = np.pi / 2 - _cal_angle(v2, s2e_l)
    e0_l = -_cal_angle(v3_l, v4_l)
    e1_l = _cal_angle(s2e_l, e2w_l)
    s0_r = np.pi / 4 - _cal_angle(v1_r, v3_r)
    s1_r = np.pi / 2 - _cal_angle(v2, s2e_r)
    e0_r = _cal_angle(v3_r, v4_r)
    e1_r = _cal_angle(s2e_r, e2w_r)
    return s0_l - np.pi / 4, s1_l, e0_l, -e1_l, s0_r + np.pi / 4, -s1_r, e0_r, e1_r


class OracleJoints2Angles:
    """Joints2Angles.__call__ (joints2angles.py:44-57): the eight angles through eight OneEuroFilters (120 Hz, 0.5, 0.5, 1)."""

    def __init__(self, clock=time.time):
        self.clock = clock
        self.filters = [OneEuroFilter(freq=120, mincutoff=0.5, beta=0.5, dcutoff=1.0) for _ in range(8)]

    def __call__(self, joints_3d):
        return [self.filters[i](a, self.clock()) for i, a in enumerate(joints2angles(joints_3d))]
