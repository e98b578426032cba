"""The tracked video loop against the reference, step for step and bit for bit (run_estimator.py:98-119).

One step of a tracked stream crops the full frame by the stream's box (clip_box, make_frame_geom), runs the CNN and the
post-process with that frame's geometry (the `geoms` branch of postprocess_kernel: filter in box pixels, rescale by the
per-frame scaler and offsets, add the crop origin) and updates the box (track_box_update).  The filters and the box
carry state from one step to the next, so a one-ulp difference surfaces steps later, or never.

The reference is oracle.prepost.OracleTracker around an OracleEstimator whose forward returns the maps the device
used, with an injected clock, one per stream.  Every GPU comparison is np.array_equal: joints_2d, joints_3d, the raw
argmax, boxes_used and the box left behind after every step, and every few steps the whole exported stream state.

* Leg A (vnect_track_postprocess on maps built here): the test chooses each joint's heat-map cell, so where the
  joints land -- and which branch of the box update runs -- is fixed by construction.  The scenarios of _streams
  name the branches their streams exist for; the CPU tests run the reference on the same inputs and prove that
  together they reach every branch of BRANCHES, that no scenario can be dropped, and that seven mutated references
  diverge from the true one.
* Leg B (the shipped tracked entry points, W1 weights): after each call the maps the CNN produced (vnect_get_maps) feed
  the reference, so the CNN's fp16 error drops out and the comparison is exact for every step of every stream.
"""
import functools
import math

import cv2
import numpy as np
import pytest

from oracle import prepost
from vnect_b200 import _capi
from vnect_b200.estimator import check_maps, nhwc_to_planar, planar_to_nhwc

# (name, scales, box size): <2, 1> and <2, -1> (the run-time identity mask) both carry the geoms branch
CONFIGS = [("s2_368", [1.0, 0.7], 368), ("s2_alias_448", [0.7, 1.0], 448)]
STEPS = 60
N_STREAMS = 40  # streams of engine A (the migrated stream continues on engine B as MIGRATED_ID)
N_FRAMES = 24   # frames per call: the streams of a call are drawn, in a new order, every step
STATE_EVERY = 6
MIGRATED_ID = 3
HUGE = 1 << 30  # the box of an unseeded or reset stream (vnect_reset_stream), clipped to the frame

# ------------------------------------------------------------------------------------------------ scenarios
# Each stream: (full frame (h, w), seeded box or None, joint pattern, clock, events by own step).
# A stream's events and clock readings are indexed by its own step count, so they hold whichever calls draw it.


def _streams(S):
    hs = S // 8
    tall = (700, 500)  # frames of the narrow crops
    m1 = (2 * S + 64, 2 * S - 100)
    return {
        # plain path with epoch-like clocks: 1.76e9 + k/30 + jitter, 2D and 3D readings apart
        "spread_epoch": [
            ((540, 960), (300, 100, 360, 380), "spread", "epoch", {}),
            ((481, 641), (100, 50, 400, 300), "spread", "epoch", {}),
            ((720, 1280), (500, 200, 300, 500), "spread", "epoch", {}),
        ] + [(hw, (40 + 7 * i, 30 + 5 * i, 200 + 9 * i, 220 + 4 * i), "spread", "epoch", {})
             for i, hw in enumerate([(540, 960), (480, 640), (360, 640), (600, 800), (479, 853), (720, 540)] * 3)],
        # the frame's edges: x and y clamped to 0 at the top-left; w = FW - x and h = FH - y at the bottom-right; tall
        # and wide narrow crops at an edge with the joints in the padded surround (coordinates outside the frame,
        # negative w / h, clip_box holding x at FW - 2 or y at FH - 2); dt of 5 s and of 1e-4 s
        "edges": [
            ((540, 960), (0, 0, 200, 180), "top_left", "plain", {}),
            ((400, 300), (3, 2, 150, 120), "top_left", "plain", {}),
            ((540, 960), (700, 300, 260, 240), "bottom_right", "plain", {}),
            ((333, 517), (300, 180, 217, 153), "bottom_right", "plain", {}),
            (tall, (480, 0, 20, 400), "right_surround", "dt_jumps", {}),
            (tall, (0, 690, 400, 10), "bottom_surround", "dt_jumps", {}),
            ((300, 300), (290, 10, 10, 280), "right_surround", "plain", {}),
        ],
        # every joint on one cell: w = h = int(0.8) = 0, a 2 x 2 box next step; a 2 x 2 full frame; odd sizes;
        # a first clock reading of 0 and t = 0 readings in mid-run (2D in one stream, 3D in another)
        "degenerate": [
            ((540, 960), (400, 200, 120, 160), "one_cell", "zero_first", {}),
            ((2, 2), (0, 0, 2, 2), "spread", "zero_2d_mid", {}),
            ((3, 5), (1, 1, 4, 2), "spread", "zero_3d_mid", {}),
            ((255, 257), (11, 13, 101, 99), "one_cell", "plain", {}),
        ],
        # crops whose longer side is exactly 2S (inverse scale 2: squarify mode 1), and small crops that are enlarged
        "mode1_small": [
            (m1, (7, 5, 2 * S - 300, 2 * S), "spread", "plain", {10: [("set_box", (21, 17, 2 * S, 2 * S - 101))],
                                                                20: [("set_box", (0, 0, 2 * S - 301, 2 * S))]}),
            (m1, (10, 10, 2 * S, 40), "spread", "plain", {}),
            ((540, 960), (100, 100, hs, hs + 7), "spread", "plain", {}),
        ],
        # an unseeded stream; a reset stream restarted with an earlier clock; set_boxes with x >= FW, y >= FH; one
        # stream exported in mid-run and continued on a second engine
        "reset_seed": [
            ((360, 640), None, "spread", "plain", {}),
            ((540, 960), (200, 100, 300, 300), "spread", "plain", {12: [("reset",)]}),
            ((540, 960), (200, 100, 300, 300), "spread", "plain", {8: [("set_box", (1000, 40, 50, 300))]}),
            ((480, 640), (200, 100, 300, 300), "spread", "plain", {9: [("set_box", (30, 500, 400, 60))]}),
            ((540, 960), (250, 60, 400, 420), "spread", "plain", {15: [("migrate",)]}),
        ],
    }


def stream_table(S):
    """[(scenario, frame_hw, seed, pattern, clock, events)] in stream-id order."""
    return [(name, *s) for name, ss in _streams(S).items() for s in ss]


def clock_readings(kind, seed, n=STEPS):
    """(t2, t3) per own step of one stream."""
    rng = np.random.default_rng(seed)
    t2 = 500 + np.cumsum(rng.uniform(0.015, 0.09, n))
    if kind == "epoch":
        t2 = 1.76e9 + np.arange(n) / 30 + rng.uniform(-0.004, 0.004, n)
    t3 = t2 + rng.uniform(0.001, 0.006, n)
    if kind == "dt_jumps":
        d = rng.uniform(0.02, 0.05, n)
        d[5], d[8], d[9], d[20] = 5.0, 1e-4, 1e-4, 5.0
        t2 = 40 + np.cumsum(d)
        t3 = t2 + 2e-5
    elif kind == "zero_first":
        t2[0] = t3[0] = 0.0
    elif kind == "zero_2d_mid":
        t2[[7, 8]] = 0.0
    elif kind == "zero_3d_mid":
        t3[[6, 11]] = 0.0
    return t2, t3


def restart_clock(t2, t3, step):
    """A stream reset at `step` restarts its clock below the readings before the reset."""
    t2, t3 = t2.copy(), t3.copy()
    t2[step:] -= 300.0
    t3[step:] -= 300.0
    return t2, t3


def joint_cells(pattern, hs, rng):
    """[21] (row, col) heat-map cells: where the joints land in box pixels."""
    if pattern == "spread":
        return np.stack([rng.integers(hs // 8, 7 * hs // 8, 21), rng.integers(hs // 4, 3 * hs // 4, 21)], axis=1)
    if pattern == "top_left":
        return rng.integers(0, hs // 4, (21, 2))
    if pattern == "bottom_right":
        return rng.integers(hs // 2, hs, (21, 2))
    if pattern == "one_cell":
        return np.repeat(rng.integers(hs // 4, 3 * hs // 4, (1, 2)), 21, axis=0)
    if pattern == "right_surround":  # rows over the picture, columns right of a narrow crop's picture
        return np.stack([rng.integers(hs // 4, 3 * hs // 4, 21), rng.integers(hs - hs // 6, hs, 21)], axis=1)
    if pattern == "bottom_surround":
        return np.stack([rng.integers(hs - hs // 6, hs, 21), rng.integers(hs // 4, 3 * hs // 4, 21)], axis=1)
    raise ValueError(pattern)


def stream_maps(cfg, sid, step):
    """(hm, xm, ym, zm) of one frame, each [NS, hs, hs, 21] float32: one sharp peak per joint at its cell in the
    identity scale over a weak background, smooth location maps (like oracle.synth)."""
    name, scales, S = cfg
    hs, ns = S // 8, len(scales)
    pattern = stream_table(S)[sid][3] if sid < N_STREAMS else "spread"
    rng = np.random.default_rng([sum(map(ord, name)), sid, step])
    cells = joint_cells(pattern, hs, rng)
    hm = (0.2 * rng.random((ns, hs, hs, 21))).astype(np.float32)
    ident = [i for i, s in enumerate(scales) if s == 1.0][0]
    hm[ident, cells[:, 0], cells[:, 1], np.arange(21)] = np.float32(2.0) + rng.uniform(0, 0.5, 21).astype(np.float32)
    loc = []
    nc = -(-hs // 8)
    for _ in range(3):
        coarse = rng.uniform(-5, 5, size=(ns, nc, nc, 21))
        fine = np.kron(coarse, np.ones((1, 8, 8, 1)))[:, :hs, :hs, :]
        loc.append((fine + 0.05 * rng.standard_normal(fine.shape)).astype(np.float32))
    return (hm, *loc)


# ------------------------------------------------------------------------------------------------ schedule
def schedule(cfg):
    """Per global step: [(stream, own step)] drawn in a new order, N_FRAMES of the live streams; the rest skip."""
    out = []
    for g in range(STEPS):
        order = np.random.default_rng([sum(map(ord, cfg[0])), 1000 + g]).permutation(N_STREAMS)
        out.append([int(s) for s in order[:N_FRAMES]])
    return out


class _Clock:
    def __init__(self):
        self.q = []

    def __call__(self):
        return self.q.pop(0)


class _Stream:
    """The reference side of one stream: its tracker, clock, own step count and host timestamp mirror."""

    def __init__(self, cfg, sid, tracker_cls, estimator_cls):
        name, scales, S = cfg
        self.cfg, self.sid = cfg, sid
        self.scenario, self.hw, self.seed, self.pattern, self.clock_kind, self.events = stream_table(S)[sid]
        self.t2, self.t3 = clock_readings(self.clock_kind, [sum(map(ord, name)), sid])
        for k, evs in self.events.items():
            if ("reset",) in evs:
                self.t2, self.t3 = restart_clock(self.t2, self.t3, k)
        self.tracker_cls, self.estimator_cls = tracker_cls, estimator_cls
        self.frame = np.zeros((*self.hw, 3), np.uint8)  # the forward is injected: only the frame's size matters
        self.k = 0
        self.engine = 0
        self.fresh(self.seed if self.seed is not None else (0, 0, HUGE, HUGE))

    def fresh(self, rect):
        name, scales, S = self.cfg
        self.clock = _Clock()
        est = self.estimator_cls(None, scales, clock=self.clock, promotion="legacy", box_size=S)
        self.tracker = self.tracker_cls(est, rect)
        self.last_t = (math.nan, math.nan)
        self.since_reset = 0

    def step(self, maps):
        """One reference step on the frame's maps -> record."""
        t2, t3 = float(self.t2[self.k]), float(self.t3[self.k])
        self.tracker.estimator.forward = lambda batch, m=maps: m
        self.clock.q = [t2, t3]
        rect_before = self.tracker.rect
        j2, j3, used = self.tracker(self.frame)
        last = self.tracker.estimator.last
        rec = dict(sid=self.sid, k=self.k, t2=t2, t3=t3, last_t=self.last_t, first=self.since_reset == 0,
                   rect_before=rect_before, used=tuple(used), j2=j2, j3=j3, rect=self.tracker.rect,
                   raw=last["joints_2d_raw"].astype(np.int32), hw=self.hw, S=self.cfg[2])
        self.last_t = (t2, t3)
        self.k += 1
        self.since_reset += 1
        return rec


def _events(streams, active):
    """Events of this step's streams, applied before the call: [(stream, event)]."""
    return [(s, ev) for s in (streams[i] for i in active) for ev in s.events.get(s.k, [])]


def run_reference(cfg, tracker_cls=prepost.OracleTracker, estimator_cls=prepost.OracleEstimator, until=None):
    """The reference over the whole schedule -> per global step {"events": [...], "calls": [[record per frame]]}.
    `until(g, records)`: stop early when it returns True (the mutation tests)."""
    streams = [_Stream(cfg, sid, tracker_cls, estimator_cls) for sid in range(N_STREAMS)]
    steps = []
    for g, active in enumerate(schedule(cfg)):
        evs = _events(streams, active)
        for s, ev in evs:
            if ev[0] == "reset":
                s.fresh((0, 0, HUGE, HUGE))
            elif ev[0] == "set_box":
                s.tracker.rect = tuple(ev[1])
            elif ev[0] == "migrate":
                s.engine = 1
        calls = [[], []]
        for sid in active:
            s = streams[sid]
            calls[s.engine].append(s.step(stream_maps(cfg, sid, s.k)))
        steps.append(dict(active=active, events=[(s.sid, ev) for s, ev in evs], calls=calls))
        if until is None and (g % STATE_EVERY == STATE_EVERY - 1 or g == STEPS - 1):
            steps[-1]["states"] = [oracle_state(s) for s in streams]
        if until is not None and until(g, steps[-1]):
            break
    return steps, streams


@functools.lru_cache(maxsize=None)
def reference(cfg_name):
    cfg = [c for c in CONFIGS if c[0] == cfg_name][0]
    return run_reference(cfg)


# ------------------------------------------------------------------------------------------------ branch classifier
BRANCHES = [
    # track_box_update (run_estimator.py:110-119)
    "track_x_clamp0", "track_y_clamp0", "track_w_spread", "track_h_spread", "track_w_frame", "track_h_frame",
    "track_w_lt2", "track_h_lt2", "track_w_neg", "track_h_neg",
    # clip_box: x <= FW - 2, y <= FH - 2, w <= FW - x, h <= FH - y, w, h >= 2 (x, y >= 0 holds for every box the API
    # accepts: the tracker clamps them and set_box refuses negative values)
    "clip_x_hi", "clip_y_hi", "clip_w_cut", "clip_h_cut", "clip_w_min", "clip_h_min",
    # the box of an unseeded or reset stream, (0, 0, 1 << 30, 1 << 30): the whole frame
    "box_reset",
    # make_frame_geom
    "geom_off_x", "geom_off_y", "geom_mode1", "geom_enlarge", "geom_shrink",
    # OneEuroFilter.__call__ (the truthiness test of OneEuroFilter.py:65), per filter group
    "f2_first", "f2_lasttime0", "f2_t0", "f2_freq_update", "f3_first", "f3_lasttime0", "f3_t0", "f3_freq_update",
    # clock regimes of the frequency update
    "clock_epoch", "dt_large", "dt_small",
]


def classify(rec):
    """The branches one step of one stream takes, restated from the kernel's lines (clip_box, make_frame_geom,
    track_box_update) and OneEuroFilter's control flow, on the reference's own values."""
    out = set()
    FH, FW = rec["hw"]
    S = rec["S"]
    x, y, w, h = rec["rect_before"]
    if (x, y, w, h) == (0, 0, HUGE, HUGE):
        out.add("box_reset")
    if x > FW - 2:
        out.add("clip_x_hi")
    if y > FH - 2:
        out.add("clip_y_hi")
    cx, cy = min(max(x, 0), FW - 2), min(max(y, 0), FH - 2)
    if w > FW - cx and FW - cx >= 2:
        out.add("clip_w_cut")
    if h > FH - cy and FH - cy >= 2:
        out.add("clip_h_cut")
    if min(w, FW - cx) < 2:
        out.add("clip_w_min")
    if min(h, FH - cy) < 2:
        out.add("clip_h_min")
    ux, uy, uw, uh = rec["used"]
    assert (ux, uy) == (cx, cy) and uw == max(min(w, FW - cx), 2) and uh == max(min(h, FH - cy), 2)
    scaler = S / max(uh, uw)
    dw, dh = prepost.cv_round(uw * scaler), prepost.cv_round(uh * scaler)
    out.add("geom_off_x" if dh > dw else "geom_off_y")
    if 1.0 / scaler == 2.0:
        out.add("geom_mode1")
    out.add("geom_enlarge" if scaler > 1 else "geom_shrink" if scaler < 1 else "geom_unit")
    j = rec["j2"]
    ymin, ymax, xmin, xmax = j[:, 0].min(), j[:, 0].max(), j[:, 1].min(), j[:, 1].max()
    bx, by = 0.8 * (xmax - xmin + 1), 0.2 * (ymax - ymin + 1)
    nx, ny = int(xmin - bx / 2), int(ymin - by / 2)
    if nx < 0:
        out.add("track_x_clamp0")
    if ny < 0:
        out.add("track_y_clamp0")
    nx, ny = max(nx, 0), max(ny, 0)
    for axis, spread, room in (("w", xmax - xmin + bx, FW - nx), ("h", ymax - ymin + by, FH - ny)):
        v = int(min(spread, room))
        out.add(f"track_{axis}_spread" if spread <= room else f"track_{axis}_frame")
        if v < 0:
            out.add(f"track_{axis}_neg")
        elif v < 2:
            out.add(f"track_{axis}_lt2")
    assert rec["rect"] == (nx, ny, int(min(xmax - xmin + bx, FW - nx)), int(min(ymax - ymin + by, FH - ny)))
    for dim, t, last in (("f2", rec["t2"], rec["last_t"][0]), ("f3", rec["t3"], rec["last_t"][1])):
        if rec["first"]:
            out.add(f"{dim}_first")
            continue
        if last == 0.0:
            out.add(f"{dim}_lasttime0")
        elif t == 0.0:
            out.add(f"{dim}_t0")
        else:
            out.add(f"{dim}_freq_update")
            dt = t - last
            if t > 1e9:
                out.add("clock_epoch")
            if dt >= 1.0:
                out.add("dt_large")
            if dt <= 1e-3:
                out.add("dt_small")
    return out


def scenario_branches(cfg):
    """{scenario: branches its streams take} over the whole reference run of one configuration."""
    steps, streams = reference(cfg[0])
    out = {}
    for st in steps:
        for call in st["calls"]:
            for rec in call:
                out.setdefault(streams[rec["sid"]].scenario, set()).update(classify(rec))
    return out


# ------------------------------------------------------------------------------------------------ mutated references
def _mutant_filter(f, x, t, f32_diff, f64_diff=False, truthy_zero=False):
    """OneEuroFilter step (the 2D float64 one, or the legacy float32 one) with one defect switched on."""
    if (f.lasttime is not None and t is not None) if truthy_zero else (f.lasttime and t):
        f.freq = 1.0 / (t - f.lasttime)
    f.lasttime = t
    prev = f.x.y
    if f32_diff:
        x = np.float32(x)
    if prev is None:
        dx = 0.0
    elif f32_diff and not f64_diff:
        dx = float(np.float32(x - np.float32(prev))) * f.freq
    else:
        dx = (float(x) - float(prev)) * f.freq
    edx = f.dx(dx, f.alpha(f.dcutoff))
    alpha = f.alpha(f.mincutoff + f.beta * math.fabs(edx))
    s = float(x) if prev is None else alpha * float(x) + (1.0 - alpha) * f.x.s
    f.x.y, f.x.s = x, s
    return s


class _TruthyZero(prepost.OracleEstimator):
    """t = 0 taken as a clock reading: the frequency update runs after and at a 0 reading."""

    def joint_filter(self, joints, dim=2):
        t = self.clock()
        filt = self.filter_2d if dim == 2 else self.filter_3d
        for i in range(21):
            for c in range(dim):
                joints[i, c] = _mutant_filter(filt[i][c], joints[i, c], t, dim == 3, truthy_zero=True)
        return joints


class _F64Diff(prepost.OracleEstimator):
    """The 3D filters' raw difference x - x_prev taken in float64 instead of float32."""

    def joint_filter(self, joints, dim=2):
        if dim == 2:
            return super().joint_filter(joints, dim)
        t = self.clock()
        for i in range(21):
            for c in range(3):
                joints[i, c] = _mutant_filter(self.filter_3d[i][c], joints[i, c], t, True, f64_diff=True)
        return joints


class _RescaleFirst(prepost.OracleEstimator):
    """The 2D joints rescaled to input pixels before the filter instead of after it."""

    def __call__(self, img):
        batch, scaler, (ox, oy) = prepost.gen_input_batch(img, self.box_size, self.scales)
        maps = self.forward(batch)
        hm, xm, ym, zm = prepost.average_scales(maps, self.scales, self.box_size, self.hm_factor)
        j2 = prepost.extract_2d_joints(hm, self.box_size, self.hm_factor)
        raw2 = j2.copy()
        j3 = prepost.extract_3d_joints(j2, xm, ym, zm, self.hm_factor)
        j3 = self.joint_filter(j3, 3)
        j2[:, 0] = (j2[:, 0] - oy) / scaler
        j2[:, 1] = (j2[:, 1] - ox) / scaler
        j2 = self.joint_filter(j2, 2)
        self.last = dict(joints_2d_raw=raw2, joints_2d_box=j2.copy(), scaler=scaler, offsets=(ox, oy))
        return j2, j3


class _BoxFromRaw(prepost.OracleTracker):
    """The box updated from the unfiltered joints (rescaled to the frame)."""

    def __call__(self, frame):
        j2, j3, used = super().__call__(frame)
        last = self.estimator.last
        raw = last["joints_2d_raw"].astype(np.float64)
        ox, oy = last["offsets"]
        raw[:, 0] = (raw[:, 0] - oy) / last["scaler"] + used[1]
        raw[:, 1] = (raw[:, 1] - ox) / last["scaler"] + used[0]
        self.rect = prepost.tracker_update(raw, frame.shape[1], frame.shape[0])
        return j2, j3, used


class _BoxFromBoxPixels(prepost.OracleTracker):
    """The box updated from the filtered joints in box pixels (before the rescale and the crop origin)."""

    def __call__(self, frame):
        j2, j3, used = super().__call__(frame)
        self.rect = prepost.tracker_update(self.estimator.last["joints_2d_box"].copy(), frame.shape[1], frame.shape[0])
        return j2, j3, used


class _NoOrigin(prepost.OracleTracker):
    """The crop origin not added to the 2D joints."""

    def __call__(self, frame):
        j2, j3, used = super().__call__(frame)
        j2[:, 0] -= used[1]
        j2[:, 1] -= used[0]
        self.rect = prepost.tracker_update(j2, frame.shape[1], frame.shape[0])
        return j2, j3, used


class _ClipOffByOne(prepost.OracleTracker):
    """clip_box keeping one pixel instead of two: x <= FW - 1, y <= FH - 1, w, h >= 1."""

    def __call__(self, frame):
        h_img, w_img = frame.shape[:2]
        x, y, w, h = self.rect
        x, y = min(max(x, 0), w_img - 1), min(max(y, 0), h_img - 1)
        w, h = max(min(w, w_img - x), 1), max(min(h, h_img - y), 1)
        j2, j3 = self.estimator(np.ascontiguousarray(frame[y:y + h, x:x + w, :]))
        j2[:, 0] += y
        j2[:, 1] += x
        self.rect = prepost.tracker_update(j2, w_img, h_img)
        return j2, j3, (x, y, w, h)


MUTATIONS = {
    "box_from_unfiltered_joints": (_BoxFromRaw, prepost.OracleEstimator),
    "box_from_box_pixel_joints": (_BoxFromBoxPixels, prepost.OracleEstimator),
    "rescale_before_filter": (prepost.OracleTracker, _RescaleFirst),
    "t0_truthy": (prepost.OracleTracker, _TruthyZero),
    "diff_3d_float64": (prepost.OracleTracker, _F64Diff),
    "clip_box_off_by_one": (_ClipOffByOne, prepost.OracleEstimator),
    "crop_origin_not_added": (_NoOrigin, prepost.OracleEstimator),
}


def _records_equal(a, b):
    return (np.array_equal(a["j2"], b["j2"]) and np.array_equal(a["j3"], b["j3"]) and a["used"] == b["used"]
            and tuple(a["rect"]) == tuple(b["rect"]))


# ------------------------------------------------------------------------------------------------ stream state
def oracle_state(s):
    """The exported stream state (VNECT_STREAM_STATE_DOUBLES) of a reference stream: 105 filters x {prev, s_x, s_dx,
    lasttime, freq, has_prev, has_time} (None -> 0 with the flag 0), the last clock readings (NaN: none since the
    reset) and the box."""
    est = s.tracker.estimator
    filters = [f for pair in est.filter_2d for f in pair] + [f for tri in est.filter_3d for f in tri]
    out = []
    for f in filters:
        has_prev, has_time = f.x.y is not None, f.lasttime is not None
        out += [float(f.x.y) if has_prev else 0.0, float(f.x.s) if has_prev else 0.0,
                float(f.dx.s) if f.dx.s is not None else 0.0, float(f.lasttime) if has_time else 0.0, f.freq,
                float(has_prev), float(has_time)]
    out += [s.last_t[0], s.last_t[1], *[float(v) for v in s.tracker.rect]]
    return np.array(out, np.float64)


# ------------------------------------------------------------------------------------------------ CPU
def test_layout_helpers_follow_postprocess_nhwc_convention():
    """planar channel 21 * m + j is joint j of map m (hm, xm, ym, zm), like the CNN's output and vnect_forward's
    transposition; maps() gives the NHWC arrays vnect_postprocess takes."""
    rng = np.random.default_rng(0)
    planar = rng.standard_normal((6, 84, 46, 46)).astype(np.float32)
    maps = planar_to_nhwc(planar)
    assert len(maps) == 4 and all(m.shape == (6, 46, 46, 21) and m.dtype == np.float32 for m in maps)
    for m in range(4):
        for j in (0, 7, 20):
            assert np.array_equal(maps[m][3, :, :, j], planar[3, 21 * m + j])
    assert np.array_equal(maps[2][5, 10, 11], planar[5, 42:63, 10, 11])
    assert np.array_equal(nhwc_to_planar(maps), planar)
    with pytest.raises(ValueError):
        planar_to_nhwc(planar[:, :80])
    with pytest.raises(ValueError):
        nhwc_to_planar([m[..., :20] for m in maps])


def test_maps_of_the_wrong_shape_are_refused():
    """postprocess() / track_postprocess() hand the C side raw pointers: every map must be [n*n_scales, hs, hs, 21]."""
    ok = [np.zeros((4, 46, 46, 21), np.float64) for _ in range(4)]
    maps, n = check_maps(ok, 2, 46)
    assert n == 2 and all(m.dtype == np.float32 and m.flags.c_contiguous for m in maps)
    bad = [
        ok[:3],                                              # a map missing
        [ok[0], ok[1], ok[2][:2], ok[3]],                    # a short xm / ym / zm
        [m[:, :45, :45] for m in ok],                        # another heat-map size
        [m[..., :20] for m in ok],                           # 20 joints
        [m[:1] for m in ok],                                 # fewer rows than one frame of scales
        [m[:3] for m in ok],                                 # not a whole number of frames
        [m[0] for m in ok],                                  # no batch axis
    ]
    for maps in bad:
        with pytest.raises(ValueError):
            check_maps(maps, 2, 46)


def test_capi_prototypes():
    sig = _capi.SIGNATURES
    import ctypes as C
    P, I32 = C.c_void_p, C.c_int32
    assert sig["vnect_track_postprocess"] == (C.c_int, [P, P, P, P, P, I32, P, P, P, P, P, P, P])
    assert sig["vnect_get_maps"] == (C.c_int, [P, I32, P, C.c_int64, C.POINTER(C.c_int32)])


def test_clocks_are_valid_reference_clocks():
    """Every stream's readings only go forward (or are 0), so the reference raises nowhere; the readings that matter
    are present."""
    for cfg in CONFIGS:
        for sid in range(N_STREAMS):
            s = _Stream(cfg, sid, prepost.OracleTracker, prepost.OracleEstimator)
            for t in (s.t2, s.t3):
                starts = [0] + sorted(k for k, e in s.events.items() if ("reset",) in e)
                for a, b in zip(starts, starts[1:] + [STEPS]):
                    nz = t[a:b][t[a:b] != 0]
                    assert np.all(np.diff(nz) > 0), (cfg[0], sid)


def test_leg_a_reaches_every_branch():
    seen = set()
    for cfg in CONFIGS:
        for br in scenario_branches(cfg).values():
            seen |= br
    seen.discard("geom_unit")
    assert seen == set(BRANCHES), (sorted(set(BRANCHES) - seen), sorted(seen - set(BRANCHES)))


def test_no_scenario_can_be_dropped():
    per = {}
    for cfg in CONFIGS:
        for name, br in scenario_branches(cfg).items():
            per.setdefault(name, set()).update(br)
    for name in per:
        rest = set().union(*(b for n, b in per.items() if n != name))
        assert per[name] - rest, f"scenario {name} reaches nothing the others do not"


def test_every_stream_runs_and_events_happen():
    steps, streams = reference(CONFIGS[0][0])
    assert all(s.k >= 12 for s in streams), [s.k for s in streams]
    evs = [ev[0] for st in steps for _, ev in st["events"]]
    assert sorted(set(evs)) == ["migrate", "reset", "set_box"] and evs.count("set_box") == 4
    assert sum(len(st["calls"][1]) for st in steps) >= 10  # the migrated stream continues on engine B
    assert sum(len(st["active"]) < N_STREAMS for st in steps) == STEPS  # streams skip steps every step


@pytest.mark.parametrize("mutation", sorted(MUTATIONS))
def test_mutated_reference_diverges(mutation):
    """A kernel with this defect would fail the GPU test: the mutated reference leaves the true one on these inputs."""
    cfg = CONFIGS[0]
    true_steps, _ = reference(cfg[0])
    hit = {}

    def until(g, step):
        for e, call in enumerate(step["calls"]):
            for a, b in zip(call, true_steps[g]["calls"][e]):
                if not _records_equal(a, b):
                    hit["at"] = (g, a["sid"])
                    return True
        return False

    run_reference(cfg, *MUTATIONS[mutation], until=until)
    assert "at" in hit, mutation
    print(f"{mutation}: diverges at step {hit['at'][0]}, stream {hit['at'][1]}")


# ------------------------------------------------------------------------------------------------ GPU, leg A
def _assert_step(tag, got, rec, raw):
    j2, j3, used = got
    assert np.array_equal(raw, rec["raw"]), (tag, "raw argmax")
    assert np.array_equal(j2, rec["j2"]), (tag, "joints_2d", np.abs(j2 - rec["j2"]).max())
    assert np.array_equal(j3, rec["j3"]), (tag, "joints_3d", np.abs(j3 - rec["j3"]).max())
    assert tuple(int(v) for v in used) == rec["used"], (tag, "boxes_used", tuple(used), rec["used"])


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_track_postprocess_bit_exact(cfg):
    from vnect_b200 import VNectEngine
    name, scales, S = cfg
    steps, streams = reference(name)
    engs = [VNectEngine(False, scales, box_size=S, max_frames=N_FRAMES, max_streams=N_STREAMS) for _ in range(2)]
    ids = [list(range(N_STREAMS)), {}]  # engine B: reference stream id -> its id there
    try:
        seeds = [(sid, s.seed) for sid, s in enumerate(streams) if s.seed is not None]
        engs[0].set_boxes([i for i, _ in seeds], [b for _, b in seeds])
        n_exports = checked = 0
        for g, st in enumerate(steps):
            boxes = [(sid, ev[1]) for sid, ev in st["events"] if ev[0] == "set_box"]
            for sid, ev in st["events"]:
                if ev[0] == "reset":
                    engs[0].reset(sid)
                elif ev[0] == "migrate":
                    engs[1].import_stream_state(engs[0].export_stream_state(sid), MIGRATED_ID)
                    ids[1][sid] = MIGRATED_ID
            if boxes:
                engs[0].set_boxes([s for s, _ in boxes], [b for _, b in boxes])
            for e, call in enumerate(st["calls"]):
                if not call:
                    continue
                per = [stream_maps(cfg, r["sid"], r["k"]) for r in call]
                maps = tuple(np.concatenate([m[c] for m in per]) for c in range(4))
                sids = [ids[e][r["sid"]] for r in call]
                got = engs[e].track_postprocess(maps, [r["hw"] for r in call], sids, [r["t2"] for r in call],
                                                [r["t3"] for r in call])
                raw = engs[e].raw_argmax(len(call))
                for f, r in enumerate(call):
                    tag = (name, g, "engine AB"[e + 1], r["sid"], r["k"], streams[r["sid"]].scenario)
                    _assert_step(tag, (got[0][f], got[1][f], got[2][f]), r, raw[f])
                    assert engs[e].get_box(sids[f]) == tuple(r["rect"]), (tag, "box")
                    checked += 1
            if "states" in st:
                for sid, s in enumerate(streams):
                    e = 1 if sid in ids[1] else 0
                    got = engs[e].export_stream_state(ids[e][sid])
                    want = st["states"][sid]
                    assert np.array_equal(got, want, equal_nan=True), (name, g, sid, np.nonzero(
                        ~((got == want) | (np.isnan(got) & np.isnan(want))))[0][:8])
                    n_exports += 1
        print(f"{name}: {checked} stream steps bit-exact, {n_exports} stream states equal")
    finally:
        for e in engs:
            e.close()


@pytest.mark.gpu
def test_track_postprocess_refusals_touch_nothing():
    """A refused call -- a side below 2, an id out of range, a duplicate id, a repeated or an earlier timestamp --
    changes no box, filter state or timestamp: every stream's exported state and box are as before, and the call
    that follows gives what it gives on an engine that never saw the refused ones."""
    from vnect_b200 import VNectEngine
    cfg = CONFIGS[0]
    name, scales, S = cfg
    maps = lambda step: tuple(np.concatenate([m[c] for m in (stream_maps(cfg, 0, step), stream_maps(cfg, 1, step))])
                              for c in range(4))
    hw = [(540, 960), (481, 641)]
    engs = [VNectEngine(False, scales, box_size=S, max_frames=2, max_streams=3) for _ in range(2)]
    try:
        for e in engs:
            e.set_boxes([0, 1], [(300, 100, 360, 380), (100, 50, 400, 300)])
            e.track_postprocess(maps(0), hw, [0, 1], [10.0, 20.0], [10.002, 20.002])
        before = [engs[0].export_stream_state(s) for s in range(3)]
        t2, t3 = [10.04, 20.04], [10.042, 20.042]  # the readings of the call that follows
        refused = [
            (ValueError, dict(frame_hw=[(540, 960), (1, 641)])),
            (ValueError, dict(frame_hw=[(540, 960), (481, 1)])),
            (ValueError, dict(ids=[0, 3])),
            (ValueError, dict(ids=[1, 1])),
            (ZeroDivisionError, dict(t2=[10.04, 20.0])),        # stream 1: repeated 2D reading
            (ZeroDivisionError, dict(t3=[10.042, 20.002])),     # stream 1: repeated 3D reading
            (ValueError, dict(t2=[10.04, 19.9])),               # stream 1: earlier 2D reading
            (ValueError, dict(t3=[10.042, 19.9])),              # stream 1: earlier 3D reading
        ]
        for exc, bad in refused:
            with pytest.raises(exc):
                engs[0].track_postprocess(maps(1), bad.get("frame_hw", hw), bad.get("ids", [0, 1]), bad.get("t2", t2),
                                          bad.get("t3", t3))
            after = [engs[0].export_stream_state(s) for s in range(3)]
            for s in range(3):
                assert np.array_equal(after[s], before[s], equal_nan=True), (bad, s)
        got = [e.track_postprocess(maps(1), hw, [0, 1], t2, t3) for e in engs]
        for a, b in zip(*got):
            assert np.array_equal(a, b)
        assert np.array_equal(engs[0].raw_argmax(2), engs[1].raw_argmax(2))
        for s in range(3):
            assert np.array_equal(engs[0].export_stream_state(s), engs[1].export_stream_state(s), equal_nan=True)
    finally:
        for e in engs:
            e.close()


# ------------------------------------------------------------------------------------------------ GPU, leg B
LEG_B_STEPS = 15
LEG_B_STREAMS = 6


def _leg_b_frames(video, k, sizes):
    """Full frames of the golden video for step k: per stream shifted by a few pixels per step and padded / cut to
    its own size (a real moving picture, so the boxes move)."""
    out = []
    for i, (h, w) in enumerate(sizes):
        src = video[(k + 2 * i) % len(video)]
        f = np.zeros((h, w, 3), np.uint8)
        dy, dx = (3 * k + 17 * i) % 40, (5 * k + 29 * i) % 60
        part = src[dy:dy + h, dx:dx + w]
        f[:part.shape[0], :part.shape[1]] = part
        out.append(f)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["track", "track_nv12", "track_frames", "submit_track_frames", "track_device_frames"])
def test_tracked_entry_points_bit_exact_on_cnn_maps(entry, w1, golden):
    import torch
    from vnect_b200 import VNectEngine
    scales, S = [1.0, 0.7], 368
    video = golden("video.npz")["frames"]
    uniform = entry in ("track", "track_nv12")
    sizes = [(480, 864)] * LEG_B_STREAMS if uniform else [(540, 960), (480, 640), (301, 517), (500, 900), (256, 256),
                                                            (431, 777)]
    eng = VNectEngine(w1, scales, max_frames=LEG_B_STREAMS, max_streams=16, max_input=(540, 960))
    try:
        seeds = {0: (100, 40, 400, 400), 2: (0, 0, 200, 150), 3: (600, 300, 400, 300), 5: (700, 50, 100, 380)}
        sids = np.array([9, 2, 14, 5, 0, 11], np.int32)  # not in frame order
        clocks = [_Clock() for _ in range(LEG_B_STREAMS)]
        refs = []
        for i in range(LEG_B_STREAMS):
            est = prepost.OracleEstimator(None, scales, clock=clocks[i], promotion="legacy", box_size=S)
            refs.append(prepost.OracleTracker(est, seeds.get(i, (0, 0, HUGE, HUGE))))
        eng.set_boxes([int(sids[i]) for i in seeds], list(seeds.values()))
        rng = np.random.default_rng(77)
        t2 = 1.76e9 + np.cumsum(rng.uniform(0.02, 0.05, (LEG_B_STEPS, LEG_B_STREAMS)), axis=0)
        t3 = t2 + rng.uniform(0.001, 0.004, t2.shape)
        dev_j2 = torch.empty((LEG_B_STREAMS, 21, 2), dtype=torch.float64, device="cuda")
        dev_j3 = torch.empty((LEG_B_STREAMS, 21, 3), dtype=torch.float32, device="cuda")
        dev_boxes = torch.empty((LEG_B_STREAMS, 4), dtype=torch.int32, device="cuda")
        launches = []
        for k in range(LEG_B_STEPS):
            frames = _leg_b_frames(video, k, sizes)
            n = len(frames)
            before = eng.launch_count()
            if entry == "track":
                got = eng.track(np.stack(frames), sids, t2[k], t3[k])
            elif entry == "track_nv12":
                yuv = np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420) for f in frames])
                nv12 = yuv.copy()  # I420 -> NV12: interleave the chroma planes
                h, w = sizes[0]
                q = (h // 2) * (w // 2)
                for i in range(n):
                    u = yuv[i, h:].reshape(-1)[:q]
                    v = yuv[i, h:].reshape(-1)[q:]
                    nv12[i, h:] = np.stack([u, v], axis=1).reshape(h // 2, w)
                got = eng.track(nv12, sids, t2[k], t3[k], pixel_format="nv12")
                frames = [cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12) for f in nv12]
            elif entry == "track_frames":
                got = eng.track_frames(frames, sids, t2[k], t3[k])
            elif entry == "submit_track_frames":
                eng.submit_track_frames(k % 2, frames, sids, t2[k], t3[k])
                got = eng.wait(k % 2)
            else:
                dev = [torch.from_numpy(f).cuda() for f in frames]
                torch.cuda.synchronize()
                eng.track_device_frames([dict(ptr=d.data_ptr(), h=d.shape[0], w=d.shape[1]) for d in dev],
                                        dev_j2.data_ptr(), dev_j3.data_ptr(), dev_boxes.data_ptr(), sids, t2[k], t3[k])
                eng.synchronize()
                got = (dev_j2.cpu().numpy(), dev_j3.cpu().numpy(), dev_boxes.cpu().numpy())
            launches.append(eng.launch_count() - before)
            maps = eng.maps(n)
            raw = eng.raw_argmax(n)
            ns = len(scales)
            for i in range(n):
                m_i = tuple(m[i * ns:(i + 1) * ns] for m in maps)
                refs[i].estimator.forward = lambda batch, m=m_i: m
                clocks[i].q = [float(t2[k, i]), float(t3[k, i])]
                r2, r3, used = refs[i](frames[i])
                tag = (entry, k, i)
                rec = dict(j2=r2, j3=r3, used=tuple(used), raw=refs[i].estimator.last["joints_2d_raw"].astype(np.int32))
                _assert_step(tag, (got[0][i], got[1][i], got[2][i]), rec, raw[i])
                assert eng.get_box(int(sids[i])) == tuple(refs[i].rect), (tag, "box")
        # the first call also writes the pyramid's constant surround once (ensure_surround); later calls replay a graph
        assert len(set(launches[1:])) == 1 and eng.info("cached_graphs") >= 1, launches
        print(f"{entry}: {LEG_B_STEPS} steps x {LEG_B_STREAMS} streams bit-exact; launches per call {launches[:3]}..., "
              f"{eng.info('cached_graphs'):.0f} cached graph(s)")
    finally:
        eng.close()
