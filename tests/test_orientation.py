"""Per-stream frame orientation (vnect_set_orientations): cameras mounted sideways, upside down or mirrored.

The contract (include/vnect_b200.h): a stream with orientation o given stored frame F produces bit for bit what a stream
with identity orientation produces for the materialised frame orient(F, o).  Engine A (orientations set, stored frames)
and engine B (identity, materialised frames) are two disjoint ranges of stream ids of one engine, fed the same clock
readings; the CNN is batch-invariant, so every output is compared with np.array_equal.

CPU: `orient` / `orient_yuv` (this file's numpy restatement of the header's table) against cv2 and numpy, the property
the YUV semantics rest on, the kernel's affine index map, and the Python code table against the header.
GPU: the stem input and every result on every entry point that takes stream ids, mixed orientations in one call,
ordering against submission, the untouched identity path, and refusals.
"""
import itertools
import os
import re

import cv2
import numpy as np
import pytest

from tests.test_yuv_input import _device_surface, _padded, random_yuv
from vnect_b200.estimator import ORIENTATIONS, yuv_layout

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
CV_CODE = {"nv12": cv2.COLOR_YUV2BGR_NV12, "i420": cv2.COLOR_YUV2BGR_I420}
SWAPS = (1, 3, 6, 7)


# ------------------------------------------------------------------------------------------------ the definition
def orient(f, code):
    """The oriented frame of stored frame f ([H, W] or [H, W, C]) for VNECT_ORIENT_* `code` (the header's table)."""
    return [f, np.rot90(f, 3), np.rot90(f, 2), np.rot90(f, 1), f[:, ::-1], f[::-1], f.swapaxes(0, 1),
            np.rot90(f, 2).swapaxes(0, 1)][code]


def orient_yuv(yuv, code, fmt):
    """A 4:2:0 frame in cv2's contiguous [3H/2, W] layout -> the materialised oriented frame in the same layout:
    luma and chroma planes oriented separately (NV12's interleaved pairs move as one sample)."""
    h, w = yuv.shape[0] * 2 // 3, yuv.shape[1]
    y = orient(yuv[:h], code)
    ho, wo = y.shape
    if fmt == "nv12":
        uv = orient(yuv[h:].reshape(h // 2, w // 2, 2), code)
        chroma = uv.reshape(ho // 2, wo)
    else:
        q = (h // 2) * (w // 2)
        flat = yuv[h:].reshape(-1)
        u = orient(flat[:q].reshape(h // 2, w // 2), code)
        v = orient(flat[q:].reshape(h // 2, w // 2), code)
        chroma = np.concatenate([u.reshape(-1), v.reshape(-1)]).reshape(ho // 2, wo)
    return np.ascontiguousarray(np.concatenate([y, chroma]))


def stored_pixel(code, H, W, yo, xo):
    """(ys, xs) of the header's table."""
    return [(yo, xo), (H - 1 - xo, yo), (H - 1 - yo, W - 1 - xo), (xo, W - 1 - yo), (yo, W - 1 - xo),
            (H - 1 - yo, xo), (xo, yo), (H - 1 - xo, W - 1 - yo)][code]


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("hw", [(3, 5), (4, 6), (7, 7), (1, 9), (481, 643)])
def test_orient_matches_numpy_and_cv2(hw):
    rng = np.random.default_rng(hw[0] * 1000 + hw[1])
    f = rng.integers(0, 256, (*hw, 3), dtype=np.uint8)
    cv = [f, cv2.rotate(f, cv2.ROTATE_90_CLOCKWISE), cv2.rotate(f, cv2.ROTATE_180),
          cv2.rotate(f, cv2.ROTATE_90_COUNTERCLOCKWISE), cv2.flip(f, 1), cv2.flip(f, 0), cv2.transpose(f),
          cv2.flip(cv2.transpose(f), -1)]
    npy = [f, np.rot90(f, 3), np.rot90(f, 2), np.rot90(f, 1), f[:, ::-1], f[::-1], f.transpose(1, 0, 2),
           np.rot90(f, 2).transpose(1, 0, 2)]
    H, W = hw
    for code in range(8):
        o = orient(f, code)
        assert np.array_equal(o, cv[code].reshape(o.shape)) and np.array_equal(o, npy[code]), code
        assert o.shape[:2] == ((W, H) if code in SWAPS else (H, W))
        for yo, xo in [(0, 0), (o.shape[0] - 1, 0), (0, o.shape[1] - 1), (o.shape[0] // 2, o.shape[1] // 3)]:
            assert np.array_equal(o[yo, xo], f[stored_pixel(code, H, W, yo, xo)]), (code, yo, xo)


def kernel_map(code, H, W, yo, xo):
    """The index map as prepost_kernels.cuh's Oriented<> sources build it: bit masks, origin and two steps."""
    swap, ry, rx = (0xCA >> code) & 1, (0xA6 >> code) & 1, (0x9C >> code) & 1
    dy, dx = np.array([-1 if ry else 1, 0]), np.array([0, -1 if rx else 1])  # stored (y, x) steps
    ey, ex = (dx, dy) if swap else (dy, dx)
    origin = np.array([H - 1 if ry else 0, W - 1 if rx else 0])
    return tuple(origin + yo * ey + xo * ex)


@pytest.mark.parametrize("hw", [(3, 5), (6, 4)])
def test_kernel_index_map_is_the_table(hw):
    H, W = hw
    for code in range(8):
        ho, wo = (W, H) if code in SWAPS else (H, W)
        for yo, xo in itertools.product(range(ho), range(wo)):
            assert kernel_map(code, H, W, yo, xo) == stored_pixel(code, H, W, yo, xo)
        # chroma: every 2x2 oriented block maps onto one stored 2x2 block when the sides are even
        if H % 2 == 0 and W % 2 == 0:
            for yo, xo in itertools.product(range(0, ho, 2), range(0, wo, 2)):
                blocks = {tuple(v // 2 for v in kernel_map(code, H, W, yo + a, xo + b)) for a in (0, 1) for b in (0, 1)}
                assert len(blocks) == 1


@pytest.mark.parametrize("fmt", ["nv12", "i420"])
@pytest.mark.parametrize("hw", [(2, 2), (6, 10), (48, 32), (480, 640)])
def test_converting_oriented_planes_is_orienting_the_conversion(fmt, hw):
    rng = np.random.default_rng(7 + hw[0])
    yuv = random_yuv(rng, 1, *hw)[0]
    bgr = cv2.cvtColor(yuv, CV_CODE[fmt])
    for code in range(8):
        assert np.array_equal(cv2.cvtColor(orient_yuv(yuv, code, fmt), CV_CODE[fmt]), orient(bgr, code)), code


def test_orientation_names_match_the_header():
    header = open(os.path.join(ROOT, "include", "vnect_b200.h")).read()
    defines = {m.group(1).lower(): int(m.group(2)) for m in re.finditer(r"#define VNECT_ORIENT_(\w+) (\d+)", header)}
    assert defines == ORIENTATIONS
    assert sorted(ORIENTATIONS.values()) == list(range(8))


# ------------------------------------------------------------------------------------------------ GPU helpers
SCALE_LISTS = {"s2": [1.0, 0.7], "s3": [1.0, 0.85, 0.7]}
MAXF, REF = 64, 64  # engine B's stream id = engine A's + REF
_clock = itertools.count()


def ticks(n):
    """n fresh clock readings (2D, 3D), increasing over the whole module so streams may be reused."""
    t = 1000.0 + 0.0333 * np.array([next(_clock) for _ in range(n)], np.float64)
    return t, t + 0.004


@pytest.fixture(scope="module", params=sorted(SCALE_LISTS))
def eng(request, w1):
    from vnect_b200 import VNectEngine
    e = VNectEngine(w1, SCALE_LISTS[request.param], max_frames=MAXF, max_streams=2 * REF, max_input=(1920, 1920))
    e.tag = request.param
    yield e
    e.close()


def set_codes(eng, ids, codes):
    eng.set_orientations(list(ids), list(codes))
    eng.set_orientations([i + REF for i in ids], [0] * len(ids))


def check_same(a, b, what):
    for k in a:
        assert np.array_equal(a[k], b[k]), f"{what}: {k} differs"


def geometry_note(S, h, w, code):
    """The pre-processing branches a frame of oriented size h x w reaches (preprocess_exact.log's notation)."""
    m = max(h, w)
    mode = "area" if m == 2 * S else "linear"
    partial = mode == "area" and (h % 2 or w % 2)
    return f"code {code} oriented {h}x{w}: {mode}{' partial-block' if partial else ''}" + (
        " (identity alias skipped)" if h == w == S and code else "")


def to_dev(arrs):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs]


def dev_out(n):
    import torch
    return (torch.empty((n, 21, 2), dtype=torch.float64, device="cuda"),
            torch.empty((n, 21, 3), dtype=torch.float32, device="cuda"),
            torch.empty((n, 4), dtype=torch.int32, device="cuda"))


def host_frames(rng, fmt, h, w, n):
    if fmt == "bgr":
        return list(rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8))
    return list(random_yuv(rng, n, h, w))


def materialise(frames, codes, fmt):
    return [orient(f, c) if fmt == "bgr" else orient_yuv(f, c, fmt) for f, c in zip(frames, codes)]


def run_call(eng, kind, frames, ids, fmt, t, lane=0, layout=None):
    """One call of entry point `kind` -> dict of everything it returns plus the stem input and the raw argmax."""
    import torch
    n = len(frames)
    t2, t3 = t
    out = {}
    if kind in ("estimate", "submit0", "submit1", "track"):
        arr = np.stack(frames)
        if kind == "estimate":
            out["j2"], out["j3"] = eng.estimate(arr, ids, t2, t3, pixel_format=fmt)
        elif kind == "track":
            out["j2"], out["j3"], out["boxes"] = eng.track(arr, ids, t2, t3, pixel_format=fmt)
        else:
            ln = int(kind[-1])
            j2, j3 = eng.submit(ln, arr, ids, t2, t3, pixel_format=fmt)
            eng.wait(ln)
            out["j2"], out["j3"] = j2.copy(), j3.copy()
    elif kind in ("estimate_device", "track_device"):
        h, w = frames[0].shape[:2]
        if fmt != "bgr":
            h = h * 2 // 3
        lay = layout(fmt, h, w) if (layout and fmt != "bgr") else None
        if lay is not None:
            ylay = yuv_layout(fmt, h, w, **lay)
            buf = _device_surface(np.stack(frames), fmt, ylay)
        else:
            buf = np.stack(frames)
        (d,) = to_dev([buf])
        j2d, j3d, bd = dev_out(n)
        if kind == "estimate_device":
            eng.estimate_device(d.data_ptr(), n, h, w, j2d.data_ptr(), j3d.data_ptr(), ids, t2, t3, pixel_format=fmt,
                                layout=lay)
        else:
            eng.track_device(d.data_ptr(), n, h, w, j2d.data_ptr(), j3d.data_ptr(), bd.data_ptr(), ids, t2, t3,
                             pixel_format=fmt, layout=lay)
            out["boxes"] = bd
        torch.cuda.synchronize()
        out["j2"], out["j3"] = j2d, j3d
    elif kind in ("estimate_frames", "submit_frames1", "track_frames", "submit_track_frames0", "submit_track_frames1",
                  "estimate_sequence"):
        if kind == "estimate_frames":
            out["j2"], out["j3"] = eng.estimate_frames(frames, ids, t2, t3, pixel_format=fmt)
        elif kind == "estimate_sequence":
            out["j2"], out["j3"] = eng.estimate_sequence(frames, ids, t2, t3, pixel_format=fmt)
        elif kind == "submit_frames1":
            j2, j3 = eng.submit_frames(1, frames, ids, t2, t3, pixel_format=fmt)
            eng.wait(1)
            out["j2"], out["j3"] = j2.copy(), j3.copy()
        elif kind == "track_frames":
            out["j2"], out["j3"], out["boxes"] = eng.track_frames(frames, ids, t2, t3, pixel_format=fmt)
        else:
            ln = int(kind[-1])
            j2, j3, b = eng.submit_track_frames(ln, frames, ids, t2, t3, pixel_format=fmt)
            eng.wait(ln)
            out["j2"], out["j3"], out["boxes"] = j2.copy(), j3.copy(), b.copy()
    elif kind in ("estimate_device_frames", "track_device_frames", "estimate_device_sequence"):
        devs = to_dev(frames)
        desc = []
        for f, d in zip(frames, devs):
            h, w = f.shape[:2]
            desc.append(dict(ptr=d.data_ptr(), h=h if fmt == "bgr" else h * 2 // 3, w=w))
        j2d, j3d, bd = dev_out(n)
        if kind == "estimate_device_frames":
            eng.estimate_device_frames(desc, j2d.data_ptr(), j3d.data_ptr(), ids, t2, t3, pixel_format=fmt)
        elif kind == "estimate_device_sequence":
            eng.estimate_device_sequence(desc, j2d.data_ptr(), j3d.data_ptr(), ids, t2, t3, pixel_format=fmt)
        else:
            eng.track_device_frames(desc, j2d.data_ptr(), j3d.data_ptr(), bd.data_ptr(), ids, t2, t3, pixel_format=fmt)
            out["boxes"] = bd
        torch.cuda.synchronize()
        out["j2"], out["j3"] = j2d, j3d
    else:
        raise AssertionError(kind)
    out = {k: (v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)) for k, v in out.items()}
    eng.synchronize()
    out["stem"] = eng.stem_input(n * len(eng.scales))
    out["argmax"] = eng.raw_argmax(n)
    return out


def compare_pair(eng, kind, stored, codes, ids, fmt, lane_note="", layout=None, state=True):
    """Call A (codes set on `ids`, stored frames) and B (identity on ids + REF, materialised frames); compare."""
    set_codes(eng, ids, codes)
    t = ticks(len(ids))
    a = run_call(eng, kind, stored, ids, fmt, t, layout=layout)
    b = run_call(eng, kind, materialise(stored, codes, fmt), [i + REF for i in ids], fmt, t, layout=layout)
    check_same(a, b, f"{kind} {fmt} codes {codes} {lane_note}")
    if state:
        for i in ids:
            assert np.array_equal(eng.export_stream_state(i), eng.export_stream_state(i + REF)), (kind, i)
    return a


def oriented_hw(fmt, f, code):
    h, w = f.shape[:2]
    if fmt != "bgr":
        h = h * 2 // 3
    return (w, h) if code in SWAPS else (h, w)


BGR_SIZES = [(481, 643), (368, 368), (735, 736)]  # odd sides; the identity alias; oriented long side 2S, partial block
YUV_SIZES = [(480, 640), (736, 480)]


# ------------------------------------------------------------------------------------------------ GPU
@gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12", "i420"])
def test_uniform_entry_points(eng, fmt):
    """estimate, submit on lanes 0 and 1, estimate_device (YUV on a padded decoder surface too): every code, every
    size, stem input and results bit for bit."""
    rng = np.random.default_rng(1)
    sizes = BGR_SIZES if fmt == "bgr" else YUV_SIZES
    kinds = ["estimate", "submit0", "submit1", "estimate_device"]
    for (h, w), kind, code in itertools.product(sizes, kinds, range(8)):
        stored = host_frames(rng, fmt, h, w, 2)
        compare_pair(eng, kind, stored, [code, code], [0, 1], fmt)
        if kind == "estimate_device" and fmt != "bgr":
            compare_pair(eng, kind, stored, [code, code], [0, 1], fmt, layout=_padded)
    for h, w in sizes:
        print(f"[{eng.tag} {fmt}] {h}x{w}: " + "; ".join(
            geometry_note(eng.box_size, *oriented_hw(fmt, np.zeros((h if fmt == 'bgr' else h * 3 // 2, w)), c), c)
            for c in range(8)))


@gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12", "i420"])
def test_table_and_sequence_entry_points(eng, fmt):
    """estimate_frames, submit_frames (lane 1), estimate_device_frames and the two sequence calls: one call carries
    all eight codes on frames of different sizes; packed results too."""
    import torch
    packed = torch.zeros((MAXF, 21, 5), dtype=torch.float64, device="cuda")
    eng.set_packed_results(packed.data_ptr())
    try:
        rng = np.random.default_rng(2)
        sizes = BGR_SIZES if fmt == "bgr" else YUV_SIZES
        codes = list(range(8))
        stored = [host_frames(rng, fmt, *sizes[i % len(sizes)], 1)[0] for i in range(8)]
        for kind in ["estimate_frames", "submit_frames1", "estimate_device_frames"]:
            set_codes(eng, range(8), codes)
            t = ticks(8)
            a = run_call(eng, kind, stored, list(range(8)), fmt, t)
            pa = packed[:8].cpu().numpy()
            b = run_call(eng, kind, materialise(stored, codes, fmt), [i + REF for i in range(8)], fmt, t)
            check_same(a, b, f"{kind} {fmt}")
            assert np.array_equal(pa, packed[:8].cpu().numpy()), kind
        # sequences: streams 10 and 11, four frames each, interleaved, every code once
        ids = [10, 11, 10, 11, 10, 11, 10, 11]
        for kind in ["estimate_sequence", "estimate_device_sequence"]:
            seq_codes = [2, 5]  # one code per stream; the frames of a stream carry all sizes
            set_codes(eng, [10, 11], seq_codes)
            t = ticks(8)
            per = [seq_codes[i % 2] for i in range(8)]
            a = run_call(eng, kind, stored, ids, fmt, t)
            b = run_call(eng, kind, materialise(stored, per, fmt), [i + REF for i in ids], fmt, t)
            check_same(a, b, f"{kind} {fmt}")
            for s in (10, 11):
                assert np.array_equal(eng.export_stream_state(s), eng.export_stream_state(s + REF))
    finally:
        eng.set_packed_results(0)


def seed_boxes(fmt, frames, codes):
    """Boxes in the oriented frame: partly outside, odd offsets, and one clipped to 2x2."""
    boxes = []
    for i, (f, c) in enumerate(zip(frames, codes)):
        h, w = oriented_hw(fmt, f, c)
        boxes.append([(w // 3 | 1, h // 5 | 1, w // 2, h // 2),      # odd offsets, inside
                      (w - w // 4, h // 3, w // 2, h),                # partly outside (right and bottom)
                      (w - 1, h - 1, 40, 40),                         # clipped to 2x2
                      (37, 51, 3 * w // 4 + 1, 3 * h // 4 + 1)][i % 4])
    return boxes


@gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12", "i420"])
def test_tracked_entry_points(eng, fmt):
    """track, track_device (uniform), track_frames, submit_track_frames on both lanes and track_device_frames: 8 steps
    per stream from seeded boxes; boxes_used, the box left behind and the exported state every step."""
    rng = np.random.default_rng(3)
    sizes = BGR_SIZES if fmt == "bgr" else YUV_SIZES
    uniform = ["track", "track_device"]
    table = ["track_frames", "submit_track_frames0", "submit_track_frames1", "track_device_frames"]
    for kind in uniform + table:
        if kind in uniform:
            cases = [(sizes[k % len(sizes)], [c, c, c, c]) for k, c in enumerate(range(8))]
        else:
            cases = [(None, list(range(8)))]
        for size, codes in cases:
            n = len(codes)
            ids = list(range(20, 20 + n))
            if size is None:
                stored0 = [host_frames(rng, fmt, *sizes[i % len(sizes)], 1)[0] for i in range(n)]
            else:
                stored0 = host_frames(rng, fmt, *size, n)
            boxes = seed_boxes(fmt, stored0, codes)
            set_codes(eng, ids, codes)
            eng.set_boxes(ids + [i + REF for i in ids], boxes + boxes)
            for step in range(8):
                # the scene moves: a fresh noise frame at the same stored size each step
                stored = [host_frames(rng, fmt, *(f.shape[:2] if fmt == "bgr" else (f.shape[0] * 2 // 3, f.shape[1])),
                                      1)[0] for f in stored0]
                compare_pair(eng, kind, stored, codes, ids, fmt, f"step {step}", state=False)
                for i in ids:
                    assert eng.get_box(i) == eng.get_box(i + REF), (kind, step, i)
                    assert np.array_equal(eng.export_stream_state(i), eng.export_stream_state(i + REF)), (kind, step)


@gpu
def test_mixed_orientations_in_one_call(eng):
    """64 streams, all eight codes, three camera sizes, in one track_device_frames / submit_track_frames /
    estimate_sequence call: frame i equals its materialised identity call."""
    rng = np.random.default_rng(4)
    cams = [(480, 640), (720, 1280), (1080, 1920)]
    codes = [i % 8 for i in range(64)]
    # 64 streams of A take ids 0..63 and B 64..127: the engine's stream range
    for kind in ["track_device_frames", "submit_track_frames1", "estimate_sequence"]:
        stored = [rng.integers(0, 256, (*cams[(i // 8) % 3], 3), dtype=np.uint8) for i in range(64)]
        ids = list(range(64))
        set_codes(eng, ids, codes)
        if kind != "estimate_sequence":
            boxes = seed_boxes("bgr", stored, codes)
            eng.set_boxes(ids + [i + REF for i in ids], boxes + boxes)
        compare_pair(eng, kind, stored, codes, ids, "bgr")


@gpu
def test_orientation_applies_in_submission_order(eng):
    """set_orientations between two submitted calls on different lanes, before either is waited on, affects only the
    later one; a stream changing orientation mid-track matches materialised frames changing at the same step."""
    rng = np.random.default_rng(5)
    f0 = host_frames(rng, "bgr", 481, 643, 2)
    f1 = host_frames(rng, "bgr", 481, 643, 2)
    set_codes(eng, [30, 31], [1, 6])
    t_a, t_b = ticks(2), ticks(2)
    a0 = eng.submit(0, np.stack(f0), [30, 31], *t_a)
    eng.set_orientations([30, 31], ["flip_h", "rot180"])  # host-only: the lane-0 call keeps codes 1 and 6
    a1 = eng.submit(1, np.stack(f1), [30, 31], *t_b)
    eng.wait(0)
    eng.wait(1)
    b0 = eng.estimate_frames(materialise(f0, [1, 6], "bgr"), [30 + REF, 31 + REF], *t_a)
    b1 = eng.estimate_frames(materialise(f1, [4, 2], "bgr"), [30 + REF, 31 + REF], *t_b)
    assert all(np.array_equal(x, y) for x, y in zip(a0 + a1, b0 + b1))
    assert eng.orientation(30) == 4 and eng.orientation(31) == 2
    # mid-track change: rot90_cw for four steps, then transpose (the box stays in oriented coordinates)
    ids = [40, 41]
    set_codes(eng, ids, [1, 1])
    eng.set_boxes(ids + [i + REF for i in ids], [(100, 200, 300, 240)] * 4)
    for step in range(8):
        code = 1 if step < 4 else 6
        eng.set_orientations(ids, [code, code])
        stored = host_frames(rng, "bgr", 481, 643, 2)
        t = ticks(2)
        a = run_call(eng, "submit_track_frames1", stored, ids, "bgr", t)
        b = run_call(eng, "submit_track_frames1", materialise(stored, [code, code], "bgr"), [i + REF for i in ids],
                     "bgr", t)
        check_same(a, b, f"mid-track step {step}")
        for i in ids:
            assert np.array_equal(eng.export_stream_state(i), eng.export_stream_state(i + REF))


@gpu
def test_identity_path_is_untouched(w1):
    """With no orientation set, and with every stream set to identity explicitly, a fixed call sequence makes the same
    launches per call and caches the same graphs; an oriented call runs the table pipeline's launches."""
    from vnect_b200 import VNectEngine
    rng = np.random.default_rng(6)
    frames = rng.integers(0, 256, (3, 481, 643, 3), dtype=np.uint8)
    square = rng.integers(0, 256, (3, 368, 368, 3), dtype=np.uint8)

    def sequence(e):
        counts = []
        for k in range(3):
            for arr, call in [(frames, "estimate"), (square, "estimate"), (frames, "track"), (frames, "frames")]:
                t = ticks(3)
                before = e.launch_count()
                if call == "estimate":
                    e.estimate(arr, [0, 1, 2], *t)
                elif call == "track":
                    e.track(arr, [0, 1, 2], *t)
                else:
                    e.estimate_frames(list(arr), [0, 1, 2], *t)
                counts.append(e.launch_count() - before)
        return counts, e.info("cached_graphs")

    engines = [VNectEngine(w1, [1.0, 0.7], max_frames=4, max_streams=4, max_input=(1080, 1080)) for _ in range(2)]
    try:
        engines[1].set_orientations([0, 1, 2, 3], ["identity"] * 4)
        plain, explicit = sequence(engines[0]), sequence(engines[1])
        assert plain == explicit
        print("launches per call", plain[0], "cached graphs", plain[1])
        # an oriented uniform call runs the table pipeline: the launches of estimate_frames
        e = engines[1]
        e.set_orientations([0], ["rot90_cw"])
        t = ticks(3)
        before = e.launch_count()
        e.estimate(frames, [0, 1, 2], *t)
        oriented = e.launch_count() - before
        assert oriented == plain[0][3], (oriented, plain[0])
    finally:
        for e in engines:
            e.close()


@gpu
def test_refusals_change_nothing(eng):
    import ctypes as C
    from vnect_b200 import _capi
    lib, h = eng._lib, eng._h
    eng.set_orientations([50, 51], ["transpose", "rot90_ccw"])
    eng.set_boxes([50, 51], [(3, 5, 40, 60), (7, 9, 20, 30)])
    before = ([eng.orientation(s) for s in range(2 * REF)], [eng.get_box(s) for s in (50, 51)],
              [eng.export_stream_state(s) for s in (50, 51)])

    def raw(n, ids, codes):
        a = None if ids is None else (C.c_int32 * max(len(ids), 1))(*ids)
        b = None if codes is None else (C.c_int32 * max(len(codes), 1))(*codes)
        return lib.vnect_set_orientations(h, n, a, b)

    for n, ids, codes in [(-1, [50], [1]), (1, None, [1]), (1, [50], None), (2, [50, 2 * REF], [1, 1]),
                          (2, [50, -1], [1, 1]), (2, [51, 51], [1, 2]), (2, [50, 51], [1, 8]), (2, [50, 51], [-1, 1])]:
        assert raw(n, ids, codes) == _capi.E_INVALID, (n, ids, codes)
    with pytest.raises(ValueError):
        eng.set_orientations([50], ["sideways"])
    with pytest.raises(ValueError):
        eng.set_orientations([50, 51], [1])
    out = C.c_int32()
    assert lib.vnect_get_orientation(h, 2 * REF, C.byref(out)) == _capi.E_INVALID
    assert raw(0, None, None) == _capi.OK
    after = ([eng.orientation(s) for s in range(2 * REF)], [eng.get_box(s) for s in (50, 51)],
             [eng.export_stream_state(s) for s in (50, 51)])
    assert before[0] == after[0] and before[1] == after[1]
    assert all(np.array_equal(x, y) for x, y in zip(before[2], after[2]))
    # configuration, not temporal state: reset keeps it
    eng.reset(50)
    assert eng.orientation(50) == ORIENTATIONS["transpose"]
