"""The numpy/cv2 oracle for pre/post-processing, pinned against the reference's own code.

Fixtures under tests/golden/ were minted by tests/golden/make_golden.py from the reference's unchanged
src/estimator.py, src/utils.py and src/OneEuroFilter.py; every comparison here runs on those stored outputs.
"""
import hashlib

import cv2
import numpy as np
import pytest

from oracle import prepost, synth
from tests.golden.make_golden import POST_CASES, PRE_CASES, post_frame_maps


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


# ------------------------------------------------------------------------------------------------ OpenCV restatements
@pytest.mark.parametrize("seed", range(14))
def test_resize_u8_int_matches_cv2(seed):
    rng = np.random.default_rng(seed)
    h, w = int(rng.integers(16, 640)), int(rng.integers(16, 640))
    s = [0.7, 0.85, 368 / max(h, w), float(rng.uniform(0.3, 1.8))][seed % 4]
    if seed >= 12:  # both sides round back to themselves: cv2 copies the image although s != 1
        s = 1 - 0.45 / max(h, w) if seed == 12 else 1 + 0.45 / max(h, w)
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    ref = cv2.resize(img, (0, 0), fx=s, fy=s, interpolation=cv2.INTER_LINEAR)
    got = prepost.resize_u8_int(img, s, s)
    assert got.shape == ref.shape
    assert np.array_equal(got, ref)


@pytest.mark.parametrize("s", [0.7, 0.85, 0.6, 0.99, 0.995, 0.999])  # the last three keep 46 cells: cv2 copies
def test_resize_f32_np_matches_cv2(s):
    m = (np.random.default_rng(3).standard_normal((46, 46, 21)) * 0.01).astype(np.float32)
    ref = cv2.resize(m, (0, 0), fx=1 / s, fy=1 / s, interpolation=cv2.INTER_LINEAR)
    got = prepost.resize_f32_np(m, 1 / s, 1 / s)
    assert got.shape == ref.shape
    assert np.array_equal(got, ref)


def test_upsample8_f64_is_lerp_fma():
    rng = np.random.default_rng(4)
    hm = rng.standard_normal((46, 46)) * 0.01
    ref = cv2.resize(hm, (0, 0), fx=8, fy=8, interpolation=cv2.INTER_LINEAR)
    pts = [(int(a), int(b)) for a, b in rng.integers(0, 368, (300, 2))] + [(0, 0), (3, 3), (4, 4), (363, 364), (367, 367)]
    for dy, dx in pts:
        assert prepost.upsample8_f64_point(hm, dy, dx) == ref[dy, dx]
    # replicated borders are exact ties (SURVEY.md App. C.4)
    assert np.array_equal(ref[0], ref[3]) and np.array_equal(ref[:, 0], ref[:, 3])
    assert np.array_equal(ref[364], ref[367]) and np.array_equal(ref[:, 364], ref[:, 367])


# ------------------------------------------------------------------------------------------------ golden fixtures
@pytest.mark.parametrize("case", PRE_CASES, ids=[c[0] for c in PRE_CASES])
def test_gen_input_batch_golden(case, golden):
    name, h, w, seed, scales = case
    g = golden("pre.npz")
    img = np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
    batch, scaler, (ox, oy) = prepost.gen_input_batch(img, 368, scales)
    assert batch.dtype == np.float32 and batch.shape == (len(scales), 368, 368, 3)
    assert np.array_equal(np.array([scaler, ox, oy], np.float64), g[name + "/meta"])
    assert np.array_equal(batch[:, ::37, ::41, :], g[name + "/sample"])
    assert sha(batch) == str(g[name + "/sha"])


def test_one_euro_filter_golden(golden):
    g = golden("filter.npz")
    f2 = prepost.OneEuroFilter(**prepost.FILTER_2D)
    f3 = prepost.OneEuroFilter(**prepost.FILTER_3D)
    y2 = np.array([f2(float(x), float(t)) for x, t in zip(g["x"], g["t"])])
    y3 = np.array([f3(float(x), float(t)) for x, t in zip(g["x"], g["t"])])
    assert np.array_equal(y2, g["y2"]) and np.array_equal(y3, g["y3"])
    assert y2[0] == g["x"][0]  # first sample passes through


def test_one_euro_filter_errors():
    with pytest.raises(ValueError):
        prepost.OneEuroFilter(freq=0)
    with pytest.raises(ValueError):
        prepost.OneEuroFilter(freq=30, mincutoff=0)
    f = prepost.OneEuroFilter(**prepost.FILTER_2D)
    f(1.0, 5.0)
    with pytest.raises(ZeroDivisionError):
        f(2.0, 5.0)


class _Clock:
    def __init__(self):
        self.q = []

    def __call__(self):
        return self.q.pop(0)


def _run_post_case(case, promotion):
    name, seed, scales, nf, pat = case
    state = {}
    clock = _Clock()
    est = prepost.OracleEstimator(lambda b: state["maps"], scales, clock=clock, promotion=promotion)
    from tests.golden.make_golden import timestamps
    t2, t3 = timestamps(pat, nf, seed)
    img = np.zeros((368, 368, 3), np.uint8)
    j2s, j3s = [], []
    for k in range(nf):
        state["maps"] = post_frame_maps(seed, k, scales)
        clock.q = [float(t2[k]), float(t3[k])]
        j2, j3 = est(img)
        j2s.append(j2)
        j3s.append(j3)
    return np.array(j2s), np.array(j3s)


@pytest.mark.parametrize("case", POST_CASES, ids=[c[0] for c in POST_CASES])
def test_estimator_postprocess_golden(case, golden):
    g = golden("post.npz")
    j2, j3 = _run_post_case(case, "numpy")
    assert j2.dtype == np.float64 and j3.dtype == np.float32
    assert np.array_equal(j2, g[case[0] + "/j2"])
    assert np.array_equal(j3, g[case[0] + "/j3"])
    # numpy-1.x ("legacy") promotion of the 3D filter, which the CUDA path implements, is the same to float32 noise
    l2, l3 = _run_post_case(case, "legacy")
    assert np.array_equal(l2, j2)
    assert np.max(np.abs(l3.astype(np.float64) - j3)) < 1e-2  # mm (float32 filter arithmetic vs float64)


def test_border_peaks_resolve_like_reference(golden):
    """First frame of s2_border has peaks forced onto map borders/corners: exact-tie rule of SURVEY.md App. C.4."""
    g = golden("post.npz")
    j2 = g["s2_border/j2"][0]
    assert tuple(j2[0]) == (0.0, 0.0) and tuple(j2[3]) == (364.0, 364.0)
    assert j2[4][0] == 0.0 and j2[5][0] == 364.0 and j2[6][1] == 0.0 and j2[7][1] == 364.0


def test_hm_pt_interp_quirks():
    src = np.arange(46 * 46, dtype=np.float64).reshape(46, 46)
    assert prepost.hm_pt_interp_bilinear(src, 8, (363.5, 100.0)) == 0.0  # far border: x1 == x0 weights cancel
    assert prepost.hm_pt_interp_bilinear(src, 8, (100.0, 367.0)) == 0.0
    v = prepost.hm_pt_interp_bilinear(src, 8, (0.0, 0.0))  # extrapolates (weights 1.4375 / -0.4375 per axis)
    assert v == pytest.approx(1.4375 * (1.4375 * src[0, 0] - 0.4375 * src[0, 1])
                              - 0.4375 * (1.4375 * src[1, 0] - 0.4375 * src[1, 1]))


def test_e2e_golden(golden, oracle_net_w0):
    """Whole estimator with the CNN restatement.  The CNN runs on this machine's CPU, so low-order bits of the maps can
    differ from the machine that minted the fixture: 2D joints must agree except documented near-ties (none observed),
    3D joints to 0.05 mm."""
    g = golden("e2e.npz")
    pic = golden("test_pic.npz")["img"]
    clock = _Clock()
    est = prepost.OracleEstimator(oracle_net_w0, [1.0], clock=clock, promotion="numpy")
    clock.q = [1000.0, 1000.004]
    j2, j3 = est(pic)
    assert np.array_equal(j2, g["c1/j2"])
    assert np.max(np.abs(j3 - g["c1/j3"])) < 0.05
    est = prepost.OracleEstimator(oracle_net_w0, [1.0, 0.7], clock=clock, promotion="numpy")
    for k in range(4):
        clock.q = [1000 + k / 30, 1000 + k / 30 + 0.004]
        j2, j3 = est(synth.stream_frame(0, k))
        assert np.max(np.abs(j2 - g["c4/j2"][k])) < 1e-6
        assert np.max(np.abs(j3 - g["c4/j3"][k])) < 0.05


# ------------------------------------------------------------------------------------------------ reference script lines
def test_tracker_update_matches_reference_script_lines(golden):
    """oracle.prepost.tracker_update against run_estimator.py:110-119 executed verbatim (the script's text is stored in
    tests/golden/ref_scripts.npz)."""
    import textwrap
    src = bytes(golden("ref_scripts.npz")["run_estimator.py"]).decode("utf-8").splitlines()
    first = next(i for i, line in enumerate(src) if "y_min = (np.min(joints_2d[:, 0]))" in line)
    body = textwrap.dedent("\n".join(src[first:first + 10]))
    assert "H_img - y" in body
    rng = np.random.default_rng(21)
    for _ in range(200):
        w_img, h_img = int(rng.integers(200, 2000)), int(rng.integers(200, 2000))
        j2 = np.stack([rng.uniform(-20, h_img + 20, 21), rng.uniform(-20, w_img + 20, 21)], axis=1)
        ns = dict(np=np, joints_2d=j2.copy(), W_img=w_img, H_img=h_img)
        exec(body, ns)
        assert prepost.tracker_update(j2, w_img, h_img) == (ns["x"], ns["y"], ns["w"], ns["h"])


def test_tracker_update_known_values():
    j2 = np.zeros((21, 2))
    j2[:, 0] = np.linspace(100.0, 400.0, 21)   # rows
    j2[:, 1] = np.linspace(300.5, 420.25, 21)  # cols
    assert prepost.tracker_update(j2, 960, 540) == (252, 69, 216, 360)


# ------------------------------------------------------------------------------------------------ round-2 fixtures
def test_joint_filter_golden(golden):
    """tests/golden/filter_joint.npz: the reference's VNectEstimator.joint_filter (estimator.py:83-95) called directly,
    dim 2 on a float64 array and dim 3 on a float32 one, irregular timestamps."""
    from tests.golden.make_golden import JF_STEPS, joint_filter_inputs
    g = golden("filter_joint.npz")
    for dim in (2, 3):
        x, t = joint_filter_inputs(dim)
        assert np.array_equal(x, g[f"d{dim}/x"]) and np.array_equal(t, g[f"d{dim}/t"])  # inputs are reproducible
        clock = _Clock()
        est = prepost.OracleEstimator(None, [1.0], clock=clock, promotion="numpy")
        legacy = prepost.OracleEstimator(None, [1.0], clock=_Clock(), promotion="legacy")
        for k in range(JF_STEPS):
            clock.q = [float(t[k])]
            legacy.clock.q = [float(t[k])]
            y = est.joint_filter(x[k].copy(), dim)
            assert y.dtype == g[f"d{dim}/y"].dtype and np.array_equal(y, g[f"d{dim}/y"][k]), (dim, k)
            yl = legacy.joint_filter(x[k].copy(), dim)
            if dim == 2:
                assert np.array_equal(yl, y)
            else:  # numpy-1.x promotion (what the CUDA path implements) vs numpy >= 2: float32 rounding noise only
                assert np.abs(yl.astype(np.float64) - y).max() < 1e-2


def test_video_golden_tracked_loop(golden, oracle_net_w0):
    """tests/golden/video.npz: the first frames of pic/test_video.mp4 through the reference's estimator + the verbatim
    bounding-box lines of run_estimator.py:98-119 (C3).  OracleTracker + OracleEstimator must walk the same boxes."""
    g = golden("video.npz")
    frames, t = g["frames"], g["t"]
    assert frames.shape[1:] == (540, 960, 3) and frames.dtype == np.uint8
    clock = _Clock()
    trk = prepost.OracleTracker(prepost.OracleEstimator(oracle_net_w0, [1.0, 0.7], clock=clock, promotion="numpy"),
                                (0, 0, 960, 540))
    for k in range(6):
        clock.q = [float(t[k]), float(t[k])]
        j2, j3, used = trk(frames[k])
        assert used == tuple(int(v) for v in g["boxes"][k]), k
        assert np.max(np.abs(j2 - g["j2"][k])) < 1e-6
        assert np.max(np.abs(j3 - g["j3"][k])) < 0.05


def test_area2x_partial_blocks_match_cv2():
    """Exact 2x decimation of an odd-sided image (OpenCV switches INTER_LINEAR to INTER_AREA, and the last partial
    block averages only its in-range pixels): the arithmetic squarify_kernel mode 1 implements."""
    import cv2
    rng = np.random.default_rng(3)
    for h, w in ((36, 35), (35, 36), (35, 35), (7, 8)):
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        ref = cv2.resize(img, (0, 0), fx=0.5, fy=0.5, interpolation=cv2.INTER_LINEAR)
        assert np.array_equal(prepost.area2x_u8(img), ref), (h, w)


def test_joints2angles_golden(golden):
    """tests/golden/angles.npz (src/joints2angles.py run unchanged): static angles bit for bit, filtered ones too."""
    g = golden("angles.npz")
    for p, want in zip(g["poses"], g["static"]):
        assert np.array_equal(np.array([float(a) for a in prepost.joints2angles(p)]), want)
    ts = iter(np.repeat(g["t"], 8))
    obj = prepost.OracleJoints2Angles(clock=lambda: float(next(ts)))
    for frame, want in zip(g["traj"], g["filtered"]):
        assert np.array_equal(np.array([float(a) for a in obj(frame)]), want)
