#!/usr/bin/env python3
"""Mint the golden fixtures of tests/golden/ by running the reference's OWN code.

    VNECT_REFERENCE_ROOT=<checkout of XinArkh/VNect> python tests/golden/make_golden.py

The reference tree is only read.  The reference's ``src/utils.py``, ``src/OneEuroFilter.py`` and ``src/estimator.py``
are imported unchanged through ``oracle.ref_shim``; TensorFlow is replaced by a stub whose ``Session.run`` returns
either seeded synthetic maps (post-processing fixtures, machine independent) or ``oracle.forward.OracleNet`` output
(end-to-end fixtures).  Library versions are recorded in every file.

Fixtures (all small):
  pre.npz     gen_input_batch (estimator.py:70-81): sha256 of the float32 batch + scaler/offsets per case
  post.npz    multi-frame VNectEstimator.__call__ on synthetic maps: joints_2d / joints_3d per frame
  filter.npz  OneEuroFilter on a seeded noisy signal (float64), irregular timestamps
  e2e.npz     VNectEstimator.__call__ with the CNN restatement (W0) on test_pic + synthetic frames
  test_pic.npz  decoded pixels of pic/test_pic.jpg (C1 input; the GPU box has no reference tree)
  filter_joint.npz  VNectEstimator.joint_filter (estimator.py:83-95) called directly: dim 2 (float64) and dim 3 (float32)
  video.npz   first 12 decoded frames of pic/test_video.mp4 (C3 input) + the reference's video loop on them
              (run_estimator.py:98-119 executed verbatim around the reference estimator, CNN restatement W0)

  ref_scripts.npz  the text of the reference's CALLER scripts run_pic.py and run_estimator.py (bytes + sha256): test
              vectors for SURVEY.md T5 -- the scripts are executed unchanged against the drop-in on the GPU box, which
              has no reference tree.  Not product code; nothing under vnect_b200/ reads it.

  angles.npz  src/joints2angles.py run unchanged: the static joints2angles() on seeded 3D joints and the filtered
              Joints2Angles.__call__ over a joint trajectory with scripted clock readings

`python tests/golden/make_golden.py filter_joint video ref_scripts angles` regenerates only the named fixtures.
"""
import hashlib
import os
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_shim, synth  # noqa: E402
from oracle.forward import OracleNet  # noqa: E402
from oracle.weights import make_weights  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
VERSIONS = dict(cv2=cv2.__version__, numpy=np.__version__)

PRE_CASES = [  # (name, H, W, seed, scales)
    ("square368", 368, 368, 11, [1.0, 0.7]),
    ("square368_3s", 368, 368, 12, [1, 0.85, 0.7]),
    ("wide960x540", 540, 960, 13, [1.0, 0.7]),
    ("tall300x200", 300, 200, 14, [1, 0.85, 0.7]),
    ("small100x180", 100, 180, 15, [1.0, 0.7]),
    ("half736", 736, 736, 16, [1.0]),
    ("odd367x251", 367, 251, 17, [1.0, 0.7]),
]
POST_CASES = [  # (name, seed, scales, n_frames, dt pattern)
    ("s2_border", 101, [1.0, 0.7], 6, "regular30"),
    ("s3_default", 102, [1, 0.85, 0.7], 5, "irregular"),
    ("s1_single", 103, [1.0], 4, "regular25"),
    ("s2_interior", 104, [1.0, 0.7], 5, "irregular"),
]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def savez_bzip2(path, **arrays):
    """np.savez_compressed with bzip2 instead of deflate entries (np.load reads either).  The decoded video frames
    shrink to about 60 % of their deflate size, which keeps video.npz well under 1 MB."""
    import zipfile
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_BZIP2) as z:
        for name, a in arrays.items():
            with z.open(name + ".npy", "w", force_zip64=True) as f:
                np.lib.format.write_array(f, np.asanyarray(a), allow_pickle=False)


def timestamps(pattern, n, seed):
    if pattern == "regular30":
        t = 1000 + np.arange(n) / 30.0
    elif pattern == "regular25":
        t = 1000 + np.arange(n) / 25.0
    else:
        t = 1000 + np.cumsum(np.random.default_rng(seed).uniform(0.01, 0.09, n))
    return t, t + 0.004  # 2D-group and 3D-group clock readings


def post_frame_maps(seed, k, scales):
    """Frame k of a synthetic map stream: blob centres drift with k so the filters see motion."""
    return synth.synthetic_maps(seed * 100 + k, len(scales), border_joints=(k % 2 == 0))


JF_STEPS = 7
VIDEO_FRAMES = 12
VIDEO_SCALES = [1.0, 0.7]


def joint_filter_inputs(dim):
    """Seeded joint trajectories for the standalone joint_filter fixture: [JF_STEPS, 21, dim] + irregular timestamps."""
    rng = np.random.default_rng(300 + dim)
    base = rng.uniform(20, 340, (21, dim)) if dim == 2 else rng.uniform(-600, 600, (21, dim))
    x = base[None] + np.cumsum(rng.standard_normal((JF_STEPS, 21, dim)) * 4, axis=0)
    t = 2000 + np.cumsum(rng.uniform(0.012, 0.07, JF_STEPS))
    if dim == 2:
        x = np.rint(x)  # argmax output is integer valued
    return (x.astype(np.float64) if dim == 2 else x.astype(np.float32)), t


def video_timestamps(n):
    return 1000 + np.arange(n) / 25.0  # SURVEY.md section 8d C3: t_k = 1000 + k/25 for both filter groups


def reference_tracker_lines():
    """run_estimator.py:110-119 (the bounding-box update), as source text to be exec'd verbatim."""
    import textwrap
    src = open(os.path.join(ref_shim.REFERENCE_ROOT, "run_estimator.py")).read().splitlines()
    first = next(i for i, line in enumerate(src) if "y_min = (np.min(joints_2d[:, 0]))" in line)
    body = textwrap.dedent("\n".join(src[first:first + 10]))
    assert "H_img - y" in body
    return body


def make_filter_joint(est_mod):
    out = dict(versions=str(VERSIONS))
    for dim in (2, 3):
        est, em = ref_shim.make_reference_estimator(lambda b: None, [1.0])
        x, t = joint_filter_inputs(dim)
        ys = []
        real_time = em.time
        try:
            for k in range(JF_STEPS):
                em.time = ref_shim.ScriptedClock([float(t[k])])
                j = x[k].copy()
                r = est.joint_filter(j, dim=dim)
                assert r is j  # in place, like the reference's callers rely on
                ys.append(j.copy())
        finally:
            em.time = real_time
        out[f"d{dim}/x"], out[f"d{dim}/t"], out[f"d{dim}/y"] = x, t, np.array(ys)
    np.savez_compressed(os.path.join(OUT, "filter_joint.npz"), **out)


def make_video():
    cap = cv2.VideoCapture(os.path.join(ref_shim.REFERENCE_ROOT, "pic", "test_video.mp4"))
    assert cap.isOpened()
    frames = []
    for _ in range(VIDEO_FRAMES):
        ok, f = cap.read()
        assert ok
        frames.append(f)
    frames = np.stack(frames)
    H_img, W_img = frames.shape[1:3]
    net = OracleNet(make_weights("W0"))
    est, em = ref_shim.make_reference_estimator(net, VIDEO_SCALES)
    body = reference_tracker_lines()
    t = video_timestamps(VIDEO_FRAMES)
    x, y, w, h = 0, 0, W_img, H_img  # run_estimator.py:68, no HOG click (C3: fixed initial crop = full frame)
    j2s, j3s, boxes = [], [], []
    for k in range(VIDEO_FRAMES):
        frame = frames[k]
        boxes.append((x, y, w, h))
        frame_cropped = frame[y: y + h, x: x + w, :]            # run_estimator.py:100
        joints_2d, joints_3d = ref_shim.run_reference(est, em, frame_cropped, float(t[k]), float(t[k]))
        joints_2d[:, 0] += y                                    # :104-105
        joints_2d[:, 1] += x
        ns = dict(np=np, joints_2d=joints_2d, W_img=W_img, H_img=H_img)
        exec(body, ns)                                          # :110-119 verbatim
        x, y, w, h = ns["x"], ns["y"], ns["w"], ns["h"]
        j2s.append(joints_2d.copy())
        j3s.append(joints_3d.copy())
    savez_bzip2(os.path.join(OUT, "video.npz"), frames=frames, t=t, j2=np.array(j2s), j3=np.array(j3s),
                boxes=np.array(boxes, np.int32), versions=str(VERSIONS))


REF_SCRIPTS = ("run_pic.py", "run_estimator.py")


def make_ref_scripts():
    out = dict(versions=str(VERSIONS))
    for name in REF_SCRIPTS:
        data = open(os.path.join(ref_shim.REFERENCE_ROOT, name), "rb").read()
        out[name] = np.frombuffer(data, dtype=np.uint8)
        out[name + "/sha256"] = hashlib.sha256(data).hexdigest()
    np.savez_compressed(os.path.join(OUT, "ref_scripts.npz"), **out)


ANGLE_FRAMES = 40


def angle_inputs():
    """Seeded 3D joints (float32 mm, root-relative like the estimator's output) and clock readings: a random pose per
    frame for the static function, plus a smooth trajectory for the filtered call."""
    rng = np.random.default_rng(77)
    poses = rng.uniform(-600, 600, (ANGLE_FRAMES, 21, 3)).astype(np.float32)
    start = rng.uniform(-500, 500, (21, 3))
    traj = (start[None] + np.cumsum(rng.standard_normal((ANGLE_FRAMES, 21, 3)) * 6, axis=0)).astype(np.float32)
    t = 3000 + np.cumsum(rng.uniform(0.006, 0.05, ANGLE_FRAMES))
    return poses, traj, t


def make_angles():
    import contextlib
    import importlib
    import io
    ref_shim.load_reference_modules()
    j2a = importlib.import_module("joints2angles")
    poses, traj, t = angle_inputs()
    static = np.array([[float(a) for a in j2a.Joints2Angles.joints2angles(p)] for p in poses])
    with contextlib.redirect_stdout(io.StringIO()):
        obj = j2a.Joints2Angles()
        real = j2a.time
        filtered = []
        try:
            for k in range(ANGLE_FRAMES):
                j2a.time = ref_shim.ScriptedClock([float(t[k])] * 8)   # one time.time() per angle (joints2angles.py:49)
                filtered.append([float(a) for a in obj(traj[k])])
        finally:
            j2a.time = real
    np.savez_compressed(os.path.join(OUT, "angles.npz"), poses=poses, traj=traj, t=t, static=static,
                        filtered=np.array(filtered), versions=str(VERSIONS))


def main():
    assert ref_shim.reference_available(), "set VNECT_REFERENCE_ROOT to a checkout of XinArkh/VNect"
    utils, oef, est_mod = ref_shim.load_reference_modules()
    only = set(sys.argv[1:])
    if only:
        if "filter_joint" in only:
            make_filter_joint(est_mod)
        if "video" in only:
            make_video()
        if "ref_scripts" in only:
            make_ref_scripts()
        if "angles" in only:
            make_angles()
        return
    make_filter_joint(est_mod)
    make_video()
    make_ref_scripts()
    make_angles()

    # ---- pre.npz
    pre = dict(versions=str(VERSIONS))
    for name, h, w, seed, scales in PRE_CASES:
        img = np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
        batch, scaler, (ox, oy) = est_mod.VNectEstimator.gen_input_batch(img, 368, scales)
        pre[name + "/sha"] = sha(batch)
        pre[name + "/meta"] = np.array([scaler, ox, oy], np.float64)
        pre[name + "/sample"] = batch[:, ::37, ::41, :].copy()
    np.savez_compressed(os.path.join(OUT, "pre.npz"), **pre)

    # ---- filter.npz
    rng = np.random.default_rng(5)
    n = 200
    t = 10.0 + np.cumsum(rng.uniform(0.005, 0.08, n))
    sig = np.sin(t * 3.0) * 50 + rng.standard_normal(n) * 2
    f2 = oef.OneEuroFilter(freq=30, mincutoff=1.7, beta=0.3, dcutoff=0.4)
    f3 = oef.OneEuroFilter(freq=30, mincutoff=0.8, beta=0.4, dcutoff=0.4)
    np.savez_compressed(os.path.join(OUT, "filter.npz"), t=t, x=sig,
                        y2=np.array([f2(float(x), float(tt)) for x, tt in zip(sig, t)]),
                        y3=np.array([f3(float(x), float(tt)) for x, tt in zip(sig, t)]), versions=str(VERSIONS))

    # ---- post.npz
    post = dict(versions=str(VERSIONS))
    for name, seed, scales, nf, pat in POST_CASES:
        state = {}
        est, em = ref_shim.make_reference_estimator(lambda batch: state["maps"], scales)
        t2, t3 = timestamps(pat, nf, seed)
        img = np.zeros((368, 368, 3), np.uint8)
        j2s, j3s = [], []
        for k in range(nf):
            state["maps"] = post_frame_maps(seed, k, scales)
            j2, j3 = ref_shim.run_reference(est, em, img, float(t2[k]), float(t3[k]))
            j2s.append(j2.copy())
            j3s.append(j3.copy())
        post[name + "/j2"] = np.array(j2s)
        post[name + "/j3"] = np.array(j3s)
        post[name + "/t2"] = t2
        post[name + "/t3"] = t3
    np.savez_compressed(os.path.join(OUT, "post.npz"), **post)

    # ---- test_pic.npz + e2e.npz
    pic = cv2.imread(os.path.join(ref_shim.REFERENCE_ROOT, "pic", "test_pic.jpg"))
    np.savez_compressed(os.path.join(OUT, "test_pic.npz"), img=pic)
    net = OracleNet(make_weights("W0"))
    e2e = dict(versions=str(VERSIONS))
    est, em = ref_shim.make_reference_estimator(net, [1.0])  # C1: run_pic-like, single scale
    j2, j3 = ref_shim.run_reference(est, em, pic, 1000.0, 1000.004)
    e2e["c1/j2"], e2e["c1/j3"] = j2, j3
    est, em = ref_shim.make_reference_estimator(net, [1.0, 0.7])  # C2-like: independent frames, fresh filters each
    for i in range(3):
        est, em = ref_shim.make_reference_estimator(net, [1.0, 0.7])
        j2, j3 = ref_shim.run_reference(est, em, synth.frame_c2(i), 1000.0, 1000.004)
        e2e[f"c2_{i}/j2"], e2e[f"c2_{i}/j3"] = j2, j3
    est, em = ref_shim.make_reference_estimator(net, [1.0, 0.7])  # C4-like: one stream, 4 frames, filters live
    j2s, j3s = [], []
    for k in range(4):
        j2, j3 = ref_shim.run_reference(est, em, synth.stream_frame(0, k), 1000 + k / 30, 1000 + k / 30 + 0.004)
        j2s.append(j2.copy())
        j3s.append(j3.copy())
    e2e["c4/j2"], e2e["c4/j3"] = np.array(j2s), np.array(j3s)
    np.savez_compressed(os.path.join(OUT, "e2e.npz"), **e2e)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
