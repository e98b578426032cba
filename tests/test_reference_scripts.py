"""SURVEY.md T5: the reference's own run scripts, executed UNCHANGED, against the drop-in.

The scripts' text comes from tests/golden/ref_scripts.npz (minted from the reference checkout by make_golden.py), so no
reference tree is needed.  A working directory is laid out like the reference checkout:

    src/__init__.py
    src/estimator.py   <- the binding under test: on a GPU machine the 4-line block of INTEGRATION.md section 1,
                          parsed out of that file; on a CPU box an oracle-backed stand-in (harness self-check)
    src/hog_box.py     <- re-exports the headless HOGBox replacement (vnect_b200/hog_box.py)
    src/utils.py       <- the only two helpers the scripts call outside drawing: img_scale (utils.py:13-21) + drawing no-ops
    pic/test_pic.jpg   <- tests/golden/test_pic.npz, stored losslessly

tests/script_runner.py stubs the OpenCV GUI, serves the video frames of tests/golden/video.npz, scripts the clock and
records what the script hands to its drawing code.  The test then walks the same frames with the oracle
(OracleEstimator + the tracker restatement of run_estimator.py:110-119) using the very timestamps the estimator saw.
"""
import os
import re
import subprocess
import sys

import cv2
import numpy as np
import pytest

from oracle import prepost, ref_shim
from oracle.compare import StreamComparer

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

UTILS_STUB = '''\
import cv2


def img_scale(img, scale):
    return cv2.resize(img, (0, 0), fx=scale, fy=scale, interpolation=cv2.INTER_LINEAR)


def draw_limbs_2d(img, joints_2d, limb_parents, rect):
    return img


def draw_limbs_3d(joints_3d, joint_parents):
    pass


def plot_3d_init(joint_parents, joints_iter_gen):
    pass
'''

HOG_BINDING = '''\
import os, sys
sys.path.insert(0, os.environ.get("VNECT_B200_HOME", "/opt/vnect_b200"))
from vnect_b200.hog_box import HOGBox  # noqa: F401
'''

STANDIN_BINDING = '''\
import os, sys
sys.path.insert(0, os.environ["VNECT_B200_HOME"])
from tests.cpu_standin import VNectEstimator  # noqa: F401
'''


def integration_binding():
    """The estimator binding exactly as INTEGRATION.md section 1 prints it."""
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    m = re.search(r"## 1\..*?```python\n(.*?)```", text, flags=re.S)
    assert m and "from vnect_b200 import VNectEstimator" in m.group(1)
    return m.group(1)


def script_text(name):
    g = np.load(os.path.join(GOLDEN, "ref_scripts.npz"))
    return bytes(g[name]).decode("utf-8")


def lay_out(tmp_path, estimator_binding):
    (tmp_path / "src").mkdir()
    (tmp_path / "pic").mkdir()
    (tmp_path / "src" / "__init__.py").write_text("")
    (tmp_path / "src" / "estimator.py").write_text(estimator_binding)
    (tmp_path / "src" / "hog_box.py").write_text(HOG_BINDING)
    (tmp_path / "src" / "utils.py").write_text(UTILS_STUB)
    pic = np.load(os.path.join(GOLDEN, "test_pic.npz"))["img"]
    ok, png = cv2.imencode(".png", pic)  # lossless; cv2.imread sniffs the format from the content, not the suffix
    assert ok
    (tmp_path / "pic" / "test_pic.jpg").write_bytes(png.tobytes())
    for name in ("run_pic.py", "run_estimator.py"):
        (tmp_path / name).write_text(script_text(name))
    return pic


def run_script(tmp_path, name, max_iter):
    out = tmp_path / (name + ".npz")
    env = dict(os.environ, VNECT_B200_HOME=ROOT, VNECT_B200_WEIGHTS="random:W0",
               VNECT_TEST_VIDEO_NPZ=os.path.join(GOLDEN, "video.npz"), PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "script_runner.py"), str(tmp_path / name),
                        str(tmp_path), str(out), str(max_iter)], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return np.load(out), r.stdout


def estimator_clock(res, module_suffix):
    """Timestamps consumed inside the estimator's module, in call order."""
    return [float(t) for t, who in zip(res["clock_t"], res["clock_who"]) if str(who).endswith(module_suffix)]


class _Clock:
    def __init__(self, q):
        self.q = list(q)

    def __call__(self):
        return self.q.pop(0)


def check_run_pic(res, stdout, pic, net, module_suffix, exact):
    """run_pic.py: HOG box on the picture (hog.clicked = True), crop, estimate, shift to picture coordinates."""
    from vnect_b200.hog_box import HOGBox
    assert "Initializing VNect Estimator" in stdout and "FPS:" in stdout and "Initializing HOGBox" in stdout
    hog = HOGBox(verbose=False)
    hog.clicked = True
    _, rect = hog(pic.copy())
    x, y, w, h = (int(v) for v in rect)
    assert tuple(res["rect"][0]) == (x, y, w, h)
    ts = estimator_clock(res, module_suffix)
    assert len(ts) == 4                                    # estimator.py:98, :84 twice, :141
    ref = prepost.OracleEstimator(net, [1, 0.85, 0.7], clock=_Clock(ts[1:3]))   # the class default scales (:32)
    r2, r3 = ref(np.ascontiguousarray(pic[y:y + h, x:x + w, :]))
    r2[:, 0] += y
    r2[:, 1] += x
    j2, j3 = res["j2"][0], res["j3"][0]
    assert j2.shape == (21, 2) and j3.shape == (21, 3)
    return ref, r2, r3, j2, j3


def walk_run_estimator(res, net, module_suffix, exact):
    """run_estimator.py: HOG loop until a box is chosen (:66-83), then per frame crop / estimate / shift / update the box
    (:98-119).  Replays the same frames through the oracle tracker with the timestamps the estimator saw; returns the set
    of joints that ever differed (near-ties on the CUDA path; must be empty when `exact`)."""
    from vnect_b200.hog_box import HOGBox
    frames = np.load(os.path.join(GOLDEN, "video.npz"))["frames"]
    hog = HOGBox(verbose=False)
    k = 0
    while True:
        choose, rect = hog(frames[k].copy())
        k += 1
        if choose:
            break
    # the main loop starts with the NEXT frame (run_estimator.py:95)
    ts = estimator_clock(res, module_suffix)
    n = len(res["j2"])
    assert n >= 3 and len(ts) == 4 * n          # estimator.py:98, :84 twice, :141 per frame
    clock = _Clock([])
    trk = prepost.OracleTracker(prepost.OracleEstimator(net, [1, 0.85, 0.7], clock=clock), rect)  # default scales (:32)
    tainted = set()
    for i in range(n):
        clock.q = ts[4 * i + 1:4 * i + 3]
        r2, r3, used = trk(frames[k + i])
        assert tuple(res["rect"][i]) == used, i
        same = np.all(res["j2"][i] == r2, axis=1)
        newly = set(np.nonzero(~same)[0].tolist()) - tainted
        if exact:
            assert not newly, (i, newly)
        assert len(newly) <= 2, (i, newly)
        tainted |= newly
        if tainted:  # keep the two loops on the same box so later frames stay comparable
            trk.rect = prepost.tracker_update(res["j2"][i], frames.shape[2], frames.shape[1])
    return tainted


# ------------------------------------------------------------------------------------------------ fixture provenance
# sha256 of the reference's run_pic.py and run_estimator.py, taken when ref_scripts.npz was minted from them
REF_SCRIPT_SHA256 = {
    "run_pic.py": "da6ec6c628b3fbd819185ebe29accc606791575fddb07f4ec04247d18efd7970",
    "run_estimator.py": "db3835a346ba0d9cdf4cf16b583c5b72a5d174997da6defeb2d38b8c1aaad4b1",
}


def test_script_fixture_is_the_unmodified_reference_text():
    """The stored script text hashes to what the reference files hashed to (and equals them when the tree is present)."""
    import hashlib
    g = np.load(os.path.join(GOLDEN, "ref_scripts.npz"))
    for name, digest in REF_SCRIPT_SHA256.items():
        data = bytes(g[name])
        assert hashlib.sha256(data).hexdigest() == digest == str(g[name + "/sha256"])
        if ref_shim.reference_available():
            assert open(os.path.join(ref_shim.REFERENCE_ROOT, name), "rb").read() == data


def test_hogbox_cal_rect_matches_reference_arithmetic():
    """vnect_b200.hog_box.HOGBox.cal_rect against src/hog_box.py:47-58 (live when the tree is present, and on known
    values everywhere)."""
    from vnect_b200.hog_box import HOGBox
    assert [int(v) for v in HOGBox.cal_rect((300, 100, 120, 260), 540, 960)] == [108, 46, 504, 368]
    assert [int(v) for v in HOGBox.cal_rect((10, 5, 50, 90), 540, 960)] == [0, 0, 252, 149]
    assert [int(v) for v in HOGBox.cal_rect((800, 400, 150, 130), 540, 960)] == [608, 346, 352, 194]
    if ref_shim.reference_available():
        ref_shim.load_reference_modules()
        src = open(os.path.join(ref_shim.REFERENCE_ROOT, "src", "hog_box.py")).read()
        body = src[src.index("    def cal_rect(rect, H, W):"):src.index("    @staticmethod\n    def draw_rect")]
        import textwrap
        ns = {"np": np}
        exec(textwrap.dedent(body), ns)
        rng = np.random.default_rng(5)
        for _ in range(300):
            H, W = int(rng.integers(100, 1200)), int(rng.integers(100, 2000))
            x, y = int(rng.integers(0, W - 10)), int(rng.integers(0, H - 10))
            w, h = int(rng.integers(5, W - x)), int(rng.integers(5, H - y))
            assert [int(v) for v in HOGBox.cal_rect((x, y, w, h), H, W)] == [int(v) for v in ns["cal_rect"]((x, y, w, h), H, W)]


# ------------------------------------------------------------------------------------------------ CPU: harness self-check
def test_scripts_run_unchanged_with_cpu_standin(tmp_path, oracle_net_w0):
    """No GPU needed: the same harness with an oracle-backed estimator behind src/estimator.py.  Proves the scripts
    execute unchanged in the laid-out tree, that the headless HOGBox satisfies both scripts' loops, and that the
    bookkeeping the GPU variant relies on (clock log, recorded joints, rect walk) is right."""
    pic = lay_out(tmp_path, STANDIN_BINDING)
    res, out = run_script(tmp_path, "run_pic.py", 100)
    assert str(res["estimator_class"]) == "tests.cpu_standin.VNectEstimator"
    ref, r2, r3, j2, j3 = check_run_pic(res, out, pic, oracle_net_w0, "tests.cpu_standin", True)
    assert np.array_equal(j2, r2) and np.array_equal(j3, r3)
    res, out = run_script(tmp_path, "run_estimator.py", 5)
    assert not walk_run_estimator(res, oracle_net_w0, "tests.cpu_standin", True)


# ------------------------------------------------------------------------------------------------ GPU: the real thing
@pytest.mark.gpu
def test_scripts_run_unchanged_against_the_dropin(tmp_path, oracle_net_w0):
    """run_pic.py and 5 frames of run_estimator.py, unchanged, with src/estimator.py = the binding INTEGRATION.md
    prints: joints handed to the drawing code equal the oracle's except proven near-ties (2D exact, 3D < 1 mm)."""
    pic = lay_out(tmp_path, integration_binding())
    res, out = run_script(tmp_path, "run_pic.py", 100)
    assert str(res["estimator_class"]) == "vnect_b200.estimator.VNectEstimator"
    ref, r2, r3, j2, j3 = check_run_pic(res, out, pic, oracle_net_w0, "vnect_b200.estimator", False)
    # no raw-argmax tap through the script: untainted joints are those whose 2D result is bit-identical
    same = np.all(j2 == r2, axis=1)
    assert same.sum() >= 17, "more than 4 joints differ on the C1 picture"
    up_bound_checked = 0
    hm = ref.last["hm_avg"]
    x, y = int(res["rect"][0][0]), int(res["rect"][0][1])
    scaler, (ox, oy) = ref.last["scaler"], ref.last["offsets"]
    for j in np.nonzero(~same)[0]:   # first frame: filters pass through, so box coordinates can be reconstructed
        row = int(round((j2[j, 0] - y) * scaler + oy))
        col = int(round((j2[j, 1] - x) * scaler + ox))
        up = cv2.resize(hm[:, :, j], (0, 0), fx=8, fy=8, interpolation=cv2.INTER_LINEAR)
        gap = float(up.max() - up[row, col])
        print(f"run_pic near-tie joint {j}: gap {gap:.3e} bound {3e-3 * np.abs(hm).max():.3e}")
        assert gap <= 3e-3 * np.abs(hm).max()
        up_bound_checked += 1
    if same[14]:
        assert np.abs(j3[same].astype(np.float64) - r3[same]).max() < 1.0

    res, out = run_script(tmp_path, "run_estimator.py", 6)
    tainted = walk_run_estimator(res, oracle_net_w0, "vnect_b200.estimator", False)
    print("run_estimator.py: joints that met a near-tie:", sorted(tainted))
    assert len(tainted) <= 3
