"""The fused post-process kernel (postprocess_kernel, vnect_b200/csrc/prepost_kernels.cuh) against the reference on
every branch it can take.

The kernel is specialised at compile time on the scale count NS and the identity mask (MASK = 1: only scale 0 is a
plain copy; MASK = -1: any other mask, read at run time), picks 8, 4 or 2 heat-map rows per pass from the batch size,
and prunes the exact argmax with a float32 pass whose survivors take one of three paths (one warp: <= 32 quads; one
thread per quad: <= 192; in-place scan of every cell: more).  Each configuration of MATRIX and each map family exists
to reach one of these branches; the CPU tests below prove that the inputs reach them, so the GPU test cannot lose its
reach silently.  The reference is oracle.prepost.OracleEstimator (cv2 where the reference calls cv2) and every
comparison is bit-exact.
"""
import cv2
import numpy as np
import pytest

from oracle import prepost

# (name, scales, box size, frames per call)
MATRIX = [
    ("s2_1f", [1.0, 0.7], 368, 1),                # <2, 1>, 8 rows per pass
    ("s2_13f", [1.0, 0.7], 368, 13),              # <2, 1>, 4 rows
    ("s2_64f", [1.0, 0.7], 368, 64),              # <2, 1>, 2 rows
    ("s1", [1.0], 368, 2),                        # <1, 1>
    ("s1_resized", [0.7], 368, 13),               # <1, -1>, 4 rows: no identity scale, the sums get their own plane
    ("s2_resized", [0.85, 0.7], 368, 1),          # <2, -1>, 8 rows: alias_scale = -1
    ("s2_alias1", [0.7, 1.0], 368, 64),           # <2, -1>, 2 rows: alias_scale = 1, read back from L2
    ("s3_alias1", [0.85, 1.0, 0.7], 368, 2),      # <3, -1>: __ddiv_rn(acc, 3) with a run-time mask
    ("s4", [1, 0.9, 0.8, 0.7], 368, 2),           # <4, 1>: * 0.25 and the four-term tvmax margin
    ("s4_resized0", [0.5, 1.0, 0.6, 0.3], 368, 2),  # <4, -1>: exact 2x, a narrow staged row window for 0.3
    ("copy_0995", [1.0, 0.995], 368, 2),          # 0.995 keeps 46 cells: cv2 copies it (mask 3 -> <2, -1>)
    ("copy_095_box64", [1, 0.95], 64, 2),         # the same at hs = 8: rows per pass >= hs, y_split = 0
    ("copy_0999_box512", [1, 0.999], 512, 2),     # the same at hs = 64: 512 threads, kMaxHm
    ("s3_box448", [1, 0.85, 0.7], 448, 2),        # <3, 1>: __ddiv_rn(acc, 3) at hs = 56
]
STEPS = 3
SCALER, OFFSETS = 0.684, (58, 11)  # offsets = (x, y)

# families assigned per joint, and the survivor path each one exists to reach
FAMILIES = {
    "peak": "one_warp",          # one blob
    "border": "one_warp",        # the blob on an edge or a corner: replicated borders tie exactly
    "ridge": "per_thread",       # a crest of equal cells along part of a row
    "noise": "full_scan",        # a constant plus noise far below the pruning margin
    "constant": "full_scan",     # every sample ties: the first one wins
    "cancel": "one_warp",        # NS >= 3: large per-scale values cancelling to a blob (the tvmax margin)
    "plateau": "one_warp",       # a float32 plateau + ~2e-16 in the other scales: quads flat to a few ulps
    "saddle": "one_warp",        # the same with +-2e-16 in a checkerboard: saddle-shaped quads
    "plateau_wide": "per_thread",  # a wider plateau: the near-flat quads on the per-thread path
    "plateau_full": "full_scan",   # the whole map: the near-flat quads on the in-place scan
}
DEFECT2 = ("plateau", "saddle", "plateau_wide", "plateau_full")
REGIMES = {"one_warp": (1, 32), "per_thread": (33, 192), "full_scan": (193, 1 << 30)}


def identity_mask(scales, hs):
    """Bit i: scale i is a plain copy.  cv2.resize copies when dsize == ssize, i.e. when round(hs / s) == hs."""
    return sum(1 << i for i, s in enumerate(scales) if prepost.cv_round(hs * (1.0 / s)) == hs)


def kernel_key(scales, box):
    """(NS, MASK) of the postprocess_kernel instantiation a scale list launches."""
    return len(scales), 1 if identity_mask(scales, box // 8) == 1 else -1


def rows_per_pass(n_frames):
    return 2 if n_frames >= 48 else 4 if n_frames >= 12 else 8


def families_for(scales, hs):
    """The families a scale list can carry: cancellation needs three scales, near-flat sums two, and an 8 x 8 map has
    too few quads for the per-thread path."""
    ns = len(scales)
    return [f for f in FAMILIES if (f != "cancel" or ns >= 3) and (f not in DEFECT2 or ns >= 2)
            and (FAMILIES[f] != "per_thread" or hs >= 16)]


def joint_family(scales, hs, frame, joint):
    fams = families_for(scales, hs)
    return fams[(joint + 3 * frame) % len(fams)]


# ------------------------------------------------------------------------------------------------ inputs
def _family_planes(fam, scales, hs, rng):
    """Heat-map planes [NS, hs, hs] of one joint."""
    ns = len(scales)
    yy, xx = np.mgrid[0:hs, 0:hs].astype(np.float64)
    out = np.zeros((ns, hs, hs), np.float32)
    if fam in ("peak", "border", "cancel"):
        if fam == "border":
            c = [(0, 0), (0, hs - 1), (hs - 1, 0), (hs - 1, hs - 1), (0, hs // 3), (hs - 1, hs // 2),
                 (hs // 2, 0), (hs // 5, hs - 1)][int(rng.integers(0, 8))]
        else:
            c = rng.uniform(3, hs - 4, 2)
        sig = rng.uniform(1.0, 2.5)
        for i, s in enumerate(scales):  # a shrunken copy per scale, like a real pyramid
            cy, cx = (c[0] - hs / 2) * s + hs / 2, (c[1] - hs / 2) * s + hs / 2
            blob = np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * (sig * s) ** 2))
            out[i] = blob + 0.02 * rng.standard_normal((hs, hs))
        if fam == "cancel":  # +-300-ish per scale, cancelling in the sum: float32 partial sums far above |sum|
            big = rng.uniform(200, 400)
            out[0] += np.float32(big)
            out[1] -= np.float32(big)
            if ns == 4:
                out[2] += np.float32(big * 0.5)
                out[3] -= np.float32(big * 0.5)
    elif fam == "ridge":  # in scale 0, two rows of 1.0 over a run of columns; the other scales are flat
        r, x0 = int(rng.integers(hs // 3, hs // 2)), int(rng.integers(hs // 6, hs // 4))
        width = int(rng.integers(3 * hs // 4, 5 * hs // 6))
        out[0] = 0.2 * rng.random((hs, hs))
        out[0, r:r + 2, x0:x0 + width] = 1.0
        out[1:] = 0.125
    elif fam == "noise":
        out[:] = np.float32(0.3) + (1e-9 * rng.standard_normal((ns, hs, hs))).astype(np.float32)
    elif fam == "constant":
        out[:] = np.float32(-0.25)
    else:  # the near-flat families: a plateau of 0.5 (a power of two: every resize keeps it exact) in scale 0 ...
        out[0] = 0.3 * rng.random((hs, hs))
        if fam == "plateau_full":
            out[0] = 0.5
        else:  # 3 x 3 raw cells, or about 7 x 9 cells after the resize of scale 0
            h, w = (3, 3) if fam != "plateau_wide" else (round(7 * scales[0]), round(9 * scales[0]))
            y, x = rng.integers(hs // 3, hs // 2, 2)
            out[0, y:y + h, x:x + w] = 0.5
        # ... and values of ~2e-16 in the others: the averaged quads then differ by a few float64 ulps
        for i in range(1, ns):
            if fam == "saddle":
                out[i] = 2e-16 * (1 - 2 * ((yy + xx) % 2))
            else:
                out[i] = 2e-16 * rng.standard_normal((hs, hs))
    return out


def frame_maps(name, scales, box, frame, step):
    """(hm, xm, ym, zm) of one frame, each [NS, hs, hs, 21] float32."""
    hs = box // 8
    rng = np.random.default_rng([sum(map(ord, name)), frame, step])
    hm = np.zeros((len(scales), hs, hs, 21), np.float32)
    for j in range(21):
        hm[..., j] = _family_planes(joint_family(scales, hs, frame, j), scales, hs, rng)
    loc = []
    nc = -(-hs // 8)
    for _ in range(3):  # smooth location maps, like oracle.synth
        coarse = rng.uniform(-5, 5, size=(len(scales), nc, nc, 21))
        fine = np.kron(coarse, np.ones((1, 8, 8, 1)))[:, :hs, :hs, :]
        loc.append((fine + 0.05 * rng.standard_normal(fine.shape)).astype(np.float32))
    return (hm, *loc)


def clock_readings(name, n_frames):
    """[STEPS, n_frames] 2D and 3D clock readings: irregular steps, different per stream."""
    rng = np.random.default_rng(sum(map(ord, name)) + 7)
    t2 = 500 + np.cumsum(rng.uniform(0.015, 0.09, (STEPS, n_frames)), axis=0)
    return t2, t2 + rng.uniform(0.001, 0.006, (STEPS, n_frames))


# ------------------------------------------------------------------------------------------------ kernel restatements
def _resized_f32(plane, s, hs):
    """What the kernel's resize tables give for scale s: cv2's resize by 1/s and centre crop, float32."""
    sm = cv2.resize(plane, (0, 0), fx=1.0 / s, fy=1.0 / s, interpolation=cv2.INTER_LINEAR)
    m = sm.shape[0] // 2
    return sm[m - hs // 2:m + hs // 2, m - hs // 2:m + hs // 2]


def _f32_rd(x):
    """__double2float_rd"""
    f = np.float32(x)
    return np.nextafter(f, np.float32(-np.inf)) if float(f) > x else f


def _fmaf(a, b, c):
    # the product of two float32 is exact in float64; the double rounding of the sum is far inside the margin
    return np.float32(np.float64(a) * np.float64(b) + np.float64(c))


def survivor_count(planes, scales):
    """Quads that survive steps B and C of the kernel for one (frame, joint): float32 sums in scale order, the bound
    from the 4 x 4 candidates around the largest cell (the first one here; ties in these families are exact), the
    margin, the cell test and the fmaf cap test."""
    ns, hs = len(scales), planes.shape[1]
    v = [_resized_f32(planes[i], s, hs) for i, s in enumerate(scales)]
    ssum = v[0].copy()
    for t in v[1:]:
        ssum = (ssum + t).astype(np.float32)
    bamax = max(abs(float(ssum.max())), abs(float(ssum.min())))
    if ns > 2:
        bamax = max(bamax, max(float(np.abs(t).max()) for t in v))
    r0, c0 = np.unravel_index(int(np.argmax(ssum)), ssum.shape)

    def cand(k):  # upsample_candidate: (source cell, fraction)
        if k == 0:
            return 0, 0.0
        if k == 2 * hs - 1:
            return hs - 1, 0.0
        return (k - 1) >> 1, (0.9375 if (k - 1) & 1 else 0.0625)

    best = -np.inf
    for a in range(4):
        for b in range(4):
            iy, fy = cand(min(max(2 * r0 - 1, 0) + a, 2 * hs - 1))
            ix, fx = cand(min(max(2 * c0 - 1, 0) + b, 2 * hs - 1))
            iy1, ix1 = min(iy + 1, hs - 1), min(ix + 1, hs - 1)
            s00, s01, s10, s11 = (float(ssum[iy, ix]), float(ssum[iy, ix1]), float(ssum[iy1, ix]),
                                  float(ssum[iy1, ix1]))
            h0 = (s01 - s00) * fx + s00
            h1 = (s11 - s10) * fx + s10
            best = max(best, (h1 - h0) * fy + h0)
    thr = _f32_rd(best - bamax * (1e-6 * ns))
    quads = set()
    for y, x in zip(*np.nonzero(ssum >= thr)):
        for qy in range(max(y - 1, 0), y + 1):
            for qx in range(max(x - 1, 0), x + 1):
                quads.add((qy, qx))
    f = np.float32(0.9375)
    n = 0
    for qy, qx in quads:
        qy1, qx1 = min(qy + 1, hs - 1), min(qx + 1, hs - 1)
        s00, s01, s10, s11 = ssum[qy, qx], ssum[qy, qx1], ssum[qy1, qx], ssum[qy1, qx1]
        h0, h1 = _fmaf(s01 - s00, f, s00), _fmaf(s11 - s10, f, s10)
        cap = max(s00, h0, _fmaf(s10 - s00, f, s00), _fmaf(h1 - h0, f, h0))
        n += bool(cap >= thr)
    return n


def candidate_argmax(hm_avg, box):
    """Step D before the fix: the first maximum over the upsample candidates only (two ends of every x8 segment)."""
    hs = hm_avg.shape[0]
    k = [0] + [d for r in range(hs - 1) for d in (8 * r + 4, 8 * r + 11)] + [8 * (hs - 1) + 4]
    out = np.zeros((hm_avg.shape[2], 2))
    for j in range(hm_avg.shape[2]):
        up = cv2.resize(hm_avg[:, :, j], (0, 0), fx=8, fy=8, interpolation=cv2.INTER_LINEAR)
        i = int(np.argmax(up[np.ix_(k, k)]))
        out[j] = (k[i // len(k)], k[i % len(k)])
    return out


# ------------------------------------------------------------------------------------------------ CPU
def test_identity_mask_follows_cv2_copy_rule():
    m = np.random.default_rng(0).standard_normal((46, 46, 3)).astype(np.float32)
    for s in (1.0, 0.995, 0.99, 0.989, 0.95, 0.7):
        copied = np.array_equal(cv2.resize(m, (0, 0), fx=1 / s, fy=1 / s, interpolation=cv2.INTER_LINEAR), m)
        assert bool(identity_mask([s], 46)) == copied, s
    assert identity_mask([1, 0.95], 8) == 3 and identity_mask([1, 0.9], 8) == 1
    assert identity_mask([1, 0.999], 64) == 3 and identity_mask([1, 0.99], 64) == 1


def test_matrix_reaches_every_instantiation_and_block_shape():
    keys = {kernel_key(s, b) for _, s, b, _ in MATRIX}
    assert keys == {(ns, m) for ns in (1, 2, 3, 4) for m in (1, -1)}
    for rows in (8, 4, 2):
        masks = {kernel_key(s, b)[1] for _, s, b, n in MATRIX if rows_per_pass(n) == rows}
        assert masks == {1, -1}, rows
    masks = {name: identity_mask(s, b // 8) for name, s, b, _ in MATRIX}
    assert masks["s1_resized"] == 0 and masks["s2_resized"] == 0  # the sums in their own plane
    assert masks["s2_alias1"] == 2 and masks["s3_alias1"] == 2  # alias_scale = 1
    assert masks["copy_0995"] == masks["copy_095_box64"] == masks["copy_0999_box512"] == 3
    assert {b // 8 for _, _, b, _ in MATRIX} >= {8, 46, 56, 64}


@pytest.mark.parametrize("case", MATRIX, ids=[c[0] for c in MATRIX])
def test_families_reach_their_survivor_path(case):
    """Survivor counts of the restated steps B and C, with margin for the three plain families."""
    name, scales, box, _ = case
    hm = frame_maps(name, scales, box, 0, 0)[0]
    seen = set()
    for j in range(21):
        fam = joint_family(scales, box // 8, 0, j)
        n = survivor_count(hm[..., j], scales)
        path = FAMILIES[fam]
        if path == "full_scan" and (box // 8) ** 2 <= 192:  # an 8 x 8 map has 64 quads: flat maps take the per-thread path
            path = "per_thread"
        lo, hi = REGIMES[path]
        assert lo <= n <= hi, (fam, j, n)
        if fam in ("peak", "border", "cancel"):
            assert n <= 10, (fam, j, n)
        if fam == "ridge":
            assert 38 <= n <= 160, (fam, j, n)
        if path == "full_scan":
            assert n > 400, (fam, j, n)
        seen.add(fam)
    assert seen == set(families_for(scales, box // 8))


@pytest.mark.parametrize("case", [c for c in MATRIX if len(c[1]) >= 2], ids=[c[0] for c in MATRIX if len(c[1]) >= 2])
def test_near_flat_inputs_defeat_the_candidate_argmax(case):
    """The committed near-flat families really separate the candidate-only reduction from np.argmax over the whole
    cv2 upsample, on every survivor path, so the GPU test would catch a kernel that looks at the candidates only."""
    name, scales, box, n_frames = case
    split = {f: 0 for f in DEFECT2}
    for frame in range(n_frames):
        maps = frame_maps(name, scales, box, frame, 0)
        hm = prepost.average_scales(maps, scales, box)[0]
        want = prepost.extract_2d_joints(hm, box)
        got = candidate_argmax(hm, box)
        for j in np.nonzero((want != got).any(axis=1))[0]:
            fam = joint_family(scales, box // 8, frame, j)
            assert fam in DEFECT2, (frame, j, fam)  # every other family is exact with the candidates alone
            split[fam] += 1
    assert sum(split.values()) >= 1, split
    if n_frames >= 13:  # on each survivor path, a near-flat family split at least once
        assert split["plateau"] + split["saddle"] and split["plateau_wide"] and split["plateau_full"], split


# ------------------------------------------------------------------------------------------------ GPU
class _Clock:
    def __init__(self):
        self.q = []

    def __call__(self):
        return self.q.pop(0)


@pytest.mark.gpu
@pytest.mark.parametrize("case", MATRIX, ids=[c[0] for c in MATRIX])
def test_postprocess_bit_exact_on_every_branch(case):
    from vnect_b200 import VNectEngine
    name, scales, box, n = case
    t2, t3 = clock_readings(name, n)
    clocks = [_Clock() for _ in range(n)]
    refs = [prepost.OracleEstimator(None, scales, clock=clocks[i], promotion="legacy", box_size=box) for i in range(n)]
    img = np.zeros((box, box, 3), np.uint8)
    eng = VNectEngine(False, scales, box_size=box, max_frames=64, max_streams=64)
    try:
        ids = np.arange(n)[::-1].copy()  # every frame its own stream, not in frame order
        for step in range(STEPS):
            per_frame = [frame_maps(name, scales, box, f, step) for f in range(n)]
            batch = tuple(np.concatenate([m[c] for m in per_frame]) for c in range(4))
            j2, j3, raw = eng.postprocess(batch, SCALER, OFFSETS, ids, t2[step], t3[step])
            for f in range(n):
                refs[f].forward = lambda b, m=per_frame[f]: m
                clocks[f].q = [float(t2[step, f]), float(t3[step, f])]
                _, r3 = refs[f](img)
                last = refs[f].last
                r2 = last["joints_2d_box"].copy()
                r2[:, 0] = (r2[:, 0] - OFFSETS[1]) / SCALER
                r2[:, 1] = (r2[:, 1] - OFFSETS[0]) / SCALER
                fams = [joint_family(scales, box // 8, f, j) for j in range(21)]
                bad = np.nonzero((raw[f] != last["joints_2d_raw"].astype(np.int32)).any(axis=1))[0]
                assert bad.size == 0, [(int(j), fams[j], tuple(raw[f, j]), tuple(last["joints_2d_raw"][j]))
                                       for j in bad]
                assert np.array_equal(j2[f], r2), (step, f)
                assert np.array_equal(j3[f], r3), (step, f)
    finally:
        eng.close()


@pytest.mark.gpu
def test_preprocess_copies_a_scale_that_keeps_the_box_size():
    """0.999 * 368 rounds to 368: cv2 copies the box image, the pyramid kernel must too."""
    from vnect_b200 import VNectEngine
    scales = [1.0, 0.999]
    eng = VNectEngine(False, scales, max_frames=1, max_input=(540, 960))
    try:
        img = np.random.default_rng(31).integers(0, 256, (540, 960, 3), dtype=np.uint8)
        got, scaler, offs = eng.preprocess(img)
        ref, rs, ro = prepost.gen_input_batch(img, 368, scales)
        assert (scaler, offs) == (rs, ro)
        assert np.array_equal(ref[0], ref[1])
        assert np.array_equal(got, ref.astype(np.float16).astype(np.float32))
    finally:
        eng.close()
