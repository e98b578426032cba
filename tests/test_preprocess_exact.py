"""The network input every pre-processing path writes, read back as the stem reads it and compared with cv2 bit for bit.

Pre-processing is integer and table work (squarify_kernel, pyramid_kernel and the geometry kernels in
vnect_b200/csrc/prepost_kernels.cuh): it must equal estimator.gen_input_batch (cv2.resize, then float32 / 255 - 0.4,
then fp16) exactly.  `VNectEngine.stem_input` returns the raw fp16 bits of x1, the parity-split, zero-padded NHWC4
buffer the stem reads (DESIGN.md §2), so the check covers the picture, the black surround of the shrunken scales, the
TF-SAME zero border and the 4th channel.

The expected buffer is built on the CPU from cv2 through oracle.prepost.gen_input_batch: YUV frames go through
cv2.cvtColor first, tracked frames are cropped numpy-style with the box the call reports (which must equal the seeded
box clipped as `clip_box` clips it).  Each case of CASES exists for the branches it reaches; `case_branches` derives
them from a restatement of the host geometry (squarify_geometry / make_frame_geom, the alias rule, the pyramid's R,
pad0, row tables and staged rows, the `aligned` flag), and the CPU tests check that every branch of BRANCHES is
reached and that no case can be dropped without losing one.  Every case makes three calls with fresh frames (the
third replays a captured graph) and checks the input of each.
"""
import time

import cv2
import numpy as np
import pytest

from oracle import prepost

PYR_ROWS, PYR_THREADS, PYR_MAX_SMEM = 8, 256, 160 * 1024  # kPyrRows, kPyrThreads, kPyrMaxSmem
CALLS = 3

# ------------------------------------------------------------------------------------------------ host restatement


def squarify_geometry(S, h, w):
    """squarify_geometry (host) / make_frame_geom (device) for an h x w picture: (scaler, dh, dw, off_x, off_y, mode)."""
    scaler = S / max(h, w)
    dw, dh = prepost.cv_round(w * scaler), prepost.cv_round(h * scaler)
    off_x = off_y = 0
    if dh > dw:
        off_x = S // 2 - dw // 2
    else:
        off_y = S // 2 - dh // 2
    return scaler, dh, dw, off_x, off_y, 1 if 1.0 / scaler == 2.0 else 0


def clip_box(box, fh, fw):
    """clip_box: numpy slicing frame[y:y+h, x:x+w] of an FH x FW frame, at least 2 x 2."""
    x, y, w, h = box
    x = min(max(x, 0), fw - 2)
    y = min(max(y, 0), fh - 2)
    return x, y, max(min(w, fw - x), 2), max(min(h, fh - y), 2)


def pyramid_scale(S, s):
    """The pyramid's per-scale plan: R, pad0, the row table (r0, r1) and the most source rows one block stages."""
    R = prepost.cv_round(S * s) if s < 1 else S
    plan = dict(R=R, pad0=(S - R) // 2, rows=1, r0=None, r1=None)
    if R != S:
        iy, _ = prepost.linear_coords(R, S, 1.0 / s, False)
        r0, r1 = np.clip(iy, 0, S - 1), np.clip(iy + 1, 0, S - 1)
        y0 = np.arange(R)
        y1 = np.minimum(y0 + PYR_ROWS, R) - 1
        plan.update(r0=r0, r1=r1, rows=int((r1[y1] - r0[y0] + 1).max()))
    return plan


def staged_rows(S, scales):
    """pyr_src_rows: what vnect_create checks against the 160 KB of dynamic shared memory."""
    return max(pyramid_scale(S, s)["rows"] for s in scales)


def magic(d):
    """floor(2^32 / d) + 1: the r_magic / q_magic divisors."""
    return (1 << 32) // d + 1


# ------------------------------------------------------------------------------------------------ reference buffer


def stem_layout(batch_f32):
    """float32 [n, S, S, 3] network input -> the fp16 bits of x1, uint16 [n, 2, S/2 + 3, (S + 6) * 4]: pixel (y, x)
    at padded (y + 2, x + 2) in parity plane (y + 2) & 1, row (y + 2) >> 1; channel 3 and the border are zero."""
    n, S = batch_f32.shape[:2]
    P = np.zeros((n, S + 6, S + 6, 4), np.uint16)
    P[:, 2:S + 2, 2:S + 2, :3] = batch_f32.astype(np.float16).view(np.uint16)
    return P.reshape(n, S // 2 + 3, 2, (S + 6) * 4).transpose(0, 2, 1, 3).copy()


def expected_input(pictures, S, scales):
    """The x1 buffer of a call whose frames are the BGR `pictures` (already converted and cropped)."""
    return np.concatenate([stem_layout(prepost.gen_input_batch(p, S, scales)[0]) for p in pictures])


def region_map(S, scales):
    """Per forward of one frame, every element of x1 by region: 0 picture, 1 surround, 2 zero border, 3 4th channel."""
    out = []
    pr = np.arange(S + 6)[:, None, None]
    pc = np.arange(S + 6)[None, :, None]
    c = np.arange(4)[None, None, :]
    for s in scales:
        p = pyramid_scale(S, s)
        lo, hi = p["pad0"] + 2, p["pad0"] + 2 + p["R"]
        border = (pr < 2) | (pr >= S + 2) | (pc < 2) | (pc >= S + 2)
        pic = (pr >= lo) & (pr < hi) & (pc >= lo) & (pc < hi)
        reg = np.where(border, 2, np.where(c == 3, 3, np.where(pic, 0, 1))).astype(np.int8)
        out.append(reg.reshape(S // 2 + 3, 2, (S + 6) * 4).transpose(1, 0, 2))
    return np.stack(out)


REGIONS = ("picture", "surround", "zero border", "4th channel")


def diff_report(got, want, S, scales):
    """None when the bits are equal; otherwise the first differing (forward, y, x, c) in image coordinates and the
    count of differing elements per region."""
    if got.shape == want.shape and np.array_equal(got, want):
        return None
    if got.shape != want.shape:
        return f"shape {got.shape} != {want.shape}"
    bad = got != want
    regs = region_map(S, scales)
    counts = {}
    for k, name in enumerate(REGIONS):
        counts[name] = int(sum((bad[f] & (regs[f % len(scales)] == k)).sum() for f in range(bad.shape[0])))
    f, par, r, col = (int(v) for v in np.argwhere(bad)[0])
    y, x, c = 2 * r + par - 2, col // 4 - 2, col % 4
    return (f"{int(bad.sum())} elements differ; first at forward {f} (scale {scales[f % len(scales)]}), y {y}, x {x}, "
            f"c {c}: got 0x{int(got[f, par, r, col]):04x}, want 0x{int(want[f, par, r, col]):04x}; by region {counts}")


# ------------------------------------------------------------------------------------------------ the matrix
# engines: weights ("random:W0", or False for pre-processing only), box, scales, max_frames, max_input
ENGINES = {
    "w0_368": ("random:W0", 368, [1.0, 0.7], 3, (736, 960)),
    "pre_448": (False, 448, [1.0, 0.55], 2, (540, 960)),
    "pre_64": (False, 64, [1.0, 0.7, 0.5, 0.3], 2, (300, 500)),
    "pre_400": (False, 400, [1.0, 0.85], 2, (540, 960)),
    "pre_512": (False, 512, [1.0, 0.999], 1, (512, 512)),
    "pre_368_copy": (False, 368, [1.0, 0.999], 1, (540, 960)),
    "pre_512_min": (False, 512, [1.0, 0.0898], 1, (540, 960)),
}

# entry point -> (where the frames are, frame table, tracked)
ENTRIES = {
    "estimate": ("host", False, False), "submit0": ("host", False, False), "submit1": ("host", False, False),
    "estimate_device": ("device", False, False), "track": ("host", False, True),
    "estimate_frames": ("host", True, False), "submit_frames": ("host", True, False),
    "estimate_device_frames": ("device", True, False), "track_frames": ("host", True, True),
    "submit_track_frames": ("host", True, True), "track_device_frames": ("device", True, True),
    "preprocess": ("host", False, False),
}

# name, engine, entry point, format, frames: (H, W) of each (full frames when tracked), extra:
#   boxes: the seeded (x, y, w, h) per frame; dev: (byte offset of the first frame, pitch - 3W) of aliased device
#   BGR frames; padded: a decoder surface (luma pitch > W, chroma plane at an aligned offset)
CASES = [
    ("estimate_bgr_shrink", "w0_368", "estimate", "bgr", [(540, 960)] * 2, {}),
    ("submit0_bgr_enlarge", "w0_368", "submit0", "bgr", [(101, 97)], {}),
    ("submit1_i420_unit", "w0_368", "submit1", "i420", [(368, 200)] * 2, {}),
    ("device_alias_0", "w0_368", "estimate_device", "bgr", [(368, 368)] * 2, {"dev": (0, 0)}),
    ("device_alias_1", "w0_368", "estimate_device", "bgr", [(368, 368)] * 2, {"dev": (1, 1)}),
    ("device_alias_2", "w0_368", "estimate_device", "bgr", [(368, 368)], {"dev": (2, 2)}),
    ("device_nv12_surface", "w0_368", "estimate_device", "nv12", [(736, 736)] * 2, {"padded": True}),
    ("track_bgr", "w0_368", "track", "bgr", [(480, 640)] * 2, {"boxes": [(31, 17, 201, 333), (500, 300, 250, 260)]}),
    ("track_i420", "w0_368", "track", "i420", [(480, 640)] * 2, {"boxes": [(33, 45, 161, 299), (700, 500, 60, 60)]}),
    ("frames_bgr_partial", "w0_368", "estimate_frames", "bgr", [(736, 735), (735, 736), (2, 2)], {}),
    ("submit_frames_nv12", "w0_368", "submit_frames", "nv12", [(540, 960), (2, 2)], {}),
    ("device_frames_i420", "w0_368", "estimate_device_frames", "i420", [(480, 640), (2, 2)], {}),
    ("track_frames_bgr", "w0_368", "track_frames", "bgr", [(480, 640), (600, 800)],
     {"boxes": [(101, 51, 300, 220), (560, 590, 400, 300)]}),
    ("submit_track_frames_nv12", "w0_368", "submit_track_frames", "nv12", [(480, 640), (600, 800)],
     {"boxes": [(7, 9, 333, 271), (700, 550, 150, 90)]}),
    ("track_device_frames_i420", "w0_368", "track_device_frames", "i420", [(480, 640), (600, 800)],
     {"boxes": [(900, 700, 50, 50), (77, 131, 389, 247)]}),
    ("pre_448_r246", "pre_448", "preprocess", "bgr", [(300, 500)] * 2, {}),
    ("pre_64_four_scales", "pre_64", "preprocess", "bgr", [(300, 500)] * 2, {}),
    ("pre_400_qpr100", "pre_400", "preprocess", "bgr", [(400, 400)] * 2, {}),
    ("pre_512_r511", "pre_512", "preprocess", "bgr", [(512, 512)], {}),
    ("pre_368_copy", "pre_368_copy", "preprocess", "bgr", [(540, 960)], {}),
    ("pre_512_min_scale", "pre_512_min", "preprocess", "bgr", [(540, 960)], {}),
]

BRANCHES = {
    # squarify_kernel instantiations, with and without per-frame geometry
    "squarify<BgrSrc>", "squarify<BgrSrc> tracked", "squarify<Yuv420Src>", "squarify<Yuv420Src> tracked",
    "squarify<FrameTableSrc<BgrSrc>>", "squarify<FrameTableSrc<BgrSrc>> tracked",
    "squarify<FrameTableSrc<Yuv420Src>>", "squarify<FrameTableSrc<Yuv420Src>> tracked",
    "format nv12", "format i420",
    # squarify geometry
    "mode 0 shrink", "mode 0 enlarge", "mode 0 unit scale, short side smaller", "placement off_x", "placement off_y",
    "mode 1 full blocks", "mode 1 partial column", "mode 1 partial row",
    # YUV layouts and tracked boxes
    "yuv padded surface", "yuv crop odd x", "yuv crop odd y", "box partly outside", "box clipped to 2x2",
    # entry points
    *(f"entry {e}" for e in ENTRIES),
    # pyramid, scale-1 path
    "scale 1 from d_sq", "scale 1 aliased host-staged", "scale 1 aliased device +0, pitch 3S",
    "scale 1 aliased device +1, pitch 3S+1", "scale 1 aliased device +2, pitch 3S+2", "scale 1 at S / 4 = 100 (box 400)",
    # pyramid, shrunken path
    "R > 256", "128 < R <= 256", "R < 128", "R odd", "R even", "pad0 % 8 != 0", "blocks wholly in the surround",
    "four scales", "scale 0.5 (cv2 INTER_AREA)", "pad0 = 0", "R == S copied", "largest staged-row count",
    "byte-wise loads, shrunken path",
}


def _picture_branches(S, h, w):
    _, dh, dw, _, _, mode = squarify_geometry(S, h, w)
    out = {"placement off_x" if dh > dw else "placement off_y"} if dh != dw else set()
    if mode == 1:
        out.add("mode 1 full blocks" if h % 2 == 0 and w % 2 == 0 else
                "mode 1 partial column" if w % 2 else "mode 1 partial row")
    else:
        sc = S / max(h, w)
        out.add("mode 0 shrink" if sc < 1 else "mode 0 enlarge" if sc > 1 else
                "mode 0 unit scale, short side smaller" if min(h, w) < S else "mode 0 unit scale, square")
    return out


def case_pictures(case):
    """(H, W) of the picture each frame's squarify resizes (the clipped crop when tracked) and each clipped box."""
    _, _, entry, _, frames, extra = case
    tracked = ENTRIES[entry][2]
    boxes = [clip_box(b, fh, fw) for b, (fh, fw) in zip(extra["boxes"], frames)] if tracked else None
    pics = [(b[3], b[2]) for b in boxes] if tracked else list(frames)
    return pics, boxes


def case_branches(case):
    name, eng, entry, fmt, frames, extra = case
    _, S, scales, _, _ = ENGINES[eng]
    where, table, tracked = ENTRIES[entry]
    pics, boxes = case_pictures(case)
    out = {f"entry {entry}"}
    if fmt != "bgr":
        out.add(f"format {fmt}")
    alias = fmt == "bgr" and not table and not tracked and all(hw == (S, S) for hw in frames)
    if not alias:
        src = "BgrSrc" if fmt == "bgr" else "Yuv420Src"
        out.add(f"squarify<{f'FrameTableSrc<{src}>' if table else src}>{' tracked' if tracked else ''}")
        for h, w in pics:
            out |= _picture_branches(S, h, w)
    if fmt != "bgr" and extra.get("padded"):
        out.add("yuv padded surface")
    if tracked:
        for (x, y, w, h), seed, (fh, fw) in zip(boxes, extra["boxes"], frames):
            if fmt != "bgr":
                out |= {"yuv crop odd x"} if x % 2 else set()
                out |= {"yuv crop odd y"} if y % 2 else set()
            sx, sy, sw, sh = seed
            if sx < 0 or sy < 0 or sx + sw > fw or sy + sh > fh:
                out.add("box partly outside")
            if (w, h) == (2, 2):
                out.add("box clipped to 2x2")
    # the pyramid: where its source is and whether it is read word-wise (`aligned`)
    aligned = True
    if alias and where == "device":
        off, extra_pitch = extra["dev"]
        aligned = ((off | (3 * S + extra_pitch)) & 3) == 0
        src = f"scale 1 aliased device +{off}, pitch 3S" + (f"+{extra_pitch}" if extra_pitch else "")
    else:
        src = "scale 1 aliased host-staged" if alias else "scale 1 from d_sq"
    Rs = [pyramid_scale(S, s) for s in scales]
    if any(p["R"] == S for p in Rs):
        out.add(src)
        if S // 4 == 100:
            out.add("scale 1 at S / 4 = 100 (box 400)")
    for s, p in zip(scales, Rs):
        R, pad0 = p["R"], p["pad0"]
        if R == S:
            if s < 1:
                out.add("R == S copied")
            continue
        out.add("R > 256" if R > 256 else "128 < R <= 256" if R > 128 else "R < 128")
        out.add("R odd" if R % 2 else "R even")
        if pad0 % 8:
            out.add("pad0 % 8 != 0")
        if pad0 == 0:
            out.add("pad0 = 0")
        if pad0 >= PYR_ROWS:
            out.add("blocks wholly in the surround")
        if 2 * R == S:
            out.add("scale 0.5 (cv2 INTER_AREA)")
        if not aligned:
            out.add("byte-wise loads, shrunken path")
    if len(scales) == 4:
        out.add("four scales")
    if (staged_rows(S, scales) + 1) * S * 4 > PYR_MAX_SMEM:
        out.add("largest staged-row count")
    return out


# ------------------------------------------------------------------------------------------------ CPU tests


def test_matrix_reaches_every_branch():
    reached = set().union(*(case_branches(c) for c in CASES))
    assert reached - BRANCHES == set(), sorted(reached - BRANCHES)
    assert BRANCHES - reached == set(), sorted(BRANCHES - reached)


def test_no_case_can_be_dropped():
    for i, c in enumerate(CASES):
        others = set().union(*(case_branches(o) for j, o in enumerate(CASES) if j != i))
        assert case_branches(c) - others, f"case {c[0]} reaches nothing the other cases do not"


def test_case_shapes_fit_their_engines():
    for name, eng, entry, fmt, frames, extra in CASES:
        _, S, scales, max_frames, max_input = ENGINES[eng]
        assert 1 <= len(frames) <= max_frames, name
        if ENTRIES[entry][0] == "host":
            assert all(h <= max_input[0] and w <= max_input[1] for h, w in frames), name
        if fmt != "bgr":
            assert all(h % 2 == 0 and w % 2 == 0 for h, w in frames), name
        if not ENTRIES[entry][1]:
            assert len(set(frames)) == 1, name
        assert ("boxes" in extra) == ENTRIES[entry][2], name
        assert staged_rows(S, scales) * S * 4 <= PYR_MAX_SMEM, name


def test_the_named_geometries():
    """The numbers the matrix is chosen for, from the restatement."""
    assert [pyramid_scale(368, 0.7)[k] for k in ("R", "pad0")] == [258, 55]
    assert pyramid_scale(448, 0.55)["R"] == 246
    assert [pyramid_scale(64, s)["R"] for s in (0.7, 0.5, 0.3)] == [45, 32, 19]
    assert [pyramid_scale(512, 0.999)[k] for k in ("R", "pad0")] == [511, 0]
    assert pyramid_scale(368, 0.999)["R"] == 368
    assert squarify_geometry(368, 368, 200)[0] == 1.0
    assert squarify_geometry(368, 736, 736)[5] == 1 and squarify_geometry(368, 735, 735)[5] == 0


def test_mode1_corner_block_cannot_occur():
    """A block partial in both directions needs both sides odd, but mode 1 (exact 2x) needs max(h, w) == 2S, which is
    even; so the corner case of the exact-2x decimation is unreachable and the matrix has no case for it."""
    for S in range(64, 513, 16):
        for m in range(2 * S - 3, 2 * S + 4):
            for o in range(m - 3, m + 1):
                if squarify_geometry(S, m, o)[5] == 1 or squarify_geometry(S, o, m)[5] == 1:
                    assert m == 2 * S and o <= m
                    assert not (m % 2 and o % 2)


def test_staged_row_boundary_at_box_512():
    """The smallest scale (in steps of 1e-4) whose staged rows fit 160 KB at box 512, recomputed from the tables."""
    fits = [s for s in np.round(np.arange(0.0850, 0.0950, 0.0001), 4) if staged_rows(512, [float(s)]) * 512 * 4
            <= PYR_MAX_SMEM]
    assert fits[0] == 0.0898
    assert staged_rows(512, [0.0898]) == 80 and 80 * 512 * 4 == PYR_MAX_SMEM
    assert staged_rows(512, [0.0897]) == 81
    assert staged_rows(512, [1.0, 0.0898]) == 80  # pre_512_min


def test_constructor_refuses_a_scale_whose_rows_do_not_fit():
    """vnect_create refuses the scale before anything touches a device (so this runs without one too)."""
    from vnect_b200 import VNectEngine
    with pytest.raises(ValueError, match="pyramid scale too small"):
        VNectEngine(False, [1.0, 0.0897], box_size=512, max_frames=1)
    with pytest.raises(ValueError, match="pyramid scale too small"):
        VNectEngine(False, [0.0897], box_size=512, max_frames=1)


def _umulhi(a, m):
    return ((a.astype(np.uint64) * np.uint64(m)) >> np.uint64(32)).astype(np.int64)


def _walk(width, rows, mg):
    """pyramid_kernel's flat walk of `rows` x `width` items by 256 threads: start at (umulhi(tid, magic), remainder),
    step (256 / width rows, 256 % width columns), one wrap correction, stop past the last row.  -> visited (row, col)."""
    tid = np.arange(PYR_THREADS, dtype=np.int64)
    step_rows = PYR_THREADS // width
    step_cols = PYR_THREADS - step_rows * width
    ly = _umulhi(tid, mg)
    c = tid - ly * width
    assert ((c >= 0) & (c < width)).all()
    seen = []
    active = ly < rows
    while active.any():
        wrap = active & (c >= width)
        c = np.where(wrap, c - width, c)
        ly = np.where(wrap, ly + 1, ly)
        active &= ly < rows
        assert (c[active] < width).all()  # one wrap is enough
        seen.append(ly[active] * width + c[active])
        ly = ly + step_rows
        c = c + step_cols
        active &= ly < rows
    return np.concatenate(seen) if seen else np.zeros(0, np.int64)


def _visits_once(width, rows, mg):
    idx = _walk(width, rows, mg)
    return idx.size == rows * width and np.array_equal(np.sort(idx), np.arange(rows * width))


def test_magic_divisions_are_exact_for_every_thread():
    tid = np.arange(PYR_THREADS, dtype=np.int64)
    for d in range(1, 513):
        assert np.array_equal(_umulhi(tid, magic(d)), tid // d), d


def test_pyramid_walks_visit_every_item_once():
    """Every box size 64..512 in steps of 16: the scale-1 loop (S/4 groups x 1..8 rows), the staging loop (S/4 groups
    x every staged-row count that fits) and the shrunken loop (every R in 1..S x 1..8 rows)."""
    for S in range(64, 513, 16):
        qpr = S // 4
        for rows in range(1, PYR_ROWS + 1):
            assert _visits_once(qpr, rows, magic(qpr)), (S, rows)
        for rows in range(1, PYR_MAX_SMEM // (S * 4) + 1):
            assert _visits_once(qpr, rows, magic(qpr)), (S, "staged", rows)
        for R in range(1, S + 1):
            for rows in range(1, PYR_ROWS + 1):
                assert _visits_once(R, rows, magic(R)), (S, R, rows)


def _cpu_case(S=64, scales=(1.0, 0.7, 0.3), seed=3):
    img = np.random.default_rng(seed).integers(0, 256, (45, 61, 3), dtype=np.uint8)
    return expected_input([img], S, list(scales)), S, list(scales)


def _first_pixel(region, S, scales, fwd=1):
    reg = region_map(S, scales)[fwd % len(scales)]
    return tuple(int(v) for v in np.argwhere(reg == region)[len(np.argwhere(reg == region)) // 2])


def test_reference_layout_places_pixels_as_the_stem_reads_them():
    want, S, scales = _cpu_case()
    batch = np.concatenate([prepost.gen_input_batch(np.random.default_rng(3).integers(0, 256, (45, 61, 3),
                                                                                    dtype=np.uint8), S, scales)[0]])
    for y, x in [(0, 0), (1, 0), (0, 1), (S - 1, S - 1), (17, 40)]:
        pr, pc = y + 2, x + 2
        for c in range(3):
            assert want[1, pr & 1, pr >> 1, pc * 4 + c] == np.float16(batch[1, y, x, c]).view(np.uint16)
        assert want[1, pr & 1, pr >> 1, pc * 4 + 3] == 0
    regs = region_map(S, scales)
    assert {int(v) for v in np.unique(regs)} == {0, 1, 2, 3}
    for f in range(want.shape[0]):
        assert not want[f][regs[f % len(scales)] >= 2].any()


@pytest.mark.parametrize("mutation", ["picture_lsb", "surround", "border", "channel4", "parity_swap", "shift"])
def test_comparison_rejects_mutations(mutation):
    want, S, scales = _cpu_case()
    got = want.copy()
    regs = region_map(S, scales)
    expect = None
    if mutation == "picture_lsb":  # one channel of one picture pixel off by one 8-bit level
        f, par, r, col = 1, *_first_pixel(0, S, scales)
        col -= col % 4
        y, x = 2 * r + par - 2, col // 4 - 2
        lut = {int(np.float16(np.float32(v) / np.float32(255) - np.float32(0.4)).view(np.uint16)): v for v in range(256)}
        v = lut[int(got[f, par, r, col])]
        got[f, par, r, col] = np.float16(np.float32((v + 1) % 256) / np.float32(255) - np.float32(0.4)).view(np.uint16)
        expect = "picture"
    elif mutation == "surround":
        f, par, r, col = 1, *_first_pixel(1, S, scales)
        got[f, par, r, col] ^= 1
        expect = "surround"
    elif mutation == "border":
        got[2, 1, 0, 5] = 0x3c00
        expect = "zero border"
    elif mutation == "channel4":
        f, par, r, col = 0, *_first_pixel(3, S, scales, fwd=0)
        got[f, par, r, col] = 0x0001
        expect = "4th channel"
    elif mutation == "parity_swap":  # padded rows 10 and 11 trade places
        got[0, 0, 5], got[0, 1, 5] = want[0, 1, 5].copy(), want[0, 0, 5].copy()
    else:  # the picture one column to the right
        got[:, :, :, 12:] = want[:, :, :, 8:-4]
    msg = diff_report(got, want, S, scales)
    assert msg is not None
    if expect:
        counts = {k: int(v) for k, v in (item.split(": ") for item in
                                         msg.split("by region {")[1].rstrip("}").replace("'", "").split(", "))}
        assert counts[expect] == 1 and sum(counts.values()) == 1, msg
    assert diff_report(want.copy(), want, S, scales) is None
    assert regs.shape[0] == len(scales)


# ------------------------------------------------------------------------------------------------ GPU


def _frame_data(fmt, h, w, rng):
    """A fresh frame: BGR uint8 [h, w, 3], or YUV 4:2:0 uint8 [3h/2, w] in cv2's layout."""
    return rng.integers(0, 256, (h, w, 3) if fmt == "bgr" else (h * 3 // 2, w), dtype=np.uint8)


def _to_bgr(fmt, f):
    if fmt == "bgr":
        return f
    return cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12 if fmt == "nv12" else cv2.COLOR_YUV2BGR_I420)


def _surface(fmt, f, h, w):
    """A decoder-like surface of a YUV frame: luma pitch w + 64, chroma plane after 16 padding rows, aligned to 256."""
    yp = w + 64
    u_off = yp * (h + 16)
    nv12 = fmt == "nv12"
    uvp = yp if nv12 else yp // 2
    v_off = u_off + 1 if nv12 else u_off + uvp * (h // 2)
    stride = ((v_off if not nv12 else u_off) + uvp * (h // 2) + 255) // 256 * 256
    buf = np.zeros(stride, np.uint8)
    buf[:h * yp].reshape(h, yp)[:, :w] = f[:h]
    if nv12:
        buf[u_off:u_off + uvp * (h // 2)].reshape(h // 2, uvp)[:, :w] = f[h:]
    else:
        q = (h // 2) * (w // 2)
        u, v = f[h:].reshape(-1)[:q].reshape(h // 2, w // 2), f[h:].reshape(-1)[q:].reshape(h // 2, w // 2)
        buf[u_off:u_off + uvp * (h // 2)].reshape(h // 2, uvp)[:, :w // 2] = u
        buf[v_off:v_off + uvp * (h // 2)].reshape(h // 2, uvp)[:, :w // 2] = v
    return buf, dict(y_pitch=yp, uv_pitch=uvp, u_offset=u_off, v_offset=v_off)


class _Run:
    """One engine and the device buffers its cases reuse across their three calls (the same addresses each time, so
    the third call replays the graph the second one captured)."""

    def __init__(self, key):
        from vnect_b200 import VNectEngine
        weights, self.S, self.scales, mf, max_input = ENGINES[key]
        self.eng = VNectEngine(weights, self.scales, box_size=self.S, max_frames=mf, max_streams=mf,
                               max_input=max_input)
        self.t = 1000.0
        self.dev = {}

    def clock(self, n):
        self.t += 0.05
        return np.full(n, self.t), np.full(n, self.t + 0.004)

    def device(self, name, host):
        import torch
        if name not in self.dev:
            self.dev[name] = torch.empty(host.size, dtype=torch.uint8, device="cuda")
        buf = self.dev[name]
        buf.copy_(torch.from_numpy(host.reshape(-1)))
        torch.cuda.synchronize()  # the engine's stream does not wait for torch's
        return buf.data_ptr()

    def outputs(self, name, n):
        import torch
        key = ("out", name)
        if key not in self.dev:
            self.dev[key] = (torch.empty((n, 21, 2), dtype=torch.float64, device="cuda"),
                             torch.empty((n, 21, 3), dtype=torch.float32, device="cuda"),
                             torch.empty((n, 4), dtype=torch.int32, device="cuda"))
        return self.dev[key]


def _call(run, case, frames):
    """One call of the case's entry point; returns the boxes it reports (tracked entries) or None."""
    name, _, entry, fmt, sizes, extra = case
    eng, n = run.eng, len(frames)
    ids = np.arange(n, dtype=np.int32)
    t2, t3 = run.clock(n)
    if ENTRIES[entry][2]:
        for i, b in enumerate(extra["boxes"]):
            eng.set_box(i, b)
    if entry == "estimate":
        eng.estimate(np.stack(frames), ids, t2, t3)
    elif entry in ("submit0", "submit1"):
        lane = int(entry[-1])
        eng.submit(lane, np.stack(frames), ids, t2, t3, pixel_format=fmt)
        eng.wait(lane)
    elif entry == "preprocess":
        eng.preprocess(np.stack(frames))
    elif entry == "track":
        return eng.track(np.stack(frames), ids, t2, t3, pixel_format=fmt)[2]
    elif entry == "estimate_frames":
        eng.estimate_frames(frames, ids, t2, t3, pixel_format=fmt)
    elif entry == "submit_frames":
        eng.submit_frames(1, frames, ids, t2, t3, pixel_format=fmt)
        eng.wait(1)
    elif entry == "track_frames":
        return eng.track_frames(frames, ids, t2, t3, pixel_format=fmt)[2]
    elif entry == "submit_track_frames":
        boxes = eng.submit_track_frames(0, frames, ids, t2, t3, pixel_format=fmt)[2]
        eng.wait(0)
        return boxes
    else:  # device entry points
        j2, j3, bx = run.outputs(name, n)
        if entry == "estimate_device" and fmt == "bgr":
            (h, w), (off, xp) = sizes[0], extra["dev"]
            pitch = 3 * w + xp
            stride = pitch * h + 4
            host = np.zeros(off + stride * n, np.uint8)
            for i, f in enumerate(frames):
                host[off + i * stride:off + i * stride + pitch * h].reshape(h, pitch)[:, :3 * w] = f.reshape(h, 3 * w)
            ptr = run.device(name, host) + off
            eng.estimate_device(ptr, n, h, w, j2.data_ptr(), j3.data_ptr(), ids, t2, t3, pitch=pitch,
                                frame_stride=stride)
        elif entry == "estimate_device":
            h, w = sizes[0]
            surf = [_surface(fmt, f, h, w) for f in frames]
            ptr = run.device(name, np.concatenate([s[0] for s in surf]))
            eng.estimate_device(ptr, n, h, w, j2.data_ptr(), j3.data_ptr(), ids, t2, t3, pixel_format=fmt,
                                layout=dict(surf[0][1], frame_stride=surf[0][0].size))
        else:
            descs, parts, pos = [], [], 0
            for (h, w), f in zip(sizes, frames):  # packed frames (cv2's layout for YUV), 256 bytes apart
                part = f.reshape(-1)
                descs.append((pos, dict(h=h, w=w)))
                parts.append(part)
                pos += (part.size + 255) // 256 * 256
            host = np.zeros(pos, np.uint8)
            for (p, _), part in zip(descs, parts):
                host[p:p + part.size] = part
            base = run.device(name, host)
            table = [dict(ptr=base + p, **d) for p, d in descs]
            if entry == "estimate_device_frames":
                eng.estimate_device_frames(table, j2.data_ptr(), j3.data_ptr(), ids, t2, t3, pixel_format=fmt)
            else:
                eng.track_device_frames(table, j2.data_ptr(), j3.data_ptr(), bx.data_ptr(), ids, t2, t3,
                                        pixel_format=fmt)
                eng.synchronize()
                return bx.cpu().numpy()
    return None


@pytest.fixture(scope="module")
def runs():
    made = {}

    def get(key):
        if key not in made:
            made[key] = _Run(key)
        return made[key]
    yield get
    for r in made.values():
        r.eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_stem_input_bit_exact(case, runs):
    name, eng_key, entry, fmt, sizes, extra = case
    run = runs(eng_key)
    S, scales = run.S, run.scales
    t0 = time.perf_counter()
    pics, boxes = case_pictures(case)
    n = len(sizes)
    compared = 0
    for call in range(CALLS):
        rng = np.random.default_rng([sum(map(ord, name)), call])
        frames = [_frame_data(fmt, h, w, rng) for h, w in sizes]
        used = _call(run, case, frames)
        got = run.eng.stem_input(n * len(scales))
        bgr = [_to_bgr(fmt, f) for f in frames]
        if boxes is not None:
            used = np.asarray(used).reshape(n, 4)
            assert [tuple(int(v) for v in b) for b in used] == boxes, (call, used, boxes)
            bgr = [np.ascontiguousarray(f[y:y + h, x:x + w]) for f, (x, y, w, h) in zip(bgr, boxes)]
        want = expected_input(bgr, S, scales)
        msg = diff_report(got, want, S, scales)
        assert msg is None, f"{name}, call {call}: {msg}"
        compared += got.size
    Rs = [pyramid_scale(S, s)["R"] for s in scales]
    print(f"\n[{name}] entry={entry} format={fmt} S={S} scales={scales} R={Rs} frames={sizes} "
          f"pictures={pics}\n    branches={sorted(case_branches(case))}\n    forwards={CALLS * n * len(scales)} "
          f"elements={compared} bit-exact ({time.perf_counter() - t0:.2f} s)")


@pytest.mark.gpu
def test_smallest_accepted_scale_builds_at_box_512():
    """0.0898 at box 512 stages exactly 160 KB: built (and bit-exact, pre_512_min_scale); 0.0897 is refused."""
    from vnect_b200 import VNectEngine
    eng = VNectEngine(False, [0.0898], box_size=512, max_frames=1, max_input=(300, 500))
    try:
        img = np.random.default_rng(5).integers(0, 256, (300, 500, 3), dtype=np.uint8)
        eng.preprocess(img)
        assert diff_report(eng.stem_input(1), expected_input([img], 512, [0.0898]), 512, [0.0898]) is None
    finally:
        eng.close()
    with pytest.raises(ValueError, match="pyramid scale too small"):
        VNectEngine(False, [0.0897], box_size=512, max_frames=1)
