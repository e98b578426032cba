"""Every launch of the CNN forward, checked in isolation against a float64 evaluation of that one operation.

Each launch's inputs are read back from the device with ``VNectEngine.tap`` (exact fp16 values; the stem's input is
the ``forward()`` batch, fp16-representable), its parameters are rounded to fp16 exactly as ``vnect_finalize`` rounds
them, and the operation is evaluated in float64 with torch convolutions.  The comparison is per element, so one wrong
tap block, pixel, image or tile fails it; the tolerance does not accumulate over the layers before the launch.

The bound.  A launch computes ``s = sum_k a_k w_k + bias (+ residual)`` over K multiply-adds and rounds it to fp16
(or stores it as fp32).  fp16 x fp16 products are exact in fp32 (11 + 11 significand bits, exponents far inside the
fp32 range, fp16 subnormals included), so only the additions round.  There are K + 1 of them (K products, the bias,
the residual), in an order that is not known (tensor-core MMAs, K blocks, CTA-pair halves) and possibly truncating
inside an MMA, so every addition is allowed a relative error of u = 2^-23 (round toward zero; round to nearest is
2^-24).  A term that passes through d roundings carries at most ((1 + u)^d - 1) |term|; summed over the terms this is
at most ((1 + u)^(K+1) - 1) A, with A = sum_k |a_k w_k| + |bias| (+ |residual|) evaluated in float64 as conv(|a|, |w|)
+ |bias| (+ |res|).  (1 + u)^d - 1 <= (d + 1) u while d (d - 1) u / 2 <= 1, i.e. for any chain of up to 4096 roundings;
the longest chain of an MMA-based sum is far shorter (each MMA adds 16 products before the accumulator sees them), so
for every K here (at most 4608) the fp32 error is below (K + 2) u A.  ReLU and max-pooling do not increase an error
(|relu(x) - relu(y)| <= |x - y|, |max x - max y| <= max |x - y|).  Rounding the fp32 result to fp16 (round to
nearest) adds at most 2^-11 |got| for a normal result and 2^-25 in the subnormal range.  Per element:

    |got - relu(ref)| <= (K + 2) 2^-23 A + 2^-11 |got| + 2^-25

* K is the launch's multiply-add count: taps x padded Cin (224 for the stem's 7 rows x 8 px x 4 ch), plus the
  shortcut's Cin for a folded projection, 4 taps x 256 for the transposed conv.  The second output of a fused block
  tail is its own 1x1 conv of K = the first output's channels, read from the first output's tap.
* planar fp32 outputs (the maps ``forward()`` returns): the last two terms become 2^-24 |got|.
* conv1 + pool1: the bound of a pooled element is the largest bound of its window.
* bone lengths sqrt(dx^2 + dy^2 + dz^2) are computed from the fp32 deltas: sqrt(3) times the largest component bound,
  plus 4 2^-24 bone for the fp32 squares, sums and square root, plus the fp16 term.

Sensitivity.  For every launch the same checker must reject three mutations of the reference: (a) one 64-channel block
removed at one tap (the last K block, and for a folded projection also the shortcut's first block), (b) the output
shifted by one pixel in x within each image, (c) the residual dropped, where there is one.
"""
import math
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import synth

U = 2.0 ** -23
EPI_PLANAR_F32, EPI_DECONV_HEAD, EPI_TMA, EPI_TMA_RES = 1, 2, 3, 4

# ------------------------------------------------------------------------------------------------ graph restatement
BLOCK_INPUT = {"res2a": "pool1", "res2b": "res2a", "res2c": "res2b", "res3a": "res2c", "res3b": "res3a",
               "res3c": "res3b", "res3d": "res3c", "res4a": "res3d", "res4b": "res4a", "res4c": "res4b",
               "res4d": "res4c", "res4e": "res4d", "res4f": "res4e", "res5a": "res4f"}
EVEN_ONLY = {"res2b", "res2c", "res3d"}  # blocks evaluated at even pixels only (their output feeds stride-2 1x1s)
CHAIN = {"res5b_branch2a_new": "res5a", "res5b_branch2b_new": "res5b_branch2a_new",
         "res5b_branch2c_new": "res5b_branch2b_new", "res5c_branch2b": "res5c_branch2a_feat"}


def restate(name):
    """Step name -> what the launch reads and writes: kind, scope(s), k, in / in_stride, in2, res / res_stride, out,
    tail (scope of a fused block tail's second conv, which is also its output's name)."""
    st = dict(name=name, k=1, in_stride=1, in2=None, res=None, res_stride=1, tail=None, scope=None)
    if name == "conv1+pool1":
        return dict(st, kind="stem", k=7, input="<input>", out="pool1")
    if name == "res5c_deconv_head":
        return dict(st, kind="deconv", k=4, input="res5b_branch2c_new", out="res5c_branch2a_feat")
    if name == "res5c_branch2c":
        return dict(st, kind="planar", scope=name, input="res5c_branch2b", out="<maps>")
    main, _, tail = name.partition(">")
    st["tail"] = tail or None
    if "+" in main:
        s2c, s1 = main.split("+")
        pre, suf = s2c.split("_branch")[0], "_new" if s2c.endswith("_new") else ""
        return dict(st, kind="fold", scope=s2c, scope1=s1, input=f"{pre}_branch2b{suf}", in2=BLOCK_INPUT[pre], out=pre)
    if main in CHAIN:
        return dict(st, kind="conv", scope=main, k=3 if "branch2b" in main else 1, input=CHAIN[main], out=main)
    pre, br = main.split("_branch")
    suf = "_new" if br.endswith("_new") else ""
    if br.startswith("2a"):
        return dict(st, kind="conv", scope=main, input=BLOCK_INPUT[pre], out=main)
    if br.startswith("2b"):
        return dict(st, kind="conv", scope=main, k=3, input="res2b_branch2a" if pre == "res2c" else f"{pre}_branch2a{suf}",
                    in_stride=2 if pre in EVEN_ONLY else 1, out=main)
    # last 1x1 with the identity shortcut: read at stride 2 from a full-size block input (res2b from res2a, res3d from
    # res3c), at stride 1 from res2b, which is itself even-pixel only
    return dict(st, kind="conv", scope=main, input=f"{pre}_branch2b{suf}", res=BLOCK_INPUT[pre],
                res_stride=2 if pre in ("res2b", "res3d") else 1, out=pre)


def io_names(st):
    ins = [st["input"]] + [x for x in (st["in2"], st["res"]) if x]
    return ins, [st["out"]] + ([st["tail"]] if st["tail"] else [])


# ------------------------------------------------------------------------------------------------ parameters
def _h(a):
    """float32 parameters -> their fp16 values (round to nearest even, as __float2half_rn) in float64"""
    return torch.from_numpy(np.asarray(a, np.float32).astype(np.float16).astype(np.float64))


def _f(a):
    return torch.from_numpy(np.asarray(a, np.float32).astype(np.float64))


def _oihw(w_hwio, cin_pad=None):
    w = _h(w_hwio).permute(3, 2, 0, 1)
    if cin_pad and cin_pad > w.shape[1]:
        w = F.pad(w, (0, 0, 0, 0, 0, cin_pad - w.shape[1]))
    return w.contiguous()


class Params:
    """The launch's parameters exactly as vnect_finalize packs them, in float64 on `dev`."""

    def __init__(self, weights, dev):
        self.w, self.dev, self.cache = weights, dev, {}

    def get(self, key, make):
        if key not in self.cache:
            self.cache[key] = tuple(t.to(self.dev) for t in make())
        return self.cache[key]

    def conv(self, scope, cin_pad):
        return self.get((scope, cin_pad), lambda: (_oihw(self.w[scope + "/weights"], cin_pad),
                                                   _f(self.w[scope + "/biases"])))

    def fold(self, s2c, s1):
        # [W_2c | W_1], bias b_2c + b_1 summed in float32
        b = np.float32(self.w[s2c + "/biases"]) + np.float32(self.w[s1 + "/biases"])
        return self.get((s2c, s1), lambda: (_oihw(self.w[s2c + "/weights"]), _oihw(self.w[s1 + "/weights"]), _f(b)))

    def deconv(self):
        def make():
            g, be = (np.asarray(self.w["bn5c_branch2a/" + v], np.float32) for v in ("gamma", "beta"))
            mu, var = (np.asarray(self.w["bn5c_branch2a/" + v], np.float32) for v in ("moving_mean", "moving_variance"))
            scale = g / np.sqrt(var + np.float32(0.001))  # float32 throughout, as the host code
            bias = be - mu * scale
            w2a = np.asarray(self.w["res5c_branch2a/kernel"], np.float32) * scale[None, None, :, None]  # before rounding
            w = torch.cat([_h(w2a), _h(self.w["res5c_branch1a/kernel"])], dim=2)  # [kh, kw, 191, 256]
            return w.permute(3, 2, 0, 1).contiguous(), torch.cat([_f(bias), torch.zeros(63, dtype=torch.float64)])
        return self.get("deconv", make)

    def planar(self):
        return self.get("planar", lambda: (_oihw(self.w["res5c_branch2c/kernel"]),))

    def stem(self):
        return self.get("stem", lambda: (_oihw(self.w["conv1/weights"]), _f(self.w["conv1/biases"])))


# ------------------------------------------------------------------------------------------------ reference
def _conv(x, w, stride=1, padding=0):
    return F.conv2d(x, w, stride=stride, padding=padding)


def reference(st, get, P, drop=None, no_res=False, bounds=True):
    """float64 evaluation of one launch -> {output name: (ref, accumulation bound, fp16 output?)}.  `get(name)` gives
    an activation as float64 NCHW.  drop = (which, channel slice, (ky, kx)): zero that block of the weights of the
    launch's main input ("in"), its folded shortcut ("in2") or its fused tail's conv ("tail").  no_res: drop the
    residual."""
    out = {}
    kind = st["kind"]

    def dropped(w, which):
        if drop is None or drop[0] != which:
            return w
        w = w.clone()
        w[:, drop[1], drop[2][0], drop[2][1]] = 0
        return w

    if kind == "stem":
        x = get("<input>")
        w, b = P.stem()
        w = dropped(w, "in")
        pad = lambda t: F.pad(t, (2, 3, 2, 3))  # SAME for 7x7 / 2 on an even side
        y = F.relu(_conv(pad(x), w, 2) + b[None, :, None, None])
        ref = F.max_pool2d(F.pad(y, (0, 1, 0, 1), value=-math.inf), 3, 2)
        accb = None
        if bounds:
            A = _conv(pad(x.abs()), w.abs(), 2) + b.abs()[None, :, None, None]
            accb = F.max_pool2d(F.pad((224 + 2) * U * A, (0, 1, 0, 1)), 3, 2)  # bounds >= 0: zero pad = ignored
        out["pool1"] = (ref, accb, True)
        return out
    if kind == "deconv":
        x = get(st["input"])
        w, b = P.deconv()
        w = dropped(w.permute(1, 0, 2, 3), "in").permute(1, 0, 2, 3)  # [in, out, kh, kw]: drop over input channels
        d = F.conv_transpose2d(x, w, stride=2, padding=1) + b[None, :, None, None]
        d1 = d[:, 128:191]
        bone = torch.sqrt(d1[:, 0:21] ** 2 + d1[:, 21:42] ** 2 + d1[:, 42:63] ** 2)
        ref = torch.cat([F.relu(d[:, :128]), d1, bone], dim=1)
        accb = None
        if bounds:
            A = F.conv_transpose2d(x.abs(), w.abs(), stride=2, padding=1) + b.abs()[None, :, None, None]
            cb = (1024 + 2) * U * A
            c1 = cb[:, 128:191]
            comp = torch.maximum(torch.maximum(c1[:, 0:21], c1[:, 21:42]), c1[:, 42:63])
            accb = torch.cat([cb[:, :128], c1, math.sqrt(3) * comp + 4 * 2.0 ** -24 * bone], dim=1)
        out["res5c_branch2a_feat"] = (ref, accb, True)
        return out
    if kind == "planar":
        x = get(st["input"])
        (w,) = P.planar()
        w = dropped(w, "in")
        ref = _conv(x, w)
        out["<maps>"] = (ref, (128 + 2) * U * _conv(x.abs(), w.abs()) if bounds else None, False)
        return out
    x = get(st["input"])
    s, ss = st["in_stride"], slice(None, None, st["res_stride"])
    if kind == "fold":
        w2c, w1, b = P.fold(st["scope"], st["scope1"])
        x2 = get(st["in2"])
        w2c, w1 = dropped(w2c, "in"), dropped(w1, "in2")
        y = _conv(x, w2c) + _conv(x2, w1) + b[None, :, None, None]
        A = (_conv(x.abs(), w2c.abs()) + _conv(x2.abs(), w1.abs()) + b.abs()[None, :, None, None]) if bounds else None
        K = x.shape[1] + x2.shape[1]
    else:
        w, b = P.conv(st["scope"], x.shape[1])
        w = dropped(w, "in")
        pad = 1 if st["k"] == 3 else 0
        y = _conv(x, w, s, pad) + b[None, :, None, None]
        A = (_conv(x.abs(), w.abs(), s, pad) + b.abs()[None, :, None, None]) if bounds else None
        K = st["k"] ** 2 * x.shape[1]
        if st["res"]:
            r = get(st["res"])[:, :, ss, ss]
            if not no_res:
                y = y + r
            if bounds:
                A = A + r.abs()
    out[st["out"]] = (F.relu(y), (K + 2) * U * A if bounds else None, True)
    if st["tail"]:
        t = get(st["out"])  # the tail's conv reads the first output as stored (fp16)
        w2, b2 = P.conv(st["tail"], t.shape[1])
        w2 = dropped(w2, "tail")
        ref2 = F.relu(_conv(t, w2) + b2[None, :, None, None])
        A2 = _conv(t.abs(), w2.abs()) + b2.abs()[None, :, None, None] if bounds else None
        out[st["tail"]] = (ref2, (t.shape[1] + 2) * U * A2 if bounds else None, True)
    return out


def check(got, ref, accb, fp16):
    """-> (elements over the bound, largest err / bound, largest share of the fp32 term used by what the output
    rounding does not explain).  Rounding to fp16 alone reaches err / bound ~ 1 at the bottom of a binade, so the second
    number sits near 1 for any correct fp16 output; the third shows how much of (K + 2) 2^-23 A the sum really used."""
    err = (got - ref).abs()
    rounding = 2.0 ** -11 * got.abs() + 2.0 ** -25 if fp16 else 2.0 ** -24 * got.abs()
    bound = accb + rounding
    ratio = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, math.inf, 0.0))
    share = ((err - rounding).clamp_min(0) / accb.clamp_min(1e-300)).max()
    return int((err > bound).sum()), float(ratio.max()), float(share)


def mutations(st, cin, cin2=None, ctail=None):
    """(label, reference() keyword arguments) of the mutations every launch must be caught by"""
    k = st["k"]
    if st["kind"] == "stem":
        m = [("block", dict(drop=("in", slice(0, 3), (6, 6))))]  # all three channels at one of the 49 taps
    elif st["kind"] == "deconv":
        m = [("block", dict(drop=("in", slice(192, 256), (3, 3))))]
    elif st["kind"] == "fold":
        m = [("block", dict(drop=("in2", slice(cin2 - 64, cin2), (0, 0)))),
             ("short0", dict(drop=("in2", slice(0, 64), (0, 0))))]
    else:
        m = [("block", dict(drop=("in", slice(cin - 64, cin), (k - 1, k - 1))))]
    if st["tail"]:
        m.append(("tail", dict(drop=("tail", slice(ctail - 64, ctail), (0, 0)))))
    m.append(("shift", None))
    if st["res"]:
        m.append(("res", dict(no_res=True)))
    return m


def check_launch(st, get, P):
    """All outputs of one launch against the reference, then every mutation.  -> ([largest err / bound, largest share
    of the fp32 term], {mutation: elements flagged}); asserts that the launch passes and that each mutation is
    rejected."""
    base = reference(st, get, P)
    worst = [0.0, 0.0]
    for name, (ref, accb, fp16) in base.items():
        got = get(name)
        assert bool(torch.isfinite(got).all()), f"{st['name']}: non-finite values in {name}"
        if name == "res5c_branch2a_feat":
            assert got.shape[1] == 256 and bool((got[:, 212:] == 0).all()), "deconv head: columns 212-255 must be 0"
            got = got[:, :212]
        assert got.shape == ref.shape, (st["name"], name, tuple(got.shape), tuple(ref.shape))
        bad, r, share = check(got, ref, accb, fp16)
        assert bad == 0, f"{st['name']} -> {name}: {bad} elements over the bound (largest err / bound {r:.3g})"
        worst = [max(worst[0], r), max(worst[1], share)]
    x = get(st["input"])
    cin2 = get(st["in2"]).shape[1] if st["in2"] else None
    ctail = get(st["out"]).shape[1] if st["tail"] else None
    flagged = {}
    for label, kw in mutations(st, x.shape[1], cin2, ctail):
        mut = {n: (torch.roll(v[0], 1, dims=3),) for n, v in base.items()} if kw is None else \
            reference(st, get, P, bounds=False, **kw)
        flagged[label] = sum(check(get(n)[:, :mut[n][0].shape[1]], mut[n][0], base[n][1], base[n][2])[0] for n in base)
        assert flagged[label] > 0, f"{st['name']}: mutation '{label}' is not rejected"
    return worst, flagged


# ------------------------------------------------------------------------------------------------ CPU tests
class Float32Params:
    """Params in float32: the arithmetic of a correct kernel, for the CPU tests"""

    def __init__(self, P):
        self.P = P

    def __getattr__(self, meth):
        return lambda *a: tuple(t.float() for t in getattr(self.P, meth)(*a))


def emulate_launch(st, acts, P32):
    """What a correct device stores for one launch: float32 arithmetic, fp16 (or fp32 planar) outputs, in `acts`"""
    get32 = lambda k: acts[k].float()
    # a fused tail reads the first output as stored: store it, then evaluate the tail from it
    for step in ([dict(st, tail=None), st] if st["tail"] else [st]):
        for k, (v, _, fp16) in reference(step, get32, P32, bounds=False).items():
            acts[k] = (v.half() if fp16 else v).double()
    if st["kind"] == "deconv":  # stored with 44 zero columns of padding
        acts["res5c_branch2a_feat"] = F.pad(acts["res5c_branch2a_feat"], (0, 0, 0, 0, 0, 44))


class EmulatedEngine:
    """The 368 throughput plan's launches in float32 on the CPU, at any box size: lets the GPU test's walk over a
    forward run without a GPU"""

    def __init__(self, weights, box):
        self.box_size, self.scales, self.P32 = box, [1.0], Float32Params(Params(weights, "cpu"))

    def step_names(self):
        return [s[0] for s in STEPS_368]

    def info(self, key):
        assert key == "launches_per_forward"
        return float(len(STEPS_368))

    def forward(self, x):
        self.acts = {"<input>": torch.from_numpy(x).double().permute(0, 3, 1, 2)}
        for name in self.step_names():
            emulate_launch(restate(name), self.acts, self.P32)
        maps = self.acts["<maps>"].permute(0, 2, 3, 1).float().numpy()
        return tuple(np.ascontiguousarray(maps[..., 21 * i:21 * (i + 1)]) for i in range(4))

    def tap(self, name, n):
        return self.acts[name][:n].permute(0, 2, 3, 1).float().numpy()

STEPS_368 = [  # the throughput plan at box 368 (CTA pairs, 256-column tiles, fused block tails): (name, ins, outs)
    ("conv1+pool1", ["<input>"], ["pool1"]),
    ("res2a_branch2a", ["pool1"], ["res2a_branch2a"]),
    ("res2a_branch2b", ["res2a_branch2a"], ["res2a_branch2b"]),
    ("res2a_branch2c+res2a_branch1>res2b_branch2a", ["res2a_branch2b", "pool1"], ["res2a", "res2b_branch2a"]),
    ("res2b_branch2b", ["res2b_branch2a"], ["res2b_branch2b"]),
    ("res2b_branch2c", ["res2b_branch2b", "res2a"], ["res2b"]),
    ("res2c_branch2b", ["res2b_branch2a"], ["res2c_branch2b"]),
    ("res2c_branch2c>res3a_branch2a", ["res2c_branch2b", "res2b"], ["res2c", "res3a_branch2a"]),
    ("res3a_branch2b", ["res3a_branch2a"], ["res3a_branch2b"]),
    ("res3a_branch2c+res3a_branch1", ["res3a_branch2b", "res2c"], ["res3a"]),
    ("res3b_branch2a", ["res3a"], ["res3b_branch2a"]),
    ("res3b_branch2b", ["res3b_branch2a"], ["res3b_branch2b"]),
    ("res3b_branch2c>res3c_branch2a", ["res3b_branch2b", "res3a"], ["res3b", "res3c_branch2a"]),
    ("res3c_branch2b", ["res3c_branch2a"], ["res3c_branch2b"]),
    ("res3c_branch2c>res3d_branch2a", ["res3c_branch2b", "res3b"], ["res3c", "res3d_branch2a"]),
    ("res3d_branch2b", ["res3d_branch2a"], ["res3d_branch2b"]),
    ("res3d_branch2c", ["res3d_branch2b", "res3c"], ["res3d"]),
    ("res4a_branch2a", ["res3d"], ["res4a_branch2a"]),
    ("res4a_branch2b", ["res4a_branch2a"], ["res4a_branch2b"]),
    ("res4a_branch2c+res4a_branch1", ["res4a_branch2b", "res3d"], ["res4a"]),
] + [s for p, q in zip("bcdef", "abcde") for s in (
    (f"res4{p}_branch2a", [f"res4{q}"], [f"res4{p}_branch2a"]),
    (f"res4{p}_branch2b", [f"res4{p}_branch2a"], [f"res4{p}_branch2b"]),
    (f"res4{p}_branch2c", [f"res4{p}_branch2b", f"res4{q}"], [f"res4{p}"]))] + [
    ("res5a_branch2a_new", ["res4f"], ["res5a_branch2a_new"]),
    ("res5a_branch2b_new", ["res5a_branch2a_new"], ["res5a_branch2b_new"]),
    ("res5a_branch2c_new+res5a_branch1_new", ["res5a_branch2b_new", "res4f"], ["res5a"]),
    ("res5b_branch2a_new", ["res5a"], ["res5b_branch2a_new"]),
    ("res5b_branch2b_new", ["res5b_branch2a_new"], ["res5b_branch2b_new"]),
    ("res5b_branch2c_new", ["res5b_branch2b_new"], ["res5b_branch2c_new"]),
    ("res5c_deconv_head", ["res5b_branch2c_new"], ["res5c_branch2a_feat"]),
    ("res5c_branch2b", ["res5c_branch2a_feat"], ["res5c_branch2b"]),
    ("res5c_branch2c", ["res5c_branch2b"], ["<maps>"]),
]


def test_graph_restatement_names_every_input_and_output():
    assert len(STEPS_368) == 44
    for name, ins, outs in STEPS_368:
        assert io_names(restate(name)) == (ins, outs), name
    # geometry the names alone do not show
    assert [restate(n)["in_stride"] for n in ("res2b_branch2b", "res2c_branch2b", "res3d_branch2b", "res3a_branch2b")] \
        == [2, 2, 2, 1]
    assert [restate(n)["res_stride"] for n in ("res2b_branch2c", "res2c_branch2c>res3a_branch2a", "res3d_branch2c",
                                               "res4b_branch2c")] == [2, 1, 2, 1]
    # the latency plan runs the same graph with every block tail unfused
    for name, ins, outs in STEPS_368:
        main, _, tail = name.partition(">")
        if tail:
            assert io_names(restate(main)) == (ins, outs[:1])
            assert io_names(restate(tail)) == ([outs[0]], [tail])
    # every activation is written by exactly one launch before it is read
    written = {"<input>"}
    for name, ins, outs in STEPS_368:
        assert set(ins) <= written, name
        assert not set(outs) & written, name
        written |= set(outs)


def _rn(x):
    return x.astype(np.float32)


def _rz_add(s, p):
    """float32 s + p rounded toward zero (float64 sum, then truncated)"""
    t = s.astype(np.float64) + p.astype(np.float64)
    r = t.astype(np.float32)
    over = np.abs(r.astype(np.float64)) > np.abs(t)
    r[over] = np.nextafter(r[over], np.float32(0))
    return r


@pytest.mark.parametrize("K", [64, 320, 576, 1024, 2304, 4608])
def test_bound_holds_for_fp32_sums_in_any_order(K):
    rng = np.random.default_rng(K)
    rows = 64
    # fp16 operands over a wide range of magnitudes, subnormals included, mostly one sign (large A, small |s|)
    a = (rng.standard_normal((rows, K)) * 2.0 ** rng.integers(-20, 4, (rows, K))).astype(np.float16)
    w = (rng.standard_normal((rows, K)) * 0.05 + 0.01).astype(np.float16)
    prods = a.astype(np.float32) * w.astype(np.float32)  # exact
    assert np.array_equal(prods.astype(np.float64), a.astype(np.float64) * w.astype(np.float64))
    bias = rng.standard_normal(rows).astype(np.float32)
    exact = (a.astype(np.float64) * w.astype(np.float64)).sum(1) + bias
    A = np.abs(a.astype(np.float64) * w.astype(np.float64)).sum(1) + np.abs(bias)
    orders = [np.arange(K), np.argsort(np.abs(prods[0])), np.argsort(-np.abs(prods[0]))] + \
             [rng.permutation(K) for _ in range(3)]
    for order in orders:
        p = prods[:, order]
        for rz in (False, True):
            s = np.zeros(rows, np.float32)
            for k in range(K):  # sequential: the longest possible rounding chain
                s = _rz_add(s, p[:, k]) if rz else _rn(s + p[:, k])
            s = _rz_add(s, bias) if rz else _rn(s + bias)
            for relu in (False, True):
                got = np.maximum(s, 0) if relu else s
                ref = np.maximum(exact, 0) if relu else exact
                g16 = got.astype(np.float16).astype(np.float64)
                n, r, _ = check(torch.from_numpy(g16), torch.from_numpy(ref), torch.from_numpy((K + 2) * U * A), True)
                assert n == 0 and r < 1, (K, rz, relu, r)
                n, r, _ = check(torch.from_numpy(got.astype(np.float64)), torch.from_numpy(ref),
                             torch.from_numpy((K + 2) * U * A), False)
                assert n == 0 and r < 1, (K, rz, relu, r)
        # MMA-like order: 16-product groups summed in a tree, then accumulated
        g = p.reshape(rows, -1, 16)
        while g.shape[2] > 1:
            g = _rn(g[:, :, 0::2] + g[:, :, 1::2])
        s = np.zeros(rows, np.float32)
        for k in range(g.shape[1]):
            s = _rn(s + g[:, k, 0])
        g16 = _rn(s + bias).astype(np.float16).astype(np.float64)
        assert check(torch.from_numpy(g16), torch.from_numpy(exact), torch.from_numpy((K + 2) * U * A), True)[0] == 0


@pytest.mark.parametrize("name", ["res2b_branch2c", "res2a_branch2c+res2a_branch1>res2b_branch2a", "res3d_branch2b",
                                  "conv1+pool1", "res5c_deconv_head", "res5c_branch2c"])
def test_mutations_are_rejected_on_cpu(w1, name):
    """A float32 evaluation of the launch (what a correct kernel stores) passes the checker; each mutation of the
    reference fails it.  Small geometry, same code as the GPU test."""
    rng = np.random.default_rng(5)
    st = restate(name)
    P = Params(w1, "cpu")
    S, n = 64, 2
    shapes = {"<input>": (n, 3, S, S), "pool1": (n, 64, 16, 16), "res2a_branch2b": (n, 64, 16, 16),
              "res2a": (n, 256, 16, 16), "res2b_branch2b": (n, 64, 8, 8), "res2b_branch2a": (n, 64, 16, 16),
              "res3d_branch2a": (n, 128, 8, 8), "res5b_branch2c_new": (n, 256, 4, 4), "res5c_branch2b": (n, 128, 8, 8)}
    acts = {k: torch.from_numpy(rng.uniform(-1, 1, s).astype(np.float16).astype(np.float64)) for k, s in shapes.items()}
    acts["<input>"] = acts["<input>"] * 0.5
    for k in ("pool1", "res2a", "res2b_branch2b", "res2b_branch2a", "res3d_branch2a", "res5b_branch2c_new"):
        acts[k] = acts[k].abs()  # post-ReLU activations
    get = acts.__getitem__
    emulate_launch(st, acts, Float32Params(P))
    worst, flagged = check_launch(st, get, P)
    assert worst[0] < 1
    assert set(flagged) >= {"block", "shift"} and all(v > 0 for v in flagged.values())
    if st["res"]:
        assert flagged["res"] > 0


def test_walk_over_an_emulated_forward(w1):
    """The GPU test's walk, on a float32 emulation of the 368 plan at box 64: the restated graph chains (every
    launch's inputs have the shapes its reference needs) and a correct forward passes every launch."""
    report = {"params": Params(w1, "cpu"), "worst": {}, "failures": []}
    x = np.random.default_rng(3).uniform(-0.4, 0.6, (2, 64, 64, 3)).astype(np.float16).astype(np.float32)
    _check_forward(EmulatedEngine(w1, 64), x, "emulated 64", report)
    assert not report["failures"], report["failures"]
    assert len(report["worst"]) == 44 and max(w[0] for w in report["worst"].values()) < 1


# ------------------------------------------------------------------------------------------------ GPU
def _stem_units(S, n, n_xt, sms):
    """items and grid of stem_roll_set_batch (conv_plan.cuh)"""
    PH, best_rows, best = S // 4, S // 4, -1
    for rows in range(1, PH + 1):
        segs = -(-PH // rows)
        cost = -(-(n * segs * n_xt) // sms) * (4 * rows + 7)
        if best < 0 or cost <= best:
            best, best_rows = cost, rows
    items = n * -(-PH // best_rows) * n_xt
    grid = max(min(items, sms) & ~1, 1)
    return items, grid


def _units_per_worker(path, cout, n, S, sms):
    """most tiles (or tail units, or stem items) one CTA / CTA pair walks in this launch"""
    if path["kind"] == "stem":
        items, grid = _stem_units(S, n, path["n_xt"], sms)
        return -(-items // grid)  # a CTA pair takes both x tiles of a segment: one item per CTA either way
    H, W = path["H"], path["W"]
    m_tiles = -(-(n * H * W) // 128) if path["mode"] == 0 else n * -(-W // path["tw"]) * -(-H // path["th"])
    if path["n2"]:
        units, workers = -(-m_tiles // 2), sms // 2
    else:
        phases = 4 if path["epi"] == EPI_DECONV_HEAD else 1
        n_pad = {EPI_DECONV_HEAD: 192, EPI_PLANAR_F32: 96}.get(path["epi"], cout)
        units, workers = phases * -(-m_tiles // path["cg"]) * (n_pad // path["block_n"]), sms // path["cg"]
    return -(-units // min(units, workers))


class DeviceTaps:
    """Activations of the engine's last forward of n images as float64 NCHW on `dev`, each read back once"""

    def __init__(self, eng, n, x, maps, dev):
        self.eng, self.n, self.dev, self.cache = eng, n, dev, {}
        self.cache["<input>"] = torch.from_numpy(x).to(dev, torch.float16)
        self.cache["<maps>"] = torch.from_numpy(np.concatenate(maps, axis=-1)).to(dev)

    def __call__(self, name):
        if name not in self.cache:
            t = self.eng.tap(name, self.n)
            self.cache[name] = torch.from_numpy(t).to(self.dev, torch.float16)  # exact: the tap holds fp16 values
        return self.cache[name].to(torch.float64).permute(0, 3, 1, 2).contiguous()


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return f"{name}, power limit {pl}"


MATRIX = [  # (box, scales, max_frames, forwards checked, why)
    (368, [1.0, 0.7], 64, [128, 5], "throughput plan, bench batch: every persistent loop wraps; then an odd batch "
                                    "after a larger call"),
    (368, [1.0, 0.7], 1, [2, 1], "latency plan: 64-column tiles, no tails"),
    (368, [1.0, 0.7], 4, [7], "latency plan at its largest capacity: the launches only it has (unfused block tails) "
                              "walk several tiles per CTA"),
    (448, [1.0, 0.85, 0.7], 32, [96], "C5's plan"),
    (512, [1.0, 0.7], 8, [5], "three-x-tile single-CTA stem, every grid a multiple of 128 rows"),
    (400, [1.0, 0.7], 8, [7], "resident-weight spatial res2 3x3, im2col res3 on CTA pairs, odd res4 grid, pair stem"),
    (64, [1.0, 0.7], 20, [37], "tiles larger than the image, many images per tile, single-x-tile stem"),
    (64, [1.0, 0.7], 1, [2, 1], "box 64 on the latency plan"),
]

GEMM_INSTANTIATIONS = {  # every (block_n, epilogue, cg, b_resident, halo) find_conv_kernel returns a kernel for
    (64, EPI_TMA, 1, 1, 1), (64, EPI_TMA, 1, 0, 1), (64, EPI_TMA, 1, 1, 0), (64, EPI_TMA, 1, 0, 0),
    (128, EPI_TMA, 2, 0, 1), (128, EPI_TMA, 2, 0, 0), (256, EPI_TMA, 2, 0, 0), (64, EPI_TMA_RES, 1, 0, 0),
    (256, EPI_TMA_RES, 2, 0, 0), (96, EPI_PLANAR_F32, 1, 0, 0), (192, EPI_DECONV_HEAD, 2, 0, 0)}


def _inputs(eng, n):
    frames = np.stack([synth.frame_c2(i, eng.box_size) for i in range(-(-n // len(eng.scales)))])
    return eng.preprocess(frames)[0][:n]  # the fp16 network input, as float32


def _check_forward(eng, x, label, report):
    """forward(x), then every launch of it against its float64 reference; -> the maps"""
    assert np.array_equal(x.astype(np.float16).astype(np.float32), x)
    maps = eng.forward(x)
    n = x.shape[0]
    P = report["params"]
    get = DeviceTaps(eng, n, x, maps, P.dev)
    names = eng.step_names()
    checked = 0
    for name in names:
        try:
            worst, flagged = check_launch(restate(name), get, P)
        except AssertionError as e:  # report every failing launch of the matrix, then fail
            report["failures"].append(f"[{label} n={n}] {e}")
            print(f"  [{label} n={n}] {name:46s} FAILED: {e}")
            continue
        checked += 1
        report["worst"][name] = [max(a, b) for a, b in zip(report["worst"].get(name, (0.0, 0.0)), worst)]
        print(f"  [{label} n={n}] {name:46s} max err/bound {worst[0]:.4f} (fp32 term used {worst[1]:.4f})  rejected: "
              + " ".join(f"{k}={v}" for k, v in flagged.items()))
    assert len(names) == eng.info("launches_per_forward")
    print(f"  [{label} n={n}] launches checked: {checked} of launches_per_forward = "
          f"{int(eng.info('launches_per_forward'))}")
    del get
    torch.cuda.empty_cache()
    return maps


def _host_taps(eng, n):
    return {o: eng.tap(o, n) for name in eng.step_names() for o in io_names(restate(name))[1] if o != "<maps>"}


@pytest.mark.gpu
def test_every_launch_against_float64(w1):
    from vnect_b200 import VNectEngine
    print(f"\ncard: {_card()}")
    report = {"params": Params(w1, "cuda"), "worst": {}, "failures": []}
    paths, spread = [], {}
    for box, scales, max_frames, ns, why in MATRIX:
        eng = VNectEngine(w1, scales, box, max_frames=max_frames, max_streams=max_frames)
        try:
            cap = int(eng.info("max_forwards"))
            plan = "throughput" if cap > 8 else "latency"
            label = f"{box}/{plan}({cap})"
            print(f"{label}: {why}")
            sp = eng.step_paths()
            paths.append(sp)
            sms = int(eng.info("num_sms"))
            for n in ns:
                x = _inputs(eng, n)
                maps = _check_forward(eng, x, label, report)
                for name, path in zip(eng.step_names(), sp):
                    st = restate(name)
                    cout = eng.tap(st["out"], 1).shape[-1] if st["out"] != "<maps>" else 84
                    spread[name] = max(spread.get(name, 0), _units_per_worker(path, cout, n, box, sms))
            if box == 368 and plan == "throughput":
                # the 5-forward call after the 128-forward one equals a fresh engine's, launch by launch
                after, maps_after = _host_taps(eng, 5), maps
                fresh = VNectEngine(w1, scales, box, max_frames=max_frames, max_streams=max_frames)
                try:
                    maps_fresh = fresh.forward(x)
                    ref = _host_taps(fresh, 5)
                finally:
                    fresh.close()
                assert after.keys() == ref.keys()
                for k in after:
                    assert np.array_equal(after[k], ref[k]), f"5 forwards after 128: {k} differs from a fresh engine"
                assert all(np.array_equal(a, b) for a, b in zip(maps_after, maps_fresh))
                print(f"  [{label}] 5 forwards after 128: {len(after)} activations and the maps bit-identical to a "
                      "fresh engine's")
                # graph path: the third estimate replays a captured graph; its activations are forward()'s
                frames = np.stack([synth.frame_c2(50 + i, box) for i in range(3)])
                for k in range(3):
                    eng.estimate(frames, t2d=np.full(3, 10.0 + k), t3d=np.full(3, 10.0 + k))
                assert eng.info("cached_graphs") >= 1
                replay = _host_taps(eng, 3 * len(scales))
                eng.forward(eng.preprocess(frames)[0])
                direct = _host_taps(eng, 3 * len(scales))
                for k in replay:
                    assert np.array_equal(replay[k], direct[k]), f"graph replay: {k} differs from forward()"
                print(f"  [{label}] third estimate (graph replay): {len(replay)} activations bit-identical to "
                      "forward(preprocess(frames))")
        finally:
            eng.close()
        torch.cuda.empty_cache()

    # coverage, from what the library reports
    convs = [p for sp in paths for p in sp if p["kind"] == "conv"]
    inst = {(p["block_n"], p["epi"], p["cg"], p["b_resident"], p["halo"]) for p in convs if not p["n2"]}
    tails = {(p["n2"], p["epi"]) for p in convs if p["n2"]}
    stems = {(p["cg"], p["n_xt"]) for sp in paths for p in sp if p["kind"] == "stem"}
    kinds = {"flat": any(p["mode"] == 0 and not p["im2col"] for p in convs),
             "spatial": any(p["mode"] == 1 and not p["halo"] and not p["b_resident"] for p in convs),
             "halo": any(p["halo"] for p in convs), "resident": any(p["b_resident"] for p in convs),
             "im2col": any(p["im2col"] for p in convs)}
    print(f"coverage: GEMM instantiations {sorted(inst)}")
    print(f"coverage: block tails (n2, epilogue) {sorted(tails)}; stem (cg, x tiles) {sorted(stems)}; paths {kinds}")
    assert inst == GEMM_INSTANTIATIONS
    assert tails == {(64, EPI_TMA), (128, EPI_TMA_RES)}
    assert stems == {(1, 1), (2, 2), (1, 3)}
    assert all(kinds.values())
    print("largest tiles / units per CTA over the matrix, per launch: "
          + ", ".join(f"{k} {v}" for k, v in spread.items()))
    assert all(v >= 2 for v in spread.values()), {k: v for k, v in spread.items() if v < 2}
    print(f"largest err / bound over the matrix: {max(w[0] for w in report['worst'].values()):.4f}; largest share of "
          f"the fp32 term used: {max(w[1] for w in report['worst'].values()):.4f}")
    assert not report["failures"], "\n".join(report["failures"])
