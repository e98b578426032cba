#!/usr/bin/env python3
"""What joint scores and lost-person recovery cost, each leg timed for at least --seconds with CUDA events on the
engine's stream, seeded W0 weights, random frames:

* c2: 64 frames of 368x368 per call, scales [1.0, 0.7], device frames and results (estimate_device), without and with
  dev_scores_ptr (a pool of four score buffers in rotation);
* tracked: the 64-stream mixed-size workload of track_bench.py (22 x 480x640, 21 x 720x1280, 21 x 1080x1920 in one
  call), device-resident (track_device_frames), recovery off and on.  The "on" leg gives every stream a threshold
  below every mean score seen in warm-up, so its crops are those of the "off" leg (checked: boxes_used of the first
  timed steps of both legs are compared, and the result is recorded).

The legs of each pair alternate twice (off, on, off, on) so that drift shows up as spread.  Prints ms per step and
frames/s with the card's name and power limit read in the same run, and writes the same as JSON to --out.  Needs a
CUDA device.
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from mixed_bench import BOX, GROUPS, N, SCALES  # noqa: E402
from yuv_bench import ROOT, card, timed  # noqa: E402

sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--out", default=None, help="JSON results file")
    args = ap.parse_args()
    import torch
    from vnect_b200 import VNectEngine
    from vnect_b200.weights import seeded_init

    w = seeded_init("W0")
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    clock = {"t": 1000.0}

    def stamps(n):
        clock["t"] += 1.0 / 30
        return np.full(n, clock["t"]), np.full(n, clock["t"] + 0.004)

    res = {"card": card(), "min_seconds": args.seconds, "legs": []}
    rng = np.random.default_rng(0)
    ids = np.arange(N, dtype=np.int32)
    pool = [torch.empty((N, 21), dtype=torch.float64, device="cuda") for _ in range(4)]
    d_j2 = torch.empty((N, 21, 2), dtype=torch.float64, device="cuda")
    d_j3 = torch.empty((N, 21, 3), dtype=torch.float32, device="cuda")
    d_boxes = torch.empty((N, 4), dtype=torch.int32, device="cuda")

    def record(leg, steps, ms, n_frames):
        leg.update(steps=steps, ms=round(ms, 2), ms_per_step=round(ms / steps, 3),
                   frames_per_s=round(steps * n_frames / (ms * 1e-3), 1))
        res["legs"].append(leg)
        print(json.dumps(leg), flush=True)

    # ---- c2: 64 box-size frames per call
    eng = VNectEngine(w, SCALES, BOX, max_frames=N, max_streams=N)
    eng.set_cuda_stream(stream.cuda_stream)
    frames = torch.from_numpy(rng.integers(0, 256, (N, BOX, BOX, 3), dtype=np.uint8)).cuda()
    k = {"i": 0}

    def c2(scores):
        def step():
            t2, t3 = stamps(N)
            sc = pool[k["i"] % len(pool)].data_ptr() if scores else None
            k["i"] += 1
            eng.estimate_device(frames.data_ptr(), N, BOX, BOX, d_j2.data_ptr(), d_j3.data_ptr(), ids, t2, t3,
                                dev_scores_ptr=sc)
        return step

    for rep in range(2):
        for scores in (False, True):
            eng.reset()
            steps, ms = timed(c2(scores), stream, args.seconds)
            record({"workload": "c2_device", "scores": scores, "rep": rep}, steps, ms, N)
    res["c2_cached_graphs"] = eng.info("cached_graphs")
    eng.close()
    del frames

    # ---- tracked: 64 mixed-size streams, device-resident
    eng = VNectEngine(w, SCALES, BOX, max_frames=N, max_streams=N, max_input=(1080, 1920))
    eng.set_cuda_stream(stream.cuda_stream)
    sizes = [hw for n, hw in GROUPS for _ in range(n)]
    rects = np.array([(w_ // 4, h // 4, w_ // 2, h // 2) for h, w_ in sizes], np.int32)
    dev = [torch.from_numpy(rng.integers(0, 256, (h, w_, 3), dtype=np.uint8)).cuda() for h, w_ in sizes]
    descs = [dict(ptr=d.data_ptr(), h=h, w=w_) for d, (h, w_) in zip(dev, sizes)]

    def tracked(scores_to=None):
        t2, t3 = stamps(N)
        eng.track_device_frames(descs, d_j2.data_ptr(), d_j3.data_ptr(), d_boxes.data_ptr(), ids, t2, t3,
                                dev_scores_ptr=scores_to)

    # warm-up with scores on: the least mean score any stream shows
    eng.reset()
    eng.set_boxes(ids, rects)
    means = []
    for _ in range(8):
        tracked(pool[0].data_ptr())
        torch.cuda.synchronize()
        means.append(pool[0].cpu().numpy().sum(axis=1) / 21)
    least = float(np.min(means))
    tau = least / 2 if least > 0 else 0.0
    res["tracked_warmup_least_mean_score"] = least
    res["tracked_threshold"] = tau
    first_boxes = {}
    for rep in range(2):
        for on in (False, True):
            eng.set_track_recovery(ids, np.full(N, tau if on else 0.0))
            eng.reset()
            eng.set_boxes(ids, rects)
            used = []
            for _ in range(4):
                tracked()
                used.append(d_boxes.cpu().numpy().copy())
            first_boxes.setdefault(on, used)
            steps, ms = timed(tracked, stream, args.seconds)
            record({"workload": "tracked_64_mixed_device", "recovery": on and tau > 0, "rep": rep}, steps, ms, N)
    res["tracked_crops_identical"] = all(np.array_equal(a, b) for a, b in zip(first_boxes[False], first_boxes[True]))
    print("card:", res["card"], "least warm-up mean score:", least, "threshold:", tau,
          "crops identical:", res["tracked_crops_identical"])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
