#!/usr/bin/env python3
"""Tracked video streams, synchronous against pipelined and device-resident, on the workload of mixed_bench.py: 64
streams per step (22 frames of 480x640, 21 of 720x1280, 21 of 1080x1920) in one mixed-size call, scales [1.0, 0.7],
seeded W0 weights, random frames, BGR and NV12, every stream's box seeded once per leg with set_boxes.  Legs, each
timed for at least --seconds with CUDA events on the engine's stream:

* tracked_sync: track_frames, which waits for every step;
* tracked_2lanes: submit_track_frames on pinned host frames into pinned results, alternating the two lanes (wait for
  a lane, then submit on it), so the upload of one step overlaps the kernels of the other;
* tracked_device: track_device_frames on device frames, each in its own allocation, device results;
* untracked_2lanes / untracked_device: submit_frames and estimate_device_frames on the same frames, the same way --
  the ceilings the tracked legs can approach.

Prints frames/s and ms per step with the card's name and power limit read in the same run, and writes the same as
JSON to --out.  Needs a CUDA device.
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

    eng = VNectEngine(seeded_init("W0"), SCALES, BOX, max_frames=N, max_streams=N, max_input=(1080, 1920))
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng.set_cuda_stream(stream.cuda_stream)
    clock = {"t": 1000.0}

    def stamps(n):
        clock["t"] += 1.0 / 30
        return np.full(n, clock["t"]), np.full(n, clock["t"] + 0.004)

    ids = np.arange(N, dtype=np.int32)
    sizes = [hw for n, hw in GROUPS for _ in range(n)]
    # a quarter of each frame, centred: a box a person detector might give
    rects = np.array([(w // 4, h // 4, w // 2, h // 2) for h, w in sizes], np.int32)
    d_j2 = torch.empty((N, 21, 2), dtype=torch.float64, device="cuda")
    d_j3 = torch.empty((N, 21, 3), dtype=torch.float32, device="cuda")
    d_boxes = torch.empty((N, 4), dtype=torch.int32, device="cuda")
    pinned = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()  # noqa: E731
    h_out = [(pinned((N, 21, 2), torch.float64), pinned((N, 21, 3), torch.float32), pinned((N, 4), torch.int32))
             for _ in range(2)]
    res = {"card": card(), "streams": N, "groups": [f"{n} x {h}x{w}" for n, (h, w) in GROUPS], "scales": SCALES,
           "box": BOX, "min_seconds": args.seconds, "legs": []}
    rng = np.random.default_rng(0)
    for fmt in ("bgr", "nv12"):
        shape = (lambda h, w: (h, w, 3)) if fmt == "bgr" else (lambda h, w: (h * 3 // 2, w))
        host = [torch.from_numpy(rng.integers(0, 256, shape(h, w), dtype=np.uint8)).pin_memory() for h, w in sizes]
        host_frames = [f.numpy() for f in host]
        dev_frames = [f.cuda() for f in host]
        torch.cuda.synchronize()
        descs = [dict(ptr=d.data_ptr(), h=h, w=w) for d, (h, w) in zip(dev_frames, sizes)]
        kw = {} if fmt == "bgr" else {"pixel_format": fmt}
        lane = {"k": 0}

        def next_lane():
            k = lane["k"] % 2
            lane["k"] += 1
            eng.wait(k)  # the step this lane carried two calls ago
            return k

        def tracked_sync():
            t2, t3 = stamps(N)
            eng.track_frames(host_frames, ids, t2, t3, **kw)

        def tracked_2lanes():
            k = next_lane()
            t2, t3 = stamps(N)
            eng.submit_track_frames(k, host_frames, ids, t2, t3, out=h_out[k], **kw)

        def tracked_device():
            t2, t3 = stamps(N)
            eng.track_device_frames(descs, d_j2.data_ptr(), d_j3.data_ptr(), d_boxes.data_ptr(), ids, t2, t3, **kw)

        def untracked_2lanes():
            k = next_lane()
            t2, t3 = stamps(N)
            eng.submit_frames(k, host_frames, ids, t2, t3, out=h_out[k][:2], **kw)

        def untracked_device():
            t2, t3 = stamps(N)
            eng.estimate_device_frames(descs, d_j2.data_ptr(), d_j3.data_ptr(), ids, t2, t3, **kw)

        for path, step in (("tracked_sync", tracked_sync), ("tracked_2lanes", tracked_2lanes),
                           ("tracked_device", tracked_device), ("untracked_2lanes", untracked_2lanes),
                           ("untracked_device", untracked_device)):
            eng.reset()
            eng.set_boxes(ids, rects)
            steps, ms = timed(step, stream, args.seconds)
            eng.wait(0)
            eng.wait(1)
            leg = {"format": fmt, "path": path, "steps": steps, "ms": round(ms, 2), "ms_per_step": round(ms / steps, 3),
                   "frames_per_s": round(steps * N / (ms * 1e-3), 1)}
            res["legs"].append(leg)
            print(json.dumps(leg), flush=True)
        del dev_frames
    print("card:", res["card"])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
