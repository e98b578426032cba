#!/usr/bin/env python3
"""One mixed-size call against three calls grouped by size, on a multi-camera batch: 64 streams (22 frames of 480x640,
21 of 720x1280, 21 of 1080x1920), scales [1.0, 0.7], seeded W0 weights, random frames, BGR and NV12.  Legs, each timed
for at least --seconds with CUDA events on the engine's stream:

* device: frames resident in device memory.  mixed = one estimate_device_frames call per step, every frame in its own
  allocation; grouped = three estimate_device calls per step on one strided buffer per size (frames already grouped,
  i.e. without the gather copy a caller with separately allocated frames would need: the grouped path's best case);
* host_pinned_2lanes: frames in pinned host memory, calls alternating the two lanes (wait for a lane, then submit on
  it).  mixed = one submit_frames call per step, grouped = three submit calls per step;
* tracked: host frames, one track_frames call against three track calls per step (each synchronises).

Prints frames/s with the card's name and power limit read in the same run, and writes the same as JSON to --out.
Needs a CUDA device.
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from yuv_bench import ROOT, card, timed  # noqa: E402

sys.path.insert(0, ROOT)

GROUPS, SCALES, BOX = [(22, (480, 640)), (21, (720, 1280)), (21, (1080, 1920))], [1.0, 0.7], 368
N = sum(n for n, _ in GROUPS)


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
    group_ids, lo = [], 0
    for n, _ in GROUPS:
        group_ids.append(ids[lo:lo + n])
        lo += n
    d_j2 = torch.empty((N, 21, 2), dtype=torch.float64, device="cuda")
    d_j3 = torch.empty((N, 21, 3), dtype=torch.float32, device="cuda")
    h_out = [(torch.empty((N, 21, 2), dtype=torch.float64).pin_memory().numpy(),
              torch.empty((N, 21, 3), dtype=torch.float32).pin_memory().numpy()) for _ in range(2)]
    res = {"card": card(), "streams": N, "groups": [f"{n} x {h}x{w}" for n, (h, w) in GROUPS], "scales": SCALES,
           "box": BOX, "min_seconds": args.seconds, "legs": []}
    rng = np.random.default_rng(0)
    for fmt in ("bgr", "nv12"):
        shape = (lambda h, w: (h, w, 3)) if fmt == "bgr" else (lambda h, w: (h * 3 // 2, w))
        # one pinned host array per size (what the grouped calls take); the mixed calls take its frames one by one
        pinned = [torch.from_numpy(rng.integers(0, 256, (n, *shape(h, w)), dtype=np.uint8)).pin_memory()
                  for n, (h, w) in GROUPS]
        host_groups = [p.numpy() for p in pinned]
        host_frames = [f for g in host_groups for f in g]
        dev_groups = [p.cuda() for p in pinned]
        dev_frames = [torch.empty_like(p[i], device="cuda").copy_(p[i]) for p in pinned for i in range(len(p))]
        torch.cuda.synchronize()
        sizes = [hw for n, hw in GROUPS for _ in range(n)]
        descs = [dict(ptr=d.data_ptr(), h=h, w=w) for d, (h, w) in zip(dev_frames, sizes)]
        kw = {} if fmt == "bgr" else {"pixel_format": fmt}

        def device_mixed():
            t2, t3 = stamps(N)
            eng.estimate_device_frames(descs, d_j2.data_ptr(), d_j3.data_ptr(), ids, t2, t3, **kw)

        def device_grouped():
            t2, t3 = stamps(N)
            o = 0
            for g, gid, (n, (h, w)) in zip(dev_groups, group_ids, GROUPS):
                eng.estimate_device(g.data_ptr(), n, h, w, d_j2[o].data_ptr(), d_j3[o].data_ptr(), gid, t2[:n],
                                    t3[:n], **kw)
                o += n

        lane = {"k": 0}

        def next_lane():
            k = lane["k"] % 2
            lane["k"] += 1
            eng.wait(k)  # the batch this lane carried two calls ago
            return k

        def host_mixed():
            k = next_lane()
            t2, t3 = stamps(N)
            eng.submit_frames(k, host_frames, ids, t2, t3, out=h_out[k], **kw)

        def host_grouped():
            t2, t3 = stamps(N)
            o = 0
            for g, gid in zip(host_groups, group_ids):
                k = next_lane()
                n = len(g)
                eng.submit(k, g, gid, t2[:n], t3[:n], out=(h_out[k][0][o:o + n], h_out[k][1][o:o + n]), **kw)
                o += n

        def tracked_mixed():
            t2, t3 = stamps(N)
            eng.track_frames(host_frames, ids, t2, t3, **kw)

        def tracked_grouped():
            t2, t3 = stamps(N)
            for g, gid in zip(host_groups, group_ids):
                eng.track(g, gid, t2[:len(g)], t3[:len(g)], **kw)

        for path, legs in (("device", (("mixed", device_mixed), ("grouped", device_grouped))),
                           ("host_pinned_2lanes", (("mixed", host_mixed), ("grouped", host_grouped))),
                           ("tracked", (("mixed", tracked_mixed), ("grouped", tracked_grouped)))):
            for mode, step in legs:
                eng.reset()
                steps, ms = timed(step, stream, args.seconds)
                eng.wait(0)
                eng.wait(1)
                leg = {"format": fmt, "path": path, "mode": mode, "calls_per_step": 1 if mode == "mixed" else 3,
                       "steps": steps, "ms": round(ms, 2), "ms_per_step": round(ms / steps, 3),
                       "frames_per_s": round(steps * N / (ms * 1e-3), 1)}
                res["legs"].append(leg)
                print(json.dumps(leg), flush=True)
        del dev_groups, dev_frames
    print("card:", res["card"])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
