#!/usr/bin/env python3
"""Oriented streams against identity ones, and against what callers without per-stream orientation do instead, on the
mixed_bench workload: 64 streams (22 frames of 480x640, 21 of 720x1280, 21 of 1080x1920), scales [1.0, 0.7], seeded
W0 weights, random frames, BGR and NV12.  Legs, each timed for at least --seconds with CUDA events on the engine's
stream, every leg run --rounds times in turn so the spread between rounds of one leg is visible next to the gaps:

* device: frames resident in device memory, one estimate_device_frames call per step with every stream set to
  identity, rot90_cw, transpose or rot180;
* host_pinned_2lanes: frames in pinned host memory, one submit_frames call per step alternating the two lanes, the
  same four orientations;
* workaround legs (BGR): device = torch.rot90(frame, -1).contiguous() per frame into a second buffer, then the identity
  device call; host = np.ascontiguousarray(np.rot90(frame, 3)) per frame on the host (its time included: the events
  span the host loop), then the identity two-lane host call.

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
ORIENTED = ("identity", "rot90_cw", "transpose", "rot180")


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None, help="JSON results file")
    args = ap.parse_args()
    import torch
    from vnect_b200 import VNectEngine
    from vnect_b200.weights import seeded_init

    eng = VNectEngine(seeded_init("W0"), SCALES, BOX, max_frames=N, max_streams=N, max_input=(1920, 1920))
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng.set_cuda_stream(stream.cuda_stream)
    clock = {"t": 1000.0}

    def stamps(n):
        clock["t"] += 1.0 / 30
        return np.full(n, clock["t"]), np.full(n, clock["t"] + 0.004)

    ids = np.arange(N, dtype=np.int32)
    d_j2 = torch.empty((N, 21, 2), dtype=torch.float64, device="cuda")
    d_j3 = torch.empty((N, 21, 3), dtype=torch.float32, device="cuda")
    h_out = [(torch.empty((N, 21, 2), dtype=torch.float64).pin_memory().numpy(),
              torch.empty((N, 21, 3), dtype=torch.float32).pin_memory().numpy()) for _ in range(2)]
    res = {"card": card(), "streams": N, "groups": [f"{n} x {h}x{w}" for n, (h, w) in GROUPS], "scales": SCALES,
           "box": BOX, "min_seconds": args.seconds, "rounds": args.rounds, "legs": []}
    rng = np.random.default_rng(0)
    sizes = [hw for n, hw in GROUPS for _ in range(n)]
    lane = {"k": 0}

    def next_lane():
        k = lane["k"] % 2
        lane["k"] += 1
        eng.wait(k)  # the batch this lane carried two calls ago
        return k

    for fmt in ("bgr", "nv12"):
        shape = (lambda h, w: (h, w, 3)) if fmt == "bgr" else (lambda h, w: (h * 3 // 2, w))
        pinned = [torch.from_numpy(rng.integers(0, 256, shape(h, w), dtype=np.uint8)).pin_memory() for h, w in sizes]
        host_frames = [p.numpy() for p in pinned]
        dev_frames = [p.cuda() for p in pinned]
        torch.cuda.synchronize()
        descs = [dict(ptr=d.data_ptr(), h=h, w=w) for d, (h, w) in zip(dev_frames, sizes)]
        kw = {"pixel_format": fmt}

        def device_call(descs_=descs):
            t2, t3 = stamps(N)
            eng.estimate_device_frames(descs_, d_j2.data_ptr(), d_j3.data_ptr(), ids, t2, t3, **kw)

        def host_call(frames_=host_frames):
            k = next_lane()
            t2, t3 = stamps(N)
            eng.submit_frames(k, frames_, ids, t2, t3, out=h_out[k], **kw)

        legs = [("device", o, device_call) for o in ORIENTED] + [("host_pinned_2lanes", o, host_call) for o in ORIENTED]
        if fmt == "bgr":
            rotated = [torch.empty((w, h, 3), dtype=torch.uint8, device="cuda") for h, w in sizes]
            rot_descs = [dict(ptr=r.data_ptr(), h=w, w=h) for r, (h, w) in zip(rotated, sizes)]

            def device_workaround():
                for r, d in zip(rotated, dev_frames):
                    r.copy_(torch.rot90(d, -1, dims=(0, 1)).contiguous())
                device_call(rot_descs)

            def host_workaround():
                host_call([np.ascontiguousarray(np.rot90(f, 3)) for f in host_frames])

            legs += [("device", "workaround_torch_rot90", device_workaround),
                     ("host_pinned_2lanes", "workaround_np_rot90", host_workaround)]
        for rnd in range(args.rounds):
            for path, orient, step in legs:
                eng.reset()
                eng.set_orientations(ids, ["identity" if orient.startswith("workaround") else orient] * N)
                steps, ms = timed(step, stream, args.seconds)
                eng.wait(0)
                eng.wait(1)
                leg = {"format": fmt, "path": path, "orientation": orient, "round": rnd, "steps": steps,
                       "ms": round(ms, 2), "ms_per_step": round(ms / steps, 3),
                       "frames_per_s": round(steps * N / (ms * 1e-3), 1)}
                res["legs"].append(leg)
                print(json.dumps(leg), flush=True)
        del dev_frames, pinned
        if fmt == "bgr":
            del rotated
    print("card:", res["card"])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
