#!/usr/bin/env python3
"""BGR vs NV12 input on C2-like batches (64 frames, scales [1.0, 0.7], seeded W0 weights, random frames), two frame
sizes, at least --seconds of work per leg, timed with CUDA events on the engine's stream:

* device: frames resident in device memory, VNectEngine.estimate_device back to back;
* host: frames in pinned host memory, submit / wait alternating the two lanes (the copy of one batch overlaps the
  kernels of the other).

Prints frames/s and the bytes copied to the device per frame (from the shapes), with the card's name and power limit
read in the same run, and writes the same as JSON to --out.  Needs a CUDA device.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, SCALES, BOX = 64, [1.0, 0.7], 368


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def timed(step, stream, seconds):
    """Runs step() until `seconds` of device time have passed (after a warm-up); returns (steps, ms)."""
    import torch
    for _ in range(3):  # warm-up, graph capture, first replay
        step()
    torch.cuda.synchronize()
    reps = 8
    while True:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            step()
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if ms >= seconds * 1e3:
            return reps, ms
        reps = int(reps * min(8.0, 1.2 * seconds * 1e3 / max(ms, 1e-3))) + 1


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--out", default=None, help="JSON results file")
    args = ap.parse_args()
    import cv2
    import torch
    from vnect_b200 import VNectEngine
    from vnect_b200.weights import seeded_init

    eng = VNectEngine(seeded_init("W0"), SCALES, BOX, max_frames=N, max_streams=N, max_input=(540, 960))
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng.set_cuda_stream(stream.cuda_stream)
    ids = np.arange(N, dtype=np.int32)
    clock = {"t": 1000.0}

    def stamps():
        clock["t"] += 1.0 / 30
        return np.full(N, clock["t"]), np.full(N, clock["t"] + 0.004)

    d_j2 = torch.empty((N, 21, 2), dtype=torch.float64, device="cuda")
    d_j3 = torch.empty((N, 21, 3), dtype=torch.float32, device="cuda")
    h_out = [(torch.empty((N, 21, 2), dtype=torch.float64).pin_memory().numpy(),
              torch.empty((N, 21, 3), dtype=torch.float32).pin_memory().numpy()) for _ in range(2)]
    res = {"card": card(), "frames_per_batch": N, "scales": SCALES, "box": BOX, "min_seconds": args.seconds,
           "legs": []}
    rng = np.random.default_rng(0)
    for h, w in [(368, 368), (540, 960)]:
        nv12 = rng.integers(0, 256, (N, h * 3 // 2, w), dtype=np.uint8)
        bgr = np.stack([cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12) for f in nv12])
        for fmt, frames in (("bgr", bgr), ("nv12", nv12)):
            bytes_per_frame = frames[0].nbytes
            pinned = torch.from_numpy(frames).pin_memory()
            dev = pinned.cuda()
            torch.cuda.synchronize()
            kw = {} if fmt == "bgr" else {"pixel_format": fmt}

            def device_step():
                t2, t3 = stamps()
                eng.estimate_device(dev.data_ptr(), N, h, w, d_j2.data_ptr(), d_j3.data_ptr(), ids, t2, t3, **kw)

            host = pinned.numpy()
            lane = {"k": 0}

            def host_step():
                k = lane["k"] % 2
                lane["k"] += 1
                eng.wait(k)  # the batch this lane carried two steps ago
                t2, t3 = stamps()
                eng.submit(k, host, ids, t2, t3, out=h_out[k], **kw)

            for path, step, h2d in (("device", device_step, 0), ("host_pinned_2lanes", host_step, bytes_per_frame)):
                steps, ms = timed(step, stream, args.seconds)
                eng.wait(0)
                eng.wait(1)
                leg = {"size": f"{h}x{w}", "format": fmt, "path": path, "steps": steps, "ms": round(ms, 2),
                       "frames_per_s": round(steps * N / (ms * 1e-3), 1), "h2d_bytes_per_frame": h2d}
                res["legs"].append(leg)
                print(json.dumps(leg), flush=True)
    print("card:", res["card"])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    eng.close()


if __name__ == "__main__":
    main()
