#!/usr/bin/env python3
"""One recorded video through the engine: frames per second of a single stream at 540x960 (scales [1.0, 0.7], seeded
W0 weights, random frames), BGR and NV12, at least --seconds of work per leg, timed with CUDA events on the engine's
stream:

* one_per_call: one frame per call on a max_frames = 1 engine (estimate_device), the only exact option without
  sequence calls;
* seq64_host_2lanes / seq64_device: one stream as 64-frame sequence calls, pinned host frames submitted on alternating
  lanes (submit_sequence) or device-resident frames (estimate_device_sequence);
* seq8x8_device: 8 streams x 8 consecutive frames per call, interleaved;
* ceiling_host_2lanes / ceiling_device: 64 distinct streams per call (submit_frames / estimate_device_frames).

With --profile, instead: one torch.profiler run (CUDA activities) of 64-frame sequence calls and of 64-stream calls,
printing the device time of the post-process kernels (argmax, sequence scan, ordinary post-process) per call.
Prints the card's name and power limit read in the same run and writes everything as JSON to --out.  Needs a CUDA
device.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, SCALES, BOX, H, W = 64, [1.0, 0.7], 368, 540, 960


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def timed(step, stream, seconds):
    """Runs step() until `seconds` of device time have passed (after a warm-up); returns (steps, ms)."""
    import torch
    for _ in range(4):  # warm-up, graph capture, first replays (both lanes)
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


class Clock:
    """Per stream 1/30 s steps of an epoch-like clock."""

    def __init__(self):
        self.t = {}

    def take(self, ids):
        out = np.empty(len(ids))
        for i, s in enumerate(ids):
            self.t[s] = self.t.get(s, 1.7e9 + s) + 1.0 / 30
            out[i] = self.t[s]
        return out, out + 0.004


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--seconds", type=float, default=2.0)
    ap.add_argument("--profile", action="store_true", help="torch.profiler run of the post-process kernels instead")
    ap.add_argument("--out", default=None, help="JSON results file")
    args = ap.parse_args()
    import cv2
    import torch
    from vnect_b200 import VNectEngine
    from vnect_b200.weights import seeded_init

    w = seeded_init("W0")
    eng = VNectEngine(w, SCALES, BOX, max_frames=N, max_streams=N, max_input=(H, W))
    eng1 = VNectEngine(w, SCALES, BOX, max_frames=1, max_streams=1, max_input=(H, W))
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    for e in (eng, eng1):
        e.set_cuda_stream(stream.cuda_stream)
    clock = Clock()
    d_j2 = torch.empty((N, 21, 2), dtype=torch.float64, device="cuda")
    d_j3 = torch.empty((N, 21, 3), dtype=torch.float32, device="cuda")
    h_out = [(torch.empty((N, 21, 2), dtype=torch.float64).pin_memory().numpy(),
              torch.empty((N, 21, 3), dtype=torch.float32).pin_memory().numpy()) for _ in range(2)]
    res = {"card": card(), "size": f"{H}x{W}", "scales": SCALES, "box": BOX, "min_seconds": args.seconds, "legs": []}
    rng = np.random.default_rng(0)
    nv12 = rng.integers(0, 256, (N, H * 3 // 2, W), dtype=np.uint8)
    bgr = np.stack([cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12) for f in nv12])
    one = [0] * N
    ids8 = [int(s) for s in np.random.default_rng(1).permutation(np.repeat(np.arange(8), 8))]
    distinct = list(range(N))
    for fmt, frames in (("bgr", bgr), ("nv12", nv12)):
        pinned = torch.from_numpy(frames).pin_memory()
        dev = pinned.cuda()
        torch.cuda.synchronize()
        host = [pinned.numpy()[i] for i in range(N)]
        dtab = [dict(ptr=dev[i].data_ptr(), h=H, w=W) for i in range(N)]
        lane = {"k": 0}

        def one_per_call():
            t2, t3 = clock.take([0])
            eng1.estimate_device(dev[0].data_ptr(), 1, H, W, d_j2.data_ptr(), d_j3.data_ptr(), [0], t2, t3,
                                 pixel_format=fmt)

        def host_2lanes(submit, ids):
            def step():
                k = lane["k"] % 2
                lane["k"] += 1
                eng.wait(k)  # the batch this lane carried two steps ago
                t2, t3 = clock.take(ids)
                submit(k, host, ids, t2, t3, out=h_out[k], pixel_format=fmt)
            return step

        def device(fn, ids):
            def step():
                t2, t3 = clock.take(ids)
                fn(dtab, d_j2.data_ptr(), d_j3.data_ptr(), ids, t2, t3, pixel_format=fmt)
            return step

        legs = [("one_per_call", one_per_call, 1),
                ("seq64_host_2lanes", host_2lanes(eng.submit_sequence, one), N),
                ("seq64_device", device(eng.estimate_device_sequence, one), N),
                ("seq8x8_device", device(eng.estimate_device_sequence, ids8), N),
                ("ceiling_host_2lanes", host_2lanes(eng.submit_frames, distinct), N),
                ("ceiling_device", device(eng.estimate_device_frames, distinct), N)]
        if args.profile:
            from torch.profiler import ProfilerActivity, profile
            for name, step, n in legs:
                if name not in ("seq64_device", "seq8x8_device", "ceiling_device"):
                    continue
                for _ in range(4):
                    step()
                torch.cuda.synchronize()
                calls = 20
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(calls):
                        step()
                    torch.cuda.synchronize()
                kern = {}
                for ev in prof.key_averages():
                    if "postprocess_kernel" in ev.key or "sequence_filter_kernel" in ev.key:
                        dt = getattr(ev, "device_time_total", None)
                        if dt is None:
                            dt = ev.cuda_time_total
                        kern[ev.key[:90]] = round(dt / calls, 2)
                total = sum(getattr(ev, "device_time_total", 0) or 0 for ev in prof.key_averages()
                            if ev.device_type is not None and str(ev.device_type).endswith("CUDA"))
                leg = {"format": fmt, "leg": name, "profiled_calls": calls, "us_per_call": kern,
                       "all_kernels_us_per_call": round(total / calls, 1)}
                res["legs"].append(leg)
                print(json.dumps(leg), flush=True)
            continue
        for name, step, n in legs:
            steps, ms = timed(step, stream, args.seconds)
            eng.wait(0)
            eng.wait(1)
            leg = {"format": fmt, "leg": name, "frames_per_call": n, "steps": steps, "ms": round(ms, 2),
                   "frames_per_s": round(steps * n / (ms * 1e-3), 1), "ms_per_call": round(ms / steps, 4)}
            res["legs"].append(leg)
            print(json.dumps(leg), flush=True)
    print("card:", res["card"])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    eng.close()
    eng1.close()


if __name__ == "__main__":
    main()
