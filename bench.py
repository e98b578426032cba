#!/usr/bin/env python3
"""Benchmark of the VNect per-frame hot path (BASELINE.json: frames/s @368x368, 2 scales, on 1/2/4/8 B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A step = one pass of the hot path over one batch of 64 synthetic 368x368 BGR frames per GPU (config C2 of
SURVEY.md section 8d: scales [1.0, 0.7] => 128 CNN forwards), OneEuroFilter state live across steps (each frame slot is
a video stream).  For N > 1 launch with torchrun (one rank per GPU); streams are sharded, nothing is exchanged on the
compute path, and the per-step results are all-gathered with NCCL inside the timed region (weak scaling).
Extra keys of the same line: `sustained` (>= 2 s of back-to-back steps), `c4_strong_scaling` (BASELINE config 4: 256
streams sharded i mod G for 32 steps, total work fixed, plus the bit-for-bit check of the gathered results against a
single-GPU run), batch-1 latency.

value  = frames/s with the frames already resident in HBM (device-timed with CUDA events on the launch stream).
e2e    = frames/s through the public host API (pinned host frames in, host joints out; H2D/D2H inside the timed region).
roofline = the implicit-GEMM convolution kernel family (the dominant kernel): algorithmic FLOPs of the CNN
           (BASELINE.md section 3) / summed device time of its launches, against the measured bf16 tensor peak.
cpu_baseline = the CPU restatement of the reference (oracle/: torch-CPU fp32 CNN + cv2/numpy pre/post) on a bounded
           sample, timed on this box's host cores.  `--impl reference` times only that.

--dump-outputs DIR writes what the last of the K timed `value` steps returned to its caller: DIR/joints_2d.npy
(float64 [frames, 21, 2]) and DIR/joints_3d.npy (float32 [frames, 21, 3]) of rank 0, plus DIR/results_all.npy (the
gathered float64 [streams, 21, 5] rows) when N > 1.  Frames, weights and clock readings are seeded and the filter state
at that point depends only on --warmup and --steps, so two builds run with the same arguments can be compared file by
file.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BOX = 368
SCALES = [1.0, 0.7]
FRAMES_PER_GPU = 64
FLOPS_PER_FORWARD = 23_830_290_432  # BASELINE.md section 3 (reference graph, every conv at full resolution)
# res2c / res3d feed only stride-2 1x1 convs, and res2b feeds only res2c's residual add (src/vnect_model.py:56 wires
# res2c's 3x3 to res2b_branch2a), so the 3x3, last 1x1 and add of those three blocks are evaluated at even pixels only
# (identical results, DESIGN.md section 3): 3/4 of those six convs' MACs are not executed.  The roofline uses EXECUTED flops.
SKIPPED_FLOPS = 2 * 3 * (2 * (92 * 92 // 4) * (576 * 64 + 64 * 256) + (46 * 46 // 4) * (1152 * 128 + 128 * 512))
EXECUTED_FLOPS_PER_FORWARD = FLOPS_PER_FORWARD - SKIPPED_FLOPS
METRIC = "frames/sec @368x368 2-scale"
WORKLOAD = "C2: 64 synthetic 368x368 BGR frames per GPU per step, scales [1.0, 0.7] (128 CNN forwards), W0 seeded random-init weights, filters on"


def frame_c2(i, size=BOX):
    """C2 frame i (SURVEY.md section 8d): uniform-noise BGR image, seed 1000 + i."""
    return np.random.default_rng(1000 + i).integers(0, 256, (size, size, 3), dtype=np.uint8)


def stream_frame(stream, k, size=BOX):
    """C4 (SURVEY.md section 8d): frame k of synthetic stream `stream` = a fixed noise image (seed 2000 + stream)
    circularly shifted by (k, 2k) pixels, so the argmaxes move and the filters see motion."""
    base = np.random.default_rng(2000 + stream).integers(0, 256, (size, size, 3), dtype=np.uint8)
    return np.ascontiguousarray(np.roll(base, shift=(k, 2 * k), axis=(0, 1)))


C4_STREAMS = 256
C4_STEPS = 32


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                              ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_arm(n_frames, threads=None):
    """The reference's CPU path on the oracle restatement (TensorFlow 1.x is not installable: SURVEY.md section 8c).
    Returns frames/s over n_frames two-scale frames (after one warm-up frame)."""
    import torch
    from oracle import prepost, synth
    from oracle.forward import OracleNet
    from oracle.weights import make_weights
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    net = OracleNet(make_weights("W0"))
    clock = {"t": 1000.0}

    def tick():
        clock["t"] += 0.004
        return clock["t"]
    est = prepost.OracleEstimator(net, SCALES, clock=tick)
    est(synth.frame_c2(0))
    t0 = time.perf_counter()
    for i in range(n_frames):
        est(synth.frame_c2(i))
    dt = time.perf_counter() - t0
    return n_frames / dt, threads


def run_reference(args, out=sys.stdout):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = 8
    vals = []
    for _ in range(args.warmup):
        cpu_reference_arm(2)
    threads = os.cpu_count()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v, threads = cpu_reference_arm(n)
        vals.append(v)
    wall = time.perf_counter() - t0
    v = statistics.mean(vals)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": "CPU restatement of the reference (TensorFlow 1.x not installable); each step = %d frames" % n},
        "cpu_baseline": {"value": v, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": "%d two-scale 368x368 frames per step, oracle estimator (torch-CPU fp32 CNN + cv2/numpy pre/post)" % n},
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=out, flush=True)


def run_c4(eng, parallel, dev, stream, rank, world, local, barrier):
    """BASELINE.json config 4 as specified: 256 synthetic video streams x 32 steps, stream i on rank i mod G, results of
    every step all-gathered (NCCL).  Total work is fixed, so this is the STRONG-scaling curve.  Outside the timed region
    rank 0 recomputes all 256 streams alone and asserts the gathered [256, 21, 5] equal it bit for bit (SURVEY T6)."""
    import torch
    import torch.distributed as dist
    from vnect_b200 import VNectEngine
    from vnect_b200.weights import seeded_init
    per = parallel.slots_per_rank(C4_STREAMS, world)
    mine = parallel.owned_streams(C4_STREAMS, rank, world)
    assert len(mine) == per, "256 streams divide evenly over 1/2/4/8 ranks"
    ceng = VNectEngine(seeded_init("W0"), SCALES, BOX, max_frames=per, max_streams=per, device=local)
    ceng.set_cuda_stream(stream.cuda_stream)
    base = torch.from_numpy(np.stack([np.random.default_rng(2000 + s).integers(0, 256, (BOX, BOX, 3), dtype=np.uint8)
                                      for s in mine])).to(dev)
    frames = [torch.roll(base, shifts=(k, 2 * k), dims=(1, 2)).contiguous() for k in range(C4_STEPS)]  # == stream_frame
    d2 = torch.empty((per, 21, 2), dtype=torch.float64, device=dev)
    d3 = torch.empty((per, 21, 3), dtype=torch.float32, device=dev)
    packed = torch.zeros((per, 21, 5), dtype=torch.float64, device=dev)
    gathered = torch.empty((C4_STEPS, world * per, 21, 5), dtype=torch.float64, device=dev)
    ceng.set_packed_results(packed.data_ptr())
    ids = np.arange(per, dtype=np.int32)

    def run(record):
        ceng.reset()
        for k in range(C4_STEPS):
            t = 1000 + k / 30
            ceng.estimate_device(frames[k].data_ptr(), per, BOX, BOX, d2.data_ptr(), d3.data_ptr(), ids,
                                 np.full(per, t), np.full(per, t + 0.004))
            if world > 1:
                parallel.all_gather_packed(packed, gathered[k] if record else gathered[0])
            elif record:
                gathered[k].copy_(packed)

    run(False)  # warm-up: function attributes, CUDA graph capture, NCCL channels
    run(False)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    run(True)
    e1.record(stream)
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    out = {"streams": C4_STREAMS, "steps": C4_STEPS, "streams_per_gpu": per, "scaling": "strong",
           "value": C4_STREAMS * C4_STEPS / (ms * 1e-3), "unit": "frames/s", "ms_total": ms,
           "data": "synth.stream_frame streams resident in HBM, results all-gathered every step"}
    ceng.close()
    # ---- T6: the gathered results equal the single-GPU answer bit for bit (outside the timed region, rank 0 only)
    if rank == 0:
        got = gathered.cpu().numpy()[:, parallel.unshard_index(C4_STREAMS, world)]          # [steps, 256, 21, 5]
        chunk = 64
        seng = VNectEngine(seeded_init("W0"), SCALES, BOX, max_frames=chunk, max_streams=C4_STREAMS, device=local)
        seng.set_cuda_stream(stream.cuda_stream)
        sp = torch.zeros((chunk, 21, 5), dtype=torch.float64, device=dev)
        s2 = torch.empty((chunk, 21, 2), dtype=torch.float64, device=dev)
        s3 = torch.empty((chunk, 21, 3), dtype=torch.float32, device=dev)
        seng.set_packed_results(sp.data_ptr())
        want = np.empty_like(got)
        for c0 in range(0, C4_STREAMS, chunk):
            sb = torch.from_numpy(np.stack([np.random.default_rng(2000 + s).integers(0, 256, (BOX, BOX, 3), dtype=np.uint8)
                                            for s in range(c0, c0 + chunk)])).to(dev)
            for k in range(C4_STEPS):
                fr = torch.roll(sb, shifts=(k, 2 * k), dims=(1, 2)).contiguous()
                tt = 1000 + k / 30
                seng.estimate_device(fr.data_ptr(), chunk, BOX, BOX, s2.data_ptr(), s3.data_ptr(),
                                     np.arange(c0, c0 + chunk, dtype=np.int32), np.full(chunk, tt), np.full(chunk, tt + 0.004))
                torch.cuda.synchronize()
                want[k, c0:c0 + chunk] = sp.cpu().numpy()
        seng.close()
        same = bool(np.array_equal(got, want))
        out["bit_identical_to_single_gpu"] = same
        if not same:
            bad = np.argwhere(np.any(got != want, axis=(2, 3)))
            out["first_mismatch_step_stream"] = [int(v) for v in bad[0]]
        assert same, "C4: gathered multi-GPU results differ from the single-GPU run"
    return out


def claim_stdout():
    """stdout must carry exactly ONE JSON line, but NCCL (and anything else in C) writes its log to file descriptor 1
    unless NCCL_DEBUG_FILE says otherwise.  Point fd 1 at stderr for the whole run and keep the real stdout for the
    result line: nothing is muted, it just lands on stderr."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main():
    out = claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=FRAMES_PER_GPU, help="frames per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="skip the C4 strong-scaling leg (256 streams x 32 steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args, out)

    import torch
    import torch.distributed as dist
    from vnect_b200 import VNectEngine
    from vnect_b200.weights import seeded_init
    from vnect_b200 import parallel

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}; launch with torchrun for N>1", file=sys.stderr)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # stdout carries exactly one JSON line; NCCL's own log (version, "nranks N" of the communicator) goes to
        # stderr instead of being muted, so the rank count of the gather can be read from the run's log
        # (whatever the launcher set wins; the image's default level VERSION is raised to INFO so that the communicator's
        # "nranks" line exists in the log, wherever NCCL_DEBUG_FILE points)
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "INFO"
            os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
        dist.init_process_group("nccl", device_id=dev)
    nf = args.frames
    n_streams = nf * world

    eng = VNectEngine(seeded_init("W0"), SCALES, BOX, max_frames=nf, max_streams=nf, device=local)
    # a dedicated (capturable) torch stream is made current and handed to the engine: the engine's kernels, the
    # torch.cuda.Event timers and the NCCL gather all live on it
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    eng.set_cuda_stream(stream.cuda_stream)

    # synthetic frames: stream s = global frame slot; pinned host copy for the e2e leg, device copy for `value`
    my_streams = parallel.owned_streams(n_streams, rank, world)
    host_frames = torch.empty((nf, BOX, BOX, 3), dtype=torch.uint8).pin_memory()
    hf = host_frames.numpy()
    for i, s in enumerate(my_streams):
        hf[i] = frame_c2(s)
    dev_frames = host_frames.to(dev)
    d_j2 = torch.empty((nf, 21, 2), dtype=torch.float64, device=dev)
    d_j3 = torch.empty((nf, 21, 3), dtype=torch.float32, device=dev)
    # the exchange buffer of the gather: the post-process kernel itself writes (row, col, x, y, z) float64 here
    d_packed = torch.zeros((nf, 21, 5), dtype=torch.float64, device=dev)
    g_all = torch.empty((world * nf, 21, 5), dtype=torch.float64, device=dev)
    eng.set_packed_results(d_packed.data_ptr())
    ids = np.arange(nf, dtype=np.int32)
    tclock = {"t": 1000.0}

    def stamps():
        tclock["t"] += 1.0 / 30
        return np.full(nf, tclock["t"]), np.full(nf, tclock["t"] + 0.004)

    def device_step():
        t2, t3 = stamps()
        eng.estimate_device(dev_frames.data_ptr(), nf, BOX, BOX, d_j2.data_ptr(), d_j3.data_ptr(), ids, t2, t3)
        if world > 1:
            parallel.all_gather_packed(d_packed, g_all)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- value: device-resident, CUDA-event timed
    for _ in range(max(args.warmup, 3)):
        device_step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = eng.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        device_step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = eng.launch_count() - launches0
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = n_streams * args.steps / (ms_max * 1e-3)
    # results of the last timed step, taken before the legs below move the filters on by a timing-dependent step count
    if args.dump_outputs and rank == 0:
        dump = {"joints_2d": d_j2.cpu().numpy(), "joints_3d": d_j3.cpu().numpy()}
        if world > 1:
            dump["results_all"] = g_all.cpu().numpy()[parallel.unshard_index(n_streams, world)]
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    # the GEMM family's own time for the roofline, taken here: same thermal / power state as the `value` leg just timed
    # (after the 2 s sustained leg further down the chip sits at its power cap and the forward measures 10-15 % longer)
    fwd_ms, per = eng.time_forward(nf * len(SCALES), reps=3, per_layer=True)
    conv_ms = sum(per.values())  # every launch of one forward batch is an implicit-GEMM kernel (pool1 is fused)
    # A timed step is: pyramid kernel, the family's launches, post-process kernel -- nothing else sits in the stream.  The
    # family's time INSIDE the timed region is therefore this rank's step time minus the two small kernels (timed alone,
    # ~2 % of a step); fwd_ms above is the same forward launched kernel by kernel outside the graph, kept as a second view.
    pre_ms, post_ms = eng.time_prepost(nf, reps=5)
    tclock["t"] += 10.0  # time_prepost advanced the streams' clocks on its own
    fam_ms = ms / args.steps - pre_ms - post_ms

    # ---------------------------------------------------------------- e2e: host frames in, host joints out
    # Public host API, pinned host frames -> pinned host joints, two submission lanes so the H2D copy of batch k+1
    # overlaps the kernels of batch k.  Every step copies its 26 MB of frames to the device and its joints back.
    outs = []
    for _ in range(2):
        a = torch.empty((nf, 21, 2), dtype=torch.float64).pin_memory()
        b = torch.empty((nf, 21, 3), dtype=torch.float32).pin_memory()
        outs.append((a.numpy(), b.numpy(), a, b))
    j2h, j3h = outs[0][0], outs[0][1]

    # cross-rank gather of a finished step's results: device-side, asynchronous, waited one step later so that it
    # never stalls the submission pipeline (the only collective on the path, 21 x 5 numbers per frame)
    g_in = [torch.empty((nf, 21, 5), dtype=torch.float64, device=dev) for _ in range(2)]
    g_out = [torch.empty((world * nf, 21, 5), dtype=torch.float64, device=dev) for _ in range(2)]
    g_work = [None, None]

    def gather(lane):
        if world == 1:
            return
        if g_work[lane] is not None:
            g_work[lane].wait()
        # the batch of this lane has completed (wait(lane)); d_packed holds a LATER batch by now, so the slots are
        # refilled from the lane's host results (vnect_b200.parallel layout)
        g_in[lane][:, :, :2].copy_(outs[lane][2], non_blocking=True)
        g_in[lane][:, :, 2:].copy_(outs[lane][3], non_blocking=True)
        _, g_work[lane] = parallel.all_gather_packed(g_in[lane], g_out[lane], async_op=True)

    def e2e_steps(k):
        for i in range(k):
            lane = i & 1
            if i >= 2:
                eng.wait(lane)
                gather(lane)
            t2, t3 = stamps()
            eng.submit(lane, hf, ids, t2, t3, out=(outs[lane][0], outs[lane][1]))
        for i in range(max(k - 2, 0), k):
            eng.wait(i & 1)
            gather(i & 1)
        for w in g_work:
            if w is not None:
                w.wait()

    e2e_steps(3)
    barrier()
    t0 = time.perf_counter()
    e2e_steps(args.steps)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = n_streams * args.steps / float(t.item())
    clocks = sampler.stop() if rank == 0 else None  # sampled across both timed regions (value and e2e)

    # ---------------------------------------------------------------- sustained figure (>= 2 s of back-to-back steps)
    barrier()
    sus_steps = max(args.steps, int(2.2 / max(ms_max / args.steps * 1e-3, 1e-5)))
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record(stream)
    for _ in range(sus_steps):
        device_step()
    s1.record(stream)
    barrier()
    t = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sustained = {"value": n_streams * sus_steps / (float(t.item()) * 1e-3), "unit": "frames/s", "steps": sus_steps,
                 "seconds": float(t.item()) * 1e-3}

    # ---------------------------------------------------------------- C4: 256 streams sharded i mod G, strong scaling
    c4 = run_c4(eng, parallel, dev, stream, rank, world, local, barrier) if not args.no_c4 else None

    # ---------------------------------------------------------------- roofline of the conv-GEMM kernel family
    # (fwd_ms / per were taken right after the `value` leg, see there)
    peaks, peak_src = measured_peaks()
    # the family's launch time inside a step (fam_ms, see above); the forward launched outside the graph (fwd_ms) and the
    # sum of the layers timed one by one (conv_ms, a launch ramp per layer) are kept as second views.
    # Flops: the ones EXECUTED (res2b / res2c / res3d are evaluated at even pixels only); the reference graph's count
    # (SURVEY.md section 8d, 23.83 GFLOP per forward) gives frac_algorithmic.
    achieved = EXECUTED_FLOPS_PER_FORWARD * nf * len(SCALES) / (fam_ms * 1e-3) / 1e12
    achieved_alg = FLOPS_PER_FORWARD * nf * len(SCALES) / (fam_ms * 1e-3) / 1e12
    achieved_ser = EXECUTED_FLOPS_PER_FORWARD * nf * len(SCALES) / (conv_ms * 1e-3) / 1e12
    peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    traffic, traffic_note = None, None
    try:  # DRAM traffic of the same launches from the committed ncu capture (profiles/conv_traffic.json names its source)
        with open(os.path.join(ROOT, "profiles", "conv_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("frames_per_step") == nf:
            import hashlib
            traffic = tj["conv_family_dram_bytes_per_step"]
            with open(os.path.join(ROOT, "profiles", "conv_traffic.json"), "rb") as fb:
                digest = hashlib.sha256(fb.read()).hexdigest()[:16]
            traffic_note = ("dram__bytes_read.sum + dram__bytes_write.sum summed over the family's launches of one step, "
                            + tj["source"] + "; NOT measured in this run: read from profiles/conv_traffic.json (sha256 "
                            + digest + ", captured at commit " + str(tj.get("captured_at_commit")) + ")")
    except Exception:
        pass
    roofline = {"bound": "tensor", "kernel": "conv_gemm_kernel<*> (implicit-GEMM conv family, %d launches per forward batch)" % (len(per) - 1),
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "peak_source": "%s MEASURED_PEAKS.json bf16_tflops_sustained (burst %.1f)" % (peak_src, peaks["bf16_tflops"]),
                "traffic": traffic, "traffic_note": traffic_note,
                "hbm_view": None if traffic is None else {
                    "achieved_gbs": traffic / (fam_ms * 1e-3) / 1e9, "peak_gbs": peaks["hbm_gbs"],
                    "frac": traffic / (fam_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                    "note": "the family mixes tensor-bound 3x3 convs with HBM-bound 1x1 expand convs; per-launch numbers in profiles/r02_step_traffic.txt"},
                "frac_of_burst": achieved / peaks["bf16_tflops"],
                "frac_algorithmic": achieved_alg / peak, "frac_algorithmic_of_burst": achieved_alg / peaks["bf16_tflops"],
                "frac_layers_timed_one_by_one": achieved_ser / peak,
                "time_basis": "family_ms_in_step: this rank's timed step (CUDA events over the %d steps of `value`) minus the pyramid and post-process kernels timed alone; a step's stream holds nothing but those two and the family's %d launches" % (args.steps, len(per)),
                "family_ms_in_step": fam_ms, "pre_ms": pre_ms, "post_ms": post_ms,
                "frac_forward_outside_graph": EXECUTED_FLOPS_PER_FORWARD * nf * len(SCALES) / (fwd_ms * 1e-3) / 1e12 / peak,
                "conv_ms_per_batch": conv_ms, "forward_ms_per_batch": fwd_ms,
                "flops_per_forward_executed": EXECUTED_FLOPS_PER_FORWARD, "flops_per_forward_reference": FLOPS_PER_FORWARD}

    # ---------------------------------------------------------------- batch-1 latency (C3-style: one stream, filters on)
    # measured on a latency plan (max_frames = 1, what the drop-in VNectEstimator builds): host frame in, host joints out
    lat = []
    if rank == 0:
        lat_eng = VNectEngine(seeded_init("W0"), SCALES, BOX, max_frames=1, max_streams=1, device=local)
        one = hf[:1]
        o2 = np.empty((1, 21, 2), np.float64)
        o3 = np.empty((1, 21, 3), np.float32)
        for k in range(60):
            tclock["t"] += 1.0 / 30
            t0 = time.perf_counter()
            lat_eng.estimate(one, [0], [tclock["t"]], [tclock["t"] + 0.004], out=(o2, o3))
            lat.append((time.perf_counter() - t0) * 1e3)
        lat = sorted(lat[10:])
        lat_eng.close()

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world >= 1:
            n_cpu = 12
            v, threads = cpu_reference_arm(n_cpu)
            cpu = {"value": v, "unit": "frames/s", "cores": threads, "kind": "port",
                   "sample": "%d two-scale 368x368 frames of the same workload through the oracle estimator (torch-CPU fp32 CNN + cv2/numpy pre/post; TF1 not installable)" % n_cpu}
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_gpu_per_step": nf, "box_size": BOX, "scales": SCALES,
                       "precision": "fp16 operands, fp32 accumulate (TMEM)",
                       "l2": "per-step working set (~8 GB of activations) exceeds the 126 MB L2; no flush needed",
                       "sharding": "streams round-robin over ranks, results all-gathered (NCCL) each step" if world > 1 else "single GPU"},
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": int(hf.nbytes) * world,
                    "d2h_bytes_per_step": int(j2h.nbytes + j3h.nbytes) * world},
            "gpu_launches": int(launches) * world,
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "sustained": sustained,
            "c4_strong_scaling": c4,
            "latency_ms_p50_batch1": statistics.median(lat) if lat else None,
            "latency_ms_p95_batch1": lat[int(0.95 * (len(lat) - 1))] if lat else None,
        }
        print(json.dumps(line), file=out, flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
