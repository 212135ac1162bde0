#!/usr/bin/env python
"""Benchmark of the B200-native Unicorn per-frame hot path (contract: see the task statement / DESIGN.md §Measurement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NAME] [--size H W] [--dump-outputs DIR]

A step = one steady-state SOT frame (BASELINE.json configs[1]: unicorn_track_large, 800x1280): backbone+neck ->
deformable interaction -> 2x embedding upsample -> fused correlation/propagation -> head -> NMS, on synthetic video
with seeded random weights.  `value` = frames/s with frames resident in HBM (CUDA events, max over ranks);
`e2e` = frames/s through UnicornSOTTrack.track_tensor with pinned HOST frames (H2D + D2H inside the timed region).
`--impl reference` times the reference algorithm's CPU restatement (oracle/, validated against the real reference)
on the host cores for the same workload.
Every frames/s figure of either impl times exactly `--steps` frames; only the kernel microbenchmarks and the `cpu_baseline`
sample have fixed counts of their own.  Inputs and weights are seeded, so `--dump-outputs` of two builds run with
the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAME_GFLOP = {"unicorn_track_large": 1997.0, "unicorn_track_tiny": 54.9}  # SURVEY.md §2.3 / BASELINE.md §2 (800x1280 / 320x320)
CORR_GFLOP = lambda n, c=128, k=1: 2.0 * n * n * c / 1e9 + 2.0 * n * n * k / 1e9  # noqa: E731
CORR_BYTES = lambda n, c=128, k=1, s=2: 2 * n * c * s + 2 * k * n * 4  # noqa: E731


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sus=p.get("bf16_tflops_sustained", p["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def host_threads():
    """CPU threads this process may really use: min(affinity, cgroup CPU quota).  The GPU boxes expose 128 logical
    CPUs but a 16-CPU cgroup quota; 128 torch threads there are ~20x slower than 16."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            n = min(n, max(1, int(int(q[0]) / int(q[1]))))
    except Exception:
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = min(n, max(1, quota // period))
        except Exception:
            pass
    return n


def run_reference(args):
    """The reference's own algorithm on the host CPU cores (oracle port; see oracle/unicorn_oracle.py header)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import unicorn_oracle as orc
    from unicorn_b200.synthetic import make_video
    from unicorn_b200.weights import make_state_dict
    cores = host_threads()
    torch.set_num_threads(cores)
    H, W = args.size
    steps, warm = args.steps, min(args.warmup, 1)
    sd = make_state_dict(args.config, 0)
    frames, boxes = make_video(steps + warm + 1, H, W, seed=0)
    o = orc.SOTOracle(sd, args.config)
    o.initialize(frames[0:1], boxes[0, 0])
    for i in range(warm):
        o.track(frames[1 + i:2 + i])
    t0 = time.perf_counter()
    for i in range(steps):
        o.track(frames[1 + warm + i:2 + warm + i])
    dt = time.perf_counter() - t0
    fps = steps / dt
    print(json.dumps({
        "impl": "reference", "metric": "frames/sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.config} SOT steady-state frame {H}x{W} (BASELINE configs[1])", "parallelism": "cpu"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{steps} full frames after {warm} warm-up, torch CPU fp32, {cores} threads"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def cpu_baseline_sample(cfg, H, W, budget_s=25.0):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import unicorn_oracle as orc
    from unicorn_b200.synthetic import make_video
    from unicorn_b200.weights import make_state_dict
    cores = host_threads()
    torch.set_num_threads(cores)
    sd = make_state_dict(cfg, 0)
    frames, boxes = make_video(6, H, W, seed=0)
    o = orc.SOTOracle(sd, cfg)
    t0 = time.perf_counter()
    o.initialize(frames[0:1], boxes[0, 0])
    o.track(frames[1:2])  # warm-up frame
    n, t1 = 0, time.perf_counter()
    while n < 4 and (time.perf_counter() - t0) < budget_s:  # ~10 s of CPU work on 16 cores, bounded at budget_s
        o.track(frames[2 + n:3 + n])
        n += 1
    dt = time.perf_counter() - t1
    n = max(n, 1)
    return {"value": n / dt, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"{n} full {H}x{W} SOT frame(s) after 1 warm-up frame, oracle (torch CPU fp32), {cores} threads"}


def extra_workloads(dev, rank, world, K, sync_all, save_tuning=None):
    """BASELINE configs[2] (ConvNeXt-L MOT at 1536x2048, ByteTrack association of 100 synthetic objects per frame) and configs[3]
    (ConvNeXt-L + CondInst mask head VOS at 800x1280, 1 and 3 objects) through the product drivers.  Per workload: `_dt_dev` =
    seconds for K CUDA-graph replays with the frames resident in HBM (CUDA events), `_dt_e2e` = wall clock of K frames through the
    driver's public call with pinned uint8 HOST frames (H2D, association / result D2H inside)."""
    import types
    from unicorn_b200.engine import UnicornEngine
    from unicorn_b200.mot import UnicornMOTTracker
    from unicorn_b200.synthetic import make_detections, make_video
    from unicorn_b200.tracker.byte_tracker import BYTETracker
    from unicorn_b200.vos import UnicornVOSTrack
    from unicorn_b200.weights import make_state_dict
    to_u8 = lambda f: f.round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()  # noqa: E731
    out = {}

    def timed(replay, step, n, warm=3):
        for i in range(warm):
            step(i)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            replay(i)
        e1.record()
        sync_all()
        dt_dev = e0.elapsed_time(e1) / 1e3
        t0 = time.perf_counter()
        for i in range(n):
            step(i)
        torch.cuda.synchronize()
        return dt_dev, time.perf_counter() - t0

    # ---------------- configs[2]: MOT 1536x2048
    H, W = 1536, 2048
    cfg = "unicorn_track_large_mot_challenge"
    eng = UnicornEngine(make_state_dict(cfg, 0), cfg, device=dev)
    frames, _ = make_video(4, H, W, seed=10 + rank, n_obj=6)
    host = [to_u8(frames[i:i + 1]).pin_memory() for i in range(4)]
    devf = [h.to(dev) for h in host]
    bargs = types.SimpleNamespace(track_thresh=0.5, track_buffer=30, match_thresh=0.8, mot20=False)
    bt100 = BYTETracker(bargs, device=dev)
    dets100 = make_detections(n_frames=2 * K + 16, n_obj=100, seed=3, W=float(W), H=float(H))
    MD = 3  # frames in flight on the device: the ByteTrack arm's frames are independent (own stream + engine context each)
    trk = UnicornMOTTracker(eng, (H, W), assoc="byte", tracker=BYTETracker(bargs, device=dev), use_graph=True, depth=MD)
    for i in range(MD - 1):
        trk.submit(host[i % 4])
    cnt = [0]

    def mot_step(i):  # submit(t+MD-1); collect(t): the host association of frame t overlaps the device work of the frames behind it
        trk.submit(host[(i + MD - 1) % 4])
        trk.collect()
        bt100.update(dets100[cnt[0] % len(dets100)][0].numpy(), (H, W), (H, W))  # seeded random weights detect few boxes of their own:
        cnt[0] += 1                                                                # the 100-object association cost is paid here

    main = torch.cuda.current_stream()

    def mot_replay(i):  # device-resident: input copy + graph replay on the context's stream, no result copies
        c = trk._ctxs[i % MD]
        if i < MD:
            c.stream.wait_stream(main)
        with torch.cuda.stream(c.stream):
            c.img_in_u8.copy_(devf[i % 4], non_blocking=True)
            c.graph.replay()
        if i >= K - MD:
            main.wait_stream(c.stream)
    for i in range(2 * MD + 1):
        mot_step(i)  # a context's first frame runs eagerly (autotuning), its second one captures the graph
    dt_dev, dt_e2e = timed(mot_replay, mot_step, K)
    for i in range(MD - 1):
        trk.collect()
    if save_tuning:
        eng.save_tuning(os.path.join(save_tuning, f"{cfg}.json"))
    out["mot_1536x2048"] = dict(_frames=K, _dt_dev=dt_dev, _dt_e2e=dt_e2e, gflop_per_frame=1887.7 * 3.072,
                                workload=f"{cfg} MOT detector (mode whole, 64512 anchors) + ByteTrack association of 100 synthetic objects per frame, "
                                         f"1536x2048 (BASELINE configs[2]); device half = CUDA graph, {MD} frames in flight on their own streams, association of frame t overlapped with them",
                                h2d_bytes_per_step=int(host[0].numel()), d2h_bytes_per_step=int(trk.max_dets * 7 * 4 + 4))
    del trk
    # the reference's own association arm (mot_evaluator.py:1005-1057): interaction with the previous frame, embedding upsample, sampling,
    # QuasiDenseEmbedTracker — the s16 feature of frame t-1 is carried, so the device halves run on one stream (host half overlapped)
    from unicorn_b200.tracker import QuasiDenseEmbedTracker
    trq = UnicornMOTTracker(eng, (H, W), tracker=QuasiDenseEmbedTracker(device=dev), use_graph=True)
    trq.submit(host[0])

    def qd_step(i):
        trq.submit(host[(i + 1) % 4])
        trq.collect()

    def qd_replay(i):
        trq.img_in_u8.copy_(devf[i % 4], non_blocking=True)
        trq._graphs[i & 1][0].replay()
    for i in range(4):
        qd_step(i)  # frames 1-2 eager, 3-4 capture the two parity graphs
    dt_dev, dt_e2e = timed(qd_replay, qd_step, K)
    trq.collect()
    out["mot_1536x2048_qd"] = dict(_frames=K, _dt_dev=dt_dev, _dt_e2e=dt_e2e, gflop_per_frame=(1887.7 + 43.8) * 3.072,  # + interaction and embedding branch of the SOT frame count (1997 - 1887.7 - 65.5 correlation)
                                   workload=f"{cfg} MOT detector + interaction with the previous frame + embedding + QuasiDense association (the reference's arm), "
                                            "1536x2048; device half = CUDA graph on one stream (frame t needs the s16 feature of t-1), association overlapped",
                                   h2d_bytes_per_step=int(host[0].numel()), d2h_bytes_per_step=int(trq.max_dets * (7 + 128) * 4 + 4))
    del trq, eng
    # ---------------- configs[3]: VOS with the CondInst mask head, 800x1280
    H, W = 800, 1280
    cfg = "unicorn_track_large_mask"
    eng = UnicornEngine(make_state_dict(cfg, 0), cfg, device=dev)
    for n_obj in (1, 3):
        frames, boxes = make_video(4, H, W, seed=20 + rank, n_obj=n_obj)
        host = [to_u8(frames[i:i + 1]).pin_memory() for i in range(4)]
        devf = [h.to(dev) for h in host]
        VD = 3  # frames in flight (worker drivers on engine forks; a VOS frame depends only on the reference frames of its objects)
        vos = UnicornVOSTrack(eng, (H, W), use_graph=True, depth=VD)
        vos.initialize_tensor(host[0], {o + 1: boxes[0, o] for o in range(n_obj)})
        for i in range(VD - 1):
            vos.submit(host[1 + i % 3])

        def vos_step(i):  # submit(t + VD - 1); collect(t)
            vos.submit(host[1 + (i + VD - 1) % 3])
            vos.collect()

        def vos_replay(i):  # device-resident: input copy + graph replay on the worker's stream
            w = vos._workers[i % VD]
            if i < VD:
                w._stream.wait_stream(main)
            with torch.cuda.stream(w._stream):
                w.img_in_u8.copy_(devf[1 + i % 3], non_blocking=True)
                w._graph.replay()
            if i >= K - VD:
                main.wait_stream(w._stream)
        for i in range(2 * VD + 1):
            vos_step(i)  # a worker's first frame runs eagerly, its second one captures the graph
        dt_dev, dt_e2e = timed(vos_replay, vos_step, K)
        for i in range(VD - 1):
            vos.collect()
        out[f"vos_800x1280_{n_obj}obj"] = dict(_frames=K, _dt_dev=dt_dev, _dt_e2e=dt_e2e, gflop_per_frame=2062.0 + (n_obj - 1) * 337.0,
                                                workload=f"{cfg} VOS, {n_obj} object(s), 800x1280 (BASELINE configs[3]): backbone, interaction, "
                                                         f"fused correlation, per-object mask head + NMS + dynamic mask, device soft aggregation; one CUDA graph per frame, {VD} frames in flight",
                                                h2d_bytes_per_step=int(host[0].numel()), d2h_bytes_per_step=int(n_obj * 32),
                                                launches_per_frame=vos.launches_per_frame)
        del vos
    if save_tuning:
        eng.save_tuning(os.path.join(save_tuning, f"{cfg}.json"))
    return out


def roofline_inputs():
    """Per-launch DRAM traffic of the kernels quoted below, from the committed ncu captures of the CURRENT kernels
    (profiles/r2_roofline_inputs.json, written by tools/make_roofline_inputs.py from profiles/r2_ncu_*.csv)."""
    path = os.path.join(ROOT, "profiles", "r2_roofline_inputs.json")
    return json.load(open(path)) if os.path.exists(path) else {"kernels": {}}


def pk_burst():
    return peaks()["tf_burst"]


def last_step_outputs(ctx, max_inst):
    """Host copies of what one SOT frame of an engine context produced: the detections collect() hands back (`dets`, rows
    x1 y1 x2 y2 obj_conf cls_conf cls; `count`, the number NMS kept) and the dense maps behind them that the tracker exposes
    as `last` (`head`, the decoded [A, 6] predictions; `priors`, the stride-8 label map propagated by the correlation)."""
    n = int(ctx.ws.count.item())
    out = {"dets": ctx.ws.dets[:min(n, max_inst)], "head": ctx.last["head"][0], "priors": ctx.last["priors"][0]}
    out = {k: v.float().cpu().numpy() for k, v in out.items()}
    out["count"] = np.array([n], dtype=np.float64)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", default="unicorn_track_large")
    ap.add_argument("--size", type=int, nargs=2, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--depth", type=int, default=3, help="frames in flight of the headline measurement (>= 2; the sequential numbers are always reported too)")
    ap.add_argument("--no-extra", action="store_true", help="skip the configs[2] (MOT 1536x2048) and configs[3] (VOS mask) workloads")
    ap.add_argument("--save-tuning", default=None, help="directory: write every engine's per-layer N-tile table (with UC_NO_TUNED=1: fresh autotuning)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the outputs of the headline measurement's last timed frame as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.size is None:
        args.size = (320, 320) if "tiny" in args.config else (800, 1280)
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to --impl ours")
        return run_reference(args)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from unicorn_b200 import ops
    from unicorn_b200.engine import UnicornEngine
    from unicorn_b200.sot import UnicornSOTTrack
    from unicorn_b200.synthetic import make_video
    from unicorn_b200.weights import make_state_dict

    H, W = args.size
    K, Wm = args.steps, max(args.warmup, 3)
    sd = make_state_dict(args.config, 0)
    n_frames = min(K, 16) + 1
    frames, boxes = make_video(n_frames, H, W, seed=rank)  # one independent sequence per rank (SURVEY §8e)
    eng = UnicornEngine(sd, args.config, device=dev)
    trk = UnicornSOTTrack(eng, (H, W), use_graph=True)
    # frames as the decoder delivers them: uint8 HWC BGR (quantised synthetic video; the oracle / reference arm gets
    # the same values as fp32 NCHW)
    to_u8 = lambda f: f.round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()  # noqa: E731
    frames_u8 = to_u8(frames)
    trk.initialize_tensor(frames_u8[0:1], boxes[0, 0])
    host_frames = [frames_u8[1 + i:2 + i].contiguous().pin_memory() for i in range(n_frames - 1)]
    dev_frames = [f.to(dev) for f in host_frames]
    # warm-up (builds the CUDA graph on the first call)
    trk.track_tensor(host_frames[0])
    for i in range(Wm):
        trk.track_tensor(host_frames[i % len(host_frames)])
    launches_per_frame = trk.launches_per_frame  # counted while the frame was captured into the CUDA graph

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---------------- device-resident throughput: frames already in HBM, graph replays only
    sampler = ClockSampler(local_rank)
    sync_all()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        trk.img_in_u8.copy_(dev_frames[i % len(dev_frames)], non_blocking=True)
        trk.graph.replay()
    e1.record()
    sync_all()
    dt_dev = e0.elapsed_time(e1) / 1e3
    # ---------------- the headline: `depth` frames in flight (sot.py submit / collect).  The frames of a sequence are independent — the
    # network never sees the previous frame's result (unicorn_sot.py:57-109) — so each runs on its own stream and engine context and
    # fills the SMs that one frame's small kernels and launch gaps leave idle; results are bit-identical to the sequential tracker
    # (tests/test_engine_gpu.py::test_pipelined_tracker_matches_sequential).  The sequential numbers are reported next to it.
    main = torch.cuda.current_stream()

    def measure_pipe(depth):
        pipe = UnicornSOTTrack(eng, (H, W), use_graph=True, depth=depth)
        pipe.initialize_tensor(frames_u8[0:1], boxes[0, 0])
        for i in range(2 * depth):
            pipe.track_tensor(host_frames[i % len(host_frames)])
        sync_all()
        e0.record()
        for c in pipe._ctxs:
            c.stream.wait_stream(main)
        for i in range(K):
            c = pipe._ctxs[i % depth]
            with torch.cuda.stream(c.stream):
                c.img_in_u8.copy_(dev_frames[i % len(dev_frames)], non_blocking=True)
                c.graph.replay()
        for c in pipe._ctxs:
            main.wait_stream(c.stream)
        e1.record()
        sync_all()
        return pipe, e0.elapsed_time(e1) / 1e3
    D = max(2, args.depth)
    pipe, dt_dev_pipe = measure_pipe(D)
    # timed step i ran on context i % D; the later measurements reuse these buffers, so copy the last step's results now
    dumped = last_step_outputs(pipe._ctxs[(K - 1) % D], pipe.max_inst) if args.dump_outputs and rank == 0 else None
    dt_dev_pipe3 = measure_pipe(D + 1)[1]
    # ---------------- end to end through the public API with pinned host frames, driven by the product's multi-GPU module:
    # one sequence per rank (parallel.shard_sequences), start barrier, wall clock of the slowest rank, one all_gather of the
    # per-rank [frames, seconds, tracks] (parallel.gather_stats) — no data-path collective (SURVEY 8e)
    from unicorn_b200 import parallel

    def sot_worker_seq(seq_index, seq):
        tracked = 0
        for i in range(K):
            dets, n = trk.track_tensor(seq[i % len(seq)])
            tracked += int(n > 0)
        torch.cuda.synchronize()
        return K, tracked

    def sot_worker_pipe(seq_index, seq):
        tracked = 0
        for i in range(K):
            if i >= D:
                tracked += int(pipe.collect()[1] > 0)
            pipe.submit(seq[i % len(seq)])
        for i in range(min(D, K)):
            tracked += int(pipe.collect()[1] > 0)
        torch.cuda.synchronize()
        return K, tracked
    seqs = [host_frames if r == rank else None for r in range(world)]
    sync_all()
    dt_e2e = parallel.run_sharded(seqs, sot_worker_seq, device=dev)["seconds"]
    sync_all()
    sharded = parallel.run_sharded(seqs, sot_worker_pipe, device=dev)
    dt_e2e_pipe = sharded["seconds"]
    clocks = sampler.stop()
    # ---------------- correlation kernel alone (L2 flushed between launches)
    hh, ww = H // 8, W // 8
    n_pos = hh * ww
    e_pre, e_cur = trk.last["embed_pre"].view(-1, 128), trk.last["embed_cur"].view(-1, 128)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    ts = []
    for _ in range(10):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ops.corr_propagate(e_pre, e_cur, trk.lbs_pre, out=eng.buf("corr.out", (1, n_pos), torch.float32))
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / 1e3)
    t_corr = sorted(ts)[len(ts) // 2]
    # ---------------- dominant kernel: conv_gemm on the two stage-3 pointwise GEMM shapes (54 of the 172 conv launches of
    # a frame, 37 % of its device time), timed the way the frame runs them: kernel nodes of a CUDA graph, CUDA events.
    conv_roof = dw_roof = mlp_roof = None
    RI = roofline_inputs()
    if "large" in args.config and (H, W) == (800, 1280):
        xs = torch.randn(1, 50, 80, 768, device=dev).bfloat16()
        w1 = ops.pack_conv_weight(torch.randn(3072, 768, 1, 1, device=dev) / 768 ** 0.5)
        w2 = ops.pack_conv_weight(torch.randn(768, 3072, 1, 1, device=dev) / 3072 ** 0.5)
        b1, b2, gm = torch.randn(3072, device=dev), torch.randn(768, device=dev), torch.randn(768, device=dev)
        hid = torch.empty(1, 50, 80, 3072, device=dev, dtype=torch.bfloat16)
        res = torch.randn(1, 50, 80, 768, device=dev).bfloat16()
        yo = torch.empty_like(res)

        def pair():
            eng.conv(xs, w1, 1, bias=b1, act=ops.ACT_GELU, out=hid)
            eng.conv(hid, w2, 1, bias=b2, gamma=gm, res=res, out=yo)
        pair()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(10):
                pair()
        g.replay()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(3):
            g.replay()
        b.record()
        torch.cuda.synchronize()
        t_pair = a.elapsed_time(b) / 1e3 / 30  # seconds per (pwconv1 + pwconv2)
        fl = 2 * 2.0 * 4000 * 768 * 3072
        conv_roof = {"bound": "tensor", "achieved": fl / t_pair / 1e12, "peak": pk_burst(), "unit": "TFLOP/s",
                     "frac": fl / t_pair / 1e12 / pk_burst(), "us_per_launch": t_pair * 1e6 / 2,
                     "traffic": RI["kernels"].get("r2_ncu_conv_s3pw2", {}).get("dram_bytes"),
                     "traffic_note": "dram__bytes_read + write of the pwconv2 launch (conv_gemm_kernel<192,7,2>), ncu --set full, cold L2: A 24.6 + W 4.7 + residual "
                                     "6.1 MB = the algorithmic bytes; profiles/r2_ncu_conv_gn.csv (pwconv1: r2_ncu_conv_s3pw1, 10.9 MB = A 6.1 + W 4.7)",
                     "kernel": "uc::conv_gemm_kernel, ConvNeXt-L stage-3 pwconv1 (768->3072, GELU) + pwconv2 (3072->768, layer-scale + residual), "
                               "M = 4000 pixels, CUDA-graph nodes",
                     "peak_source": "measured bf16_tflops (burst)"}

        # ---- the two other hand-written hot kernels of a ConvNeXt block on its stage-1 shape: the tensor-core depthwise 7x7 and the fused
        # LayerNorm + MLP (CUDA-graph nodes, 10 launches per replay; the 49 MB working set stays L2 resident like inside the frame)
        def graph_time(fn, reps=10):
            fn()
            torch.cuda.synchronize()
            gg = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gg):
                for _ in range(reps):
                    fn()
            gg.replay()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(3):
                gg.replay()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / 1e3 / (3 * reps)
        M1, C1 = 200 * 320, 192
        x1 = torch.randn(1, 200, 320, C1, device=dev).bfloat16()
        y1 = torch.empty_like(x1)
        qt = ops.pack_dw_weight_mma(torch.randn(C1, 1, 7, 7, device=dev) / 7, torch.randn(C1, device=dev))
        t_dw = graph_time(lambda: ops.dwconv7_mma(x1, qt, out=y1))
        dw_bytes = 4.0 * M1 * C1  # read + write the bf16 map once
        dw_roof = {"bound": "hbm", "achieved": dw_bytes / t_dw / 1e9, "peak": peaks()["hbm"], "unit": "GB/s", "frac": dw_bytes / t_dw / 1e9 / peaks()["hbm"],
                   "us_per_launch": t_dw * 1e6, "traffic": RI["kernels"].get("r2_ncu_dwmma_s1", {}).get("dram_bytes"),
                   "kernel": "uc::dwconv7_mma_kernel<4> (depthwise 7x7 as Toeplitz blocks on mma.sync), ConvNeXt-L stage 1: 200x320x192, static item schedule",
                   "note": "algorithmic bytes (49 MB: the map read and written once) over the launch time; the kernel is bound by shared-memory wavefronts "
                           "(ldmatrix), not by HBM — DESIGN.md 4.3", "peak_source": "measured hbm_gbs"}
        w1f = ops.pack_conv_weight(torch.randn(4 * C1, C1, 1, 1, device=dev) / C1 ** 0.5)
        w2s = ops.pack_conv_weight(torch.randn(C1, 4 * C1, 1, 1, device=dev) / (4 * C1) ** 0.5)
        c1v, b2v, gmv = torch.randn(4 * C1, device=dev), torch.randn(C1, device=dev), torch.randn(C1, device=dev) * 0.1
        t_mlp = graph_time(lambda: ops.convnext_mlp(y1.view(-1, C1), w1f, c1v, w2s, b2v, gmv, x1.view(-1, C1)))
        fl_mlp = 2 * 2.0 * M1 * C1 * 4 * C1
        mlp_roof = {"bound": "tensor", "achieved": fl_mlp / t_mlp / 1e12, "peak": pk_burst(), "unit": "TFLOP/s", "frac": fl_mlp / t_mlp / 1e12 / pk_burst(),
                    "us_per_launch": t_mlp * 1e6, "traffic": RI["kernels"].get("r2_ncu_mlp_s1", {}).get("dram_bytes"),
                    "kernel": "uc::convnext_mlp_kernel<192> (LayerNorm + pwconv1 + GELU + pwconv2 + layer scale + residual), ConvNeXt-L stage 1: M = 64000 pixels",
                    "note": "the GELU of the 64000 x 768 hidden activations (2 MUFU operations per element, 16 per clock and SM) bounds this kernel at "
                            "~26 us, not the tensor pipe; the separate kernels it replaces take 120 us (profiles/r2_mlp_fused_microbench.txt)",
                    "peak_source": "measured bf16_tflops (burst)"}

    extra = {} if args.no_extra else extra_workloads(dev, rank, world, K, sync_all, args.save_tuning if rank == 0 else None)
    if args.save_tuning and rank == 0:
        eng.save_tuning(os.path.join(args.save_tuning, f"{args.config}.json"))
    RI_frame = RI.get("frame", {})
    if world > 1:
        t = torch.tensor([dt_dev, dt_e2e, dt_dev_pipe, dt_e2e_pipe, dt_dev_pipe3] + [v for k in sorted(extra) for v in (extra[k]["_dt_dev"], extra[k]["_dt_e2e"])], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t = t.tolist()
        dt_dev, dt_e2e, dt_dev_pipe, dt_e2e_pipe, dt_dev_pipe3 = t[0], t[1], t[2], t[3], t[4]
        for j, k in enumerate(sorted(extra)):
            extra[k]["_dt_dev"], extra[k]["_dt_e2e"] = t[5 + 2 * j], t[6 + 2 * j]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    fps = world * K / dt_dev_pipe
    fps_e2e = world * K / dt_e2e_pipe
    gflop = FRAME_GFLOP.get(args.config, 0.0) * (H * W) / ((800 * 1280) if "large" in args.config else (320 * 320))
    ach = gflop * K / dt_dev_pipe / 1e3  # TFLOP/s per GPU
    out = {
        "metric": "frames/sec", "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": 1e3 * dt_dev_pipe / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{args.config} SOT steady-state frame {H}x{W}, 1 object (BASELINE configs[1])",
                   "parallelism": f"dp{world} (one sequence per GPU, no data-path collective)",
                   "l2": "per-frame working set (0.52 GB bf16 weights + activations) exceeds the 126 MB L2; a different frame every step",
                   "weights": "seeded random init (unicorn_b200.weights.make_state_dict)", "cuda_graph": True,
                   "frames_in_flight": D, "frames_in_flight_note": "independent frames of one sequence on separate streams / engine contexts; "
                                                                "ms_per_step = timed region / steps; per-frame latency is the `sequential` entry's",
                   "input": "uint8 HWC BGR frames (3.07 MB H2D per frame); float conversion fused into the stem kernel"},
        "roofline": {"bound": "tensor", "achieved": ach, "peak": pk["tf_sus"], "unit": "TFLOP/s", "frac": ach / pk["tf_sus"],
                     "traffic": RI_frame.get("dram_bytes"), "traffic_note": RI_frame.get("note"),
                     "kernel": "whole-frame CUDA graph (1997 GFLOP algorithmic per 800x1280 frame, SURVEY §8d)",
                     "peak_source": pk["src"] + " bf16_tflops_sustained"},
        "roofline_conv": conv_roof,
        "roofline_dwconv": dw_roof, "roofline_mlp": mlp_roof,
        "roofline_corr": {"bound": "tensor", "traffic": RI["kernels"].get("r2_ncu_corr", {}).get("dram_bytes"),
                          "hbm_note": "the fused kernel moves only its algorithmic 8.26 MB (the 16000^2 similarity matrix never leaves the SM), so it is bound "
                                      "by the tensor / MUFU / issue pipes, not by HBM: hbm_frac is reported because BASELINE.json's metric asks for it, it is not a "
                                      "utilisation target", "achieved": CORR_GFLOP(n_pos) / t_corr / 1e3, "peak": pk["tf_burst"], "unit": "TFLOP/s",
                          "frac": CORR_GFLOP(n_pos) / t_corr / 1e3 / pk["tf_burst"], "us_per_launch": t_corr * 1e6,
                          "hbm_gbs_algorithmic": CORR_BYTES(n_pos) / t_corr / 1e9, "hbm_frac": CORR_BYTES(n_pos) / t_corr / 1e9 / pk["hbm"],
                          "kernel": "uc::corr_kernel<1> (fused K^TQ + softmax + PV), L2 flushed between launches",
                          "peak_source": pk["src"] + " bf16_tflops (burst)"},
        "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": int(host_frames[0].numel() * host_frames[0].element_size()),
                "d2h_bytes_per_step": int(trk.host_dets.numel() * 4 + 4)},
        "sequential": {"value": world * K / dt_dev, "e2e": world * K / dt_e2e, "unit": "frames/s", "ms_per_step": 1e3 * dt_dev / K,
                       "roofline_frac": gflop * K / dt_dev / 1e3 / pk["tf_sus"],
                       "note": "one frame in flight (UnicornSOTTrack.track_tensor: frame in, its result out) = the per-frame latency"},
        f"pipelined_{D + 1}_frames": {"value": world * K / dt_dev_pipe3, "unit": "frames/s", "note": "device-resident, one more frame in flight"},
        "multi_gpu": {"module": "unicorn_b200.parallel.run_sharded + gather_stats", "shard": sharded["shard"], "per_rank_frames_seconds_tracks": sharded["per_rank"]},
        "gpu_launches": launches_per_frame * K * 2,  # K device-resident steps + K end-to-end steps
        "launches_per_frame": launches_per_frame,
        "clocks": clocks,
    }
    pk_sus = pk["tf_sus"]
    for k in sorted(extra):  # BASELINE configs[2] / configs[3], measured in the same run (whole-job numbers over `world` GPUs)
        e = extra[k]
        n_fr, dtd, dte = e.pop("_frames"), e.pop("_dt_dev"), e.pop("_dt_e2e")
        e.update(value=world * n_fr / dtd, e2e=world * n_fr / dte, unit="frames/s", ms_per_step=1e3 * dtd / n_fr, steps=n_fr,
                 roofline_frac=e["gflop_per_frame"] * n_fr / dtd / 1e3 / pk_sus)
        out[k] = e
    if not args.no_cpu_baseline and world == 1:
        out["cpu_baseline"] = cpu_baseline_sample(args.config, H, W)
    else:
        out["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": os.cpu_count(), "kind": "port", "sample": "skipped (N>1 or --no-cpu-baseline)"}
        out["cpu_baseline"]["cores"] = host_threads()
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
