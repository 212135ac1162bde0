"""Frames/s of the other BASELINE.json workloads on ONE B200 (bench.py is the contract line for configs[1]):
  mot : configs[2] — ConvNeXt-L MOT detector + embedding path at 1536x2048 (mode="whole", NMS, embedding sampling), then
        (a) the QDTrack association of the reference's MOT evaluator on the model's own detections and
        (b) ByteTrack association on 100 synthetic objects per frame (random weights give few detections of their own).
  vos : configs[3] — ConvNeXt-L + CondInst mask head at 800x1280, n objects propagated from the first frame.
  mots: configs[3] MOTS — the same model at 800x1280 on 1080x1920 frames: (a) sequential step_tensor, (b) CUDA graphs with the
        association and mask encoding of frame t overlapped with frame t+1, (c) the mask tail alone (ops.mots_masks_rle) on
        K = 8 / 32 / 64 synthetic masks against the host path it replaced; prints the card and its power limit first.
Wall clock around synchronised steps (eager launches unless stated), synthetic video, seeded weights.
usage: bench_workloads.py mot|vos|mots [frames]"""
import json, os, sys, time, types
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from unicorn_b200 import _lib
from unicorn_b200.engine import UnicornEngine
from unicorn_b200.synthetic import make_video, make_detections
from unicorn_b200.weights import make_state_dict

what = sys.argv[1] if len(sys.argv) > 1 else "mot"
n = int(sys.argv[2]) if len(sys.argv) > 2 else 12
dev = "cuda"


def timed(fn, n, warm=3):
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize()
    l0, t0 = _lib.LAUNCHES, time.perf_counter()
    for i in range(n):
        fn(warm + i)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return n / dt, 1e3 * dt / n, (_lib.LAUNCHES - l0) // n


if what == "mot":
    from unicorn_b200.mot import UnicornMOTTracker
    from unicorn_b200.tracker.byte_tracker import BYTETracker
    H, W = 1536, 2048
    cfg = "unicorn_track_large_mot_challenge"
    eng = UnicornEngine(make_state_dict(cfg, 0), cfg)
    frames, _ = make_video(4, H, W, seed=0, n_obj=6)
    frames = [f[None].to(dev) for f in frames]
    args = types.SimpleNamespace(track_thresh=0.5, track_buffer=30, match_thresh=0.8, mot20=False)
    dets100 = make_detections(n_frames=n + 8, n_obj=100, seed=3, W=float(W), H=float(H))

    def pipelined(trk, extra=None):
        """submit(t+1); collect(t): host association of frame t overlaps the device work of frame t+1"""
        trk.submit(frames[0])
        def step(i):
            trk.submit(frames[(i + 1) % 4])
            trk.collect()
            if extra:
                extra(i)
        r = timed(step, n, warm=5)
        trk.collect()
        return r

    trk = UnicornMOTTracker(eng, (H, W))
    fps, ms, launches = timed(lambda i: trk.step_tensor(frames[i % 4]), n)
    print(json.dumps({"workload": "configs[2] MOT 1536x2048 ConvNeXt-L: detector + embedding + QDTrack association, sequential eager",
                      "frames_per_s": round(fps, 2), "ms_per_frame": round(ms, 2), "kernels_per_frame": launches, "n_gpus": 1}))
    trk = UnicornMOTTracker(eng, (H, W), use_graph=True)
    fps, ms, launches = pipelined(trk)
    print(json.dumps({"workload": "configs[2] same, device half as CUDA graphs, association of frame t overlapped with frame t+1",
                      "frames_per_s": round(fps, 2), "ms_per_frame": round(ms, 2), "kernels_per_frame": launches, "n_gpus": 1}))
    # ByteTrack arm: detector (no embedding branch) + BYTETracker.update.  Seeded random weights give only a handful of
    # detections, so a second tracker is fed 100 synthetic objects per frame inside the same loop: the measured rate
    # includes the host cost of a 100-object association while the device runs the next frame.
    bt100 = BYTETracker(args, device=dev)
    trk = UnicornMOTTracker(eng, (H, W), assoc="byte", tracker=BYTETracker(args, device=dev), use_graph=True)
    fps, ms, launches = pipelined(trk, extra=lambda i: bt100.update(dets100[i][0].numpy(), (H, W), (H, W)))
    print(json.dumps({"workload": "configs[2] MOT 1536x2048 ConvNeXt-L detector (CUDA graphs) + ByteTrack association of 100 synthetic "
                                  "objects per frame, pipelined", "frames_per_s": round(fps, 2), "ms_per_frame": round(ms, 2),
                      "kernels_per_frame": launches, "n_gpus": 1}))
    bt = BYTETracker(args, device=dev)
    fps2, ms2, l2 = timed(lambda i: bt.update(dets100[i][0].numpy(), (H, W), (H, W)), n)
    print(json.dumps({"workload": "configs[2] ByteTrack update alone, 100 synthetic objects per frame (host Kalman + LAP, IoU on the GPU)",
                      "frames_per_s": round(fps2, 1), "ms_per_frame": round(ms2, 3), "kernels_per_frame": l2}))
elif what == "mots":
    import ctypes
    import subprocess
    import torch.nn.functional as F
    from unicorn_b200 import ops, results as R
    from unicorn_b200.mots import UnicornMOTSTracker
    H, W, img_h, img_w = 800, 1280, 1080, 1920
    cfg = "unicorn_track_large_mask"
    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=uuid,name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout
    card = [l for l in smi.splitlines() if str(props.uuid) in l] or smi.splitlines()[:1]
    print(json.dumps({"device": props.name, "nvidia_smi": card[0].split(", ", 1)[-1] if card else "unavailable",
                      "fields": "name, power.limit, clocks.max.sm"}))
    eng = UnicornEngine(make_state_dict(cfg, 0), cfg)
    frames, _ = make_video(4, H, W, seed=1, n_obj=3)
    frames = [f[None].to(dev) for f in frames]
    trk = UnicornMOTSTracker(eng, (H, W))
    fps, ms, launches = timed(lambda i: trk.step_tensor(frames[i % 4], img_h, img_w), n)
    print(json.dumps({"workload": f"configs[3] MOTS {H}x{W} from {img_h}x{img_w} frames, ConvNeXt-L + CondInst mask head: detector + masks + "
                                  "embedding + QDTrack association + device RLE, sequential eager step_tensor",
                      "frames_per_s": round(fps, 2), "ms_per_frame": round(ms, 2), "kernels_per_frame": launches, "n_gpus": 1}))
    trk = UnicornMOTSTracker(eng, (H, W), use_graph=True)
    trk.submit(frames[0], img_h, img_w)

    def step(i):
        trk.submit(frames[(i + 1) % 4], img_h, img_w)
        trk.collect()
    fps, ms, launches = timed(step, n, warm=5)
    trk.collect()
    print(json.dumps({"workload": "configs[3] MOTS same, device half as CUDA graphs, association + encoding of frame t overlapped with frame t+1",
                      "frames_per_s": round(fps, 2), "ms_per_frame": round(ms, 2), "kernels_per_frame": launches, "n_gpus": 1}))
    # The seeded random weights give only a few tracked instances, so the mask tail is also timed alone on K synthetic soft
    # ellipses at the network resolution, encoded to the 1080x1920 frame, against the host path it replaces.
    sf = 1 / min(H / float(img_h), W / float(img_w))
    thres = 0.3
    for K in (8, 32, 64):
        g = torch.Generator().manual_seed(K)
        c = (torch.rand(K, 2, generator=g) * torch.tensor([H, W])).to(dev)
        r = ((0.05 + 0.2 * torch.rand(K, 2, generator=g)) * torch.tensor([H, W])).to(dev)
        yy = torch.arange(H, device=dev, dtype=torch.float32)[None, :, None]
        xx = torch.arange(W, device=dev, dtype=torch.float32)[None, None, :]
        d2 = ((yy - c[:, 0, None, None]) / r[:, 0, None, None]) ** 2 + ((xx - c[:, 1, None, None]) / r[:, 1, None, None]) ** 2
        masks = torch.sigmoid(8.0 * (1.0 - d2)).contiguous()
        del d2
        sel = torch.stack([torch.arange(K, dtype=torch.int32), torch.ones(K, dtype=torch.int32)]).to(dev)
        ws = ops.MotsRleWorkspace(dev)
        got = ops.mots_masks_rle(masks, sel[0], sel[1], img_h, img_w, thres, sf, ws)  # sizes the workspace
        reps = 20
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            ops.mots_masks_rle(masks, sel[0], sel[1], img_h, img_w, thres, sf, ws)
        op_ms = 1e3 * (time.perf_counter() - t0) / reps
        # the three kernels alone (uc_mots_masks_rle, no host copies), CUDA events over repeated launches
        lib, S = _lib.lib(), _lib.stream_ptr()
        meta = ws.meta[:2 * K + 1]
        call = lambda: _lib.check(lib.uc_mots_masks_rle(
            ctypes.c_void_p(masks.data_ptr()), K, H, W, ctypes.c_void_p(sel[0].data_ptr()), ctypes.c_void_p(sel[1].data_ptr()), K, img_h, img_w,
            ctypes.c_float(thres), ctypes.c_double(sf), ctypes.c_void_p(ws.bits.data_ptr()), ctypes.c_long(ws.bits.numel()),
            ctypes.c_void_p(meta.data_ptr()), ctypes.c_void_p(meta[K:].data_ptr()), ctypes.c_void_p(meta[2 * K:].data_ptr()),
            ctypes.c_void_p(ws.chars.data_ptr()), ctypes.c_long(ws.chars.numel()), S), "uc_mots_masks_rle", 3)
        for _ in range(3):
            call()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            call()
        e1.record()
        torch.cuda.synchronize()
        kern_ms = e0.elapsed_time(e1) / reps
        # host path of the previous driver on the same masks: resize + threshold on the device, bool masks to the host, overlap
        # free + RLE in Python (results.mots_frame_result); 2 repetitions after one warm-up
        ids = torch.arange(K)
        boxes = torch.tensor([[0.0, 0.0, 100.0, 100.0, 1.0]]).repeat(K, 1)

        def host():
            m = F.interpolate(masks[:, None], scale_factor=sf, mode="bilinear", align_corners=False)[:, 0, :img_h, :img_w] > thres
            return R.mots_frame_result(1, boxes, ids, m.cpu(), img_h, img_w, 100)[5]
        ref = host()
        t0 = time.perf_counter()
        for _ in range(2):
            host()
        host_ms = 1e3 * (time.perf_counter() - t0) / 2
        bound_ms = 1e3 * K * H * W * 4 / 7.7e12
        print(json.dumps({"workload": f"MOTS mask tail, {K} soft ellipse masks {H}x{W} -> RLE of the {img_h}x{img_w} frame",
                          "identical_to_host": got == ref, "rle_bytes": sum(len(s) for s in got),
                          "device_op_ms": round(op_ms, 3), "device_kernels_ms": round(kern_ms, 3),
                          "hbm_bound_ms": round(bound_ms, 4), "fraction_of_hbm_bound": round(bound_ms / kern_ms, 3),
                          "masks_fit_l2": K * H * W * 4 < 126e6, "host_path_ms": round(host_ms, 1),
                          "host_threads": torch.get_num_threads(), "speedup_op_vs_host": round(host_ms / op_ms, 1)}))
        del masks
else:
    from unicorn_b200.vos import UnicornVOSTrack
    H, W = 800, 1280
    cfg = "unicorn_track_large_mask"
    eng = UnicornEngine(make_state_dict(cfg, 0), cfg)
    for n_obj in (1, 3):
        frames, boxes = make_video(4, H, W, seed=1, n_obj=n_obj)
        frames = [f[None].to(dev) for f in frames]
        trk = UnicornVOSTrack(eng, (H, W))
        trk.initialize_tensor(frames[0], {o + 1: boxes[0, o].tolist() for o in range(n_obj)})
        fps, ms, launches = timed(lambda i: trk.track_tensor(frames[1 + i % 3]), n)
        print(json.dumps({"workload": f"configs[3] VOS 800x1280 ConvNeXt-L + CondInst mask head, {n_obj} object(s) (eager)",
                          "frames_per_s": round(fps, 2), "ms_per_frame": round(ms, 2), "kernels_per_frame": launches, "n_gpus": 1}))
