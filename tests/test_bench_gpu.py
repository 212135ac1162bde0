"""bench.py --dump-outputs: the files hold the result of the headline measurement's last timed frame, and --steps sets how many
frames were timed (with K steps over min(K, 16) distinct frames, the last one is frame K; one step more or less would dump another)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_last_timed_frame(tmp_path):
    from unicorn_b200.engine import UnicornEngine
    from unicorn_b200.sot import UnicornSOTTrack
    from unicorn_b200.synthetic import make_video
    from unicorn_b200.weights import make_state_dict
    name, K, H, W = "unicorn_track_tiny", 5, 320, 320
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", name, "--steps", str(K), "--warmup", "1",
                        "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=1200, cwd=tmp_path)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == K
    got = {n: np.load(out / f"{n}.npy") for n in ("dets", "count", "head", "priors")}
    assert sorted(os.listdir(out)) == sorted(f"{n}.npy" for n in got)
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20

    # the same seeded sequence through the synchronous tracker: bench.py's frame K
    frames, boxes = make_video(K + 1, H, W, seed=0)
    u8 = frames.round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()
    trk = UnicornSOTTrack(UnicornEngine(make_state_dict(name, 0), name), (H, W), use_graph=True)
    trk.initialize_tensor(u8[0:1], boxes[0, 0])
    dets, n = trk.track_tensor(u8[K:K + 1].pin_memory())
    head, priors = trk.last["head"][0].cpu().numpy(), trk.last["priors"][0].cpu().numpy()
    assert got["count"].tolist() == [n]
    assert got["head"].shape == head.shape and got["priors"].shape == priors.shape
    np.testing.assert_allclose(got["priors"], priors, atol=1e-4)
    np.testing.assert_allclose(got["head"], head, rtol=1e-4, atol=1e-3)
    np.testing.assert_allclose(got["dets"], dets.numpy(), rtol=1e-4, atol=1e-3)
