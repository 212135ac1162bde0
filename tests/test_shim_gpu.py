"""The `unicorn` shim on the GPU: a tracker written against the REFERENCE'S API only (`from unicorn.exp import get_exp`,
`model(..., mode=...)`, `model.head(...)`, `unicorn.utils.boxes.postprocess`; the call sequence of
external/lib/test/tracker/unicorn_sot.py:26-109, torch fp16 mm + softmax(dim=0) correlation included) must produce the boxes of the
product driver UnicornSOTTrack.  Mask model: shim postprocess_inst against the kernels' direct result."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def shim():
    import unicorn_b200.shim as s
    s.install()
    return s


def _rgb_frames(n, H, W, seed):
    from unicorn_b200.synthetic import make_video
    frames, boxes = make_video(n, H, W, seed=seed)
    rgb = frames.permute(0, 2, 3, 1).round().clamp(0, 255).to(torch.uint8).numpy()
    xywh = boxes[:, 0].clone()
    xywh[:, 2:] -= xywh[:, :2]
    return rgb, xywh


class ApiOnlySOT:
    """initialize/track written with nothing but the reference's public API (what unicorn_sot.py does, in this test's words)."""

    def __init__(self, exp_name, ckpt, input_size):
        from unicorn.exp import get_exp
        exp = get_exp(f"exps/default/{exp_name}", None)
        self.model = exp.get_model(load_pretrain=False)
        self.model.load_state_dict(torch.load(ckpt, map_location="cpu")["model"])
        self.model.cuda()
        self.model.eval()
        self.size = input_size

    def _prep(self, img):
        import cv2
        h, w = img.shape[:2]
        r = min(self.size[0] / h, self.size[1] / w)
        rs = cv2.resize(cv2.cvtColor(img, cv2.COLOR_RGB2BGR), (int(w * r), int(h * r)), interpolation=cv2.INTER_LINEAR)
        t = torch.full((1, 3, self.size[0], self.size[1]), 114.0, device="cuda")
        t[:, :, :rs.shape[0], :rs.shape[1]] = torch.tensor(rs, device="cuda", dtype=torch.float).permute(2, 0, 1)[None]
        return t, r

    def initialize(self, image, box_xywh):
        x, r = self._prep(image)
        _, self.pre = self.model(imgs=x, mode="backbone")
        b = torch.tensor(box_xywh).float()
        b[2:] += b[:2]
        x1, y1, x2, y2 = torch.round(b * r).int().tolist()
        lab = torch.zeros(1, 1, *self.size, device="cuda")
        lab[0, 0, max(0, y1):max(0, y2), max(0, x1):max(0, x2)] = 1.0
        self.lbs = F.interpolate(lab, scale_factor=1 / 8, mode="bilinear", align_corners=False)[0].flatten(-2)
        self.state = list(box_xywh)

    def track(self, image):
        from unicorn.utils.boxes import postprocess
        x, r = self._prep(image)
        fpn, cur = self.model(imgs=x, mode="backbone")
        f0, f1 = self.model(seq_dict0=self.pre, seq_dict1=cur, mode="interaction")
        e0 = self.model(feat=f0, mode="upsample").flatten(-2).squeeze().half()
        e1 = self.model(feat=f1, mode="upsample").flatten(-2).squeeze().half()
        trans = torch.softmax(torch.mm(e0.transpose(1, 0), e1), dim=0)
        coarse = (self.lbs.half() @ trans).view(1, -1, self.pre["h"] * 2, self.pre["w"] * 2).float()
        pri = (coarse, F.interpolate(coarse, scale_factor=1 / 2, mode="bilinear", align_corners=False),
               F.interpolate(coarse, scale_factor=1 / 4, mode="bilinear", align_corners=False))
        out = postprocess(self.model.head(fpn, pri, mode="sot"), 1, 0.001, 0.65)[0]
        if out is not None:
            b = out[0, :4].clone()
            b[0::2] = b[0::2].clamp(0, self.size[1])
            b[1::2] = b[1::2].clamp(0, self.size[0])
            b = (b / r).cpu().numpy()
            self.state = [int(b[0]), int(b[1]), int(b[2] - b[0]), int(b[3] - b[1])]
        return {"target_bbox": self.state}


def test_api_only_tracker_matches_product_driver(shim, tmp_path):
    from unicorn_b200.engine import UnicornEngine
    from unicorn_b200.sot import UnicornSOTTrack
    from unicorn_b200.weights import make_state_dict
    name, size = "unicorn_track_tiny", (320, 320)
    sd = make_state_dict(name, 0)
    ckpt = str(tmp_path / "ckpt.pth")
    torch.save({"model": sd}, ckpt)
    rgb, xywh = _rgb_frames(6, 256, 400, seed=9)
    a = ApiOnlySOT(name, ckpt, size)
    a.initialize(rgb[0], xywh[0].tolist())
    b = UnicornSOTTrack(UnicornEngine(sd, name), size, use_graph=True)
    b.initialize(rgb[0], {"init_bbox": xywh[0].tolist()})
    diffs = []
    for t in range(1, 6):
        sa, sb = a.track(rgb[t])["target_bbox"], b.track(rgb[t])["target_bbox"]
        diffs.append(np.abs(np.array(sa, dtype=np.float32) - np.array(sb, dtype=np.float32)).max())
    print("API-only tracker vs UnicornSOTTrack, max |box difference| per frame (pixels):", diffs)
    # same engine kernels; the only difference is the unfused fp16 correlation of the reference flow vs the fused kernel
    assert np.median(diffs) <= 1.0, diffs


def test_shim_postprocess_inst_matches_kernels(shim):
    from unicorn.exp import get_exp
    from unicorn.utils.boxes import postprocess_inst
    from unicorn_b200 import ops
    from unicorn_b200.synthetic import make_video
    from unicorn_b200.weights import make_state_dict
    name = "unicorn_track_tiny_mask"
    model = get_exp(f"exps/default/{name}.py", None).get_model(load_pretrain=False)
    model.load_state_dict(make_state_dict(name, 0), strict=False)
    model.cuda().eval()
    frames, _ = make_video(1, 320, 320, seed=1, n_obj=3)
    (outs, locs, dyn, lvls, mf, um), seq = model(imgs=frames[0:1].cuda(), mode="whole")
    assert outs.shape == (1, 2100, 13) and locs.shape == (2100, 2) and dyn.shape == (1, 2100, 169) and lvls.shape == (1, 2100)
    assert mf.shape == (1, 8, 40, 40) and um.shape == (1, 144, 40, 40) and set(seq) == {"feat", "pos", "h", "w"}
    keep = outs.clone()
    dets, masks = postprocess_inst(outs, locs, dyn, lvls, mf, model.head.mask_head, 8, 0.02, 0.7, d_rate=2, up_masks=um[0:1])
    assert torch.allclose(outs[0, :, 2] - outs[0, :, 0], keep[0, :, 2], atol=1e-3)  # converted to corners in place, like the reference
    d, m = dets[0], masks[0]
    assert d.shape[1] == 7 and m.shape == (d.shape[0], 1, 320, 320) and float(m.min()) >= 0 and float(m.max()) <= 1
    e = model.engine
    ws = ops.PostWorkspace(2100, "cuda")
    d2, cnt = ops.postprocess_device(keep[0].contiguous(), 8, 0.02, 0.7, ws)
    assert int(cnt.item()) == d.shape[0] and torch.equal(d2[:d.shape[0]], d)
