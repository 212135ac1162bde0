"""MOTS mask encoding on the device (ops.mots_masks_rle / uc_mots_masks_rle) against the host path it replaces (F.interpolate +
threshold + results.overlap_free + results.rle_encode), and the MOTS driver's pipelined submit / collect against its sequential
step_tensor and the previous host formula."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
dev = "cuda"


def _device(masks, rows, emit, img_h, img_w, thres=0.5, sf=1.0, ws=None):
    from unicorn_b200 import ops
    sel = torch.tensor([rows, emit], dtype=torch.int32, device=dev)
    out = ops.mots_masks_rle(masks.to(dev, torch.float32).contiguous(), sel[0], sel[1], img_h, img_w, thres, sf, ws)
    torch.cuda.synchronize()
    return out


def _host(bits, rows, emit):
    """bits: bool [n, H, W] (any device) -> rle_encode(overlap_free(bits[rows]))[emitted]."""
    from unicorn_b200 import results as R
    free = R.overlap_free(bits[torch.as_tensor(rows, device=bits.device)]).cpu().numpy()
    return [R.rle_encode(free[i]) for i in range(len(rows)) if emit[i]]


def _exact(bits, rows=None, emit=None, ws=None):
    n, H, W = bits.shape
    rows = list(range(n)) if rows is None else rows
    emit = [1] * len(rows) if emit is None else emit
    got = _device(bits.float(), rows, emit, H, W, ws=ws)
    ref = _host(bits, rows, emit)
    assert got == ref
    return got


def _ellipses(K, H, W, seed, device=dev):
    g = torch.Generator(device="cpu").manual_seed(seed)
    c = torch.rand(K, 2, generator=g) * torch.tensor([H, W])
    r = (0.05 + 0.3 * torch.rand(K, 2, generator=g)) * torch.tensor([H, W])
    yy = torch.arange(H, device=device, dtype=torch.float32)[None, :, None]
    xx = torch.arange(W, device=device, dtype=torch.float32)[None, None, :]
    c, r = c.to(device), r.to(device)
    return ((yy - c[:, 0, None, None]) / r[:, 0, None, None]) ** 2 + ((xx - c[:, 1, None, None]) / r[:, 1, None, None]) ** 2 < 1


# ------------------------------------------------------------------------------------------------ 1. bit logic (sf = 1, 0/1 masks)
@pytest.mark.parametrize("H,W", [(20, 30), (37, 53), (64, 1), (1, 77), (1, 1), (33, 2)])
def test_rle_exact_edge_masks(H, W):
    z = torch.zeros(1, H, W, dtype=torch.bool)
    first = z.clone()
    first[0, 0, 0] = True
    last = z.clone()
    last[0, -1, -1] = True
    for m in (z, ~z, first, last):
        _exact(m)
    g = torch.Generator().manual_seed(H * 1000 + W)
    _exact(torch.rand(3, H, W, generator=g) > 0.5)


@pytest.mark.parametrize("K", [1, 64])
def test_rle_exact_ellipses_fullhd(K):
    bits = _ellipses(K, 1080, 1920, seed=K)
    got = _exact(bits)
    assert len(got) == K


def test_rle_exact_row_order_and_non_emitted_rows_claim():
    bits = _ellipses(6, 123, 97, seed=3)
    bits[:, 40:80, 30:70] = True  # every mask overlaps every other one
    _exact(bits, rows=[3, 0, 5, 2])
    _exact(bits, rows=[4, 1, 2, 0, 5, 3], emit=[0, 1, 0, 1, 1, 0])
    # a non-emitted first row still takes its pixels from the others: the second string is empty inside the first mask
    got = _device(bits.float(), [0, 1], [0, 1], 123, 97)
    assert len(got) == 1 and got == _host(bits, [0, 1], [0, 1])


def test_rle_capacity_growth():
    from unicorn_b200 import ops
    ws = ops.MotsRleWorkspace(dev, capacity=16)
    board = (torch.arange(61)[:, None] + torch.arange(45)[None, :]) % 2 == 0
    bits = torch.stack([board, ~board, board])
    got = _exact(bits, ws=ws)
    assert ws.chars.numel() >= sum(len(s) for s in got) > 16
    again = _exact(bits, ws=ws)  # the grown buffer is kept
    assert again == got


# ------------------------------------------------------------------------------------------------ 2. resize + threshold
@pytest.mark.parametrize("Hin,Win,img_h,img_w", [(800, 1280, 1080, 1920), (320, 320, 480, 640), (320, 320, 160, 240), (800, 1280, 402, 640)])
def test_rle_resize_threshold_vs_interpolate(Hin, Win, img_h, img_w):
    from unicorn_b200 import results as R
    K, thres = 6, 0.3
    g = torch.Generator().manual_seed(Hin + img_h)
    coarse = torch.rand(K, 1, Hin // 32, Win // 32, generator=g)
    m = F.interpolate(coarse, size=(Hin, Win), mode="bilinear", align_corners=False)[:, 0]
    m = (m + 0.02 * torch.rand(K, Hin, Win, generator=g)).to(dev).contiguous()  # fp32 soft masks, not piecewise linear
    scale = min(Hin / float(img_h), Win / float(img_w))
    sf = 1 / scale
    v = F.interpolate(m[:, None], scale_factor=sf, mode="bilinear", align_corners=False)[:, 0, :img_h, :img_w]
    ref_bits = v > thres
    he, we = ref_bits.shape[1:]
    rows, emit = [2, 0, 5, 1, 4, 3], [1, 1, 0, 1, 1, 1]
    got = _device(m, rows, emit, img_h, img_w, thres=thres, sf=sf)
    ref = R.overlap_free(ref_bits[rows]).cpu().numpy()
    near = torch.cumsum(((v - thres).abs() < 1e-6)[rows].int(), 0).cpu().numpy() > 0  # a flip there may move to later rows
    dec = [R.rle_decode(s, he, we) for s in got]
    ref = [ref[i] for i in range(K) if emit[i]]
    near = [near[i] for i in range(K) if emit[i]]
    assert len(dec) == len(ref)
    flips = sum(int((d != r).sum()) for d, r in zip(dec, ref))
    outside = sum(int(((d != r) & ~n).sum()) for d, r, n in zip(dec, ref, near))
    print(f"{Hin}x{Win} -> {img_h}x{img_w} (encoded {he}x{we}): {flips} pixel(s) differ, {outside} of them farther than 1e-6 "
          "from the threshold")
    assert outside == 0


# ------------------------------------------------------------------------------------------------ 3. driver equivalence
def test_mots_driver_pipelined_graphs_and_sequential_match_host_formula():
    from unicorn_b200 import results as R
    from unicorn_b200.engine import UnicornEngine
    from unicorn_b200.mots import UnicornMOTSTracker
    from unicorn_b200.synthetic import make_video
    from unicorn_b200.tracker import QuasiDenseEmbedTracker
    from unicorn_b200.weights import make_state_dict
    name = "unicorn_track_tiny_mask"
    eng = UnicornEngine(make_state_dict(name, 0), name)
    frames, _ = make_video(6, 320, 320, seed=1, n_obj=3)
    frames = frames.round().clamp(0, 255)  # the uint8 arm below sees the same pixels
    u8 = frames.to(torch.uint8).permute(0, 2, 3, 1).contiguous()
    img_h, img_w = 480, 640
    kw = dict(conf=0.01, nms=0.7, score_thr=0.02, max_dets=16, min_box_area=0)

    def qd():
        return QuasiDenseEmbedTracker(init_score_thr=0.05, obj_score_thr=0.03)

    seq = UnicornMOTSTracker(eng, (320, 320), tracker=qd(), **kw)
    old_trk = qd()
    scale = min(320 / img_h, 320 / img_w)
    a, c = [], []
    for t in range(6):
        a.append(seq.step_tensor(frames[t:t + 1], img_h, img_w))
        # the previous driver's host half on the same device outputs
        last = seq.last
        d, f, masks = last["dets"], last["feats"], last["masks"]
        n = d.shape[0]
        if n == 0:
            c.append((t + 1, [], 2, img_h, img_w, []))
            continue
        m = F.interpolate(masks[:, None], scale_factor=1 / scale, mode="bilinear", align_corners=False)[:, 0, :img_h, :img_w] > seq.mask_thres
        scores = d[:, 4] * d[:, 5]
        keep = scores > seq.score_thr
        boxes = torch.cat([d[keep, :4] / scale, scores[keep, None]], 1)
        m, f = m[keep.to(m.device)], f[keep]
        ob, _, oid, idx = old_trk.match(boxes, torch.ones(boxes.size(0)), f, t + 1, return_index=True)
        m = m[idx.to(m.device)]
        valid = oid > -1
        c.append(R.mots_frame_result(t + 1, ob[valid], oid[valid], m[valid.to(m.device)].cpu(), img_h, img_w, seq.min_box_area))

    pipe = UnicornMOTSTracker(eng, (320, 320), tracker=qd(), use_graph=True, **kw)
    b = []
    pipe.submit(u8[0:1], img_h, img_w)
    for t in range(1, 6):
        pipe.submit(u8[t:t + 1].pin_memory(), img_h, img_w)
        b.append(pipe.collect())
    b.append(pipe.collect())
    assert len(pipe._graphs) == 2  # frames 3-6 replayed the two parity graphs

    for t in range(6):
        assert a[t] == c[t], (t, a[t][:2], c[t][:2])
        assert b[t] == a[t], (t, b[t][:2], a[t][:2])
    assert any(r[1] for r in a), "no tracked instance in 6 frames"
    print("tracked ids per frame:", [r[1] for r in a])
