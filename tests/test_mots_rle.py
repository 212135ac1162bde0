"""MOTS mask encoding without a GPU: uc_mots_masks_rle validates its arguments before any launch, and the host row selection of
the MOTS driver (mots.mots_rows) picks, orders and filters the masks exactly as results.mots_frame_result does."""
import ctypes

import numpy as np
import pytest
import torch

P = ctypes.c_void_p
A, B, C, D, E = (P(0x10000 * i) for i in range(1, 6))  # never dereferenced: validation comes first


def _call(lib, masks=A, n_max=8, Hin=32, Win=48, rows=B, emit=C, K=4, img_h=48, img_w=72, thres=0.3, sf=1.5, ws=D, ws_bytes=1 << 20,
          out_len=E, out_off=E, out_total=E, chars=A, capacity=1024):
    return lib.uc_mots_masks_rle(masks, n_max, Hin, Win, rows, emit, K, img_h, img_w, ctypes.c_float(thres), ctypes.c_double(sf), ws,
                                 ctypes.c_long(ws_bytes), out_len, out_off, out_total, chars, ctypes.c_long(capacity), None)


@pytest.mark.parametrize("bad,msg", [
    (dict(masks=None), b"null pointer"), (dict(rows=None), b"null pointer"), (dict(emit=None), b"null pointer"),
    (dict(ws=None), b"null pointer"), (dict(out_len=None), b"null pointer"), (dict(out_total=None), b"null pointer"),
    (dict(chars=None), b"null pointer"),
    (dict(K=9), b"n_max"), (dict(K=0), b"n_max"),
    (dict(Hin=0), b"non-positive sizes"), (dict(Win=-1), b"non-positive sizes"), (dict(img_h=0), b"non-positive sizes"),
    (dict(img_w=0), b"non-positive sizes"),
    (dict(sf=0.0), b"scale_factor"), (dict(sf=-1.5), b"scale_factor"), (dict(sf=float("nan")), b"scale_factor"),
    (dict(sf=0.01), b"empty"),
    (dict(capacity=0), b"capacity"),
    (dict(ws_bytes=16), b"workspace"),
])
def test_masks_rle_rejects_bad_arguments_before_any_launch(bad, msg):
    from unicorn_b200 import _lib
    lib = _lib.lib()
    lib.uc_last_error.restype = ctypes.c_char_p
    assert _call(lib, **bad) == -1  # UC_EINVAL: no launch was attempted (without a GPU a launch would give a CUDA error)
    assert msg in lib.uc_last_error()


def test_workspace_bytes_follows_the_cropped_resized_map():
    from unicorn_b200 import _lib
    fn = _lib.lib().uc_mots_rle_workspace_bytes
    fn.restype = ctypes.c_long
    d = ctypes.c_double
    # 800x1280 at 1.5 -> 1200x1920, cropped to the 1080x1920 frame: 1920 columns of 34 words
    assert fn(64, 800, 1280, 1080, 1920, d(1.5)) == 64 * 1920 * 34 * 4
    # the short-map case: a 402x640 frame at 800x1280 has scale_factor 402/800; 800 * sf = 401.99999999999994 in double, so the
    # resized map is 401x643 and the encoded mask 401x640
    sf = 1 / min(800 / 402, 1280 / 640)
    assert fn(1, 800, 1280, 402, 640, d(sf)) == 640 * ((401 + 31) // 32) * 4
    assert fn(0, 800, 1280, 402, 640, d(sf)) == 0 and fn(1, 800, 1280, 402, 640, d(0.0)) == 0


def _reference(keep, index, boxes, ids, masks, min_box_area):
    """The previous driver's host path: masks[keep][index][ids > -1] -> results.mots_frame_result."""
    from unicorn_b200 import results as R
    m = masks[keep][index]
    valid = ids > -1
    return R.mots_frame_result(7, boxes[valid], ids[valid], m[valid], masks.shape[1], masks.shape[2], min_box_area)


def _via_rows(keep, index, boxes, ids, masks, min_box_area):
    from unicorn_b200 import results as R
    from unicorn_b200.mots import mots_rows
    rows, emit, out_ids = mots_rows(keep, index, boxes, ids, min_box_area)
    assert len(rows) == len(emit) and sum(emit) == len(out_ids)
    free = R.overlap_free(masks[rows]) if rows else masks[:0]
    return 7, out_ids, 2, masks.shape[1], masks.shape[2], [R.rle_encode(free[i].numpy()) for i in range(len(rows)) if emit[i]]


def _box(x1, y1, w, h, s=0.9):
    return [x1, y1, x1 + w, y1 + h, s]


def _masks(n, H=24, W=20, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, H, W, generator=g) > 0.5


CASES = {
    # unsorted ids; every box above the area limit
    "unsorted": (torch.tensor([1, 1, 1, 1], dtype=torch.bool), torch.tensor([True, True, True, True]),
                 torch.tensor([_box(0, 0, 20, 20), _box(5, 5, 30, 10), _box(1, 1, 11, 11), _box(2, 2, 50, 3)]), torch.tensor([7, 2, 9, 0])),
    # -1 ids (unmatched / not initialised) drop out of the ordering but not the rest
    "minus_one": (torch.tensor([1, 0, 1, 1, 1], dtype=torch.bool), torch.tensor([True, True, True, True]),
                  torch.tensor([_box(0, 0, 20, 20), _box(5, 5, 30, 10), _box(1, 1, 11, 11), _box(2, 2, 50, 3)]), torch.tensor([3, -1, 1, -1])),
    # area exactly at the limit (100 = 10 x 10, not emitted), just above it, and below it: the rows still claim their pixels
    "area_limit": (torch.tensor([1, 1, 1, 1], dtype=torch.bool), torch.tensor([True, True, True, True]),
                   torch.tensor([_box(0, 0, 10, 10), _box(3.5, 2.25, 10, 10.0001), _box(0, 0, 4, 4), _box(1, 1, 25, 4)]),
                   torch.tensor([4, 1, 0, 2])),
    # match() dropped a duplicate: its index is a boolean mask over the kept rows (applied as the reference applies it)
    "index_mask": (torch.tensor([1, 1, 0, 1, 1, 1], dtype=torch.bool), torch.tensor([True, False, True, True, True]),
                   torch.tensor([_box(0, 0, 20, 20), _box(5, 5, 30, 10), _box(1, 1, 11, 11), _box(2, 2, 50, 3)]), torch.tensor([5, 6, -1, 2])),
    "all_invalid": (torch.tensor([1, 1], dtype=torch.bool), torch.tensor([True, True]),
                    torch.tensor([_box(0, 0, 20, 20), _box(5, 5, 30, 10)]), torch.tensor([-1, -1])),
}


@pytest.mark.parametrize("name", sorted(CASES))
@pytest.mark.parametrize("min_box_area", [0, 100])
def test_mots_rows_matches_mots_frame_result(name, min_box_area):
    keep, index, boxes, ids = CASES[name]
    masks = _masks(keep.numel(), seed=len(name))
    ref = _reference(keep, index, boxes, ids, masks, min_box_area)
    got = _via_rows(keep, index, boxes, ids, masks, min_box_area)
    assert got == ref


def test_mots_rows_random():
    rng = np.random.default_rng(5)
    for trial in range(50):
        n = int(rng.integers(1, 12))
        keep = torch.as_tensor(rng.random(n) < 0.8)
        nk = int(keep.sum())
        index = torch.as_tensor(rng.random(nk) < 0.9)
        m = int(index.sum())
        xy = rng.uniform(0, 50, (m, 2))
        wh = rng.choice([5.0, 10.0, 12.5, 20.0], (m, 2))
        boxes = torch.as_tensor(np.concatenate([xy, xy + wh, rng.random((m, 1))], 1), dtype=torch.float32)
        ids = torch.as_tensor(rng.permutation(40)[:m] - 5)
        ids[ids < -1] = -1
        masks = _masks(n, seed=trial)
        assert _via_rows(keep, index, boxes, ids, masks, 100) == _reference(keep, index, boxes, ids, masks, 100)
