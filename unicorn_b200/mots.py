"""MOTS per-frame driver: the per-frame body of MOTEvaluator.evaluate_omni_mots (unicorn/evaluators/mot_evaluator.py:776-897) on
the B200 engine: whole-mode detector with the CondInst controllers -> NMS -> dynamic-conv masks of the kept detections -> embedding
sampling -> QuasiDenseEmbedTracker.match(return_index=True) -> masks of the tracked boxes in ascending-id order, overlap free,
area filter, COCO RLE.

Like UnicornMOTTracker's QDTrack arm (mot.py) the frame is split in a device half and a host half:

  submit(frame, img_h, img_w)  enqueues every kernel of the frame (optionally as one of two CUDA-graph replays, by frame parity)
                               and asynchronous copies of (count, detections, sampled embeddings) into a pinned slot, and records
                               an event; the soft masks stay on the device, in a buffer of the frame's parity;
  collect()                    waits for the oldest slot, runs the association on the host (mots_rows), then resizes, thresholds,
                               makes overlap free and run-length encodes the selected masks on the device (ops.mots_masks_rle, on
                               a side stream): only the RLE lengths and bytes come back, never a full-resolution mask.

`submit(t+1); collect(t)` overlaps the association and encoding of frame t with the device work of frame t+1; the results are
those of the sequential `step_tensor`.  tests/test_mots_gpu.py and tests/test_mots_rle_gpu.py check the driver on a B200."""
import torch

from . import ops
from .engine import UnicornEngine
from .tracker import QuasiDenseEmbedTracker


def mots_rows(keep, index, boxes, ids, min_box_area=100):
    """Host row selection of one MOTS frame after QuasiDenseEmbedTracker.match (mot_evaluator.py:846-884).  keep: bool [n], the
    score filter over the n NMS rows; (boxes [m,5], ids [m], index) = match(..., return_index=True) on the kept rows.  The masks
    are indexed as the reference indexes them (masks[keep][index][ids > -1], :857-858), then ordered by ascending id.  Returns
    (rows, emit, out_ids): the NMS row of every valid track in ascending-id order, 1 where its box area exceeds min_box_area
    (the rows with 0 still take part in the overlap-free step), and the 1-based ids of the emitted rows — what
    results.mots_frame_result computes from the masks themselves."""
    rows = torch.nonzero(torch.as_tensor(keep, dtype=torch.bool)).view(-1)[torch.as_tensor(index)]
    ids = torch.as_tensor(ids).long()
    boxes = torch.as_tensor(boxes, dtype=torch.float32)
    valid = ids > -1
    rows, boxes, ids = rows[valid], boxes[valid], ids[valid]
    order = ids.sort()[1]
    rows, boxes, ids = rows[order].tolist(), boxes[order], ids[order].tolist()
    emit, out_ids = [], []
    for i, tid in enumerate(ids):
        x1, y1, x2, y2 = boxes[i, :4].tolist()
        e = (x2 - x1) * (y2 - y1) > min_box_area
        emit.append(int(e))
        if e:
            out_ids.append(tid + 1)  # 1-based ids for the MOTS files
    return rows, emit, out_ids


class UnicornMOTSTracker:
    def __init__(self, engine: UnicornEngine, input_size, conf=0.01, nms=0.7, score_thr=0.1, max_dets=64, mask_thres=0.3, d_rate=2,
                 min_box_area=100, tracker=None, use_graph=False):
        assert engine.cfg["mask"], "MOTS needs a *_mask model"
        self.eng, self.input_size = engine, tuple(input_size)
        self.conf, self.nms, self.score_thr, self.max_dets = conf, nms, score_thr, max_dets
        self.mask_thres, self.d_rate, self.min_box_area = mask_thres, d_rate, min_box_area
        self.tracker = tracker or QuasiDenseEmbedTracker(device=engine.dev)
        H, W = self.input_size
        A = (H // 8) * (W // 8) + (H // 16) * (W // 16) + (H // 32) * (W // 32)
        dev = engine.dev
        self.ws = ops.PostWorkspace(A, dev)
        self.img_in = torch.empty(1, 3, H, W, dtype=torch.float32, device=dev)
        self.img_in_u8 = torch.empty(1, H, W, 3, dtype=torch.uint8, device=dev)  # letterboxed BGR frame as cv2 / the decoder delivers it
        self._u8 = False
        self.feats = torch.zeros(max_dets, 128, dtype=torch.float32, device=dev)
        # soft masks by frame parity: collect(t) encodes frame t's masks while frame t+1's are written
        h, w, up = H // 8, W // 8, 8 // d_rate
        self._masks = [torch.zeros(max_dets, h * up * d_rate, w * up * d_rate, dtype=torch.float32, device=dev) for _ in range(2)]
        self._mask_scratch = torch.empty(max_dets * h * w * (1 + up * up), dtype=torch.float32, device=dev)
        self.frame_id = 0       # frames submitted
        self.collected = 0      # frames associated
        self._prev_feat = torch.zeros(1, H // 16, W // 16, engine.dims[2], dtype=torch.bfloat16, device=dev)
        self._has_prev = torch.zeros(1, dtype=torch.int32, device=dev)
        self._slots = [dict(cnt=torch.zeros(1, dtype=torch.int32).pin_memory(), dets=torch.zeros(max_dets, 7).pin_memory(),
                            feats=torch.zeros(max_dets, 128).pin_memory(), ev=torch.cuda.Event(), img=(0, 0), frame_id=0, dev={})
                       for _ in range(2)]
        self.use_graph = use_graph
        self._graphs = {}
        self._rle_stream = torch.cuda.Stream(device=dev)
        self._rle_ws = ops.MotsRleWorkspace(dev)
        self.last = {}

    # ------------------------------------------------------------------------------------------ device half
    def _device_frame(self, parity):
        e = self.eng
        e.begin_frame()
        fpn, seq = e.backbone(self.img_in_u8 if self._u8 else self.img_in, tag="mots%d" % parity)
        out = e.head(fpn, None, "mot", with_masks=True)
        dets, cnt = ops.postprocess_device(out[0], e.ncls, self.conf, self.nms, self.ws)
        mf, um = e.mask_branch(fpn)
        hw = [(t.shape[1], t.shape[2]) for t in e.dyn_levels]
        ops.dynamic_masks(mf, um, e.dyn_levels, hw, self.ws, self.max_dets, up_rate=8 // self.d_rate, d_rate=self.d_rate,
                          out=self._masks[parity], scratch=self._mask_scratch)
        ops.copy_rows_if(self._has_prev, seq["feat"], self._prev_feat, invert=True)  # first frame with detections: pre_dict = cur_dict (:812-813)
        _, f_cur = e.interaction(self._prev_feat, seq["feat"])
        emb = e.upsample(f_cur, "mots.emb")
        ops.sample_embed(emb, dets, self.max_dets, 8.0, count=cnt, out=self.feats)
        ops.copy_rows_if(cnt, seq["feat"], self._prev_feat)  # pre_dict advances only on frames with detections (:803,818)
        self._has_prev.bitwise_or_((cnt > 0).to(torch.int32))
        self.last = dict(head=out, mask_feats=mf, up_masks=um, dyn=[t for t in e.dyn_levels])

    def submit(self, frame, img_h, img_w):
        """frame: preprocessed fp32 [1,3,H,W] or letterboxed uint8 [1,H,W,3] (the float conversion happens in the stem kernel), host
        or device; (img_h, img_w): original image size.  Enqueues the frame; returns immediately."""
        assert self.frame_id - self.collected < 2, "collect() the previous frame first"
        self.frame_id += 1
        parity = self.frame_id & 1
        u8 = frame.dtype == torch.uint8
        if u8 != self._u8:
            self._u8, self._graphs = u8, {}  # the captured graphs read one of the two static input buffers
        (self.img_in_u8 if u8 else self.img_in).copy_(frame, non_blocking=True)
        if self.use_graph and self.frame_id > 2:
            g = self._graphs.get(parity)
            if g is None:  # frames 1-2 ran eagerly (plan-time autotuning, buffer allocation); 3 and 4 are captured
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._device_frame(parity)
                self._graphs[parity] = g = (g, self.last)
            g[0].replay()
            dev_out = g[1]
        else:
            self._device_frame(parity)
            dev_out = self.last
        s = self._slots[parity]
        s["cnt"].copy_(self.ws.count.view(-1)[:1], non_blocking=True)
        s["dets"].copy_(self.ws.dets[:self.max_dets], non_blocking=True)
        s["feats"].copy_(self.feats, non_blocking=True)
        s["img"], s["frame_id"], s["dev"] = (img_h, img_w), self.frame_id, dev_out
        s["ev"].record()

    # ------------------------------------------------------------------------------------------ host half
    def collect(self):
        """Association and mask encoding of the oldest submitted frame.  Returns the tuple write_results_mots() consumes:
        (frame_id, ids (1-based), cat_id, img_h, img_w, rles)."""
        assert self.collected < self.frame_id, "nothing submitted"
        self.collected += 1
        parity = self.collected & 1
        s = self._slots[parity]
        s["ev"].synchronize()
        n = min(int(s["cnt"][0]), self.max_dets)
        d, f = s["dets"][:n].clone(), s["feats"][:n].clone()
        img_h, img_w = s["img"]
        H, W = self.input_size
        scale = min(H / float(img_h), W / float(img_w))
        masks = self._masks[parity]
        # head / mask_feats / up_masks / dyn are engine buffers: they describe this frame until the next one is submitted
        self.last = dict(s["dev"], dets=d, feats=f, masks=masks[:n])
        if n == 0:  # outputs[0] is None: no tracking for this frame (mot_evaluator.py:803)
            return s["frame_id"], [], 2, img_h, img_w, []
        scores = d[:, 4] * d[:, 5]
        keep = scores > self.score_thr
        boxes = torch.cat([d[keep, :4] / scale, scores[keep, None]], 1)
        ob, _, oid, idx = self.tracker.match(boxes, torch.ones(boxes.size(0)), f[keep], s["frame_id"], return_index=True)
        rows, emit, ids = mots_rows(keep, idx, ob, oid, self.min_box_area)
        rles = []
        if rows:
            with torch.cuda.stream(self._rle_stream):
                self._rle_stream.wait_event(s["ev"])
                sel = torch.tensor([rows, emit], dtype=torch.int32).to(masks.device, non_blocking=True)
                rles = ops.mots_masks_rle(masks, sel[0], sel[1], img_h, img_w, self.mask_thres, 1 / scale, self._rle_ws)
        return s["frame_id"], ids, 2, img_h, img_w, rles

    def step_tensor(self, frame, img_h, img_w):
        """Sequential protocol of the reference: one frame in (preprocessed fp32 [1,3,H,W] or uint8 [1,H,W,3]; original image size
        (img_h, img_w)), its MOTS tuple out."""
        self.submit(frame, img_h, img_w)
        return self.collect()
