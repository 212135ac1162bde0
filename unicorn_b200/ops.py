"""Python wrappers over the C ABI.  Tensors are torch CUDA tensors used purely as device memory:
activations are NHWC views (B, H, W, C) with unit channel stride and a constant pixel stride (so a channel
slice of a wider buffer is a valid operand, which is how concatenations are formed without copies)."""
import ctypes

import torch

from . import _lib
from ._lib import BF16, F32, F16, ACT_NONE, ACT_RELU, ACT_GELU, ACT_SILU, ACT_SIGMOID  # noqa: F401

_DT = {torch.bfloat16: BF16, torch.float32: F32, torch.float16: F16}


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _nhwc_ld(t):
    """pixel stride of an NHWC view; validates the layout."""
    assert t.dim() == 4 and t.is_cuda, "expected a CUDA NHWC tensor"
    B, H, W, C = t.shape
    ld = t.stride(2) if W > 1 else (t.stride(1) // W if H > 1 else max(C, t.stride(2)))
    assert t.stride(3) == 1 or C == 1
    if W > 1:
        assert t.stride(2) == ld
    if H > 1:
        assert t.stride(1) == W * ld, (t.shape, t.stride())
    if B > 1:
        assert t.stride(0) == H * W * ld
    return ld


def pack_conv_weight(w, dtype=torch.bfloat16, cout_pad=8):
    """[Cout, Cin, KH, KW] (or [Cout, Cin] for Linear) fp32 -> [Cout_pad, KH*KW, Cin] 16-bit, K-major."""
    if w.dim() == 2:
        w = w[:, :, None, None]
    Cout, Cin, KH, KW = w.shape
    Cp = (Cout + cout_pad - 1) // cout_pad * cout_pad
    out = torch.zeros(Cp, KH * KW, Cin, dtype=dtype, device=w.device)
    out[:Cout] = w.permute(0, 2, 3, 1).reshape(Cout, KH * KW, Cin).to(dtype)
    return out.contiguous()


CONV_TRACE = None


def conv2d(x, w_packed, KH, KW, stride=1, pad=0, bias=None, act=ACT_NONE, gamma=None, res=None, out=None,
           out_dtype=None, block_n=0, gn_stats=None, gn_groups=0, row_stats=None, col_s=None, row_eps=1e-6):
    """x: NHWC view (B,H,W,Cin) bf16/f16.  w_packed: [Cout, KH*KW, Cin].  Returns NHWC (B,Ho,Wo,Cout)."""
    B, H, W, Cin = x.shape
    Cout = w_packed.shape[0]
    assert w_packed.shape[1] == KH * KW and w_packed.shape[2] == Cin and w_packed.is_contiguous()
    assert w_packed.dtype == x.dtype
    Ho = (H + 2 * pad - KH) // stride + 1
    Wo = (W + 2 * pad - KW) // stride + 1
    if out is None:
        out = torch.empty(B, Ho, Wo, Cout, dtype=out_dtype or x.dtype, device=x.device)
    assert out.shape == (B, Ho, Wo, Cout), (out.shape, (B, Ho, Wo, Cout))
    d = _lib.UcConv2d()
    d.x, d.x_dtype = _p(x), _DT[x.dtype]
    d.B, d.H, d.W, d.Cin, d.ldx = B, H, W, Cin, _nhwc_ld(x)
    d.w = _p(w_packed)
    d.Cout, d.KH, d.KW, d.stride, d.pad = Cout, KH, KW, stride, pad
    d.bias, d.act, d.gamma = _p(bias), act, _p(gamma)
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() >= Cout
    if gamma is not None:
        assert gamma.dtype == torch.float32 and gamma.numel() >= Cout
    d.res, d.ldres = _p(res), (_nhwc_ld(res) if res is not None else 0)
    if res is not None:
        assert res.dtype == out.dtype and res.shape == out.shape
    d.y, d.ldy, d.y_dtype = _p(out), _nhwc_ld(out), _DT[out.dtype]
    d.block_n = block_n
    d.gn_stats, d.gn_groups = _p(gn_stats), gn_groups
    d.row_stats, d.col_s, d.row_eps = _p(row_stats), _p(col_s), row_eps
    if row_stats is not None:
        assert row_stats.dtype == torch.int64 and row_stats.numel() == B * H * W * 2 and col_s is not None and col_s.numel() >= Cout
    if CONV_TRACE is not None:  # tools/profile_frame.py: conv launches in issue order, to label an ncu launch list
        CONV_TRACE.append(dict(M=B * Ho * Wo, N=Cout, K=Cin * KH * KW, k=KH, s=stride, bn=block_n, act=act, gn=gn_groups,
                               f32=int(out.dtype == torch.float32)))
    _lib.check(_lib.lib().uc_conv2d(ctypes.byref(d), _lib.stream_ptr()), "uc_conv2d")
    return out


def linear(x2d, w_packed, **kw):
    """x2d: [M, K] rows (unit inner stride).  Returns [M, N]."""
    M, K = x2d.shape
    assert x2d.stride(1) == 1
    x4 = x2d.as_strided((1, 1, M, K), (M * x2d.stride(0), M * x2d.stride(0), x2d.stride(0), 1))
    out = kw.pop("out", None)
    res = kw.pop("res", None)
    if out is not None:
        out = out.as_strided((1, 1, M, out.shape[1]), (M * out.stride(0), M * out.stride(0), out.stride(0), 1))
    if res is not None:
        res = res.as_strided((1, 1, M, res.shape[1]), (M * res.stride(0), M * res.stride(0), res.stride(0), 1))
    y = conv2d(x4, w_packed, 1, 1, out=out, res=res, **kw)
    return y.as_strided((M, y.shape[3]), (y.stride(2), 1))


# ------------------------------------------------------------------------------------------- other entry points
def _L():
    return _lib.lib()


def _S():
    return _lib.stream_ptr()


_f = ctypes.c_float
_i = ctypes.c_int
_l = ctypes.c_long


def pack_stem_weight(w):
    """[C0,3,4,4] -> [48, C0] fp32 (k = (ci*4+kh)*4+kw)."""
    return w.reshape(w.shape[0], 48).t().contiguous().float()


def pack_dw_weight(w):
    """[C,1,7,7] -> [49, C] fp32."""
    return w.reshape(w.shape[0], 49).t().contiguous().float()


def pack_dw_weight_mma(w, bias):
    """[C,1,7,7], [C] -> int32 [ceil(C/32), 1824]: per 32-channel chunk the bf16 tap pairs {e[j-1], e[j]}, j = 0..7, of every channel
    and filter row ([32][7][8] words; e = the row padded with zeros, lower index in the low half) followed by the 32 fp32 biases; zero
    for the channels that pad C to a multiple of 32 — the operand of uc_dwconv7_mma, which builds the B fragments of its Toeplitz
    blocks T[k][n] = e[k-n-1] from it."""
    C = w.shape[0]
    Cp = -(-C // 32) * 32
    e = torch.zeros(Cp, 7, 9, dtype=torch.bfloat16, device=w.device)  # e[-1] .. e[7]
    e[:C, :, 1:8] = w.reshape(C, 7, 7).to(torch.bfloat16)
    bits = e.view(torch.int16).to(torch.int32) & 0xffff
    pairs = (bits[:, :, 0:8] | (bits[:, :, 1:9] << 16)).to(torch.int32).reshape(Cp // 32, 32 * 7 * 8)
    bp = torch.zeros(Cp, dtype=torch.float32, device=w.device)
    bp[:C] = bias.float()
    return torch.cat([pairs, bp.view(torch.int32).reshape(Cp // 32, 32)], dim=1).contiguous()


def dwconv7_mma(x, qtab, out=None, work_counter=None):
    B, H, W, C = x.shape
    assert x.is_contiguous() and x.dtype == torch.bfloat16 and qtab.dtype == torch.int32 and qtab.shape == (-(-C // 32), 1824)
    if out is None:
        out = torch.empty_like(x)
    _lib.check(_L().uc_dwconv7_mma(_p(x), _p(qtab), _p(out), B, H, W, C, _p(work_counter), _S()), "uc_dwconv7_mma")
    return out


def convnext_mlp_supported(C):
    return bool(_L().uc_convnext_mlp_supported(int(C)))


def convnext_mlp(t, w1f, c1, w2, b2, gamma, x, eps=1e-6):
    """x[M,C] += gamma * (W2 . GELU(W1f . LN0(t) + c1) + b2) in one launch (uc_convnext_mlp); t, x: [M, C] bf16 contiguous."""
    M, C = t.shape
    assert t.is_contiguous() and x.is_contiguous() and x.shape == t.shape and t.dtype == x.dtype == torch.bfloat16
    assert w1f.dtype == torch.bfloat16 and w1f.numel() == 4 * C * C and w2.dtype == torch.bfloat16 and w2.numel() == 4 * C * C
    _lib.check(_L().uc_convnext_mlp(_p(t), _p(w1f), _p(c1), _p(w2), _p(b2), _p(gamma), _p(x), M, C, ctypes.c_float(eps), _S()), "uc_convnext_mlp")
    return x


def stem_ln(img, w48, bias, lnw, lnb, eps=1e-6):
    """img: fp32 NCHW [B,3,H,W] or uint8 NHWC [B,H,W,3] (BGR)."""
    u8 = img.dtype == torch.uint8
    if u8:
        B, H, W, _ = img.shape
    else:
        B, _, H, W = img.shape
        assert img.dtype == torch.float32
    assert img.is_contiguous()
    C0 = w48.shape[1]
    out = torch.empty(B, H // 4, W // 4, C0, dtype=torch.bfloat16, device=img.device)
    _lib.check(_L().uc_stem_ln(_p(img), int(u8), _p(w48), _p(bias), _p(lnw), _p(lnb), _p(out), B, H, W, C0, _f(eps), _S()), "uc_stem_ln")
    return out


def dwconv7_ln(x, w49, bias, lnw, lnb, eps=1e-6, out=None):
    B, H, W, C = x.shape
    assert x.is_contiguous() and x.dtype == torch.bfloat16
    if out is None:
        out = torch.empty_like(x)
    _lib.check(_L().uc_dwconv7_ln(_p(x), _p(w49), _p(bias), _p(lnw), _p(lnb), _p(out), B, H, W, C, _f(eps), _S()), "uc_dwconv7_ln")
    return out


def dwconv7(x, w49, bias, out=None, ln_stats=None, work_counter=None):
    B, H, W, C = x.shape
    assert x.is_contiguous() and x.dtype == torch.bfloat16
    if out is None:
        out = torch.empty_like(x)
    if ln_stats is not None:
        assert ln_stats.dtype == torch.int64 and ln_stats.is_contiguous() and ln_stats.numel() == B * H * W * 2
    if work_counter is not None:
        assert work_counter.dtype == torch.int32 and work_counter.numel() >= 1
    _lib.check(_L().uc_dwconv7(_p(x), _p(w49), _p(bias), _p(out), B, H, W, C, _p(ln_stats), _p(work_counter), _S()), "uc_dwconv7")
    return out


def layernorm(x2d, w, b, eps, res=None, out=None):
    """rows [M, C] (unit inner stride)."""
    M, C = x2d.shape
    if out is None:
        out = torch.empty(M, C, dtype=x2d.dtype, device=x2d.device)
    _lib.check(_L().uc_layernorm(_p(x2d), x2d.stride(0), _p(res), res.stride(0) if res is not None else 0, _p(w), _p(b),
                                 _p(out), out.stride(0), _l(M), C, _f(eps), _DT[x2d.dtype], _S()), "uc_layernorm")
    return out


def groupnorm_apply(x, stats, w, b, G, eps, act, out=None, prior=None, beta=None, add2=None, out2=None):
    """x NHWC view; in-place when out is None."""
    B, H, W, C = x.shape
    if out is None:
        out = x
    ld2 = _nhwc_ld(add2) if add2 is not None else 0
    _lib.check(_L().uc_groupnorm_apply(_p(x), _nhwc_ld(x), _p(stats), _p(w), _p(b), _p(out), _nhwc_ld(out), B, _l(H * W), C, G,
                                       _f(eps), act, _p(prior), _p(beta), _p(add2), ld2, _p(out2),
                                       _nhwc_ld(out2) if out2 is not None else 0, _S()), "uc_groupnorm_apply")
    return out


def copy_upsample(src, dst, up):
    B, Hs, Ws, C = src.shape
    assert dst.shape == (B, Hs * up, Ws * up, C)
    _lib.check(_L().uc_copy_upsample(_p(src), _nhwc_ld(src), _p(dst), _nhwc_ld(dst), B, Hs, Ws, C, up, _S()), "uc_copy_upsample")
    return dst


def pixel_shuffle2(x, out=None):
    B, H, W, C4 = x.shape
    Co = C4 // 4
    if out is None:
        out = torch.empty(B, 2 * H, 2 * W, Co, dtype=x.dtype, device=x.device)
    _lib.check(_L().uc_pixel_shuffle2(_p(x), _nhwc_ld(x), _p(out), _nhwc_ld(out), B, H, W, Co, _S()), "uc_pixel_shuffle2")
    return out


def bilinear(src, Hd, Wd, scale_h=0.0, scale_w=0.0, out=None):
    """src fp32 [..., Hs, Ws] contiguous planes."""
    Hs, Ws = src.shape[-2:]
    P = src.numel() // (Hs * Ws)
    if out is None:
        out = torch.empty(*src.shape[:-2], Hd, Wd, dtype=torch.float32, device=src.device)
    _lib.check(_L().uc_bilinear_f32(_p(src), _p(out), P, Hs, Ws, Hd, Wd, _f(scale_h), _f(scale_w), _S()), "uc_bilinear_f32")
    return out


def add(a2d, b2d, out=None):
    M, C = a2d.shape
    if out is None:
        out = torch.empty(M, C, dtype=a2d.dtype, device=a2d.device)
    _lib.check(_L().uc_add(_p(a2d), a2d.stride(0), _p(b2d), b2d.stride(0), _p(out), out.stride(0), _l(M), C, _DT[a2d.dtype], _S()), "uc_add")
    return out


def copy_rows_if(flag, src, dst, invert=False):
    """dst <- src (NHWC views of equal shape, channel-contiguous) when (flag[0] != 0) != invert — decided on the device."""
    assert src.shape == dst.shape and src.dtype == dst.dtype and flag.dtype == torch.int32
    C = src.shape[-1]
    rows = src.numel() // C
    es = src.element_size()
    _lib.check(_L().uc_copy_rows_if(_p(flag), int(bool(invert)), _p(src), _l(_nhwc_ld(src) * es), _p(dst), _l(_nhwc_ld(dst) * es), _l(rows), C * es, _S()),
               "uc_copy_rows_if")
    return dst


def letterbox_u8(src, input_size, swap_rb=True, pad=114, out=None):
    """src: uint8 [h,w,3] device tensor (RGB when swap_rb) -> (uint8 [1,H,W,3] letterboxed frame, r) — the preprocessing of
    external/lib/test/tracker/unicorn_sot.py:114-123 (swap_rb=True) / data_augment.py:194-214 (swap_rb=False)."""
    assert src.dtype == torch.uint8 and src.is_cuda and src.is_contiguous() and src.dim() == 3 and src.shape[2] == 3
    h, w = src.shape[:2]
    H, W = input_size
    r = min(H / h, W / w)
    if out is None:
        out = torch.empty(1, H, W, 3, dtype=torch.uint8, device=src.device)
    _lib.check(_L().uc_letterbox_u8(_p(src), h, w, _p(out), H, W, int(h * r), int(w * r), int(bool(swap_rb)), int(pad), _S()), "uc_letterbox_u8")
    return out, r


def nchw_to_nhwc(x, dtype=torch.bfloat16, out=None):
    B, C, H, W = x.shape
    assert x.dtype == torch.float32 and x.is_contiguous()
    if out is None:
        out = torch.empty(B, H, W, C, dtype=dtype, device=x.device)
    _lib.check(_L().uc_nchw_f32_to_nhwc(_p(x), _p(out), _nhwc_ld(out), B, C, _l(H * W), _DT[out.dtype], _S()), "uc_nchw_f32_to_nhwc")
    return out


def nhwc_to_nchw(x):
    B, H, W, C = x.shape
    assert x.dtype in (torch.bfloat16, torch.float16), "uc_nhwc_to_nchw_f32 converts 16-bit NHWC maps"
    out = torch.empty(B, C, H, W, dtype=torch.float32, device=x.device)
    _lib.check(_L().uc_nhwc_to_nchw_f32(_p(x), _nhwc_ld(x), _p(out), B, C, _l(H * W), _DT[x.dtype], _S()), "uc_nhwc_to_nchw_f32")
    return out


def msda_forward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight):
    """Reference operator semantics (fp32)."""
    B, S, M, D = value.shape
    _, Lq, _, L, P, _ = sampling_loc.shape
    out = torch.empty(B, Lq, M * D, dtype=torch.float32, device=value.device)
    _lib.check(_L().uc_msda_forward_f32(_p(value), _p(spatial_shapes), _p(level_start_index), _p(sampling_loc), _p(attn_weight),
                                        B, S, M, D, L, Lq, P, _p(out), _S()), "uc_msda_forward_f32")
    return out


def msda_fused(value, offlog, level_hw, M=8, P=4, out=None):
    L = len(level_hw)
    Lq = sum(h * w for h, w in level_hw)
    assert value.shape == (Lq, M * 32) and value.dtype == torch.bfloat16 and value.is_contiguous()
    assert offlog.dtype == torch.float32 and offlog.shape[0] == Lq and offlog.shape[1] >= M * L * P * 3
    if out is None:
        out = torch.empty(Lq, M * 32, dtype=torch.bfloat16, device=value.device)
    hw = (ctypes.c_int * (2 * L))(*[v for pair in level_hw for v in pair])
    _lib.check(_L().uc_msda_fused_bf16(_p(value), _p(offlog), offlog.stride(0), _p(out), hw, L, M, P, _S()), "uc_msda_fused_bf16")
    return out


def corr_propagate(embed_ref, embed_cur, values, out=None):
    """embed_* [n, 128] 16-bit rows; values fp32 [n_obj, n_ref] -> fp32 [n_obj, n_cur]."""
    n_ref, C = embed_ref.shape
    n_cur = embed_cur.shape[0]
    n_obj = values.shape[0]
    assert values.dtype == torch.float32 and values.stride(1) == 1 and values.shape[1] == n_ref
    if out is None:
        out = torch.empty(n_obj, n_cur, dtype=torch.float32, device=values.device)
    _lib.check(_L().uc_corr_propagate(_p(embed_ref), embed_ref.stride(0), n_ref, _p(embed_cur), embed_cur.stride(0), n_cur, C,
                                      _DT[embed_ref.dtype], _p(values), values.stride(0), n_obj, _p(out), out.stride(0), _S()),
               "uc_corr_propagate")
    return out


def head_decode(regobj, cls, hw, strides, ncls, out=None):
    A = sum(h * w for h, w in hw)
    if out is None:
        out = torch.empty(1, A, 5 + ncls, dtype=torch.float32, device=regobj[0].device)
    ro = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in regobj])
    cl = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in cls])
    hwa = (ctypes.c_int * 6)(*[v for pair in hw for v in pair])
    st = (ctypes.c_int * 3)(*strides)
    _lib.check(_L().uc_head_decode(ro, cl, hwa, st, regobj[0].shape[-1], cls[0].shape[-1], ncls, _p(out), _S()), "uc_head_decode")
    return out


class PostWorkspace:
    def __init__(self, max_anchors, device):
        fn = _L().uc_postprocess_workspace_bytes
        fn.restype = ctypes.c_long
        self.nbytes = fn(max_anchors)
        self.buf = torch.empty(self.nbytes, dtype=torch.uint8, device=device)
        self.dets = torch.empty(max_anchors, 7, dtype=torch.float32, device=device)
        self.count = torch.zeros(1, dtype=torch.int32, device=device)
        self.anchors = torch.zeros(max_anchors, dtype=torch.int32, device=device)
        self.max_anchors = max_anchors


def postprocess_device(pred, ncls, conf, nms, ws, max_keep=0):
    """pred fp32 [A, 5+ncls] (decoded).  Launches only; ws.dets / ws.count hold the result.
    max_keep > 0 returns exactly the first max_keep rows of the full NMS result."""
    A = pred.shape[0]
    assert pred.is_contiguous() and pred.dtype == torch.float32 and A <= ws.max_anchors
    _lib.check(_L().uc_postprocess(_p(pred), A, ncls, _f(conf), _f(nms), int(max_keep), _p(ws.buf), _l(ws.nbytes), _p(ws.dets), _p(ws.count), _p(ws.anchors), _S()),
               "uc_postprocess", 4)
    return ws.dets, ws.count


def sample_embed(embed, boxes, n_max, stride=8.0, count=None, out=None):
    """embed NHWC 16-bit [1,h,w,C]; boxes fp32 [>=n_max, >=4] (device); returns fp32 [n_max, C]."""
    _, h, w, C = embed.shape
    if out is None:
        out = torch.zeros(n_max, C, dtype=torch.float32, device=embed.device)
    _lib.check(_L().uc_sample_embed(_p(embed), _nhwc_ld(embed), h, w, C, _DT[embed.dtype], _p(boxes), boxes.stride(0), _p(count), n_max,
                                    _f(stride), _p(out), _S()), "uc_sample_embed")
    return out


def bisoftmax(det_embeds, memo_embeds, det_labels=None, memo_labels=None):
    N, C = det_embeds.shape
    M = memo_embeds.shape[0]
    ws = torch.empty(N * M + 2 * N + 2 * M, dtype=torch.float32, device=det_embeds.device)
    scores = torch.empty(N, M, dtype=torch.float32, device=det_embeds.device)
    _lib.check(_L().uc_bisoftmax(_p(det_embeds), _p(memo_embeds), N, M, C, _p(det_labels), _p(memo_labels), _p(ws), _p(scores), _S()),
               "uc_bisoftmax", 3)
    return scores


def qd_assign(scores, memo_ids, boxes5, match_thr, obj_thr, nms_conf_thr):
    """scores f32 [N,M] (device), memo_ids int64 [M], boxes5 f32 [N,5] (score in column 4) -> ids int64 [N] (device)."""
    N, M = scores.shape
    ids = torch.full((N,), -1, dtype=torch.int64, device=boxes5.device)
    if N == 0:
        return ids
    taken = torch.empty(max(M, 1), dtype=torch.uint8, device=boxes5.device)
    _lib.check(_L().uc_qd_assign(_p(scores), N, M, _p(memo_ids), _p(boxes5[:, 4]), boxes5.stride(0), _f(match_thr), _f(obj_thr), _f(nms_conf_thr),
                                 _p(ids), _p(taken), _S()), "uc_qd_assign")
    return ids


def box_iou(a, b, plus_one=False):
    N, M = a.shape[0], b.shape[0]
    out = torch.empty(N, M, dtype=torch.float32, device=a.device)
    if N and M:
        _lib.check(_L().uc_box_iou(_p(a), a.stride(0), N, _p(b), b.stride(0), M, _p(out), int(plus_one), _S()), "uc_box_iou")
    return out


def aligned_bilinear_add(src, dst, factor):
    _, hs, ws, C = src.shape
    assert dst.shape == (1, hs * factor, ws * factor, C)
    _lib.check(_L().uc_aligned_bilinear_add(_p(src), _nhwc_ld(src), hs, ws, _p(dst), _nhwc_ld(dst), C, factor, _S()), "uc_aligned_bilinear_add")
    return dst


def dynamic_masks(mask_feats, up_masks, dyn_levels, level_hw, ws, n_max, up_rate=4, d_rate=2, strides=(8, 16, 32), soi=(64.0, 128.0, 256.0),
                  out=None, scratch=None):
    """mask_feats fp32 [1,h,w,8]; up_masks fp32 [1,h,w,9*up^2]; dyn_levels: 3 fp32 [1,hk,wk,ld] controller outputs;
    ws: PostWorkspace after postprocess_device.  Returns fp32 [n_max, h*up*d, w*up*d]."""
    _, h, w, _ = mask_feats.shape
    H, W = h * up_rate * d_rate, w * up_rate * d_rate
    if out is None:
        out = torch.zeros(n_max, H, W, dtype=torch.float32, device=mask_feats.device)
    if scratch is None:
        scratch = torch.empty(n_max * h * w * (1 + up_rate * up_rate), dtype=torch.float32, device=mask_feats.device)
    dl = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in dyn_levels])
    hw = (ctypes.c_int * 6)(*[v for pair in level_hw for v in pair])
    st = (ctypes.c_int * 3)(*strides)
    so = (ctypes.c_float * 3)(*soi)
    _lib.check(_L().uc_dynamic_masks(_p(mask_feats), _p(up_masks), h, w, up_rate, d_rate, dl, dyn_levels[0].shape[-1], hw, st, so,
                                     _p(ws.anchors), _p(ws.count), n_max, _p(scratch), _p(out), _S()), "uc_dynamic_masks", 3)
    return out


class MotsRleWorkspace:
    """Device buffers of mots_masks_rle: bit-packed masks, per-row lengths / offsets and the string bytes.  Allocated on first use
    and grown when a frame needs more (the string buffer when the kernel reports that the strings did not fit)."""

    def __init__(self, device, capacity=1 << 16):
        self.dev = torch.device(device)
        self.bits = torch.empty(0, dtype=torch.uint8, device=self.dev)
        self.meta = torch.empty(0, dtype=torch.int64, device=self.dev)
        self.chars = torch.empty(capacity, dtype=torch.uint8, device=self.dev)


def mots_masks_rle(masks, rows, emit, img_h, img_w, thres, scale_factor, ws=None):
    """COCO RLE strings of the MOTS masks of one frame (uc_mots_masks_rle): masks fp32 [n_max, Hin, Win] (device); rows / emit int32
    [K] device tensors (mask rows in ascending track-id order, area-filter flags).  Row k is resized with F.interpolate(scale_factor,
    bilinear, align_corners=False)[:img_h, :img_w], thresholded (> thres) and made overlap free against rows 0..k-1.  Returns the
    strings of the emitted rows, in order; only the lengths and the string bytes are copied to the host."""
    K = rows.numel()
    if K == 0:
        return []
    n_max, Hin, Win = masks.shape
    assert masks.dtype == torch.float32 and masks.is_contiguous() and masks.is_cuda
    assert rows.dtype == torch.int32 and emit.dtype == torch.int32 and emit.numel() == K and rows.is_cuda and emit.is_cuda
    ws = ws or MotsRleWorkspace(masks.device)
    fn = _L().uc_mots_rle_workspace_bytes
    fn.restype = ctypes.c_long
    need = fn(K, Hin, Win, img_h, img_w, ctypes.c_double(scale_factor))
    if need > ws.bits.numel():
        ws.bits = torch.empty(need, dtype=torch.uint8, device=masks.device)
    if ws.meta.numel() < 2 * K + 1:
        ws.meta = torch.empty(2 * K + 1, dtype=torch.int64, device=masks.device)
    while True:
        meta = ws.meta[:2 * K + 1]
        _lib.check(_L().uc_mots_masks_rle(_p(masks), n_max, Hin, Win, _p(rows), _p(emit), K, img_h, img_w, _f(thres), ctypes.c_double(scale_factor),
                                          _p(ws.bits), _l(ws.bits.numel()), _p(meta), _p(meta[K:]), _p(meta[2 * K:]), _p(ws.chars),
                                          _l(ws.chars.numel()), _S()), "uc_mots_masks_rle", 3)
        m = meta.cpu().tolist()
        total = m[2 * K]
        if total <= ws.chars.numel():
            break
        ws.chars = torch.empty(max(total, 2 * ws.chars.numel()), dtype=torch.uint8, device=masks.device)  # run again, never truncate
    data = ws.chars[:total].cpu().numpy().tobytes()
    return [data[m[K + k]:m[K + k] + m[k]].decode("ascii") for k in range(K) if m[k] > 0]
