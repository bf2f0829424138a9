"""Python-side wrappers over the C ABI (include/groma_b200.h).  torch is used only for device memory and the
current stream; every computation below runs in libgroma_b200.so.  CPU tensors are rejected -- there is no fallback."""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence

import torch

from . import lib as _lib

ACT_NONE, ACT_GELU, ACT_RELU, ACT_SWIGLU = 0, 1, 2, 3
GF_OUT_F32, GF_BIAS_ALONG_M, GF_PARTIAL, GF_CONV_ROWS, GF_CONV_COMPACT = 1, 2, 4, 8, 16

LAUNCHES = 0  # number of C-ABI kernel-launching calls made (bench.py reports it)


def _L():
    return _lib.load()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.GromaError("groma_b200 ops need CUDA tensors (no CPU fallback)")
    return t.data_ptr()


def _chk(rc: int, what: str):
    global LAUNCHES
    LAUNCHES += 1
    _lib.check(rc, what)


def _i32_array(vals: Sequence[int]):
    return (ctypes.c_int32 * len(vals))(*vals)


def _bf16(t: torch.Tensor, name: str):
    if t.dtype != torch.bfloat16:
        raise _lib.GromaError(f"{name} must be bfloat16, got {t.dtype}")


def _f32(t: Optional[torch.Tensor], name: str):
    if t is not None and t.dtype != torch.float32:
        raise _lib.GromaError(f"{name} must be float32, got {t.dtype}")


# --------------------------------------------------------------------------------------------- GEMM / conv
def gemm(a: torch.Tensor, w: torch.Tensor, *, bias: Optional[torch.Tensor] = None, act: int = ACT_NONE,
         gamma: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
         out: Optional[torch.Tensor] = None, out_f32: bool = False, block_n: int = 0,
         k: Optional[int] = None) -> torch.Tensor:
    """out[M,N] = epilogue(a[M,K] @ w[N,K]^T).  a, w: 2-D bf16, unit inner stride, row stride % 8 == 0."""
    _bf16(a, "a"); _bf16(w, "w"); _f32(bias, "bias"); _f32(gamma, "gamma")
    assert a.dim() == 2 and w.dim() == 2 and a.stride(1) == 1 and w.stride(1) == 1
    M, K = a.shape if k is None else (a.shape[0], k)
    N = w.shape[0]
    n_out = N // 2 if act == ACT_SWIGLU else N
    if out is None:
        out = torch.empty((M, n_out), dtype=torch.float32 if out_f32 else torch.bfloat16, device=a.device)
    assert out.stride(1) == 1
    flags = GF_OUT_F32 if out.dtype == torch.float32 else 0
    if residual is not None:
        _bf16(residual, "residual")
        assert residual.stride() == out.stride()
    rc = _L().groma_gemm_bf16(_p(a), a.shape[0], a.stride(0), _p(w), w.shape[0], w.stride(0), M, N, K, 1, None,
                              _p(out), out.stride(0), 1, flags, act, _p(bias), _p(gamma), _p(residual), None, 1, 0, 0,
                              block_n, _stream())
    _chk(rc, "groma_gemm_bf16")
    return out


def gemm_qkv_rope(x: torch.Tensor, w_qkv: torch.Tensor, q_out: torch.Tensor, cache_k: torch.Tensor, cache_v: torch.Tensor,
                  cos_t: torch.Tensor, sin_t: torch.Tensor, B: int, T: int, H: int, D: int, pos0: int = 0,
                  block_n: int = 256) -> torch.Tensor:
    """qkv projection + RoPE + KV-cache append in one GEMM launch (`groma_gemm_qkv_rope`): x [B*T, K], w_qkv [3*H*D, K];
    q_out [B*T, H*D]; cache_k/v [B, H, cap, D] (views of the engine's KV arena, unit stride over (cap, D))."""
    _bf16(x, "x"); _bf16(w_qkv, "w_qkv"); _bf16(q_out, "q_out"); _bf16(cache_k, "cache_k"); _bf16(cache_v, "cache_v")
    _f32(cos_t, "cos_t"); _f32(sin_t, "sin_t")
    assert x.shape[0] == B * T and w_qkv.shape[0] == 3 * H * D and q_out.is_contiguous()
    assert cache_k.is_contiguous() and cache_v.is_contiguous() and cache_k.shape[1] == H and cache_k.shape[3] == D
    rc = _L().groma_gemm_qkv_rope(_p(x), x.stride(0), _p(w_qkv), w_qkv.stride(0), B, T, H, D, x.shape[1], _p(q_out),
                                  _p(cache_k), _p(cache_v), _p(cos_t), _p(sin_t), pos0, cache_k.shape[2], block_n, _stream())
    _chk(rc, "groma_gemm_qkv_rope")
    return q_out


def gemm_splitk(a: torch.Tensor, w: torch.Tensor, split_k: int, *, bias=None, act=ACT_NONE, gamma=None, residual=None,
                out: Optional[torch.Tensor] = None, out_f32: bool = False, ws: Optional[torch.Tensor] = None,
                block_n: int = 0) -> torch.Tensor:
    """Split-K GEMM: fp32 partials to a workspace, then the reduce kernel applies the epilogue."""
    _bf16(a, "a"); _bf16(w, "w")
    M, K = a.shape
    N = w.shape[0]
    if ws is None:
        ws = torch.empty((split_k, M, N), dtype=torch.float32, device=a.device)
    rc = _L().groma_gemm_bf16(_p(a), M, a.stride(0), _p(w), N, w.stride(0), M, N, K, 1, None, None, 0, 0, GF_PARTIAL,
                              ACT_NONE, None, None, None, _p(ws), split_k, 0, 0, block_n, _stream())
    _chk(rc, "groma_gemm_bf16(split-k)")
    n_out = N // 2 if act == ACT_SWIGLU else N
    if out is None:
        out = torch.empty((M, n_out), dtype=torch.float32 if out_f32 else torch.bfloat16, device=a.device)
    flags = GF_OUT_F32 if out.dtype == torch.float32 else 0
    rc = _L().groma_splitk_reduce(_p(ws), split_k, M, N, act, flags, _p(bias), _p(gamma), _p(residual), _p(out),
                                  out.stride(0), 1, _stream())
    _chk(rc, "groma_splitk_reduce")
    return out


GF_PDL, GF_PARTIAL_T = 64, 128


def gemm_swap_ab(x: torch.Tensor, w: torch.Tensor, ws: torch.Tensor, split_k: int = 1, block_n: int = 0,
                 pdl: bool = False, transposed: bool = False) -> torch.Tensor:
    """Skinny-M GEMM for decode: computes (w[N,K] @ x[M,K]^T) with the weight as the 128-row MMA operand and the
    M<=256 activation rows as the MMA N dimension; raw fp32 partials land in ws[split][N][M].
    pdl: programmatic dependent launch."""
    _bf16(x, "x"); _bf16(w, "w")
    M, K = x.shape
    N = w.shape[0]
    flags = GF_PARTIAL | (GF_PDL if pdl else 0) | (GF_PARTIAL_T if transposed else 0)
    rc = _L().groma_gemm_bf16(_p(w), N, w.stride(0), _p(x), M, x.stride(0), N, M, K, 1, None, None, 0, 0, flags,
                              ACT_NONE, None, None, None, _p(ws), split_k, 0, 0, block_n, _stream())
    _chk(rc, "groma_gemm_bf16(swap-ab)")
    return ws


def conv3x3_flat(x_pad: torch.Tensor, w_taps: torch.Tensor, n_img: int, hp: int, wp: int, *, bias=None, act=ACT_NONE,
                 out: Optional[torch.Tensor] = None, compact: bool = True, level_rows: Optional[Sequence[int]] = None,
                 block_n: int = 0) -> torch.Tensor:
    """3x3 / pad 1 convolution as a shifted-row GEMM over zero-bordered flat NHWC maps.

    x_pad: [L * n_img*hp*wp, C] bf16 (L stacked input maps, each with its own 9 taps -> the L convs are summed);
    w_taps: [Cout, L*9*C] bf16, tap-major (level, ky, kx, cin).  Output rows: interior pixels only,
    [n_img*(hp-2)*(wp-2), Cout] when compact."""
    _bf16(x_pad, "x_pad"); _bf16(w_taps, "w_taps")
    C = x_pad.shape[1]
    Cout = w_taps.shape[0]
    L = w_taps.shape[1] // (9 * C)
    rows = n_img * hp * wp
    assert x_pad.shape[0] == L * rows
    offs = []
    for lv in range(L):
        for ky in range(3):
            for kx in range(3):
                offs.append(lv * rows + (ky - 1) * wp + (kx - 1))
    m_out = n_img * (hp - 2) * (wp - 2) if compact else rows
    if out is None:
        out = torch.empty((m_out, Cout), dtype=torch.bfloat16, device=x_pad.device)
    flags = GF_CONV_ROWS | (GF_CONV_COMPACT if compact else 0)
    rc = _L().groma_gemm_bf16(_p(x_pad), x_pad.shape[0], x_pad.stride(0), _p(w_taps), Cout, w_taps.stride(0), rows,
                              Cout, C, L * 9, _i32_array(offs), _p(out), out.stride(0), 1, flags, act, _p(bias), None,
                              None, None, 1, hp, wp, block_n, _stream())
    _chk(rc, "groma_gemm_bf16(conv3x3)")
    return out


def splitk_reduce(ws: torch.Tensor, out: torch.Tensor, *, act=ACT_NONE, bias=None, gamma=None, residual=None,
                  bias_along_m: bool = False, ld_m: Optional[int] = None, ld_n: int = 1) -> torch.Tensor:
    splits, M, N = ws.shape
    flags = (GF_OUT_F32 if out.dtype == torch.float32 else 0) | (GF_BIAS_ALONG_M if bias_along_m else 0)
    rc = _L().groma_splitk_reduce(_p(ws), splits, M, N, act, flags, _p(bias), _p(gamma), _p(residual), _p(out),
                                  out.stride(0) if ld_m is None else ld_m, ld_n, _stream())
    _chk(rc, "groma_splitk_reduce")
    return out


# --------------------------------------------------------------------------------------------- attention
def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, causal: bool, scale: float, q_pos0: int = 0,
              kv_len: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None, sk: Optional[int] = None) -> torch.Tensor:
    """q [B,Sq,H,D] (any batch/row strides, unit head/d strides), k/v [B,H,Sk,D] or [B,Sk,H,D] views (strided)."""
    _bf16(q, "q"); _bf16(k, "k"); _bf16(v, "v")
    B, Sq, H, D = q.shape
    assert q.stride(3) == 1 and q.stride(2) == D
    # k, v given as [B, H, Sk, D] logical views
    assert k.shape[0] == B and k.shape[1] == H and k.shape[3] == D and k.stride(3) == 1
    Sk = k.shape[2] if sk is None else sk
    if out is None:
        out = torch.empty((B, Sq, H * D), dtype=torch.bfloat16, device=q.device)
    if kv_len is not None:
        assert kv_len.dtype == torch.int32
    rc = _L().groma_attention(_p(q), q.stride(0), q.stride(1), _p(k), k.stride(0), k.stride(1), k.stride(2), _p(v),
                              v.stride(0), v.stride(1), v.stride(2), _p(out), out.stride(0), out.stride(1), _p(kv_len),
                              B, H, Sq, Sk, D, 1 if causal else 0, q_pos0, float(scale), _stream())
    _chk(rc, "groma_attention")
    return out


def _view2d(t: torch.Tensor, kind: str):
    """Describe a [B, S, H, D] (kind 'bshd') or [B, H, S, D] (kind 'bhsd') strided view as a 2-D row-major matrix for
    groma_attention_tc: returns (ptr tensor, rows, cols, ld, batch_rows, head_rows, head_cols)."""
    if kind == "bshd":
        B, S, H, D = t.shape
        sb, ss, sh, sd = t.stride()
        assert sd == 1 and sh == D and sb == S * ss, "expect rows = b*S + s, cols = h*D + d"
        return t, B * S, H * D, ss, S, 0, D
    B, H, S, D = t.shape
    sb, sh, ss, sd = t.stride()
    assert sd == 1
    if ss == D and sb == H * sh:            # contiguous cache [B, H, cap, D]: rows = (b*H + h)*cap + s
        cap = sh // D
        return t, B * H * cap, D, D, H * cap, cap, 0
    assert sh == D and sb == S * ss, "expect a permuted [B,S,H,D] activation view"
    return t, B * S, H * D, ss, S, 0, D


def attention_tc(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, causal: bool, scale: float, q_pos0: int = 0,
                 kv_len: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None, sk: Optional[int] = None) -> torch.Tensor:
    """tcgen05 flash attention.  q [B,Sq,H,D] view; k, v [B,H,Sk,D] views (KV cache or permuted fused-qkv slices)."""
    _bf16(q, "q"); _bf16(k, "k"); _bf16(v, "v")
    B, Sq, H, D = q.shape
    Sk = k.shape[2] if sk is None else sk
    if out is None:
        out = torch.empty((B, Sq, H * D), dtype=torch.bfloat16, device=q.device)
    qd, kd, vd = _view2d(q, "bshd"), _view2d(k, "bhsd"), _view2d(v, "bhsd")
    rc = _L().groma_attention_tc(_p(qd[0]), qd[1], qd[2], qd[3], qd[4], qd[6],
                                 _p(kd[0]), kd[1], kd[2], kd[3], kd[4], kd[5], kd[6],
                                 _p(vd[0]), vd[1], vd[2], vd[3], vd[4], vd[5], vd[6],
                                 _p(out), out.stride(1), _p(kv_len), B, H, Sq, Sk, D, 1 if causal else 0, q_pos0, float(scale), _stream())
    _chk(rc, "groma_attention_tc")
    return out


def decode_attention(q: torch.Tensor, cache_k: torch.Tensor, cache_v: torch.Tensor, kv_len: torch.Tensor, scale: float,
                     out: torch.Tensor, pdl: bool = False) -> torch.Tensor:
    """q/out [B, H*D] bf16, cache_k/v [B, H, cap, D] contiguous, kv_len int32 [B] on device."""
    _bf16(q, "q")
    B, H, cap, D = cache_k.shape
    assert cache_k.is_contiguous() and cache_v.is_contiguous() and q.is_contiguous() and out.is_contiguous()
    rc = _L().groma_decode_attention(_p(q), _p(cache_k), _p(cache_v), _p(out), _p(kv_len), B, H, D, cap, float(scale), 1 if pdl else 0, _stream())
    _chk(rc, "groma_decode_attention")
    return out


# --------------------------------------------------------------------------------------------- norms
def rmsnorm(x: torch.Tensor, w: torch.Tensor, eps: float, *, residual: Optional[torch.Tensor] = None,
            h_out: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _bf16(x, "x"); _f32(w, "w")
    assert x.is_contiguous()
    dim = x.shape[-1]
    rows = x.numel() // dim
    if out is None:
        out = torch.empty_like(x)
    rc = _L().groma_rmsnorm(_p(x), _p(residual), _p(w), _p(out), _p(h_out), rows, dim, float(eps), _stream())
    _chk(rc, "groma_rmsnorm")
    return out


def layernorm(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, eps: float, *, residual: Optional[torch.Tensor] = None,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _bf16(x, "x"); _f32(w, "w"); _f32(b, "b")
    dim = x.shape[-1]
    x2 = x.reshape(-1, dim) if x.is_contiguous() else x
    assert x2.dim() == 2 and x2.stride(1) == 1
    rows = x2.shape[0]
    if out is None:
        out = torch.empty((rows, dim), dtype=torch.bfloat16, device=x.device)
    o2 = out.reshape(-1, dim) if out.is_contiguous() else out
    if residual is not None:
        assert residual.is_contiguous() and x2.stride(0) == dim
    rc = _L().groma_layernorm(_p(x2), _p(residual), _p(w), _p(b), _p(o2), rows, dim, float(eps), x2.stride(0),
                              o2.stride(0), _stream())
    _chk(rc, "groma_layernorm")
    return out.reshape(x.shape) if out.numel() == x.numel() else out


def groupnorm_relu(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, groups: int, eps: float, n_img: int,
                   out: Optional[torch.Tensor] = None, chunks: int = 0) -> torch.Tensor:
    """x: [n_img * P, C] bf16 (NHWC pixels)."""
    _bf16(x, "x")
    C = x.shape[-1]
    P = x.shape[0] // n_img
    if chunks <= 0:
        chunks = max(1, min(64, P // 256))
    part = torch.empty((n_img * chunks * groups * 2,), dtype=torch.float32, device=x.device)
    stats = torch.empty((n_img * groups * 2,), dtype=torch.float32, device=x.device)
    if out is None:
        out = torch.empty_like(x)
    rc = _L().groma_groupnorm_relu(_p(x), _p(gamma), _p(beta), _p(out), _p(part), _p(stats), n_img, P, C, groups,
                                   float(eps), chunks, _stream())
    _chk(rc, "groma_groupnorm_relu")
    return out


def groupnorm_stats(x: torch.Tensor, groups: int, eps: float, n_img: int, chunks: int = 0) -> torch.Tensor:
    """x: [n_img * P, C] bf16 -> fp32 stats [n_img, groups, 2] (mean, rstd); the first half of groupnorm_relu."""
    _bf16(x, "x")
    C = x.shape[-1]
    P = x.shape[0] // n_img
    if chunks <= 0:
        chunks = max(1, min(64, P // 256))
    part = torch.empty((n_img * chunks * groups * 2,), dtype=torch.float32, device=x.device)
    stats = torch.empty((n_img, groups, 2), dtype=torch.float32, device=x.device)
    _chk(_L().groma_groupnorm_stats(_p(x), _p(part), _p(stats), n_img, P, C, groups, float(eps), chunks, _stream()), "groma_groupnorm_stats")
    return stats


def groupnorm_apply_relu(x: torch.Tensor, stats: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, groups: int, n_img: int,
                         out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """relu((x - mean) * rstd * gamma + beta) with the statistics of groupnorm_stats; the second half of groupnorm_relu."""
    _bf16(x, "x"); _f32(stats, "stats")
    C = x.shape[-1]
    P = x.shape[0] // n_img
    if out is None:
        out = torch.empty_like(x)
    _chk(_L().groma_groupnorm_apply_relu(_p(x), _p(stats), _p(gamma), _p(beta), _p(out), n_img, P, C, groups, _stream()),
         "groma_groupnorm_apply_relu")
    return out


# --------------------------------------------------------------------------------------------- detection ops
def msda(value: torch.Tensor, proj: torch.Tensor, ref: torch.Tensor, level_hw: Sequence[Sequence[int]],
         n_heads: int, n_points: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _bf16(value, "value"); _f32(proj, "proj"); _f32(ref, "ref")
    B, S = value.shape[0], value.shape[1]
    Q = ref.shape[1]
    L = len(level_hw)
    hw = [int(v) for pair in level_hw for v in pair]
    starts, acc = [], 0
    for h, w in level_hw:
        starts.append(acc); acc += h * w
    assert acc == S and value.is_contiguous() and proj.is_contiguous() and ref.is_contiguous()
    if out is None:
        out = torch.empty((B, Q, n_heads * 32), dtype=torch.bfloat16, device=value.device)
    rc = _L().groma_msda_forward(_p(value), _p(proj), _p(ref), _p(out), B, Q, S, n_heads, L, n_points, ref.shape[-1],
                                 _i32_array(hw), _i32_array(starts), _stream())
    _chk(rc, "groma_msda_forward")
    return out


def roi_align(feat: torch.Tensor, rois: torch.Tensor, out_size: int, spatial_scale: float, sampling_ratio: int,
              aligned: bool = True, pad: bool = False, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """feat [N,H,W,C] bf16 NHWC; rois [K,5] fp32 -> [K, out+2p, out+2p, C] bf16."""
    _bf16(feat, "feat"); _f32(rois, "rois")
    N, H, W, C = feat.shape
    K = rois.shape[0]
    p = 1 if pad else 0
    if out is None:
        out = torch.empty((K, out_size + 2 * p, out_size + 2 * p, C), dtype=torch.bfloat16, device=feat.device)
    assert feat.is_contiguous() and rois.is_contiguous() and out.is_contiguous()
    rc = _L().groma_roi_align_forward(_p(feat), _p(rois), _p(out), K, C, H, W, out_size, out_size, float(spatial_scale),
                                      sampling_ratio, 1 if aligned else 0, p, _stream())
    _chk(rc, "groma_roi_align_forward")
    return out


def nms_batched(boxes: torch.Tensor, scores: torch.Tensor, iou_thr: float, score_thr: float, max_num: int,
                counts: Optional[torch.Tensor] = None, offset: int = 0):
    """boxes [B,N,4] xyxy fp32, scores [B,N] -> (keep int64 [B,max_out], num_keep int32 [B], argmax int32 [B])."""
    _f32(boxes, "boxes"); _f32(scores, "scores")
    B, N = scores.shape
    max_out = max_num if max_num > 0 else N
    keep = torch.empty((B, max_out), dtype=torch.int64, device=boxes.device)
    num = torch.empty((B,), dtype=torch.int32, device=boxes.device)
    amax = torch.empty((B,), dtype=torch.int32, device=boxes.device)
    assert boxes.is_contiguous() and scores.is_contiguous()
    rc = _L().groma_nms_batched(_p(boxes), _p(scores), _p(counts), B, N, float(iou_thr), float(score_thr), offset,
                                max_num, _p(keep), max_out, _p(num), _p(amax), _stream())
    _chk(rc, "groma_nms_batched")
    return keep, num, amax


def topk_desc(scores: torch.Tensor, k: int) -> torch.Tensor:
    _f32(scores, "scores")
    B, N = scores.shape
    out = torch.empty((B, k), dtype=torch.int64, device=scores.device)
    rc = _L().groma_topk_desc(_p(scores), scores.stride(0), B, N, k, _p(out), _stream())
    _chk(rc, "groma_topk_desc")
    return out


def ddetr_select(delta: torch.Tensor, proposals: torch.Tensor, topk: torch.Tensor, num_pos_feats: int):
    B, S, _ = delta.shape
    k = topk.shape[1]
    ref = torch.empty((B, k, 4), dtype=torch.float32, device=delta.device)
    pos = torch.empty((B, k, 4 * num_pos_feats), dtype=torch.bfloat16, device=delta.device)
    rc = _L().groma_ddetr_select(_p(delta), _p(proposals), _p(topk), _p(ref), _p(pos), B, S, k, num_pos_feats, _stream())
    _chk(rc, "groma_ddetr_select")
    return ref, pos


def ddetr_finalize(d4, d5, ref0, coco, sa1b, pred_cxcywh, pred_xyxy, score):
    B, Q = ref0.shape[0], ref0.shape[1]
    rc = _L().groma_ddetr_finalize(_p(d4), _p(d5), _p(ref0), _p(coco), _p(sa1b), _p(pred_cxcywh), _p(pred_xyxy),
                                   _p(score), B, Q, pred_cxcywh.shape[1], score.shape[1], _stream())
    _chk(rc, "groma_ddetr_finalize")


def mask_rows(x: torch.Tensor, valid_u8: torch.Tensor):
    B, S, D = x.shape
    _chk(_L().groma_mask_rows(_p(x), _p(valid_u8), B, S, D, _stream()), "groma_mask_rows")
    return x


# --------------------------------------------------------------------------------------------- resampling
def upsample_coords(tokens: torch.Tensor, skip: int, g: int, Ho: int, Wo: int, ld: int, xs: torch.Tensor,
                    ys: torch.Tensor) -> torch.Tensor:
    B, _, C = tokens.shape
    out = torch.empty((B, Ho, Wo, ld), dtype=torch.bfloat16, device=tokens.device)
    rc = _L().groma_upsample_coords(_p(tokens), skip, g, C, _p(out), B, Ho, Wo, ld, _p(xs), _p(ys), _stream())
    _chk(rc, "groma_upsample_coords")
    return out


def fuse_shuffle(tar: torch.Tensor, top: torch.Tensor, down: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """tar/top/down: [B,H,W,C] compact NHWC; returns zero-bordered [B,H+2,W+2,C]."""
    B, Ht, Wt, C = tar.shape
    if out is None:
        out = torch.empty((B, Ht + 2, Wt + 2, C), dtype=torch.bfloat16, device=tar.device)
    rc = _L().groma_fuse_shuffle(_p(tar), _p(top), _p(down), _p(out), B, C, Ht, Wt, top.shape[1], top.shape[2],
                                 down.shape[1], down.shape[2], _stream())
    _chk(rc, "groma_fuse_shuffle")
    return out


def fuse_shuffle_gn(tar: torch.Tensor, top: torch.Tensor, down: torch.Tensor, st_tar: torch.Tensor, st_top: torch.Tensor,
                    st_down: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, groups: int,
                    out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """fuse_shuffle over RAW conv outputs: relu(GroupNorm) (per-level stats from groupnorm_stats, shared gamma / beta) is applied
    to every tap; bit-identical to groupnorm_apply_relu on each map followed by fuse_shuffle."""
    B, Ht, Wt, C = tar.shape
    for t in (st_tar, st_top, st_down):
        _f32(t, "stats")
    if out is None:
        out = torch.empty((B, Ht + 2, Wt + 2, C), dtype=torch.bfloat16, device=tar.device)
    rc = _L().groma_fuse_shuffle_gn(_p(tar), _p(top), _p(down), _p(out), B, C, Ht, Wt, top.shape[1], top.shape[2],
                                    down.shape[1], down.shape[2], _p(st_tar), _p(st_top), _p(st_down), _p(gamma), _p(beta),
                                    groups, _stream())
    _chk(rc, "groma_fuse_shuffle_gn")
    return out


# --------------------------------------------------------------------------------------------- ViT / token plumbing
def vit_patchify(images: torch.Tensor, ld: int) -> torch.Tensor:
    _f32(images, "images")
    B, _, S, _ = images.shape
    out = torch.empty((B * (S // 14) ** 2, ld), dtype=torch.bfloat16, device=images.device)
    _chk(_L().groma_vit_patchify(_p(images.contiguous()), _p(out), B, S, ld, _stream()), "groma_vit_patchify")
    return out


def vit_embed(patch: torch.Tensor, cls: torch.Tensor, pos: torch.Tensor, B: int, NP: int) -> torch.Tensor:
    C = patch.shape[-1]
    out = torch.empty((B, NP + 1, C), dtype=torch.bfloat16, device=patch.device)
    _chk(_L().groma_vit_embed(_p(patch), _p(cls), _p(pos), _p(out), B, NP, C, _stream()), "groma_vit_embed")
    return out


def mean_tokens(ts: Sequence[torch.Tensor], skip: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    B, T, C = ts[0].shape
    if out is None:
        out = torch.empty((B, T - skip, C), dtype=torch.bfloat16, device=ts[0].device)
    ptrs = [_p(t) for t in ts] + [None] * (4 - len(ts))
    _chk(_L().groma_mean_tokens(ptrs[0], ptrs[1], ptrs[2], ptrs[3], len(ts), _p(out), B, T, C, skip, _stream()),
         "groma_mean_tokens")
    return out


def space_to_depth(tokens: torch.Tensor, g: int) -> torch.Tensor:
    B, _, C = tokens.shape
    out = torch.empty((B, (g // 2) ** 2, 4 * C), dtype=torch.bfloat16, device=tokens.device)
    _chk(_L().groma_space_to_depth(_p(tokens), _p(out), B, g, C, _stream()), "groma_space_to_depth")
    return out


def gather_rows(idx: torch.Tensor, t0: torch.Tensor, t1: Optional[torch.Tensor] = None, split: int = 0,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
    assert idx.dtype == torch.int64 and idx.is_contiguous()
    n, D = idx.numel(), t0.shape[-1]
    if out is None:
        out = torch.empty((n, D), dtype=torch.bfloat16, device=t0.device)
    _chk(_L().groma_gather_rows(_p(idx), _p(t0), _p(t1), split if t1 is not None else (1 << 62), _p(out), n, D,
                                _stream()), "groma_gather_rows")
    return out


def scatter_rows(idx: torch.Tensor, src: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    assert idx.dtype == torch.int64 and idx.is_contiguous() and src.is_contiguous()
    n, D = idx.numel(), src.shape[-1]
    _chk(_L().groma_scatter_rows(_p(idx), _p(src), _p(out), n, D, _stream()), "groma_scatter_rows")
    return out


def add(a: torch.Tensor, b: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    if out is None:
        out = torch.empty_like(a)
    _chk(_L().groma_add(_p(a), _p(b), _p(out), a.numel(), _stream()), "groma_add")
    return out


def add_bcast(a: torch.Tensor, b: torch.Tensor, period: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    D = a.shape[-1]
    if out is None:
        out = torch.empty_like(a)
    _chk(_L().groma_add_bcast(_p(a), _p(b), _p(out), a.numel() // D, period, D, _stream()), "groma_add_bcast")
    return out


def rope_kv(qkv: torch.Tensor, q_out: torch.Tensor, cache_k: torch.Tensor, cache_v: torch.Tensor, cos_t: torch.Tensor,
            sin_t: torch.Tensor, B: int, T: int, H: int, D: int, pos0: int, pos_ptr: Optional[torch.Tensor] = None):
    _chk(_L().groma_rope_kv(_p(qkv), _p(q_out), _p(cache_k), _p(cache_v), _p(cos_t), _p(sin_t), B, T, H, D, pos0,
                            _p(pos_ptr), cache_k.shape[2], _stream()), "groma_rope_kv")


def argmax(logits: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _f32(logits, "logits")
    rows, V = logits.shape
    if out is None:
        out = torch.empty((rows,), dtype=torch.int64, device=logits.device)
    _chk(_L().groma_argmax(_p(logits), _p(out), rows, V, logits.stride(0), _stream()), "groma_argmax")
    return out


def to_bf16(x: torch.Tensor) -> torch.Tensor:
    _f32(x, "x")
    out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    _chk(_L().groma_cast_f32_bf16(_p(x.contiguous()), _p(out), x.numel(), _stream()), "groma_cast_f32_bf16")
    return out


def linear_smallk(x: torch.Tensor, w: torch.Tensor, b: Optional[torch.Tensor], relu: bool) -> torch.Tensor:
    _f32(x, "x"); _f32(w, "w"); _f32(b, "b")
    M, K = x.shape
    N = w.shape[0]
    out = torch.empty((M, N), dtype=torch.bfloat16, device=x.device)
    _chk(_L().groma_linear_smallk(_p(x.contiguous()), _p(w), _p(b), _p(out), M, N, K, 1 if relu else 0, _stream()),
         "groma_linear_smallk")
    return out


def decode_advance(pos: torch.Tensor, kv_len: torch.Tensor):
    _chk(_L().groma_decode_advance(_p(pos), _p(kv_len), kv_len.numel(), _stream()), "groma_decode_advance")


def decode_reduce_norm(ws: torch.Tensor, x: torch.Tensor, w: torch.Tensor, y: torch.Tensor, eps: float, pdl: bool = True):
    """ws [S, B, N] fp32 token-major partials; x [B, N] bf16 residual stream (updated in place); y = RMSNorm(x) * w."""
    S, B, N = ws.shape
    _chk(_L().groma_decode_reduce_norm(_p(ws), S, B, N, _p(x), _p(w), _p(y), float(eps), 1 if pdl else 0, _stream()),
         "groma_decode_reduce_norm")


def decode_reduce_swiglu(ws: torch.Tensor, out: torch.Tensor, pdl: bool = True):
    S, B, N = ws.shape
    _chk(_L().groma_decode_reduce_swiglu(_p(ws), S, B, N, _p(out), 1 if pdl else 0, _stream()), "groma_decode_reduce_swiglu")


def decode_head_argmax(ws: torch.Tensor, logits: torch.Tensor, ids: torch.Tensor, pos: torch.Tensor, kv_len: torch.Tensor,
                       pdl: bool = False) -> torch.Tensor:
    """ws [S, B, V] fp32 head partials -> logits [B, V] fp32, ids [B] int64 (greedy), pos / kv_len advanced: one launch."""
    S, B, V = ws.shape
    _f32(ws, "ws"); _f32(logits, "logits")
    assert logits.shape == (B, V) and logits.is_contiguous() and ids.dtype == torch.int64 and ids.numel() == B
    assert pos.dtype == torch.int32 and kv_len.dtype == torch.int32 and kv_len.numel() == B
    _chk(_L().groma_decode_head_argmax(_p(ws), S, B, V, _p(logits), _p(ids), _p(pos), _p(kv_len), 1 if pdl else 0, _stream()),
         "groma_decode_head_argmax")
    return logits


def decode_reduce_rope_kv(ws: torch.Tensor, q_out: torch.Tensor, cache_k: torch.Tensor, cache_v: torch.Tensor, cos_t: torch.Tensor,
                          sin_t: torch.Tensor, pos_ptr: torch.Tensor, H: int, D: int, pdl: bool = True):
    S, B, N = ws.shape
    assert N == 3 * H * D
    _chk(_L().groma_decode_reduce_rope_kv(_p(ws), S, B, H, D, _p(q_out), _p(cache_k), _p(cache_v), _p(cos_t), _p(sin_t),
                                          _p(pos_ptr), cache_k.shape[2], 1 if pdl else 0, _stream()), "groma_decode_reduce_rope_kv")


def decode_rope_attention(ws: torch.Tensor, cache_k: torch.Tensor, cache_v: torch.Tensor, kv_len: torch.Tensor, pos_ptr: torch.Tensor,
                          cos_t: torch.Tensor, sin_t: torch.Tensor, scale: float, out: torch.Tensor, pdl: bool = True) -> torch.Tensor:
    """decode_reduce_rope_kv + decode_attention in one launch: ws [S, B, 3*H*D] fp32 qkv partials; the new K/V row is appended
    to cache_k/v [B, H, cap, 128] at *pos_ptr; out [B, H*D] bf16."""
    S, B, N = ws.shape
    _, H, cap, D = cache_k.shape
    assert N == 3 * H * D and cache_k.is_contiguous() and cache_v.is_contiguous() and out.is_contiguous() and ws.is_contiguous()
    _chk(_L().groma_decode_rope_attention(_p(ws), S, _p(cache_k), _p(cache_v), _p(out), _p(kv_len), _p(pos_ptr), _p(cos_t), _p(sin_t),
                                          B, H, D, cap, float(scale), 1 if pdl else 0, _stream()), "groma_decode_rope_attention")
    return out


# ----------------------------------------------------------------------------------------------------------------------
# image preprocessing (SURVEY §8f N3)
PREPROCESS_KMAX = 64


def preprocess_image(img: torch.Tensor, lut: torch.Tensor, out_size: int, out_f32: Optional[torch.Tensor] = None,
                     out_u8: Optional[torch.Tensor] = None) -> None:
    """Pillow-exact bicubic resize of one uint8 HWC RGB cuda image to out_size^2, then the byte->float32 table `lut` [3,256]
    (rescale + normalize) into out_f32 [3,S,S]; out_u8 [S,S,3] receives the resized bytes.  See include/groma_b200.h."""
    if img.dtype != torch.uint8 or img.dim() != 3 or img.shape[2] != 3 or not img.is_cuda or img.stride(2) != 1 or img.stride(1) != 3:
        raise ValueError("img must be a cuda uint8 [H, W, 3] tensor with packed RGB pixels")
    H, W = int(img.shape[0]), int(img.shape[1])
    tmp = torch.empty((H, out_size, 3), dtype=torch.uint8, device=img.device)
    coef = torch.empty((2 * out_size * (2 + PREPROCESS_KMAX),), dtype=torch.int32, device=img.device)
    if out_f32 is not None and (out_f32.dtype != torch.float32 or not out_f32.is_contiguous() or out_f32.numel() != 3 * out_size * out_size):
        raise ValueError("out_f32 must be contiguous float32 [3, S, S]")
    if out_u8 is not None and (out_u8.dtype != torch.uint8 or not out_u8.is_contiguous() or out_u8.numel() != 3 * out_size * out_size):
        raise ValueError("out_u8 must be contiguous uint8 [S, S, 3]")
    if out_f32 is not None and (lut is None or lut.dtype != torch.float32 or lut.numel() != 768 or not lut.is_contiguous()):
        raise ValueError("lut must be contiguous float32 [3, 256]")
    rc = _L().groma_preprocess_image(_p(img), H, W, img.stride(0), _p(lut), out_size, _p(tmp), _p(coef), _p(out_f32), _p(out_u8),
                                     _stream())
    _chk(rc, "groma_preprocess_image")
