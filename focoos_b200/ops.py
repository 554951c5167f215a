"""Operator surface of focoos_b200: torch tensors in, hand-written sm_100a kernels underneath.

Every function below validates/allocates on the host and then calls ONE entry point of the C ABI
declared in `include/focoos_b200.h` (loaded with ctypes from `focoos_b200/lib/libfocoos_b200.so`,
built in-tree by `focoos_b200/csrc/build.py`).  The same functions are registered as PyTorch custom
ops in the `focoos_b200::` namespace (see `_register_torch_ops`).

There is NO CPU or eager-PyTorch fallback: without the compiled library, or with non-CUDA tensors,
every op raises.  (`_backend` exists so that `tests/` can exercise the host-side orchestration on a
GPU-less machine by installing the reference backend from `oracle/ops_ref.py`; product code never
sets it.)

Layout: activations are NHWC; a tensor argument may be a channel-slice view of a wider NHWC buffer
(`t[..., a:b]`): only the last-dim stride must be 1, the pixel pitch is taken from `stride(-2)`.
"""
from __future__ import annotations

import ctypes
import os
import re
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

F32, F16, F16PAIR = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_SILU, ACT_GELU = 0, 1, 2, 3
ACT = {None: 0, "none": 0, "relu": 1, "silu": 2, "gelu": 3}
ALGO_AUTO, ALGO_SIMT, ALGO_TCGEN05, ALGO_TCGEN05_SPLIT3 = 0, 1, 2, 3

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libfocoos_b200.so")
_lib = None
_backend = None  # tests only


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.float16:
        return F16
    raise TypeError(f"focoos_b200: unsupported dtype {t.dtype}")


def torch_dtype(code: int) -> torch.dtype:
    return torch.float32 if code == F32 else torch.float16


_HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "focoos_b200.h")
_RESTYPES = {"int": ctypes.c_int, "int64_t": ctypes.c_int64, "const char*": ctypes.c_char_p}
_ARGTYPES = {"int": ctypes.c_int, "int64_t": ctypes.c_int64, "float": ctypes.c_float}  # and every pointer: c_void_p


def _ctype(table, decl: str, fn: str):
    if decl in table:
        return table[decl]
    if table is _ARGTYPES and "*" in decl:
        return ctypes.c_void_p
    raise RuntimeError(f"focoos_b200: {fn} in {_HEADER} uses the type `{decl}`, which the ctypes binding does not map")


def _prototypes():
    """{name: (restype, argtypes)} of every `ret fb200_name(params);` declared in include/focoos_b200.h"""
    text = re.sub(r"/\*.*?\*/", "", open(_HEADER).read(), flags=re.S)
    protos = {}
    for ret, name, params in re.findall(r"^\s*([\w ]+\**)\s*\b(fb200_\w+)\s*\(([^)]*)\)\s*;", text, flags=re.M):
        params = [] if params.strip() in ("", "void") else [re.sub(r"\s*\b\w+$", "", p.strip()) for p in params.split(",")]
        protos[name] = (_ctype(_RESTYPES, ret.strip(), name), [_ctype(_ARGTYPES, p, name) for p in params])
    return protos


_PROTOTYPES = _prototypes()
EXPORTED_SYMBOLS = tuple(sorted(_PROTOTYPES))


def load_library():
    """Load the C-ABI library with the prototypes of include/focoos_b200.h; raises if it has not been built (no silent fallback)
    or does not export a declared entry point."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(
            f"focoos_b200: CUDA library not found at {_LIB_PATH}. Build it with "
            "`python -m focoos_b200.csrc.build` (or `__graft_entry__.build()`); there is no CPU fallback."
        )
    lib = ctypes.CDLL(_LIB_PATH)
    for name, (restype, argtypes) in _PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
    _lib = lib
    return lib

_launch_count = 0
_trace = None       # profiling aid (tools/layer_roofline.py): list of [symbol, note, start_event, end_event]
_trace_note = []


def enable_trace(on: bool = True):
    global _trace
    _trace = [] if on else None
    return _trace


def launch_count() -> int:
    """Number of kernels launched through this module since import (for bench.py's `gpu_launches`)."""
    return _launch_count


def _check(rc: int, what: str):
    if rc != 0:
        msg = load_library().fb200_last_error()
        raise RuntimeError(f"focoos_b200.{what} failed ({rc}): {msg.decode() if msg else '?'}")


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _ws(nbytes: int, device):
    return torch.empty(int(nbytes), dtype=torch.uint8, device=device)


def _pitch(t: torch.Tensor, free_batch_stride: bool = False) -> int:
    """pixel pitch (elements) of an NHWC / [.., L, C] tensor that may be a channel slice of a wider buffer."""
    assert t.stride(-1) == 1, "last dim must be contiguous"
    p = t.stride(-2) if t.dim() >= 2 else t.shape[-1]
    # outer dims must be dense w.r.t. the pitch
    exp = p
    for d in range(t.dim() - 2, -1, -1):
        if t.shape[d] != 1 and not (d == 0 and free_batch_stride and t.dim() == 4):
            assert t.stride(d) == exp, f"unsupported view strides {t.stride()} for shape {tuple(t.shape)}"
        exp *= t.shape[d]
    return p


def _batch_stride(t: torch.Tensor) -> int:
    return t.stride(0) if (t.dim() == 4 and t.shape[0] > 1) else 0


class CudaBackend:
    """Thin marshalling layer: tensors -> raw pointers/sizes -> C ABI."""

    def __init__(self):
        self.lib = load_library()

    @staticmethod
    def _cuda(*ts):
        for t in ts:
            if t is not None and not t.is_cuda:
                raise RuntimeError("focoos_b200: tensors must live on a CUDA device (no CPU fallback)")

    def _call(self, name, *args):
        global _launch_count
        _launch_count += 1
        if _trace is None:
            _check(getattr(self.lib, name)(*args), name)
            return
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _check(getattr(self.lib, name)(*args), name)
        e1.record()
        _trace.append([name, _trace_note.pop() if _trace_note else "", e0, e1])

    def stem_conv(self, img, w, scale, bias, mean, std, act, out):
        self._cuda(img, w, out.buf if isinstance(out, Pair) else out)
        u8 = img.dtype == torch.uint8
        B, H, W = (img.shape[0], img.shape[1], img.shape[2]) if u8 else (img.shape[0], img.shape[2], img.shape[3])
        m = (ctypes.c_float * 3)(*mean)
        s = (ctypes.c_float * 3)(*std)
        if isinstance(out, Pair):
            self._call("fb200_stem_conv3x3s2_u8" if u8 else "fb200_stem_conv3x3s2", _p(img), B, H, W, _p(w), _p(scale), _p(bias), m, s, act, _p(out.buf), F16PAIR, out.C, _stream())
            return
        self._call("fb200_stem_conv3x3s2_u8" if u8 else "fb200_stem_conv3x3s2", _p(img), B, H, W, _p(w), _p(scale), _p(bias), m, s, act, _p(out), _dt(out), out.shape[-1], _stream())

    def conv2d(self, x, w, scale, bias, stride, pad, act, residual, out, algo):
        self._cuda(x, w, out)
        B, H, W, Cin = x.shape
        Cout, KH, KW, _ = w.shape
        if _trace is not None:
            _trace_note.append(dict(op="conv", B=B, H=H, W=W, Cin=Cin, Cout=Cout, k=KH, stride=stride, res=residual is not None, xdt=str(x.dtype)[6:], odt=str(out.dtype)[6:], algo=algo))
        self._call("fb200_conv2d", _p(x), _dt(x), B, H, W, Cin, _pitch(x), _p(w), KH, KW, stride, pad, _p(scale), _p(bias), _p(residual),
                   0 if residual is None else _pitch(residual), act, _p(out), _dt(out), _pitch(out, True), _batch_stride(out), Cout, algo, _stream())

    def conv2d_per_image(self, x, w, act, out, algo):
        self._cuda(x, w, out)
        B, H, W, Cin = x.shape
        _, Cout, KH, KW, _ = w.shape
        self._call("fb200_conv2d_per_image_weights", _p(x), _dt(x), B, H, W, Cin, _pitch(x), _p(w), w.stride(0), KH, KW, 1, (KH - 1) // 2, None, None, act,
                   _p(out), _dt(out), _pitch(out, True), Cout, algo, _stream())

    def linear_rowmax(self, x2d, w, bias, out):
        self._cuda(x2d, w, out)
        self._call("fb200_linear_rowmax", _p(x2d), x2d.shape[0], x2d.shape[1], x2d.stride(0), _p(w), _p(bias), w.shape[0], _p(out), _stream())

    def conv2d_pair(self, x, w3, scale, bias, stride, pad, act, residual, out):
        """x / residual / out: `Pair` (hi + lo fp16 planes) - residual and out may also be plain fp32 tensors (both, or neither)"""
        out_pair = isinstance(out, Pair)
        xh = x.hi
        self._cuda(xh, w3, out.hi if out_pair else out)
        B, H, W, C = xh.shape
        Cout, KH, KW, _ = w3.shape
        oh = out.hi if out_pair else out
        rh = None if residual is None else (residual.hi if out_pair else residual)
        if _trace is not None:
            _trace_note.append(dict(op="conv", B=B, H=H, W=W, Cin=C, Cout=Cout, k=KH, stride=stride, res=residual is not None, xdt="pair", odt="pair" if out_pair else "float32", algo=3))
        self._call("fb200_conv2d_pair", _p(xh), B, H, W, C, _pitch(xh), x.lo_off, _p(w3), KH, KW, stride, pad, _p(scale), _p(bias), _p(rh),
                   0 if rh is None else _pitch(rh), residual.lo_off if (out_pair and residual is not None) else 0, act, _p(oh), F16PAIR if out_pair else F32,
                   _pitch(oh, True), out.lo_off if out_pair else 0, _batch_stride(oh), Cout, _stream())

    def image_resize(self, images, out):
        self._cuda(images, out)
        u8 = images.dtype == torch.uint8
        B = images.shape[0]
        H, W = (images.shape[1], images.shape[2]) if u8 else (images.shape[2], images.shape[3])
        self._call("fb200_image_resize", _p(images), 1 if u8 else 0, B, H, W, _p(out), out.shape[2], out.shape[3], _stream())

    def pair_pool(self, mode, x, out):
        xh, oh = x.hi, out.hi
        self._cuda(xh, oh)
        B, H, W, C = xh.shape
        self._call("fb200_pair_pool", mode, _p(xh), x.lo_off, _pitch(xh), B, H, W, C, _p(oh), out.lo_off, _pitch(oh), oh.shape[1], oh.shape[2], _stream())

    def linear_rowmax_pair(self, xp, w3, bias, out):
        xh = xp.hi
        self._cuda(xh, w3, out)
        M = xh.numel() // xh.shape[-1]
        self._call("fb200_linear_rowmax_pair", _p(xh), M, xh.shape[-1], _pitch(xh), xp.lo_off, _p(w3), _p(bias), w3.shape[0], _p(out), _stream())

    def split_pair(self, x, out):
        self._cuda(x, out)
        C = x.shape[-1]
        self._call("fb200_split_f32_pair", _p(x), x.numel() // C, C, _pitch(x), _p(out), _stream())

    def maxpool3x3s2(self, x, out):
        self._cuda(x, out)
        B, H, W, C = x.shape
        self._call("fb200_maxpool3x3s2", _p(x), _dt(x), B, H, W, C, _p(out), _stream())

    def avgpool2x2(self, x, out):
        self._cuda(x, out)
        B, H, W, C = x.shape
        self._call("fb200_avgpool2x2_ceil", _p(x), _dt(x), B, H, W, C, _p(out), _stream())

    def resize_bilinear(self, x, out):
        self._cuda(x, out)
        B, H, W, C = x.shape
        self._call("fb200_resize_bilinear", _p(x), _dt(x), B, H, W, C, _pitch(x), _p(out), out.shape[1], out.shape[2], _pitch(out), _stream())

    def add(self, a, b, out):
        self._cuda(a, b, out)
        C = a.shape[-1]
        self._call("fb200_add", _p(a), _p(b), _p(out), _dt(a), a.numel() // C, b.numel() // C, C, _stream())

    def layernorm(self, x, res, gamma, beta, out, eps):
        self._cuda(x, out)
        C = x.shape[-1]
        self._call("fb200_layernorm", _p(x), _p(res), _p(gamma), _p(beta), _p(out), _dt(x), x.numel() // C, C, eps, _stream())

    def attention(self, q, k, v, out, heads, scale, split=False):
        self._cuda(q, k, v)
        B, Lq, C = q.shape
        if split and q.dtype == torch.float32:
            pair = isinstance(out, Pair)
            o = out.buf if pair else out
            self._cuda(o)
            self._call("fb200_attention_split", _p(q), _pitch(q), _p(k), _pitch(k), _p(v), _pitch(v), _p(o), F16PAIR if pair else F32, _pitch(o), B, Lq, k.shape[1],
                       heads, C // heads, scale, _stream())
            return
        self._call("fb200_attention", _p(q), _pitch(q), _p(k), _pitch(k), _p(v), _pitch(v), _p(out), _pitch(out), _dt(q), B, Lq, k.shape[1],
                   heads, C // heads, scale, _stream())

    def msda(self, value, oa, ref, shapes, P, heads, out):
        self._cuda(value, oa, ref)
        B, S, _ = value.shape
        Q = oa.shape[1]
        flat = [int(v) for hw in shapes for v in hw]
        sh = (ctypes.c_int * len(flat))(*flat)
        pair = isinstance(out, Pair)
        o = out.buf if pair else out
        self._cuda(o)
        self._call("fb200_msda", _p(value), _dt(value), _pitch(value), _p(oa), _dt(oa), _pitch(oa), _p(ref), sh, len(shapes), P, B, S, Q, heads,
                   _p(o), F16PAIR if pair else _dt(o), _pitch(o), _stream())

    def layernorm_ex(self, x, res, gather, valid, fill, gamma, beta, eps, M, out_f32, out_pair, pos, out_pair_pos):
        """x [.., C] fp32 rows (last-dim pitch); gather int32 [B, K] or None; valid uint8 [S] or None; outputs: fp32 tensor / Pair / Pair (each optional)"""
        self._cuda(x, gamma, beta)
        C = x.shape[-1]
        S = 0 if valid is None else valid.numel()
        if gather is not None and valid is None:
            S = x.shape[-2]
        self._call("fb200_layernorm_ex", _p(x), _pitch(x), _p(res), _p(gather), 0 if gather is None else gather.shape[-1], _p(valid), S, _p(fill), _p(gamma), _p(beta),
                   eps, M, C, _p(out_f32), _p(None if out_pair is None else out_pair.buf), _p(pos),
                   0 if pos is None else pos.numel() // C, _p(None if out_pair_pos is None else out_pair_pos.buf), _stream())

    def split_pair_ex(self, x, act, pos, out_pair, out_pair_pos):
        self._cuda(x)
        C = x.shape[-1]
        self._call("fb200_split_pair_ex", _p(x), x.numel() // C, C, _pitch(x), act, _p(pos), 0 if pos is None else pos.numel() // C,
                   _p(None if out_pair is None else out_pair.buf), _p(None if out_pair_pos is None else out_pair_pos.buf), _stream())

    def box_refine_qpos(self, delta, ref_in, ref_out, w0, b0, qpos_pair):
        self._cuda(ref_in)
        self._call("fb200_box_refine_qpos", _p(delta), _p(ref_in), _p(ref_out), _p(w0), _p(b0), 0 if w0 is None else w0.shape[0],
                   _p(None if qpos_pair is None else qpos_pair.buf), ref_in.numel() // 4, _stream())

    def sigmoid_rows(self, x, out):
        self._cuda(x, out)
        C = x.shape[-1]
        self._call("fb200_sigmoid_rows", _p(x), _pitch(x), x.numel() // C, C, _p(out), _stream())

    def row_select(self, x, valid, fill, out):
        self._cuda(x, valid, fill, out)
        C = x.shape[-1]
        self._call("fb200_row_select", _p(x), _p(valid), _p(fill), _p(out), _dt(x), x.numel() // C, valid.numel(), C, _stream())

    def rowmax(self, x, out):
        self._cuda(x, out)
        N = x.shape[-1]
        self._call("fb200_rowmax", _p(x), _dt(x), out.numel(), N, _pitch(x), _p(out), _stream())

    def topk(self, x, K, out_idx, out_val):
        self._cuda(x, out_idx)
        B, N = x.shape
        self._call("fb200_topk", _p(x), B, N, K, _p(out_idx), _p(out_val), _stream())

    def gather_rows(self, src, idx, out):
        self._cuda(src, idx, out)
        B, S, C = src.shape
        self._call("fb200_gather_rows", _p(src), _dt(src), B, S, C, _pitch(src), _p(idx), idx.shape[1], _p(out), _stream())

    def box_op(self, mode, x, ref, idx, out):
        self._cuda(x, out)
        self._call("fb200_box_op", mode, _p(x), _p(ref), _p(idx), _p(out), x.numel(), _stream())

    def detr_postprocess(self, scores, boxes, sizes, K, thr, out_scores, out_labels, out_boxes, out_query, out_count):
        self._cuda(scores, boxes, sizes)
        B, Q, C = scores.shape
        self._call("fb200_detr_postprocess", _p(scores), _p(boxes), _p(sizes), B, Q, C, K, thr, _p(out_scores), _p(out_labels),
                   _p(out_boxes), _p(out_query), _p(out_count), _stream())


    def detr_eval_postprocess(self, scores, boxes, sizes, K, out_scores, out_labels, out_boxes, out_count):
        self._cuda(scores, boxes, sizes)
        B, Q, C = scores.shape
        self._call("fb200_detr_eval_postprocess", _p(scores), _p(boxes), _p(sizes), B, Q, C, K, _p(out_scores), _p(out_labels), _p(out_boxes), _p(out_count), _stream())

    # ---- MaskFormer-family operators -------------------------------------------------------------------------
    def upsample_nearest_add(self, y, cur, out):
        self._cuda(y, cur, out)
        B, h, w, C = y.shape
        self._call("fb200_upsample_nearest_add", _p(y), _p(cur), _p(out), _dt(y), B, h, w, cur.shape[1], cur.shape[2], C, _stream())

    def attn_mask_build(self, x, Q, mask, allowed):
        self._cuda(x, mask, allowed)
        B, h, w, Qp = x.shape
        self._call("fb200_attn_mask_build", _p(x), _dt(x), B, h * w, Qp, Q, _p(mask), mask.shape[2], _p(allowed), _stream())

    def attention_masked(self, q, k, v, mask, allowed, out, heads, scale):
        self._cuda(q, k, v, mask, allowed, out)
        B, Lq, C = q.shape
        self._call("fb200_attention_masked", _p(q), _pitch(q), _p(k), _pitch(k), _p(v), _pitch(v), _p(mask), mask.shape[2], _p(allowed), _p(out), _pitch(out),
                   _dt(q), B, Lq, k.shape[1], heads, C // heads, scale, _stream())

    def attention_masked_split(self, q, k, v, mask, allowed, out, heads, scale):
        """k / v: fp32 tensors [B,Lk,C] or `Pair`s (hi / lo fp16 planes written by their projection)"""
        pair = isinstance(k, Pair)
        kh, vh = (k.hi, v.hi) if pair else (k, v)
        self._cuda(q, kh, vh, mask, allowed, out)
        B, Lq, C = q.shape
        self._call("fb200_attention_masked_split", _p(q), _pitch(q), _p(kh), _pitch(kh), _p(vh), _pitch(vh), F16PAIR if pair else F32, k.lo_off if pair else 0,
                   _p(mask), mask.shape[2], _p(allowed), _p(out), _pitch(out), B, Lq, kh.shape[1], heads, C // heads, scale, _stream())

    def softmax_drop_last(self, x, out):
        self._cuda(x, out)
        N = x.shape[-1]
        self._call("fb200_softmax_drop_last", _p(x), x.numel() // N, N, _pitch(x), _p(out), _stream())

    def mask_sigmoid_upsample(self, x, Q, out):
        self._cuda(x, out)
        B, h, w, Qp = x.shape
        self._call("fb200_mask_sigmoid_upsample", _p(x), _dt(x), B, h, w, Qp, Q, _p(out), out.shape[2], out.shape[3], _stream())

    def mask_sigmoid_upsample_argmax(self, x, Q, scores, labels, counts):
        self._cuda(x, scores, labels, counts)
        B, h, w, Qp = x.shape
        self._call("fb200_mask_sigmoid_upsample_argmax", _p(x), _dt(x), B, h, w, Qp, Q, _p(scores), labels.shape[1], labels.shape[2], _p(labels), _p(counts), _stream())

    def mask_sigmoid_upsample_stats(self, x, Q, size, thr, count, psum):
        self._cuda(x, count, psum)
        B, h, w, Qp = x.shape
        self._call("fb200_mask_sigmoid_upsample_stats", _p(x), _dt(x), B, h, w, Qp, Q, size[0], size[1], thr, _p(count), _p(psum), _stream())

    def mask_sigmoid_upsample_select(self, x, bq, out):
        self._cuda(x, bq, out)
        _, h, w, Qp = x.shape
        self._call("fb200_mask_sigmoid_upsample_select", _p(x), _dt(x), h, w, Qp, _p(bq), bq.shape[0], _p(out), out.shape[1], out.shape[2], _stream())

    def mask_stats(self, masks, thr, count, psum):
        self._cuda(masks, count, psum)
        B, Q, H, W = masks.shape
        self._call("fb200_mask_stats", _p(masks), B * Q, H * W, thr, _p(count), _p(psum), _stream())

    def mask_resize_bbox(self, masks, bq, thr, out_masks, out_bbox):
        self._cuda(masks, bq, out_masks, out_bbox)
        B, Q, H, W = masks.shape
        self._call("fb200_mask_resize_bbox", _p(masks), Q, H, W, _p(bq), bq.shape[0], thr, _p(out_masks), out_masks.shape[1], out_masks.shape[2], _p(out_bbox), _stream())

    # ---- BiSeNetFormer-family operators ----------------------------------------------------------------------
    def dwconv3x3s2(self, x, w9c, scale, bias, out):
        self._cuda(x, w9c, out)
        B, H, W, C = x.shape
        self._call("fb200_dwconv3x3s2_bn", _p(x), _dt(x), B, H, W, C, _p(w9c), _p(scale), _p(bias), _p(out), _stream())

    def avgpool3x3s2(self, x, out):
        self._cuda(x, out)
        B, H, W, C = x.shape
        self._call("fb200_avgpool3x3s2", _p(x), _dt(x), B, H, W, C, _p(out), _pitch(out), _stream())

    def global_avgpool(self, x, out):
        self._cuda(x, out)
        B, C = x.shape[0], x.shape[-1]
        self._call("fb200_global_avgpool", _p(x), _dt(x), B, x.numel() // (B * C), C, _p(out), _stream())

    def channel_scale(self, x, gate, addvec, addt, self_add, out):
        self._cuda(x, gate, out)
        B, C = x.shape[0], x.shape[-1]
        self._call("fb200_channel_scale", _p(x), _p(gate), _p(addvec), _p(addt), int(self_add), _p(out), _dt(x), B, x.numel() // (B * C), C, _stream())

    def mask_argmax(self, masks, scores, labels, counts):
        self._cuda(masks, scores, labels, counts)
        B, Q, H, W = masks.shape
        self._call("fb200_mask_argmax", _p(masks), _p(scores), B, Q, H * W, _p(labels), _p(counts), _stream())

    def label_resize_bbox(self, labels, bq, out_masks, out_bbox):
        self._cuda(labels, bq, out_masks, out_bbox)
        self._call("fb200_label_resize_bbox", _p(labels), labels.shape[1], labels.shape[2], _p(bq), bq.shape[0], _p(out_masks), out_masks.shape[1], out_masks.shape[2],
                   _p(out_bbox), _stream())

    # ---- backward / training-mode operators (autograd_ops.py and the training graph) -------------------------
    def conv_wgrad(self, x, dy, KH, KW, stride, pad, dw):
        self._cuda(x, dy, dw)
        B, H, W, Cin = x.shape
        _, Ho, Wo, Cout = dy.shape
        ws = _ws(self.lib.fb200_conv_wgrad_workspace_bytes(B, Ho, Wo, Cin, Cout, KH, KW), x.device)
        self._call("fb200_conv_wgrad", _p(x), B, H, W, Cin, x.stride(2), _p(dy), Ho, Wo, Cout, dy.stride(2), KH, KW, stride, pad, _p(dw), 0, _p(ws), _stream())

    def conv_wgrad_tc_supported(self, x_shape, dy_shape, KH, KW, stride, pad):
        B, H, W, Cin = x_shape
        _, Ho, Wo, Cout = dy_shape
        return bool(self.lib.fb200_conv_wgrad_tc_supported(B, H, W, Cin, Ho, Wo, Cout, KH, KW, stride, pad))

    def conv_wgrad_tc(self, x_pair, dy_pair, KH, KW, stride, pad, dw):
        self._cuda(x_pair, dy_pair, dw)
        B, H, W, C2 = x_pair.shape
        Cin, Cout = C2 // 2, dy_pair.shape[-1] // 2
        ws = _ws(self.lib.fb200_conv_wgrad_tc_workspace_bytes(B, dy_pair.shape[1], dy_pair.shape[2], Cin, Cout, KH, KW), x_pair.device)
        self._call("fb200_conv_wgrad_tc", _p(x_pair), B, H, W, Cin, _p(dy_pair), Cout, KH, KW, stride, pad, _p(dw), 0, _p(ws), _stream())

    def conv_wgrad_tc_f16(self, x16, dy16, KH, KW, stride, pad, dw):
        self._cuda(x16, dy16, dw)
        B, H, W, Cin = x16.shape
        Cout = dy16.shape[-1]
        ws = _ws(self.lib.fb200_conv_wgrad_tc_workspace_bytes(B, dy16.shape[1], dy16.shape[2], Cin, Cout, KH, KW), x16.device)
        self._call("fb200_conv_wgrad_tc_f16", _p(x16), B, H, W, Cin, _p(dy16), Cout, KH, KW, stride, pad, _p(dw), 0, _p(ws), _stream())

    def dilate2(self, dy, out):
        self._cuda(dy, out)
        B, Ho, Wo, C = dy.shape
        self._call("fb200_dilate2", _p(dy), B, Ho, Wo, C, out.shape[1], out.shape[2], _p(out), _stream())

    def _col_ws(self, C, device):
        return _ws(self.lib.fb200_col_workspace_bytes(C), device)

    def colsum(self, x2d, out):
        self._cuda(x2d, out)
        R, C = x2d.shape
        self._call("fb200_colsum", _p(x2d), R, C, x2d.stride(0), _p(out), 0, _p(self._col_ws(C, x2d.device)), _stream())

    def bn_train_fwd(self, x2d, gamma, beta, res2d, act, eps, momentum, rmean, rvar, save_mean, save_rstd, y2d):
        self._cuda(x2d, gamma, beta, y2d)
        R, C = x2d.shape
        self._call("fb200_bn_train_fwd", _p(x2d), x2d.stride(0), R, C, _p(gamma), _p(beta), _p(res2d), 0 if res2d is None else res2d.stride(0), act, eps,
                   momentum, _p(rmean), _p(rvar), _p(save_mean), _p(save_rstd), _p(y2d), y2d.stride(0), _p(self._col_ws(C, x2d.device)), _stream())

    def bn_train_bwd(self, x2d, dy2d, y2d, gamma, beta, save_mean, save_rstd, act, dx2d, dres2d, dgamma, dbeta):
        self._cuda(x2d, dy2d, dx2d)
        R, C = x2d.shape
        self._call("fb200_bn_train_bwd", _p(x2d), x2d.stride(0), _p(dy2d), dy2d.stride(0), _p(y2d), 0 if y2d is None else y2d.stride(0), R, C, _p(gamma), _p(beta),
                   _p(save_mean), _p(save_rstd), act, _p(dx2d), dx2d.stride(0), _p(dres2d), 0 if dres2d is None else dres2d.stride(0), _p(dgamma), _p(dbeta), 0,
                   _p(self._col_ws(C, x2d.device)), _stream())

    def bn_stats(self, x2d, mean, var):
        self._cuda(x2d, mean, var)
        R, C = x2d.shape
        self._call("fb200_bn_stats", _p(x2d), x2d.stride(0), R, C, _p(mean), _p(var), _p(self._col_ws(C, x2d.device)), _stream())

    def bn_sync_combine(self, allst, eps, momentum, rmean, rvar, mean, rstd, inv_total):
        self._cuda(allst, mean, rstd, inv_total)
        world, width = allst.shape
        self._call("fb200_bn_sync_combine", _p(allst), world, (width - 1) // 2, eps, momentum, _p(rmean), _p(rvar), _p(mean), _p(rstd), _p(inv_total), _stream())

    def bn_apply(self, x2d, mean, rstd, gamma, beta, res2d, act, y2d):
        self._cuda(x2d, mean, rstd, gamma, beta, y2d)
        R, C = x2d.shape
        self._call("fb200_bn_apply", _p(x2d), x2d.stride(0), R, C, _p(mean), _p(rstd), _p(gamma), _p(beta), _p(res2d), 0 if res2d is None else res2d.stride(0), act,
                   _p(y2d), y2d.stride(0), _stream())

    def bn_bwd_reduce(self, x2d, dy2d, y2d, gamma, beta, mean, rstd, act, sum_dy, sum_dy_xhat):
        self._cuda(x2d, dy2d, sum_dy, sum_dy_xhat)
        R, C = x2d.shape
        self._call("fb200_bn_bwd_reduce", _p(x2d), x2d.stride(0), _p(dy2d), dy2d.stride(0), _p(y2d), 0 if y2d is None else y2d.stride(0), R, C, _p(gamma), _p(beta),
                   _p(mean), _p(rstd), act, _p(sum_dy), _p(sum_dy_xhat), _p(self._col_ws(C, x2d.device)), _stream())

    def bn_bwd_apply(self, x2d, dy2d, y2d, gamma, beta, mean, rstd, sum_dy, sum_dy_xhat, inv_count, act, dx2d, dres2d):
        self._cuda(x2d, dy2d, dx2d)
        R, C = x2d.shape
        self._call("fb200_bn_bwd_apply", _p(x2d), x2d.stride(0), _p(dy2d), dy2d.stride(0), _p(y2d), 0 if y2d is None else y2d.stride(0), R, C, _p(gamma), _p(beta),
                   _p(mean), _p(rstd), _p(sum_dy), _p(sum_dy_xhat), inv_count, act, _p(dx2d), dx2d.stride(0), _p(dres2d), 0 if dres2d is None else dres2d.stride(0), _stream())

    def add_act(self, a, b, dy, act, out):
        self._cuda(a, out)
        self._call("fb200_add_act", _p(a), _p(b), _p(dy), act, a.numel(), _p(out), _stream())

    def maxpool_bwd(self, x, dy, dx):
        self._cuda(x, dy, dx)
        B, H, W, C = x.shape
        self._call("fb200_maxpool3x3s2_bwd", _p(x), _p(dy), B, H, W, C, _p(dx), _stream())

    def avgpool_bwd(self, dy, dx):
        self._cuda(dy, dx)
        B, H, W, C = dx.shape
        self._call("fb200_avgpool2x2_ceil_bwd", _p(dy), B, H, W, C, _p(dx), _stream())

    def resize_bwd(self, dy, dx):
        self._cuda(dy, dx)
        B, H, W, C = dx.shape
        self._call("fb200_resize_bilinear_bwd", _p(dy), dy.stride(2), B, H, W, C, dy.shape[1], dy.shape[2], _p(dx), _stream())

    def layernorm_bwd(self, x2d, res2d, gamma, dy2d, eps, dx2d, dgamma, dbeta):
        self._cuda(x2d, dy2d, dx2d)
        M, C = x2d.shape
        self._call("fb200_layernorm_bwd", _p(x2d), _p(res2d), _p(gamma), _p(dy2d), M, C, eps, _p(dx2d), _p(dgamma), _p(dbeta), 0,
                   _p(self._col_ws(C, x2d.device)), _stream())

    def attention_bwd(self, q, k, v, o, do, heads, scale, dq, dk, dv):
        self._cuda(q, k, v, o, do, dq, dk, dv)
        B, Lq, C = q.shape
        self._call("fb200_attention_bwd", _p(q), q.stride(1), _p(k), k.stride(1), _p(v), v.stride(1), _p(o), o.stride(1), _p(do), do.stride(1), B, Lq, k.shape[1], heads,
                   C // heads, scale, _p(dq), dq.stride(1), _p(dk), dk.stride(1), _p(dv), dv.stride(1), _stream())

    def msda_bwd(self, value, oa, ref, do, shapes, P, heads, dvalue, doa):
        self._cuda(value, oa, ref, do, dvalue, doa)
        B, S, _ = value.shape
        Q = oa.shape[1]
        arr = (ctypes.c_int * (2 * len(shapes)))(*[int(v) for hw in shapes for v in hw])
        self._call("fb200_msda_bwd", _p(value), value.stride(1), _p(oa), oa.stride(1), _p(ref), _p(do), do.stride(1), arr, len(shapes), P, B, S, Q, heads, _p(dvalue),
                   dvalue.stride(1), _p(doa), doa.stride(1), _stream())

    # ---- DETR training criterion (criterion.py) --------------------------------------------------------------
    def detr_match_cost(self, logits, boxes, tl, tb, toff, wts, alpha, gamma, cost):
        self._cuda(logits, boxes, tl, tb, toff, cost)
        L, B, Q, C = logits.shape
        self._call("fb200_detr_match_cost", _p(logits), _p(boxes), _p(tl), _p(tb), _p(toff), L, B, Q, C, tl.shape[0],
                   wts[0], wts[1], wts[2], alpha, gamma, _p(cost), _stream())

    def hungarian(self, cost, toff, B, max_targets, match_q):
        self._cuda(cost, toff, match_q)
        L, T, Q = cost.shape
        self._call("fb200_hungarian", _p(cost), _p(toff), L, B, Q, T, max_targets, _p(match_q), _stream())

    def detr_loss(self, logits, boxes, tl, tb, toff, match_q, num_boxes, wts, alpha, gamma, losses, g_logits, g_l1, g_giou):
        self._cuda(logits, boxes, toff, losses, g_logits, g_l1, g_giou)
        L, B, Q, C = logits.shape
        ws = _ws(self.lib.fb200_detr_loss_workspace_bytes(L, B, Q), logits.device)
        self._call("fb200_detr_loss", _p(logits), _p(boxes), _p(tl), _p(tb), _p(toff), _p(match_q), L, B, Q, C, 0 if tl is None else tl.shape[0],
                   num_boxes, wts[0], wts[1], wts[2], alpha, gamma,
                   _p(losses), _p(g_logits), _p(g_l1), _p(g_giou), _p(ws), _stream())

    # ---- optimiser step (train_step.py) ----------------------------------------------------------------------
    def optim_workspace(self, device):
        return torch.zeros(int(self.lib.fb200_optim_workspace_bytes()), dtype=torch.uint8, device=device)

    def grad_stats(self, grads, ws):
        self._cuda(grads, ws)
        self._call("fb200_grad_stats", _p(grads), grads.numel(), _p(ws), _stream())

    def optim_finalize(self, ws, ctrl, max_norm, clip_passes, inv_world, use_scaler, growth, backoff, growth_interval, beta1, beta2):
        self._cuda(ws, ctrl)
        self._call("fb200_optim_finalize", _p(ws), _p(ctrl), max_norm, int(clip_passes), inv_world, int(use_scaler),
                   growth, backoff, int(growth_interval), beta1, beta2, _stream())

    def adamw_step(self, params, grads, m, v, chunk_start, chunk_len, chunk_seg, seg_lr, seg_wd, seg_active, lr_factor, beta1, beta2, eps, ctrl):
        self._cuda(params, grads, m, v, chunk_start, chunk_len, chunk_seg, seg_lr, seg_wd, ctrl)
        self._call("fb200_adamw_step", _p(params), _p(grads), _p(m), _p(v), _p(chunk_start), _p(chunk_len), _p(chunk_seg), chunk_len.shape[0], _p(seg_lr), _p(seg_wd), _p(seg_active),
                   lr_factor, beta1, beta2, eps, _p(ctrl), _stream())


class Pair:
    """An fp32 NHWC activation stored as TWO fp16 planes (hi = fp16(v), lo = fp16(v - hi), exact to ~2^-22) inside one buffer `buf` [..., 2 * Ctot]:
    hi planes of all channels in buf[..., :Ctot], lo planes in buf[..., Ctot:] - the operand format of the fp32-accurate tensor-core convs, which also
    WRITE it (conv2d_pair), so activations never pass through a separate split kernel between two convs.  A Pair may be a channel slice [c0, c0 + C)
    of a wider pair buffer (concat-free CSP / FPN blocks): hi and lo are then strided views with the same pixel pitch."""

    __slots__ = ("buf", "c0", "C")

    def __init__(self, buf: torch.Tensor, c0: int = 0, C: Optional[int] = None):
        assert buf.dtype == torch.float16 and buf.shape[-1] % 2 == 0
        self.buf, self.c0 = buf, c0
        self.C = buf.shape[-1] // 2 - c0 if C is None else C

    @staticmethod
    def empty(shape, device) -> "Pair":
        return Pair(torch.empty((*shape[:-1], 2 * shape[-1]), dtype=torch.float16, device=device))

    @property
    def Ctot(self) -> int:
        return self.buf.shape[-1] // 2

    @property
    def hi(self) -> torch.Tensor:
        return self.buf[..., self.c0:self.c0 + self.C]

    @property
    def lo(self) -> torch.Tensor:
        return self.buf[..., self.Ctot + self.c0:self.Ctot + self.c0 + self.C]

    @property
    def lo_off(self) -> int:
        return self.Ctot

    @property
    def shape(self):
        return (*self.buf.shape[:-1], self.C)

    @property
    def device(self):
        return self.buf.device

    def slice(self, a: int, b: int) -> "Pair":
        return Pair(self.buf, self.c0 + a, b - a)

    def float(self) -> torch.Tensor:
        """the fp32 values (a torch op: taps / tests only, never on the forward path)"""
        return self.hi.float() + self.lo.float()


_cuda_backend = None


def _be():
    global _cuda_backend
    if _backend is not None:
        return _backend
    if _cuda_backend is None:
        _cuda_backend = CudaBackend()
    return _cuda_backend


OPT_CONV_CTA_PAIR = 0


def set_option(option: int, value: int) -> int:
    """process-wide tuning option of the C library (include/focoos_b200.h fb200_option); returns the previous value"""
    rc = load_library().fb200_set_option(int(option), int(value))
    if rc < 0:
        _check(rc, "set_option")
    return rc


def set_conv_trace(buf: Optional[torch.Tensor]):
    """debug timeline of conv_tc launches (see include/focoos_b200.h fb200_set_conv_trace); buf: int64 CUDA tensor [>= 296 * 128] or None"""
    _check(load_library().fb200_set_conv_trace(_p(buf)), "set_conv_trace")


def supports_tcgen05() -> bool:
    return load_library().fb200_device_supports_tcgen05() == 1


_tc_ok = None


def supports_tcgen05_cached() -> bool:
    """tcgen05 path usable (real sm_100 device; False under the tests' CPU backend hook)"""
    global _tc_ok
    if _backend is not None:
        return False
    if _tc_ok is None:
        _tc_ok = supports_tcgen05()
    return _tc_ok


# ------------------------------------------------------------------------------------------------
# public tensor-level API
# ------------------------------------------------------------------------------------------------
def stem_conv(img: torch.Tensor, w, scale, bias, mean: Sequence[float], std: Sequence[float], act=ACT_RELU, out_dtype=torch.float32, out_pair: bool = False):
    """[B,3,H,W] fp32 NCHW 0..255 -> normalise -> conv3x3/s2 + BN + act -> NHWC [B,H/2,W/2,32]."""
    assert img.dim() == 4 and img.is_contiguous()
    if img.dtype == torch.uint8:  # decoded images as they come: [B,H,W,3] uint8
        assert img.shape[3] == 3
        B, H, W, _ = img.shape
    else:
        assert img.dtype == torch.float32 and img.shape[1] == 3
        B, _, H, W = img.shape
    if out_pair:  # the result as a Pair: [hi(Cout) | lo(Cout)] fp16 per pixel
        pr = Pair.empty((B, (H - 1) // 2 + 1, (W - 1) // 2 + 1, w.shape[0]), img.device)
        _be().stem_conv(img, w, scale, bias, [float(v) for v in mean], [float(v) for v in std], act, pr)
        return pr
    out = torch.empty((B, (H - 1) // 2 + 1, (W - 1) // 2 + 1, w.shape[0]), dtype=out_dtype, device=img.device)
    _be().stem_conv(img, w, scale, bias, [float(v) for v in mean], [float(v) for v in std], act, out)
    return out


def conv2d(x, w, scale=None, bias=None, *, stride=1, pad=0, act=ACT_NONE, residual=None, out=None, out_dtype=None, algo=ALGO_AUTO):
    """NHWC conv with fused per-channel scale/bias (folded BN), residual add and activation.
    w: [Cout,KH,KW,Cin] (same dtype as x).  `out` may be a channel slice of a wider NHWC buffer."""
    assert x.dim() == 4 and w.dim() == 4 and w.is_contiguous() and w.dtype == x.dtype
    if algo == ALGO_TCGEN05_SPLIT3:  # x = [hi|lo] pair (2C channels), w = [W_hi|W_lo|W_hi] (3C)
        assert x.dtype == torch.float16 and w.shape[3] * 2 == x.shape[3] * 3
    else:
        assert w.shape[3] == x.shape[3]
    B, H, W, _ = x.shape
    Cout, KH, KW, _ = w.shape
    Ho, Wo = (H + 2 * pad - KH) // stride + 1, (W + 2 * pad - KW) // stride + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, Cout), dtype=out_dtype or x.dtype, device=x.device)
    assert tuple(out.shape) == (B, Ho, Wo, Cout), (tuple(out.shape), (B, Ho, Wo, Cout))
    if residual is not None:
        assert residual.shape == out.shape and residual.dtype == out.dtype
    _be().conv2d(x, w, scale, bias, stride, pad, act, residual, out, algo)
    return out


def conv2d_per_image(x, w, *, act=ACT_NONE, out=None, out_dtype=None, algo=ALGO_AUTO):
    """conv with one weight set per image: x [B,H,W,Cin], w [B,Cout,KH,KW,Cin] -> [B,H,W,Cout]  (the per-query mask product, one launch per batch)."""
    assert x.dim() == 4 and w.dim() == 5 and w.shape[0] == x.shape[0] and w.dtype == x.dtype and w.stride(-1) == 1
    if algo == ALGO_TCGEN05_SPLIT3:  # fp32-accurate: x = the [hi|lo] pair of the fp32 activation (2C channels), w = per-image [W_hi|W_lo|W_hi] triples (3C), fp32 out
        assert x.dtype == torch.float16 and w.shape[-1] * 2 == x.shape[-1] * 3, (w.shape, x.shape)
        out_dtype = out_dtype or torch.float32
    else:
        assert w.shape[-1] == x.shape[-1]
    B, H, W, _ = x.shape
    Cout = w.shape[1]
    if out is None:
        out = torch.empty((B, H, W, Cout), dtype=out_dtype or x.dtype, device=x.device)
    assert tuple(out.shape) == (B, H, W, Cout)
    _be().conv2d_per_image(x, w.contiguous(), act, out, algo)
    return out


def linear_rowmax(x, w, bias=None):
    """max over the output features of x @ w.T + bias, per row, without materialising the product (fp16 x [..., K], w [N, K]) -> fp32 [...]."""
    assert x.dtype == torch.float16 and w.dtype == torch.float16 and x.stride(-1) == 1
    lead = x.shape[:-1]
    x2 = x.reshape(-1, x.shape[-1])
    out = torch.full((x2.shape[0],), float("-inf"), dtype=torch.float32, device=x.device)
    _be().linear_rowmax(x2, w.reshape(w.shape[0], -1).contiguous(), bias, out)
    return out.reshape(lead)


def linear_rowmax_pair(xp: "Pair", w3, bias=None):
    """linear_rowmax on pair-format rows with the split weight triple: fp32-accurate row maxima, the [rows, N] product never materialised"""
    lead = xp.shape[:-1]
    out = torch.full((int(np.prod(lead)),), float("-inf"), dtype=torch.float32, device=xp.device)
    _be().linear_rowmax_pair(xp, w3.reshape(w3.shape[0], -1).contiguous(), bias, out)
    return out.reshape(lead)


def split_pair(x):
    """fp32 [..., C] (rows may be pitched) -> fp16 [..., 2C] = [hi | lo] with hi = fp16(x), lo = fp16(x - hi): operands of the
    split-precision tensor-core mode (three fp16 products reproduce the fp32 product to ~2^-21)."""
    assert x.dtype == torch.float32
    out = torch.empty((*x.shape[:-1], 2 * x.shape[-1]), dtype=torch.float16, device=x.device)
    _be().split_pair(x, out)
    return out


def to_pair(x) -> Pair:
    """fp32 tensor -> Pair (one split launch); a Pair passes through"""
    return x if isinstance(x, Pair) else Pair(split_pair(x))


def conv2d_pair(x: Pair, w3, scale=None, bias=None, *, stride=1, pad=0, act=ACT_NONE, residual=None, out=None, out_pair: bool = True):
    """fp32-accurate conv (three fp16 tcgen05 products) on a pair-format input.  `out_pair`: write the result as a Pair (for a following conv / pair pool) or
    as a plain fp32 tensor (for the non-conv consumers: LayerNorm, attention, deformable attention, selection).  The residual has the output's format."""
    assert isinstance(x, Pair) and w3.dtype == torch.float16 and w3.shape[3] == 3 * x.C, (w3.shape, x.C)
    B, H, W, _ = x.shape
    Cout, KH, KW, _ = w3.shape
    Ho, Wo = (H + 2 * pad - KH) // stride + 1, (W + 2 * pad - KW) // stride + 1
    if out is None:
        out = Pair.empty((B, Ho, Wo, Cout), x.device) if out_pair else torch.empty((B, Ho, Wo, Cout), dtype=torch.float32, device=x.device)
    assert tuple(out.shape) == (B, Ho, Wo, Cout), (tuple(out.shape), (B, Ho, Wo, Cout))
    if residual is not None:
        assert isinstance(residual, Pair) == isinstance(out, Pair) and tuple(residual.shape) == tuple(out.shape)
    _be().conv2d_pair(x, w3, scale, bias, stride, pad, act, residual, out)
    return out


def image_resize(images, size: Tuple[int, int]):
    """a batch of decoded images - uint8 NHWC [B,H,W,3] or float32 NCHW [B,3,H,W] - resized (bilinear, align_corners=False on the float values, like the reference's
    F.interpolate in processor/base_processor.py:284-294) to float32 NCHW [B,3,size[0],size[1]] in ONE launch."""
    images = images.contiguous()
    assert (images.dtype == torch.uint8 and images.dim() == 4 and images.shape[3] == 3) or (images.dtype == torch.float32 and images.dim() == 4 and images.shape[1] == 3)
    out = torch.empty((images.shape[0], 3, int(size[0]), int(size[1])), dtype=torch.float32, device=images.device)
    _be().image_resize(images, out)
    return out


def pair_maxpool3x3s2(x: Pair) -> Pair:
    B, H, W, C = x.shape
    out = Pair.empty((B, (H - 1) // 2 + 1, (W - 1) // 2 + 1, C), x.device)
    _be().pair_pool(0, x, out)
    return out


def pair_avgpool2x2(x: Pair) -> Pair:
    B, H, W, C = x.shape
    out = Pair.empty((B, (H + 1) // 2, (W + 1) // 2, C), x.device)
    _be().pair_pool(1, x, out)
    return out


def pair_resize_bilinear(x: Pair, size: Tuple[int, int], out: Optional[Pair] = None) -> Pair:
    B, H, W, C = x.shape
    if out is None:
        out = Pair.empty((B, size[0], size[1], C), x.device)
    assert tuple(out.shape) == (B, size[0], size[1], C)
    _be().pair_pool(2, x, out)
    return out


def linear(x, w, bias=None, *, act=ACT_NONE, residual=None, out=None, out_dtype=None, algo=ALGO_AUTO):
    """y = act(x @ w.T + bias (+ residual)); x [..., K] (rows may be pitched), w [N, K]."""
    lead = x.shape[:-1]
    K = x.shape[-1]
    N = w.shape[0]
    x4 = x.reshape(1, 1, -1, K) if x.is_contiguous() else _as4(x)
    r4 = None if residual is None else (residual.reshape(1, 1, -1, N) if residual.is_contiguous() else _as4(residual))
    o4 = None if out is None else (out.reshape(1, 1, -1, N) if out.is_contiguous() else _as4(out))
    y = conv2d(x4, w.reshape(N, 1, 1, w.shape[-1]), None, bias, act=act, residual=r4, out=o4, out_dtype=out_dtype, algo=algo)
    return out if out is not None else y.reshape(*lead, N)


def _as4(t):
    """[..., L, C] pitched view -> [1,1,M,C] view (requires uniform pitch, checked by _pitch)."""
    p = _pitch(t)
    M = t.numel() // t.shape[-1]
    return t.as_strided((1, 1, M, t.shape[-1]), (M * p, M * p, p, 1), t.storage_offset())


def maxpool3x3s2(x):
    B, H, W, C = x.shape
    out = torch.empty((B, (H - 1) // 2 + 1, (W - 1) // 2 + 1, C), dtype=x.dtype, device=x.device)
    _be().maxpool3x3s2(x.contiguous(), out)
    return out


def avgpool2x2(x):
    B, H, W, C = x.shape
    out = torch.empty((B, (H + 1) // 2, (W + 1) // 2, C), dtype=x.dtype, device=x.device)
    _be().avgpool2x2(x.contiguous(), out)
    return out


def resize_bilinear(x, size: Tuple[int, int], out=None):
    B, H, W, C = x.shape
    if out is None:
        out = torch.empty((B, size[0], size[1], C), dtype=x.dtype, device=x.device)
    assert tuple(out.shape) == (B, size[0], size[1], C)
    _be().resize_bilinear(x, out)
    return out


def add(a, b):
    """a + b with b broadcast over leading dims (a [B,L,C], b [L,C] or [1,L,C] or same shape)."""
    a = a.contiguous()
    b = b.contiguous()
    out = torch.empty_like(a)
    _be().add(a, b, out)
    return out


def layernorm(x, gamma, beta, residual=None, eps=1e-5):
    x = x.contiguous()
    if residual is not None:
        residual = residual.contiguous()
        assert residual.shape == x.shape
    out = torch.empty_like(x)
    _be().layernorm(x, residual, gamma, beta, out, eps)
    return out


def attention(q, k, v, heads: int, scale: float, split: bool = False, out_pair: bool = False):
    """softmax(q k^T * scale) v per head; q [B,Lq,C], k,v [B,Lk,C] (may be column slices of one buffer).
    split=True (fp32 tensors only): tensor-core kernel with split-precision products instead of the CUDA-core fp32 kernel."""
    B, Lq, C = q.shape
    if out_pair:  # fp32 split kernel writing the [hi | lo] pair rows the out_proj linear reads
        assert split and q.dtype == torch.float32
        out = Pair.empty((B, Lq, C), q.device)
        _be().attention(q, k, v, out, heads, scale, True)
        return out
    out = torch.empty((B, Lq, C), dtype=q.dtype, device=q.device)
    if split and q.dtype == torch.float32:
        _be().attention(q, k, v, out, heads, scale, True)
    else:
        _be().attention(q, k, v, out, heads, scale)
    return out


def msda(value, oa, ref, shapes, num_points: int, heads: int, out_dtype=None, out_pair: bool = False):
    """value [B,S,heads*32]; oa [B,Q,heads*L*P*3] (offsets then logits); ref [B,Q,4] fp32 -> [B,Q,heads*32]."""
    B, Q = oa.shape[0], oa.shape[1]
    if out_pair:
        out = Pair.empty((B, Q, heads * 32), value.device)
    else:
        out = torch.empty((B, Q, heads * 32), dtype=out_dtype or value.dtype, device=value.device)
    _be().msda(value, oa, ref.contiguous(), [tuple(s) for s in shapes], num_points, heads, out)
    return out


def layernorm_ex(x, gamma, beta, *, residual=None, gather=None, valid=None, fill=None, pos=None, want_f32=True, want_pair=True, want_pair_pos=False, eps=1e-5):
    """Fused row glue of the fp32-accurate head (csrc/head_fused.cu): LayerNorm of fp32 rows x [B, S, C] - optionally gathered by top-k indices `gather` [B, K]
    and masked by `valid` [S] / `fill` [C] - returned as (fp32 tensor | None, Pair | None, Pair of (y + pos) | None)."""
    C = x.shape[-1]
    if gather is not None:
        lead = (x.shape[0], gather.shape[-1])
    else:
        lead = tuple(x.shape[:-1])
    M = 1
    for d in lead:
        M *= d
    of = torch.empty((*lead, C), dtype=torch.float32, device=x.device) if want_f32 else None
    op = Pair.empty((*lead, C), x.device) if want_pair else None
    opp = Pair.empty((*lead, C), x.device) if want_pair_pos else None
    _be().layernorm_ex(x, residual, gather, valid, fill, gamma, beta, eps, M, of, op, pos if want_pair_pos else None, opp)
    return of, op, opp


def split_pair_ex(x, *, act=ACT_NONE, pos=None, want_pair=True, want_pair_pos=False):
    """(Pair of act(x) | None, Pair of (x + pos) | None) of an fp32 tensor in one pass; pos broadcasts over leading rows"""
    x = x if x.stride(-1) == 1 else x.contiguous()
    op = Pair.empty(tuple(x.shape), x.device) if want_pair else None
    opp = Pair.empty(tuple(x.shape), x.device) if want_pair_pos else None
    _be().split_pair_ex(x, act, pos if want_pair_pos else None, op, opp)
    return op, opp


def box_refine_qpos(delta, ref, w0=None, b0=None):
    """(new reference boxes, Pair of relu(boxes . w0^T + b0) | None): bbox refinement (delta may be None: boxes = ref) + first query_pos_head layer"""
    ref = ref.contiguous()
    new_ref = torch.empty_like(ref) if delta is not None else ref
    qp = Pair.empty((*ref.shape[:-1], w0.shape[0]), ref.device) if w0 is not None else None
    _be().box_refine_qpos(None if delta is None else delta.contiguous(), ref, new_ref if delta is not None else None, w0, b0, qp)
    return new_ref, qp


def sigmoid_rows(x):
    """dense sigmoid(x) of a (possibly pitched) fp32 [.., C] view"""
    out = torch.empty(tuple(x.shape), dtype=torch.float32, device=x.device)
    _be().sigmoid_rows(x, out)
    return out


def row_select(x, valid_u8, fill_f32):
    x = x.contiguous()
    out = torch.empty_like(x)
    _be().row_select(x, valid_u8, fill_f32, out)
    return out


def rowmax(x):
    out = torch.empty(x.shape[:-1], dtype=torch.float32, device=x.device)
    _be().rowmax(x, out)
    return out


def topk(x, k: int):
    assert x.dtype == torch.float32 and x.dim() == 2 and x.is_contiguous()
    idx = torch.empty((x.shape[0], k), dtype=torch.int32, device=x.device)
    val = torch.empty((x.shape[0], k), dtype=torch.float32, device=x.device)
    _be().topk(x, k, idx, val)
    return val, idx


def gather_rows(src, idx):
    B, S, C = src.shape
    out = torch.empty((B, idx.shape[1], C), dtype=src.dtype, device=src.device)
    _be().gather_rows(src, idx, out)
    return out


def box_sigmoid(x):
    x = x.contiguous()
    out = torch.empty_like(x)
    _be().box_op(0, x, None, None, out)
    return out


def box_refine(delta, ref):
    delta, ref = delta.contiguous(), ref.contiguous()
    out = torch.empty_like(delta)
    _be().box_op(1, delta, ref, None, out)
    return out


def box_add_anchors(x, anchors, idx):
    x = x.contiguous()
    out = torch.empty_like(x)
    _be().box_op(2, x, anchors, idx.contiguous(), out)
    return out


def box_cxcywh_to_xyxy(x):
    x = x.contiguous()
    out = torch.empty_like(x)
    _be().box_op(3, x, None, None, out)
    return out


def detr_postprocess(scores, boxes, sizes_i32, top_k: int, threshold: float):
    """-> (scores [B,K], labels [B,K] i32, boxes [B,K,4] i32, query [B,K] i32, count [B] i32), sorted by score."""
    B = scores.shape[0]
    dev = scores.device
    o_s = torch.empty((B, top_k), dtype=torch.float32, device=dev)
    o_l = torch.empty((B, top_k), dtype=torch.int32, device=dev)
    o_b = torch.empty((B, top_k, 4), dtype=torch.int32, device=dev)
    o_q = torch.empty((B, top_k), dtype=torch.int32, device=dev)
    o_c = torch.empty((B,), dtype=torch.int32, device=dev)
    _be().detr_postprocess(scores.contiguous(), boxes.contiguous(), sizes_i32, top_k, float(threshold), o_s, o_l, o_b, o_q, o_c)
    return o_s, o_l, o_b, o_q, o_c


def detr_eval_postprocess(scores, boxes, sizes_i32, top_k: int):
    """evaluator variant: -> (scores [B,K], labels [B,K] i32, boxes [B,K,4] fp32 in pixels of sizes[b], count [B] i32); rows [0, count[b]) are valid"""
    B = scores.shape[0]
    dev = scores.device
    o_s = torch.empty((B, top_k), dtype=torch.float32, device=dev)
    o_l = torch.empty((B, top_k), dtype=torch.int32, device=dev)
    o_b = torch.empty((B, top_k, 4), dtype=torch.float32, device=dev)
    o_c = torch.empty((B,), dtype=torch.int32, device=dev)
    _be().detr_eval_postprocess(scores.contiguous(), boxes.contiguous(), sizes_i32, top_k, o_s, o_l, o_b, o_c)
    return o_s, o_l, o_b, o_c


# ------------------------------------------------------------------------------------------------
# torch.library registration: focoos_b200::<op>  (out-variant schemas; the python API above allocates)
# ------------------------------------------------------------------------------------------------
_torch_lib = None


def _register_torch_ops():
    global _torch_lib
    if _torch_lib is not None:
        return
    lib = torch.library.Library("focoos_b200", "DEF")
    defs = {
        "conv2d": ("(Tensor x, Tensor w, Tensor? scale, Tensor? bias, int stride, int pad, int act, Tensor? residual, Tensor(a!) out, int algo) -> ()",
                   lambda x, w, scale, bias, stride, pad, act, residual, out, algo: _be().conv2d(x, w, scale, bias, stride, pad, act, residual, out, algo)),
        "maxpool3x3s2": ("(Tensor x, Tensor(a!) out) -> ()", lambda x, out: _be().maxpool3x3s2(x, out)),
        "avgpool2x2": ("(Tensor x, Tensor(a!) out) -> ()", lambda x, out: _be().avgpool2x2(x, out)),
        "resize_bilinear": ("(Tensor x, Tensor(a!) out) -> ()", lambda x, out: _be().resize_bilinear(x, out)),
        "add": ("(Tensor a, Tensor b, Tensor(a!) out) -> ()", lambda a, b, out: _be().add(a, b, out)),
        "layernorm": ("(Tensor x, Tensor? res, Tensor gamma, Tensor beta, Tensor(a!) out, float eps) -> ()",
                      lambda x, res, gamma, beta, out, eps: _be().layernorm(x, res, gamma, beta, out, eps)),
        "attention": ("(Tensor q, Tensor k, Tensor v, Tensor(a!) out, int heads, float scale) -> ()",
                      lambda q, k, v, out, heads, scale: _be().attention(q, k, v, out, heads, scale)),
        "msda": ("(Tensor value, Tensor oa, Tensor ref, int[] shapes, int points, int heads, Tensor(a!) out) -> ()",
                 lambda value, oa, ref, shapes, points, heads, out: _be().msda(value, oa, ref, [tuple(shapes[i:i + 2]) for i in range(0, len(shapes), 2)], points, heads, out)),
        "rowmax": ("(Tensor x, Tensor(a!) out) -> ()", lambda x, out: _be().rowmax(x, out)),
        "topk": ("(Tensor x, int k, Tensor(a!) out_idx, Tensor(b!) out_val) -> ()", lambda x, k, oi, ov: _be().topk(x, k, oi, ov)),
        "gather_rows": ("(Tensor src, Tensor idx, Tensor(a!) out) -> ()", lambda src, idx, out: _be().gather_rows(src, idx, out)),
        "box_op": ("(int mode, Tensor x, Tensor? ref, Tensor? idx, Tensor(a!) out) -> ()", lambda mode, x, ref, idx, out: _be().box_op(mode, x, ref, idx, out)),
    }
    for name, (schema, fn) in defs.items():
        lib.define(name + schema)
        lib.impl(name, fn, "CUDA")
    _torch_lib = lib


try:  # registration itself needs no GPU and no compiled library
    _register_torch_ops()
except Exception:  # pragma: no cover - e.g. double import under a different module name
    pass


# ------------------------------------------------------------------------------------------------
# MaskFormer-family operators (SURVEY §8 rows a14-a17)
# ------------------------------------------------------------------------------------------------


def upsample_nearest_add(y, cur):
    """cur + F.interpolate(y, size=cur.shape, mode="nearest")  (fai_mf/modelling.py:364), NHWC."""
    out = torch.empty_like(cur)
    _be().upsample_nearest_add(y.contiguous(), cur.contiguous(), out)
    return out


def attn_mask_build(mask_logits_nhwc, num_queries: int):
    """[B,h,w,Qp] mask logits at the target level size -> (uint8 mask [B,Q,LkP] with 1 = NOT allowed (logit < 0), int32 allowed-key
    count [B,Q]).  A row whose count is 0 attends everywhere (fai_mf/modelling.py:96-105,510-513)."""
    B, h, w, _ = mask_logits_nhwc.shape
    LkP = (h * w + 3) // 4 * 4
    mask = torch.empty((B, num_queries, LkP), dtype=torch.uint8, device=mask_logits_nhwc.device)
    allowed = torch.zeros((B, num_queries), dtype=torch.int32, device=mask_logits_nhwc.device)
    _be().attn_mask_build(mask_logits_nhwc.contiguous(), num_queries, mask, allowed)
    return mask, allowed


def attention_masked(q, k, v, mask, allowed, heads: int, scale: float, split: bool = False):
    """masked cross-attention: q [B,Lq,C], k/v [B,Lk,C]; mask/allowed from attn_mask_build (shared by all heads).
    split (fp32 tensors, precision "fp32_tc"): fp32-accurate tensor-core products instead of the CUDA-core fp32 kernel."""
    B, Lq, C = q.shape
    out = torch.empty((B, Lq, C), dtype=q.dtype, device=q.device)
    if split and q.dtype == torch.float32:
        if isinstance(k, Pair):
            assert isinstance(v, Pair) and k.lo_off == v.lo_off and k.C == C and v.C == C
        _be().attention_masked_split(q, k, v, mask, allowed, out, heads, scale)
    else:
        _be().attention_masked(q, k, v, mask, allowed, out, heads, scale)
    return out


def softmax_drop_last(x):
    """F.softmax(x, -1)[..., :-1] on fp32 rows (fai_mf/modelling.py:618)."""
    assert x.dtype == torch.float32
    out = torch.empty((*x.shape[:-1], x.shape[-1] - 1), dtype=torch.float32, device=x.device)
    _be().softmax_drop_last(x, out)
    return out


def mask_sigmoid_upsample(mask_logits_nhwc, num_queries: int, size):
    """[B,h,w,Qp] logits -> sigmoid -> bilinear (align_corners=False) to `size` -> [B,Q,H,W] fp32 probabilities
    (fai_mf/modelling.py:619,722-723: sigmoid at low resolution THEN upsample)."""
    B = mask_logits_nhwc.shape[0]
    out = torch.empty((B, num_queries, size[0], size[1]), dtype=torch.float32, device=mask_logits_nhwc.device)
    _be().mask_sigmoid_upsample(mask_logits_nhwc.contiguous(), num_queries, out)
    return out


def mask_sigmoid_upsample_argmax(mask_logits_nhwc, num_queries: int, size, scores):
    """semantic labels straight from the low-resolution mask logits: argmax_q(scores[b,q] * bilinear(sigmoid(x))[b,q]) -> (labels uint8 [B,H,W],
    counts int32 [B,Q]) without materialising the [B,Q,H,W] probabilities."""
    B = mask_logits_nhwc.shape[0]
    labels = torch.empty((B, size[0], size[1]), dtype=torch.uint8, device=mask_logits_nhwc.device)
    counts = torch.empty((B, num_queries), dtype=torch.int32, device=mask_logits_nhwc.device)
    _be().mask_sigmoid_upsample_argmax(mask_logits_nhwc.contiguous(), num_queries, scores.contiguous().float(), labels, counts)
    return labels, counts


def mask_sigmoid_upsample_stats(mask_logits_nhwc, num_queries: int, size, thr: float):
    """(count [B,Q] int32, psum [B,Q] fp32) of mask_stats(mask_sigmoid_upsample(x)) without materialising the [B,Q,H,W] probabilities."""
    B = mask_logits_nhwc.shape[0]
    count = torch.empty((B, num_queries), dtype=torch.int32, device=mask_logits_nhwc.device)
    psum = torch.empty((B, num_queries), dtype=torch.float32, device=mask_logits_nhwc.device)
    _be().mask_sigmoid_upsample_stats(mask_logits_nhwc.contiguous(), num_queries, (int(size[0]), int(size[1])), float(thr), count, psum)
    return count, psum


def mask_sigmoid_upsample_select(mask_logits_nhwc, bq_i32, size):
    """upsampled probabilities [n,H,W] of the kept (b,q) pairs only (same values as mask_sigmoid_upsample(x)[b,q])."""
    n = bq_i32.shape[0]
    out = torch.empty((n, int(size[0]), int(size[1])), dtype=torch.float32, device=mask_logits_nhwc.device)
    if n:
        _be().mask_sigmoid_upsample_select(mask_logits_nhwc.contiguous(), bq_i32.contiguous(), out)
    return out


def mask_stats(masks, thr: float):
    """per (b,q): number of pixels with prob >= thr and the sum of those probabilities (fai_mf/processor.py:222-257)."""
    B, Q = masks.shape[:2]
    count = torch.empty((B, Q), dtype=torch.int32, device=masks.device)
    psum = torch.empty((B, Q), dtype=torch.float32, device=masks.device)
    _be().mask_stats(masks.contiguous(), thr, count, psum)
    return count, psum


def mask_resize_bbox(masks, bq_i32, thr: float, size):
    """kept (b,q) pairs -> binary masks (prob >= thr) bilinearly resized to `size` and re-binarised (> 0), plus their xyxy boxes
    (fai_mf/processor.py:275-283, utils/vision.py:344-370)."""
    n = bq_i32.shape[0]
    om = torch.empty((n, size[0], size[1]), dtype=torch.uint8, device=masks.device)
    ob = torch.empty((n, 4), dtype=torch.int32, device=masks.device)
    if n:
        _be().mask_resize_bbox(masks.contiguous(), bq_i32.contiguous(), thr, om, ob)
    return om, ob


# ------------------------------------------------------------------------------------------------
# BiSeNetFormer-family operators (SURVEY §8 rows a18-a19)
# ------------------------------------------------------------------------------------------------
ACT_SIGMOID = 4


def dwconv3x3s2(x, w9c, scale, bias):
    """depthwise 3x3/s2/p1 conv + folded BN (CatBottleneck.avd_layer); w9c fp32 [9, C]."""
    B, H, W, C = x.shape
    out = torch.empty((B, (H - 1) // 2 + 1, (W - 1) // 2 + 1, C), dtype=x.dtype, device=x.device)
    _be().dwconv3x3s2(x.contiguous(), w9c, scale, bias, out)
    return out


def avgpool3x3s2(x, out=None):
    B, H, W, C = x.shape
    if out is None:
        out = torch.empty((B, (H - 1) // 2 + 1, (W - 1) // 2 + 1, C), dtype=x.dtype, device=x.device)
    _be().avgpool3x3s2(x.contiguous(), out)
    return out


def global_avgpool(x):
    """[B,H,W,C] (or [B,L,C]) -> [B,C] mean over the middle dims."""
    out = torch.empty((x.shape[0], x.shape[-1]), dtype=x.dtype, device=x.device)
    _be().global_avgpool(x.contiguous(), out)
    return out


def channel_scale(x, gate, addvec=None, addt=None, self_add=False):
    """x * gate[b,c] (+ addvec[b,c]) (+ addt) (+ x)."""
    out = torch.empty_like(x)
    _be().channel_scale(x.contiguous(), gate.contiguous(), None if addvec is None else addvec.contiguous(), None if addt is None else addt.contiguous(), self_add, out)
    return out


def mask_argmax(masks, scores):
    """-> (labels uint8 [B,H,W] = argmax_q(score_q * mask_q), counts int32 [B,Q])."""
    B, Q, H, W = masks.shape
    labels = torch.empty((B, H, W), dtype=torch.uint8, device=masks.device)
    counts = torch.zeros((B, Q), dtype=torch.int32, device=masks.device)
    _be().mask_argmax(masks.contiguous(), scores.contiguous(), labels, counts)
    return labels, counts


def label_resize_bbox(labels, bq_i32, size):
    n = bq_i32.shape[0]
    om = torch.empty((n, size[0], size[1]), dtype=torch.uint8, device=labels.device)
    ob = torch.empty((n, 4), dtype=torch.int32, device=labels.device)
    if n:
        _be().label_resize_bbox(labels.contiguous(), bq_i32.contiguous(), om, ob)
    return om, ob
