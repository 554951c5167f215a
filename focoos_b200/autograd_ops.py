"""torch.autograd.Function wrappers whose forward AND backward run the hand-written kernels (SURVEY §8 a21).

The reference fine-tunes through torch autograd (trainer/trainer.py:757 `losses.backward()`): every op below replaces one
torch op of the reference's training graph together with its aten backward.  Layout is NHWC fp32 (tokens [B,L,C] = NHWC with
H=1); weights stay in the reference's state_dict layout (OIHW / [N,K]) and are re-packed per call (they change every step).

    Conv2dFn          nn.Conv2d                    data grad = forward conv kernel on dy (zero-dilated for stride 2) with
                                                   flipped/transposed weights; weight grad = conv_wgrad kernel
    BatchNormTrainFn  nn.BatchNorm2d.train()       (+ fused residual add and ReLU/SiLU)
    LayerNormFn       nn.LayerNorm(x + res)
    LinearFn          nn.Linear (+ ReLU)
    AddActFn          act(a + b)                   RepVggBlock sum + SiLU, GELU of the AIFI FFN
    MaxPoolFn / AvgPoolFn / ResizeFn               F.max_pool2d(3,2,1) / AvgPool2d(2,2,ceil) / F.interpolate(bilinear)
    AttentionFn       nn.MultiheadAttention core   softmax(QK^T s)V per head
    MSDAFn            ms_deform_attn_core_pytorch  (+ softmax over levels*points, sampling-location arithmetic)

`conv_precision`: "fp32" = SIMT fp32 kernels; "fp32_tc" = tcgen05 split-precision products (fp32 storage) where the shape allows;
"amp" = ONE tcgen05 product on fp16-rounded operands with fp32 accumulation and fp32 storage - the arithmetic class of the reference's own
training (torch.autocast(fp16) + GradScaler, trainer/trainer.py:645,735-771), a third of the tensor work of "fp32_tc".
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch

from . import ops


# ---- conv through either fp32 engine ----------------------------------------------------------------------------------
def _split3_weights(w):
    """[Cout,KH,KW,C] fp32 -> [Cout,KH,KW,3C] fp16 = [W_hi | W_lo | W_hi] (operand layout of ALGO_TCGEN05_SPLIT3)."""
    hi = w.half()
    lo = (w - hi.float()).half()
    return torch.cat([hi, lo, hi], dim=-1).contiguous()


def _to_half_contiguous(t):
    """fp16, contiguous copy of a (possibly permuted) fp32 view in ONE copy kernel (cast + layout change) - `.contiguous().half()` is two"""
    return torch.empty(t.shape, dtype=torch.float16, device=t.device).copy_(t)


def conv_any(x, w_khwc, bias, stride: int, pad: int, precision: str, act=ops.ACT_NONE, x_pair=None, return_pair=False):
    """x NHWC fp32, w [Cout,KH,KW,Cin] fp32 -> NHWC fp32 through the SIMT fp32 or the split-precision tcgen05 kernel.
    x_pair: the [hi|lo] fp16 pair of x if the caller already has it; return_pair: also return the pair used (None on the SIMT path)."""
    B, H, W, C = x.shape
    Cout, KH, KW, _ = w_khwc.shape
    Ho, Wo = (H + 2 * pad - KH) // stride + 1, (W + 2 * pad - KW) // stride + 1
    geom = (stride == 1 and (2 * pad == KH - 1)) or (stride == 2 and KH == 3 and pad == 1 and H % 2 == 0 and W % 2 == 0)  # conv_tc.cu: conv2d_tc_supported
    ok = (precision in ("fp32_tc", "amp") and (x.is_cuda or ops._backend is not None) and C % 32 == 0 and Cout % 4 == 0 and B * Ho * Wo >= 64 and x.is_contiguous()
          and KH == KW and geom and act in (ops.ACT_NONE, ops.ACT_RELU, ops.ACT_SILU))
    if ok and precision == "amp":  # fp16 operands (x_pair carries the fp16 copy of x when the caller already has it), one product, fp32 out
        x16 = x_pair if x_pair is not None else x.half()
        w16 = w_khwc if w_khwc.dtype == torch.float16 else _to_half_contiguous(w_khwc)
        y = ops.conv2d(x16, w16, None, bias, stride=stride, pad=pad, act=act, out_dtype=torch.float32, algo=ops.ALGO_TCGEN05)
        return (y, x16) if return_pair else y
    if ok:
        xp = x_pair if x_pair is not None else ops.split_pair(x)
        y = ops.conv2d(xp, _split3_weights(w_khwc), None, bias, stride=stride, pad=pad, act=act, out_dtype=torch.float32, algo=ops.ALGO_TCGEN05_SPLIT3)
        return (y, xp) if return_pair else y
    if w_khwc.dtype != x.dtype:  # an "amp" caller packed the weight in fp16 but the shape does not take the tensor-core path: the CUDA-core kernel wants one dtype
        w_khwc = w_khwc.to(x.dtype)
    if C % 4:  # the 3-channel image: zero-pad the channel dimension (the SIMT kernel reads 16-byte vectors)
        padc = 4 - C % 4
        x = torch.nn.functional.pad(x, (0, padc))
        w_khwc = torch.nn.functional.pad(w_khwc, (0, padc))
    y = ops.conv2d(x, w_khwc, None, bias, stride=stride, pad=pad, act=act, algo=ops.ALGO_SIMT)
    return (y, None) if return_pair else y


def wgrad_on_tensor_cores(x_shape, dy_shape, KH, KW, stride, pad, precision) -> bool:
    return precision in ("fp32_tc", "amp") and ops._be().conv_wgrad_tc_supported(tuple(x_shape), tuple(dy_shape), KH, KW, stride, pad)


def tc_operand(x, precision):
    """the tensor-core operand form of an fp32 NHWC tensor: its [hi | lo] fp16 pair ("fp32_tc") or its fp16 rounding ("amp")"""
    return x.half() if precision == "amp" else ops.split_pair(x)


def weight_grad(x, dy, KH, KW, stride, pad, precision, x_pair=None, dy_pair=None):
    """dW [Cout,KH,KW,Cin] fp32 of a conv (or a linear as 1x1 over [1,1,M,K]): tensor cores (split precision) when the shape allows, else SIMT fp32.
    x / dy may be None when the corresponding pair is given and the shape takes the tensor-core path."""
    be = ops._be()
    planes = 1 if precision == "amp" else 2
    Cout = dy.shape[-1] if dy is not None else dy_pair.shape[-1] // planes
    xs = tuple(x.shape) if x is not None else (*x_pair.shape[:-1], x_pair.shape[-1] // planes)
    ds = (*xs[:1], (xs[1] + 2 * pad - KH) // stride + 1, (xs[2] + 2 * pad - KW) // stride + 1, Cout)
    dev = (dy if dy is not None else dy_pair).device
    dwk = torch.empty((Cout, KH, KW, xs[-1]), dtype=torch.float32, device=dev)
    if wgrad_on_tensor_cores(xs, ds, KH, KW, stride, pad, precision):
        xp = x_pair if x_pair is not None else tc_operand(x.contiguous(), precision)
        dp = dy_pair if dy_pair is not None else tc_operand(dy.contiguous(), precision)
        (be.conv_wgrad_tc_f16 if precision == "amp" else be.conv_wgrad_tc)(xp, dp, KH, KW, stride, pad, dwk)
    else:
        be.conv_wgrad(x, dy, KH, KW, stride, pad, dwk)
    return dwk


class Conv2dFn(torch.autograd.Function):
    """x [B,H,W,Cin] NHWC, w [Cout,Cin,KH,KW] (state_dict layout), bias [Cout] or None.
    In the tensor-core mode the activation is saved for backward as its [hi|lo] fp16 pair (same bytes as fp32) - the operand format of both
    the forward conv and the weight-gradient kernel - so it is split once, not three times."""

    @staticmethod
    def forward(ctx, x, w, bias, stride, pad, precision):
        x = x.contiguous()
        Cout, _, KH, KW = w.shape
        wk = w.permute(0, 2, 3, 1)
        wk = _to_half_contiguous(wk) if (precision == "amp" and x.shape[-1] % 32 == 0) else wk.contiguous()  # amp: the packed weight straight in fp16 (one kernel)
        y, xp = conv_any(x, wk, bias, stride, pad, precision, return_pair=True)
        keep_pair = xp is not None and wgrad_on_tensor_cores(x.shape, y.shape, KH, KW, stride, pad, precision)
        ctx.save_for_backward(xp if keep_pair else x, w)
        ctx.cfg = (stride, pad, precision, bias is not None, keep_pair, tuple(x.shape))
        return y

    @staticmethod
    def backward(ctx, dy):
        saved, w = ctx.saved_tensors
        stride, pad, precision, has_bias, keep_pair, xshape = ctx.cfg
        dy = dy.contiguous()
        B, H, W, Cin = xshape
        Cout, _, KH, KW = w.shape
        be = ops._be()
        dx = dw = db = None
        dyp = None
        if keep_pair or (precision in ("fp32_tc", "amp") and stride == 1 and ctx.needs_input_grad[0] and Cout % 32 == 0):
            dyp = tc_operand(dy, precision)  # shared by the data-gradient conv and the weight-gradient GEMM
        if ctx.needs_input_grad[0]:
            # data gradient: correlation of (dilated) dy with the spatially flipped, in/out-transposed filter
            wsrc = (w if KH == 1 and KW == 1 else w.flip(2, 3)).permute(1, 2, 3, 0)  # [Cin,KH,KW,Cout] (a 1x1 filter has nothing to flip)
            wt = _to_half_contiguous(wsrc) if (precision == "amp" and Cout % 32 == 0) else wsrc.contiguous()
            g, gp = dy, dyp
            if stride == 2:
                Hd, Wd = H + 2 * pad - KH + 1, W + 2 * pad - KW + 1
                g, gp = torch.empty((B, Hd, Wd, Cout), dtype=torch.float32, device=dy.device), None
                be.dilate2(dy, g)
            elif stride != 1:
                raise NotImplementedError("focoos_b200: conv data gradient for stride > 2")
            dx = conv_any(g, wt, None, 1, KH - 1 - pad, precision, x_pair=gp)
            assert tuple(dx.shape) == tuple(xshape), (dx.shape, xshape)
        if ctx.needs_input_grad[1]:
            if keep_pair:
                dw = weight_grad(None, dy, KH, KW, stride, pad, precision, x_pair=saved, dy_pair=dyp).permute(0, 3, 1, 2)
            else:
                dw = weight_grad(saved, dy, KH, KW, stride, pad, precision).permute(0, 3, 1, 2)
        if has_bias and ctx.needs_input_grad[2]:
            db = torch.empty(Cout, dtype=torch.float32, device=dy.device)
            be.colsum(dy.reshape(-1, Cout), db)
        return dx, dw, db, None, None, None


class BatchNormTrainFn(torch.autograd.Function):
    """y = act(BN_batchstats(x) + res); running statistics updated in place (momentum 0.1, unbiased variance) like nn.BatchNorm2d.train()."""

    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, res, act, eps, momentum):
        x = x.contiguous()
        C = x.shape[-1]
        x2 = x.reshape(-1, C)
        y = torch.empty_like(x)
        mean = torch.empty(C, dtype=torch.float32, device=x.device)
        rstd = torch.empty(C, dtype=torch.float32, device=x.device)
        r2 = None if res is None else res.contiguous().reshape(-1, C)
        ops._be().bn_train_fwd(x2, gamma, beta, r2, act, eps, momentum, running_mean, running_var, mean, rstd, y.reshape(-1, C))
        # the ReLU mask is recomputed from x (sign of the normalised value) unless a residual was added before the activation: saves the output from
        # being kept alive and two passes over it in backward
        ctx.save_for_backward(x, gamma, beta, mean, rstd, y if (act != ops.ACT_NONE and res is not None) else None)
        ctx.cfg = (act, res is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, gamma, beta, mean, rstd, y = ctx.saved_tensors
        act, has_res = ctx.cfg
        C = x.shape[-1]
        dy = dy.contiguous()
        dx = torch.empty_like(x)
        dres = torch.empty_like(x) if has_res else None
        dgamma = torch.empty(C, dtype=torch.float32, device=x.device)
        dbeta = torch.empty(C, dtype=torch.float32, device=x.device)
        ops._be().bn_train_bwd(x.reshape(-1, C), dy.reshape(-1, C), None if y is None else y.reshape(-1, C), gamma, beta, mean, rstd, act, dx.reshape(-1, C),
                               None if dres is None else dres.reshape(-1, C), dgamma, dbeta)
        return dx, dgamma, dbeta, None, None, dres, None, None, None


class SyncBatchNormTrainFn(torch.autograd.Function):
    """BatchNormTrainFn with the statistics taken over ALL data-parallel ranks - what torch.nn.SyncBatchNorm (trainer/trainer.py:334) computes:
    forward: local mean / biased variance -> all_gather with the local row counts -> combined mean / variance (aten batch_norm_gather_stats_with_counts);
    backward: local sum(g), sum(g * xhat) -> all_reduce -> dx with the global sums over the global row count; dgamma / dbeta stay LOCAL (the gradient
    exchange sums them like every other parameter gradient).  Two small collectives per layer and pass; everything else is the single-GPU kernels."""

    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, res, act, eps, momentum, group):
        import torch.distributed as dist
        x = x.contiguous()
        C = x.shape[-1]
        x2 = x.reshape(-1, C)
        be = ops._be()
        stats = torch.empty((2 * C + 1,), dtype=torch.float32, device=x.device)
        be.bn_stats(x2, stats[:C], stats[C:2 * C])
        stats[2 * C:].fill_(float(x2.shape[0]))  # a fill kernel: no host -> device copy in the middle of the launch stream
        world = dist.get_world_size(group)
        allst = torch.empty((world, 2 * C + 1), dtype=torch.float32, device=x.device)
        dist.all_gather_into_tensor(allst.view(-1), stats, group=group)
        mean = torch.empty(C, dtype=torch.float32, device=x.device)
        rstd = torch.empty(C, dtype=torch.float32, device=x.device)
        inv_total = torch.empty(1, dtype=torch.float32, device=x.device)
        # global moments, running statistics (unbiased variance over the GLOBAL count) and 1 / total in one launch; nothing of it is read back by the host
        be.bn_sync_combine(allst, eps, momentum, running_mean, running_var, mean, rstd, inv_total)
        y = torch.empty_like(x)
        r2 = None if res is None else res.contiguous().reshape(-1, C)
        be.bn_apply(x2, mean, rstd, gamma, beta, r2, act, y.reshape(-1, C))
        ctx.save_for_backward(x, gamma, beta, mean, rstd, y if (act != ops.ACT_NONE and res is not None) else None, inv_total)
        ctx.cfg = (act, res is not None, group)
        return y

    @staticmethod
    def backward(ctx, dy):
        import torch.distributed as dist
        x, gamma, beta, mean, rstd, y, inv_total = ctx.saved_tensors
        act, has_res, group = ctx.cfg
        C = x.shape[-1]
        dy = dy.contiguous()
        be = ops._be()
        sums = torch.empty((2, C), dtype=torch.float32, device=x.device)
        y2 = None if y is None else y.reshape(-1, C)
        be.bn_bwd_reduce(x.reshape(-1, C), dy.reshape(-1, C), y2, gamma, beta, mean, rstd, act, sums[0], sums[1])
        local = sums.clone()
        dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
        sums.mul_(inv_total)  # the global sums over the global row count, scaled on the device (the kernel's own factor is 1): sum * (1 / total) is the same product it forms
        dx = torch.empty_like(x)
        dres = torch.empty_like(x) if has_res else None
        be.bn_bwd_apply(x.reshape(-1, C), dy.reshape(-1, C), y2, gamma, beta, mean, rstd, sums[0], sums[1], 1.0, act, dx.reshape(-1, C),
                        None if dres is None else dres.reshape(-1, C))
        return dx, local[1], local[0], None, None, dres, None, None, None, None


class FrozenBatchNormFn(torch.autograd.Function):
    """FrozenBatchNorm2d (nn/backbone/resnet.py:226-250; TrainerArgs.freeze_bn): the affine of the RUNNING statistics in training too - nothing is
    updated, weight / bias receive no gradient; dx = gamma * rstd * g."""

    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, res, act, eps):
        x = x.contiguous()
        C = x.shape[-1]
        rstd = torch.rsqrt(running_var + eps)
        y = torch.empty_like(x)
        r2 = None if res is None else res.contiguous().reshape(-1, C)
        ops._be().bn_apply(x.reshape(-1, C), running_mean, rstd, gamma, beta, r2, act, y.reshape(-1, C))
        ctx.save_for_backward(x, gamma, beta, running_mean.clone(), rstd, y if (act != ops.ACT_NONE and res is not None) else None)
        ctx.cfg = (act, res is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, gamma, beta, mean, rstd, y = ctx.saved_tensors
        act, has_res = ctx.cfg
        C = x.shape[-1]
        dy = dy.contiguous()
        zero = torch.zeros(C, dtype=torch.float32, device=x.device)
        dx = torch.empty_like(x)
        dres = torch.empty_like(x) if has_res else None
        ops._be().bn_bwd_apply(x.reshape(-1, C), dy.reshape(-1, C), None if y is None else y.reshape(-1, C), gamma, beta, mean, rstd, zero, zero, 0.0, act, dx.reshape(-1, C),
                               None if dres is None else dres.reshape(-1, C))
        return dx, None, None, None, None, dres, None, None


class LayerNormFn(torch.autograd.Function):
    """LayerNorm(x + res) * gamma + beta."""

    @staticmethod
    def forward(ctx, x, res, gamma, beta, eps):
        x = x.contiguous()
        res = None if res is None else res.contiguous()
        ctx.save_for_backward(x, res, gamma)
        ctx.eps = eps
        return ops.layernorm(x, gamma, beta, residual=res, eps=eps)

    @staticmethod
    def backward(ctx, dy):
        x, res, gamma = ctx.saved_tensors
        C = x.shape[-1]
        dx = torch.empty_like(x)
        dg = torch.empty(C, dtype=torch.float32, device=x.device)
        db = torch.empty(C, dtype=torch.float32, device=x.device)
        ops._be().layernorm_bwd(x.reshape(-1, C), None if res is None else res.reshape(-1, C), gamma, dy.contiguous().reshape(-1, C), ctx.eps, dx.reshape(-1, C), dg, db)
        return dx, (dx if res is not None else None), dg, db, None


class LinearFn(torch.autograd.Function):
    """y = act(x @ w.T + b), act in {none, relu}; x [..., K], w [N, K]."""

    @staticmethod
    def forward(ctx, x, w, bias, act, precision):
        assert act in (ops.ACT_NONE, ops.ACT_RELU)
        x = x.contiguous()
        K, N = x.shape[-1], w.shape[0]
        x4 = x.reshape(1, 1, -1, K)
        w4 = w.reshape(N, 1, 1, K)
        w4 = _to_half_contiguous(w4) if (precision == "amp" and K % 32 == 0) else w4.contiguous()
        y4, xp = conv_any(x4, w4, bias, 1, 0, precision, act=act, return_pair=True)
        y = y4.reshape(*x.shape[:-1], N)
        keep_pair = xp is not None and wgrad_on_tensor_cores(x4.shape, y4.shape, 1, 1, 1, 0, precision)
        ctx.save_for_backward(xp if keep_pair else x, w, y if act == ops.ACT_RELU else None)
        ctx.cfg = (act, precision, bias is not None, keep_pair, tuple(x.shape))
        return y

    @staticmethod
    def backward(ctx, dy):
        saved, w, y = ctx.saved_tensors
        act, precision, has_bias, keep_pair, xshape = ctx.cfg
        K, N = xshape[-1], w.shape[0]
        be = ops._be()
        g = dy.contiguous()
        if act == ops.ACT_RELU:  # dy * relu'(y): y > 0 <=> pre-activation > 0
            gm = torch.empty_like(g)
            be.add_act(y, None, g, ops.ACT_RELU, gm)
            g = gm
        g2 = g.reshape(1, 1, -1, N)
        gp = tc_operand(g2, precision) if (keep_pair or (precision in ("fp32_tc", "amp") and N % 32 == 0 and g2.shape[2] >= 64 and ctx.needs_input_grad[0])) else None
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            wt = _to_half_contiguous(w.t()) if (precision == "amp" and N % 32 == 0) else w.t().contiguous()
            dx = conv_any(g2, wt.reshape(K, 1, 1, N), None, 1, 0, precision, x_pair=gp).reshape(xshape)
        if ctx.needs_input_grad[1]:
            if keep_pair:
                dw = weight_grad(None, g2, 1, 1, 1, 0, precision, x_pair=saved, dy_pair=gp).reshape(N, K)
            else:
                dw = weight_grad(saved.reshape(1, 1, -1, K), g2, 1, 1, 1, 0, precision).reshape(N, K)
        if has_bias and ctx.needs_input_grad[2]:
            db = torch.empty(N, dtype=torch.float32, device=g.device)
            be.colsum(g2.reshape(-1, N), db)
        return dx, dw, db, None, None


class AddActFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b, act):
        a = a.contiguous()
        b = None if b is None else b.contiguous()
        ctx.save_for_backward(a, b)
        ctx.act = act
        out = torch.empty_like(a)
        ops._be().add_act(a, b, None, act, out)
        return out

    @staticmethod
    def backward(ctx, dy):
        a, b = ctx.saved_tensors
        g = torch.empty_like(a)
        ops._be().add_act(a, b, dy.contiguous(), ctx.act, g)
        return g, (g if b is not None else None), None


class MaxPoolFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        x = x.contiguous()
        ctx.save_for_backward(x)
        return ops.maxpool3x3s2(x)

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        dx = torch.empty_like(x)
        ops._be().maxpool_bwd(x, dy.contiguous(), dx)
        return dx


class AvgPoolFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        ctx.shape = x.shape
        return ops.avgpool2x2(x.contiguous())

    @staticmethod
    def backward(ctx, dy):
        dx = torch.empty(ctx.shape, dtype=torch.float32, device=dy.device)
        ops._be().avgpool_bwd(dy.contiguous(), dx)
        return dx


class ResizeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, size):
        ctx.shape = x.shape
        return ops.resize_bilinear(x.contiguous(), size)

    @staticmethod
    def backward(ctx, dy):
        dx = torch.empty(ctx.shape, dtype=torch.float32, device=dy.device)
        ops._be().resize_bwd(dy.contiguous(), dx)
        return dx, None


class AttentionFn(torch.autograd.Function):
    """q [B,Lq,C], k/v [B,Lk,C] (already projected), heads of 32 channels."""

    @staticmethod
    def forward(ctx, q, k, v, heads, scale, split=False):
        q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        o = ops.attention(q, k, v, heads, scale, split=split)
        ctx.save_for_backward(q, k, v, o)
        ctx.cfg = (heads, scale)
        return o

    @staticmethod
    def backward(ctx, do):
        q, k, v, o = ctx.saved_tensors
        heads, scale = ctx.cfg
        dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        ops._be().attention_bwd(q, k, v, o, do.contiguous(), heads, scale, dq, dk, dv)
        return dq, dk, dv, None, None, None


class MSDAFn(torch.autograd.Function):
    """value [B,S,heads*32], oa [B,Q,heads*L*P*3] (offsets then logits), ref [B,Q,4] (no gradient: detached in the reference)."""

    @staticmethod
    def forward(ctx, value, oa, ref, shapes, num_points, heads):
        value, oa, ref = value.contiguous(), oa.contiguous(), ref.contiguous()
        ctx.save_for_backward(value, oa, ref)
        ctx.cfg = (tuple(tuple(s) for s in shapes), num_points, heads)
        return ops.msda(value, oa, ref, shapes, num_points, heads, out_dtype=torch.float32)

    @staticmethod
    def backward(ctx, do):
        value, oa, ref = ctx.saved_tensors
        shapes, P, heads = ctx.cfg
        dvalue = torch.zeros_like(value)
        doa = torch.empty_like(oa)
        ops._be().msda_bwd(value, oa, ref, do.contiguous(), shapes, P, heads, dvalue, doa)
        return dvalue, doa, None, None, None, None


def conv2d(x, w, bias=None, stride=1, pad=0, precision="fp32"):
    return Conv2dFn.apply(x, w, bias, stride, pad, precision)


def batch_norm_train(x, bn: torch.nn.BatchNorm2d, res=None, act=ops.ACT_NONE, sync_group=None, frozen=False):
    """train-mode BatchNorm2d: batch statistics (default), statistics over all ranks of `sync_group` (SyncBatchNorm), or the frozen running statistics"""
    if frozen:
        return FrozenBatchNormFn.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, res, act, bn.eps)
    with torch.no_grad():
        bn.num_batches_tracked += 1  # nn.BatchNorm2d.train() bookkeeping (a state_dict buffer)
    momentum = 0.1 if bn.momentum is None else bn.momentum
    if sync_group is not None:
        return SyncBatchNormTrainFn.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, res, act, bn.eps, momentum, None if sync_group is True else sync_group)
    return BatchNormTrainFn.apply(x, bn.weight, bn.bias, bn.running_mean, bn.running_var, res, act, bn.eps, momentum)


def layer_norm(x, ln: torch.nn.LayerNorm, res=None):
    return LayerNormFn.apply(x, res, ln.weight, ln.bias, ln.eps)


def linear(x, w, bias=None, act=ops.ACT_NONE, precision="fp32"):
    return LinearFn.apply(x, w, bias, act, precision)
