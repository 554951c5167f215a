"""Per-operator CPU references with the SAME signatures as `focoos_b200.ops.CudaBackend`.

TEST INFRASTRUCTURE — NOT PRODUCT CODE (see oracle/detr_oracle.py header for the import rules).
Two uses: (1) `-m gpu` tests compare each CUDA kernel against these on seeded inputs;
(2) `-m "not gpu"` tests install `RefBackend()` as `focoos_b200.ops._backend` to run the HOST
orchestration (weight packing, fused NHWC graph, level ordering, slices) on a GPU-less machine
and compare it with the golden fixtures.  Everything computes in fp32 with plain torch ops
(F.conv2d, F.grid_sample, ...) — i.e. the reference's own library calls — and rounds to the output
dtype at the end.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F


def _act(x, act):
    return [lambda v: v, F.relu, F.silu, F.gelu, torch.sigmoid][act](x)


def _f(t):
    return None if t is None else t.float()


def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _nhwc(t):
    return t.permute(0, 2, 3, 1)


def _act_bw(act, z):
    return {0: lambda t: t, 1: F.relu, 2: F.silu, 3: F.gelu}[act](z)


def _bn_g(x2d, dy2d, y2d, gamma, beta, mean, rstd, act):
    xh = (x2d - mean) * rstd
    g = dy2d
    if act == 1:
        g = dy2d * ((y2d if y2d is not None else xh * gamma + beta) > 0)
    elif act == 2:
        z = (xh * gamma + beta).detach().requires_grad_(True)
        with torch.enable_grad():
            (g,) = torch.autograd.grad(F.silu(z), z, dy2d)
    return xh, g


def _via_autograd(fn, x, dy):
    xx = x.detach().clone().requires_grad_(True)
    with torch.enable_grad():
        (g,) = torch.autograd.grad(fn(xx), xx, dy)
    return g


def _mha_core(q, k, v, heads, scale):
    B, Lq, C = q.shape
    hd = C // heads
    qh, kh, vh = (t.reshape(B, -1, heads, hd).transpose(1, 2) for t in (q, k, v))
    p = torch.softmax(qh @ kh.transpose(-1, -2) * scale, -1)
    return (p @ vh).transpose(1, 2).reshape(B, Lq, C)


class RefBackend:
    def stem_conv(self, img, w, scale, bias, mean, std, act, out):
        if img.dtype == torch.uint8:
            img = img.permute(0, 3, 1, 2).float()
        x = (img - torch.tensor(mean).view(1, 3, 1, 1)) / torch.tensor(std).view(1, 3, 1, 1)
        y = F.conv2d(x, w.permute(0, 3, 1, 2).float(), None, 2, 1)
        if scale is not None:
            y = y * scale.view(1, -1, 1, 1)
        if bias is not None:
            y = y + bias.view(1, -1, 1, 1)
        if hasattr(out, "hi"):
            self._pair_write(out, _act(y, act).permute(0, 2, 3, 1))
            return
        out.copy_(_act(y, act).permute(0, 2, 3, 1).to(out.dtype))

    def conv2d(self, x, w, scale, bias, stride, pad, act, residual, out, algo):
        if algo == 3:  # split-precision operands: x = [hi|lo], w = [W_hi|W_lo|W_hi] -> the fp32 values they encode
            C = x.shape[-1] // 2
            x = x[..., :C].float() + x[..., C:].float()
            w = w[..., :C].float() + w[..., C:2 * C].float()
        y = F.conv2d(x.float().permute(0, 3, 1, 2), w.float().permute(0, 3, 1, 2), None, stride, pad)
        if scale is not None:
            y = y * scale.view(1, -1, 1, 1)
        if bias is not None:
            y = y + bias.view(1, -1, 1, 1)
        y = y.permute(0, 2, 3, 1)
        post = bool(act & 16)  # FB200_ACT_RESIDUAL_AFTER
        r = 0.0 if residual is None else residual.float()
        y = _act(y, act & 15) + r if post else _act(y + r, act & 15)
        out.copy_(y.to(out.dtype))

    def conv2d_per_image(self, x, w, act, out, algo):
        for b in range(x.shape[0]):
            self.conv2d(x[b:b + 1], w[b], None, None, 1, (w.shape[2] - 1) // 2, act, None, out[b:b + 1], algo)

    @staticmethod
    def _pair_write(pr, v):
        hi = v.half()
        pr.hi.copy_(hi)
        pr.lo.copy_((v - hi.float()).half())

    def conv2d_pair(self, x, w3, scale, bias, stride, pad, act, residual, out):
        """the fp32 conv the pair operands encode; pair outputs are re-split exactly as the CUDA epilogue does (hi = fp16(v), lo = fp16(v - hi))"""
        C = x.C
        xv = x.float()
        w = w3[..., :C].float() + w3[..., C:2 * C].float()
        y = F.conv2d(xv.permute(0, 3, 1, 2), w.permute(0, 3, 1, 2), None, stride, pad)
        if scale is not None:
            y = y * scale.view(1, -1, 1, 1)
        if bias is not None:
            y = y + bias.view(1, -1, 1, 1)
        y = y.permute(0, 2, 3, 1)
        r = 0.0 if residual is None else residual.float()
        y = _act(y, act & 15) + r if (act & 16) else _act(y + r, act & 15)
        if hasattr(out, "hi"):
            self._pair_write(out, y)
        else:
            out.copy_(y)

    def linear_rowmax(self, x2d, w, bias, out):
        y = x2d.float() @ w.float().t()
        if bias is not None:
            y = y + bias
        out.copy_(y.max(-1).values)

    def linear_rowmax_pair(self, xp, w3, bias, out):
        K = xp.C
        w = w3[..., :K].float() + w3[..., K:2 * K].float()
        y = xp.float().reshape(-1, K) @ w.reshape(w.shape[0], K).t()
        out.copy_((y + (bias if bias is not None else 0.0)).max(-1).values)

    def image_resize(self, images, out):
        x = images.permute(0, 3, 1, 2).float() if images.dtype == torch.uint8 else images.float()
        out.copy_(F.interpolate(x, size=tuple(out.shape[2:]), mode="bilinear", align_corners=False))

    def pair_pool(self, mode, x, out):
        v = x.float().permute(0, 3, 1, 2)
        if mode == 0:
            y = F.max_pool2d(v, 3, 2, 1)
        elif mode == 1:
            y = F.avg_pool2d(v, 2, 2, 0, ceil_mode=True)
        else:
            y = F.interpolate(v, size=(out.shape[1], out.shape[2]), mode="bilinear", align_corners=False)
        self._pair_write(out, y.permute(0, 2, 3, 1))

    def split_pair(self, x, out):
        C = x.shape[-1]
        hi = x.half()
        out[..., :C] = hi
        out[..., C:] = (x - hi.float()).half()

    def maxpool3x3s2(self, x, out):
        out.copy_(F.max_pool2d(x.float().permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1).to(out.dtype))

    def avgpool2x2(self, x, out):
        out.copy_(F.avg_pool2d(x.float().permute(0, 3, 1, 2), 2, 2, 0, ceil_mode=True).permute(0, 2, 3, 1).to(out.dtype))

    def resize_bilinear(self, x, out):
        y = F.interpolate(x.float().permute(0, 3, 1, 2), size=(out.shape[1], out.shape[2]), mode="bilinear", align_corners=False)
        out.copy_(y.permute(0, 2, 3, 1).to(out.dtype))

    def add(self, a, b, out):
        C = a.shape[-1]
        rows, brows = a.numel() // C, b.numel() // C
        out.copy_((a.float().reshape(rows // brows, brows, C) + b.float().reshape(1, brows, C)).reshape(a.shape).to(out.dtype))

    def layernorm(self, x, res, gamma, beta, out, eps):
        v = x.float() if res is None else x.float() + res.float()
        out.copy_(F.layer_norm(v, (v.shape[-1],), gamma, beta, eps).to(out.dtype))

    def attention(self, q, k, v, out, heads, scale, split=False):
        B, Lq, C = q.shape
        Lk = k.shape[1]
        hd = C // heads
        qh = q.float().reshape(B, Lq, heads, hd).transpose(1, 2)
        kh = k.float().reshape(B, Lk, heads, hd).transpose(1, 2)
        vh = v.float().reshape(B, Lk, heads, hd).transpose(1, 2)
        a = torch.softmax((qh @ kh.transpose(-1, -2)) * scale, dim=-1)
        o = (a @ vh).transpose(1, 2).reshape(B, Lq, C)
        if hasattr(out, "hi"):
            self._pair_write(out, o)
        else:
            out.copy_(o.to(out.dtype))

    def msda(self, value, oa, ref, shapes, P, heads, out):
        B, S, C = value.shape
        Q = oa.shape[1]
        L = len(shapes)
        hd = C // heads
        oa = oa.float()
        off = oa[..., : heads * L * P * 2].reshape(B, Q, heads, L, P, 2)
        aw = torch.softmax(oa[..., heads * L * P * 2 : heads * L * P * 3].reshape(B, Q, heads, L * P), -1).reshape(B, Q, heads, L, P)
        r = ref.float().reshape(B, Q, 1, 1, 1, 4)
        loc = r[..., :2] + off / P * r[..., 2:] * 0.5
        val = value.float().reshape(B, S, heads, hd)
        vals = val.split([h * w for h, w in shapes], dim=1)
        grids = 2 * loc - 1
        sampled = []
        for lid, (H_, W_) in enumerate(shapes):
            vl = vals[lid].flatten(2).transpose(1, 2).reshape(B * heads, hd, H_, W_)
            g = grids[:, :, :, lid].transpose(1, 2).flatten(0, 1)
            sampled.append(F.grid_sample(vl, g, mode="bilinear", padding_mode="zeros", align_corners=False))
        awt = aw.transpose(1, 2).reshape(B * heads, 1, Q, L * P)
        o = (torch.stack(sampled, dim=-2).flatten(-2) * awt).sum(-1).view(B, heads * hd, Q).transpose(1, 2)
        if hasattr(out, "hi"):
            self._pair_write(out, o)
        else:
            out.copy_(o.to(out.dtype))

    def layernorm_ex(self, x, res, gather, valid, fill, gamma, beta, eps, M, out_f32, out_pair, pos, out_pair_pos):
        """fb200_layernorm_ex: optional valid-mask fill and top-k gather of the source rows, LayerNorm, outputs as fp32 / pair / pair(y + pos)"""
        C = x.shape[-1]
        v = x.float()
        if valid is not None:
            S = valid.numel()
            v = torch.where(valid.bool().view(1, S, 1), v.reshape(-1, S, C), fill.view(1, 1, C))
        if gather is not None:
            v = v.reshape(gather.shape[0], -1, C)
            v = torch.gather(v, 1, gather.long().unsqueeze(-1).expand(-1, -1, C))
        v = v.reshape(M, C)
        if res is not None:
            v = v + res.float().reshape(M, C)
        y = F.layer_norm(v, (C,), gamma, beta, eps)
        if out_f32 is not None:
            out_f32.copy_(y.reshape(out_f32.shape))
        if out_pair is not None:
            self._pair_write(out_pair, y.reshape(out_pair.shape))
        if out_pair_pos is not None:
            pr = pos.numel() // C
            yp = (y.reshape(M // pr, pr, C) + pos.float().reshape(1, pr, C)).reshape(out_pair_pos.shape)
            self._pair_write(out_pair_pos, yp)

    def split_pair_ex(self, x, act, pos, out_pair, out_pair_pos):
        C = x.shape[-1]
        v = x.float()
        if out_pair is not None:
            self._pair_write(out_pair, _act(v, act & 15))
        if out_pair_pos is not None:
            pr = pos.numel() // C
            rows = v.numel() // C
            self._pair_write(out_pair_pos, (v.reshape(rows // pr, pr, C) + pos.float().reshape(1, pr, C)).reshape(v.shape))

    def box_refine_qpos(self, delta, ref_in, ref_out, w0, b0, qpos_pair):
        r = ref_in.float()
        if delta is not None:
            x = r.clamp(0, 1)
            r = torch.sigmoid(delta.float() + torch.log(x.clamp(min=1e-5) / (1 - x).clamp(min=1e-5)))
            ref_out.copy_(r)
        if qpos_pair is not None:
            self._pair_write(qpos_pair, torch.relu(r @ w0.float().t() + b0.float()))

    def sigmoid_rows(self, x, out):
        out.copy_(torch.sigmoid(x.float()))

    def row_select(self, x, valid, fill, out):
        C = x.shape[-1]
        S = valid.numel()
        xv = x.float().reshape(-1, S, C)
        m = valid.bool().view(1, S, 1)
        out.copy_(torch.where(m, xv, fill.view(1, 1, C)).reshape(x.shape).to(out.dtype))

    def rowmax(self, x, out):
        out.copy_(x.float().max(-1).values)

    def topk(self, x, K, out_idx, out_val):
        v, i = torch.sort(x, dim=-1, descending=True, stable=True)
        out_idx.copy_(i[:, :K].to(torch.int32))
        if out_val is not None:
            out_val.copy_(v[:, :K])

    def gather_rows(self, src, idx, out):
        out.copy_(src.gather(1, idx.long().unsqueeze(-1).expand(-1, -1, src.shape[-1])))

    def box_op(self, mode, x, ref, idx, out):
        if mode == 0:
            out.copy_(torch.sigmoid(x))
        elif mode == 1:
            r = ref.clip(0.0, 1.0)
            out.copy_(torch.sigmoid(x + torch.log(r.clip(min=1e-5) / (1 - r).clip(min=1e-5))))
        elif mode == 2:
            out.copy_(x + ref[idx.long().reshape(-1)].reshape(x.shape))
        else:
            xc, yc, w, h = x.unbind(-1)
            out.copy_(torch.stack([xc - 0.5 * w, yc - 0.5 * h, xc + 0.5 * w, yc + 0.5 * h], -1))

    def detr_postprocess(self, scores, boxes, sizes, K, thr, out_scores, out_labels, out_boxes, out_query, out_count):
        B, Q, C = scores.shape
        for b in range(B):
            v, i = torch.sort(scores[b].flatten(), descending=True, stable=True)
            v, i = v[:K], i[:K]
            q = i // C
            bx = boxes[b][q].clone()
            bx[:, 0::2] *= float(sizes[b, 1])
            bx[:, 1::2] *= float(sizes[b, 0])
            out_scores[b] = v
            out_labels[b] = (i % C).to(torch.int32)
            out_query[b] = q.to(torch.int32)
            out_boxes[b] = bx.round().to(torch.int32)
            out_count[b] = int((v > thr).sum())


    def detr_eval_postprocess(self, scores, boxes, sizes, K, out_scores, out_labels, out_boxes, out_count):
        """fai_detr/processor.py:121-144 + detector_postprocess :19-57 per image (top-k, scale, clip, drop empty boxes), compacted."""
        B, Q, C = scores.shape
        for b in range(B):
            v, i = torch.sort(scores[b].flatten(), descending=True, stable=True)
            v, i = v[:K], i[:K]
            bx = boxes[b][i // C].clone()
            H, W = float(sizes[b, 0]), float(sizes[b, 1])
            bx[:, 0::2] = (bx[:, 0::2] * W).clamp(0, W)
            bx[:, 1::2] = (bx[:, 1::2] * H).clamp(0, H)
            keep = ((bx[:, 2] - bx[:, 0]) > 0) & ((bx[:, 3] - bx[:, 1]) > 0)
            n = int(keep.sum())
            out_scores[b, :n] = v[keep]
            out_labels[b, :n] = (i % C)[keep].to(torch.int32)
            out_boxes[b, :n] = bx[keep]
            out_count[b] = n

    # ---- MaskFormer-family operators -------------------------------------------------------------------------
    def upsample_nearest_add(self, y, cur, out):
        up = F.interpolate(y.float().permute(0, 3, 1, 2), size=(cur.shape[1], cur.shape[2]), mode="nearest").permute(0, 2, 3, 1)
        out.copy_((cur.float() + up).to(out.dtype))

    def attn_mask_build(self, x, Q, mask, allowed):
        B, h, w, Qp = x.shape
        m = (x.float().reshape(B, h * w, Qp)[:, :, :Q] < 0).permute(0, 2, 1)  # [B,Q,hw], True = not allowed
        mask.zero_()
        mask[:, :, : h * w] = m.to(torch.uint8)
        allowed.copy_((~m).sum(-1).to(torch.int32))

    def attention_masked(self, q, k, v, mask, allowed, out, heads, scale):
        B, Lq, C = q.shape
        Lk = k.shape[1]
        hd = C // heads
        qh = q.float().reshape(B, Lq, heads, hd).transpose(1, 2)
        kh = k.float().reshape(B, Lk, heads, hd).transpose(1, 2)
        vh = v.float().reshape(B, Lk, heads, hd).transpose(1, 2)
        m = mask[:, :, :Lk].bool() & (allowed > 0).unsqueeze(-1)
        s = (qh @ kh.transpose(-1, -2)) * scale
        s = s.masked_fill(m.unsqueeze(1), float("-inf"))
        out.copy_((torch.softmax(s, -1) @ vh).transpose(1, 2).reshape(B, Lq, C).to(out.dtype))

    def attention_masked_split(self, q, k, v, mask, allowed, out, heads, scale):
        """fb200_attention_masked_split: k / v as fp32 tensors or as Pairs (the fp32 values they encode)"""
        kf = k.float() if hasattr(k, "hi") else k
        vf = v.float() if hasattr(v, "hi") else v
        self.attention_masked(q, kf, vf, mask, allowed, out, heads, scale)

    def softmax_drop_last(self, x, out):
        out.copy_(F.softmax(x.float(), dim=-1)[..., :-1])

    def mask_sigmoid_upsample(self, x, Q, out):
        p = torch.sigmoid(x.float()[..., :Q]).permute(0, 3, 1, 2)
        out.copy_(F.interpolate(p, size=(out.shape[2], out.shape[3]), mode="bilinear", align_corners=False))

    def mask_sigmoid_upsample_argmax(self, x, Q, scores, labels, counts):
        B, h, w, _ = x.shape
        probs = torch.empty((B, Q, labels.shape[1], labels.shape[2]), dtype=torch.float32)
        self.mask_sigmoid_upsample(x, Q, probs)
        self.mask_argmax(probs, scores, labels, counts)

    def mask_sigmoid_upsample_stats(self, x, Q, size, thr, count, psum):
        probs = torch.empty((x.shape[0], Q, size[0], size[1]), dtype=torch.float32)
        self.mask_sigmoid_upsample(x, Q, probs)
        self.mask_stats(probs, thr, count, psum)

    def mask_sigmoid_upsample_select(self, x, bq, out):
        Q = int(bq[:, 1].max()) + 1
        probs = torch.empty((x.shape[0], Q, out.shape[1], out.shape[2]), dtype=torch.float32)
        self.mask_sigmoid_upsample(x, Q, probs)
        for i in range(bq.shape[0]):
            out[i] = probs[int(bq[i, 0]), int(bq[i, 1])]

    def mask_stats(self, masks, thr, count, psum):
        b = masks >= thr
        count.copy_(b.sum(dim=(-2, -1)).to(torch.int32))
        psum.copy_((masks * b).sum(dim=(-2, -1)))

    def mask_resize_bbox(self, masks, bq, thr, out_masks, out_bbox):
        for i in range(bq.shape[0]):
            b, q = int(bq[i, 0]), int(bq[i, 1])
            m = (masks[b, q] >= thr).float()[None, None]
            r = F.interpolate(m, size=(out_masks.shape[1], out_masks.shape[2]), mode="bilinear", align_corners=False)[0, 0].bool()
            out_masks[i] = r.to(torch.uint8)
            rows, cols = r.any(1).nonzero(), r.any(0).nonzero()
            out_bbox[i] = torch.tensor([int(cols[0]), int(rows[0]), int(cols[-1]), int(rows[-1])] if len(rows) else [0, 0, 0, 0], dtype=torch.int32)

    # ---- BiSeNetFormer-family operators ----------------------------------------------------------------------
    def dwconv3x3s2(self, x, w9c, scale, bias, out):
        C = x.shape[-1]
        w = w9c.t().reshape(C, 1, 3, 3)
        y = F.conv2d(x.float().permute(0, 3, 1, 2), w, None, 2, 1, 1, C) * scale.view(1, -1, 1, 1) + bias.view(1, -1, 1, 1)
        out.copy_(y.permute(0, 2, 3, 1).to(out.dtype))

    def avgpool3x3s2(self, x, out):
        out.copy_(F.avg_pool2d(x.float().permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1).to(out.dtype))

    def global_avgpool(self, x, out):
        B, C = x.shape[0], x.shape[-1]
        out.copy_(x.float().reshape(B, -1, C).mean(1).to(out.dtype))

    def channel_scale(self, x, gate, addvec, addt, self_add, out):
        B, C = x.shape[0], x.shape[-1]
        xs = x.float().reshape(B, -1, C)
        y = xs * gate.float().view(B, 1, C)
        if addvec is not None:
            y = y + addvec.float().view(B, 1, C)
        if addt is not None:
            y = y + addt.float().reshape(B, -1, C)
        if self_add:
            y = y + xs
        out.copy_(y.reshape(x.shape).to(out.dtype))

    def mask_argmax(self, masks, scores, labels, counts):
        B, Q = scores.shape
        lab = (scores.view(B, Q, 1, 1) * masks).argmax(dim=1)
        labels.copy_(lab.to(torch.uint8))
        for b in range(B):
            counts[b] = torch.bincount(lab[b].flatten(), minlength=Q).to(torch.int32)

    def label_resize_bbox(self, labels, bq, out_masks, out_bbox):
        for i in range(bq.shape[0]):
            b, q = int(bq[i, 0]), int(bq[i, 1])
            m = (labels[b] == q).float()[None, None]
            r = F.interpolate(m, size=(out_masks.shape[1], out_masks.shape[2]), mode="bilinear", align_corners=False)[0, 0].bool()
            out_masks[i] = r.to(torch.uint8)
            rows, cols = r.any(1).nonzero(), r.any(0).nonzero()
            out_bbox[i] = torch.tensor([int(cols[0]), int(rows[0]), int(cols[-1]), int(rows[-1])] if len(rows) else [0, 0, 0, 0], dtype=torch.int32)

    # ---- backward / training-mode operators (autograd_ops.py and the training graph) -------------------------
    def conv_wgrad(self, x, dy, KH, KW, stride, pad, dw):
        Cout, Cin = dy.shape[-1], x.shape[-1]
        g = torch.nn.grad.conv2d_weight(_nchw(x).contiguous(), (Cout, Cin, KH, KW), _nchw(dy).contiguous(), stride=stride, padding=pad)
        dw.copy_(g.permute(0, 2, 3, 1))

    def conv_wgrad_tc_supported(self, x_shape, dy_shape, KH, KW, stride, pad):
        B, H, W, Cin = x_shape
        Cout = dy_shape[-1]
        return stride in (1, 2) and KH == KW and KH in (1, 3) and 2 * pad == KH - 1 and not (stride == 2 and KH != 3) and Cin % 8 == 0 and Cout % 8 == 0 and B * dy_shape[1] * dy_shape[2] >= 512

    def conv_wgrad_tc(self, x_pair, dy_pair, KH, KW, stride, pad, dw):
        Cin, Cout = x_pair.shape[-1] // 2, dy_pair.shape[-1] // 2
        xh, xl = x_pair[..., :Cin].float(), x_pair[..., Cin:].float()
        dh, dl = dy_pair[..., :Cout].float(), dy_pair[..., Cout:].float()
        g = lambda a, b: torch.nn.grad.conv2d_weight(_nchw(a).contiguous(), (Cout, Cin, KH, KW), _nchw(b).contiguous(), stride=stride, padding=pad)
        dw.copy_((g(xh, dh) + g(xl, dh) + g(xh, dl)).permute(0, 2, 3, 1))

    def conv_wgrad_tc_f16(self, x16, dy16, KH, KW, stride, pad, dw):
        """fb200_conv_wgrad_tc_f16: the weight gradient of the fp16-rounded operands, fp32 accumulation (the "amp" training precision)"""
        Cin, Cout = x16.shape[-1], dy16.shape[-1]
        g = torch.nn.grad.conv2d_weight(_nchw(x16.float()).contiguous(), (Cout, Cin, KH, KW), _nchw(dy16.float()).contiguous(), stride=stride, padding=pad)
        dw.copy_(g.permute(0, 2, 3, 1))

    def dilate2(self, dy, out):
        out.zero_()
        out[:, : 2 * dy.shape[1] : 2, : 2 * dy.shape[2] : 2] = dy

    def colsum(self, x2d, out):
        out.copy_(x2d.double().sum(0).float())

    def bn_train_fwd(self, x2d, gamma, beta, res2d, act, eps, momentum, rmean, rvar, save_mean, save_rstd, y2d):
        R = x2d.shape[0]
        mean = x2d.double().mean(0)
        var = ((x2d.double() - mean) ** 2).mean(0)
        save_mean.copy_(mean.float())
        save_rstd.copy_((1.0 / torch.sqrt(var + eps)).float())
        if rmean is not None:
            rmean.mul_(1 - momentum).add_(momentum * save_mean)
            rvar.mul_(1 - momentum).add_(momentum * (var * R / max(R - 1, 1)).float())
        z = (x2d - save_mean) * save_rstd * gamma + beta
        if res2d is not None:
            z = z + res2d
        y2d.copy_(_act_bw(act, z))

    def bn_train_bwd(self, x2d, dy2d, y2d, gamma, beta, save_mean, save_rstd, act, dx2d, dres2d, dgamma, dbeta):
        R = x2d.shape[0]
        xh = (x2d - save_mean) * save_rstd
        g = dy2d
        if act == 1:
            g = dy2d * ((y2d if y2d is not None else xh * gamma + beta) > 0)
        elif act == 2:
            z = (xh * gamma + beta).detach().requires_grad_(True)
            with torch.enable_grad():
                (gz,) = torch.autograd.grad(F.silu(z), z, dy2d)
            g = gz
        db = g.double().sum(0).float()
        dg = (g.double() * xh.double()).sum(0).float()
        dx2d.copy_(gamma * save_rstd * (g - db / R - xh * dg / R))
        if dres2d is not None:
            dres2d.copy_(g)
        dgamma.copy_(dg)
        dbeta.copy_(db)

    def bn_stats(self, x2d, mean, var):
        m = x2d.double().mean(0)
        mean.copy_(m.float())
        var.copy_(((x2d.double() - m) ** 2).mean(0).float())

    def bn_sync_combine(self, allst, eps, momentum, rmean, rvar, mean, rstd, inv_total):
        """fb200_bn_sync_combine: aten batch_norm_gather_stats_with_counts on the gathered [world, 2C+1] rows"""
        C = (allst.shape[1] - 1) // 2
        a = allst.double()
        n = a[:, 2 * C:2 * C + 1]
        total = n.sum()
        m = (a[:, :C] * n).sum(0) / total
        v = ((a[:, C:2 * C] + (a[:, :C] - m) ** 2) * n).sum(0) / total
        mean.copy_(m.float())
        rstd.copy_((1.0 / torch.sqrt(v + eps)).float())
        inv_total.copy_((1.0 / total).float().reshape(1))
        if rmean is not None:
            rmean.mul_(1 - momentum).add_(m.float(), alpha=momentum)
            rvar.mul_(1 - momentum).add_((v * total / (total - 1).clamp(min=1)).float(), alpha=momentum)

    def bn_apply(self, x2d, mean, rstd, gamma, beta, res2d, act, y2d):
        z = (x2d - mean) * rstd * gamma + beta
        if res2d is not None:
            z = z + res2d
        y2d.copy_(_act_bw(act, z))

    def bn_bwd_reduce(self, x2d, dy2d, y2d, gamma, beta, mean, rstd, act, sum_dy, sum_dy_xhat):
        xh, g = _bn_g(x2d, dy2d, y2d, gamma, beta, mean, rstd, act)
        sum_dy.copy_(g.double().sum(0).float())
        sum_dy_xhat.copy_((g.double() * xh.double()).sum(0).float())

    def bn_bwd_apply(self, x2d, dy2d, y2d, gamma, beta, mean, rstd, sum_dy, sum_dy_xhat, inv_count, act, dx2d, dres2d):
        xh, g = _bn_g(x2d, dy2d, y2d, gamma, beta, mean, rstd, act)
        dx2d.copy_(gamma * rstd * (g - sum_dy * inv_count - xh * sum_dy_xhat * inv_count))
        if dres2d is not None:
            dres2d.copy_(g)

    def add_act(self, a, b, dy, act, out):
        z = (a if b is None else a + b).detach().requires_grad_(dy is not None)
        if dy is None:
            out.copy_(_act_bw(act, z))
        else:
            with torch.enable_grad():
                (g,) = torch.autograd.grad(_act_bw(act, z), z, dy)
            out.copy_(g)

    def maxpool_bwd(self, x, dy, dx):
        dx.copy_(_nhwc(_via_autograd(lambda t: F.max_pool2d(t, 3, 2, 1), _nchw(x), _nchw(dy))))

    def avgpool_bwd(self, dy, dx):
        dx.copy_(_nhwc(_via_autograd(lambda t: F.avg_pool2d(t, 2, 2, 0, ceil_mode=True), _nchw(torch.zeros_like(dx)), _nchw(dy))))

    def resize_bwd(self, dy, dx):
        size = dy.shape[1:3]
        dx.copy_(_nhwc(_via_autograd(lambda t: F.interpolate(t, size=tuple(size), mode="bilinear", align_corners=False), _nchw(torch.zeros_like(dx)), _nchw(dy))))

    def layernorm_bwd(self, x2d, res2d, gamma, dy2d, eps, dx2d, dgamma, dbeta):
        s = (x2d if res2d is None else x2d + res2d).detach().clone().requires_grad_(True)
        g = gamma.detach().clone().requires_grad_(True)
        b = torch.zeros_like(gamma).requires_grad_(True)
        with torch.enable_grad():
            ds, dg, db = torch.autograd.grad(F.layer_norm(s, (s.shape[-1],), g, b, eps), (s, g, b), dy2d)
        dx2d.copy_(ds)
        dgamma.copy_(dg)
        dbeta.copy_(db)

    def attention_bwd(self, q, k, v, o, do, heads, scale, dq, dk, dv):
        qq, kk, vv = (t.detach().clone().requires_grad_(True) for t in (q, k, v))
        with torch.enable_grad():
            gq, gk, gv = torch.autograd.grad(_mha_core(qq, kk, vv, heads, scale), (qq, kk, vv), do)
        dq.copy_(gq)
        dk.copy_(gk)
        dv.copy_(gv)

    def msda_bwd(self, value, oa, ref, do, shapes, P, heads, dvalue, doa):
        vv, oo = value.detach().clone().requires_grad_(True), oa.detach().clone().requires_grad_(True)
        out = torch.empty((value.shape[0], oa.shape[1], value.shape[2]))
        with torch.enable_grad():
            B, S, C = vv.shape
            Q, L, hd = oo.shape[1], len(shapes), C // heads
            off = oo[..., : heads * L * P * 2].reshape(B, Q, heads, L, P, 2)
            aw = torch.softmax(oo[..., heads * L * P * 2 : heads * L * P * 3].reshape(B, Q, heads, L * P), -1).reshape(B, Q, heads, L, P)
            r = ref.reshape(B, Q, 1, 1, 1, 4)
            loc = r[..., :2] + off / P * r[..., 2:] * 0.5
            vals = vv.reshape(B, S, heads, hd).split([h * w for h, w in shapes], dim=1)
            grids = 2 * loc - 1
            sampled = []
            for lid, (H_, W_) in enumerate(shapes):
                vl = vals[lid].flatten(2).transpose(1, 2).reshape(B * heads, hd, H_, W_)
                g = grids[:, :, :, lid].transpose(1, 2).flatten(0, 1)
                sampled.append(F.grid_sample(vl, g, mode="bilinear", padding_mode="zeros", align_corners=False))
            awt = aw.transpose(1, 2).reshape(B * heads, 1, Q, L * P)
            o = (torch.stack(sampled, dim=-2).flatten(-2) * awt).sum(-1).view(B, heads * hd, Q).transpose(1, 2)
            gv, go = torch.autograd.grad(o, (vv, oo), do)
        dvalue.add_(gv)
        doa.copy_(go)

    # ---- DETR training criterion (criterion.py) --------------------------------------------------------------
    def detr_match_cost(self, logits, boxes, tl, tb, toff, wts, alpha, gamma, cost):
        from oracle import criterion_oracle as CO
        L, B, Q, C = logits.shape
        for l in range(L):
            for b in range(B):
                t0, t1 = int(toff[b]), int(toff[b + 1])
                if t1 > t0:
                    cost[l, t0:t1] = CO.match_cost(logits[l, b], boxes[l, b], tl[t0:t1].long(), tb[t0:t1], wts[0], wts[1], wts[2], alpha, gamma).T

    def hungarian(self, cost, toff, B, max_targets, match_q):
        from scipy.optimize import linear_sum_assignment
        for l in range(cost.shape[0]):
            for b in range(B):
                t0, t1 = int(toff[b]), int(toff[b + 1])
                if t1 > t0:
                    r, c = linear_sum_assignment(cost[l, t0:t1].numpy())
                    match_q[l, t0 + torch.as_tensor(r)] = torch.as_tensor(c, dtype=torch.int32)

    def detr_loss(self, logits, boxes, tl, tb, toff, match_q, num_boxes, wts, alpha, gamma, losses, g_logits, g_l1, g_giou):
        from oracle import criterion_oracle as CO
        L, B, Q, C = logits.shape
        has = tl is not None
        targets = [(tl[int(toff[b]):int(toff[b + 1])].long(), tb[int(toff[b]):int(toff[b + 1])]) if has else (torch.zeros(0, dtype=torch.long), torch.zeros((0, 4))) for b in range(B)]
        with torch.enable_grad():
            for l in range(L):
                lg = logits[l].detach().clone().requires_grad_(True)
                bx = boxes[l].detach().clone().requires_grad_(True)
                idx = [(match_q[l, int(toff[b]):int(toff[b + 1])].long() if has else torch.zeros(0, dtype=torch.long), torch.arange(len(targets[b][0]))) for b in range(B)]
                v, b1, gi = CO.layer_losses(lg, bx, targets, idx, num_boxes, alpha, gamma, wts)
                losses[l] = torch.stack([v, b1, gi]).detach()
                g_logits[l] = torch.autograd.grad(v, lg, retain_graph=True)[0]
                g_l1[l] = torch.autograd.grad(b1, bx, retain_graph=True)[0] if has else 0
                g_giou[l] = torch.autograd.grad(gi, bx)[0] if has else 0

    # ---- optimiser step (train_step.py; same control-block layout) -------------------------------------------
    def optim_workspace(self, device):
        return torch.zeros(4, dtype=torch.float64)

    def grad_stats(self, grads, ws):
        ws[0] = float((grads.double() ** 2).sum())
        ws[1] = 0.0 if bool(torch.isfinite(grads).all()) else 1.0

    def optim_finalize(self, ws, ctrl, max_norm, clip_passes, inv_world, use_scaler, growth, backoff, growth_interval, beta1, beta2):
        ic = ctrl.view(torch.int32)
        scale = float(ctrl[0]) if use_scaler else 1.0
        pre = inv_world / scale
        norm = math.sqrt(float(ws[0])) * pre if math.isfinite(float(ws[0])) else float("inf")
        bad = int(ws[1] != 0 or not math.isfinite(norm))
        coef, nrm = 1.0, norm
        for _ in range(clip_passes if max_norm > 0 else 0):
            c = min(max_norm / (nrm + 1e-6), 1.0) if math.isfinite(nrm) else 0.0
            coef *= c
            nrm *= c
        ic[2] = bad
        ctrl[3], ctrl[4], ctrl[8] = norm, pre * coef, coef
        if not bad:
            ic[5] += 1
            ctrl[6] = 1.0 - beta1 ** int(ic[5])
            ctrl[7] = math.sqrt(1.0 - beta2 ** int(ic[5]))
        if use_scaler:
            if bad:
                ctrl[0] = scale * backoff
                ic[1] = 0
            elif int(ic[1]) + 1 == growth_interval:
                ctrl[0] = scale * growth
                ic[1] = 0
            else:
                ic[1] += 1

    def adamw_step(self, params, grads, m, v, chunk_start, chunk_len, chunk_seg, seg_lr, seg_wd, seg_active, lr_factor, beta1, beta2, eps, ctrl):
        if int(ctrl.view(torch.int32)[2]):
            return
        gmul, bc1, bc2s = float(ctrl[4]), float(ctrl[6]), float(ctrl[7])
        for s0, ln, sg in zip(chunk_start.tolist(), chunk_len.tolist(), chunk_seg.tolist()):
            if seg_active is not None and not int(seg_active[sg]):
                continue
            sl = slice(s0, s0 + ln)
            lr, wd = float(seg_lr[sg]) * lr_factor, float(seg_wd[sg])
            g = grads[sl] * gmul
            params[sl] *= 1.0 - lr * wd
            m[sl] = m[sl] + (g - m[sl]) * (1.0 - beta1)
            v[sl] = v[sl] * beta2 + (1.0 - beta2) * (g * g)
            params[sl] -= (lr / bc1) * (m[sl] / (v[sl].sqrt() / bc2s + eps))
